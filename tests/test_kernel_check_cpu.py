"""
The per-element checker of tests/kernel_check.py catches the faults a whole-tensor relative L2 lets through.
A CPU fp64 convolution stands in for the kernel: its correctly bf16-rounded result must pass, and each injected
defect (the kind a kernel makes at a tile edge, a channel-block tail or a persistent-loop wrap) must fail with the
coordinates of the element it broke.
"""
import re

import pytest
import torch
import torch.nn.functional as F

from tests.kernel_check import (BF16_ROUNDING, assert_elementwise, check_poisoned, normalize_kernel_name,
                                poisoned)

N, H, W, C, K = 2, 16, 16, 64, 32


def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


@pytest.fixture(scope="module")
def conv_case():
    g = torch.Generator().manual_seed(0)
    x = (torch.randn(N, H, W, C, generator=g) + 0.5).bfloat16().double()
    w = (torch.randn(K, 3, 3, C, generator=g) / (9 * C) ** 0.5).bfloat16().double()
    wt = w.permute(0, 3, 1, 2)
    ref = nhwc(F.conv2d(nchw(x), wt, padding=1))
    mag = nhwc(F.conv2d(nchw(x).abs(), wt.abs(), padding=1))
    return x, w, ref, mag


def _check(out, case, label):
    _, _, ref, mag = case
    return assert_elementwise(out, ref, mag, BF16_ROUNDING, label=label)


def _fails_at(out, case, label, n=None, h=None, w=None, c=None):
    with pytest.raises(AssertionError) as e:
        _check(out, case, label)
    msg = str(e.value)
    m = re.search(r"\(n, h, w, c\) = \((\d+), (\d+), (\d+), (\d+)\)", msg)
    assert m, msg
    got = tuple(int(v) for v in m.groups())
    for want, have in zip((n, h, w, c), got):
        assert want is None or want == have, msg
    return got


def test_rounded_reference_passes(conv_case):
    out = conv_case[2].bfloat16()
    worst, worst_acc = _check(out, conv_case, "bf16(ref)")
    assert worst <= 1.0 and worst_acc == 0.0


def test_bf16_output_with_residual_passes():
    g = torch.Generator().manual_seed(1)
    acc = torch.randn(4, 4, 4, 16, generator=g, dtype=torch.float64) * 3
    res = torch.randn(4, 4, 4, 16, generator=g).bfloat16().double()
    out = (acc.bfloat16().double() + res).bfloat16()   # the kernel's two rounding points
    assert_elementwise(out, acc + res, acc.abs(), 2 * BF16_ROUNDING, addends=(res,), label="conv + residual")
    with pytest.raises(AssertionError):   # one rounding point's worth does not cover two
        assert_elementwise(out, acc + res, acc.abs(), BF16_ROUNDING, addends=(res,), label="one rounding")


def test_zeroed_pixel_fails(conv_case):
    out = conv_case[2].bfloat16()
    out[1, 5, 7, :] = 0
    _fails_at(out, conv_case, "zeroed pixel", 1, 5, 7)


def test_pixel_from_neighbouring_image_fails(conv_case):
    out = conv_case[2].bfloat16()
    out[1, 9, 3, :] = out[0, 9, 3, :]
    _fails_at(out, conv_case, "pixel of the other image", 1, 9, 3)


def test_missing_tap_in_one_tile_fails(conv_case):
    x, w, ref, _ = conv_case
    # one 8 (w) x 16 (h) pixel tile at w = 8..15 of image 0 loses its tap (r, s) = (0, 2)
    tap = F.pad(nchw(x), (1, 1, 1, 1))[:, :, 0:H, 2:W + 2]
    contrib = nhwc(F.conv2d(tap, w.permute(0, 3, 1, 2)[:, :, 0:1, 2:3]))
    out = ref.clone()
    out[0, :, 8:16, :] -= contrib[0, :, 8:16, :]
    got = _fails_at(out.bfloat16(), conv_case, "tap (0, 2) missing in one tile", n=0)
    assert 8 <= got[2] < 16


def test_missing_channel_block_in_one_tile_fails(conv_case):
    x, w, ref, _ = conv_case
    # the input channels 32..63 (one 32-channel block) left out of one 8 x 16 tile of image 1
    part = nhwc(F.conv2d(nchw(x[..., 32:]), w[..., 32:].permute(0, 3, 1, 2), padding=1))
    out = ref.clone()
    out[1, :, 0:8, :] -= part[1, :, 0:8, :]
    got = _fails_at(out.bfloat16(), conv_case, "channel block missing in one tile", n=1)
    assert got[2] < 8


def test_one_channel_scaled_fails(conv_case):
    out = conv_case[2].clone()
    out[..., 13] *= 1 + 2.0 ** -6
    _fails_at(out.bfloat16(), conv_case, "channel 13 scaled by 1 + 2^-6", c=13)


def test_poisoned_layout():
    for dt in (torch.bfloat16, torch.float32):
        t = poisoned((3, 5, 7, 16), dt, device="cpu")
        assert t.data_ptr() % 1024 == 0 and t.is_contiguous() and t.dtype == dt
        assert bool(torch.isnan(t).all())
        t.zero_()
        check_poisoned(t, "fully written")


def test_unwritten_element_fails():
    t = poisoned((2, 4, 4, 8), torch.bfloat16, device="cpu")
    t.fill_(1.0)
    t[1, 2, 3, 5] = float("nan")
    with pytest.raises(AssertionError, match=r"never written; first at \(n, h, w, c\) = \(1, 2, 3, 5\)"):
        check_poisoned(t, "one element left")
    # the checker itself also refuses a NaN
    ref = torch.ones(2, 4, 4, 8, dtype=torch.float64)
    with pytest.raises(AssertionError, match=r"\(1, 2, 3, 5\)"):
        assert_elementwise(t, ref, ref, BF16_ROUNDING, label="NaN in the output")


@pytest.mark.parametrize("side", ["before", "after"])
def test_write_into_guard_fails(side):
    t = poisoned((2, 4, 4, 8), torch.float32, device="cpu")
    t.fill_(0.0)
    buf, lo, hi, guard = t._poison
    if side == "before":
        buf[lo - 4:lo] = 0                       # one fp32 element just before the start
    else:
        buf[hi + 100] = 0x3F                     # one byte a little past the end
    with pytest.raises(AssertionError, match=f"guard bytes {side}"):
        check_poisoned(t, "stray write")


def test_kernel_name_normalisation():
    assert normalize_kernel_name("void b200::conv_tc2h_kernel<64, 1, 1, 1>(CUtensorMap, CUtensorMap)") == \
        "conv_tc2h_kernel<64,1,1,1>"
    assert normalize_kernel_name("void b200::conv_tc2_kernel<32, 1>(CUtensorMap, ConvTcArgs)") == \
        "conv_tc2_kernel<32,1,0>"
    assert normalize_kernel_name("void b200::conv_tc2_kernel<16, 2, false>(CUtensorMap)") == \
        "conv_tc2_kernel<16,2,0>"
    assert normalize_kernel_name("void b200::wgrad_tc_kernel<32, 1, (bool)0, true>(int)") == \
        "wgrad_tc_kernel<32,1,0,1>"
    assert normalize_kernel_name("void b200::repitch_rows_kernel<__nv_bfloat16>(const T*, T*)") == \
        "repitch_rows_kernel<bf16>"
    assert normalize_kernel_name("parity_merge_add_kernel(const __nv_bfloat16*, int)") == "parity_merge_add_kernel"
    assert normalize_kernel_name("b200::wgrad_tc2h_kernel(CUtensorMap, CUtensorMap, WgradHaloArgs)") == \
        "wgrad_tc2h_kernel"
