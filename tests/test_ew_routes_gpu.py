"""
The kernels between the convolutions by dispatch route: batch-norm statistics, the fused BN + skip + ReLU + dropout
forward and backward, pooling, the classifier head, the layout kernels and the fp32 evaluation path. Every row
asserts the exact set of kernels it launched, that no byte outside an output was written and no output element left
unwritten (NaN-poisoned float outputs between guards; uint8 outputs run twice, poisoned with 0x00 and with 0xFF, and
must equal the reference exactly both times), and every output element against an fp64 reference
(tests/kernel_check.py). Summation bounds come from the reduction structure of each kernel (gamma_n = n u / (1 - n u)
with n the longest chain of fp32 additions), not from a fixed tolerance; dropout keep bits are recomputed exactly
from a port of the kernels' counter RNG.
"""
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.kernel_check import (BF16_ROUNDING, assert_elementwise, check_poisoned, drop_threshold, dropout_keep,
                                kernels_launched, poisoned)

pytestmark = pytest.mark.gpu

EPS = 1e-5
U32 = 2.0 ** -24            # unit roundoff of fp32
EW_THREADS = 256
# fp32 / rounding-order slack of the element-wise affine x * sc + sh (sc = gamma * invstd, sh = beta - mean * sc in
# fp32, rsqrtf for a variance) and the second-order terms of chained bf16 roundings, per unit of |operands|
AFFINE_ACC = 2.0 ** -12


def _ops():
    from pytorch_ddp_resnet_b200 import _lib, ops
    return ops, _lib


def gamma_n(n):
    """Higham's gamma_n: a chain of n fp32 additions errs by at most gamma_n * sum |terms|."""
    return n * U32 / (1 - n * U32)


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def reduce_chain(rows, C, bps):
    """Longest fp32 addition chain of the reduction kernels (bn_stats_kernel, bn_act_bwd_reduce_kernel) as api.cu
    bn_blocks and elementwise.cuh ReduceGeom / block_row_range lay them out: a thread sums its rows of the block's
    range (stride RP), then one thread sums the RP row lanes of the block; blocks meet in fp64. The grid is sized by
    the first channel chunk; a second chunk (blockIdx.y > 0) may have fewer groups and so a longer lane sum."""
    CG = C // 8
    RP0 = EW_THREADS // min(EW_THREADS, CG)
    grid = max(1, min(_sms() * bps, -(-rows // RP0)))
    n = 0
    for cg0 in range(0, CG, EW_THREADS):
        RP = EW_THREADS // min(EW_THREADS, CG - cg0)
        passes = -(-rows // RP)
        n = max(n, -(-passes // grid) + RP)
    return n


def _gen(label):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(label.encode()))


def _assert_kernels(launched, expected, label):
    assert sorted(launched) == sorted(expected), f"{label}: launched {launched}, expected {sorted(expected)}"


def _report(label, launched, worst):
    print(f"[route] {label}: {'+'.join(launched)}; worst ratio {worst[0]:.4f}, accumulation term {worst[1]:.4f}")


def _worst(*ws):
    return max(w[0] for w in ws), max(w[1] for w in ws)


def _assert_bytes_equal(got, ref, label, bits_per_byte=None):
    """uint8 outputs exactly; names the first differing element ((n, h, w, c) of the unit for a bit mask)."""
    if torch.equal(got, ref):
        return
    diff = (got != ref).reshape(-1).nonzero()
    i = int(diff[0].item())
    shape = tuple(got.shape)
    coords = []
    rem = i
    for s in reversed(shape):
        coords.append(rem % s)
        rem //= s
    coords = list(reversed(coords))
    g, r = int(got.reshape(-1)[i].item()), int(ref.reshape(-1)[i].item())
    if bits_per_byte:
        j = ((g ^ r) & -(g ^ r)).bit_length() - 1
        coords[-1] = coords[-1] * 8 + j
        raise AssertionError(f"{label}: {diff.numel()} mask bytes differ; first at (n, h, w, c) = {tuple(coords)}: "
                             f"bit {(g >> j) & 1}, reference {(r >> j) & 1} (bytes {g:#04x} / {r:#04x})")
    raise AssertionError(f"{label}: {diff.numel()} bytes differ; first at {tuple(coords)}: {g} != {r}")


def _pack_bits(bits):
    """bool [..., C] -> uint8 [..., C/8], bit j of byte g = channel 8 g + j."""
    shp = bits.shape
    b = bits.reshape(*shp[:-1], shp[-1] // 8, 8).to(torch.int32)
    w = (1 << torch.arange(8, device=bits.device, dtype=torch.int32))
    return (b * w).sum(-1).to(torch.uint8)


# ---------------------------------------------------------------------------------------------------------------
# 1. batch statistics: bn_stats, bn_stats_finalize, bn_running_update
# ---------------------------------------------------------------------------------------------------------------
# (C, rows, data); RP = 256 / min(256, C/8) rows per pass
STATS = [
    (8, 1, "normal"), (8, 255, "normal"), (8, 3_000_001, "normal"),        # RP = 256; several unrolled batches
    (24, 84, "normal"), (24, 50_001, "shifted"),                            # RP = 85 does not divide 256
    (160, 11, "normal"), (160, 131_072, "normal"), (160, 131_072, "shifted"),   # WRN 128x32x32x160
    (640, 7, "normal"), (640, 8_191, "normal"),                             # RP = 3 (ragged last pass)
    (2048, 1, "normal"), (2048, 4_099, "shifted"),                          # one group per thread
    (2056, 3_001, "normal"),                                                # second chunk: one group, RP = 256
    (4096, 2_049, "normal"), (4096, 600, "shifted"),                        # two full chunks
]
CONST_C, ZERO_C, CONST_V = 3, 5, 1.5      # a constant channel (var = 0, exact sums) and an all-zero one


def _stats_input(rows, C, data, g):
    mu, sd = (0.5, 1.0) if data == "normal" else (8.0, 0.25)
    x = (torch.randn(rows, C, device="cuda", generator=g) * sd + mu).bfloat16()
    x[:, CONST_C] = CONST_V
    x[:, ZERO_C] = 0
    return x


def _stats_ref(x, n):
    """fp64 mean / biased var of x [rows, C] and the gamma_n bounds of the kernel's fp32 sums on them."""
    xd = x.double()
    rows = xd.shape[0]
    m = xd.mean(0)
    var = (xd - m).pow(2).mean(0)
    gm = gamma_n(n)
    dmean = gm * xd.abs().sum(0) / rows
    dvar = gm * (xd * xd).sum(0) / rows + 2 * m.abs() * dmean + dmean * dmean
    return m, var, dmean, dvar


def _invstd_bound(var, dvar):
    """|invstd' - invstd| for any var' within dvar of var (monotone in var; var' < 0 clamps to 0)."""
    f = lambda v: (v.clamp_min(0) + np.float32(EPS).item()).rsqrt()
    return torch.maximum(f(var - dvar) - f(var), f(var) - f(var + dvar))


def _check_stats(mean, invstd, x, n, label):
    m, var, dmean, dvar = _stats_ref(x, n)
    ref_is = (var + float(np.float32(EPS))).rsqrt()
    w1 = assert_elementwise(mean, m, dmean, U32, acc=1.0, label=f"{label} mean")
    w2 = assert_elementwise(invstd, ref_is, _invstd_bound(var, dvar), U32, acc=1.0, label=f"{label} invstd")
    # the constant and the zero channel: exact sums, var = 0, invstd = eps^-1/2 bit for bit
    is0 = np.float32(1.0 / math.sqrt(float(np.float32(EPS))))
    for c, v in ((CONST_C, CONST_V), (ZERO_C, 0.0)):
        if c < x.shape[1]:
            assert mean[c].item() == v and invstd[c].item() == is0, \
                f"{label}: channel {c} (constant {v}): mean {mean[c].item()!r}, invstd {invstd[c].item()!r} != {is0!r}"
    return _worst(w1, w2), (m, var, dmean, dvar)


def _check_running(rm, rv, rm0, rv0, m, var, dmean, dvar, rows, mom, label, var_operands=None):
    """torch.nn.BatchNorm2d: running = (1 - momentum) running + momentum * batch stat, the UNBIASED variance.
    dmean / dvar: bounds of the batch statistics' summation error; the fp32 update itself rounds up to four times
    (the variance recovered from invstd as 1 / invstd^2 - eps: var_operands = 1 / invstd^2 joins that scale)."""
    corr = rows / (rows - 1) if rows > 1 else 1.0
    ref_m = (1 - mom) * rm0.double() + mom * m
    ref_v = (1 - mom) * rv0.double() + mom * var * corr
    scale_m = (1 - mom) * rm0.double().abs() + mom * m.abs()
    scale_v = (1 - mom) * rv0.double().abs() + mom * corr * (var.abs() if var_operands is None else var_operands)
    w1 = assert_elementwise(rm, ref_m, mom * dmean, 4 * U32, acc=1.0, scale64=scale_m, label=f"{label} running_mean")
    w2 = assert_elementwise(rv, ref_v, mom * dvar * corr, 4 * U32, acc=1.0, scale64=scale_v,
                            label=f"{label} running_var")
    return _worst(w1, w2)


def _stats_id(r):
    return f"C{r[0]}-rows{r[1]}-{r[2]}"


@pytest.mark.parametrize("row", STATS, ids=_stats_id)
def test_bn_stats_route(row):
    ops, _lib = _ops()
    C, rows, data = row
    label = f"bn_stats {_stats_id(row)}"
    g = _gen(label)
    x = _stats_input(rows, C, data, g)
    mean, invstd = poisoned((C,), torch.float32), poisoned((C,), torch.float32)
    rm0 = torch.randn(C, device="cuda", generator=g) * 0.1
    rv0 = torch.rand(C, device="cuda", generator=g) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.full((), 7, dtype=torch.int64, device="cuda")
    mom = 0.1
    nws = _lib.load().b200_bn_workspace_bytes(rows, C)
    ws = ops.bn_accumulators(x.device, nws)

    def call():
        _lib.call("b200_bn_stats", x.data_ptr(), rows, C, EPS, mom, mean.data_ptr(), invstd.data_ptr(), rm.data_ptr(),
                  rv.data_ptr(), nbt.data_ptr(), ws.data_ptr(), nws, ops._stream())

    _, launched = kernels_launched(call)
    _assert_kernels(launched, ["bn_stats_kernel"], label)
    check_poisoned(mean, "mean")
    check_poisoned(invstd, "invstd")
    w, (m, var, dmean, dvar) = _check_stats(mean, invstd, x, reduce_chain(rows, C, 4), label)
    w = _worst(w, _check_running(rm, rv, rm0, rv0, m, var, dmean, dvar, rows, mom, label))
    assert nbt.item() == 8, f"{label}: num_batches_tracked {nbt.item()} (must go up by exactly one)"
    assert not bool(ws[:2 * C].any()), f"{label}: accumulators not cleared"
    _report(label, launched, w)


@pytest.mark.parametrize("C", [24, 4096])
def test_bn_stats_finalize_and_running_update(C):
    """bn_stats_finalize_kernel from hand-filled fp64 slots (they must be drained to zero), and
    bn_running_update_kernel from given mean / invstd (the update of statistics a conv epilogue produced)."""
    ops, _lib = _ops()
    label = f"bn_stats_finalize C{C}"
    g = _gen(label)
    rows = 1000
    x = _stats_input(rows, C, "normal", g).double()
    nws = _lib.load().b200_bn_workspace_bytes(rows, C)
    ws = torch.zeros((nws + 7) // 8, dtype=torch.float64, device="cuda")
    stride = max(512, (2 * C + 31) // 32 * 32) + 32      # common.cuh bn_slot_stride
    parts = torch.chunk(x, 8)                           # BN_SLOTS = 8 copies, one partial per slot
    for k, part in enumerate(parts):
        ws[k * stride:k * stride + C] = part.sum(0)
        ws[k * stride + C:k * stride + 2 * C] = (part * part).sum(0)
    mean, invstd = poisoned((C,), torch.float32), poisoned((C,), torch.float32)
    rm0 = torch.randn(C, device="cuda", generator=g) * 0.1
    rv0 = torch.rand(C, device="cuda", generator=g) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")

    def call():
        _lib.call("b200_bn_stats_finalize", rows, C, EPS, 0.1, mean.data_ptr(), invstd.data_ptr(), rm.data_ptr(),
                  rv.data_ptr(), nbt.data_ptr(), ws.data_ptr(), nws, ops._stream())

    _, launched = kernels_launched(call)
    _assert_kernels(launched, ["bn_stats_finalize_kernel"], label)
    check_poisoned(mean, "mean")
    check_poisoned(invstd, "invstd")
    assert not bool(ws.any()), f"{label}: slots not drained"
    # fp64 sums in: only the fp64 finalize (16 ulps of fp64 here) and the fp32 outputs round
    w, (m, var, dmean, dvar) = _check_stats(mean, invstd, x.bfloat16(), 1, label)
    w = _worst(w, _check_running(rm, rv, rm0, rv0, m, var, dmean, dvar, rows, 0.1, label))
    assert nbt.item() == 1
    _report(label, launched, w)

    # bn_running_update_kernel: var = 1 / invstd^2 - eps in fp32 from the given fp32 invstd
    label = f"bn_running_update C{C}"
    rm, rv = rm0.clone(), rv0.clone()

    def call2():
        _lib.call("b200_bn_running_update", mean.data_ptr(), invstd.data_ptr(), rows, C, EPS, 0.1, rm.data_ptr(),
                  rv.data_ptr(), nbt.data_ptr(), ops._stream())

    _, launched = kernels_launched(call2)
    _assert_kernels(launched, ["bn_running_update_kernel"], label)
    isd = invstd.double()
    var_in = (1 / (isd * isd) - float(np.float32(EPS))).clamp_min(0)
    zero = torch.zeros_like(isd)
    w2 = _check_running(rm, rv, rm0, rv0, mean.double(), var_in, zero, zero, rows, 0.1, label,
                        var_operands=1 / (isd * isd))
    assert nbt.item() == 2, f"{label}: num_batches_tracked {nbt.item()} != 2"
    _report(label, launched, w2)


# ---------------------------------------------------------------------------------------------------------------
# 2./3. bn_act_fwd: the five instantiations, exact dropout bits, mask bytes bit for bit
# ---------------------------------------------------------------------------------------------------------------
FWD = "bn_act_fwd_kernel<{}>"
# (rule: the api.cu b200_bn_act_fwd branch, N, H, W, C, options, kernel template arguments)
BN_FWD = [
    ("!skip, !drop -> <4,4,false,0>", 4, 16, 16, 160, dict(relu=True), "4,4,0,0"),
    ("!skip, !drop, no ReLU, no affine", 2, 8, 8, 64, dict(relu=False, affine=False), "4,4,0,0"),
    ("!skip, !drop, eval mode (stat_is_var)", 2, 8, 8, 640, dict(relu=True, eval=True), "4,4,0,0"),
    ("!skip, !drop, fused running update, two channel chunks", 2, 4, 4, 4096, dict(relu=True, running=True),
     "4,4,0,0"),
    ("!skip, !drop, C = 2056: second chunk of one group", 2, 5, 3, 2056, dict(relu=True), "4,4,0,0"),
    ("skip SAME, !drop -> <2,3,true,0>", 4, 16, 16, 160, dict(relu=True, skip="same"), "2,3,1,0"),
    ("skip SUBSAMPLE_PAD (skip_C < C), !drop", 2, 8, 8, 640, dict(relu=True, skip="pad"), "2,3,1,0"),
    ("drop + ReLU -> <2,4,false,1>", 4, 16, 16, 160, dict(relu=True, p=0.3), "2,4,0,1"),
    ("drop + ReLU, C = 4096", 2, 3, 5, 4096, dict(relu=True, p=0.3), "2,4,0,1"),
    ("drop, no ReLU, no mask -> <2,4,false,1>", 2, 8, 8, 160, dict(relu=False, p=0.3, mask=False), "2,4,0,1"),
    ("drop, no ReLU, mask -> keepbits <4,3,false,2>", 4, 16, 16, 160, dict(relu=False, p=0.3), "4,3,0,2"),
    ("drop, no ReLU, mask, C = 2056", 2, 5, 3, 2056, dict(relu=False, p=0.5), "4,3,0,2"),
    ("skip SAME + drop + ReLU -> <2,3,true,2>", 4, 16, 16, 160, dict(relu=True, skip="same", p=0.3), "2,3,1,2"),
    ("skip SUBSAMPLE_PAD + drop + ReLU", 2, 8, 8, 640, dict(relu=True, skip="pad", p=0.3), "2,3,1,2"),
    ("skip SAME + drop + ReLU, C = 4096", 2, 3, 5, 4096, dict(relu=True, skip="same", p=0.3), "2,3,1,2"),
    ("skip SAME + drop, no ReLU -> <2,3,true,2>", 4, 8, 8, 160, dict(relu=False, skip="same", p=0.3), "2,3,1,2"),
    ("drop + ReLU after a tick (step counter 3)", 2, 8, 8, 160, dict(relu=True, p=0.1, ticks=3), "2,4,0,1"),
]


def _fwd_id(r):
    o = r[5]
    parts = [f"{r[1]}x{r[2]}x{r[3]}x{r[4]}"] + [k if v is True else f"{k}{v}" for k, v in sorted(o.items())]
    return "-".join(parts)


def _fwd_inputs(N, H, W, C, o, g):
    x = (torch.randn(N, H, W, C, device="cuda", generator=g) * 1.3 + 0.4).bfloat16()
    mean = torch.randn(C, device="cuda", generator=g) * 0.3 + 0.4
    var = torch.rand(C, device="cuda", generator=g) * 1.5 + 0.3
    invstd = (var.double() + EPS).rsqrt().float()
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.3
    skip = None
    if o.get("skip") == "same":
        skip = torch.randn(N, H, W, C, device="cuda", generator=g).bfloat16()
    elif o.get("skip") == "pad":
        skip = torch.randn(N, 2 * H, 2 * W, C // 2 - 8 * (C >= 64), device="cuda", generator=g).bfloat16()
    return x, mean, var, invstd, gamma, beta, skip


def fwd_reference(x, mean, stat, gamma, beta, skip, o, seed, offset, y_kernel):
    """fp64 y of bn_act_fwd at the kernel's rounding points, its bound operands, and the reference mask byte.
    Returns (ref, scale64, mag, npts, keep, gate) with gate = active AND kept (the mask bits)."""
    N, H, W, C = x.shape
    xd = x.double()
    relu, p = o.get("relu", True), o.get("p", 0.0)
    if o.get("affine", True):
        is64 = (stat.double() + float(np.float32(EPS))).rsqrt() if o.get("eval") else stat.double()
        sc = gamma.double() * is64
        sh = beta.double() - mean.double() * sc
    else:
        sc = torch.ones(C, dtype=torch.float64, device=x.device)
        sh = torch.zeros_like(sc)
    pre = xd * sc + sh
    # operands of the fp32 x * sc + (beta - mean * sc): the shift cancels when |mean| >> std
    mag = (xd * sc).abs() + beta.double().abs() + (mean.double() * sc).abs() if o.get("affine", True) else xd.abs()
    scale = pre.abs()
    npts = 1
    if skip is not None:
        s = torch.zeros_like(pre)
        if o["skip"] == "same":
            s = skip.double()
        else:
            s[..., :skip.shape[-1]] = skip.double()[:, ::2, ::2, :]
        pre = pre + s
        scale = scale + s.abs()
        mag = mag + s.abs()
        npts += 1
    keep = torch.ones_like(pre, dtype=torch.bool)
    mult = torch.ones_like(pre)
    if p > 0:
        keep = torch.from_numpy(dropout_keep(N * H * W, C, p, seed, offset)).to(x.device).reshape(pre.shape)
        inv_keep = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
        mult = torch.where(keep, torch.full_like(pre, inv_keep), torch.zeros_like(pre))
        npts += 1
    bound_pre = npts * BF16_ROUNDING * scale + AFFINE_ACC * mag
    active = torch.ones_like(keep)
    if relu:
        active = pre > 0
        # within rounding reach of zero the kernel's own sign decides: teacher-forced from its y (0 = gated)
        near = pre.abs() <= bound_pre
        active = torch.where(near & keep, y_kernel.double() != 0, active)
    ref = torch.where(active, pre, torch.zeros_like(pre)) * mult
    gate = (active & keep) if relu else keep
    return ref, scale * mult, mag * mult, npts, keep, gate


@pytest.mark.parametrize("row", BN_FWD, ids=_fwd_id)
def test_bn_act_fwd_route(row):
    ops, _lib = _ops()
    rule, N, H, W, C, o, targs = row
    label = f"bn_act_fwd {_fwd_id(row)}"
    g = _gen(label)
    x, mean, var, invstd, gamma, beta, skip = _fwd_inputs(N, H, W, C, o, g)
    relu, p, want_mask = o.get("relu", True), o.get("p", 0.0), o.get("mask", True)
    affine = o.get("affine", True)
    stat = var if o.get("eval") else invstd
    counter = ops.step_counter(x.device)
    for _ in range(o.get("ticks", 0)):
        ops.tick(x.device)
    offset = int(counter.item()) if p > 0 else None
    seed = 0x5EED0000 + zlib.crc32(label.encode())
    skip_mode = {None: 0, "same": _lib.SKIP_SAME, "pad": _lib.SKIP_SUBSAMPLE_PAD}[o.get("skip")]
    rm0 = torch.randn(C, device="cuda", generator=g) * 0.1
    rv0 = torch.rand(C, device="cuda", generator=g) + 0.5
    nbt = torch.full((), 3, dtype=torch.int64, device="cuda")
    p_ = ops._p
    runs = []
    for fill in ((0x00, 0xFF) if want_mask else (0xFF,)):
        y = poisoned((N, H, W, C), torch.bfloat16)
        mask = poisoned((N, H, W, C // 8), torch.uint8, byte=fill) if want_mask else None
        rm, rv = rm0.clone(), rv0.clone()
        running = o.get("running", False)

        def call():
            _lib.call("b200_bn_act_fwd", x.data_ptr(), y.data_ptr(), N, H, W, C, p_(mean if affine else None),
                      p_(stat if affine else None), int(bool(o.get("eval"))), EPS, p_(gamma if affine else None),
                      p_(beta if affine else None), p_(skip), skip_mode, 0 if skip is None else skip.shape[-1],
                      int(relu), float(p), seed, counter.data_ptr() if p > 0 else None, p_(rm if running else None),
                      p_(rv if running else None), p_(nbt if running else None), 0.1, p_(mask), ops._stream())

        _, launched = kernels_launched(call)
        _assert_kernels(launched, [FWD.format(targs)], f"{label} ({rule})")
        check_poisoned(y, "y")
        if mask is not None:
            check_poisoned(mask, f"mask (fill {fill:#04x})")
        runs.append((y, mask, rm, rv))
    y, mask, rm, rv = runs[0]
    ref, scale, mag, npts, keep, gate = fwd_reference(x, mean, stat, gamma, beta, skip, o, seed, offset, y)
    w = assert_elementwise(y, ref, mag, npts * BF16_ROUNDING, acc=AFFINE_ACC, scale64=scale, label=f"{label} y")
    if p > 0:   # the exact dropout bits: a dropped unit is +-0, a kept active one is not
        bad = ((y != 0) & ~keep).nonzero()
        assert bad.numel() == 0, f"{label}: unit (n, h, w, c) = {tuple(bad[0].tolist())} dropped by the RNG is non-zero"
    for y2, mask2, _, _ in runs[1:]:
        assert torch.equal(y2.view(torch.int16), y.view(torch.int16)), f"{label}: the two runs differ"
    if want_mask:
        ref_mask = _pack_bits(gate)
        for _, m_, _, _ in runs:
            _assert_bytes_equal(m_, ref_mask, f"{label} mask", bits_per_byte=8)
    if o.get("running"):
        m = mean.double()
        # the kernel recovers the variance from invstd in fp32: 1 / invstd^2 - eps
        isd = invstd.double()
        var_in = (1 / (isd * isd) - float(np.float32(EPS))).clamp_min(0)
        rows = N * H * W
        zero = torch.zeros_like(m)
        w = _worst(w, _check_running(rm, rv, rm0, rv0, m, var_in, zero, zero, rows, 0.1, label,
                                     var_operands=1 / (isd * isd)))
        assert nbt.item() == 3 + len(runs), f"{label}: num_batches_tracked {nbt.item()} (one per launch)"
    _report(label, [FWD.format(targs)], w)


# ---------------------------------------------------------------------------------------------------------------
# 4. bn_act_bwd: both reduce and all four apply instantiations
# ---------------------------------------------------------------------------------------------------------------
RED = "bn_act_bwd_reduce_kernel<{}>"
APP = "bn_act_bwd_apply_kernel<{}>"
# (rule, N, H, W, C, path: y | mask | reduced, extras, expected)
BN_BWD = []
for _relu in (True, False):
    for _p in (0.0, 0.3):
        BN_BWD += [
            ("y path: !mask -> reduce<false> + apply<false,true,true>", 4, 8, 8, 160, _relu, _p, "y", "",
             [RED.format(0), APP.format("0,1,1")]),
            ("y path, addend + dskip", 4, 8, 8, 160, _relu, _p, "y", "addend+dskip", [RED.format(0), APP.format("0,1,1")]),
            ("mask -> reduce<true> + apply<true,false,false>", 4, 8, 8, 160, _relu, _p, "mask", "",
             [RED.format(1), APP.format("1,0,0")]),
            ("mask + addend -> apply<true,true,false>", 4, 8, 8, 160, _relu, _p, "mask", "addend",
             [RED.format(1), APP.format("1,1,0")]),
            ("mask + dskip -> apply<true,true,true>", 4, 8, 8, 160, _relu, _p, "mask", "dskip",
             [RED.format(1), APP.format("1,1,1")]),
            ("reduced= (sums given) + addend + dskip: apply only", 4, 8, 8, 160, _relu, _p, "reduced", "addend+dskip",
             [APP.format("1,1,1")]),
        ]
BN_BWD += [
    ("mask + dskip, C = 2056: second chunk of one group", 2, 5, 3, 2056, True, 0.3, "mask", "dskip",
     [RED.format(1), APP.format("1,1,1")]),
    ("y path, C = 4096: two full chunks", 2, 3, 5, 4096, True, 0.3, "y", "addend+dskip",
     [RED.format(0), APP.format("0,1,1")]),
    ("mask + addend, C = 4096", 2, 3, 5, 4096, False, 0.3, "mask", "addend", [RED.format(1), APP.format("1,1,0")]),
    ("mask, WRN 128x32x32x160", 128, 32, 32, 160, True, 0.0, "mask", "", [RED.format(1), APP.format("1,0,0")]),
]


def _bwd_id(r):
    return f"{r[1]}x{r[2]}x{r[3]}x{r[4]}-relu{int(r[5])}-p{r[6]}-{r[7]}-{r[8] or 'plain'}"


@pytest.mark.parametrize("row", BN_BWD, ids=_bwd_id)
def test_bn_act_bwd_route(row):
    from tests.test_conv_routes_gpu import _bn_bwd_ref
    ops, _lib = _ops()
    rule, N, H, W, C, relu, p, path, extras, expected = row
    label = f"bn_act_bwd {_bwd_id(row)}"
    g = _gen(label)
    o = dict(relu=relu, p=p)
    x, _, _, _, gamma, beta, _ = _fwd_inputs(N, H, W, C, o, g)
    mean, invstd = ops.bn_stats(x, EPS)
    seed = 0xB0B + zlib.crc32(label.encode())
    offset = int(ops.step_counter(x.device).item()) if p > 0 else None
    y, mask = ops.bn_act_fwd(x, mean, invstd, gamma, beta, relu=relu, dropout_p=p, seed=seed, want_mask=True)
    _, _, _, _, keep, gate = fwd_reference(x, mean, invstd, gamma, beta, None, o, seed, offset, y)
    _assert_bytes_equal(mask, _pack_bits(gate), f"{label} forward mask", bits_per_byte=8)
    dy = (torch.randn(N, H, W, C, device="cuda", generator=g) + 0.2).bfloat16()
    addend = torch.randn(N, H, W, C, device="cuda", generator=g).bfloat16() if "addend" in extras else None
    rows = N * H * W
    # g = bf16(dy / (1 - p)) where the unit was active and kept, else 0: the kernels' rounding point
    if p > 0:
        inv_keep = float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))
        gd = (dy.float() * inv_keep).bfloat16().double()
    else:
        gd = dy.double()
    gd = torch.where(gate, gd, torch.zeros_like(gd))
    n = reduce_chain(rows, C, 3)
    C_ = C
    xd = x.double().reshape(-1, C_)
    g2 = gd.reshape(-1, C_)
    md, isd = mean.double(), invstd.double()
    dbeta_ref = g2.sum(0)
    dgamma_ref = (g2 * (xd - md) * isd).sum(0)
    reduced = None
    if path == "reduced":
        reduced = (dgamma_ref.float(), dbeta_ref.float())
    dx = poisoned((N, H, W, C), torch.bfloat16)
    dskip = poisoned((N, H, W, C), torch.bfloat16) if "dskip" in extras else None
    dgamma = poisoned((C,), torch.float32) if reduced is None else reduced[0]
    dbeta = poisoned((C,), torch.float32) if reduced is None else reduced[1]
    p_ = ops._p
    nws = _lib.load().b200_bn_workspace_bytes(rows, C)
    ws = ops.bn_accumulators(dy.device, nws)        # allocated (and zeroed) outside the profiled call

    def call():
        if reduced is not None:
            _lib.call("b200_bn_act_bwd_apply", dy.data_ptr(), mask.data_ptr(), x.data_ptr(), dx.data_ptr(), p_(dskip),
                      p_(addend), rows, C, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(),
                      dbeta.data_ptr(), int(relu), float(p), ops._stream())
            return
        _lib.call("b200_bn_act_bwd", dy.data_ptr(), p_(y if path == "y" else None),
                  p_(mask if path == "mask" else None), x.data_ptr(), dx.data_ptr(), p_(dskip), p_(addend), rows, C,
                  mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), int(relu),
                  float(p), seed, ops.step_counter(dy.device).data_ptr() if p > 0 else None, ws.data_ptr(), nws,
                  ops._stream())

    _, launched = kernels_launched(call)
    _assert_kernels(launched, expected, f"{label} ({rule})")
    for name, t in (("dx", dx), ("dskip", dskip)) + ((("dgamma", dgamma), ("dbeta", dbeta)) if reduced is None else ()):
        if t is not None:
            check_poisoned(t, name)
    ws_ = []
    if reduced is None:
        # fp32 sums of g and g * x (g, x bf16: every product exact) over the reduce kernel's chain, fp64 finish
        gm = gamma_n(n)
        mag_s0 = gm * g2.abs().sum(0)
        mag_s1 = gm * (g2 * xd).abs().sum(0)
        ws_.append(assert_elementwise(dbeta, dbeta_ref, mag_s0, U32, acc=1.0, label=f"{label} dbeta"))
        ws_.append(assert_elementwise(dgamma, dgamma_ref, isd * (mag_s1 + md.abs() * mag_s0), U32, acc=1.0,
                                      label=f"{label} dgamma"))
    *_, dx_ref, mag = _bn_bwd_ref(gd, x, mean, invstd, gamma, rows)
    adds, npts = [], 1
    if addend is not None:
        dx_ref = dx_ref + addend.double()
        adds, npts = [addend], 2
    ws_.append(assert_elementwise(dx, dx_ref, mag, npts * BF16_ROUNDING, acc=2.0 ** -14, addends=adds,
                                  label=f"{label} dx"))
    if dskip is not None:
        bad = (dskip.double() != gd).nonzero()
        assert bad.numel() == 0, f"{label}: dskip != g at (n, h, w, c) = {tuple(bad[0].tolist())}"
    _report(label, launched, _worst(*ws_))


# ---------------------------------------------------------------------------------------------------------------
# 5. pooling
# ---------------------------------------------------------------------------------------------------------------
def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1)


# (rule, N, H, W, C, k, stride, pad, expected)
AVG = [
    ("global: pad 0, k == H == W (WRN head 8x8x640: RP = 3)", 128, 8, 8, 640, 8, 1, 0, "avgpool_global_kernel"),
    ("global 7x7x2048 (ImageNet head: one chunk)", 16, 7, 7, 2048, 7, 1, 0, "avgpool_global_kernel"),
    ("global, C = 2056: 257 channel groups", 4, 7, 7, 2056, 7, 1, 0, "avgpool_global_kernel"),
    ("global, C = 4104: 513 channel groups", 2, 5, 5, 4104, 5, 1, 0, "avgpool_global_kernel"),
    ("generic k3 s2 p1 on odd extents", 2, 9, 11, 24, 3, 2, 1, "avgpool_fwd_kernel"),
    ("generic k2 s2 p0", 3, 8, 6, 16, 2, 2, 0, "avgpool_fwd_kernel"),
    ("generic k = H with padding is no global pool", 2, 5, 5, 8, 5, 1, 1, "avgpool_fwd_kernel"),
]


@pytest.mark.parametrize("row", AVG, ids=lambda r: f"{r[1]}x{r[2]}x{r[3]}x{r[4]}-k{r[5]}s{r[6]}p{r[7]}")
def test_avgpool_route(row):
    ops, _lib = _ops()
    rule, N, H, W, C, k, s, pad, exp = row
    label = f"avgpool {N}x{H}x{W}x{C} k{k}s{s}p{pad}"
    g = _gen(label)
    x = (torch.randn(N, H, W, C, device="cuda", generator=g) + 0.5).bfloat16()
    P, Q = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    y = poisoned((N, P, Q, C), torch.bfloat16)
    _, launched = kernels_launched(lambda: _lib.call("b200_avgpool_fwd", x.data_ptr(), y.data_ptr(), N, H, W, C, k, s,
                                                     pad, ops._stream()))
    _assert_kernels(launched, [exp], f"{label} ({rule})")
    check_poisoned(y, "y")
    xd = nchw(x.double())
    ref = nhwc(F.avg_pool2d(xd, k, s, pad, count_include_pad=True))
    mag = nhwc(F.avg_pool2d(xd.abs(), k, s, pad, count_include_pad=True))
    # fp32 sums of at most k^2 terms (global: per-lane partials, then the lanes), times the fp32 1/k^2
    acc = gamma_n(k * k + EW_THREADS // max(1, min(EW_THREADS, C // 8)) + 2)
    w = assert_elementwise(y, ref, mag, BF16_ROUNDING, acc=acc, label=f"{label} y")
    _report(label, launched, w)
    if exp == "avgpool_global_kernel":
        return
    # backward: dx = sum over the windows of bf16(dy / k^2), each term rounded, then the bf16 sum
    label = f"avgpool_bwd {N}x{H}x{W}x{C} k{k}s{s}p{pad}"
    dy = torch.randn(N, P, Q, C, device="cuda", generator=g).bfloat16()
    dx = poisoned((N, H, W, C), torch.bfloat16)
    _, launched = kernels_launched(lambda: _lib.call("b200_avgpool_bwd", dy.data_ptr(), dx.data_ptr(), N, H, W, C, k,
                                                     s, pad, ops._stream()))
    _assert_kernels(launched, ["avgpool_bwd_kernel"], label)
    check_poisoned(dx, "dx")

    def bwd(d):
        xx = torch.zeros(N, C, H, W, dtype=torch.float64, device="cuda", requires_grad=True)
        F.avg_pool2d(xx, k, s, pad, count_include_pad=True).backward(nchw(d))
        return nhwc(xx.grad)

    ref, terms = bwd(dy.double()), bwd(dy.double().abs())
    w = assert_elementwise(dx, ref, terms, BF16_ROUNDING, acc=gamma_n(k * k + 1), addends=[terms],
                           label=f"{label} dx")
    _report(label, launched, w)


# (rule, N, H, W, C, k, stride, pad, kernel suffix)
MAXP = [
    ("ks<3,2>: ImageNet stem 112x112", 2, 112, 112, 64, 3, 2, 1, "_ks_kernel<3,2>"),
    ("ks<3,2>, C = 8, odd extents", 2, 15, 17, 8, 3, 2, 1, "_ks_kernel<3,2>"),
    ("ks<3,2>, C = 2056", 1, 9, 9, 2056, 3, 2, 1, "_ks_kernel<3,2>"),
    ("ks<3,1>", 2, 13, 11, 24, 3, 1, 1, "_ks_kernel<3,1>"),
    ("ks<2,2>", 2, 16, 14, 16, 2, 2, 0, "_ks_kernel<2,2>"),
    ("ks<2,2>, C = 2056", 1, 6, 6, 2056, 2, 2, 0, "_ks_kernel<2,2>"),
    ("generic k5 s2 p2", 2, 13, 13, 16, 5, 2, 2, "_kernel"),
    ("generic k3 s3 p1", 2, 14, 14, 8, 3, 3, 1, "_kernel"),
    ("generic k2 s1", 2, 9, 10, 24, 2, 1, 0, "_kernel"),
    ("generic k2 s1, C = 2056", 1, 7, 7, 2056, 2, 1, 0, "_kernel"),
]


def _maxpool_ref(x, k, s, pad):
    """exact max and the first maximal window position r * k + c in scan order (padding = -inf never wins)."""
    N, H, W, C = x.shape
    xd = F.pad(nchw(x.double()), (pad, pad, pad, pad), value=float("-inf"))
    win = F.unfold(xd, k, stride=s)                   # [N, C * k * k, L]
    P, Q = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    win = win.reshape(N, C, k * k, P, Q)
    m = win.max(2).values
    pos = torch.arange(k * k, device=x.device).reshape(1, 1, k * k, 1, 1)
    first = torch.where(win == m.unsqueeze(2), pos, torch.full_like(pos, 1 << 20)).min(2).values
    return nhwc(m), nhwc(first)


@pytest.mark.parametrize("row", MAXP, ids=lambda r: f"{r[1]}x{r[2]}x{r[3]}x{r[4]}-k{r[5]}s{r[6]}p{r[7]}")
def test_maxpool_route(row):
    ops, _lib = _ops()
    rule, N, H, W, C, k, s, pad, suffix = row
    label = f"maxpool {N}x{H}x{W}x{C} k{k}s{s}p{pad}"
    g = _gen(label)
    # small integers: ties everywhere, so the first-maximum rule decides most windows
    x = torch.randint(-3, 4, (N, H, W, C), device="cuda", generator=g).bfloat16()
    P, Q = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    ref_y, ref_arg = _maxpool_ref(x, k, s, pad)
    args = []
    for fill in (0x00, 0xFF):
        y = poisoned((N, P, Q, C), torch.bfloat16)
        am = poisoned((N, P, Q, C), torch.uint8, byte=fill)
        _, launched = kernels_launched(lambda: _lib.call("b200_maxpool_fwd", x.data_ptr(), y.data_ptr(), am.data_ptr(),
                                                         N, H, W, C, k, s, pad, ops._stream()))
        _assert_kernels(launched, ["maxpool_fwd" + suffix], f"{label} ({rule})")
        check_poisoned(y, "y")
        check_poisoned(am, f"argmax (fill {fill:#04x})")
        assert torch.equal(y.double(), ref_y), f"{label}: max values differ"
        _assert_bytes_equal(am, ref_arg.to(torch.uint8), f"{label} argmax (fill {fill:#04x})")
        args.append(am)
    dy = torch.randn(N, P, Q, C, device="cuda", generator=g).bfloat16()
    dx = poisoned((N, H, W, C), torch.bfloat16)
    _, launched = kernels_launched(lambda: _lib.call("b200_maxpool_bwd", dy.data_ptr(), args[0].data_ptr(),
                                                     dx.data_ptr(), N, H, W, C, k, s, pad, ops._stream()))
    _assert_kernels(launched, ["maxpool_bwd" + suffix], f"{label} bwd ({rule})")
    check_poisoned(dx, "dx")
    # dx[n, h, w, c] = sum of dy over the windows whose first maximum sits at (h, w)
    t = ref_arg.long()
    n_i, p_i, q_i, c_i = torch.meshgrid(*(torch.arange(v, device="cuda") for v in (N, P, Q, C)), indexing="ij")
    h_i = p_i * s + t // k - pad
    w_i = q_i * s + t % k - pad
    ref = torch.zeros(N, H, W, C, dtype=torch.float64, device="cuda")
    mag = torch.zeros_like(ref)
    ref.index_put_((n_i, h_i, w_i, c_i), dy.double(), accumulate=True)
    mag.index_put_((n_i, h_i, w_i, c_i), dy.double().abs(), accumulate=True)
    w = assert_elementwise(dx, ref, mag, BF16_ROUNDING, acc=gamma_n(k * k), label=f"{label} dx")
    _report(label, launched, w)


# ---------------------------------------------------------------------------------------------------------------
# 6. head: linear forward / backward, cross entropy + top-k
# ---------------------------------------------------------------------------------------------------------------
LINEAR = [(128, 640, 10), (256, 2048, 1000), (7, 33, 3), (1, 64, 100), (1024, 40, 1)]


@pytest.mark.parametrize("shape", LINEAR, ids=lambda s: "x".join(map(str, s)))
def test_linear_route(shape):
    ops, _lib = _ops()
    B, I, O = shape
    label = f"linear {B}x{I}x{O}"
    g = _gen(label)
    x = torch.randn(B, I, device="cuda", generator=g).bfloat16()
    w = torch.randn(O, I, device="cuda", generator=g) / I ** 0.5
    b = torch.randn(O, device="cuda", generator=g)
    y = poisoned((B, O), torch.bfloat16)
    _, launched = kernels_launched(lambda: _lib.call("b200_linear_fwd", x.data_ptr(), w.data_ptr(), b.data_ptr(),
                                                     y.data_ptr(), B, I, O, ops._stream()))
    _assert_kernels(launched, ["linear_fwd_kernel"], label)
    check_poisoned(y, "logits")
    wb, bb = w.bfloat16().double(), b.bfloat16().double()       # the kernel multiplies by bf16(w), adds bf16(b)
    ref = x.double() @ wb.t() + bb
    mag = x.double().abs() @ wb.abs().t() + bb.abs()
    w1 = assert_elementwise(y, ref, mag, BF16_ROUNDING, acc=gamma_n(-(-I // 32) + 6), label=f"{label} logits")
    _report(label, launched, w1)

    dy = (torch.randn(B, O, device="cuda", generator=g) * 0.1).bfloat16()
    dx = poisoned((B, I), torch.bfloat16)
    dw, db = poisoned((O, I), torch.float32), poisoned((O,), torch.float32)
    _, launched = kernels_launched(lambda: _lib.call("b200_linear_bwd", dy.data_ptr(), x.data_ptr(), w.data_ptr(),
                                                     dx.data_ptr(), dw.data_ptr(), db.data_ptr(), B, I, O,
                                                     ops._stream()))
    _assert_kernels(launched, ["linear_bwd_dw_kernel", "linear_bwd_dx_kernel"], f"{label} bwd")
    for name, t in (("dx", dx), ("dw", dw), ("db", db)):
        check_poisoned(t, name)
    dyd, xd = dy.double(), x.double()
    w2 = assert_elementwise(dx, dyd @ wb, dyd.abs() @ wb.abs(), BF16_ROUNDING, acc=gamma_n(O), label=f"{label} dx")
    w3 = assert_elementwise(dw, dyd.t() @ xd, dyd.abs().t() @ xd.abs(), 0.0, acc=gamma_n(B), label=f"{label} dw")
    w4 = assert_elementwise(db, dyd.sum(0), dyd.abs().sum(0), 0.0, acc=gamma_n(B), label=f"{label} db")
    _report(f"{label} bwd", launched, _worst(w2, w3, w4))


CE = [(1, 1), (3, 4), (33, 10), (1000, 100), (256, 1000)]
# __expf: 2 + floor(|1.173 x|) ulp; __logf: 2^-21.41 absolute on [0.5, 2], else 3 ulp (CUDA C Programming Guide,
# intrinsic functions). expf / logf of the fp32 path: 2 ulp / 1 ulp.
ULP = 2.0 ** -23


def _ce_reference(z, labels, fast):
    """fp64 loss terms, top-1 / top-5 error counts (label rank: larger logits, ties towards the lower index), softmax,
    and per-sample bounds of the kernel's lse."""
    zd = z.double()
    B, O = zd.shape
    zl = zd.gather(1, labels[:, None])
    idx = torch.arange(O, device=z.device)[None, :]
    rank = ((zd > zl) | ((zd == zl) & (idx < labels[:, None]))).sum(1)
    mx = zd.max(1, keepdim=True).values
    se = torch.exp(zd - mx).sum(1, keepdim=True)
    lse = mx + se.log()
    exp_ulps = (2 + torch.floor(1.173 * (zd - mx).abs())) if fast else torch.full_like(zd, 2.0)
    rel_se = (torch.exp(zd - mx) * exp_ulps * ULP).sum(1, keepdim=True) / se + gamma_n(-(-O // 32) + 5)
    log_err = (2.0 ** -21.41 + 3 * ULP * se.log().abs()) if fast else (ULP * se.log().abs())
    dlse = rel_se * 1.01 + log_err + U32 * (mx.abs() + lse.abs())
    return (lse - zl).squeeze(1), rank, torch.exp(zd - lse), lse, dlse.squeeze(1)


@pytest.mark.parametrize("shape", CE, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", ["bf16", "f32"])
def test_ce_topk_route(shape, dtype):
    ops, _lib = _ops()
    B, O = shape
    label = f"ce_topk {dtype} {B}x{O}"
    g = _gen(label)
    # integer logits in a narrow range: ties at the label decide the ranks
    z = torch.randint(-4, 5, (B, O), device="cuda", generator=g).float()
    labels = torch.randint(0, O, (B,), device="cuda", generator=g)
    fast = dtype == "bf16"
    if fast:
        z = z.bfloat16()
    out = poisoned((3,), torch.float32)
    dl = poisoned((B, O), torch.bfloat16) if fast else None
    gs = torch.tensor([1024.0], device="cuda") if B % 2 else None

    def call():
        if fast:
            _lib.call("b200_ce_topk", z.data_ptr(), labels.data_ptr(), out.data_ptr(), dl.data_ptr(), ops._p(gs), B, O,
                      ops._stream())
        else:
            _lib.call("b200_ce_topk_f32", z.data_ptr(), labels.data_ptr(), out.data_ptr(), B, O, ops._stream())

    _, launched = kernels_launched(call)
    _assert_kernels(launched, ["ce_topk_kernel" if fast else "ce_topk_f32_kernel"], label)
    check_poisoned(out, "out")
    loss_b, rank, prob, lse, dlse = _ce_reference(z, labels, fast)
    for j, (name, cnt) in enumerate((("top-1", int((rank >= 1).sum())), ("top-5", int((rank >= 5).sum()))), 1):
        want = np.float32(cnt) / np.float32(B)
        got = out[j].item()
        assert got == want and round(got * B) == cnt, f"{label}: {name} error {got!r} * B != {cnt} (want {want!r})"
    # the mean loss: per-sample lse error, then the fixed-order fp32 sums (per warp, then over 32 warps) and / B
    bound_loss = dlse.sum() / B + gamma_n(-(-B // 32) + 33) * loss_b.abs().sum() / B
    w = assert_elementwise(out[:1], loss_b.mean().reshape(1), bound_loss.reshape(1), U32, acc=1.0,
                           label=f"{label} loss")
    if fast:
        check_poisoned(dl, "dlogits")
        sc = float(np.float32(1024.0 if gs is not None else 1.0) / np.float32(B))
        onehot = F.one_hot(labels, O).double()
        ref = (prob - onehot) * sc
        exp_ulps = 2 + torch.floor(1.173 * (z.double() - lse).abs())
        mag = sc * (prob * (exp_ulps * ULP + dlse[:, None] * 1.01 + U32 * (z.double() - lse).abs())
                    + 2 * U32 * (prob + onehot))
        w = _worst(w, assert_elementwise(dl, ref, mag, BF16_ROUNDING, acc=1.0, label=f"{label} dlogits"))
    _report(label, launched, w)


# ---------------------------------------------------------------------------------------------------------------
# 7. layout and subsample
# ---------------------------------------------------------------------------------------------------------------
WPREP = [(64, 3, 3, 64), (33, 3, 3, 17), (10, 1, 1, 640), (7, 3, 3, 3), (100, 1, 1, 130), (96, 3, 3, 3),
         (160, 3, 3, 160), (1, 1, 1, 1)]


def test_weight_prep_routes():
    ops, _lib = _ops()
    g = _gen("weight_prep")
    ws = [torch.randn(*s, device="cuda", generator=g) for s in WPREP]
    for w in ws:
        K, R, S, C = w.shape
        label = f"weight_prep {K}x{R}x{S}x{C}"
        wk, wt = poisoned((K, R, S, C), torch.bfloat16), poisoned((C, R, S, K), torch.bfloat16)
        _, launched = kernels_launched(lambda: _lib.call("b200_weight_prep", w.data_ptr(), wk.data_ptr(), wt.data_ptr(),
                                                         K, R * S, C, ops._stream()))
        _assert_kernels(launched, ["weight_cast_kernel", "weight_transpose_kernel"], label)
        check_poisoned(wk, "wk")
        check_poisoned(wt, "wt")
        assert torch.equal(wk.view(torch.int16), w.bfloat16().view(torch.int16)), f"{label}: KRSC copy"
        assert torch.equal(wt.view(torch.int16), w.permute(3, 1, 2, 0).contiguous().bfloat16().view(torch.int16)), \
            f"{label}: CRSK copy"
    # weight_prep_multi: one launch over a table mixing the 64x64 even path and the 32x32 odd K / C scalar path
    outs = [(poisoned(tuple(w.shape), torch.bfloat16), poisoned((w.shape[3], w.shape[1], w.shape[2], w.shape[0]),
                                                                torch.bfloat16)) for w in ws]
    table = ops.weight_prep_table([(w, wk, wt) for w, (wk, wt) in zip(ws, outs)])
    _, launched = kernels_launched(lambda: ops.weight_prep_multi(table, len(ws)))
    _assert_kernels(launched, ["weight_prep_multi_kernel"], "weight_prep_multi")
    for w, (wk, wt) in zip(ws, outs):
        label = f"weight_prep_multi {'x'.join(map(str, w.shape))}"
        check_poisoned(wk, f"{label} wk")
        check_poisoned(wt, f"{label} wt")
        assert torch.equal(wk.view(torch.int16), w.bfloat16().view(torch.int16)), f"{label}: KRSC copy"
        assert torch.equal(wt.view(torch.int16), w.permute(3, 1, 2, 0).contiguous().bfloat16().view(torch.int16)), \
            f"{label}: CRSK copy"
    print(f"[route] weight_prep / weight_prep_multi: {len(ws)} filters bit-exact")


@pytest.mark.parametrize("C", [1, 3, 16])
def test_nchw_to_nhwc_routes(C):
    ops, _lib = _ops()
    g = _gen(f"nchw {C}")
    N, H, W = 3, 7, 5
    x = torch.randn(N, C, H, W, device="cuda", generator=g) * 3
    y = poisoned((N, H, W, C), torch.bfloat16)
    _, launched = kernels_launched(lambda: _lib.call("b200_nchw_f32_to_nhwc_bf16", x.data_ptr(), y.data_ptr(), N, C,
                                                     H, W, ops._stream()))
    _assert_kernels(launched, ["nchw_f32_to_nhwc_bf16_kernel"], f"nchw_f32_to_nhwc_bf16 C{C}")
    check_poisoned(y, "y")
    assert torch.equal(y.view(torch.int16), x.permute(0, 2, 3, 1).contiguous().bfloat16().view(torch.int16))
    yf = poisoned((N, H, W, C), torch.float32)
    _, launched = kernels_launched(lambda: _lib.call("b200_nchw_to_nhwc_f32", x.data_ptr(), yf.data_ptr(), N, C, H, W,
                                                     ops._stream()))
    _assert_kernels(launched, ["nchw_to_nhwc_f32_kernel"], f"nchw_to_nhwc_f32 C{C}")
    check_poisoned(yf, "y f32")
    assert torch.equal(yf, x.permute(0, 2, 3, 1).contiguous())


@pytest.mark.parametrize("dtype", ["bf16", "f32"])
def test_subsample2_route(dtype):
    ops, _lib = _ops()
    g = _gen(f"subsample2 {dtype}")
    N, H, W, C = 2, 7, 5, 24
    x = torch.randn(N, 2 * H, 2 * W, C, device="cuda", generator=g)
    if dtype == "bf16":
        x = x.bfloat16()
    y = poisoned((N, H, W, C), x.dtype)
    name = "b200_subsample2" if dtype == "bf16" else "b200_subsample2_f32"
    _, launched = kernels_launched(lambda: _lib.call(name, x.data_ptr(), y.data_ptr(), N, H, W, C, ops._stream()))
    _assert_kernels(launched, ["subsample2_kernel" if dtype == "bf16" else "subsample2_f32_kernel"], name)
    check_poisoned(y, "y")
    assert torch.equal(y, x[:, ::2, ::2, :])


@pytest.mark.parametrize("geo", [(2, 5, 3, 64, 24, 40), (1, 4, 4, 16, 16, 16), (2, 3, 7, 640, 320, 648)],
                         ids=lambda t: "x".join(map(str, t)))
def test_upsample_add_route(geo):
    """dx[n, 2h, 2w, :Cg] = bf16(dx + g[n, h, w, :Cg]) in place, g with channel pitch ldg; everything else of dx
    stays bit-identical."""
    ops, _lib = _ops()
    N, H, W, C, Cg, ldg = geo
    g_ = _gen(f"upsample {geo}")
    dx = poisoned((N, 2 * H, 2 * W, C), torch.bfloat16)
    dx.copy_(torch.randn(N, 2 * H, 2 * W, C, device="cuda", generator=g_).bfloat16())
    before = dx.clone()
    gr = torch.randn(N, H, W, ldg, device="cuda", generator=g_).bfloat16()
    _, launched = kernels_launched(lambda: _lib.call("b200_upsample_add", dx.data_ptr(), gr.data_ptr(), N, H, W, C, Cg,
                                                     ldg, ops._stream()))
    _assert_kernels(launched, ["upsample_add_kernel"], f"upsample_add {geo}")
    check_poisoned(dx, "dx")
    ref = before.clone()
    ref[:, ::2, ::2, :Cg] = (before[:, ::2, ::2, :Cg].float() + gr[..., :Cg].float()).bfloat16()
    bad = (dx.view(torch.int16) != ref.view(torch.int16)).nonzero()
    assert bad.numel() == 0, f"upsample_add {geo}: first wrong element at (n, h, w, c) = {tuple(bad[0].tolist())}"


# ---------------------------------------------------------------------------------------------------------------
# 8. the fp32 evaluation path (f32_path.cuh): no intermediate rounding
# ---------------------------------------------------------------------------------------------------------------
F32_BN = [
    ("affine + ReLU", 2, 5, 3, 24, dict(relu=True)),
    ("eval mode (variance), no ReLU", 2, 5, 3, 24, dict(relu=False, eval=True)),
    ("skip SAME", 2, 4, 4, 160, dict(relu=True, skip="same")),
    ("skip SUBSAMPLE_PAD", 2, 4, 4, 160, dict(relu=True, skip="pad")),
    ("no affine", 1, 3, 3, 8, dict(relu=True, affine=False)),
]


@pytest.mark.parametrize("row", F32_BN, ids=lambda r: r[0].replace(" ", "_"))
def test_bn_act_fwd_f32_route(row):
    ops, _lib = _ops()
    rule, N, H, W, C, o = row
    label = f"bn_act_fwd_f32 {rule}"
    g = _gen(label)
    x, mean, var, invstd, gamma, beta, skip = _fwd_inputs(N, H, W, C, o, g)
    x = x.float() + torch.randn(N, H, W, C, device="cuda", generator=g) * 1e-3   # fp32 values, not bf16 ones
    skip = None if skip is None else skip.float()
    stat = var if o.get("eval") else invstd
    affine = o.get("affine", True)
    y = poisoned((N, H, W, C), torch.float32)
    p_ = ops._p
    skip_mode = {None: 0, "same": _lib.SKIP_SAME, "pad": _lib.SKIP_SUBSAMPLE_PAD}[o.get("skip")]

    def call():
        _lib.call("b200_bn_act_fwd_f32", x.data_ptr(), y.data_ptr(), N, H, W, C, p_(mean if affine else None),
                  p_(stat if affine else None), int(bool(o.get("eval"))), EPS, p_(gamma if affine else None),
                  p_(beta if affine else None), p_(skip), skip_mode, 0 if skip is None else skip.shape[-1],
                  int(o["relu"]), ops._stream())

    _, launched = kernels_launched(call)
    _assert_kernels(launched, ["bn_act_fwd_f32_kernel"], label)
    check_poisoned(y, "y")
    ref, scale, mag, _, _, _ = fwd_reference(x, mean, stat, gamma, beta, skip, o, 0, None, y)
    # fp32: the fma and the skip add round the result (2 ulps of |bn| + |skip|); sc = gamma * invstd (rsqrtf of a
    # variance: 2 ulps more) and sh = beta - mean * sc err by a few ulps of their operands
    w = assert_elementwise(y, ref, mag, 2 * U32, acc=8 * U32, scale64=scale, label=label)
    _report(label, launched, w)


@pytest.mark.parametrize("pool", [("avg", 8, 8, 1, 0), ("avg", 3, 3, 2, 1), ("max", 3, 3, 2, 1), ("max", 2, 2, 2, 0)],
                         ids=lambda t: f"{t[0]}-k{t[2]}s{t[3]}p{t[4]}")
def test_pool_fwd_f32_route(pool):
    ops, _lib = _ops()
    kind, H, k, s, pad = pool
    N, W, C = 2, H + 1 if kind == "max" else H, 24
    label = f"pool_fwd_f32 {kind} k{k}s{s}p{pad}"
    g = _gen(label)
    x = torch.randn(N, H, W, C, device="cuda", generator=g)
    if kind == "max":
        x = torch.randint(-3, 4, (N, H, W, C), device="cuda", generator=g).float()
    P, Q = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    y = poisoned((N, P, Q, C), torch.float32)
    _, launched = kernels_launched(lambda: _lib.call("b200_pool_fwd_f32", x.data_ptr(), y.data_ptr(), N, H, W, C, k, s,
                                                     pad, int(kind == "max"), ops._stream()))
    _assert_kernels(launched, [f"pool_fwd_f32_kernel<{int(kind == 'max')}>"], label)
    check_poisoned(y, "y")
    xd = nchw(x.double())
    if kind == "max":
        assert torch.equal(y.double(), nhwc(F.max_pool2d(xd, k, s, pad))), f"{label}: not bit-exact"
        print(f"[route] {label}: {launched[0]}; bit-exact")
        return
    ref = nhwc(F.avg_pool2d(xd, k, s, pad, count_include_pad=True))
    mag = nhwc(F.avg_pool2d(xd.abs(), k, s, pad, count_include_pad=True))
    w = assert_elementwise(y, ref, mag, 0.0, acc=gamma_n(k * k + 2), label=label)
    _report(label, launched, w)


@pytest.mark.parametrize("shape", [(128, 640, 10), (7, 33, 3), (2, 2048, 1000)], ids=lambda s: "x".join(map(str, s)))
def test_linear_fwd_f32_route(shape):
    ops, _lib = _ops()
    B, I, O = shape
    label = f"linear_fwd_f32 {B}x{I}x{O}"
    g = _gen(label)
    x = torch.randn(B, I, device="cuda", generator=g)
    w = torch.randn(O, I, device="cuda", generator=g) / I ** 0.5
    b = torch.randn(O, device="cuda", generator=g)
    y = poisoned((B, O), torch.float32)
    _, launched = kernels_launched(lambda: _lib.call("b200_linear_fwd_f32", x.data_ptr(), w.data_ptr(), b.data_ptr(),
                                                     y.data_ptr(), B, I, O, ops._stream()))
    _assert_kernels(launched, ["linear_fwd_f32_kernel"], label)
    check_poisoned(y, "logits")
    ref = x.double() @ w.double().t() + b.double()
    mag = x.double().abs() @ w.double().abs().t() + b.double().abs()
    wr = assert_elementwise(y, ref, mag, 0.0, acc=gamma_n(-(-I // 32) + 6), label=label)
    _report(label, launched, wr)


# ---------------------------------------------------------------------------------------------------------------
# coverage: every non-conv kernel instantiation api.cu launches has a row (tests/test_ew_routes_cpu.py checks this
# list against api.cu without a GPU)
# ---------------------------------------------------------------------------------------------------------------
EW_REACHABLE = {
    "bn_stats_kernel": "bn_sums_launch (b200_bn_stats; conv epilogues without fused sums)",
    "bn_stats_finalize_kernel": "b200_bn_stats_finalize",
    "bn_running_update_kernel": "b200_bn_running_update",
    "bn_act_fwd_kernel<2,3,1,2>": "b200_bn_act_fwd: skip_mode != 0, drop",
    "bn_act_fwd_kernel<2,3,1,0>": "b200_bn_act_fwd: skip_mode != 0, !drop",
    "bn_act_fwd_kernel<4,4,0,0>": "b200_bn_act_fwd: !skip, !drop",
    "bn_act_fwd_kernel<4,3,0,2>": "b200_bn_act_fwd: !skip, keepbits (drop, !relu, mask_out)",
    "bn_act_fwd_kernel<2,4,0,1>": "b200_bn_act_fwd: !skip, drop, relu or no mask",
    "bn_act_bwd_reduce_kernel<1>": "bn_act_bwd_impl: affine, reduce, gate_x (mask)",
    "bn_act_bwd_reduce_kernel<0>": "bn_act_bwd_impl: affine, reduce, !gate_x (y / RNG)",
    "bn_act_bwd_apply_kernel<0,1,1>": "bn_act_bwd_impl: !gate_x",
    "bn_act_bwd_apply_kernel<1,1,1>": "bn_act_bwd_impl: gate_x, dskip",
    "bn_act_bwd_apply_kernel<1,1,0>": "bn_act_bwd_impl: gate_x, addend",
    "bn_act_bwd_apply_kernel<1,0,0>": "bn_act_bwd_impl: gate_x",
    "tick_kernel": "b200_tick",
    "subsample2_kernel": "b200_subsample2",
    "upsample_add_kernel": "b200_upsample_add",
    "avgpool_global_kernel": "b200_avgpool_fwd: pad == 0, k == H == W",
    "avgpool_fwd_kernel": "b200_avgpool_fwd: otherwise",
    "avgpool_bwd_kernel": "b200_avgpool_bwd",
    "maxpool_fwd_ks_kernel<3,2>": "b200_maxpool_fwd: k 3, stride 2",
    "maxpool_fwd_ks_kernel<3,1>": "b200_maxpool_fwd: k 3, stride 1",
    "maxpool_fwd_ks_kernel<2,2>": "b200_maxpool_fwd: k 2, stride 2",
    "maxpool_fwd_kernel": "b200_maxpool_fwd: other windows",
    "maxpool_bwd_ks_kernel<3,2>": "b200_maxpool_bwd: k 3, stride 2",
    "maxpool_bwd_ks_kernel<3,1>": "b200_maxpool_bwd: k 3, stride 1",
    "maxpool_bwd_ks_kernel<2,2>": "b200_maxpool_bwd: k 2, stride 2",
    "maxpool_bwd_kernel": "b200_maxpool_bwd: other windows",
    "linear_fwd_kernel": "b200_linear_fwd",
    "linear_bwd_dx_kernel": "b200_linear_bwd: dx",
    "linear_bwd_dw_kernel": "b200_linear_bwd: dw",
    "ce_topk_kernel": "b200_ce_topk",
    "weight_cast_kernel": "b200_weight_prep: KRSC copy",
    "weight_transpose_kernel": "b200_weight_prep: CRSK copy",
    "weight_prep_multi_kernel": "b200_weight_prep_multi",
    "nchw_f32_to_nhwc_bf16_kernel": "b200_nchw_f32_to_nhwc_bf16",
    "nchw_to_nhwc_f32_kernel": "b200_nchw_to_nhwc_f32",
    "bn_act_fwd_f32_kernel": "b200_bn_act_fwd_f32",
    "subsample2_f32_kernel": "b200_subsample2_f32",
    "pool_fwd_f32_kernel<0>": "b200_pool_fwd_f32: average",
    "pool_fwd_f32_kernel<1>": "b200_pool_fwd_f32: max",
    "linear_fwd_f32_kernel": "b200_linear_fwd_f32",
    "ce_topk_f32_kernel": "b200_ce_topk_f32",
}

# kernels of the rows that are not in the tables above (weight prep, layout, tick)
_OTHER_ROWS = {"weight_cast_kernel", "weight_transpose_kernel", "weight_prep_multi_kernel",
               "nchw_f32_to_nhwc_bf16_kernel", "nchw_to_nhwc_f32_kernel", "subsample2_kernel", "subsample2_f32_kernel",
               "upsample_add_kernel", "bn_act_fwd_f32_kernel", "pool_fwd_f32_kernel<0>", "pool_fwd_f32_kernel<1>",
               "linear_fwd_f32_kernel", "ce_topk_kernel", "ce_topk_f32_kernel", "linear_fwd_kernel",
               "linear_bwd_dx_kernel", "linear_bwd_dw_kernel", "bn_stats_kernel", "bn_stats_finalize_kernel",
               "bn_running_update_kernel", "avgpool_bwd_kernel", "tick_kernel"}


def test_tick_advances_the_dropout_seed():
    """tick_kernel adds exactly one to the step counter; the next dropout launch draws with the new offset."""
    ops, _lib = _ops()
    dev = torch.device("cuda", torch.cuda.current_device())
    before = int(ops.step_counter(dev).item())
    _, launched = kernels_launched(lambda: ops.tick(dev))
    _assert_kernels(launched, ["tick_kernel"], "tick")
    assert int(ops.step_counter(dev).item()) == before + 1


def test_route_tables_cover_every_reachable_kernel():
    covered = set(_OTHER_ROWS)
    covered.update(FWD.format(r[6]) for r in BN_FWD)
    for r in BN_BWD:
        covered.update(r[9])
    covered.update(r[8] for r in AVG)
    for r in MAXP:
        covered.update({"maxpool_fwd" + r[8], "maxpool_bwd" + r[8]})
    missing = sorted(set(EW_REACHABLE) - covered)
    assert not missing, f"kernel instantiations without a row: {missing}"
