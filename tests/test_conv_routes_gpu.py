"""
Convolution kernels by dispatch route: every route that api.cu can choose with the default environment, each row
asserting which kernels ran, that no byte outside the output was written and no output element left unwritten
(poisoned outputs with guards), and every output element against an fp64 reference (tests/kernel_check.py).

Routes (api.cu): run_conv_tc picks the halo kernel conv_tc2h_kernel<KC, MT, STATS, TAIL32> for 3x3 / stride 1 /
pad 1 maps with Q % 8 == 0, P % 16 == 0, an even number of 8x16 tiles, BN % 32 == 0 and Cin % 32 == 0; else the
SM-pair kernel conv_tc2_kernel<KC, STATS, 0> when plan_tiles gives an even tile count and BN % 32 == 0; else the
single-CTA kernel conv_tc_kernel<KC, CS> (CS = 2 halved while the tiles or BN / CS do not split). KC = pick_kc(Cin):
64 | 32 | 16; BN = pick_bn(Cout, 16, 256), lowered to <= 160 with a residual. conv2d_dgrad_impl runs stride-2
dgrad as one phased SM-pair launch, else per output phase plus parity_merge_add_kernel. run_wgrad_tc2h takes 3x3
stride-1 wgrad with C, K % 32 == 0, Q % 8 == 0 and P % 16 == 0 or 16 % P == 0 (stacked images); else
wgrad_tc_kernel<SL, 1, MT, 0> (SL 32 when C, K % 32 == 0, else 16; MT 2 when C <= 320 and two M tiles exist).
"""
import re
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests.kernel_check import BF16_ROUNDING, assert_elementwise, check_poisoned, kernels_launched, poisoned

pytestmark = pytest.mark.gpu

# Accumulation error allowed per unit of |operands| (the fp64 conv of |x|, |w|): fp32 accumulation in tensor
# memory, in any order. bf16 outputs hide it under their rounding (worst accumulation-term ratio 0.0034 on a B200
# at its 1000 W limit); the fp32 weight gradients show it: worst 0.021 of 2^-14, with the batch-128 reductions over
# 131072 pixels split 37 ways, hence 2^-16 for them (about 12x headroom).
ACC = 2.0 ** -14
WGRAD_ACC = 2.0 ** -16
# Batch statistics, bias gradients and the fused BN-backward sums: fp32 partial sums per CTA, then fp64 atomics;
# bounded against the sum of |terms| (worst measured 0.019 of 2^-17, same B200: 2^-19 keeps 13x headroom).
SUM_ACC = 2.0 ** -19
EPS = 1e-5


def _ops():
    from pytorch_ddp_resnet_b200 import _lib, ops
    return ops, _lib


def nchw(t):
    return t.permute(0, 3, 1, 2)


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def _act(shape, g, mean=0.5):
    """bf16 activations drawn from N(mean, 1): a padding fault (a neighbour read instead of a zero) is large."""
    return (torch.randn(*shape, device="cuda", generator=g) + mean).bfloat16()


def _filt(K, R, C, g):
    return (torch.randn(K, R, R, C, device="cuda", generator=g) / (R * R * C) ** 0.5).bfloat16()


# ---------------------------------------------------------------------------------------------------------------
# the route table
# ---------------------------------------------------------------------------------------------------------------
# Expected kernels: '+'-separated names (regexes) of normalised kernel names. Every one must run and nothing else
# may. '{S}' is the STATS template argument (1 for the statistics epilogues); a name prefixed 'det:' runs exactly
# in the deterministic mode (the ordered reduction of the pixel-range splits); '?' marks a helper that may run.
EPILOGUES = ["plain", "bias", "res", "bias+res", "relu", "bias+relu", "stats", "stats+res"]
BIG = ["plain", "res", "stats+res"]

# fprop: (rule, N, H, W, C, K, R, stride, pad, expected, epilogues)
# expected kernels of a statistics epilogue on a kernel without the fused sums: + bn_stats_kernel
FPROP = [
    ("halo KC 32: Cin % 64 == 32, Cin < 64", 2, 16, 16, 32, 320, 3, 1, 1, "conv_tc2h_kernel<32,1,{S},0>", EPILOGUES),
    ("halo KC 64; BN 256 -> 128 with a residual", 2, 16, 16, 64, 512, 3, 1, 1, "conv_tc2h_kernel<64,1,{S},0>",
     EPILOGUES),
    ("halo TAIL32: Cin = 64n + 32 > 64", 2, 16, 16, 160, 320, 3, 1, 1, "conv_tc2h_kernel<64,1,{S},1>", EPILOGUES),
    ("halo, N = 1", 1, 32, 32, 64, 64, 3, 1, 1, "conv_tc2h_kernel<64,1,{S},0>", ["plain", "bias+res", "stats+res"]),
    ("halo WRN 160@32x32 batch 128: persistent loop", 128, 32, 32, 160, 160, 3, 1, 1, "conv_tc2h_kernel<64,1,{S},1>",
     BIG),
    ("halo WRN 320@16x16 batch 128", 128, 16, 16, 320, 320, 3, 1, 1, "conv_tc2h_kernel<64,1,{S},0>", BIG),
    ("pair KC 16 (Cin % 32 != 0), stride 2 through strided TMA windows", 2, 32, 32, 48, 320, 3, 2, 1,
     "conv_tc2_kernel<16,{S},0>", EPILOGUES),
    ("pair KC 32, P = Q = 13: bh = 9 overhangs the map", 2, 13, 13, 32, 320, 3, 1, 1, "conv_tc2_kernel<32,{S},0>",
     EPILOGUES),
    ("pair KC 64, stride 2 to a 13x13 output (overhanging h tile)", 2, 26, 26, 64, 320, 3, 2, 1,
     "conv_tc2_kernel<64,{S},0>", EPILOGUES),
    ("pair KC 64, Q = 136: a partial 8-pixel tile in w; P = 8 is no halo map", 1, 8, 136, 64, 320, 3, 1, 1,
     "conv_tc2_kernel<64,{S},0>", EPILOGUES),
    ("pair WRN 640@8x8 batch 128: 8x8 maps are no halo maps", 128, 8, 8, 640, 640, 3, 1, 1,
     "conv_tc2_kernel<64,{S},0>", BIG),
    ("pair ImageNet 56x56x64 batch 64: P % 16 != 0", 64, 56, 56, 64, 64, 3, 1, 1, "conv_tc2_kernel<64,{S},0>", BIG),
    ("single CTA CS 1: P = Q = 23, 5 tiles (odd)", 1, 23, 23, 64, 320, 3, 1, 1, "conv_tc_kernel<64,1>", EPILOGUES),
    ("single CTA CS 2: BN = 112, BN % 32 != 0", 2, 16, 16, 64, 336, 3, 1, 1, "conv_tc_kernel<64,2>", EPILOGUES),
    ("single CTA KC 32 CS 2: BN = 48", 2, 16, 16, 32, 48, 3, 1, 1, "conv_tc_kernel<32,2>", ["plain", "res", "stats"]),
    ("single CTA KC 32 CS 1: odd tile count", 1, 23, 23, 32, 80, 3, 1, 1, "conv_tc_kernel<32,1>",
     ["plain", "bias+res", "stats"]),
    ("single CTA KC 16 CS 2", 2, 16, 16, 48, 80, 3, 1, 1, "conv_tc_kernel<16,2>", ["plain", "bias+res", "stats"]),
    ("single CTA KC 16 CS 1: odd N = 9 of 4x4 maps, 3 images stacked per tile", 9, 4, 4, 48, 336, 3, 1, 1,
     "conv_tc_kernel<16,1>", ["plain", "bias+res", "relu", "stats"]),
    ("im2col stem 3x3, C = 3: K = 16 is no pair tile", 8, 32, 32, 3, 16, 3, 1, 1,
     "im2col_kernel+repitch_rows_kernel<bf16>+conv_tc_kernel<32,2>", ["plain", "bias", "bias+relu", "stats"]),
    ("im2col stem 7x7 / 2, C = 3", 2, 64, 64, 3, 64, 7, 2, 3,
     "im2col_kernel+repitch_rows_kernel<bf16>+conv_tc2_kernel<32,{S},0>", ["plain", "bias", "bias+relu", "stats"]),
    ("direct: C, K not multiples of 16", 2, 8, 8, 24, 40, 3, 1, 1, "conv_fprop_direct_kernel", EPILOGUES),
]
FUSED_STATS = ("conv_tc2h_kernel", "conv_tc2_kernel")

# dgrad: (rule, N, H, W, C, K, R, stride, pad, expected) as the forward conv; the kernel's Cin is K, its Cout is C
DGRAD = [
    ("halo KC 32", 2, 16, 16, 320, 32, 3, 1, 1, "conv_tc2h_kernel<32,1,0,0>"),
    ("halo KC 64; BN 256 -> 128 with an addend", 2, 16, 16, 512, 64, 3, 1, 1, "conv_tc2h_kernel<64,1,0,0>"),
    ("halo TAIL32 (K = 160)", 2, 16, 16, 320, 160, 3, 1, 1, "conv_tc2h_kernel<64,1,0,1>"),
    ("halo WRN 160@32x32 batch 128", 128, 32, 32, 160, 160, 3, 1, 1, "conv_tc2h_kernel<64,1,0,1>"),
    ("halo WRN 320@16x16 batch 128", 128, 16, 16, 320, 320, 3, 1, 1, "conv_tc2h_kernel<64,1,0,0>"),
    ("pair stride 1 on 8x8 maps, KC 64", 4, 8, 8, 320, 64, 3, 1, 1, "conv_tc2_kernel<64,0,0>"),
    ("pair P = Q = 13 overhanging tiles, KC 32", 2, 13, 13, 320, 32, 3, 1, 1, "conv_tc2_kernel<32,0,0>"),
    ("pair KC 16", 4, 8, 8, 320, 48, 3, 1, 1, "conv_tc2_kernel<16,0,0>"),
    ("single CTA: BN = 112, 5 tiles", 1, 23, 23, 336, 64, 3, 1, 1, "conv_tc_kernel<64,1>"),
    ("stride 2, phased single launch (WRN 160 <- 320, batch 128)", 128, 32, 32, 160, 320, 3, 2, 1,
     "conv_tc2_kernel<64,0,0>"),
    ("stride 2, phased single launch, 13x13 phases", 2, 26, 26, 64, 320, 3, 2, 1, "conv_tc2_kernel<64,0,0>"),
    ("stride 2 fallback: 1x1 / 2 / pad 0, three phases without taps", 4, 16, 16, 320, 640, 1, 2, 0,
     "conv_tc2_kernel<64,0,0>+parity_merge_add_kernel"),
    ("stride 2 fallback: BNd = 48, BNd % 32 != 0", 2, 16, 16, 48, 64, 3, 2, 1,
     "conv_tc_kernel<64,1>+parity_merge_add_kernel"),
    ("ImageNet 56x56x64 batch 64", 64, 56, 56, 64, 64, 3, 1, 1, "conv_tc2_kernel<64,0,0>"),
    ("direct: C, K not multiples of 16", 2, 8, 8, 24, 40, 3, 1, 1, "conv_dgrad_direct_kernel"),
]

# conv_dgrad_bn_bwd (STATS = 2, stride 1): (rule, N, H, W, C, K, R, stride, pad, expected)
DGRAD_BN = [
    ("halo KC 32", 2, 16, 16, 320, 32, 3, 1, 1, "conv_tc2h_kernel<32,1,2,0>"),
    ("halo KC 64, x lowers BN 256 -> 128", 2, 16, 16, 512, 64, 3, 1, 1, "conv_tc2h_kernel<64,1,2,0>"),
    ("halo TAIL32", 2, 16, 16, 320, 160, 3, 1, 1, "conv_tc2h_kernel<64,1,2,1>"),
    ("halo WRN 160@32x32 batch 128", 128, 32, 32, 160, 160, 3, 1, 1, "conv_tc2h_kernel<64,1,2,1>"),
    ("pair KC 64 on 8x8 maps", 4, 8, 8, 320, 64, 3, 1, 1, "conv_tc2_kernel<64,2,0>"),
    ("pair KC 32, P = Q = 13", 2, 13, 13, 320, 32, 3, 1, 1, "conv_tc2_kernel<32,2,0>"),
    ("pair KC 16", 4, 8, 8, 320, 48, 3, 1, 1, "conv_tc2_kernel<16,2,0>"),
]

# wgrad: (rule, N, H, W, C, K, R, stride, pad, expected)
WGRAD = [
    ("halo wgrad, P % 16 == 0, batch 128: splits > 1", 128, 32, 32, 160, 160, 3, 1, 1,
     "wgrad_tc2h_kernel+det:wgrad_reduce_splits_kernel"),
    ("halo wgrad, 8x8 maps: two images stacked per tile", 128, 8, 8, 640, 640, 3, 1, 1,
     "wgrad_tc2h_kernel+det?:wgrad_reduce_splits_kernel"),
    ("halo wgrad, one pixel tile: splits = 1", 1, 16, 8, 64, 64, 3, 1, 1, "wgrad_tc2h_kernel"),
    ("wgrad_tc SL 32 MT 2: stride 2 (WRN 160 -> 320, batch 128)", 128, 32, 32, 160, 320, 3, 2, 1,
     "wgrad_tc_kernel<32,1,2,0>+det?:wgrad_reduce_splits_kernel"),
    ("wgrad_tc SL 32 MT 1: C > 320", 4, 8, 8, 640, 640, 1, 1, 0,
     "wgrad_tc_kernel<32,1,1,0>+det?:wgrad_reduce_splits_kernel"),
    ("wgrad_tc SL 16 MT 2: C % 32 != 0", 2, 16, 16, 48, 48, 3, 1, 1,
     "wgrad_tc_kernel<16,1,2,0>+det?:wgrad_reduce_splits_kernel"),
    ("wgrad_tc SL 16 MT 1: one M tile", 2, 16, 16, 48, 80, 1, 1, 0,
     "wgrad_tc_kernel<16,1,1,0>+det?:wgrad_reduce_splits_kernel"),
    ("wgrad_tc, N = 1, Q = 136: 16 % 8 tiles need an even N for the halo kernel", 1, 8, 136, 64, 64, 3, 1, 1,
     "wgrad_tc_kernel<32,1,2,0>+det?:wgrad_reduce_splits_kernel"),
    ("wgrad_tc ImageNet 56x56x64 batch 64 (14x8 tiles overhang)", 64, 56, 56, 64, 64, 3, 1, 1,
     "wgrad_tc_kernel<32,1,2,0>+det?:wgrad_reduce_splits_kernel"),
    ("P = Q = 13: no tile of 16k rows -> direct", 2, 13, 13, 64, 64, 3, 1, 1,
     "conv_wgrad_direct_kernel+det?:wgrad_reduce_splits_kernel"),
    ("direct: C, K not multiples of 16", 2, 8, 8, 24, 40, 3, 1, 1,
     "conv_wgrad_direct_kernel+det?:wgrad_reduce_splits_kernel"),
    ("im2col stem 3x3 + bias gradient", 8, 32, 32, 3, 16, 3, 1, 1,
     "im2col_kernel+wgrad_tc_kernel<16,1,1,0>+repitch_rows_kernel<float>+conv_dbias_kernel"
     "+det?:wgrad_reduce_splits_kernel"),
    ("im2col stem 7x7 / 2 + bias gradient", 2, 64, 64, 3, 64, 7, 2, 3,
     "im2col_kernel+wgrad_tc_kernel<32,1,2,0>+repitch_rows_kernel<float>+conv_dbias_kernel"
     "+det?:wgrad_reduce_splits_kernel"),
]

# algo = direct on shapes the tensor-core path takes
DIRECT_ALGO = [
    ("fprop", 2, 16, 16, 64, 320, 3, 1, 1, "conv_fprop_direct_kernel"),
    ("dgrad", 2, 16, 16, 64, 320, 3, 2, 1, "conv_dgrad_direct_kernel"),
    ("wgrad", 2, 16, 16, 64, 64, 3, 1, 1, "conv_wgrad_direct_kernel+det?:wgrad_reduce_splits_kernel"),
]

ROWS = []
for rule, *geo, exp, epis in FPROP:
    for epi in epis:
        ROWS.append(("fprop", *geo, epi, "auto", exp, rule))
for rule, *geo, exp in DGRAD:
    for epi in ("plain", "addend"):
        ROWS.append(("dgrad", *geo, epi, "auto", exp, rule))
for rule, *geo, exp in DGRAD_BN:
    ROWS.append(("dgrad_bn", *geo, "bn_bwd", "auto", exp, rule))
for rule, *geo, exp in WGRAD:
    for mode in ("default", "deterministic"):
        ROWS.append(("wgrad", *geo, "dbias" if geo[3] == 3 else "plain", mode, exp, rule))
for pass_, *geo, exp in DIRECT_ALGO:
    epi = {"fprop": "bias+res", "dgrad": "addend", "wgrad": "plain"}[pass_]
    ROWS.append((pass_, *geo, epi, "direct", exp, "algo=direct on a tensor-core shape"))


def _row_id(r):
    return f"{r[0]}-{'x'.join(map(str, r[1:9]))}-{r[9]}-{r[10]}"


def _expect(expected, epi, deterministic):
    """-> (required regexes, allowed-only regexes) for this row."""
    req, opt = [], []
    for tok in expected.format(S=1 if "stats" in epi else 0).split("+"):
        if tok.startswith("det?:"):
            (opt if deterministic else []).append(tok[5:])
        elif tok.startswith("det:"):
            if deterministic:
                req.append(tok[4:])
        else:
            req.append(tok)
    if "stats" in epi and not tok_any(req, FUSED_STATS):
        req.append("bn_stats_kernel")          # the kernel has no fused sums: one reduction pass over y
    return req, opt


def tok_any(toks, prefixes):
    return any(t.startswith(p) for t in toks for p in prefixes)


def _assert_kernels(launched, expected, epi, deterministic, label):
    req, opt = _expect(expected, epi, deterministic)
    esc = [re.escape(t) for t in req + opt]
    stray = [k for k in launched if not any(re.fullmatch(e, k) for e in esc)]
    missing = [t for t in req if not any(re.fullmatch(re.escape(t), k) for k in launched)]
    assert not stray and not missing, f"{label}: launched {launched}, expected {req} (+ optional {opt})"


def _conv_ref(x, w, stride, pad):
    """fp64 conv of NHWC x with KRSC w, and of |x| with |w| -> NHWC (ref, mag)."""
    xd, wd = nchw(x.double()), w.double().permute(0, 3, 1, 2)
    ref = nhwc(F.conv2d(xd, wd, stride=stride, padding=pad))
    mag = nhwc(F.conv2d(xd.abs(), wd.abs(), stride=stride, padding=pad))
    return ref, mag


def _dgrad_ref(dy, w, in_shape, stride, pad):
    N, H, W, C = in_shape
    wd = w.double().permute(0, 3, 1, 2)
    dyd = nchw(dy.double())
    ref = nhwc(torch.nn.grad.conv2d_input((N, C, H, W), wd, dyd, stride=stride, padding=pad))
    mag = nhwc(torch.nn.grad.conv2d_input((N, C, H, W), wd.abs(), dyd.abs(), stride=stride, padding=pad))
    return ref, mag


def _check_sums(got, ref, mag, label):
    """fp32 per-channel results of the fused sums / statistics against fp64."""
    return assert_elementwise(got, ref, mag, 0.0, acc=SUM_ACC, label=label)


def _check_stats(y, mean, invstd, label):
    """mean / invstd must be the fp64 statistics of the STORED bf16 output."""
    yd = y.double().reshape(-1, y.shape[-1])
    m = yd.mean(0)
    var = yd.var(0, unbiased=False)
    rows = yd.shape[0]
    _check_sums(mean, m, yd.abs().mean(0), label + " mean")
    # invstd = (E[y^2] - mean^2 + eps)^-1/2: an error d in E[y^2] moves it by invstd^3 * d / 2
    ref_is = (var + EPS).rsqrt()
    mag_is = 0.5 * ref_is ** 3 * (yd * yd).sum(0) / rows * 2
    _check_sums(invstd, ref_is, mag_is, label + " invstd")


def _algo(ops, _lib, algo):
    """'auto' (the default dispatcher) | 'direct' -> the algo argument of the C entry points"""
    return ops._algo_flags(_lib.ALGO_DIRECT if algo == "direct" else None)


def _conv_geom(N, H, W, R, stride, pad):
    return (H + 2 * pad - R) // stride + 1, (W + 2 * pad - R) // stride + 1


def _run_fprop(ops, _lib, N, H, W, C, K, R, stride, pad, epi, algo, g):
    P, Q = _conv_geom(N, H, W, R, stride, pad)
    x = _act((N, H, W, C), g)
    w = _filt(K, R, C, g)
    bias = (torch.randn(K, device="cuda", generator=g) * 0.5) if "bias" in epi else None
    res = _act((N, P, Q, K), g, 0.0) if "res" in epi else None
    relu = "relu" in epi
    stats = "stats" in epi
    y = poisoned((N, P, Q, K), torch.bfloat16)
    mean = poisoned((K,), torch.float32) if stats else None
    invstd = poisoned((K,), torch.float32) if stats else None
    a = _algo(ops, _lib, algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_FPROP, N, H, W, C, K, R, R, stride, pad, a)
    ws = ops._workspace(x.device, nws) if nws else None
    acc = ops.bn_accumulators(x.device, _lib.load().b200_bn_workspace_bytes(N * P * Q, K)) if stats else None
    p = ops._p

    def call():
        if stats:
            _lib.call("b200_conv2d_fprop_stats", x.data_ptr(), w.data_ptr(), p(bias), p(res), y.data_ptr(), N, H, W,
                      C, K, R, R, stride, pad, a, p(ws), nws, acc.data_ptr(), acc.numel() * 8, EPS, mean.data_ptr(),
                      invstd.data_ptr(), ops._stream())
        else:
            _lib.call("b200_conv2d_fprop", x.data_ptr(), w.data_ptr(), p(bias), p(res), y.data_ptr(), N, H, W, C, K,
                      R, R, stride, pad, int(relu), a, p(ws), nws, ops._stream())

    _, launched = kernels_launched(call)
    ref, mag = _conv_ref(x, w, stride, pad)
    adds, npts = [], 1
    if bias is not None:
        bb = bias.bfloat16().double()           # the epilogue adds the bf16-rounded bias
        ref = ref + bb
        adds.append(bb.expand_as(ref))
    if res is not None:
        ref = ref + res.double()
        adds.append(res)
        npts = 2
    pre = ref
    if relu:
        ref = ref.clamp_min(0)
    outs = [("y", y)] + ([("mean", mean), ("invstd", invstd)] if stats else [])
    for name, t in outs:
        check_poisoned(t, name)
    worst = assert_elementwise(y, ref, mag, npts * BF16_ROUNDING, acc=ACC, addends=adds, scale64=pre, label="y")
    if stats:
        _check_stats(y, mean, invstd, "stats")
    return launched, worst


def _run_dgrad(ops, _lib, N, H, W, C, K, R, stride, pad, epi, algo, g):
    P, Q = _conv_geom(N, H, W, R, stride, pad)
    dy = _act((N, P, Q, K), g)
    w = _filt(K, R, C, g)
    wt = w.permute(3, 1, 2, 0).contiguous()
    add = _act((N, H, W, C), g, 0.0) if epi == "addend" else None
    dx = poisoned((N, H, W, C), torch.bfloat16)
    a = _algo(ops, _lib, algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_DGRAD, N, H, W, C, K, R, R, stride, pad, a)
    ws = ops._workspace(dy.device, nws) if nws else None
    if ws is not None:
        ws.fill_(0xFF)   # the parity-split workspace of the stride-2 fallback: stale bytes must not leak through

    def call():
        _lib.call("b200_conv2d_dgrad", dy.data_ptr(), wt.data_ptr(), ops._p(add), dx.data_ptr(), N, H, W, C, K, R, R,
                  stride, pad, a, ops._p(ws), nws, ops._stream())

    _, launched = kernels_launched(call)
    check_poisoned(dx, "dx")
    ref, mag = _dgrad_ref(dy, w, (N, H, W, C), stride, pad)
    adds = []
    if add is not None:
        ref = ref + add.double()
        adds = [add]
    worst = assert_elementwise(dx, ref, mag, (2 if adds else 1) * BF16_ROUNDING, acc=ACC, addends=adds, label="dx")
    return launched, worst


def _bn_inputs(ops, N, H, W, C, p, g):
    x = (torch.randn(N, H, W, C, device="cuda", generator=g) * 1.3 + 0.4).bfloat16()
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.3
    mean, invstd = ops.bn_stats(x, EPS)
    _, mask = ops.bn_act_fwd(x, mean, invstd, gamma, beta, relu=True, dropout_p=p, seed=5, want_mask=True)
    return x, gamma, mean, invstd, mask


def _gate(mask, shape):
    bits = (mask.unsqueeze(-1) >> torch.arange(8, device=mask.device, dtype=torch.uint8)) & 1
    return bits.reshape(shape).bool()


def _masked_grad(dy, gate, p):
    """g of the BN backward: dy where the unit was active and kept, scaled by 1/(1-p) and rounded to bf16 (the
    kernels' rounding point), else 0 -> fp64."""
    if p > 0:
        inv_keep = torch.tensor(1.0, dtype=torch.float32) / (1.0 - torch.tensor(p, dtype=torch.float32))
        gd = (dy.float() * inv_keep.item()).bfloat16().double()
    else:
        gd = dy.double()
    return torch.where(gate, gd, torch.zeros_like(gd))


def _bn_sums_ref(gd, x, mean, invstd):
    """fp64 (dbeta, dgamma) and their magnitudes from g (fp64), x, the fp32 statistics."""
    C = x.shape[-1]
    g2 = gd.reshape(-1, C)
    xd = x.double().reshape(-1, C)
    md, isd = mean.double(), invstd.double()
    xhat = (xd - md) * isd
    dbeta = g2.sum(0)
    dgamma = (g2 * xhat).sum(0)
    mag_b = g2.abs().sum(0)
    mag_g = isd * ((g2 * xd).abs().sum(0) + md.abs() * mag_b)   # the kernels form invstd * (sum g*x - mean * sum g)
    return dbeta, dgamma, mag_b, mag_g, xhat


def _run_dgrad_bn(ops, _lib, N, H, W, C, K, R, stride, pad, epi, algo, g, p=0.3):
    P, Q = _conv_geom(N, H, W, R, stride, pad)
    x, gamma, mean, invstd, mask = _bn_inputs(ops, N, H, W, C, p, g)
    dy = (torch.randn(N, P, Q, K, device="cuda", generator=g) * 0.1 + 0.05).bfloat16()
    w = _filt(K, R, C, g)
    wt = w.permute(3, 1, 2, 0).contiguous()
    dx = poisoned((N, H, W, C), torch.bfloat16)
    dgamma = poisoned((C,), torch.float32)
    dbeta = poisoned((C,), torch.float32)
    a = _algo(ops, _lib, algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_DGRAD, N, H, W, C, K, R, R, stride, pad, a)
    ws = ops._workspace(dy.device, nws) if nws else None
    nst = _lib.load().b200_bn_workspace_bytes(N * H * W, C)
    st = ops.bn_accumulators(dy.device, nst)
    import ctypes
    fused = ctypes.c_int(0)

    def call():
        _lib.call("b200_conv2d_dgrad_bnbwd", dy.data_ptr(), wt.data_ptr(), dx.data_ptr(), N, H, W, C, K, R, R, stride,
                  pad, a, ops._p(ws), nws, x.data_ptr(), mask.data_ptr(), mean.data_ptr(), invstd.data_ptr(), float(p),
                  dgamma.data_ptr(), dbeta.data_ptr(), st.data_ptr(), nst, ctypes.byref(fused), ops._stream())

    _, launched = kernels_launched(call)
    assert fused.value == 1, "this route fuses the BN-backward sums"
    for name, t in (("dx", dx), ("dgamma", dgamma), ("dbeta", dbeta)):
        check_poisoned(t, name)
    ref, mag = _dgrad_ref(dy, w, (N, H, W, C), stride, pad)
    worst = assert_elementwise(dx, ref, mag, BF16_ROUNDING, acc=ACC, label="dx")
    gd = _masked_grad(dx, _gate(mask, dx.shape), p)          # from the stored bf16 dx, the kernel's rounding point
    db_ref, dg_ref, mag_b, mag_g, _ = _bn_sums_ref(gd, x, mean, invstd)
    _check_sums(dbeta, db_ref, mag_b, "dbeta")
    _check_sums(dgamma, dg_ref, mag_g, "dgamma")
    return launched, worst


def _run_wgrad(ops, _lib, N, H, W, C, K, R, stride, pad, epi, algo, g):
    P, Q = _conv_geom(N, H, W, R, stride, pad)
    x = _act((N, H, W, C), g)
    dy = _act((N, P, Q, K), g, 0.25)
    want_db = epi == "dbias"
    dw = poisoned((K, R, R, C), torch.float32)
    db = poisoned((K,), torch.float32) if want_db else None
    a = None if algo in ("default", "deterministic", "auto") else _lib.ALGO_DIRECT

    def call():
        return ops.conv_wgrad(dy, x, R, R, stride, pad, want_dbias=want_db, algo=a, out=dw, out_db=db)

    with ops.deterministic(algo == "deterministic"):
        (rw, rb), launched = kernels_launched(call)
    assert rw.data_ptr() == dw.data_ptr()
    check_poisoned(dw, "dw")
    xd, dyd = nchw(x.double()), nchw(dy.double())
    ref = torch.nn.grad.conv2d_weight(xd, (K, C, R, R), dyd, stride=stride, padding=pad).permute(0, 2, 3, 1)
    mag = torch.nn.grad.conv2d_weight(xd.abs(), (K, C, R, R), dyd.abs(), stride=stride, padding=pad).permute(0, 2, 3, 1)
    worst = assert_elementwise(dw, ref, mag, 0.0, acc=WGRAD_ACC, label="dw")
    if want_db:
        check_poisoned(db, "dbias")
        d2 = dy.double().reshape(-1, K)
        _check_sums(db, d2.sum(0), d2.abs().sum(0), "dbias")
    return launched, worst


_RUN = {"fprop": _run_fprop, "dgrad": _run_dgrad, "dgrad_bn": _run_dgrad_bn, "wgrad": _run_wgrad}


@pytest.fixture(scope="module", autouse=True)
def _fp64_references():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


@pytest.mark.parametrize("row", ROWS, ids=_row_id)
def test_conv_route(row):
    ops, _lib = _ops()
    pass_, N, H, W, C, K, R, stride, pad, epi, algo, expected, rule = row
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(_row_id(row).encode()))
    launched, (worst, worst_acc) = _RUN[pass_](ops, _lib, N, H, W, C, K, R, stride, pad, epi, algo, g)
    print(f"[route] {_row_id(row)}: {'+'.join(launched)}; worst ratio {worst:.4f}, accumulation term "
          f"{worst_acc:.4f}  ({rule})")
    _assert_kernels(launched, expected, epi, algo == "deterministic", rule)


# ---------------------------------------------------------------------------------------------------------------
# coverage: every kernel instantiation the default environment can reach has a row
# ---------------------------------------------------------------------------------------------------------------
# instantiation -> the api.cu lines that choose it
REACHABLE = {
    "conv_tc2h_kernel<32,1,0,0>": "run_conv_tc: launch_conv_tc2h<32, 1, false> (mt2 needs B200_HALO_MT=2)",
    "conv_tc2h_kernel<32,1,1,0>": "run_conv_tc: stats -> launch_conv_tc2h<32, 1, true>",
    "conv_tc2h_kernel<32,1,2,0>": "run_conv_tc: bb -> launch_conv_tc2h<32, 1, 2>",
    "conv_tc2h_kernel<64,1,0,0>": "run_conv_tc: KC == 64 -> launch_conv_tc2h<64, 1, false>",
    "conv_tc2h_kernel<64,1,1,0>": "run_conv_tc: stats, KC == 64 -> launch_conv_tc2h<64, 1, true>",
    "conv_tc2h_kernel<64,1,2,0>": "run_conv_tc: bb, KC == 64 -> launch_conv_tc2h<64, 1, 2>",
    "conv_tc2h_kernel<64,1,0,1>": "run_conv_tc: mixed -> launch_conv_tc2h<64, 1, false, true>",
    "conv_tc2h_kernel<64,1,1,1>": "run_conv_tc: stats, mixed -> launch_conv_tc2h<64, 1, true, true>",
    "conv_tc2h_kernel<64,1,2,1>": "run_conv_tc: bb, mixed -> launch_conv_tc2h<64, 1, 2, true>",
    "conv_tc2_kernel<16,0,0>": "run_conv_tc: pair -> launch_conv_tc2<16, false>",
    "conv_tc2_kernel<32,0,0>": "run_conv_tc: pair -> launch_conv_tc2<32, false>",
    "conv_tc2_kernel<64,0,0>": "run_conv_tc: pair -> launch_conv_tc2<64, false>",
    "conv_tc2_kernel<16,1,0>": "run_conv_tc: pair, stats -> launch_conv_tc2<16, true>",
    "conv_tc2_kernel<32,1,0>": "run_conv_tc: pair, stats -> launch_conv_tc2<32, true>",
    "conv_tc2_kernel<64,1,0>": "run_conv_tc: pair, stats -> launch_conv_tc2<64, true>",
    "conv_tc2_kernel<16,2,0>": "run_conv_tc: pair, bb -> launch_conv_tc2<16, 2>",
    "conv_tc2_kernel<32,2,0>": "run_conv_tc: pair, bb -> launch_conv_tc2<32, 2>",
    "conv_tc2_kernel<64,2,0>": "run_conv_tc: pair, bb -> launch_conv_tc2<64, 2>",
    # launch_conv_tc_cs: CS = 4 needs B200_CONV_CLUSTER=4 (the default cluster size is 2): not reachable
    "conv_tc_kernel<16,1>": "launch_conv_tc_cs<16>: cs halved to 1",
    "conv_tc_kernel<16,2>": "launch_conv_tc_cs<16>: cs = 2",
    "conv_tc_kernel<32,1>": "launch_conv_tc_cs<32>: cs halved to 1",
    "conv_tc_kernel<32,2>": "launch_conv_tc_cs<32>: cs = 2",
    "conv_tc_kernel<64,1>": "launch_conv_tc_cs<64>: cs halved to 1",
    "conv_tc_kernel<64,2>": "launch_conv_tc_cs<64>: cs = 2",
    "parity_merge_add_kernel": "conv2d_dgrad_impl: stride-2 per-phase fallback",
    "im2col_kernel": "conv2d_fprop_impl / b200_conv2d_wgrad: use_im2col",
    "repitch_rows_kernel<bf16>": "conv2d_fprop_impl: im2col filter repitch",
    "repitch_rows_kernel<float>": "b200_conv2d_wgrad: im2col gradient repitch",
    "conv_fprop_direct_kernel": "conv2d_fprop_impl: !tc",
    "conv_dgrad_direct_kernel": "conv2d_dgrad_impl: !tc",
    "conv_wgrad_direct_kernel": "b200_conv2d_wgrad: !tc",
    "conv_dbias_kernel": "b200_conv2d_wgrad: dbias",
    "wgrad_tc2h_kernel": "run_wgrad_tc -> run_wgrad_tc2h",
    # launch_wgrad_tc_cs: CS = 2 / 4 need B200_WGRAD_CLUSTER (default 1), SL = 64 needs B200_WGRAD_SLAB=64
    "wgrad_tc_kernel<16,1,1,0>": "run_wgrad_tc: SL 16, mt 1",
    "wgrad_tc_kernel<16,1,2,0>": "run_wgrad_tc: SL 16, mt 2",
    "wgrad_tc_kernel<32,1,1,0>": "run_wgrad_tc: SL 32, mt 1",
    "wgrad_tc_kernel<32,1,2,0>": "run_wgrad_tc: SL 32, mt 2",
    "wgrad_reduce_splits_kernel": "wgrad_reduce_splits: deterministic mode, splits > 1",
}


def test_route_table_covers_every_reachable_kernel():
    covered = set()
    for pass_, *_, epi, algo, expected, _rule in ROWS:
        for det in (False, True):
            req, opt = _expect(expected, epi, det)
            covered.update(req)
            covered.update(opt)
    missing = sorted(set(REACHABLE) - covered)
    assert not missing, f"kernel instantiations without a row in the route table: {missing}"


# ---------------------------------------------------------------------------------------------------------------
# composite references: bn_act_bwd, and conv_dgrad_bn_bwd + bn_act_bwd(reduced=...), from their definitions
# ---------------------------------------------------------------------------------------------------------------
def _bn_bwd_ref(gd, x, mean, invstd, gamma, rows):
    """fp64 dx = gamma * invstd * (g - (dbeta + xhat * dgamma) / rows) and a magnitude bounding the fp32 formula
    (k1 g + k2 x + k3) and the summation error of dbeta / dgamma."""
    C = x.shape[-1]
    dbeta, dgamma, mag_b, mag_g, xhat = _bn_sums_ref(gd, x, mean, invstd)
    gm = gamma.double()
    isd = invstd.double()
    g2 = gd.reshape(-1, C)
    k1 = gm * isd
    dx = k1 * (g2 - (dbeta + xhat * dgamma) / rows)
    xd = x.double().reshape(-1, C)
    k2 = k1 * isd * dgamma / rows
    mag = (k1 * g2).abs() + (k2 * xd).abs() + (k1 * dbeta / rows).abs() + (k2 * mean.double()).abs() \
        + k1.abs() * (mag_b + xhat.abs() * mag_g / isd) / rows
    return dbeta, dgamma, mag_b, mag_g, dx.reshape(x.shape), mag.reshape(x.shape)


def _bn_act_bwd_into(ops, _lib, dy, y, x, mean, invstd, gamma, relu, p, seed, addend, mask, want_dskip, reduced):
    """ops.bn_act_bwd with poisoned outputs (same C entry points and argument order)."""
    C = dy.shape[-1]
    rows = dy.numel() // C
    dx = poisoned(tuple(dy.shape), torch.bfloat16)
    dskip = poisoned(tuple(dy.shape), torch.bfloat16) if want_dskip else None
    p_ = ops._p
    if reduced is not None:
        dgamma, dbeta = reduced
        _lib.call("b200_bn_act_bwd_apply", dy.data_ptr(), mask.data_ptr(), x.data_ptr(), dx.data_ptr(), p_(dskip),
                  p_(addend), rows, C, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(),
                  dbeta.data_ptr(), int(relu), float(p), ops._stream())
        return dx, dgamma, dbeta, dskip
    dgamma = poisoned((C,), torch.float32)
    dbeta = poisoned((C,), torch.float32)
    nws = _lib.load().b200_bn_workspace_bytes(rows, C)
    ws = ops.bn_accumulators(dy.device, nws)
    _lib.call("b200_bn_act_bwd", dy.data_ptr(), p_(y), p_(mask), x.data_ptr(), dx.data_ptr(), p_(dskip), p_(addend),
              rows, C, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(),
              int(relu), float(p), int(seed), ops.step_counter(dy.device).data_ptr() if p > 0 else None,
              ws.data_ptr(), nws, ops._stream())
    return dx, dgamma, dbeta, dskip


def _check_bn_bwd(outs, gd, x, mean, invstd, gamma, addend, label):
    dx, dgamma, dbeta, dskip = outs
    C = x.shape[-1]
    rows = x.numel() // C
    db_ref, dg_ref, mag_b, mag_g, dx_ref, mag = _bn_bwd_ref(gd, x, mean, invstd, gamma, rows)
    for name, t in (("dx", dx), ("dgamma", dgamma), ("dbeta", dbeta)) + ((("dskip", dskip),) if dskip is not None
                                                                        else ()):
        if hasattr(t, "_poison"):
            check_poisoned(t, f"{label} {name}")
    _check_sums(dbeta, db_ref, mag_b, f"{label} dbeta")
    _check_sums(dgamma, dg_ref, mag_g, f"{label} dgamma")
    adds, npts = [], 1
    if addend is not None:
        dx_ref = dx_ref + addend.double()
        adds, npts = [addend], 2
    worst = assert_elementwise(dx, dx_ref, mag, npts * BF16_ROUNDING, acc=ACC, addends=adds, label=f"{label} dx")
    if dskip is not None:
        assert torch.equal(dskip.double(), gd), f"{label}: dskip != g"
    return worst


@pytest.mark.parametrize("path", ["y", "mask"])
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("extras", ["none", "addend", "addend+dskip"])
def test_bn_act_bwd_against_fp64(path, relu, p, extras):
    ops, _lib = _ops()
    N, H, W, C = 4, 16, 16, 160
    g = torch.Generator(device="cuda").manual_seed(17)
    x = (torch.randn(N, H, W, C, device="cuda", generator=g) * 1.3 + 0.4).bfloat16()
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.3
    dy = (torch.randn(N, H, W, C, device="cuda", generator=g) + 0.2).bfloat16()
    addend = _act((N, H, W, C), g, 0.0) if "addend" in extras else None
    mean, invstd = ops.bn_stats(x, EPS)
    y, mask = ops.bn_act_fwd(x, mean, invstd, gamma, beta, relu=relu, dropout_p=p, seed=9, want_mask=True)
    gate = _gate(mask, x.shape)                                    # the kernel's own ReLU-and-keep gate
    if relu and p == 0:
        assert torch.equal(gate, y != 0)
    gd = _masked_grad(dy, gate, p)
    outs = _bn_act_bwd_into(ops, _lib, dy, y if path == "y" else None, x, mean, invstd, gamma, relu, p, 9, addend,
                            mask if path == "mask" else None, "dskip" in extras, None)
    _check_bn_bwd(outs, gd, x, mean, invstd, gamma, addend, f"bn_act_bwd[{path}, relu={relu}, p={p}, {extras}]")


# BNBWD_SHAPES of test_kernels_gpu.py: N, H, C (BN channels), K, R, stride, pad, fused sums expected
BNBWD_SHAPES = [
    (8, 32, 160, 160, 3, 1, 1, True),
    (16, 16, 320, 320, 3, 1, 1, True),
    (32, 8, 640, 640, 3, 1, 1, True),
    (8, 32, 160, 320, 3, 2, 1, False),
    (4, 16, 64, 128, 3, 1, 1, True),
    (2, 8, 24, 40, 3, 1, 1, False),
    (64, 32, 512, 128, 1, 1, 0, False),
    (64, 32, 128, 512, 1, 1, 0, True),
]


@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("shape", BNBWD_SHAPES, ids=lambda s: "x".join(map(str, s[:7])))
def test_dgrad_bn_bwd_chain_against_fp64(shape, p):
    """conv_dgrad_bn_bwd + bn_act_bwd(reduced=...) (or + bn_act_bwd's own reduction where the sums are not fused)
    against the fp64 chain da = bf16(conv_transpose(dy, w)), g = da * keep / (1 - p), dbeta = sum g,
    dgamma = sum g * xhat, dx = bf16(gamma * invstd * (g - (dbeta + xhat * dgamma) / rows)) + addend."""
    import ctypes
    ops, _lib = _ops()
    N, H, C, K, R, stride, pad, expect = shape
    P = (H + 2 * pad - R) // stride + 1
    g = torch.Generator(device="cuda").manual_seed(11)
    x, gamma, mean, invstd, mask = _bn_inputs(ops, N, H, H, C, p, g)
    dy = (torch.randn(N, P, P, K, device="cuda", generator=g) * 0.1 + 0.05).bfloat16()
    w = _filt(K, R, C, g)
    wt = w.permute(3, 1, 2, 0).contiguous()
    addend = _act((N, H, H, C), g, 0.0)
    da = poisoned((N, H, H, C), torch.bfloat16)
    dgamma = poisoned((C,), torch.float32)
    dbeta = poisoned((C,), torch.float32)
    a = ops._algo_flags(None)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_DGRAD, N, H, H, C, K, R, R, stride, pad, a)
    ws = ops._workspace(dy.device, nws) if nws else None
    nst = _lib.load().b200_bn_workspace_bytes(N * H * H, C)
    st = ops.bn_accumulators(dy.device, nst)
    fused = ctypes.c_int(0)
    _lib.call("b200_conv2d_dgrad_bnbwd", dy.data_ptr(), wt.data_ptr(), da.data_ptr(), N, H, H, C, K, R, R, stride, pad,
              a, ops._p(ws), nws, x.data_ptr(), mask.data_ptr(), mean.data_ptr(), invstd.data_ptr(), float(p),
              dgamma.data_ptr(), dbeta.data_ptr(), st.data_ptr(), nst, ctypes.byref(fused), ops._stream())
    assert bool(fused.value) == expect
    check_poisoned(da, "da")
    ref, mag = _dgrad_ref(dy, w, (N, H, H, C), stride, pad)
    assert_elementwise(da, ref, mag, BF16_ROUNDING, acc=ACC, label="da")
    outs = _bn_act_bwd_into(ops, _lib, da, None, x, mean, invstd, gamma, True, p, 5, addend, mask, False,
                            (dgamma, dbeta) if fused.value else None)
    gd = _masked_grad(da, _gate(mask, da.shape), p)
    _check_bn_bwd(outs, gd, x, mean, invstd, gamma, addend, f"chain p={p}")
