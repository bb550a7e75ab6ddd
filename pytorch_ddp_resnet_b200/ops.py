"""
Raw kernel wrappers: torch tensors in, torch tensors out, no autograd. Every function here is one or
two launches of a kernel in libb200resnet.so on the *current* torch CUDA stream.

Conventions (see include/b200resnet.h):
  * activations: contiguous bf16 tensors of shape [N, H, W, C] (NHWC);
  * conv filters: bf16 [K, R, S, C] (KRSC) and bf16 [C, R, S, K] (CRSK) working copies;
  * everything per-channel / per-parameter is fp32.
"""
import ctypes
import os
from typing import Optional, Tuple

import torch

from pytorch_ddp_resnet_b200 import _lib

_ALGO_NAMES = {"auto": _lib.ALGO_AUTO, "direct": _lib.ALGO_DIRECT, "tc": _lib.ALGO_TC}
_workspaces = {}
_step_counters = {}


# Precision mode of the forward pass: "bf16" (training and fast evaluation: bf16 activations, fp32 accumulate)
# or "tf32" (the reference's un-autocast path, evaluation.py:32-39: fp32 activations, TF32 convolutions).
# The mode only decides what a stem does with an fp32 image batch; every later kernel follows the dtype of
# the activation it receives.
_precision = ["bf16"]


def get_precision() -> str:
    return _precision[0]


class precision:
    """with ops.precision("tf32"): logits = model(x)   # forward-only fp32 / TF32 evaluation"""

    def __init__(self, mode: str):
        if mode not in ("bf16", "tf32"):
            raise ValueError("precision must be 'bf16' or 'tf32'")
        self.mode = mode

    def __enter__(self):
        self.prev = _precision[0]
        _precision[0] = self.mode
        return self

    def __exit__(self, *exc):
        _precision[0] = self.prev
        return False


# Deterministic mode: every cross-CTA / cross-warp fp32 reduction of the step runs in a fixed order (wgrad
# pixel-range splits and bias-gradient blocks from ordered partials instead of fp32 atomics, conv-epilogue
# statistics quadrant by quadrant), so a step is bit-reproducible run after run and graph replay == eager.
# On inside `with ops.deterministic():`, after torch.use_deterministic_algorithms(True), or with
# B200_DETERMINISTIC=1 in the environment (read once at import). Off by default, like cuDNN in the reference.
_deterministic = [os.environ.get("B200_DETERMINISTIC", "0") not in ("", "0")]


def is_deterministic() -> bool:
    return _deterministic[0] or torch.are_deterministic_algorithms_enabled()


class deterministic:
    """with ops.deterministic(): loss.backward()   # bit-reproducible weight gradients and batch statistics"""

    def __init__(self, enabled: bool = True):
        self.enabled = bool(enabled)

    def __enter__(self):
        self.prev = _deterministic[0]
        _deterministic[0] = self.enabled
        return self

    def __exit__(self, *exc):
        _deterministic[0] = self.prev
        return False


def _algo_flags(algo: Optional[int]) -> int:
    algo = conv_algo() if algo is None else algo
    return (algo | _lib.ALGO_DETERMINISTIC) if is_deterministic() else algo


# Eval-mode batch-norm folding (utils/fold_util.py): on inside `with ops.fold_bn(True)`.
_fold_bn = [False]


def get_fold_bn() -> bool:
    return _fold_bn[0]


class fold_bn:
    def __init__(self, on: bool = True):
        self.on = bool(on)

    def __enter__(self):
        self.prev = _fold_bn[0]
        _fold_bn[0] = self.on
        return self

    def __exit__(self, *exc):
        _fold_bn[0] = self.prev
        return False


def step_counter(device: torch.device) -> torch.Tensor:
    """Per-device uint64 step counter (stored as int64) that the dropout kernels fold into their seed.
    It only advances through tick(): a captured training step ticks it once per replay."""
    t = _step_counters.get(device.index)
    if t is None:
        t = torch.zeros((), dtype=torch.int64, device=device)
        _step_counters[device.index] = t
    return t


_bn_accums = {}


def bn_accumulators(device: torch.device, nbytes: int = 0) -> torch.Tensor:
    """Zero-filled fp64 accumulators + ticket counter of b200_bn_stats / b200_bn_act_bwd (see
    include/b200resnet.h: zero on entry, zero again on exit). One buffer per (device, stream); all
    capturing streams of a device share one buffer that is created before any capture starts (by the
    first eager call, or by GraphedTrainStep), so that no fill kernel is recorded into a graph."""
    capturing = torch.cuda.is_current_stream_capturing()
    key = (device.index, "capture" if capturing else _stream())
    t = _bn_accums.get(key)
    if t is None or t.numel() * 8 < nbytes:
        t = torch.zeros(max(1 << 15, (nbytes + 7) // 8), dtype=torch.float64, device=device)
        _bn_accums[key] = t
        if not capturing and (device.index, "capture") not in _bn_accums:
            _bn_accums[(device.index, "capture")] = torch.zeros_like(t)
    return t


# Fused conv + BN statistics: conv_fprop(want_stats=True) sums its output per channel in the epilogue, and the
# CTA that finishes last turns the sums into mean / invstd (and clears the accumulators). The record
# (output pointer, rows, C, eps, mean, invstd) is kept here; the batch-norm statistics call that follows on
# the SAME tensor takes mean / invstd from it without launching anything. An unconsumed record is simply dropped.
_pending_stats = {}


def _accum_key(device: torch.device):
    return (device.index, "capture" if torch.cuda.is_current_stream_capturing() else _stream())


def _drop_pending_stats(device: torch.device) -> None:
    _pending_stats.pop(_accum_key(device), None)


_FUSED_BN_STATS = os.environ.get("B200_FUSED_BN_STATS", "1") != "0"   # experiment switch, read once at import


def fused_bn_stats_enabled() -> bool:
    return _FUSED_BN_STATS


def tick(device: torch.device) -> None:
    _lib.require_device(device.index or 0)
    _lib.call("b200_tick", step_counter(device).data_ptr(), _stream())



_CONV_ALGO = _ALGO_NAMES[os.environ.get("B200_CONV_ALGO", "auto")]   # experiment switch, read once at import


def conv_algo() -> int:
    """Conv algorithm from B200_CONV_ALGO (auto | direct | tc); 'auto' uses tcgen05 when it can."""
    return _CONV_ALGO


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _check_act(t: torch.Tensor, name: str) -> None:
    if not (t.is_cuda and t.dtype == torch.bfloat16 and t.is_contiguous()):
        raise _lib.B200Error(
            f"{name}: expected a contiguous CUDA bf16 tensor, got {t.dtype} {t.device} "
            f"contiguous={t.is_contiguous()}")
    if t.device.index != torch.cuda.current_device():
        raise _lib.B200Error(f"{name}: tensor lives on {t.device} but the current CUDA device is "
                             f"{torch.cuda.current_device()} (kernels launch on the current device's stream)")
    _lib.require_device(t.device.index or 0)


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    key = (device.index, _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


# --------------------------------------------------------------------------------------------------
# filters / layout
# --------------------------------------------------------------------------------------------------
def weight_prep(w_krsc_f32: torch.Tensor, want_crsk: bool = True) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """fp32 [K,R,S,C] master -> (bf16 [K,R,S,C], bf16 [C,R,S,K])."""
    assert w_krsc_f32.dtype == torch.float32 and w_krsc_f32.is_contiguous() and w_krsc_f32.is_cuda
    _lib.require_device(w_krsc_f32.device.index or 0)
    K, R, S, C = w_krsc_f32.shape
    wk = torch.empty((K, R, S, C), dtype=torch.bfloat16, device=w_krsc_f32.device)
    wt = torch.empty((C, R, S, K), dtype=torch.bfloat16, device=w_krsc_f32.device) if want_crsk else None
    _lib.call("b200_weight_prep", w_krsc_f32.data_ptr(), wk.data_ptr(), _p(wt), K, R * S, C, _stream())
    return wk, wt


def weight_prep_table(entries) -> torch.Tensor:
    """Device table for weight_prep_multi from [(w_krsc_f32, wk_bf16, wt_bf16)]: 40-byte records."""
    import struct
    blob = b"".join(struct.pack("<QQQiiii", w.data_ptr(), wk.data_ptr(), wt.data_ptr(), w.shape[0],
                                w.shape[1] * w.shape[2], w.shape[3], 0) for w, wk, wt in entries)
    host = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
    return host.to(entries[0][0].device)


def weight_prep_multi(table: torch.Tensor, n: int) -> None:
    _lib.require_device(table.device.index or 0)
    _lib.call("b200_weight_prep_multi", table.data_ptr(), n, _stream())


def nchw_f32_to_nhwc_bf16(x: torch.Tensor) -> torch.Tensor:
    assert x.dtype == torch.float32 and x.is_contiguous() and x.is_cuda and x.dim() == 4
    _lib.require_device(x.device.index or 0)
    N, C, H, W = x.shape
    y = torch.empty((N, H, W, C), dtype=torch.bfloat16, device=x.device)
    _lib.call("b200_nchw_f32_to_nhwc_bf16", x.data_ptr(), y.data_ptr(), N, C, H, W, _stream())
    return y


# --------------------------------------------------------------------------------------------------
# convolution
# --------------------------------------------------------------------------------------------------
def _out_hw(H, W, R, S, stride, pad):
    return (H + 2 * pad - R) // stride + 1, (W + 2 * pad - S) // stride + 1


def conv_fprop(x, w_krsc, stride: int, pad: int, bias=None, residual=None, algo=None,
               want_stats: bool = False, eps: float = 1e-5, relu: bool = False):
    """want_stats: also compute the batch-norm statistics (mean, invstd with `eps`) of the output in the conv
    kernel itself; the next bn_batch_stats(y) / bn_stats(y) picks them up."""
    _check_act(x, "conv_fprop.x")
    N, H, W, C = x.shape
    K, R, S, Cw = w_krsc.shape
    assert Cw == C and w_krsc.dtype == torch.bfloat16 and w_krsc.is_contiguous()
    P, Q = _out_hw(H, W, R, S, stride, pad)
    y = torch.empty((N, P, Q, K), dtype=torch.bfloat16, device=x.device)
    if residual is not None:
        _check_act(residual, "conv_fprop.residual")
        assert residual.shape == y.shape
    algo = _algo_flags(algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_FPROP, N, H, W, C, K, R, S, stride, pad, algo)
    ws = _workspace(x.device, nws) if nws else None
    if want_stats and relu:
        raise _lib.B200Error("conv_fprop: the epilogue ReLU belongs to evaluation (folded batch norm), not to training")
    if want_stats and K % 8 == 0 and fused_bn_stats_enabled():
        _drop_pending_stats(x.device)
        nacc = _lib.load().b200_bn_workspace_bytes(N * P * Q, K)
        acc = bn_accumulators(x.device, nacc)
        mean = torch.empty((K,), dtype=torch.float32, device=x.device)
        invstd = torch.empty((K,), dtype=torch.float32, device=x.device)
        _lib.call("b200_conv2d_fprop_stats", x.data_ptr(), w_krsc.data_ptr(), _p(bias), _p(residual),
                  y.data_ptr(), N, H, W, C, K, R, S, stride, pad, algo, _p(ws), nws, acc.data_ptr(),
                  acc.numel() * 8, float(eps), mean.data_ptr(), invstd.data_ptr(), _stream())
        _pending_stats[_accum_key(x.device)] = (y.data_ptr(), N * P * Q, K, float(eps), mean, invstd)
        return y
    _lib.call("b200_conv2d_fprop", x.data_ptr(), w_krsc.data_ptr(), _p(bias), _p(residual),
              y.data_ptr(), N, H, W, C, K, R, S, stride, pad, int(relu), algo, _p(ws), nws, _stream())
    return y


def conv_dgrad(dy, w_crsk, in_hw: Tuple[int, int], stride: int, pad: int, addend=None, algo=None):
    _check_act(dy, "conv_dgrad.dy")
    N, P, Q, K = dy.shape
    C, R, S, Kw = w_crsk.shape
    assert Kw == K and w_crsk.dtype == torch.bfloat16 and w_crsk.is_contiguous()
    H, W = in_hw
    assert _out_hw(H, W, R, S, stride, pad) == (P, Q)
    dx = torch.empty((N, H, W, C), dtype=torch.bfloat16, device=dy.device)
    if addend is not None:
        _check_act(addend, "conv_dgrad.addend")
        assert addend.shape == dx.shape
    algo = _algo_flags(algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_DGRAD, N, H, W, C, K, R, S, stride, pad, algo)
    ws = _workspace(dy.device, nws) if nws else None
    _lib.call("b200_conv2d_dgrad", dy.data_ptr(), w_crsk.data_ptr(), _p(addend), dx.data_ptr(),
              N, H, W, C, K, R, S, stride, pad, algo, _p(ws), nws, _stream())
    return dx


_FUSED_BN_BWD = os.environ.get("B200_FUSED_BN_BWD", "1") != "0"   # experiment switch, read once at import


def conv_dgrad_bn_bwd(dy, w_crsk, in_hw: Tuple[int, int], stride: int, pad: int, *, x_bn, mask, mean, invstd,
                      dropout_p: float = 0.0, out_dgamma=None, out_dbeta=None, algo=None):
    """conv_dgrad whose result is the dy of the BN + ReLU + dropout backward of the layer in front of the conv
    (x_bn: that batch norm's input, mask: the bytes its bn_act_fwd(want_mask=True) wrote). Returns (dx, sums):
    sums = (dgamma, dbeta) when the conv epilogue reduced them (pass it to bn_act_bwd(..., reduced=sums)), None when
    this shape has no such epilogue (then bn_act_bwd does its own reduction pass)."""
    if not _FUSED_BN_BWD:
        return conv_dgrad(dy, w_crsk, in_hw, stride, pad, algo=algo), None
    _check_act(dy, "conv_dgrad_bn_bwd.dy")
    _check_act(x_bn, "conv_dgrad_bn_bwd.x_bn")
    N, P, Q, K = dy.shape
    C, R, S, Kw = w_crsk.shape
    assert Kw == K and w_crsk.dtype == torch.bfloat16 and w_crsk.is_contiguous()
    H, W = in_hw
    assert _out_hw(H, W, R, S, stride, pad) == (P, Q) and x_bn.shape == (N, H, W, C)
    assert mask.dtype == torch.uint8 and mask.is_contiguous() and mask.numel() * 8 == x_bn.numel()
    dx = torch.empty((N, H, W, C), dtype=torch.bfloat16, device=dy.device)
    dgamma = out_dgamma.view(C) if out_dgamma is not None else torch.empty((C,), dtype=torch.float32, device=dy.device)
    dbeta = out_dbeta.view(C) if out_dbeta is not None else torch.empty((C,), dtype=torch.float32, device=dy.device)
    algo = _algo_flags(algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_DGRAD, N, H, W, C, K, R, S, stride, pad, algo)
    ws = _workspace(dy.device, nws) if nws else None
    nst = _lib.load().b200_bn_workspace_bytes(N * H * W, C)
    _drop_pending_stats(dy.device)
    st = bn_accumulators(dy.device, nst)
    fused = ctypes.c_int(0)
    _lib.call("b200_conv2d_dgrad_bnbwd", dy.data_ptr(), w_crsk.data_ptr(), dx.data_ptr(), N, H, W, C, K, R, S, stride,
              pad, algo, _p(ws), nws, x_bn.data_ptr(), mask.data_ptr(), mean.data_ptr(), invstd.data_ptr(),
              float(dropout_p), dgamma.data_ptr(), dbeta.data_ptr(), st.data_ptr(), nst, ctypes.byref(fused),
              _stream())
    return dx, ((dgamma, dbeta) if fused.value else None)


def conv_wgrad(dy, x, R: int, S: int, stride: int, pad: int, want_dbias: bool = False, algo=None,
               out=None, out_db=None):
    """Returns (dw fp32 [K,R,S,C], dbias fp32 [K] or None). `out` / `out_db`: optional preallocated
    destinations (views into the flat gradient buffer that the bucketed NCCL all-reduce covers)."""
    _check_act(dy, "conv_wgrad.dy")
    _check_act(x, "conv_wgrad.x")
    if _overlap["on"]:
        side = _wgrad_side_stream(x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        _overlap["on"] = False
        try:
            with torch.cuda.stream(side):
                res = conv_wgrad(dy, x, R, S, stride, pad, want_dbias, algo, out, out_db)
        finally:
            _overlap["on"] = True
        # The outputs are kept alive through their STORAGES, not as tensors: a second reference to the tensor
        # makes autograd's AccumulateGrad clone the gradient instead of adopting it as .grad, and that clone runs on
        # the main stream BEFORE the side stream has written it. Round 2 kept the bias gradient as a tensor: inside
        # a captured step the stem's .bias.grad was therefore the PREVIOUS replay's sum (found by the bit-exact
        # graph == eager check of the deterministic mode).
        _overlap["keep"][x.device.index].append((dy, x, res[0].untyped_storage(),
                                                 None if res[1] is None else res[1].untyped_storage()))
        if res[1] is not None and out_db is None:
            # belt and braces for a free-standing bias gradient (only top-level convs have a bias; the stem's wgrad
            # is the last kernel of backward): whatever autograd does with it on the main stream is ordered after
            # the side stream
            torch.cuda.current_stream(x.device).wait_stream(side)
        return res
    N, H, W, C = x.shape
    Nd, P, Q, K = dy.shape
    assert Nd == N and _out_hw(H, W, R, S, stride, pad) == (P, Q)
    if out is not None:
        assert out.shape == (K, R, S, C) and out.dtype == torch.float32 and out.is_contiguous()
        dw = out
    else:
        dw = torch.empty((K, R, S, C), dtype=torch.float32, device=x.device)
    db = None
    if want_dbias:
        db = out_db.view(K) if out_db is not None else torch.empty((K,), dtype=torch.float32, device=x.device)
    algo = _algo_flags(algo)
    nws = _lib.load().b200_conv2d_workspace_bytes(_lib.PASS_WGRAD, N, H, W, C, K, R, S, stride, pad, algo)
    ws = _workspace(x.device, nws) if nws else None
    _lib.call("b200_conv2d_wgrad", dy.data_ptr(), x.data_ptr(), dw.data_ptr(), _p(db),
              N, H, W, C, K, R, S, stride, pad, algo, _p(ws), nws, _stream())
    return dw, db


# ---- optional overlap of wgrad with the rest of backward ------------------------------------------
# Weight gradients are not consumed until the optimizer step, so inside `wgrad_overlap(device)` every
# conv_wgrad is enqueued on a side stream (forked from the current stream at its point of issue) and runs
# concurrently with the dgrad / BN-backward chain; `join_wgrad(device)` re-joins the streams. Tensors that
# cross streams are kept alive until the join (no allocator reuse hazard, also under graph capture).
_overlap = {"on": False, "side": {}, "keep": {}}


class wgrad_overlap:
    def __init__(self, device: torch.device, enabled: bool = True):
        self.device, self.enabled = device, enabled

    def __enter__(self):
        self.prev = _overlap["on"]
        _overlap["on"] = self.enabled
        return self

    def __exit__(self, *exc):
        _overlap["on"] = self.prev
        join_wgrad(self.device)
        return False


def join_wgrad(device: torch.device) -> None:
    side = _overlap["side"].get(device.index)
    if side is not None and _overlap["keep"].get(device.index):
        torch.cuda.current_stream(device).wait_stream(side)
        _overlap["keep"][device.index] = []


def wgrad_side_stream_if_any(device: torch.device):
    """The wgrad side stream if it holds kernels that have not been joined yet (else None): what a
    consumer of weight gradients must wait for in addition to the current stream."""
    side = _overlap["side"].get(device.index)
    return side if (side is not None and _overlap["keep"].get(device.index)) else None


def _wgrad_side_stream(device: torch.device):
    side = _overlap["side"].get(device.index)
    if side is None:
        side = torch.cuda.Stream(device=device)
        _overlap["side"][device.index] = side
        _overlap["keep"][device.index] = []
    return side


def conv_tc_supported(pass_: int, N, H, W, C, K, R, S, stride, pad) -> bool:
    return bool(_lib.load().b200_conv2d_tc_supported(pass_, N, H, W, C, K, R, S, stride, pad))


# --------------------------------------------------------------------------------------------------
# batch norm / activation / dropout / skip
# --------------------------------------------------------------------------------------------------
def bn_batch_stats(x, eps: float, momentum: float = 0.1, running_mean=None, running_var=None,
                   num_batches_tracked=None):
    """Batch statistics of an [..., C] bf16 tensor -> (mean, invstd, deferred).
    deferred = False: one reduction launch computed them and updated the running statistics in place.
    deferred = True : the conv that produced x already computed them (conv_fprop(want_stats=True)); nothing
    was launched and the running statistics have NOT been updated: pass them to bn_act_fwd(running=...)."""
    _check_act(x, "bn_stats.x")
    C = x.shape[-1]
    rows = x.numel() // C
    rec = _pending_stats.pop(_accum_key(x.device), None)
    if rec is not None and rec[:4] == (x.data_ptr(), rows, C, float(eps)):
        return rec[4], rec[5], True
    mean = torch.empty((C,), dtype=torch.float32, device=x.device)
    invstd = torch.empty((C,), dtype=torch.float32, device=x.device)
    nws = _lib.load().b200_bn_workspace_bytes(rows, C)
    ws = bn_accumulators(x.device, nws)
    _lib.call("b200_bn_stats", x.data_ptr(), rows, C, eps, momentum, mean.data_ptr(), invstd.data_ptr(),
              _p(running_mean), _p(running_var), _p(num_batches_tracked), ws.data_ptr(), nws, _stream())
    return mean, invstd, False


def bn_stats(x, eps: float, momentum: float = 0.1, running_mean=None, running_var=None,
             num_batches_tracked=None):
    """Batch statistics of an [..., C] bf16 tensor -> (mean, invstd); updates running stats in place."""
    mean, invstd, deferred = bn_batch_stats(x, eps, momentum, running_mean, running_var, num_batches_tracked)
    if deferred and running_mean is not None:
        C = x.shape[-1]
        _lib.call("b200_bn_running_update", mean.data_ptr(), invstd.data_ptr(), x.numel() // C, C, eps, momentum,
                  running_mean.data_ptr(), running_var.data_ptr(), _p(num_batches_tracked), _stream())
    return mean, invstd


def bn_act_fwd(x, mean=None, invstd=None, gamma=None, beta=None, *, stat_is_var: bool = False,
               eps: float = 1e-5, skip=None, skip_mode: int = _lib.SKIP_NONE, relu: bool = True,
               dropout_p: float = 0.0, seed: int = 0, running=None, want_mask: bool = False):
    """running: optional (running_mean, running_var, num_batches_tracked, momentum) updated from mean / invstd
    by the same launch (statistics that came out of a conv kernel: bn_batch_stats(...)[2] is True).
    want_mask: also return the ReLU/dropout bit mask (uint8 [N,H,W,C/8]) for bn_act_bwd -> (y, mask).
    fp32 x: the forward-only fp32 kernel of the fp32 / TF32 mode (no dropout, no mask)."""
    if x.dtype == torch.float32:
        if dropout_p > 0 or want_mask or running is not None:
            raise _lib.B200Error("bn_act_fwd: the fp32 / TF32 mode is forward-only (evaluation)")
        _check_f32(x, "bn_act_fwd.x")
        N, H, W, C = x.shape
        y = torch.empty_like(x)
        skip_C = 0
        if skip is not None:
            _check_f32(skip, "bn_act_fwd.skip")
            skip_C = skip.shape[-1]
        _lib.call("b200_bn_act_fwd_f32", x.data_ptr(), y.data_ptr(), N, H, W, C, _p(mean), _p(invstd),
                  int(stat_is_var), eps, _p(gamma), _p(beta), _p(skip), skip_mode if skip is not None else 0, skip_C,
                  int(relu), _stream())
        return y
    _check_act(x, "bn_act_fwd.x")
    N, H, W, C = x.shape
    y = torch.empty_like(x)
    mask = torch.empty((N, H, W, C // 8), dtype=torch.uint8, device=x.device) if want_mask else None
    rm, rv, nbt, mom = running if running is not None else (None, None, None, 0.0)
    skip_C = 0
    if skip is not None:
        _check_act(skip, "bn_act_fwd.skip")
        skip_C = skip.shape[-1]
        if skip_mode == _lib.SKIP_SAME:
            assert skip.shape == x.shape
        else:
            assert skip.shape[0] == N and skip.shape[1] == 2 * H and skip.shape[2] == 2 * W
    _lib.call("b200_bn_act_fwd", x.data_ptr(), y.data_ptr(), N, H, W, C, _p(mean), _p(invstd),
              int(stat_is_var), eps, _p(gamma), _p(beta), _p(skip), skip_mode if skip is not None else 0,
              skip_C, int(relu), float(dropout_p), int(seed) & 0xFFFFFFFFFFFFFFFF,
              step_counter(x.device).data_ptr() if dropout_p > 0 else None, _p(rm), _p(rv), _p(nbt), float(mom),
              _p(mask), _stream())
    return (y, mask) if want_mask else y


def bn_act_bwd(dy, y, x, mean=None, invstd=None, gamma=None, *, relu: bool = True,
               dropout_p: float = 0.0, seed: int = 0, addend=None, want_dskip: bool = False,
               out_dgamma=None, out_dbeta=None, mask=None, reduced=None):
    """Returns (dx, dgamma, dbeta, dskip). out_dgamma / out_dbeta: optional fp32 [C] destinations.
    mask: the uint8 bit mask of bn_act_fwd(want_mask=True); with it y may be None.
    reduced: (dgamma, dbeta) already produced by conv_dgrad_bn_bwd -> only the apply pass runs."""
    _check_act(dy, "bn_act_bwd.dy")
    C = dy.shape[-1]
    rows = dy.numel() // C
    dx = torch.empty_like(dy)
    dskip = torch.empty_like(dy) if want_dskip else None
    affine = gamma is not None
    if reduced is not None:
        assert affine and mask is not None and x is not None
        dgamma, dbeta = reduced
        if addend is not None:
            _check_act(addend, "bn_act_bwd.addend")
            assert addend.shape == dy.shape
        _lib.call("b200_bn_act_bwd_apply", dy.data_ptr(), mask.data_ptr(), x.data_ptr(), dx.data_ptr(), _p(dskip),
                  _p(addend), rows, C, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), dgamma.data_ptr(),
                  dbeta.data_ptr(), int(relu), float(dropout_p), _stream())
        return dx, dgamma, dbeta, dskip
    dgamma = dbeta = None
    if affine:
        dgamma = out_dgamma.view(C) if out_dgamma is not None else torch.empty((C,), dtype=torch.float32, device=dy.device)
        dbeta = out_dbeta.view(C) if out_dbeta is not None else torch.empty((C,), dtype=torch.float32, device=dy.device)
    nws = _lib.load().b200_bn_workspace_bytes(rows, C) if affine else 0
    if affine:
        _drop_pending_stats(dy.device)
    ws = bn_accumulators(dy.device, nws) if affine else None
    if addend is not None:
        _check_act(addend, "bn_act_bwd.addend")
        assert addend.shape == dy.shape
    if mask is not None:
        assert mask.dtype == torch.uint8 and mask.is_contiguous() and mask.numel() * 8 == dy.numel()
    _lib.call("b200_bn_act_bwd", dy.data_ptr(), _p(y), _p(mask), _p(x), dx.data_ptr(), _p(dskip), _p(addend), rows,
              C, _p(mean), _p(invstd), _p(gamma), _p(dgamma), _p(dbeta), int(relu), float(dropout_p),
              int(seed) & 0xFFFFFFFFFFFFFFFF,
              step_counter(dy.device).data_ptr() if dropout_p > 0 else None, _p(ws), nws, _stream())
    return dx, dgamma, dbeta, dskip


def subsample2(x):
    N, H2, W2, C = x.shape
    assert H2 % 2 == 0 and W2 % 2 == 0
    if x.dtype == torch.float32:
        _check_f32(x, "subsample2.x")
        y = torch.empty((N, H2 // 2, W2 // 2, C), dtype=torch.float32, device=x.device)
        _lib.call("b200_subsample2_f32", x.data_ptr(), y.data_ptr(), N, H2 // 2, W2 // 2, C, _stream())
        return y
    _check_act(x, "subsample2.x")
    y = torch.empty((N, H2 // 2, W2 // 2, C), dtype=torch.bfloat16, device=x.device)
    _lib.call("b200_subsample2", x.data_ptr(), y.data_ptr(), N, H2 // 2, W2 // 2, C, _stream())
    return y


def upsample_add_(dx, g, Cg: Optional[int] = None):
    """dx[n, 2h, 2w, :Cg] += g[n, h, w, :Cg] in place (Cg defaults to all channels of g)."""
    _check_act(dx, "upsample_add.dx")
    _check_act(g, "upsample_add.g")
    N, H, W, ldg = g.shape
    Cg = ldg if Cg is None else Cg
    assert dx.shape[0] == N and dx.shape[1] == 2 * H and dx.shape[2] == 2 * W and dx.shape[3] >= Cg
    _lib.call("b200_upsample_add", dx.data_ptr(), g.data_ptr(), N, H, W, dx.shape[3], Cg, ldg, _stream())
    return dx


# --------------------------------------------------------------------------------------------------
# pooling
# --------------------------------------------------------------------------------------------------
def _pool(name, x, k, stride, pad, want_argmax: bool = False):
    N, H, W, C = x.shape
    P, Q = _out_hw(H, W, k, k, stride, pad)
    if x.dtype == torch.float32:
        _check_f32(x, name)
        y = torch.empty((N, P, Q, C), dtype=torch.float32, device=x.device)
        _lib.call("b200_pool_fwd_f32", x.data_ptr(), y.data_ptr(), N, H, W, C, k, stride, pad,
                  int(name == "b200_maxpool_fwd"), _stream())
        return y
    _check_act(x, name)
    y = torch.empty((N, P, Q, C), dtype=torch.bfloat16, device=x.device)
    if name == "b200_maxpool_fwd":
        am = torch.empty((N, P, Q, C), dtype=torch.uint8, device=x.device) if want_argmax else None
        _lib.call(name, x.data_ptr(), y.data_ptr(), _p(am), N, H, W, C, k, stride, pad, _stream())
        return (y, am) if want_argmax else y
    _lib.call(name, x.data_ptr(), y.data_ptr(), N, H, W, C, k, stride, pad, _stream())
    return y


def avgpool_fwd(x, k, stride, pad):
    return _pool("b200_avgpool_fwd", x, k, stride, pad)


def maxpool_fwd(x, k, stride, pad, want_argmax: bool = False):
    """want_argmax: also return the uint8 argmax positions that maxpool_bwd consumes -> (y, argmax)."""
    return _pool("b200_maxpool_fwd", x, k, stride, pad, want_argmax)


def avgpool_bwd(dy, in_shape, k, stride, pad):
    _check_act(dy, "avgpool_bwd.dy")
    N, H, W, C = in_shape
    dx = torch.empty(in_shape, dtype=torch.bfloat16, device=dy.device)
    _lib.call("b200_avgpool_bwd", dy.data_ptr(), dx.data_ptr(), N, H, W, C, k, stride, pad, _stream())
    return dx


def maxpool_bwd(dy, argmax, in_shape, k, stride, pad):
    _check_act(dy, "maxpool_bwd.dy")
    N, H, W, C = in_shape
    assert argmax.dtype == torch.uint8 and argmax.shape == dy.shape and argmax.is_contiguous()
    dx = torch.empty(in_shape, dtype=torch.bfloat16, device=dy.device)
    _lib.call("b200_maxpool_bwd", dy.data_ptr(), argmax.data_ptr(), dx.data_ptr(), N, H, W, C, k, stride, pad,
              _stream())
    return dx


# --------------------------------------------------------------------------------------------------
# head
# --------------------------------------------------------------------------------------------------
def linear_fwd(x, w, b):
    B, I = x.shape
    O = w.shape[0]
    if x.dtype == torch.float32:
        _check_f32(x, "linear_fwd.x")
        y = torch.empty((B, O), dtype=torch.float32, device=x.device)
        _lib.call("b200_linear_fwd_f32", x.data_ptr(), w.data_ptr(), _p(b), y.data_ptr(), B, I, O, _stream())
        return y
    _check_act(x, "linear_fwd.x")
    y = torch.empty((B, O), dtype=torch.bfloat16, device=x.device)
    _lib.call("b200_linear_fwd", x.data_ptr(), w.data_ptr(), _p(b), y.data_ptr(), B, I, O, _stream())
    return y


def linear_bwd(dy, x, w, want_dx=True, out_dw=None, out_db=None):
    _check_act(dy, "linear_bwd.dy")
    B, O = dy.shape
    I = x.shape[1]
    dx = torch.empty((B, I), dtype=torch.bfloat16, device=dy.device) if want_dx else None
    dw = out_dw.view(O, I) if out_dw is not None else torch.empty((O, I), dtype=torch.float32, device=dy.device)
    db = out_db.view(O) if out_db is not None else torch.empty((O,), dtype=torch.float32, device=dy.device)
    _lib.call("b200_linear_bwd", dy.data_ptr(), x.data_ptr(), w.data_ptr(), _p(dx), dw.data_ptr(),
              db.data_ptr(), B, I, O, _stream())
    return dx, dw, db


def ce_topk(logits, labels, want_metrics=True, want_dlogits=False, grad_scale=None):
    """(out fp32[3] = loss, top1_err, top5_err | None, dlogits bf16 | None)."""
    if logits.dtype == torch.float32:
        if want_dlogits:
            raise _lib.B200Error("ce_topk: the fp32 / TF32 mode is forward-only (evaluation)")
        _check_f32(logits, "ce_topk.logits")
        B, O = logits.shape
        out = torch.empty((3,), dtype=torch.float32, device=logits.device)
        _lib.call("b200_ce_topk_f32", logits.data_ptr(), labels.data_ptr(), out.data_ptr(), B, O, _stream())
        return out, None
    _check_act(logits, "ce_topk.logits")
    assert labels.dtype == torch.int64 and labels.is_cuda and labels.is_contiguous()
    B, O = logits.shape
    out = torch.empty((3,), dtype=torch.float32, device=logits.device) if want_metrics else None
    dl = torch.empty_like(logits) if want_dlogits else None
    _lib.call("b200_ce_topk", logits.data_ptr(), labels.data_ptr(), _p(out), _p(dl), _p(grad_scale), B, O,
              _stream())
    return out, dl


# --------------------------------------------------------------------------------------------------
# optimizer
# --------------------------------------------------------------------------------------------------
def sgd_step(ptr_table: torch.Tensor, n: int, max_size: int, lr, momentum, dampening, weight_decay,
             nesterov, first_step, inv_scale=None, found_inf=None, lr_dev=None):
    """ptr_table: int64 CUDA tensor [4, n] = rows of param ptrs, grad ptrs, buf ptrs, sizes."""
    assert ptr_table.dtype == torch.int64 and ptr_table.is_cuda and ptr_table.shape == (4, n)
    _lib.require_device(ptr_table.device.index or 0)
    base = ptr_table.data_ptr()
    row = n * 8
    _lib.call("b200_sgd_step", base, base + row, base + 2 * row, base + 3 * row, n, max_size, float(lr),
              float(momentum), float(dampening), float(weight_decay), int(bool(nesterov)),
              int(bool(first_step)), _p(inv_scale), _p(found_inf), _p(lr_dev), _stream())


_adam_tickets = {}


def adam_tickets(device: torch.device, n: int = 0) -> torch.Tensor:
    """Zero-filled uint32 ticket counters of b200_adam_step (zero on entry, zero again on exit), at least n of
    them. Keyed like bn_accumulators: one buffer per (device, stream), and one that every capturing stream of
    the device shares, created together with the first eager buffer so that no fill kernel is recorded into a
    graph. A capture cannot allocate it: step the optimizer once eagerly before capturing."""
    capturing = torch.cuda.is_current_stream_capturing()
    key = (device.index, "capture" if capturing else _stream())
    t = _adam_tickets.get(key)
    if t is None or t.numel() < n:
        if capturing:
            raise _lib.B200Error("adam_step: ticket counters must be allocated before CUDA-graph capture "
                                 "(step the optimizer once eagerly first)")
        t = torch.zeros(max(1024, n), dtype=torch.int32, device=device)
        _adam_tickets[key] = t
        cap = _adam_tickets.get((device.index, "capture"))
        if cap is None or cap.numel() < n:
            _adam_tickets[(device.index, "capture")] = torch.zeros_like(t)
    return t


def adam_step(ptr_table: torch.Tensor, n: int, max_size: int, lr, beta1, beta2, eps, weight_decay, decoupled,
              amsgrad, inv_scale=None, found_inf=None, lr_dev=None):
    """ptr_table: int64 CUDA tensor [7, n] = rows of param, grad, exp_avg, exp_avg_sq, max_exp_avg_sq (unused
    without amsgrad) and step pointers, then sizes. One launch; it advances every step counter by one."""
    assert ptr_table.dtype == torch.int64 and ptr_table.is_cuda and ptr_table.shape == (7, n)
    _lib.require_device(ptr_table.device.index or 0)
    tickets = adam_tickets(ptr_table.device, n)
    base = ptr_table.data_ptr()
    row = n * 8
    _lib.call("b200_adam_step", *(base + r * row for r in range(7)), n, max_size, float(lr), float(beta1),
              float(beta2), float(eps), float(weight_decay), int(bool(decoupled)), int(bool(amsgrad)),
              _p(inv_scale), _p(found_inf), _p(lr_dev), tickets.data_ptr(), _stream())


# --------------------------------------------------------------------------------------------------
# input pipeline
# --------------------------------------------------------------------------------------------------
def augment_batch(data_u8, index, *, flip=None, top=None, left=None, mean=None, stddev=None, pad: int = 0,
                  pad_mirror: bool = False, out_hw=None, to_tensor: bool = True, want_f32: bool = False,
                  want_bf16: bool = True):
    """One launch: out[b] = crop(pad(flip(whiten(to_tensor(data_u8[index[b]]))))) (b200_augment_batch).
    data_u8: uint8 [M,H,W,C] on the device; index int64 [B]; flip uint8 [B]; top/left int32 [B]; mean/stddev
    fp32 [C,H,W]. Returns (fp32 [B,C,OH,OW] or None, bf16 [B,OH,OW,C] or None)."""
    if not (data_u8.is_cuda and data_u8.dtype == torch.uint8 and data_u8.is_contiguous() and data_u8.dim() == 4):
        raise _lib.B200Error("augment_batch: expected a contiguous CUDA uint8 [M,H,W,C] dataset")
    if data_u8.device.index != torch.cuda.current_device():
        raise _lib.B200Error("augment_batch: the dataset lives on another device than the current one")
    _lib.require_device(data_u8.device.index or 0)
    M, H, W, C = data_u8.shape
    B = index.numel()
    assert index.dtype == torch.int64 and index.is_cuda and index.is_contiguous()
    OH, OW = out_hw if out_hw is not None else (H + 2 * pad, W + 2 * pad)
    for t, dt in ((flip, torch.uint8), (top, torch.int32), (left, torch.int32)):
        assert t is None or (t.dtype == dt and t.is_cuda and t.is_contiguous() and t.numel() == B)
    for t in (mean, stddev):
        assert t is None or (t.dtype == torch.float32 and t.is_cuda and t.is_contiguous() and t.numel() == C * H * W)
    of = torch.empty((B, C, OH, OW), dtype=torch.float32, device=data_u8.device) if want_f32 else None
    ob = torch.empty((B, OH, OW, C), dtype=torch.bfloat16, device=data_u8.device) if want_bf16 else None
    _lib.call("b200_augment_batch", data_u8.data_ptr(), index.data_ptr(), _p(flip), _p(top), _p(left), _p(mean),
              _p(stddev), B, H, W, C, int(pad), int(bool(pad_mirror)), OH, OW, int(bool(to_tensor)), _p(of), _p(ob),
              _stream())
    return of, ob


# --------------------------------------------------------------------------------------------------
# fp32 / TF32 precision mode (the reference's un-autocast path: evaluation.py:32-39, training.py:101-102)
# --------------------------------------------------------------------------------------------------
def _check_f32(t: torch.Tensor, name: str) -> None:
    if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise _lib.B200Error(f"{name}: expected a contiguous CUDA fp32 tensor, got {t.dtype} {t.device}")
    if t.device.index != torch.cuda.current_device():
        raise _lib.B200Error(f"{name}: tensor lives on {t.device}, not on the current CUDA device")
    _lib.require_device(t.device.index or 0)


def conv_tf32_supported(pass_: int, N, H, W, C, K, R, S, stride, pad) -> bool:
    return bool(_lib.load().b200_conv2d_tf32_supported(pass_, N, H, W, C, K, R, S, stride, pad))


def conv_fprop_tf32(x, w_krsc, stride: int, pad: int, bias=None, residual=None, relu: bool = False):
    """fp32 NHWC x, fp32 KRSC filter -> fp32 NHWC y through tcgen05 kind::tf32 MMAs."""
    _check_f32(x, "conv_fprop_tf32.x")
    _check_f32(w_krsc, "conv_fprop_tf32.w")
    N, H, W, C = x.shape
    K, R, S, Cw = w_krsc.shape
    assert Cw == C
    P, Q = _out_hw(H, W, R, S, stride, pad)
    y = torch.empty((N, P, Q, K), dtype=torch.float32, device=x.device)
    if residual is not None:
        _check_f32(residual, "conv_fprop_tf32.residual")
        assert residual.shape == y.shape
    nws = _lib.load().b200_conv2d_tf32_workspace_bytes(N, H, W, C, K, R, S, stride, pad)
    ws = _workspace(x.device, nws) if nws else None
    _lib.call("b200_conv2d_fprop_tf32", x.data_ptr(), w_krsc.data_ptr(), _p(bias), _p(residual), y.data_ptr(),
              N, H, W, C, K, R, S, stride, pad, int(relu), _p(ws), nws, _stream())
    return y


def nchw_f32_to_nhwc_f32(x: torch.Tensor) -> torch.Tensor:
    _check_f32(x, "nchw_f32_to_nhwc_f32.x")
    N, C, H, W = x.shape
    y = torch.empty((N, H, W, C), dtype=torch.float32, device=x.device)
    _lib.call("b200_nchw_to_nhwc_f32", x.data_ptr(), y.data_ptr(), N, C, H, W, _stream())
    return y


def conv_dgrad_tf32(dy, w_crsk, in_hw, stride: int, pad: int, addend=None):
    _check_f32(dy, "conv_dgrad_tf32.dy")
    _check_f32(w_crsk, "conv_dgrad_tf32.w")
    N, P, Q, K = dy.shape
    C, R, S, Kw = w_crsk.shape
    assert Kw == K
    H, W = in_hw
    assert _out_hw(H, W, R, S, stride, pad) == (P, Q)
    dx = torch.empty((N, H, W, C), dtype=torch.float32, device=dy.device)
    if addend is not None:
        _check_f32(addend, "conv_dgrad_tf32.addend")
        assert addend.shape == dx.shape
    _lib.call("b200_conv2d_dgrad_tf32", dy.data_ptr(), w_crsk.data_ptr(), _p(addend), dx.data_ptr(), N, H, W, C, K,
              R, S, stride, pad, _stream())
    return dx


def conv_wgrad_tf32(dy, x, R: int, S: int, stride: int, pad: int):
    _check_f32(dy, "conv_wgrad_tf32.dy")
    _check_f32(x, "conv_wgrad_tf32.x")
    N, H, W, C = x.shape
    K = dy.shape[-1]
    dw = torch.empty((K, R, S, C), dtype=torch.float32, device=x.device)
    _lib.call("b200_conv2d_wgrad_tf32", dy.data_ptr(), x.data_ptr(), dw.data_ptr(), N, H, W, C, K, R, S, stride,
              pad, _stream())
    return dw
