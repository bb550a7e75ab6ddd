"""
Per-element checks of kernel outputs (a plain module, imported by the kernel tests).

  * assert_elementwise: every element of a kernel output against an fp64 reference, with a bound built from the
    rounding points of the output type and the magnitude of the operation (the same op on |operands|);
  * poisoned / check_poisoned: outputs that start as NaN bytes between two guard regions, so that an element the
    kernel never wrote or a write past either end of the output is seen;
  * kernels_launched: the CUDA kernels a call launched (torch.profiler / CUPTI), normalised to
    `name<args>` so that a test can assert which route of the dispatcher ran.
"""
import re

import torch

POISON_BYTE = 0xFF   # 0xFFFF is a NaN in bf16, 0xFFFFFFFF a NaN in fp32
# Unit roundoff of bf16 (8 significant bits): one round-to-nearest moves a value by at most 2^-8 of itself. An
# output with k rounding points (conv result, then the residual / addend sum: k = 2) gets rounding = k * 2^-8
# against |ref| + sum |addends|, which bounds every value that was rounded.
BF16_ROUNDING = 2.0 ** -8


def _coords(idx, shape):
    out = []
    for s in reversed(shape):
        out.append(idx % s)
        idx //= s
    return tuple(reversed(out))


def _names(ndim):
    return "(n, h, w, c)" if ndim == 4 else "index"


def assert_elementwise(out, ref64, mag64, rounding, acc=2.0 ** -14, addends=(), scale64=None, label=""):
    """|out - ref| <= rounding * (|ref| + sum |addend|) + acc * mag at every element.

    ref64: the fp64 reference; mag64: the same operation applied to |operands| in fp64 (bounds the accumulation
    error of any summation order); rounding: BF16_ROUNDING per bf16 rounding point of the output, 0 for fp32
    outputs; addends: tensors added after the accumulation (residual, bias), whose size also scales the rounding of
    the sum; scale64: replaces |ref| in the rounding term (the value before an epilogue ReLU, which a rounding moves).

    Prints, and returns, the worst ratio of the error to the whole bound and the worst ratio of what the rounding
    term leaves over to the accumulation term acc * mag (the margin of `acc`). A correctly rounded bf16 output may
    use its rounding term in full, so the first ratio of a bf16 output approaches 1 by construction. Fails with the
    worst element's coordinates."""
    o = out.detach().to(torch.float64)
    ref = ref64.detach().to(torch.float64)
    assert o.shape == ref.shape, f"{label}: shape {tuple(o.shape)} != reference {tuple(ref.shape)}"
    acc_term = acc * mag64.detach().to(torch.float64).abs()
    round_term = torch.zeros_like(ref)
    if rounding:
        scale = ref.abs() if scale64 is None else scale64.detach().to(torch.float64).abs()
        for a in addends:
            scale = scale + a.detach().to(torch.float64).abs()
        round_term = rounding * scale
    bound = acc_term + round_term
    err = (o - ref).abs()
    nan = torch.isnan(o)
    ratio = torch.where(nan, torch.full_like(err, float("inf")), err / bound.clamp_min(1e-300))
    acc_ratio = (err - round_term).clamp_min(0) / acc_term.clamp_min(1e-300)
    acc_ratio = torch.where(nan, torch.full_like(err, float("inf")), acc_ratio)
    flat = ratio.reshape(-1)
    i = int(torch.argmax(flat).item())
    worst = float(flat[i].item())
    worst_acc = float(acc_ratio.max().item())
    where = _coords(i, tuple(o.shape))
    print(f"[kernel_check] {label}: worst ratio to bound {worst:.4f} at {_names(o.dim())} = {where}; "
          f"accumulation term {worst_acc:.4f}")
    if not worst <= 1.0:
        nbad = int((flat > 1.0).sum().item()) if worst != float("inf") else int((~(flat <= 1.0)).sum().item())
        raise AssertionError(
            f"{label}: {nbad} of {flat.numel()} elements outside the bound; worst at {_names(o.dim())} = {where}: "
            f"out {o.reshape(-1)[i].item()!r}, ref {ref.reshape(-1)[i].item()!r}, bound "
            f"{bound.reshape(-1)[i].item():.3e}, ratio {worst:.3g}")
    return worst, worst_acc


def poisoned(shape, dtype, guard_bytes=4096, device="cuda", byte=POISON_BYTE):
    """A tensor of `shape` whose bytes are all 0xFF (NaN), inside a buffer with `guard_bytes` of 0xFF before and
    after it. The view starts 1024-byte aligned (TMA boxes need 16 B, the epilogues' 256-bit stores 32 B).
    byte: another fill for integer outputs, which have no NaN (run them with 0x00 and with 0xFF)."""
    esize = torch.empty((), dtype=dtype).element_size()
    nbytes = esize
    for s in shape:
        nbytes *= s
    buf = torch.full((guard_bytes + nbytes + guard_bytes + 1024,), byte, dtype=torch.uint8, device=device)
    lo = guard_bytes + (-(buf.data_ptr() + guard_bytes)) % 1024
    view = buf[lo:lo + nbytes].view(dtype).view(shape)
    assert view.data_ptr() % 1024 == 0
    view._poison = (buf, lo, lo + nbytes, guard_bytes)
    view._poison_byte = byte
    return view


def check_poisoned(view, label=""):
    """After a call: both guards of a poisoned() tensor still hold their fill bit for bit, and the view holds no NaN
    (every element was written; an integer view cannot show that: compare it exactly under both fills)."""
    buf, lo, hi, guard = view._poison
    byte = getattr(view, "_poison_byte", POISON_BYTE)
    before = buf[lo - guard:lo]
    after = buf[hi:hi + guard]
    for name, g in (("before", before), ("after", after)):
        bad = (g != byte).nonzero()
        if bad.numel():
            first = int(bad[0].item())
            off = first - guard if name == "before" else first
            raise AssertionError(f"{label}: {bad.numel()} guard bytes {name} the output were overwritten "
                                 f"(first at byte offset {off} {'before the start' if name == 'before' else 'past the end'})")
    nan = torch.isnan(view)
    if bool(nan.any()):
        n = int(nan.sum().item())
        i = int(nan.reshape(-1).nonzero()[0].item())
        raise AssertionError(f"{label}: {n} of {view.numel()} output elements were never written; first at "
                             f"{_names(view.dim())} = {_coords(i, tuple(view.shape))}")


# template arity of the project's kernels whose last template parameter has a default (TF32 = false / TAIL32 =
# false): the demangled name may or may not spell the default out
_TEMPLATE_ARITY = {"conv_tc2h_kernel": 4, "conv_tc2_kernel": 3, "wgrad_tc_kernel": 4}


def normalize_kernel_name(raw):
    """'void b200::conv_tc2_kernel<64, 1, false>(CUtensorMap, ...)' -> 'conv_tc2_kernel<64,1,0>'."""
    s = raw.strip()
    if s.startswith("void "):
        s = s[5:]
    s = s.replace("b200::", "")
    lt = s.find("<")
    par = s.find("(")
    if lt < 0 or (0 <= par < lt):
        return s[:par] if par >= 0 else s
    depth, end = 0, lt
    for i in range(lt, len(s)):
        if s[i] == "<":
            depth += 1
        elif s[i] == ">":
            depth -= 1
            if depth == 0:
                end = i
                break
    base = s[:lt]
    args = [a.strip() for a in s[lt + 1:end].split(",")]
    norm = []
    for a in args:
        a = re.sub(r"^\((?:bool|int)\)", "", a)
        a = {"true": "1", "false": "0", "__nv_bfloat16": "bf16"}.get(a, a)
        norm.append(a)
    while len(norm) < _TEMPLATE_ARITY.get(base, 0):
        norm.append("0")
    return f"{base}<{','.join(norm)}>"


def kernels_launched(fn):
    """Runs fn() under torch.profiler with CUDA activities and returns (result, sorted list of the distinct
    normalised names of the CUDA kernels it launched; memsets and copies are not kernels and are left out)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if e.name.startswith(("Memset", "Memcpy", "[memory]")):
            continue
        names.add(normalize_kernel_name(e.name))
    return res, sorted(names)


# ---------------------------------------------------------------------------------------------------------------
# the dropout RNG of csrc/common.cuh (rng_draw4, effective_seed) in numpy uint64 arithmetic, and the keep mask that
# the element-wise BN kernels derive from it
# ---------------------------------------------------------------------------------------------------------------
_M32 = 0xFFFFFFFF


def rng_draw4(seed, idx):
    """(x, y) uint32 words of rng_draw4(seed, idx) for an array of counters idx."""
    import numpy as np
    idx = np.asarray(idx, dtype=np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    c0 = idx & np.uint64(_M32)
    c1 = (idx >> np.uint64(32)) ^ np.uint64(seed >> 32)
    key = seed & _M32
    for _ in range(4):
        p = c0 * np.uint64(0xD256D193)                   # < 2^64: c0 < 2^32
        c0 = (p >> np.uint64(32)) ^ np.uint64(key) ^ c1
        c1 = p & np.uint64(_M32)
        key = (key + 0x9E3779B9) & _M32
    return c0.astype(np.uint32), c1.astype(np.uint32)


def effective_seed(seed, offset):
    """The seed a launch draws with: the host seed plus the device step counter (None: no counter)."""
    if offset is None:
        return int(seed) & 0xFFFFFFFFFFFFFFFF
    return (int(seed) + (int(offset) & 0xFFFFFFFFFFFFFFFF) * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF


def drop_threshold(p):
    """api.cu drop_threshold of the fp32 probability: an element is dropped when its 16-bit uniform is below it."""
    import numpy as np
    if p <= 0:
        return 0
    return min(65535, int(float(np.float32(p)) * 65536.0 + 0.5))


def dropout_keep(rows, C, p, seed, offset):
    """bool [rows, C]: element (r, c) reads half-word c % 4 of draw 2 * (r * C/8 + c/8) + (c % 8) / 4 and is
    kept when that value is >= drop_threshold(p)."""
    import numpy as np
    r = np.arange(rows, dtype=np.uint64)[:, None]
    c = np.arange(C, dtype=np.uint64)[None, :]
    draw = np.uint64(2) * (r * np.uint64(C // 8) + c // np.uint64(8)) + (c % np.uint64(8)) // np.uint64(4)
    x, y = rng_draw4(effective_seed(seed, offset), draw)
    h = (c % np.uint64(4)).astype(np.uint32)
    word = np.where(h < 2, x, y)
    u = np.where(h % 2 == 0, word & np.uint32(0xFFFF), word >> np.uint32(16))
    return u >= drop_threshold(p)
