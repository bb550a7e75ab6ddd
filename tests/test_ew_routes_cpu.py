"""
Without a GPU: (1) every kernel instantiation that api.cu launches outside the convolution, optimizer and input
pipeline entry points is in the hand-written list of tests/test_ew_routes_gpu.py (so a new instantiation without a
route row fails here already); (2) the numpy port of the dropout RNG (tests/kernel_check.py) draws exactly what
rng_draw4 / effective_seed of csrc/common.cuh draw, compiled by nvcc for the host.
"""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from tests.kernel_check import effective_seed, normalize_kernel_name, rng_draw4

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pytorch_ddp_resnet_b200", "csrc")

# entry points whose launches the conv route table (test_conv_routes_gpu.py), the optimizer tests and the
# augmentation oracle test own
OTHER_OWNERS = re.compile(r"conv|wgrad|im2col|sgd|adam|augment")

_FUNC = re.compile(r'^(?:extern "C" |static )[\w:<>\s\*]*?\b(\w+)\s*\(', re.M)
_LAUNCH = re.compile(r"launch_k\(\s*([A-Za-z_]\w*(?:<[^>]*>)?)\s*,")
_MACRO = re.compile(r"#define\s+(\w+)\(([^)]*)\)\s+launch_k\(\s*(\w+)<([^>]*)>")


def launched_outside_conv(src):
    """{normalised kernel name: enclosing function} of every launch_k in api.cu outside the other owners' entry
    points; launches written through a #define (the maxpool K / S variants) are expanded at each use."""
    heads = [(m.start(), m.group(1)) for m in _FUNC.finditer(src)]

    def owner(pos):
        name = None
        for start, fn in heads:
            if start > pos:
                break
            name = fn
        return name

    found = {}
    for m in _LAUNCH.finditer(src):
        fn = owner(m.start())
        if fn is None or OTHER_OWNERS.search(fn):
            continue
        line_start = src.rfind("\n", 0, m.start()) + 1
        if src[line_start:m.start()].lstrip().startswith("#define"):
            continue
        found[normalize_kernel_name(m.group(1))] = fn
    for m in _MACRO.finditer(src):
        macro, params, kernel, targs = m.group(1), [p.strip() for p in m.group(2).split(",")], m.group(3), m.group(4)
        fn = owner(m.start())
        if OTHER_OWNERS.search(fn):
            continue
        for use in re.finditer(rf"\b{macro}\(([^)]*)\)", src[m.end():]):
            vals = [v.strip() for v in use.group(1).split(",")]
            if len(vals) != len(params):
                continue
            args = targs
            for p, v in zip(params, vals):
                args = re.sub(rf"\b{p}\b", v, args)
            found[normalize_kernel_name(f"{kernel}<{args}>")] = fn
    return found


def test_every_launched_kernel_is_listed():
    from tests.test_ew_routes_gpu import EW_REACHABLE
    with open(os.path.join(CSRC, "api.cu")) as f:
        found = launched_outside_conv(f.read())
    # the parser itself: the routes this file exists for must be seen
    for k in ("bn_act_fwd_kernel<2,3,1,2>", "bn_act_bwd_apply_kernel<1,1,1>", "maxpool_fwd_ks_kernel<3,2>",
              "maxpool_bwd_ks_kernel<2,2>", "pool_fwd_f32_kernel<1>", "ce_topk_f32_kernel"):
        assert k in found, f"parser missed {k}: {sorted(found)}"
    missing = sorted(k for k in found if k not in EW_REACHABLE)
    assert not missing, ("kernels launched by api.cu without an entry in EW_REACHABLE (and so without a route "
                         f"row): {[(k, found[k]) for k in missing]}")
    stale = sorted(k for k in EW_REACHABLE if k not in found)
    assert not stale, f"EW_REACHABLE lists kernels api.cu no longer launches: {stale}"


_HOST_PROGRAM = r"""
#include <cstdio>
#include "common.cuh"
int main() {
  const unsigned long long seeds[] = {0ull, 5ull, 0x0123456789abcdefull, 0xffffffffffffffffull};
  const unsigned long long offsets[] = {0ull, 1ull, 7ull, 0x8000000000000001ull};
  for (unsigned long long s : seeds)
    for (unsigned long long o : offsets) {
      // effective_seed is device-only (it reads the counter through a device pointer): the host formula here is
      // the one it evaluates
      const unsigned long long e = s + o * 0x9E3779B97F4A7C15ull;
      for (unsigned long long i = 0; i < 200; ++i) {
        const unsigned long long idx = (i < 100) ? i : (i * 0x9E3779B1ull) ^ (i << 33);
        const uint2 d = b200::rng_draw4(e, idx);
        printf("%llu %llu %llu %llu %u %u\n", s, o, e, idx, d.x, d.y);
      }
    }
  return 0;
}
"""


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def test_numpy_rng_port_matches_common_cuh(tmp_path):
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    src = tmp_path / "rng.cu"
    src.write_text(_HOST_PROGRAM)
    exe = tmp_path / "rng"
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I", CSRC, "-o", str(exe),
                    str(src)], check=True, capture_output=True, timeout=600)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True, timeout=60).stdout
    rows = np.array([[int(v) for v in line.split()] for line in out.splitlines()], dtype=object)
    assert len(rows) == 4 * 4 * 200
    for s, o, e, idx, x, y in rows:
        assert effective_seed(s, o) == e, (s, o)
    # per (seed, offset): the vectorised port over all counters of that pair
    for k in range(0, len(rows), 200):
        e = int(rows[k][2])
        idx = np.array([int(v) for v in rows[k:k + 200, 3]], dtype=np.uint64)
        px, py = rng_draw4(e, idx)
        want_x = np.array([int(v) for v in rows[k:k + 200, 4]], dtype=np.uint32)
        want_y = np.array([int(v) for v in rows[k:k + 200, 5]], dtype=np.uint32)
        bad = np.nonzero((px != want_x) | (py != want_y))[0]
        assert bad.size == 0, f"seed {e:#x}: draw {int(idx[bad[0]])} differs: {px[bad[0]]}, {py[bad[0]]} != " \
                              f"{want_x[bad[0]]}, {want_y[bad[0]]}"
