"""
ctypes binding of libb200resnet.so (C ABI in include/b200resnet.h).

There is deliberately NO fallback: if the shared library is missing, or the device is not
sm_100, every kernel call raises. The package itself still imports on a CPU-only box so that
host-side logic (spec parsing, state_dict layout, configs) can be tested without a GPU.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_longlong, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200resnet.so")

ALGO_AUTO, ALGO_DIRECT, ALGO_TC = 0, 1, 2
ALGO_DETERMINISTIC = 0x100   # flag or-ed into an algo: fixed-order reductions (B200_ALGO_DETERMINISTIC)
PASS_FPROP, PASS_DGRAD, PASS_WGRAD = 0, 1, 2
SKIP_NONE, SKIP_SAME, SKIP_SUBSAMPLE_PAD = 0, 1, 2

_P = c_void_p
_CONV_DIMS = [c_int] * 9  # N H W C K R S stride pad

# name -> (restype, argtypes); mirrors include/b200resnet.h one to one
SIGNATURES = {
    "b200_version": (c_int, []),
    "b200_last_error": (c_char_p, []),
    "b200_launch_count": (c_longlong, []),
    "b200_device_check": (c_int, []),
    "b200_conv2d_tc_supported": (c_int, [c_int] + _CONV_DIMS),
    "b200_weight_prep": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P]),
    "b200_weight_prep_multi": (c_int, [_P, c_int, _P]),
    "b200_conv2d_workspace_bytes": (c_size_t, [c_int] + _CONV_DIMS + [c_int]),
    "b200_conv2d_fprop": (c_int, [_P, _P, _P, _P, _P] + _CONV_DIMS + [c_int, c_int, _P, c_size_t, _P]),
    "b200_conv2d_fprop_stats": (c_int, [_P, _P, _P, _P, _P] + _CONV_DIMS + [c_int, _P, c_size_t, _P, c_size_t,
                                        c_float, _P, _P, _P]),
    "b200_bn_running_update": (c_int, [_P, _P, c_int64, c_int, c_float, c_float, _P, _P, _P, _P]),
    "b200_bn_stats_finalize": (c_int, [c_int64, c_int, c_float, c_float, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "b200_conv2d_dgrad": (c_int, [_P, _P, _P, _P] + _CONV_DIMS + [c_int, _P, c_size_t, _P]),
    "b200_conv2d_wgrad": (c_int, [_P, _P, _P, _P] + _CONV_DIMS + [c_int, _P, c_size_t, _P]),
    "b200_conv2d_dgrad_bnbwd": (c_int, [_P, _P, _P] + _CONV_DIMS + [c_int, _P, c_size_t, _P, _P, _P, _P, c_float,
                                        _P, _P, _P, c_size_t, _P, _P]),
    "b200_nchw_f32_to_nhwc_bf16": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b200_bn_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "b200_bn_stats": (c_int, [_P, c_int64, c_int, c_float, c_float, _P, _P, _P, _P, _P, _P,
                              c_size_t, _P]),
    "b200_bn_act_fwd": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P, c_int, c_float, _P, _P,
                                _P, c_int, c_int, c_int, c_float, c_uint64, _P, _P, _P, _P, c_float, _P, _P]),
    "b200_bn_act_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int, _P, _P, _P, _P, _P, c_int,
                                c_float, c_uint64, _P, _P, c_size_t, _P]),
    "b200_bn_act_bwd_apply": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int, _P, _P, _P, _P, _P, c_int, c_float,
                                      _P]),
    "b200_subsample2": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b200_upsample_add": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
    "b200_avgpool_fwd": (c_int, [_P, _P] + [c_int] * 7 + [_P]),
    "b200_avgpool_bwd": (c_int, [_P, _P] + [c_int] * 7 + [_P]),
    "b200_maxpool_fwd": (c_int, [_P, _P, _P] + [c_int] * 7 + [_P]),
    "b200_maxpool_bwd": (c_int, [_P, _P, _P] + [c_int] * 7 + [_P]),
    "b200_linear_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "b200_linear_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "b200_ce_topk": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P]),
    "b200_sgd_step": (c_int, [_P, _P, _P, _P, c_int, c_int64, c_float, c_float, c_float, c_float,
                              c_int, c_int, _P, _P, _P, _P]),
    "b200_adam_step": (c_int, [_P] * 7 + [c_int, c_int64] + [c_double] * 5 + [c_int, c_int, _P, _P, _P, _P, _P]),
    "b200_tick": (c_int, [_P, _P]),
    "b200_conv2d_tf32_supported": (c_int, [c_int] + _CONV_DIMS),
    "b200_conv2d_tf32_workspace_bytes": (c_size_t, _CONV_DIMS),
    "b200_conv2d_fprop_tf32": (c_int, [_P, _P, _P, _P, _P] + _CONV_DIMS + [c_int, _P, c_size_t, _P]),
    "b200_nchw_to_nhwc_f32": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b200_bn_act_fwd_f32": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P, c_int, c_float, _P, _P, _P, c_int,
                                    c_int, c_int, _P]),
    "b200_subsample2_f32": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b200_pool_fwd_f32": (c_int, [_P, _P] + [c_int] * 8 + [_P]),
    "b200_linear_fwd_f32": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "b200_ce_topk_f32": (c_int, [_P, _P, _P, c_int, c_int, _P]),
    "b200_conv2d_dgrad_tf32": (c_int, [_P, _P, _P, _P] + _CONV_DIMS + [_P]),
    "b200_conv2d_wgrad_tf32": (c_int, [_P, _P, _P] + _CONV_DIMS + [_P]),
    "b200_augment_batch": (c_int, [_P] * 7 + [c_int] * 9 + [_P, _P, _P]),
}

_lib = None
_device_ok = set()


class B200Error(RuntimeError):
    pass


def load():
    """Loads the shared library (once) and sets the ctypes prototypes. Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200Error(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C pytorch_ddp_resnet_b200/csrc`. There is no fallback path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200_last_error().decode("utf-8", "replace")


def check(status: int, what: str) -> None:
    if status != 0:
        raise B200Error(f"{what} failed (status {status}): {last_error()}")


def require_device(device_index: int) -> None:
    """Fails loudly unless the current CUDA device is a compute-capability-10 part."""
    if device_index in _device_ok:
        return
    check(load().b200_device_check(), "b200_device_check")
    _device_ok.add(device_index)


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)


def launch_count() -> int:
    """Kernels launched by the library in this process so far."""
    return int(load().b200_launch_count())
