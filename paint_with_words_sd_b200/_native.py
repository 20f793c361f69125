"""ctypes binding of libpww_b200.so (the C ABI in include/pww_b200.h).

There is no fallback: if the library is missing or a call returns a non-zero status this module
raises.  `PWW_B200_LIB` overrides the library path.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PWW_B200_LIB", os.path.join(_HERE, "libpww_b200.so"))

PWW_STAT_MAX, PWW_STAT_STD = 0, 1

EXPORTS = (
    "pww_version", "pww_status_str", "pww_last_cuda_error", "pww_device_supported",
    "pww_xattn_workspace_bytes", "pww_xattn_stats_f16", "pww_xattn_fwd_f16", "pww_attn_fwd_f16",
    "pww_xattn_fused_workspace_bytes", "pww_xattn_fused_f16",
    "pww_groupnorm_workspace_bytes", "pww_groupnorm_nhwc_f16", "pww_geglu_f16", "pww_add_layernorm_f16",
    "pww_sampler_prepare_f16", "pww_sampler_step_f32", "pww_randn_f32",
)


class NativeError(RuntimeError):
    pass


_lib: Optional[ctypes.CDLL] = None
launch_count = 0          # kernels launched through this binding (bench.py reports it as gpu_launches)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found: build it with `python -m paint_with_words_sd_b200.csrc.build` "
            "(there is no CPU / PyTorch fallback for the attention path)")
    L = ctypes.CDLL(LIB_PATH)
    c_i, c_i64, c_vp, c_f, c_sz = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_float, ctypes.c_size_t
    L.pww_version.restype = c_i
    L.pww_status_str.restype = ctypes.c_char_p
    L.pww_status_str.argtypes = [c_i]
    L.pww_last_cuda_error.restype = ctypes.c_char_p
    L.pww_device_supported.restype = c_i
    L.pww_xattn_workspace_bytes.restype = c_sz
    L.pww_xattn_workspace_bytes.argtypes = [c_i] * 5
    L.pww_xattn_stats_f16.restype = c_i
    L.pww_xattn_stats_f16.argtypes = [c_vp, c_vp, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64, c_i, c_vp,
                                      c_vp, c_vp, c_sz, c_vp]
    L.pww_xattn_fwd_f16.restype = c_i
    L.pww_xattn_fwd_f16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64,
                                    c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_f, c_vp]
    L.pww_xattn_fused_workspace_bytes.restype = c_sz
    L.pww_xattn_fused_workspace_bytes.argtypes = []
    L.pww_xattn_fused_f16.restype = c_i
    L.pww_xattn_fused_f16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64,
                                      c_i64, c_i64, c_vp, c_i64, c_i, c_vp, c_vp, c_i, c_vp, c_f, c_vp, c_vp, c_sz, c_vp]
    L.pww_attn_fwd_f16.restype = c_i
    L.pww_attn_fwd_f16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i, c_i, c_i, c_i, c_i64, c_i64, c_i64, c_i64, c_f, c_vp]
    L.pww_groupnorm_workspace_bytes.restype = c_sz
    L.pww_groupnorm_workspace_bytes.argtypes = [c_i, c_i, c_i]
    L.pww_groupnorm_nhwc_f16.restype = c_i
    L.pww_groupnorm_nhwc_f16.argtypes = [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i, c_i, c_i, c_i, c_f, c_i, c_vp, c_sz, c_vp]
    L.pww_geglu_f16.restype = c_i
    L.pww_geglu_f16.argtypes = [c_vp, c_vp, c_i64, c_i, c_vp]
    L.pww_add_layernorm_f16.restype = c_i
    L.pww_add_layernorm_f16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i, c_f, c_vp]
    L.pww_sampler_prepare_f16.restype = c_i
    L.pww_sampler_prepare_f16.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i, c_i, c_i, c_i, c_i, c_vp]
    L.pww_sampler_step_f32.restype = c_i
    L.pww_sampler_step_f32.argtypes = [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_f, c_i, c_i, c_i,
                                       c_i, c_vp]
    L.pww_randn_f32.restype = c_i
    L.pww_randn_f32.argtypes = [c_vp, c_i64, ctypes.c_uint64, c_i, c_vp]
    _lib = L
    return L


def check(status: int, what: str) -> None:
    if status != 0:
        L = lib()
        msg = L.pww_status_str(status).decode()
        if status == -3:
            msg += ": " + L.pww_last_cuda_error().decode()
        raise NativeError(f"{what} failed: {msg} (status {status})")
