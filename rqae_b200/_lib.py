"""ctypes binding of librqae_b200.so (C ABI declared in include/rqae_b200.h).

The shared library is the product; this module only loads it and declares the
argument types.  There is no fallback: if the library has not been built the
import fails, and every call on a machine without an sm_100 GPU returns
RQAE_ENODEVICE / RQAE_ECUDA, which is raised as RuntimeError."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# RQAE_B200_LIB points the binding at another build of the same library (A/B timing of kernel variants)
LIB_PATH = os.environ.get("RQAE_B200_LIB") or os.path.join(_HERE, "librqae_b200.so")

# every symbol include/rqae_b200.h declares (tests/test_capi_symbols.py checks the list against the header)
SYMBOLS = [
    "rqae_version", "rqae_strerror", "rqae_last_cuda_error", "rqae_packed_bytes", "rqae_pack_weights",
    "rqae_forward_f32", "rqae_forward_variant", "rqae_hook_rmsnorm", "rqae_decode_f32", "rqae_forward_host_f32", "rqae_forward_host_config", "rqae_forward_host_mode", "rqae_widen_codes_host", "rqae_forward_host_release",
    "rqae_fp32_peak_probe", "rqae_intensity_again_f16", "rqae_search_tc_store_bytes", "rqae_search_tc_pack_store",
    "rqae_search_tc_workspace_bytes", "rqae_search_tc_maxima_f16", "rqae_search_rows_f16", "rqae_search_qrows_bytes",
    "rqae_search_build_qrows_f16",
    "rqae_launch_count", "rqae_intensity_workspace_bytes", "rqae_intensity_f16",
    "rqae_select_top_middle_bottom_f16", "rqae_decode_tc_workspace_bytes", "rqae_decode_tc_f32",
    "rqae_search_table_bytes", "rqae_search_build_table_f16", "rqae_search_accumulate_f16", "rqae_search_position_max_f16",
]

CODE_DTYPE = {"int16": 0, "int32": 1, "int64": 2}

_lib = None


def build_hint() -> str:
    return ("librqae_b200.so not found; build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc, cross-compiles for sm_100a)")


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(build_hint())
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i, i64, sz = c.c_void_p, c.c_int, c.c_int64, c.c_size_t
    lib.rqae_version.restype = c.c_char_p
    lib.rqae_strerror.restype = c.c_char_p
    lib.rqae_strerror.argtypes = [i]
    lib.rqae_last_cuda_error.restype = c.c_char_p
    lib.rqae_packed_bytes.restype = sz
    lib.rqae_packed_bytes.argtypes = [i, i, i, i]
    lib.rqae_pack_weights.restype = i
    lib.rqae_pack_weights.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, i, vp, sz, vp]
    lib.rqae_forward_f32.restype = i
    lib.rqae_forward_f32.argtypes = [vp, vp, i, i, i, i, i, i, vp, i64, vp, i, i64, vp, vp, vp, vp]
    lib.rqae_forward_variant.restype = i
    lib.rqae_forward_variant.argtypes = [i]
    lib.rqae_hook_rmsnorm.restype = i
    lib.rqae_hook_rmsnorm.argtypes = [vp, vp, i, i, i, i, i, i, vp, i, i64, i, vp, c.c_float, i, i, vp, i, i64, vp]
    lib.rqae_decode_f32.restype = i
    lib.rqae_decode_f32.argtypes = [vp, vp, i, i, i, i, i, vp, i, i64, vp, vp, i64, vp, vp]
    lib.rqae_forward_host_f32.restype = i
    lib.rqae_forward_host_f32.argtypes = [vp, vp, i, i, i, i, i, i, vp, i64, vp, i, vp, i64]
    lib.rqae_forward_host_config.restype = i
    lib.rqae_forward_host_config.argtypes = [i, i]
    lib.rqae_forward_host_mode.restype = i
    lib.rqae_forward_host_mode.argtypes = [c.POINTER(c.c_int), c.POINTER(c.c_int)]
    lib.rqae_widen_codes_host.restype = i
    lib.rqae_widen_codes_host.argtypes = [vp, vp, i64, i, i]
    lib.rqae_forward_host_release.restype = i
    lib.rqae_forward_host_release.argtypes = []
    lib.rqae_fp32_peak_probe.restype = i
    lib.rqae_fp32_peak_probe.argtypes = [i, i, c.POINTER(c.c_double), vp, vp]
    lib.rqae_intensity_workspace_bytes.restype = sz
    lib.rqae_intensity_workspace_bytes.argtypes = [vp, i, i, i64]
    lib.rqae_intensity_f16.restype = i
    lib.rqae_intensity_f16.argtypes = [vp, i, vp, i, i64, i64, vp, i64, i, vp, vp, i, vp, i64, vp, sz, vp]
    lib.rqae_intensity_again_f16.restype = i
    lib.rqae_intensity_again_f16.argtypes = [vp, i, i64, vp, i64, i, vp, vp, i, vp, i64, vp, sz, vp]
    lib.rqae_select_top_middle_bottom_f16.restype = i
    lib.rqae_select_top_middle_bottom_f16.argtypes = [vp, i64, i64, i64, i, vp, vp, vp]
    lib.rqae_decode_tc_workspace_bytes.restype = sz
    lib.rqae_decode_tc_workspace_bytes.argtypes = [i, i, i64, i]
    lib.rqae_decode_tc_f32.restype = i
    lib.rqae_decode_tc_f32.argtypes = [vp, vp, vp, i, i, i, i, i, vp, i, i64, vp, i64, vp, i, vp, sz, vp]
    lib.rqae_search_table_bytes.restype = sz
    lib.rqae_search_table_bytes.argtypes = [i, i]
    lib.rqae_search_build_table_f16.restype = i
    lib.rqae_search_build_table_f16.argtypes = [vp, i, vp, i64, i, i, vp, sz, vp]
    lib.rqae_search_accumulate_f16.restype = i
    lib.rqae_search_accumulate_f16.argtypes = [vp, i, vp, i, i64, i64, i, i, i, vp, vp]
    lib.rqae_search_position_max_f16.restype = i
    lib.rqae_search_position_max_f16.argtypes = [vp, i64, i, i, vp, i64, vp]
    lib.rqae_search_tc_store_bytes.restype = sz
    lib.rqae_search_tc_store_bytes.argtypes = [i64, i]
    lib.rqae_search_tc_pack_store.restype = i
    lib.rqae_search_tc_pack_store.argtypes = [vp, i, i64, i64, i, i, i, vp, sz, vp]
    lib.rqae_search_tc_workspace_bytes.restype = sz
    lib.rqae_search_tc_workspace_bytes.argtypes = [vp, i]
    lib.rqae_search_tc_maxima_f16.restype = i
    lib.rqae_search_tc_maxima_f16.argtypes = [vp, i64, i, i, vp, vp, i, i, vp, i64, i, vp, i, vp, i64, vp, sz, vp]
    lib.rqae_search_qrows_bytes.restype = sz
    lib.rqae_search_qrows_bytes.argtypes = [i, i, i]
    lib.rqae_search_build_qrows_f16.restype = i
    lib.rqae_search_build_qrows_f16.argtypes = [vp, i, vp, i64, i, i, vp, sz, vp]
    lib.rqae_search_rows_f16.restype = i
    lib.rqae_search_rows_f16.argtypes = [vp, i, vp, i, i64, i64, i, vp, i, i, vp, i, i, vp, vp]
    lib.rqae_launch_count.restype = i64
    lib.rqae_launch_count.argtypes = [i]
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        lib = load()
        msg = lib.rqae_strerror(rc).decode()
        if rc == 3:
            msg += ": " + lib.rqae_last_cuda_error().decode()
        raise RuntimeError(f"{what} failed: {msg} (code {rc})")
