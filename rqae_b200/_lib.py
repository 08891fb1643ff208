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

_s, _vp, _i, _i64, _sz, _f = (ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t,
                               ctypes.c_float)
_pi, _pd = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)

# name -> (restype, argtypes) of every function include/rqae_b200.h declares, in its order
# (tests/test_capi_symbols.py checks the names and types against the header)
BINDINGS = {
    "rqae_version": (_s, []),
    "rqae_strerror": (_s, [_i]),
    "rqae_last_cuda_error": (_s, []),
    "rqae_packed_bytes": (_sz, [_i, _i, _i, _i]),
    "rqae_pack_weights": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "rqae_forward_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _i, _i64, _vp, _vp, _vp, _vp]),
    "rqae_forward_variant": (_i, [_i]),
    "rqae_hook_rmsnorm": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _i64, _i, _vp, _f, _i, _i, _vp, _i, _i64, _vp]),
    "rqae_decode_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i64, _vp, _vp, _i64, _vp, _vp]),
    "rqae_forward_host_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _i, _vp, _i64]),
    "rqae_forward_host_config": (_i, [_i, _i]),
    "rqae_forward_host_mode": (_i, [_pi, _pi]),
    "rqae_widen_codes_host": (_i, [_vp, _vp, _i64, _i, _i]),
    "rqae_forward_host_release": (_i, []),
    "rqae_intensity_workspace_bytes": (_sz, [_vp, _i, _i, _i64]),
    "rqae_intensity_f16": (_i, [_vp, _i, _vp, _i, _i64, _i64, _vp, _i64, _i, _vp, _vp, _i, _vp, _i64, _vp, _sz, _vp]),
    "rqae_intensity_again_f16": (_i, [_vp, _i, _i64, _vp, _i64, _i, _vp, _vp, _i, _vp, _i64, _vp, _sz, _vp]),
    "rqae_intensity_exact_f16": (_i, [_vp, _i, _vp, _i, _i64, _i64, _vp, _i64, _i, _vp, _vp, _i, _vp, _i64, _vp]),
    "rqae_select_top_middle_bottom_f16": (_i, [_vp, _i64, _i64, _i64, _i, _vp, _vp, _vp]),
    "rqae_search_table_bytes": (_sz, [_i, _i]),
    "rqae_search_build_table_f16": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "rqae_search_accumulate_f16": (_i, [_vp, _i, _vp, _i, _i64, _i64, _i, _i, _i, _vp, _vp]),
    "rqae_search_position_max_f16": (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp]),
    "rqae_decode_tc_workspace_bytes": (_sz, [_i, _i, _i64, _i]),
    "rqae_decode_tc_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i64, _vp, _i64, _vp, _i, _vp, _sz, _vp]),
    "rqae_fp32_peak_probe": (_i, [_i, _i, _pd, _vp, _vp]),
    "rqae_search_tc_store_bytes": (_sz, [_i64, _i]),
    "rqae_search_qrows_bytes": (_sz, [_i, _i, _i]),
    "rqae_search_build_qrows_f16": (_i, [_vp, _i, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "rqae_search_tc_pack_store": (_i, [_vp, _i, _i64, _i64, _i, _i, _i, _vp, _sz, _vp]),
    "rqae_search_tc_workspace_bytes": (_sz, [_vp, _i]),
    "rqae_search_tc_maxima_f16": (_i, [_vp, _i64, _i, _i, _vp, _vp, _i, _i, _vp, _i64, _i, _vp, _i, _vp, _i64, _vp, _sz, _vp]),
    "rqae_search_rows_f16": (_i, [_vp, _i, _vp, _i, _i64, _i64, _i, _vp, _i, _i, _vp, _i, _i, _vp, _vp]),
    "rqae_launch_count": (_i64, [_i]),
}
SYMBOLS = list(BINDINGS)

CODE_DTYPE = {"int16": 0, "int32": 1, "int64": 2}   # the C ABI's code_dtype by dtype name

_lib = None


def code_dtype(dtype):
    """The C ABI's ``code_dtype`` for a torch dtype: 0 int16, 1 int32, 2 int64, None for any other dtype."""
    return CODE_DTYPE.get(str(dtype).split(".")[-1])


def code_tensor(t):
    """A code tensor in a dtype the C ABI takes: ``t`` itself when it is int16 / int32 / int64, else ``t`` as int64."""
    return t if code_dtype(t.dtype) is not None else t.long()


def workspace(nbytes: int, device, buf=None):
    """Device scratch of ``nbytes`` bytes at the 1024-byte alignment the tensor-core entry points require: (tensor,
    aligned pointer, usable bytes from that pointer).  ``buf`` is reused when it is on ``device`` and large enough."""
    import torch
    if buf is None or buf.device != device or buf.numel() < nbytes + 1024:
        buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    ptr = (buf.data_ptr() + 1023) // 1024 * 1024
    return buf, ptr, buf.numel() - (ptr - buf.data_ptr())


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
    for name, (restype, argtypes) in BINDINGS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        lib = load()
        msg = lib.rqae_strerror(rc).decode()
        if rc == 3:
            msg += ": " + lib.rqae_last_cuda_error().decode()
        raise RuntimeError(f"{what} failed: {msg} (code {rc})")
