"""ctypes binding of libffr_b200.so (the C ABI declared in include/ffr.h).

The product path fails loudly when the CUDA library is missing: there is no CPU fallback and nothing here
imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
import re

from ._build import LIB_PATH

FFR_OK = 0
ERR_NAMES = {-1: "FFR_ERR_INVALID", -2: "FFR_ERR_CUDA", -3: "FFR_ERR_WORKSPACE", -4: "FFR_ERR_UNSUPPORTED",
             -5: "FFR_ERR_NCCL"}
METRIC_COSINE, METRIC_EUCLID = 0, 1
DTYPE_F32, DTYPE_F16 = 0, 1
FLAG_FORCE_FP32, FLAG_FORCE_MMA, FLAG_NO_RECHECK = 1, 2, 4
SELF_OTHERS, SELF_EARLIER = 0, 1
ERR_INVALID, ERR_UNSUPPORTED = -1, -4


class FfrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


_vp, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/ffr.h declares (tests check this)
SIGNATURES = {
    "ffr_abi_version": (C.c_int, []),
    "ffr_last_error": (C.c_char_p, []),
    "ffr_build_info": (C.c_char_p, []),
    "ffr_device_count": (C.c_int, []),
    "ffr_padded_dim": (_i32, [_i32]),
    "ffr_l2norm_rows_f32": (C.c_int, [_vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp]),
    "ffr_filter_workspace_bytes": (_sz, [_i64, _i64, _i32, C.c_int, C.c_int]),
    "ffr_filter": (C.c_int, [_vp, _i64, _vp, _i64, _i32, C.c_int, _vp, _vp, C.c_int, _f32, _i64, _vp, _vp, _vp,
                             _vp, _sz, _vp]),
    "ffr_filter_ex": (C.c_int, [_vp, _i64, _vp, _i64, _i32, C.c_int, _vp, _vp, C.c_int, _f32, _i64, _vp, _vp, _vp,
                                _f32, _vp, _vp, _i64, C.c_int, _vp, _sz, _vp]),
    "ffr_filter_self_workspace_bytes": (_sz, [_i64, _i64, _i32, C.c_int]),
    "ffr_filter_self": (C.c_int, [_vp, _i64, _i64, _i64, _i32, C.c_int, C.c_int, _f32, _vp, _vp, _vp,
                                  _f32, _vp, _vp, _i64, C.c_int, _vp, _sz, _vp]),
    "ffr_filter_stats": (C.c_int, [_vp, C.POINTER(_i64), _vp]),
    "ffr_ref_mean_and_thres": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "ffr_ref_mean_and_thres_batched": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "ffr_first_match_stream": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _i32, _i32, C.c_int, _f32, _f32, _vp, _vp]),
    "ffr_ctx_create": (C.c_int, [C.c_int, _i64, _i64, _i32, C.POINTER(_vp)]),
    "ffr_ctx_destroy": (None, [_vp]),
    "ffr_ctx_filter_host": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _i32, C.c_int, _f32, _i64, _vp, _vp, _vp, C.c_int]),
    "ffr_ctx_launch_count": (_i64, [_vp]),
    "ffr_launch_count": (_i64, []),
    "ffr_nccl_unique_id": (C.c_int, [_vp]),
    "ffr_comm_create": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "ffr_comm_destroy": (None, [_vp]),
    "ffr_allgather_workspace_bytes": (_sz, [C.c_int, _i64]),
    "ffr_allgather_results": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "ffr_allgather_results_inplace": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "ffr_allreduce_best_workspace_bytes": (_sz, [_i64]),
    "ffr_allreduce_best": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i32, C.c_int, _f32, _vp, _vp, _vp,
                                     _f32, _vp, _vp, _i64, _vp, _sz, _vp]),
}
# test / tuning hooks that are not part of the public header
HOOKS = {
    "ffr_set_recheck_delta": (None, [_f32]),
    "ffr_get_recheck_delta": (_f32, []),
    "ffr_debug_set_k2_events": (None, [_vp, _vp]),
    "ffr_debug_set_prof": (None, [_vp]),
    "ffr_debug_reload_env": (None, []),
    "ffr_debug_last_k2_config": (None, [C.POINTER(_i32)]),
    "ffr_debug_mma_scores": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None


def header_symbols(header_path: str | None = None) -> list[str]:
    """Function names declared in include/ffr.h (used by the CPU test that the .so exports all of them)."""
    if header_path is None:
        header_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "ffr.h")
    text = open(header_path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ffr_[a-z0-9_]+)\s*\(", text)))


def load() -> C.CDLL:
    """Load libffr_b200.so.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in {**SIGNATURES, **HOOKS}.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ffr_abi_version() != 1:
        raise RuntimeError("libffr_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != FFR_OK:
        raise FfrError(code, load().ffr_last_error().decode("utf-8", "replace"))
