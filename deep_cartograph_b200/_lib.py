"""ctypes binding of libdcg_b200.so (the C-ABI declared in include/dcg.h).

There is NO CPU fallback: importing this module without the built library, or calling an
operator with CPU tensors, raises.  Build with ``python -m deep_cartograph_b200.build``.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_c_i64 = C.c_int64
_c_int = C.c_int
_c_sz = C.c_size_t
_p = C.c_void_p

COV_SIMT_F32 = 0
COV_TC_3XTF32 = 1
COV_TC_1XTF32 = 2
COV_TC_3XF16 = 3
COV_TC_I8X3 = 4
COV_ENGINES = {"simt_f32": COV_SIMT_F32, "tc_3xtf32": COV_TC_3XTF32, "tc_1xtf32": COV_TC_1XTF32,
               "tc_3xf16": COV_TC_3XF16, "tc_i8x3": COV_TC_I8X3}

LINKAGE_METHODS = {"single": 0, "complete": 1, "average": 2, "ward": 3}   # DCG_LINK_* (dcg.h)
HDBSCAN_MAX_MIN_SAMPLES = 64                                              # DCG_HDBSCAN_MAX_MIN_SAMPLES (dcg.h)
SILHOUETTE_MAX_SLOTS = 384                                                # DCG_SILHOUETTE_MAX_SLOTS (dcg.h)
SILHOUETTE_MAX_LABELINGS = 32                                             # DCG_SILHOUETTE_MAX_LABELINGS (dcg.h)

_SIGNATURES = {
    # name: (restype, [argtypes])
    "dcg_version": (_c_int, []),
    "dcg_error_string": (C.c_char_p, [_c_int]),
    "dcg_device_info": (_c_int, [C.POINTER(_c_int)] * 3),
    "dcg_colstats_workspace_bytes": (_c_sz, [_c_i64, _c_int]),
    "dcg_colstats_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _p, _p, _p, _p, _c_sz, _p]),
    "dcg_p2p_buffer_bytes": (_c_sz, [_c_int, _c_i64]),
    "dcg_p2p_alloc": (_c_int, [_c_sz, _p, _p]),
    "dcg_p2p_open": (_c_int, [_p, _p]),
    "dcg_p2p_close": (_c_int, [_p, _c_int]),
    "dcg_p2p_allreduce_f64": (_c_int, [_p, _p, _c_int, _c_int, _c_int, _c_int, _p, _c_i64, C.c_uint64, _p]),
    "dcg_stats_pack": (_c_int, [C.c_double, _p, _p, _p, _p, _c_int, _p, _p]),
    "dcg_stats_merge": (_c_int, [_p, _c_int, _c_int, _p, _p, _p, _p, _p, _p]),
    "dcg_standardize_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _p, _p]),
    "dcg_gather_standardize_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _c_i64, _c_i64, _p, _p, _p, _p]),
    "dcg_cov_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int, _c_int, _c_int]),
    "dcg_cov_lag_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _p, _c_int,
                                 _p, _p, _p, _p, _c_int, _p, _c_sz, _p]),
    "dcg_cov_i8_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int, _c_int]),
    "dcg_cov_lag_i8_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _p, _p, _p, _c_int,
                                    _p, _p, _p, _p, _p, _p, _c_sz, _p]),
    "dcg_cov_i8_set_timing": (_c_int, [_c_int]),
    "dcg_cov_i8_get_timing": (_c_int, [C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(_c_int)]),
    "dcg_project_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_project_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _p, _p, _c_int, _p, _p, _p,
                                 _p, _c_sz, _p]),
    "dcg_project_blocks_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_project_blocks_f32": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _p, _p, _c_int, _c_int, _p, _c_i64,
                                        _p, _c_sz, _p]),
    "dcg_kmeans_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int, _c_int]),
    "dcg_kmeans_step": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _c_int, _p,
                                 _p, _p, _p, _p, _c_int, _p, _p, _c_sz, _p]),
    "dcg_kmeans_update": (_c_int, [_p, _p, _c_int, _c_int, _p, _p, _p]),
    "dcg_kmeans_iterate": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _c_int, _p, _p, _p, _p, _c_sz, _p]),
    "dcg_kmeans_iterate_n": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _c_int, _p, _p, _p, _c_int, C.c_double,
                                      _p, _c_sz, _p]),
    "dcg_nearest_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_nearest_to_centers": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _c_int, _p,
                                        _p, _c_sz, _p]),
    "dcg_ticacov_out_doubles": (_c_sz, [_c_int]),
    "dcg_ticacov_workspace_bytes": (_c_sz, [_c_i64, _c_int]),
    "dcg_ticacov_f32": (_c_int, [_p, _p, _p, _p, _c_i64, _c_int, _p, _p, _c_sz, _p]),
    "dcg_gen_eig_small_f64": (_c_int, [_p, _p, _c_int, _c_int, _p, _p, _p, _p]),
    "dcg_tri_inv_blocks_f64": (_c_int, [_p, _p, _c_int, _c_int, _c_int, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _c_i64, _p]),
    "dcg_cluster_dispersion": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _p, _c_int, _p, _p, _p]),
    "dcg_silhouette_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_silhouette_f64": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _c_int, _p, _p, _c_int, _p, _p, _p, _c_sz, _p]),
    "dcg_linkage_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_linkage_f64": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _p, _c_sz, _p]),
    "dcg_hdbscan_workspace_bytes": (_c_sz, [_c_i64, _c_int, _c_int]),
    "dcg_core_distances_f64": (_c_int, [_p, _c_i64, _c_int, _c_i64, _c_int, _p, _p, _c_sz, _p]),
    "dcg_mreach_mst_f64": (_c_int, [_p, _c_i64, _c_int, _c_i64, _p, _p, _p, _c_sz, _p]),
    "dcg_nearest_frames_workspace_bytes": (_c_sz, [_c_i64, _c_i64, _c_int]),
    "dcg_nearest_frames_f64": (_c_int, [_p, _c_i64, _c_i64, _p, _c_i64, _c_i64, _c_int, _p, _p, _p, _c_sz, _p]),
    "dcg_fes_bin_f32": (_c_int, [_p, _c_i64, _c_i64, _c_int, _c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                                 _c_int, _c_int, _p, _p, _p]),
    "dcg_fes_smooth_f64": (_c_int, [_p, _c_int, _c_int, _c_int, C.c_double, C.c_double, C.c_double, _p, _p, _p, _p]),
    "dcg_ticaloss_out_doubles": (_c_sz, [_c_int]),
    "dcg_ticaloss_f64": (_c_int, [_p, _c_int, C.c_double, _c_int, _p, _p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class DcgError(RuntimeError):
    """A libdcg_b200 entry point returned a non-zero code."""

    def __init__(self, fn: str, code: int, msg: str):
        super().__init__(f"{fn} failed with code {code}: {msg}")
        self.code = code


_lib = None


def lib_path() -> str:
    return os.environ.get("DCG_B200_LIB", _build.LIB_PATH)


def load():
    """Load (once) and return the ctypes handle.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build the CUDA extension first "
            "(python -m deep_cartograph_b200.build).  There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(fn: str, code: int) -> None:
    if code != 0:
        msg = load().dcg_error_string(code)
        raise DcgError(fn, code, msg.decode() if msg else "?")


def call(fn: str, *args) -> None:
    """Call an int-returning entry point and raise DcgError on failure."""
    check(fn, getattr(load(), fn)(*args))
