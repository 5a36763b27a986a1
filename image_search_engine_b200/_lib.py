"""ctypes binding of libise.so (the C ABI declared in include/ise.h).

There is deliberately NO fallback: if the shared library is missing, or no B200 is
visible, every compute entry point raises.  Build with ``python __graft_entry__.py``
(or ``make -C image_search_engine_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("ISE_LIB_PATH", _PKG_DIR / "libise.so"))   # override: kernel A/B testing only

_c_void_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_f64 = C.c_double
_size = C.c_size_t

# name -> (restype, argtypes); mirrors include/ise.h one to one
PROTOTYPES = {
    "ise_version": (_int, []),
    "ise_last_error": (C.c_char_p, []),
    "ise_ctx_create": (_int, [_int, C.POINTER(_c_void_p)]),
    "ise_ctx_destroy": (None, [_c_void_p]),
    "ise_ctx_sm_count": (_int, [_c_void_p]),
    "ise_rand_perm_prefix": (_int, [_i64, _i64, _i64, _c_void_p]),
    "ise_split_plan": (_int, [_c_void_p, _i64, _i64, _c_void_p, C.POINTER(C.c_int32)]),
    "ise_split_plan_warm": (_int, [_i64]),
    "ise_pack_rows": (_int, [_c_void_p, _c_void_p, _i64, _i64, _int, _int, _int, _c_void_p, _int, C.POINTER(_int)]),
    "ise_pack_begin": (_int, [_c_void_p, _c_void_p, _c_void_p, _int, _int, _int, _int, _c_void_p, _int,
                              C.POINTER(_c_void_p)]),
    "ise_pack_wait": (_int, [_c_void_p, _int, C.POINTER(_int)]),
    "ise_pack_poll": (_int, [_c_void_p, _int, C.POINTER(_int), C.POINTER(_int)]),
    "ise_pack_claim": (_int, [_c_void_p, _int, C.POINTER(_int)]),
    "ise_pack_end": (_int, [_c_void_p]),
    "ise_prepare_planes": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _i64, _c_void_p, _c_void_p, _i64,
                                  _c_void_p, _c_void_p, _c_void_p]),
    "ise_prepare_rows": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _i64, _c_void_p, _c_void_p, _i64,
                                _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_scan_f32": (_int, [_c_void_p, _c_void_p, _i64, _int, _i64, _c_void_p, _c_void_p]),
    "ise_normalize_l2": (_int, [_c_void_p, _c_void_p, _i64, _int, _c_void_p]),
    "ise_gemm_select_workspace_bytes": (_size, [_c_void_p, _i64, _i64, _int, _int]),
    "ise_gemm_select": (_int, [_c_void_p,
                               _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p,
                               _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p,
                               _i64, _i64, _int, _int, _int, _i64, _c_void_p, _c_void_p, _c_void_p,
                               _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_assign_fused": (_int, [_c_void_p, _c_void_p, _i64, _i64, _int, _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p,
                                _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _i64, _int, _i64,
                                _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_assign_workspace_bytes": (_size, [_c_void_p, _i64, _int]),
    "ise_assign_verified_covers": (_int, [_c_void_p, _i64, _i64, _int]),
    "ise_assign_verified": (_int, [_c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p,
                                   _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _i64, _i64, _int, _int, _i64,
                                   _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_flat_search_exact_workspace_bytes": (_size, [_c_void_p, _i64, _i64, _int]),
    "ise_flat_search_exact": (_int, [_c_void_p, _c_void_p, _i64, _c_void_p, _i64, _int, _int, _int, _i64,
                                     _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_pair_scores": (_int, [_c_void_p, _c_void_p, _i64, _c_void_p, _i64, _int, _int, _c_void_p, _c_void_p]),
    "ise_scores_mask": (_int, [_c_void_p, _c_void_p, _i64, _i64, _c_void_p, _int, _i64, _int, _c_void_p]),
    "ise_rescore_topk": (_int, [_c_void_p, _c_void_p, _int, _i64, _c_void_p, _i64, _i64, _i64, _int, _int, _int, _i64,
                                _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_rescore_select": (_int, [_c_void_p, _c_void_p, _int, _i64, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p,
                                  _c_void_p, _i64, _i64, _int, _int, _int, _int, _i64, _c_void_p, _c_void_p, _c_void_p,
                                  _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_gemm_collect": (_int, [_c_void_p,
                                _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p,
                                _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p,
                                _i64, _i64, _int, _int, _i64, _c_void_p, _int,
                                _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_range_seed": (_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64, _int, _int, C.c_float,
                              _c_void_p, _c_void_p]),
    "ise_range_count": (_int, [_c_void_p, _c_void_p, _int, _i64, _c_void_p, _i64, _i64, _i64, _int, _int, C.c_float,
                               _i64, _c_void_p, _c_void_p, _int, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_range_lims_workspace_bytes": (_size, [_c_void_p, _i64]),
    "ise_range_lims": (_int, [_c_void_p, _c_void_p, _i64, _i64, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_range_fill": (_int, [_c_void_p, _i64, _int, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                              _c_void_p, _c_void_p]),
    "ise_range_sort_workspace_bytes": (_size, [_c_void_p, _i64, _i64]),
    "ise_range_sort": (_int, [_c_void_p, _i64, _c_void_p, _i64, _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_scores_range_workspace_bytes": (_size, [_c_void_p, _i64, _i64]),
    "ise_scores_range": (_int, [_c_void_p, _c_void_p, _i64, _i64, _int, C.c_float, _i64, _i64, _c_void_p, _c_void_p,
                                _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_topk_merge": (_int, [_c_void_p, _c_void_p, _c_void_p, _int, _i64, _int, _int, _c_void_p, _c_void_p,
                              _c_void_p]),
    "ise_kmeans_accumulate": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _i64, _c_void_p, _c_void_p,
                                     _c_void_p, _i64, _int, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_kmeans_accumulate_workspace_bytes": (_size, [_c_void_p, _i64, _i64]),
    "ise_kmeans_accumulate_sorted": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _i64, _c_void_p, _c_void_p, _c_void_p, _i64, _int,
                                            _c_void_p, _c_void_p, _c_void_p, _c_void_p, _size, _c_void_p]),
    "ise_kmeans_mean": (_int, [_c_void_p, _c_void_p, _c_void_p, _i64, _int, _c_void_p, _c_void_p, _c_void_p]),
    "ise_kmeans_apply_splits": (_int, [_c_void_p, _c_void_p, _i64, _int, _c_void_p, C.c_int32, _c_void_p]),
    "ise_bovw_histogram": (_int, [_c_void_p, _c_void_p, _i64, _c_void_p, _i64, _int, _int, _int, _c_void_p, _int,
                                  _f64, _f64, _f64, _f64, _c_void_p]),
    "ise_bovw_histogram_csr": (_int, [_c_void_p, _c_void_p, _c_void_p, _i64, _int, _int, _int, _c_void_p, _c_void_p,
                                      _c_void_p, _c_void_p, _int, _f64, _f64, _f64, _f64, _c_void_p]),
    "ise_scores_topk_workspace_bytes": (_size, [_c_void_p, _i64, _i64, _int]),
    "ise_scores_topk": (_int, [_c_void_p, _c_void_p, _i64, _i64, _int, _int, _i64, _c_void_p, _c_void_p, _c_void_p,
                               _size, _c_void_p]),
    "ise_ivfpq_residual": (_int, [_c_void_p, _c_void_p, _i64, _i64, _int, _c_void_p, _c_void_p, _c_void_p, _c_void_p]),
    "ise_ivfpq_scan": (_int, [_c_void_p, _c_void_p, _i64, _int, _c_void_p, _i64, _c_void_p, _int, _c_void_p, _int, _int,
                              _c_void_p, _c_void_p, _i64, _c_void_p, _c_void_p]),
    "ise_okapi_csr": (_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _i64, _f64, _f64, _f64, _f64, _c_void_p, _int,
                             _c_void_p, _c_void_p]),
    "ise_tfidf_finish": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _c_void_p, _int, _c_void_p]),
    "ise_comm_init_all": (_int, [_int, _c_void_p, C.POINTER(_c_void_p)]),
    "ise_comm_destroy": (None, [_c_void_p]),
    "ise_comm_size": (_int, [_c_void_p]),
    "ise_allreduce_sum_f32": (_int, [_c_void_p, _c_void_p, _i64, _c_void_p]),
    "ise_allgather": (_int, [_c_void_p, _c_void_p, _c_void_p, _i64, _c_void_p]),
    "ise_okapi_tf": (_int, [_c_void_p, _c_void_p, _int, _i64, _int, _f64, _f64, _f64, _f64, _c_void_p,
                            _c_void_p]),
}

METRIC_IP, METRIC_L2 = 0, 1
DTYPE_F32, DTYPE_U8, DTYPE_F16 = 0, 1, 2
HIST_NUMPY_COMPAT, HIST_BINCOUNT = 0, 1
OUT_F32, OUT_F64 = 0, 1


class IseError(RuntimeError):
    pass


_lib = None
_lib_lock = threading.RLock()
_ctxs: dict[int, int] = {}


def load():
    """Loads libise.so and binds every prototype; raises if the extension was not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not LIB_PATH.exists():
            raise IseError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python __graft_entry__.py`); there is no CPU fallback")
        lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_LOCAL if hasattr(os, "RTLD_LOCAL") else 0)
        for name, (restype, argtypes) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
        return lib


def check(rc: int):
    if rc != 0:
        msg = load().ise_last_error()
        raise IseError(msg.decode("utf-8", "replace") if msg else f"libise call failed with {rc}")


def ctx(device_index: int) -> int:
    """Per-device ise_ctx handle (created once)."""
    h = _ctxs.get(device_index)
    if h is not None:
        return h
    with _lib_lock:
        h = _ctxs.get(device_index)
        if h is None:
            out = _c_void_p()
            rc = load().ise_ctx_create(int(device_index), C.byref(out))
            check(rc)
            h = out.value
            _ctxs[device_index] = h
    return h
