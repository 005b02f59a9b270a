"""ctypes binding of the C-ABI library (include/revers_o_b200.h).

There is no CPU fallback: if the shared library is missing, loading raises with the build command;
if no sm_100 device is present, every compute call returns an error that `check()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RVO_LIB_PATH") or os.path.join(_HERE, "lib", "librevers_o_b200.so")   # override: A/B builds only

RVO_E_UNSUPPORTED = -5
RVO_MAX_K = 512
RVO_SMALL_Q = 4
RVO_KMEANS_MAX_CLUSTERS = 65536
RVO_DTYPE_BF16, RVO_DTYPE_F16 = 0, 1
RVO_PATH_AUTO, RVO_PATH_SMALL, RVO_PATH_TENSOR, RVO_PATH_DENSE = 0, 1, 2, 3

# name -> (restype, argtypes); mirrors include/revers_o_b200.h one to one
PROTOTYPES = {
    "rvo_version": (C.c_int, []),
    "rvo_last_error": (C.c_char_p, []),
    "rvo_device_sm_count": (C.c_int, [C.c_void_p]),
    "rvo_db_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "rvo_normalize_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int64,
                                     C.c_void_p, C.c_void_p]),
    "rvo_mask_pool_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rvo_mask_pool": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_mask_pool_to_db": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_size_t, C.c_void_p]),
    "rvo_exchange_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "rvo_exchange_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "rvo_exchange_free": (C.c_int, [C.c_void_p]),
    "rvo_exchange_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rvo_exchange_import": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "rvo_exchange_unimport": (C.c_int, [C.c_void_p]),
    "rvo_search_topk_push": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                       C.c_int64, C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                       C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_search_topk_fused": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                        C.c_int64, C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_merge_topk_exchange": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvo_search_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "rvo_search_topk": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int32,
                                  C.c_float, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                  C.c_void_p]),
    "rvo_search_workspace_bytes_ex": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rvo_search_topk_ex": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int32,
                                     C.c_float, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    "rvo_padded_queries": (C.c_int, [C.c_int32, C.c_int32]),
    "rvo_scan_tile_rows": (C.c_int, [C.c_int32, C.c_int32]),
    "rvo_scores_dense": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_int64,
                                   C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_packed_result_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "rvo_merge_topk_packed": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p]),
    "rvo_merge_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvo_selfjoin_workspace_bytes": (C.c_size_t, [C.c_int32]),
    "rvo_selfjoin_threshold": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_float,
                                         C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_void_p]),
    "rvo_selfjoin_workspace_bytes_ex": (C.c_size_t, [C.c_int32, C.c_int64]),
    "rvo_selfjoin_threshold_ex": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_float,
                                            C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_join_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int64]),
    "rvo_join_threshold": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                     C.c_float, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_cross_join_threshold": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                           C.c_int64, C.c_float, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_join_components": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                      C.c_float, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_components_flatten": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "rvo_components_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "rvo_knn_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "rvo_knn_join": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                               C.c_int64, C.c_int32, C.c_float, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_knn_exclude_self": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rvo_kmeans_update_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "rvo_kmeans_update": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "rvo_kmeans_finalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "rvo_kernel_launch_count": (C.c_int64, []),
    "rvo_last_scan_ms": (C.c_float, []),
    "rvo_set_option": (C.c_int, [C.c_char_p, C.c_int64]),
}

_lib = None


class RvoError(RuntimeError):
    pass


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RvoError(
                f"{LIB_PATH} is missing: the CUDA extension is the product path and there is no CPU fallback. "
                "Build it with `python -m revers_o_b200.build` (nvcc, sm_100a).")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().rvo_last_error().decode("utf-8", "replace")
        raise RvoError(f"{what} failed (code {rc}): {msg}")


option_epoch = 0   # bumped by set_option: cached plans (workspace sizes) depend on the tuning options


def set_option(name: str, value: int) -> None:
    global option_epoch
    check(load().rvo_set_option(name.encode(), int(value)), f"rvo_set_option({name})")
    option_epoch += 1


def kernel_launch_count() -> int:
    return int(load().rvo_kernel_launch_count())
