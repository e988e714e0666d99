"""ctypes binding of libkeds_knn.so (include/keds_knn.h). This is the stub a KEDs maintainer would
add; everything above it (index.py, retrieval.py, metrics.py) is host logic in the reference's own
language. There is no fallback: a missing library or a failing call raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkeds_knn.so")

METRIC_IP = 0
METRIC_L2 = 1
SEARCH_EXACT_ONLY = 1
SEARCH_NO_FALLBACK = 2
SEARCH_FORCE_IP = 4


class SearchStats(C.Structure):
    _fields_ = [
        ("n_flagged", C.c_int32 * 2),
        ("slices", C.c_int32),
        ("items", C.c_int32),
        ("grid", C.c_int32),
        ("exact_only", C.c_int32),
        ("launches", C.c_int32),
        ("err_word", C.c_uint32),
    ]


_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/keds_knn.h one to one
SIGNATURES = {
    "keds_index_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "keds_index_free": (None, [_vp]),
    "keds_index_add": (C.c_int, [_vp, _vp, C.c_int64]),
    "keds_index_add_ex": (C.c_int, [_vp, _vp, C.c_int64, C.c_uint32]),
    "keds_index_get_rows": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp]),
    "keds_index_reset": (C.c_int, [_vp]),
    "keds_index_ntotal": (C.c_int64, [_vp]),
    "keds_index_dim": (C.c_int, [_vp]),
    "keds_index_metric": (C.c_int, [_vp]),
    "keds_index_device": (C.c_int, [_vp]),
    "keds_index_rows": (_vp, [_vp]),
    "keds_index_set_id_offset": (C.c_int, [_vp, C.c_int64]),
    "keds_index_operand_format": (C.c_int, [_vp]),
    "keds_index_set_operand_format": (C.c_int, [_vp, C.c_int]),
    "keds_index_generation": (C.c_uint64, [_vp]),
    "keds_exchange_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(_vp), C.c_int64, C.POINTER(_vp)]),
    "keds_exchange_free": (None, [_vp]),
    "keds_exchange_capacity": (C.c_int64, [_vp]),
    "keds_index_search_sharded": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int, _vp]),
    "keds_index_rows_ipc": (C.c_int, [_vp, _vp]),
    "keds_exchange_attach_rows": (C.c_int, [_vp, C.c_int, C.POINTER(_vp), _i64p, _i64p]),
    "keds_retrieve2_sharded": (
        C.c_int,
        [_vp, _vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp, C.c_int, C.c_float, C.c_int64, C.c_int64,
         _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_uint32, _vp],
    ),
    "keds_exchange_stats": (
        C.c_int,
        [_vp, _vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_uint32)],
    ),
    "keds_index_search": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp]),
    "keds_index_search_ex": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int, C.c_uint32, _vp]),
    "keds_index_search2": (
        C.c_int,
        [_vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_uint32, _vp],
    ),
    "keds_retrieve2": (
        C.c_int,
        [_vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp, C.c_int, C.c_float,
         _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_uint32, _vp],
    ),
    "keds_index_range_search": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, _vp, C.c_uint32, _vp]),
    "keds_index_range_results": (C.c_int, [_vp, _vp, _vp, _vp]),
    "keds_index_label_hits": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp, C.c_int, _vp, _vp]),
    "keds_index_sync": (C.c_int, [_vp, _vp]),
    "keds_index_last_stats": (C.c_int, [_vp, C.POINTER(SearchStats)]),
    "keds_index_set_profiling": (C.c_int, [_vp, C.c_int]),
    "keds_index_profile": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "keds_index_profile_chain": (
        C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int]),
    "keds_gather_pool": (
        C.c_int,
        [_vp, C.c_int64, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp],
    ),
    "keds_topk_merge": (C.c_int, [_vp, _vp, C.c_int, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp]),
    "keds_topk_merge_strided": (
        C.c_int,
        [_vp, _vp, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp],
    ),
    "keds_p2p_push": (
        C.c_int,
        [_vp, C.c_int64, C.POINTER(_vp), C.POINTER(_vp), C.c_int, C.c_int, C.c_uint32, _vp, _vp],
    ),
    "keds_topk_merge_wait": (
        C.c_int,
        [_vp, _vp, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp, C.c_int,
         C.c_uint32, _vp, _vp],
    ),
    "keds_gallery_rank": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp]),
    "keds_index_rank": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp, _vp, _vp]),
    "keds_label_hits": (C.c_int, [_vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp]),
    "keds_consumer_create": (
        C.c_int,
        [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)],
    ),
    "keds_consumer_free": (None, [_vp]),
    "keds_consumer_set_linear": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int]),
    "keds_consumer_finalize": (C.c_int, [_vp]),
    "keds_consumer_forward": (
        C.c_int,
        [_vp, _vp, _vp, C.c_int64, _vp, C.c_int64, _vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp],
    ),
    "keds_consumer_check": (C.c_int, [_vp, _vp, C.POINTER(C.c_int64)]),
    "keds_consumer_param_count": (C.c_int64, [_vp]),
    "keds_consumer_param_offset": (
        C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                  C.POINTER(C.c_int64)]),
    "keds_consumer_bind_params": (C.c_int, [_vp, _vp]),
    "keds_consumer_forward_train": (
        C.c_int,
        [_vp, _vp, _vp, C.c_int64, _vp, C.c_int64, _vp, _vp, _vp, C.c_int64, C.c_int, C.POINTER(_vp), _vp, _vp],
    ),
    "keds_consumer_backward": (C.c_int, [_vp, _vp, _vp, _vp]),
    "keds_consumer_forward_sharded": (
        C.c_int,
        [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, _vp, _vp],
    ),
    "keds_consumer_forward_train_sharded": (
        C.c_int,
        [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.POINTER(_vp), _vp, _vp],
    ),
    "keds_consumer_debug_hidden": (C.c_int, [_vp, C.c_int, _vp, C.c_int64, _vp]),
    "keds_consumer_set_debug": (C.c_int, [_vp, C.c_int]),
    "keds_consumer_debug_timeline": (C.c_int, [_vp, C.c_int, _vp, C.c_int64]),
    "keds_clip_loss_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "keds_clip_loss_free": (None, [_vp]),
    "keds_clip_loss_forward_backward": (
        C.c_int,
        [_vp, _vp, _vp, C.c_int64, C.c_int, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp],
    ),
    "keds_clip_loss_check": (C.c_int, [_vp, _vp]),
    "keds_debug_scores": (C.c_int, [_vp, _vp, C.c_int64, _vp, _vp]),
    "keds_debug_plan": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int64, C.c_int, C.POINTER(C.c_int32)]),
    "keds_debug_linear_plan": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32)]),
    "keds_consumer_debug_linear": (
        C.c_int,
        [_vp, C.c_int, _vp, _vp, C.c_int64, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp,
         C.c_int64, C.c_int, _vp],
    ),
    "keds_consumer_debug_attend": (
        C.c_int,
        [_vp, C.c_int, C.c_int, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp, _vp, _vp,
         _vp, _vp, _vp, _vp],
    ),
    "keds_index_set_eps_scale": (C.c_int, [_vp, C.c_float]),
    "keds_index_set_pdl": (C.c_int, [_vp, C.c_int]),
    "keds_last_error": (C.c_char_p, []),
    "keds_device_count": (C.c_int, []),
    "keds_version": (C.c_char_p, []),
}

_lib = None


def load() -> C.CDLL:
    """Load the native library (building it first if sources are newer and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        _build.build()
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -m keds_b200.build` (there is no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header and library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().keds_last_error().decode("utf-8", "replace")


def check(status: int) -> None:
    if status != 0:
        raise RuntimeError(f"libkeds_knn error {status}: {last_error()}")
