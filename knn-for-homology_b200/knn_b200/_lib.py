"""ctypes binding of libknn_b200.so (the C ABI declared in include/knn_b200.h).

This is the stub a maintainer of the reference would add in place of faiss's SWIG layer
(see INTEGRATION.md).  Loading never touches CUDA; the first call that needs a device does.
There is no CPU fallback: a missing library or a missing device raises.
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("KNN_B200_LIB", _HERE.parent / "libknn_b200.so"))

c_i64 = ctypes.c_int64
c_vp = ctypes.c_void_p

# element types of caller rows for the *_typed entry points (KNN_DTYPE_* in include/knn_b200.h)
DTYPE_F32 = 0
DTYPE_F16 = 1
DTYPE_BF16 = 2

# name -> (restype, argtypes); mirrors include/knn_b200.h one to one
SIGNATURES = {
    "knn_last_error": (ctypes.c_char_p, []),
    "knn_device_count": (ctypes.c_int, []),
    "knn_kernel_launches": (c_i64, []),
    "knn_normalize_l2": (ctypes.c_int, [c_vp, c_i64, c_i64, ctypes.c_int]),
    "knn_normalize_l2_dev": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp]),
    "knn_index_create": (ctypes.c_int, [ctypes.POINTER(c_vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint]),
    "knn_index_free": (ctypes.c_int, [c_vp]),
    "knn_index_reset": (ctypes.c_int, [c_vp]),
    "knn_index_reserve": (ctypes.c_int, [c_vp, c_i64]),
    "knn_index_add": (ctypes.c_int, [c_vp, c_i64, c_vp]),
    "knn_index_add_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_vp]),
    "knn_index_ntotal": (c_i64, [c_vp]),
    "knn_index_d": (ctypes.c_int, [c_vp]),
    "knn_index_metric": (ctypes.c_int, [c_vp]),
    "knn_index_search": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "knn_index_search_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "knn_index_search_filter_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "knn_index_search_finish_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "knn_index_search_begin_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), c_vp]),
    "knn_index_search_filter_batch_dev": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp]),
    "knn_index_search_finish_batch_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "knn_index_search_end_dev": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "knn_index_add_typed": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int]),
    "knn_index_add_typed_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_vp]),
    "knn_index_search_typed": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_i64, c_vp, c_vp]),
    "knn_index_search_typed_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "knn_index_search_begin_typed_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_i64, ctypes.POINTER(c_i64),
                                                        ctypes.POINTER(c_i64), c_vp]),
    "knn_index_search_filter_typed_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "knn_index_search_finish_typed_dev": (ctypes.c_int, [c_vp, c_i64, c_vp, ctypes.c_int, c_i64, c_vp, c_vp, c_vp, c_i64,
                                                         c_vp]),
    "knn_index_reconstruct": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp]),
    "knn_merge_topk_dev": (ctypes.c_int, [ctypes.c_int, c_i64, c_i64, ctypes.c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "knn_peer_buffer_alloc": (ctypes.c_int, [ctypes.POINTER(c_vp), c_i64, ctypes.c_int]),
    "knn_peer_buffer_free": (ctypes.c_int, [c_vp]),
    "knn_peer_handle_get": (ctypes.c_int, [c_vp, c_vp]),
    "knn_peer_handle_open": (ctypes.c_int, [c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]),
    "knn_peer_handle_close": (ctypes.c_int, [c_vp]),
    "knn_bounds_push_peer_dev": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_i64, c_vp, c_vp, c_vp, ctypes.c_uint32, c_vp, c_vp]),
    "knn_bounds_wait_max_dev": (ctypes.c_int, [ctypes.c_int, c_i64, c_vp, c_vp, ctypes.c_uint32, c_vp, c_vp, c_vp]),
    "knn_merge_topk_peer_dev": (ctypes.c_int, [ctypes.c_int, c_i64, c_i64, ctypes.c_int, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "knn_eval_family_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "knn_eval_levels_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, ctypes.c_int, c_i64, c_vp, c_vp, c_vp]),
    "knn_eval_sets_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "knn_remove_self_hit_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "knn_prefilter_measure_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, ctypes.c_int,
                                                 c_vp, c_vp, c_vp, c_vp]),
    "knn_prefilter_emit_dev": (ctypes.c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, ctypes.c_int,
                                              c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "knn_index_set_param": (ctypes.c_int, [c_vp, ctypes.c_char_p, c_i64]),
    "knn_index_get_stat": (ctypes.c_int, [c_vp, ctypes.c_char_p, ctypes.POINTER(ctypes.c_double)]),
}

_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C knn-for-homology_b200/csrc`). knn_b200 has no CPU fallback."
            )
        lib = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export the ABI
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class KnnError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        msg = load().knn_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(msg)
        if rc == -3:
            raise MemoryError(msg)
        raise KnnError(f"knn_b200 error {rc}: {msg}")
