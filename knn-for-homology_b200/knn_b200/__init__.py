"""knn_b200 - B200-native exact k-nearest-neighbour search with a faiss-style API.

Host side of the drop-in for the flat-search path of konstin/knn-for-homology; all compute
happens in libknn_b200.so (hand-written sm_100a CUDA).  ``import knn_b200 as faiss`` (or
putting ``knn-for-homology_b200/`` on sys.path, which exposes a ``faiss`` alias package) lets
the reference's drivers run unchanged.
"""
from .index import (METRIC_INNER_PRODUCT, METRIC_L2, MAX_K, IndexFlat, IndexFlatIP, IndexFlatL2, IndexHNSWFlat,
                    IndexLSH, merge_topk, normalize_L2)
from .io import read_index, write_index
from .selectors import IDSelector, IDSelectorBatch, IDSelectorBitmap, IDSelectorNot, IDSelectorRange, SearchParameters
from .postproc import (compute_auc1, compute_correctness_array, compute_is_correct, evaluate_faiss, evaluate_ids,
                       format_prefilter_db, remove_self_hit, write_prefilter_db)

__all__ = ["METRIC_INNER_PRODUCT", "METRIC_L2", "MAX_K", "IndexFlat", "IndexFlatIP", "IndexFlatL2", "IndexLSH",
           "IndexHNSWFlat", "normalize_L2", "write_index", "read_index", "merge_topk", "evaluate_faiss", "evaluate_ids",
           "compute_is_correct", "compute_correctness_array", "compute_auc1", "remove_self_hit", "write_prefilter_db",
           "format_prefilter_db", "SearchParameters", "IDSelector", "IDSelectorRange", "IDSelectorBatch",
           "IDSelectorBitmap", "IDSelectorNot"]
