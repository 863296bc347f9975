"""faiss-style flat index over libknn_b200.so.

Mirrors the slice of the faiss Python surface the reference's drivers use on the flat path
(/root/reference: cath/search.py:13-26, pfam/proteins_search.py:17-57,
seqvec_search/main.py:22-50): ``normalize_L2``, ``IndexFlat(d, metric)``, ``.train``,
``.add``, ``.search -> (D, I)``, ``.d .ntotal .metric_type .is_trained``.

Inputs may be numpy arrays (host path: the library copies H2D/D2H itself) or CUDA
``torch.Tensor``s on the index's device (device path: results come back as CUDA tensors on
the current torch stream).

16-bit rows are read as they are: float16 / bfloat16 CUDA tensors, float16 numpy arrays and
contiguous float16 / bfloat16 CPU torch tensors (numpy has no bfloat16) are handed to the
library without an fp32 copy, and every call returns exactly what it returns for the same
rows up-converted to float32.  Other dtypes are converted to float32 first, as faiss's
wrapper does.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _lib

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
MAX_K = 2048


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _default_device() -> int:
    try:
        import torch

        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except Exception:
        pass
    return 0


def _h16_code(dtype):
    """KNN_DTYPE code of a 16-bit torch / numpy dtype that the library reads as it is, else None."""
    if dtype == np.float16:
        return _lib.DTYPE_F16
    if type(dtype).__module__.startswith("torch"):
        import torch

        return {torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}.get(dtype)
    return None


def _is_host_h16_tensor(x) -> bool:
    """A CPU torch tensor of a 16-bit type: searched and added through the host path (numpy has no bfloat16)."""
    return _is_torch(x) and not x.is_cuda and _h16_code(x.dtype) is not None


def _torch_stream(device: int) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream


_PINNED_RESULT_LIMIT = 1 << 30


def _result_arrays(nq: int, k: int):
    """(D, I) numpy arrays for a host-path search.  Up to 1 GiB they live in page-locked memory (owned by a torch
    tensor the arrays keep alive), so the library DMAs the result rows straight into them under the search of the next
    query batch instead of bouncing them through a staging buffer; they are ordinary numpy arrays to the caller."""
    if 0 < nq * k * 12 <= _PINNED_RESULT_LIMIT:
        try:
            import torch

            return (torch.empty((nq, k), dtype=torch.float32, pin_memory=True).numpy(),
                    torch.empty((nq, k), dtype=torch.int64, pin_memory=True).numpy())
        except Exception:
            pass
    return np.empty((nq, k), dtype=np.float32), np.empty((nq, k), dtype=np.int64)


def normalize_L2(x) -> None:
    """In-place row normalisation, faiss.normalize_L2 (cath/search.py:19, seqvec_search/main.py:31,34).

    Like faiss (swig_ptr), requires a C-contiguous float32 matrix because it must alias the
    caller's memory; zero rows are left untouched."""
    lib = _lib.load()
    if _is_torch(x):
        import torch

        if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous() or not x.is_cuda:
            raise TypeError("normalize_L2 expects a contiguous float32 CUDA matrix")
        _lib.check(lib.knn_normalize_l2_dev(x.data_ptr(), x.shape[0], x.shape[1], _torch_stream(x.device.index)))
        return None
    if not isinstance(x, np.ndarray) or x.ndim != 2:
        raise ValueError("normalize_L2 expects a 2-d array")
    if x.dtype != np.float32:
        raise TypeError("normalize_L2 expects float32, got %s" % x.dtype)
    if not x.flags.c_contiguous:
        raise ValueError("normalize_L2 expects a C-contiguous array (it normalises in place)")
    if not x.flags.writeable:
        raise ValueError("normalize_L2 expects a writeable array")
    _lib.check(lib.knn_normalize_l2(x.ctypes.data, x.shape[0], x.shape[1], _default_device()))
    return None


class IndexFlat:
    """Exact (brute-force) index: faiss.IndexFlat(d, metric) (cath/search.py:20)."""

    def __init__(self, d: int, metric: int = METRIC_L2, device: int | None = None, bf16_storage: bool = False):
        if metric not in (METRIC_INNER_PRODUCT, METRIC_L2):
            raise ValueError("unsupported metric %r (flat path: METRIC_INNER_PRODUCT or METRIC_L2)" % (metric,))
        self._lib = _lib.load()
        self.d = int(d)
        self.metric_type = int(metric)
        self.is_trained = True
        self.device = _default_device() if device is None else int(device)
        self._h = ctypes.c_void_p()
        _lib.check(self._lib.knn_index_create(ctypes.byref(self._h), self.d, self.metric_type, self.device,
                                              1 if bf16_storage else 0))

    # -- faiss attributes ---------------------------------------------------------------
    @property
    def ntotal(self) -> int:
        return int(self._lib.knn_index_ntotal(self._h))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.knn_index_free(h)
            except Exception:
                pass
            self._h = ctypes.c_void_p()

    # -- helpers --------------------------------------------------------------------------
    def _host_matrix(self, x) -> np.ndarray:
        x = np.asarray(x)
        if x.ndim != 2:
            raise ValueError("expected a 2-d array")
        assert x.shape[1] == self.d, "dimension mismatch: got %d, index has %d" % (x.shape[1], self.d)
        if x.dtype == np.float16:
            return np.ascontiguousarray(x)  # read as it is (exact up-conversion in the kernels)
        return np.ascontiguousarray(x, dtype=np.float32)  # faiss's python wrapper does the same

    def _host_rows(self, x):
        """Host rows -> (object that owns them, KNN_DTYPE code, address of the first row)."""
        if _is_host_h16_tensor(x):
            if x.dim() != 2:
                raise ValueError("expected a 2-d tensor")
            assert x.shape[1] == self.d, "dimension mismatch: got %d, index has %d" % (x.shape[1], self.d)
            x = x.contiguous()
            return x, _h16_code(x.dtype), x.data_ptr()
        x = self._host_matrix(x)
        return x, _h16_code(x.dtype) or _lib.DTYPE_F32, x.ctypes.data

    def _dev_matrix(self, x):
        """CUDA tensor -> (contiguous tensor, KNN_DTYPE code): float16 / bfloat16 as they are, anything else float32."""
        import torch

        if x.dim() != 2:
            raise ValueError("expected a 2-d tensor")
        assert x.shape[1] == self.d, "dimension mismatch: got %d, index has %d" % (x.shape[1], self.d)
        if not x.is_cuda or x.device.index != self.device:
            raise ValueError("tensor must live on cuda:%d" % self.device)
        code = _h16_code(x.dtype)
        if code is not None:
            return x.contiguous(), code
        return x.to(torch.float32).contiguous(), _lib.DTYPE_F32

    # -- faiss methods --------------------------------------------------------------------
    def train(self, x) -> None:
        """No-op for a flat index (pfam/proteins_search.py:35, seqvec_search/main.py:37)."""
        if not _is_torch(x):
            self._host_matrix(x)
        elif _is_host_h16_tensor(x):
            self._host_rows(x)

    def reserve(self, n: int) -> None:
        _lib.check(self._lib.knn_index_reserve(self._h, int(n)))

    def add(self, x) -> None:
        """Append rows; ids are the row numbers (cath/search.py:22)."""
        if _is_torch(x) and not _is_host_h16_tensor(x):
            x, code = self._dev_matrix(x)
            _lib.check(self._lib.knn_index_add_typed_dev(self._h, x.shape[0], x.data_ptr(), code, _torch_stream(self.device)))
            # the ingest kernel reads x asynchronously on the current stream; keep it alive until then
            import torch

            x.record_stream(torch.cuda.current_stream(self.device))
            return
        x, code, ptr = self._host_rows(x)
        _lib.check(self._lib.knn_index_add_typed(self._h, x.shape[0], ptr, code))

    def reset(self) -> None:
        _lib.check(self._lib.knn_index_reset(self._h))

    def _search_params(self, params, exclude, nq: int, id_base: int, on_device: bool, allow_bit0: int = 0,
                       allow_nbits: int | None = None):
        """(knn_search_params or None, the arrays it points to).  params.sel becomes one packed bitmap (built on the
        device for a device search, on the host for a host search; allow_nbits defaults to ntotal); exclude, an (nq,)
        array of ids in the space the call returns (-1: none), is passed as int64 - for a host search with the id base
        taken off, because the host call returns row numbers and the id base is added afterwards."""
        sel = getattr(params, "sel", None) if params is not None else None
        if sel is None and exclude is None:
            return None, ()
        if allow_nbits is None:
            allow_nbits = self.ntotal
        c = _lib.SearchParamsC(None, int(allow_bit0), int(allow_nbits), None)
        keep = []
        if on_device:
            import torch

            dev = torch.device("cuda", self.device)
            if sel is not None:
                bits = sel.bitmap(int(allow_nbits), device=dev)
                keep.append(bits)
                c.allow_bits = bits.data_ptr()
            if exclude is not None:
                ex = torch.as_tensor(exclude, dtype=torch.int64).to(dev).contiguous().view(-1)
                if ex.shape[0] != nq:
                    raise ValueError("exclude must hold one id per query (%d), got %d" % (nq, ex.shape[0]))
                keep.append(ex)
                c.exclude_ids = ex.data_ptr()
        else:
            if sel is not None:
                bits = np.ascontiguousarray(sel.bitmap(int(allow_nbits)))
                keep.append(bits)
                c.allow_bits = bits.ctypes.data
            if exclude is not None:
                ex = exclude.detach().cpu().numpy() if _is_torch(exclude) else exclude
                ex = np.ascontiguousarray(np.asarray(ex, dtype=np.int64).reshape(-1))
                if ex.shape[0] != nq:
                    raise ValueError("exclude must hold one id per query (%d), got %d" % (nq, ex.shape[0]))
                if id_base:
                    ex = np.ascontiguousarray(np.where(ex >= int(id_base), ex - int(id_base), -1))
                keep.append(ex)
                c.exclude_ids = ex.ctypes.data
        keep.append(c)
        return c, keep

    def search(self, x, k: int, id_base: int = 0, *, params=None, exclude=None):
        """(D, I) of the k best rows per query, best first (cath/search.py:24).

        params: faiss.SearchParameters(sel=IDSelector...) restricts the search to the selected rows.  exclude (an
        extension): an (nq,) array or tensor of ids, -1 for none; id exclude[q] is never returned for query q (ids
        include id_base).  A filtered search returns exactly what an unfiltered one returns on an index of the
        eligible rows alone, ids mapped back; queries with fewer than k eligible rows get id -1 padding."""
        k = int(k)
        if k <= 0:
            raise ValueError("k must be positive")
        if _is_torch(x) and not _is_host_h16_tensor(x):
            import torch

            x, code = self._dev_matrix(x)
            D = torch.empty((x.shape[0], k), dtype=torch.float32, device=x.device)
            I = torch.empty((x.shape[0], k), dtype=torch.int64, device=x.device)
            p, keep = self._search_params(params, exclude, x.shape[0], id_base, on_device=True)
            if p is None:
                _lib.check(self._lib.knn_index_search_typed_dev(self._h, x.shape[0], x.data_ptr(), code, k, D.data_ptr(),
                                                                I.data_ptr(), int(id_base), _torch_stream(self.device)))
            else:  # the filter arrays are read on the current stream, which later frees of them are ordered behind
                _lib.check(self._lib.knn_index_search_params_dev(self._h, x.shape[0], x.data_ptr(), code, k, D.data_ptr(),
                                                                 I.data_ptr(), int(id_base), ctypes.byref(p),
                                                                 _torch_stream(self.device)))
            return D, I
        x, code, ptr = self._host_rows(x)
        D, I = _result_arrays(x.shape[0], k)
        p, keep = self._search_params(params, exclude, x.shape[0], id_base, on_device=False)
        if p is None:
            _lib.check(self._lib.knn_index_search_typed(self._h, x.shape[0], ptr, code, k, D.ctypes.data, I.ctypes.data))
        else:
            _lib.check(self._lib.knn_index_search_params(self._h, x.shape[0], ptr, code, k, D.ctypes.data, I.ctypes.data,
                                                         ctypes.byref(p)))
        if id_base:
            I[I >= 0] += int(id_base)
        return D, I

    # -- two-phase search (row-sharded databases; see distributed.ShardedIndexFlat) ----------
    def search_filter(self, x, k: int, j: int | None = None):
        """Phase 1 on CUDA tensor x: returns `lower` (nq,) float32 - per query a lower bound of the true
        k-th best score inside this shard (combine across shards with an element-wise MAX) - and, when j is
        given, also `lower_j`, the same for the j-th best (with G shards and j = ceil(k/G), combine with an
        element-wise MIN: every shard holds j rows at or above it)."""
        import torch

        x, code = self._dev_matrix(x)
        lower = torch.empty((x.shape[0],), dtype=torch.float32, device=x.device)
        lower_j = torch.empty_like(lower) if j is not None else None
        _lib.check(self._lib.knn_index_search_filter_typed_dev(self._h, x.shape[0], x.data_ptr(), code, int(k),
                                                               lower.data_ptr(), int(j or 0),
                                                               lower_j.data_ptr() if j is not None else None,
                                                               _torch_stream(self.device)))
        self._pending_x = (x, code)  # phase 2 needs the same queries (kept alive here)
        return lower if j is None else (lower, lower_j)

    def search_finish(self, lower, k: int, id_base: int = 0):
        """Phase 2: exact rescoring of the candidates that survive the combined bound -> this shard's (D, I)."""
        import torch

        x, code = self._pending_x
        self._pending_x = None
        D = torch.empty((x.shape[0], int(k)), dtype=torch.float32, device=x.device)
        I = torch.empty((x.shape[0], int(k)), dtype=torch.int64, device=x.device)
        lower = lower.contiguous()
        _lib.check(self._lib.knn_index_search_finish_typed_dev(self._h, x.shape[0], x.data_ptr(), code, int(k),
                                                               lower.data_ptr(), D.data_ptr(), I.data_ptr(), int(id_base),
                                                               _torch_stream(self.device)))
        return D, I

    # -- the same, batch by batch (the caller overlaps exchange + finish of batch b with the filter of batch b + 1) --
    def search_begin(self, x, k: int, params=None, exclude=None, id_base: int = 0, allow_bit0: int = 0,
                     allow_nbits: int | None = None):
        """Returns (nbatches, batch_rows); x (and the filter) are kept alive until search_end.  With params / exclude
        the batches are filtered (see search); finish_batch and end must then be given the same id_base.  A shard of a
        row-sharded database passes the global selector with allow_bit0 = its first global row and allow_nbits = the
        global row count."""
        x, code = self._dev_matrix(x)
        nb, rows = ctypes.c_int64(), ctypes.c_int64()
        p, keep = self._search_params(params, exclude, x.shape[0], id_base, on_device=True, allow_bit0=allow_bit0,
                                      allow_nbits=allow_nbits)
        if p is None:
            _lib.check(self._lib.knn_index_search_begin_typed_dev(self._h, x.shape[0], x.data_ptr(), code, int(k),
                                                                  ctypes.byref(nb), ctypes.byref(rows), _torch_stream(self.device)))
        else:
            _lib.check(self._lib.knn_index_search_begin_params_dev(self._h, x.shape[0], x.data_ptr(), code, int(k),
                                                                   int(id_base), ctypes.byref(p), ctypes.byref(nb),
                                                                   ctypes.byref(rows), _torch_stream(self.device)))
        self._pending_x = x
        self._pending_filter = keep
        return nb.value, rows.value

    def search_filter_batch(self, b: int, j: int, bounds) -> None:
        """bounds: zero-initialised float32 CUDA tensor (nbatches, 2, batch_rows); slice [b] is written."""
        _lib.check(self._lib.knn_index_search_filter_batch_dev(self._h, int(b), int(j), bounds.data_ptr(), _torch_stream(self.device)))

    def search_finish_batch(self, b: int, bounds, D, I, id_base: int = 0) -> None:
        _lib.check(self._lib.knn_index_search_finish_batch_dev(self._h, int(b), bounds.data_ptr() if bounds is not None else None,
                                                               D.data_ptr(), I.data_ptr(), int(id_base), _torch_stream(self.device)))

    def search_end(self, D, I, id_base: int = 0) -> None:
        _lib.check(self._lib.knn_index_search_end_dev(self._h, D.data_ptr(), I.data_ptr(), int(id_base), _torch_stream(self.device)))
        self._pending_x = None
        self._pending_filter = ()

    def search_into(self, xq_ptr: int, nq: int, k: int, D_ptr: int, I_ptr: int, dtype: int = _lib.DTYPE_F32) -> None:
        """Host-pointer search into caller-owned (e.g. pinned) buffers: the raw C-ABI call (dtype: a KNN_DTYPE code)."""
        _lib.check(self._lib.knn_index_search_typed(self._h, int(nq), int(xq_ptr), int(dtype), int(k), int(D_ptr), int(I_ptr)))

    def reconstruct_n(self, i0: int = 0, n: int | None = None) -> np.ndarray:
        n = self.ntotal - i0 if n is None else n
        out = np.empty((n, self.d), dtype=np.float32)
        _lib.check(self._lib.knn_index_reconstruct(self._h, int(i0), int(n), out.ctypes.data))
        return out

    # -- tuning / introspection -------------------------------------------------------------
    def set_param(self, name: str, value: int) -> None:
        _lib.check(self._lib.knn_index_set_param(self._h, name.encode(), int(value)))

    def stat(self, name: str) -> float:
        out = ctypes.c_double()
        _lib.check(self._lib.knn_index_get_stat(self._h, name.encode(), ctypes.byref(out)))
        return out.value


class IndexFlatIP(IndexFlat):
    def __init__(self, d: int, **kw):
        super().__init__(d, METRIC_INNER_PRODUCT, **kw)


class IndexFlatL2(IndexFlat):
    def __init__(self, d: int, **kw):
        super().__init__(d, METRIC_L2, **kw)


class IndexLSH:
    """Name must exist (seqvec_search/main.py:23 evaluates faiss.IndexLSH at import); the LSH
    index itself is approximate and outside the flat path (SURVEY.md section 8f)."""

    def __init__(self, *a, **kw):
        from .drivers import APPROXIMATE_INDEX_HINT

        raise NotImplementedError(APPROXIMATE_INDEX_HINT % "IndexLSH")


class IndexHNSWFlat:
    def __init__(self, *a, **kw):
        from .drivers import APPROXIMATE_INDEX_HINT

        raise NotImplementedError(APPROXIMATE_INDEX_HINT % "IndexHNSWFlat")


def merge_topk(D_lists, I_lists, metric: int):
    """Merge [nlists, nq, k] CUDA tensors of per-shard results into the global (D, I)."""
    import torch

    lib = _lib.load()
    nlists, nq, k = D_lists.shape
    D_lists = D_lists.contiguous()
    I_lists = I_lists.contiguous()
    D = torch.empty((nq, k), dtype=torch.float32, device=D_lists.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=D_lists.device)
    _lib.check(lib.knn_merge_topk_dev(int(metric), nq, k, nlists, D_lists.data_ptr(), I_lists.data_ptr(),
                                      D.data_ptr(), I.data_ptr(), _torch_stream(D_lists.device.index)))
    return D, I
