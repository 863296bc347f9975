"""Filtered search, the parts that need no GPU: the header declares knn_search_params and its three entry points, the
library exports them, every IDSelector packs to the bits a numpy reference gives (faiss's bitmap byte order, bits past
the end), IndexFlat hands params / exclude to the right entry point with the right pointers and id base, and
ShardedIndexFlat gives every shard the global bitmap from its first global row on.  The kernels and the bit-exactness
contract are covered by tests/test_gpu_filtered_search.py."""
import ctypes
import os
import re
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

REPO = Path(__file__).resolve().parent.parent
HEADER = (REPO / "include" / "knn_b200.h").read_text()
CALLS = ["knn_index_search_params", "knn_index_search_params_dev", "knn_index_search_begin_params_dev"]


def test_header_declares_the_params_struct_and_calls():
    m = re.search(r"typedef struct knn_search_params \{(.*?)\} knn_search_params;", HEADER, re.S)
    assert m
    fields = " ".join(m.group(1).split())
    for f in ["const uint32_t* allow_bits;", "int64_t allow_bit0;", "int64_t allow_nbits;", "const int64_t* exclude_ids;"]:
        assert f in re.sub(r"/\*.*?\*/", "", fields), f
    for name in CALLS:
        m = re.search(r"\bint %s\(([^)]*)\);" % name, HEADER)
        assert m, name
        assert "const knn_search_params* p" in " ".join(m.group(1).split()), name


def test_ctypes_struct_matches_the_header_layout():
    from knn_b200 import _lib

    assert ctypes.sizeof(_lib.SearchParamsC) == 32
    assert [f[0] for f in _lib.SearchParamsC._fields_] == ["allow_bits", "allow_bit0", "allow_nbits", "exclude_ids"]
    for name in CALLS:
        assert name in _lib.SIGNATURES


def test_library_exports_the_params_calls():
    from knn_b200 import _lib

    if not _lib.LIB_PATH.exists():
        pytest.skip("libknn_b200.so is not built")
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in CALLS:
        assert hasattr(lib, name), name


def test_faiss_alias_exposes_the_selectors():
    import faiss

    for name in ["SearchParameters", "IDSelectorRange", "IDSelectorBatch", "IDSelectorBitmap", "IDSelectorNot"]:
        assert hasattr(faiss, name), name


# ---- selector packing ------------------------------------------------------------------------------------------
def _bits(words, n):
    """Words (numpy uint32 or torch int32) -> bool array of the first n bits (bit i: word i >> 5, bit i & 31)."""
    w = words.cpu().numpy() if hasattr(words, "cpu") else np.asarray(words)
    w = np.ascontiguousarray(w).view(np.uint32)
    assert len(w) == (n + 31) // 32
    return ((w[np.arange(n) >> 5] >> (np.arange(n) & 31).astype(np.uint32)) & 1).astype(bool)


def _selectors(n):
    import knn_b200 as k

    rng = np.random.default_rng(n)
    ids = rng.integers(-3, n + 40, 50)
    bm = (rng.random(max(1, n // 8 - 2)) * 256).astype(np.uint8)  # shorter than n bits: the rest selects nothing
    i = np.arange(n)
    bm_ref = np.zeros(n, bool)
    nb = min(n, 8 * len(bm))
    bm_ref[:nb] = (bm[i[:nb] >> 3] >> (i[:nb] & 7)) & 1  # faiss: bit i & 7 of byte i >> 3
    return [
        (k.IDSelectorRange(5, n - 17), (i >= 5) & (i < n - 17)),
        (k.IDSelectorRange(-4, n + 100), np.ones(n, bool)),
        (k.IDSelectorBatch(ids), np.isin(i, ids)),
        (k.IDSelectorBatch(10, ids), np.isin(i, ids[:10])),
        (k.IDSelectorBitmap(bm), bm_ref),
        (k.IDSelectorBitmap(3, bm), bm_ref & (i < 24)),
        (k.IDSelectorNot(k.IDSelectorRange(5, n - 17)), ~((i >= 5) & (i < n - 17))),
        (k.IDSelectorNot(k.IDSelectorBitmap(bm)), ~bm_ref),
    ]


@pytest.mark.parametrize("n", [1, 31, 32, 33, 1000, 4097])
def test_selectors_pack_like_numpy(n):
    for sel, ref in _selectors(n):
        assert np.array_equal(_bits(sel.bitmap(n), n), ref), (type(sel).__name__, n)
        assert np.array_equal(_bits(sel.bitmap(n, device="cpu"), n), ref), (type(sel).__name__, n, "torch")


def test_bitmap_bytes_are_the_words_little_endian():
    import knn_b200 as k

    bm = np.array([0x01, 0x80, 0x00, 0xFF, 0x3C], np.uint8)
    w = k.IDSelectorBitmap(bm).bitmap(40)
    assert w.dtype == np.dtype("<u4") and list(w) == [0xFF008001, 0x3C]


# ---- IndexFlat routing against a stub library ---------------------------------------------------------------------
class _StubLib:
    """Records every call; the params struct is read while the call is in progress.  ntotal is configurable."""

    def __init__(self, ntotal):
        self.calls, self.ntotal = [], ntotal

    def __getattr__(self, name):
        if not name.startswith("knn_"):
            raise AttributeError(name)

        def call(*args):
            if name == "knn_index_ntotal":
                return self.ntotal
            rec = list(args)
            for i, a in enumerate(args):
                if type(a).__name__ == "CArgObject" and isinstance(a._obj, ctypes.Structure):
                    p = a._obj
                    nw = (p.allow_nbits + 31) // 32
                    rec[i] = dict(bit0=p.allow_bit0, nbits=p.allow_nbits,
                                  bits=np.ctypeslib.as_array((ctypes.c_uint32 * nw).from_address(p.allow_bits)).copy()
                                  if p.allow_bits else None,
                                  ex=np.ctypeslib.as_array((ctypes.c_int64 * args[1]).from_address(p.exclude_ids)).copy()
                                  if p.exclude_ids else None)
            self.calls.append((name, tuple(rec)))
            return 0

        return call


def _stub_index(ntotal, d=8):
    from knn_b200.index import IndexFlat

    idx = IndexFlat.__new__(IndexFlat)
    idx._lib, idx._h, idx.d, idx.metric_type, idx.device = _StubLib(ntotal), ctypes.c_void_p(1), d, 0, 0
    return idx


def test_unfiltered_search_keeps_its_entry_point():
    import knn_b200 as k

    idx = _stub_index(100)
    x = np.zeros((4, 8), np.float32)
    idx.search(x, 3)
    idx.search(x, 3, params=k.SearchParameters())  # no selector: the unfiltered call
    assert [c[0] for c in idx._lib.calls] == ["knn_index_search_typed"] * 2


def test_host_search_passes_the_bitmap_and_exclusions_without_the_id_base():
    import knn_b200 as k

    n, nq = 100, 4
    idx = _stub_index(n)
    x = np.zeros((nq, 8), np.float32)
    ex = np.array([1005, -1, 1000, 7], np.int64)
    idx.search(x, 3, 1000, params=k.SearchParameters(sel=k.IDSelectorRange(10, 70)), exclude=ex)
    name, args = idx._lib.calls[-1]
    assert name == "knn_index_search_params" and args[1:5] == (nq, x.ctypes.data, 0, 3)
    p = args[7]
    assert p["bit0"] == 0 and p["nbits"] == n
    assert np.array_equal(_bits(p["bits"], n), (np.arange(n) >= 10) & (np.arange(n) < 70))
    assert list(p["ex"]) == [5, -1, 0, -1]  # the host call returns row numbers: the id base comes off (ids < it: none)
    # exclusions alone, as a torch tensor
    idx.search(x, 3, exclude=torch.tensor([3, 2, 1, 0]))
    p = idx._lib.calls[-1][1][7]
    assert p["bits"] is None and list(p["ex"]) == [3, 2, 1, 0]


def test_exclude_must_hold_one_id_per_query():
    idx = _stub_index(10)
    with pytest.raises(ValueError, match="one id per query"):
        idx.search(np.zeros((4, 8), np.float32), 3, exclude=np.zeros(3, np.int64))


# ---- ShardedIndexFlat: every shard gets the global bitmap, its first row as allow_bit0 and id_base --------------
class _RecShard:
    device = 0

    def __init__(self):
        self.ntotal = 0

    def add(self, x):
        self.ntotal += x.shape[0]


def _shard_worker(rank, world, port, out):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    import knn_b200 as k
    from knn_b200.distributed import ShardedIndexFlat

    seen = []

    class Rec(ShardedIndexFlat):
        def _two_phase_pipelined(self, xd, kk, mark, flt=None):
            seen.append(dict(flt, exclude=flt["exclude"].tolist(), nq=xd.shape[0]))
            D = torch.full((xd.shape[0], kk), float(rank))
            I = torch.full((xd.shape[0], kk), rank, dtype=torch.int64)
            return D, I

    merged = []
    index = Rec(8, 0, index_factory=_RecShard, peer_merge=False, shard_weights=[0.25, 0.75],
                merge_fn=lambda D, I, m: merged.append((D.shape, I.shape)) or (D[0], I[0]))
    index.add(np.zeros((40, 8), np.float32))
    x = np.zeros((5, 8), np.float32)
    ex = np.array([3, -1, 39, 10, 0])
    p = k.SearchParameters(sel=k.IDSelectorRange(0, 20))
    index.search(x, 4, params=p, exclude=ex)
    s = seen[0]
    assert len(seen) == 1
    assert s["id_base"] == s["allow_bit0"] == [0, 10][rank] and s["allow_nbits"] == 40, s
    assert s["exclude"] == list(ex) and s["params"] is p and s["nq"] == 5
    assert merged[0] == (torch.Size([2, 5, 4]), torch.Size([2, 5, 4]))
    if rank == 0:
        Path(out).write_text("ok")
    dist.destroy_process_group()


def test_sharded_filtered_search_hands_each_shard_its_offsets_world2_gloo(tmp_path):
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = tmp_path / "ok"
    mp.spawn(_shard_worker, args=(2, port, str(out)), nprocs=2, join=True)
    assert out.read_text() == "ok"


def test_grid_index_refuses_filters():
    from knn_b200.distributed import GridIndexFlat

    with pytest.raises(NotImplementedError, match="ShardedIndexFlat"):
        GridIndexFlat.search(object.__new__(GridIndexFlat), np.zeros((2, 8), np.float32), 3,
                             exclude=np.zeros(2, np.int64))
