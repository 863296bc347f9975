"""Filtered search (faiss SearchParameters / IDSelector, and one excluded id per query) on the GPU.

The contract (include/knn_b200.h, knn_search_params): a filtered search returns exactly what an unfiltered search
returns on an index that holds only the eligible rows, with ids mapped back to row numbers - bit for bit, D and I.
The oracle of every selector test is therefore "the same search on an IndexFlat built from x[allowed], I mapped
through the allowed ids"; for exclusions it is "that search with k + 1, the excluded id removed, or else the last
column dropped".  Results also pass the fp64 parity check.

1. selectors on every path: densities, clustered equal scores at the panel boundaries, both metrics, path 1 / 2, every
   GEMM kernel (nq), k from 1 to 2048, d = 1024 / 100, bf16 storage, fp32 / fp16 / bf16 queries, host (pageable,
   pinned) and device queries, id_base and an allow_bit0 that is not a multiple of 32;
2. fewer eligible rows than k, and none;
3. excluded rows that would win (duplicates of the queries);
4. all-vs-all with exclude = arange(n): the single dense panel (C2 shape) and several panels, duplicated rows;
5. overflow repair with filters on the device and host paths;
6. the adversarial error-bound data with a selector;
7. the batch-wise two-phase ABI on 2, 3 and 8 virtual shards, and ShardedIndexFlat in two processes;
8. misuse."""
import ctypes
import os
import socket
import sys
import time
from pathlib import Path

import numpy as np
import pytest

from oracle import adversarial as adv
from oracle import flat_oracle as fo
from oracle.parity import check_parity

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent
IP, L2 = 0, 1
F32, F16, BF16 = 0, 1, 2
ERR_INVALID = -1


@pytest.fixture(scope="module")
def knn():
    import knn_b200

    assert knn_b200._lib.load().knn_device_count() >= 1, "no CUDA device: the CUDA path cannot run"
    return knn_b200


def _data(n, nq, d, seed, clusters=40):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((clusters, d)).astype(np.float32)
    xb = (c[rng.integers(0, clusters, n)] + 0.6 * rng.standard_normal((n, d))).astype(np.float32)
    xq = (c[rng.integers(0, clusters, nq)] + 0.6 * rng.standard_normal((nq, d))).astype(np.float32)
    return xb, xq


def _mask(n, kind, seed=0):
    rng = np.random.default_rng(seed + 1000)
    m = np.zeros(n, dtype=bool)
    if kind == "all":
        m[:] = True
    elif kind == "single":
        m[n // 3] = True
    elif isinstance(kind, float):
        m[rng.random(n) < kind] = True
    elif kind != "none":
        raise ValueError(kind)
    return m


def _index(knn, xb, metric, params=None, bf16_storage=False):
    idx = knn.IndexFlat(xb.shape[1], metric, device=0, bf16_storage=bf16_storage)
    for name, v in (params or {}).items():
        idx.set_param(name, v)
    if xb.shape[0]:
        idx.add(xb)
    return idx


def _oracle(knn, xb, xq, k, metric, allowed, exclude=None, params=None, bf16_storage=False, id_base=0):
    """Search of the index of the allowed rows (ids mapped back, + id_base); with exclude: k + 1, then the excluded id
    removed or else the last column dropped.  Host queries, the same index parameters."""
    ids = np.flatnonzero(allowed)
    kk = k + 1 if exclude is not None else k
    nq = xq.shape[0]
    if len(ids) == 0:
        D = np.full((nq, kk), -np.finfo(np.float32).max if metric == IP else np.finfo(np.float32).max, np.float32)
        I = np.full((nq, kk), -1, np.int64)
    else:
        sub = _index(knn, xb[ids], metric, params, bf16_storage)
        D, I = sub.search(xq, kk)
        I = np.where(I >= 0, ids[np.clip(I, 0, None)] + id_base, -1)
    if exclude is None:
        return D, I
    Do, Io = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    for q in range(nq):
        hit = np.flatnonzero((I[q] == exclude[q]) & (I[q] >= 0)) if exclude[q] >= 0 else []
        keep = np.ones(kk, bool)
        keep[hit[0] if len(hit) else kk - 1] = False
        Do[q], Io[q] = D[q][keep], I[q][keep]
    return Do, Io


def _eq(D, I, Dr, Ir, tag=""):
    assert np.array_equal(I, Ir), ("ids differ from the oracle", tag, np.argwhere(I != Ir)[:5])
    assert np.array_equal(D.view(np.uint32), Dr.view(np.uint32)), ("distances differ from the oracle", tag)


def _np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else t


def _parity(D, I, xq, xb, allowed, k, metric):
    """fp64 parity of a filtered result against the oracle over the eligible rows (at least k of them)."""
    ids = np.flatnonzero(allowed)
    D_ref, I_ref = fo.knn_flat(xq, xb[ids], k, metric)
    check_parity(D, np.searchsorted(ids, I), D_ref, I_ref, xq, xb[ids], metric)


# ---- 1. selectors on every path --------------------------------------------------------------------------------
# (id, n, d, nq, k, metric, density, index params)
SEL_CASES = [
    ("none", 20000, 1024, 300, 10, IP, "none", {}),
    ("single", 20000, 1024, 300, 10, L2, "single", {}),
    ("0.1pct", 20000, 1024, 300, 10, IP, 0.001, {}),
    ("10pct", 20000, 1024, 300, 10, L2, 0.1, {}),
    ("50pct", 20000, 1024, 300, 100, IP, 0.5, {}),
    ("99.9pct", 20000, 1024, 300, 100, L2, 0.999, {}),
    ("all", 20000, 1024, 300, 10, IP, "all", {}),
    ("nq1", 20000, 1024, 1, 10, IP, 0.5, {}),
    ("nq64-l2", 20000, 1024, 64, 10, L2, 0.5, {}),
    ("nq65", 20000, 1024, 65, 100, IP, 0.5, {}),
    ("nq128-l2", 20000, 1024, 128, 10, L2, 0.1, {}),
    ("nq129", 20000, 1024, 129, 10, IP, 0.5, {}),
    ("nq20000-batches", 30000, 256, 20000, 10, IP, 0.5, {"query_batch": 4096}),
    ("cg1", 20000, 1024, 300, 10, L2, 0.5, {"cta_group": 1}),
    ("exact-path", 20000, 1024, 300, 10, IP, 0.5, {"path": 1}),
    ("exact-path-l2", 20000, 1024, 40, 100, L2, 0.1, {"path": 1}),
    ("k1", 30000, 1024, 300, 1, IP, 0.5, {}),
    ("k1000", 30000, 1024, 300, 1000, L2, 0.5, {}),
    ("k2048", 30000, 1024, 300, 2048, IP, 0.5, {}),
    ("k1000-dense-small", 14433, 1024, 500, 1000, IP, 0.5, {}),
    ("d100", 20000, 100, 300, 10, L2, 0.5, {}),
    ("stream-quad", 20000, 1024, 200, 10, IP, 0.5, {"stream_quad": 1}),
]


@pytest.mark.parametrize("name,n,d,nq,k,metric,density,params", SEL_CASES, ids=[c[0] for c in SEL_CASES])
def test_selector_matches_subset_index(knn, name, n, d, nq, k, metric, density, params):
    import torch

    xb, xq = _data(n, nq, d, seed=len(name) + n)
    allowed = _mask(n, density, seed=nq)
    idx = _index(knn, xb, metric, params)
    sel = knn.IDSelectorBatch(np.flatnonzero(allowed))
    p = knn.SearchParameters(sel=sel)
    Dr, Ir = _oracle(knn, xb, xq, k, metric, allowed, params=params)
    D, I = idx.search(xq, k, params=p)                       # host (pinned result arrays) queries
    _eq(D, I, Dr, Ir, name + " host")
    Dd, Id = idx.search(torch.from_numpy(xq).cuda(), k, params=p)  # device queries
    _eq(_np(Dd), _np(Id), Dr, Ir, name + " device")
    if nq <= 300 and k <= 100 and allowed.sum() >= k:
        _parity(D, I, xq, xb, allowed, k, metric)


@pytest.mark.parametrize("qdt", ["fp16", "bf16"])
@pytest.mark.parametrize("metric", [IP, L2])
def test_selector_16bit_queries_bf16_storage(knn, qdt, metric):
    import torch

    n, nq, d, k = 20000, 300, 1024, 50
    xb, xq = _data(n, nq, d, seed=5 + metric)
    allowed = _mask(n, 0.3, seed=metric)
    tq = torch.from_numpy(xq).to({"fp16": torch.float16, "bf16": torch.bfloat16}[qdt])
    xq32 = tq.float().numpy()
    idx = _index(knn, xb, metric, bf16_storage=True)
    p = knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed)))
    Dr, Ir = _oracle(knn, xb, xq32, k, metric, allowed, bf16_storage=True)
    D, I = idx.search(tq.cuda(), k, params=p)
    _eq(_np(D), _np(I), Dr, Ir, "device " + qdt)
    D, I = idx.search(tq, k, params=p)  # CPU 16-bit tensor: the host path
    _eq(D, I, Dr, Ir, "host " + qdt)


def test_pageable_host_results_and_all_selector_types(knn):
    """Pageable result buffers through search_into-like raw calls, and every IDSelector form against its rows."""
    n, nq, d, k = 20000, 300, 256, 20
    xb, xq = _data(n, nq, d, seed=9)
    idx = _index(knn, xb, IP)
    rng = np.random.default_rng(3)
    bm = (rng.random((n + 7) // 8) * 256).astype(np.uint8)
    bm_allowed = np.unpackbits(bm, bitorder="little")[:n].astype(bool)
    cases = [(knn.IDSelectorRange(777, 15000), (np.arange(n) >= 777) & (np.arange(n) < 15000)),
             (knn.IDSelectorBitmap(bm), bm_allowed),
             (knn.IDSelectorBitmap(bm[: n // 16]), (np.arange(n) < 8 * (n // 16)) & bm_allowed),  # bits past the end
             (knn.IDSelectorNot(knn.IDSelectorRange(0, 19000)), np.arange(n) >= 19000)]
    for sel, allowed in cases:
        Dr, Ir = _oracle(knn, xb, xq, k, IP, allowed)
        lib = knn._lib.load()
        D, I = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)  # pageable
        bits = np.ascontiguousarray(sel.bitmap(n))
        c = knn._lib.SearchParamsC(bits.ctypes.data, 0, n, None)
        knn._lib.check(lib.knn_index_search_params(idx._h, nq, xq.ctypes.data, F32, k, D.ctypes.data, I.ctypes.data,
                                                   ctypes.byref(c)))
        _eq(D, I, Dr, Ir, type(sel).__name__)


def _clustered(n, d, seed):
    """Rows that all score the same against every query except a few distinct ones: ties everywhere."""
    rng = np.random.default_rng(seed)
    row = rng.standard_normal(d).astype(np.float32)
    xb = np.tile(row, (n, 1))
    xb[::97] = rng.standard_normal((len(xb[::97]), d)).astype(np.float32)
    xq = np.tile(row, (64, 1)) + 0.01 * rng.standard_normal((64, d)).astype(np.float32)
    return xb, xq


@pytest.mark.parametrize("where", ["first", "last", "end-of-first-panel", "inside-last-panel"])
@pytest.mark.parametrize("metric", [IP, L2])
def test_selected_ties_at_panel_boundaries(knn, where, metric):
    n, d, k = 50000, 128, 100
    xb, xq = _clustered(n, d, seed=len(where))
    first_panel = 1024  # k = 100: max(1024, 4k) rows stored densely
    lo = {"first": 0, "last": n - 400, "end-of-first-panel": first_panel - 200, "inside-last-panel": 40000}[where]
    allowed = np.zeros(n, bool)
    allowed[lo:lo + 400] = True
    allowed[::97] |= np.arange(n)[::97] % 2 == 0
    idx = _index(knn, xb, metric, {"path": 2})
    D, I = idx.search(xq, k, params=knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed))))
    Dr, Ir = _oracle(knn, xb, xq, k, metric, allowed, params={"path": 2})
    _eq(D, I, Dr, Ir, where)


def test_id_base_and_unaligned_allow_bit0(knn):
    """Device ABI: a global bitmap read from bit 37 on, ids with an id base, exclusions in that id space."""
    import torch

    n, nq, d, k, bit0, base = 20000, 300, 256, 50, 37, 1000
    xb, xq = _data(n, nq, d, seed=77)
    rng = np.random.default_rng(4)
    glob = rng.random(bit0 + n + 50) < 0.4
    allowed = glob[bit0:bit0 + n].copy()
    ex = np.where(rng.random(nq) < 0.7, rng.integers(0, n, nq) + base, -1).astype(np.int64)
    ex[:5] = np.flatnonzero(allowed)[:5] + base
    idx = _index(knn, xb, L2)
    words = torch.from_numpy(np.packbits(np.concatenate([glob, np.zeros((-len(glob)) % 32, bool)]), bitorder="little").view("<u4").view(np.int32).copy()).cuda()
    ex_d = torch.from_numpy(ex).cuda()
    xq_d = torch.from_numpy(xq).cuda()
    D = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    I = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    c = knn._lib.SearchParamsC(words.data_ptr(), bit0, len(glob), ex_d.data_ptr())
    lib = knn._lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    for path in (2, 1):
        idx.set_param("path", path)
        knn._lib.check(lib.knn_index_search_params_dev(idx._h, nq, xq_d.data_ptr(), F32, k, D.data_ptr(), I.data_ptr(),
                                                       base, ctypes.byref(c), stream))
        Dr, Ir = _oracle(knn, xb, xq, k, L2, allowed, exclude=ex, id_base=base)
        _eq(_np(D), _np(I), Dr, Ir, "path %d" % path)
    # IndexFlat.search with id_base: exclusions are given in the returned id space on both paths
    for x in (xq, xq_d):
        Dp, Ip = idx.search(x, k, base, exclude=ex)
        Dr, Ir = _oracle(knn, xb, xq, k, L2, np.ones(n, bool), exclude=ex, id_base=base)
        _eq(_np(Dp), _np(Ip), Dr, Ir, "IndexFlat id_base")


# ---- 2. fewer eligible rows than k, and none -------------------------------------------------------------------
@pytest.mark.parametrize("path", [1, 2])
@pytest.mark.parametrize("metric", [IP, L2])
@pytest.mark.parametrize("n_allowed", [0, 7, 999])
def test_fewer_eligible_rows_than_k(knn, path, metric, n_allowed):
    import torch

    n, nq, d, k = 20000, 200, 256, 1000
    xb, xq = _data(n, nq, d, seed=n_allowed)
    allowed = np.zeros(n, bool)
    allowed[np.random.default_rng(1).choice(n, n_allowed, replace=False)] = True
    ex = np.where(np.arange(nq) % 2 == 0, np.flatnonzero(allowed)[0] if n_allowed else 5, -1).astype(np.int64)
    idx = _index(knn, xb, metric, {"path": path})
    p = knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed)))
    for x in (xq, torch.from_numpy(xq).cuda()):
        D, I = idx.search(x, k, params=p, exclude=ex)
        D, I = _np(D), _np(I)
        Dr, Ir = _oracle(knn, xb, xq, k, metric, allowed, exclude=ex)
        _eq(D, I, Dr, Ir)
        pad = -np.finfo(np.float32).max if metric == IP else np.finfo(np.float32).max
        for q in range(nq):
            n_q = n_allowed - (1 if ex[q] >= 0 and n_allowed and allowed[ex[q]] else 0)
            assert (I[q, n_q:] == -1).all() and (D[q, n_q:] == pad).all()
            assert allowed[I[q, :n_q]].all() and ex[q] not in I[q, :n_q]


# ---- 3. excluded rows that would win ----------------------------------------------------------------------------
@pytest.mark.parametrize("nq", [40, 300])
@pytest.mark.parametrize("metric", [IP, L2])
def test_masked_duplicates_of_the_queries_never_appear(knn, nq, metric):
    n, d, k = 30000, 512, 10
    xb, xq = _data(n, nq, d, seed=nq + metric)
    pos = np.random.default_rng(2).choice(n, nq, replace=False)
    xb[pos] = xq  # every query's exact duplicate: its top hit on both metrics
    allowed = np.ones(n, bool)
    allowed[pos] = False
    idx = _index(knn, xb, metric)
    D, I = idx.search(xq, k, params=knn.SearchParameters(sel=knn.IDSelectorNot(knn.IDSelectorBatch(pos))))
    assert not np.isin(I, pos).any()
    Dr, Ir = _oracle(knn, xb, xq, k, metric, allowed)
    _eq(D, I, Dr, Ir)
    assert idx.stat("overflow_queries") == 0


# ---- 4. all-vs-all with exclude = arange(n) ---------------------------------------------------------------------
@pytest.mark.parametrize("n,d,k,metric", [(14433, 1024, 1000, IP), (14433, 1024, 1000, L2), (40000, 256, 100, IP)],
                         ids=["c2-ip-dense", "c2-l2-dense", "multi-panel"])
def test_all_vs_all_excludes_the_self_row(knn, n, d, k, metric):
    import torch

    xb, _ = _data(n, 1, d, seed=n + metric)
    dup = np.arange(0, n, 1000)
    xb[dup + 1] = xb[dup]  # row i + 1 duplicates row i: i's duplicate must be returned, i itself never
    idx = _index(knn, xb, metric)
    ex = np.arange(n, dtype=np.int64)
    xd = torch.from_numpy(xb).cuda()
    D, I = idx.search(xd, k, exclude=torch.from_numpy(ex).cuda())
    D, I = _np(D), _np(I)
    assert not (I == ex[:, None]).any()
    assert (I[dup, 0] == dup + 1).all() and (I[dup + 1, 0] == dup).all()
    Dr, Ir = _oracle(knn, xb, xb, k, metric, np.ones(n, bool), exclude=ex)
    _eq(D, I, Dr, Ir, "all-vs-all")
    # the search-(k+1)-and-drop-column-0 workaround gets the duplicated rows wrong (ties: the lower id comes first)
    Dk, Ik = idx.search(xd, k + 1)
    assert (_np(Ik)[dup + 1, 1:] != I[dup + 1]).any()
    # combined with a selector
    allowed = _mask(n, 0.5, seed=1)
    D, I = idx.search(xd, k, params=knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed))),
                      exclude=torch.from_numpy(ex).cuda())
    Dr, Ir = _oracle(knn, xb, xb, k, metric, allowed, exclude=ex)
    _eq(_np(D), _np(I), Dr, Ir, "all-vs-all + selector")


# ---- 5. overflow repair with filters ------------------------------------------------------------------------------
@pytest.mark.parametrize("where", ["device", "host"])
def test_overflow_repair_honours_both_filters(knn, where):
    import torch

    nb, d, k, nq = 40000, 64, 10, 128
    row = np.random.default_rng(2).standard_normal(d).astype(np.float32)
    xb = np.tile(row, (nb, 1))
    xq = np.tile(row, (nq, 1))
    allowed = np.arange(nb) % 2 == 1
    ex = np.full(nq, -1, np.int64)
    ex[::2] = 1  # the first allowed row
    idx = _index(knn, xb, IP, {"path": 2})
    p = knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed)))
    x = torch.from_numpy(xq).cuda() if where == "device" else xq
    D, I = idx.search(x, k, params=p, exclude=ex)
    I = _np(I)
    assert idx.stat("overflow_queries") == nq
    first = np.flatnonzero(allowed)
    for q in range(nq):
        want = first[1:k + 1] if ex[q] == 1 else first[:k]
        assert np.array_equal(I[q], want), (q, I[q], want)


# ---- 6. adversarial error-bound data with a selector ---------------------------------------------------------------
@pytest.mark.parametrize("metric", [IP, L2])
@pytest.mark.parametrize("nq", [48, 300])
def test_adversarial_rows_with_a_selector(knn, metric, nq):
    case = adv.dy_aligned(nq, 1024, 10, metric=metric, seed=91 + nq + metric)
    n = case.xb.shape[0]
    allowed = np.ones(n, bool)
    rng = np.random.default_rng(nq)
    allowed[rng.choice(case.decoys.ravel(), case.decoys.size // 3, replace=False)] = False
    allowed[rng.choice(case.hidden.ravel(), max(1, case.hidden.size // 4), replace=False)] = False
    idx = _index(knn, case.xb, metric, {"path": 2})
    D, I = idx.search(case.xq, case.k, params=knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed))))
    assert idx.stat("overflow_queries") == 0
    Dr, Ir = _oracle(knn, case.xb, case.xq, case.k, metric, allowed, params={"path": 2})
    _eq(D, I, Dr, Ir)
    idx.set_param("path", 1)
    D1, I1 = idx.search(case.xq, case.k, params=knn.SearchParameters(sel=knn.IDSelectorBatch(np.flatnonzero(allowed))))
    _eq(D1, I1, Dr, Ir, "exact path")


# ---- 7. the batch-wise two-phase ABI on virtual shards --------------------------------------------------------------
def _pipelined_filtered(knn, shards, starts, xq, k, n_global, sel, ex):
    import torch

    G = len(shards)
    geo = [sh.search_begin(xq, k, params=knn.SearchParameters(sel=sel), exclude=ex, id_base=a, allow_bit0=a,
                           allow_nbits=n_global) for sh, a in zip(shards, starts)]
    nbatches = geo[0][0]
    bounds = [torch.zeros((nbatches, 2, rows), dtype=torch.float32, device="cuda") for _, rows in geo]
    nq = xq.shape[0]
    D = [torch.empty((nq, k), dtype=torch.float32, device="cuda") for _ in shards]
    I = [torch.empty((nq, k), dtype=torch.int64, device="cuda") for _ in shards]
    j = -(-k // G)
    for b in range(nbatches):
        for sh, bd in zip(shards, bounds):
            sh.search_filter_batch(b, j, bd)
        m = torch.stack([bd[b] for bd in bounds]).amax(0)
        for sh, bd, Ds, Is, a in zip(shards, bounds, D, I, starts):
            bd[b].copy_(m)
            sh.search_finish_batch(b, bd, Ds, Is, a)
    for sh, Ds, Is, a in zip(shards, D, I, starts):
        sh.search_end(Ds, Is, a)
    return knn.merge_topk(torch.stack(D), torch.stack(I), shards[0].metric_type)


@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("metric,k", [(IP, 10), (L2, 100), (IP, 1000)])
def test_two_phase_virtual_shards_with_filters(knn, G, metric, k):
    import torch

    n, nq, d = 48000, 700, 256
    xb, xq = _data(n, nq, d, seed=G * 10 + k)
    cuts = np.linspace(0, n, G + 1).astype(int)
    allowed = _mask(n, 0.5, seed=G)
    allowed[cuts[0]:cuts[1]] = False                     # shard 0: no eligible rows
    allowed[cuts[1]:cuts[2]] = False
    allowed[cuts[1] + np.arange(3) * 11] = True          # shard 1: fewer than j eligible rows
    ex = np.where(np.arange(nq) % 3 == 0, np.random.default_rng(5).integers(0, n, nq), -1).astype(np.int64)
    ex[1] = np.flatnonzero(allowed)[0]
    sel = knn.IDSelectorBatch(np.flatnonzero(allowed))
    shards = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        sh = knn.IndexFlat(d, metric, device=0)
        sh.set_param("query_batch", 256)
        sh.add(xb[a:b])
        shards.append(sh)
    xq_d = torch.from_numpy(xq).cuda()
    ex_d = torch.from_numpy(ex).cuda()
    Dm, Im = _pipelined_filtered(knn, shards, list(cuts[:-1]), xq_d, k, n, sel, ex_d)
    single = _index(knn, xb, metric)
    D1, I1 = single.search(xq_d, k, params=knn.SearchParameters(sel=sel), exclude=ex_d)
    assert torch.equal(Im, I1) and torch.equal(Dm, D1)
    Dr, Ir = _oracle(knn, xb, xq, k, metric, allowed, exclude=ex)
    _eq(_np(Dm), _np(Im), Dr, Ir)


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    from datetime import timedelta

    import torch
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=60))
    torch.cuda.set_device(0)
    import knn_b200
    from knn_b200.distributed import ShardedIndexFlat

    done = []
    n, d, nq = 16000, 64, 500
    xb, xq = _data(n, nq, d, seed=12)
    allowed = _mask(n, 0.3, seed=2)
    ex = np.where(np.arange(nq) % 2 == 0, np.arange(nq) * 7, -1).astype(np.int64)
    for metric, k in ((IP, 10), (L2, 100)):
        index = ShardedIndexFlat(d, metric, device=0, shard_weights=[1.2, 0.8])
        index.local.set_param("query_batch", 256)
        index.add(torch.from_numpy(xb).cuda())
        single = knn_b200.IndexFlat(d, metric, device=0)
        single.add(xb)
        p = knn_b200.SearchParameters(sel=knn_b200.IDSelectorBatch(np.flatnonzero(allowed)))
        D, I = index.search(torch.from_numpy(xq).cuda(), k, params=p, exclude=ex)
        D1, I1 = single.search(torch.from_numpy(xq).cuda(), k, params=p, exclude=ex)
        assert torch.equal(I, I1) and torch.equal(D, D1), (rank, metric, k)
        done.append((rank, metric, k))
        index.close()
        dist.barrier()
    (Path(out_dir) / ("rank%d" % rank)).write_text(repr(done))
    dist.destroy_process_group()


def test_sharded_index_filtered_two_processes_one_gpu(tmp_path):
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=False)
    deadline = time.time() + 180
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("two-process filtered sharded search did not finish in 180 s")
    done = [eval((tmp_path / ("rank%d" % r)).read_text()) for r in range(2)]
    assert len(done[0]) == len(done[1]) == 2


# ---- 8. misuse ------------------------------------------------------------------------------------------------------
def test_misuse_returns_invalid_and_the_index_stays_usable(knn):
    import torch

    n, nq, d, k = 20000, 300, 128, 10
    xb, xq = _data(n, nq, d, seed=1)
    idx = _index(knn, xb, IP)
    lib = knn._lib.load()
    xq_d = torch.from_numpy(xq).cuda()
    D = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    I = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    words = torch.zeros(((n + 31) // 32,), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    for bit0, nbits in ((-1, n), (0, -5)):
        c = knn._lib.SearchParamsC(words.data_ptr(), bit0, nbits, None)
        rc = lib.knn_index_search_params_dev(idx._h, nq, xq_d.data_ptr(), F32, k, D.data_ptr(), I.data_ptr(), 0,
                                             ctypes.byref(c), stream)
        assert rc == ERR_INVALID and b"must not be negative" in lib.knn_last_error()
    host_words = np.zeros((n + 31) // 32, np.uint32)
    c = knn._lib.SearchParamsC(host_words.ctypes.data, 0, n, None)  # a host bitmap in a device call
    assert lib.knn_index_search_params_dev(idx._h, nq, xq_d.data_ptr(), F32, k, D.data_ptr(), I.data_ptr(), 0,
                                           ctypes.byref(c), stream) == ERR_INVALID
    c = knn._lib.SearchParamsC(words.data_ptr(), 0, n, None)  # a device bitmap in a host call
    Dh, Ih = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    assert lib.knn_index_search_params(idx._h, nq, xq.ctypes.data, F32, k, Dh.ctypes.data, Ih.ctypes.data,
                                       ctypes.byref(c)) == ERR_INVALID
    # finish_batch / end with an id_base other than begin_params's
    ex = torch.full((nq,), -1, dtype=torch.int64, device="cuda")
    nb, rows = idx.search_begin(xq_d, k, exclude=ex, id_base=100)
    bounds = torch.zeros((nb, 2, rows), dtype=torch.float32, device="cuda")
    idx.search_filter_batch(0, k, bounds)
    assert lib.knn_index_search_finish_batch_dev(idx._h, 0, bounds.data_ptr(), D.data_ptr(), I.data_ptr(), 0, stream) == ERR_INVALID
    assert b"id_base" in lib.knn_last_error()
    for b in range(nb):
        if b:
            idx.search_filter_batch(b, k, bounds)
        idx.search_finish_batch(b, bounds, D, I, 100)
    assert lib.knn_index_search_end_dev(idx._h, D.data_ptr(), I.data_ptr(), 0, stream) == ERR_INVALID
    idx.search_end(D, I, 100)
    # still usable: an unfiltered and a filtered search give the oracle's answer
    D0, I0 = idx.search(xq, k)
    Dr, Ir = _oracle(knn, xb, xq, k, IP, np.ones(n, bool))
    _eq(D0, I0, Dr, Ir)
    with pytest.raises(NotImplementedError, match="ShardedIndexFlat"):
        from knn_b200.distributed import GridIndexFlat

        GridIndexFlat.search(object.__new__(GridIndexFlat), xq, k, exclude=np.zeros(nq, np.int64))
