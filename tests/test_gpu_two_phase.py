"""The pipelined two-phase sharded search on ONE GPU: the path every row-sharded multi-GPU search takes
(ShardedIndexFlat._two_phase_pipelined, the batch-wise C ABI knn_index_search_{begin,filter_batch,finish_batch,end}_dev
and the bound exchange over peer memory, knn_bounds_push_peer_dev / knn_bounds_wait_max_dev).

a. the bound-exchange kernels with G virtual ranks on cuda:0 against a torch max;
b. BoundsExchange itself, with G virtual ranks sharing torch buffers instead of IPC mappings;
c. the batch-wise ABI on G shards in one process, step for step as _two_phase_pipelined runs it, against one unsharded
   index (bit for bit) and the CPU oracle - with shards that take different paths (tensor-core filter, exact scan, empty);
d. misuse of the batch-wise ABI returns an error;
e. the real ShardedIndexFlat, two processes on cuda:0 over gloo, with one shard on the exact path.

Every pushed bound is enqueued before any wait on the same stream, so no wait kernel ever spins."""
import ctypes
import os
import socket
import sys
import time
import zlib
from pathlib import Path

import numpy as np
import pytest

from oracle import flat_oracle as fo
from oracle.parity import check_parity

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent
FLT_MAX = float(np.finfo(np.float32).max)
IP, L2 = 0, 1
ERR_INVALID = -1


@pytest.fixture(scope="module")
def knn():
    import knn_b200

    assert knn_b200._lib.load().knn_device_count() >= 1, "no CUDA device: the CUDA path cannot run"
    return knn_b200


def _stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def _ptrs(ts):
    return (ctypes.c_void_p * len(ts))(*[t if isinstance(t, int) else t.data_ptr() for t in ts])


# ---- a. bound-exchange kernels ------------------------------------------------------------------------------------
def _bound_values(gen, G, n, shard):
    """2 * rows style bounds of one virtual rank: random scores, extremes, and now and then the exact-path fill."""
    import torch

    v = torch.randn(n, device="cuda", generator=gen) * 10
    special = torch.tensor([FLT_MAX, -FLT_MAX, float("inf"), float("-inf"), 0.0, -0.0], device="cuda")
    pick = torch.randint(0, 8, (n,), device="cuda", generator=gen)
    v = torch.where(pick < 6, special[pick.clamp(max=5)], v) if shard % 2 else v
    if shard == G - 1 and G > 1:  # an exact-path shard: lower = -FLT_MAX, negated j-bound = +FLT_MAX
        h = n // 2
        v[:h] = -FLT_MAX
        v[h:] = FLT_MAX
    if shard == 0:  # -inf everywhere on one rank: the kernel's -FLT_MAX start value must show through where all agree
        v[: max(1, n // 7)] = float("-inf")
    return v


def _expected_max(srcs):
    import torch

    return torch.stack(srcs).amax(0).clamp(min=-FLT_MAX)


@pytest.mark.parametrize("G", [1, 2, 3, 8, 16])
def test_bounds_push_wait_max_kernels_equal_torch_max(knn, G):
    import torch

    lib = knn._lib.load()
    nmax = 2 * 16384
    gen = torch.Generator(device="cuda").manual_seed(G)
    slots = [torch.full((G * nmax,), 123.0, device="cuda") for _ in range(G)]  # [rank][n] per virtual rank
    flags = [torch.zeros(G, dtype=torch.int32, device="cuda") for _ in range(G)]
    counters = [torch.zeros(1, dtype=torch.int32, device="cuda") for _ in range(G)]  # one per rank, reused by every call
    timeout = torch.zeros(1, dtype=torch.int32, device="cuda")
    # largest n first: later epochs leave stale data of the previous, larger n behind in the slots
    for epoch, n in enumerate([2 * 16384, 257, 256, 255, 1, 2 * 16384, 1], start=1):
        srcs = [_bound_values(gen, G, n, r) for r in range(G)]
        # slots_peer[l] = rank l's slot array for this n: slot [rank] of it starts at rank * n
        for r in range(G):
            assert lib.knn_bounds_push_peer_dev(G, r, n, srcs[r].data_ptr(), _ptrs(slots), _ptrs(flags), epoch,
                                                counters[r].data_ptr(), _stream()) == 0, knn._lib.load().knn_last_error()
        outs = [torch.full((n,), 7.0, device="cuda") for _ in range(G)]
        for r in range(G):
            assert lib.knn_bounds_wait_max_dev(G, n, slots[r].data_ptr(), flags[r].data_ptr(), epoch, outs[r].data_ptr(),
                                               timeout.data_ptr(), _stream()) == 0
        want = _expected_max(srcs)
        for r in range(G):
            assert torch.equal(outs[r], want), (G, n, epoch, r)
            assert torch.equal(slots[r][:G * n].view(G, n), torch.stack(srcs)), "slot layout [rank][n]"
            assert flags[r].tolist() == [epoch] * G
        assert int(timeout.item()) == 0
        assert all(int(c.item()) == 0 for c in counters), "the push kernel resets its arrival counter"


def test_bounds_kernels_reject_invalid_arguments(knn):
    import torch

    lib = knn._lib.load()
    buf = torch.zeros(64, device="cuda")
    flag = torch.zeros(17, dtype=torch.int32, device="cuda")
    ctr = torch.zeros(1, dtype=torch.int32, device="cuda")
    p = buf.data_ptr()
    slots17, flags17 = _ptrs([p] * 17), _ptrs([flag.data_ptr()] * 17)
    push = lambda G, r, n, src=p, sl=slots17, fl=flags17, c=ctr.data_ptr(): lib.knn_bounds_push_peer_dev(  # noqa: E731
        G, r, n, src, sl, fl, 1, c, None)
    assert push(0, 0, 4) == ERR_INVALID
    assert push(17, 0, 4) == ERR_INVALID
    assert push(2, -1, 4) == ERR_INVALID
    assert push(2, 2, 4) == ERR_INVALID
    assert push(2, 0, 0) == ERR_INVALID
    assert push(2, 0, -3) == ERR_INVALID
    assert push(2, 0, 4, src=None) == ERR_INVALID
    assert push(2, 0, 4, sl=None) == ERR_INVALID
    assert push(2, 0, 4, fl=None) == ERR_INVALID
    assert push(2, 0, 4, c=None) == ERR_INVALID
    assert push(2, 0, 4, sl=_ptrs([p, 0])) == ERR_INVALID
    assert push(2, 0, 4, fl=_ptrs([flag.data_ptr(), 0])) == ERR_INVALID
    wait = lambda G, n, sl=p, fl=flag.data_ptr(), out=p, t=ctr.data_ptr(): lib.knn_bounds_wait_max_dev(  # noqa: E731
        G, n, sl, fl, 1, out, t, None)
    assert wait(0, 4) == ERR_INVALID
    assert wait(17, 4) == ERR_INVALID
    assert wait(2, 0) == ERR_INVALID
    assert wait(2, -1) == ERR_INVALID
    assert wait(2, 4, sl=None) == ERR_INVALID
    assert wait(2, 4, fl=None) == ERR_INVALID
    assert wait(2, 4, out=None) == ERR_INVALID
    assert wait(2, 4, t=None) == ERR_INVALID
    torch.cuda.synchronize()
    assert torch.count_nonzero(buf) == 0 and torch.count_nonzero(flag) == 0  # nothing was launched


# ---- b. BoundsExchange with G virtual ranks -----------------------------------------------------------------------
class _SharedBuffers:
    """Stands in for PeerExchange: G torch buffers on cuda:0, every virtual rank sees all of them."""

    def __init__(self, bufs, rank):
        self.bufs, self.rank = bufs, rank
        self.bases = [b.data_ptr() for b in bufs]
        self._own_tensor = bufs[rank]
        self.capacity = bufs[rank].numel()

    def ensure(self, nbytes):
        assert nbytes <= self.capacity

    def barrier(self):
        import torch

        torch.cuda.synchronize()

    def close(self):
        pass


def _virtual_exchanges(G):
    import torch

    from knn_b200.distributed import BoundsExchange

    nbytes = 1024 * G * 4 + BoundsExchange.MAX_QUERY_ROWS * 2 * G * 4
    bufs = [torch.full((nbytes,), 0xAB, dtype=torch.uint8, device="cuda") for _ in range(G)]
    return bufs, [BoundsExchange(None, None, r, G, 0, exchange=_SharedBuffers(bufs, r)) for r in range(G)]


@pytest.mark.parametrize("G", [2, 3, 8])
def test_bounds_exchange_push_then_wait_with_virtual_ranks(knn, G):
    import torch

    bufs, bxs = _virtual_exchanges(G)
    assert all(torch.count_nonzero(b) == 0 for b in bufs), "the constructor zeroes the rank's buffer"
    gen = torch.Generator(device="cuda").manual_seed(100 + G)
    # searches of different geometry on the same buffers: epochs advance, stale slots of larger searches stay behind
    for nbatches, rows in [(3, 256), (1, 768), (9, 256), (1, 1), (2, 16384), (1, 257)]:
        for bx in bxs:
            bx.begin(nbatches, rows)
        n = 2 * rows
        srcs = [torch.stack([_bound_values(gen, G, n, r) for _ in range(nbatches)]).view(nbatches, 2, rows) for r in range(G)]
        work = [s.clone() for s in srcs]
        for b in range(nbatches):        # every batch of every rank pushed before any wait
            for r, bx in enumerate(bxs):
                bx.push(b, work[r][b])
        for b in range(nbatches):
            for r, bx in enumerate(bxs):
                bx.wait_max(b, work[r][b])
        torch.cuda.synchronize()
        want = _expected_max([s.view(nbatches, n) for s in srcs]).view(nbatches, 2, rows)
        for r, bx in enumerate(bxs):
            bx.check()
            assert torch.equal(work[r], want), (G, nbatches, rows, r)
            own = bufs[r]
            for b in range(nbatches):  # slots [batch][rank][2 * rows], flags [batch][rank] = epoch
                off = bx.slots_off + b * G * n * 4
                slot = own[off:off + G * n * 4].view(torch.float32).view(G, n)
                assert torch.equal(slot, torch.stack([s[b].reshape(n) for s in srcs])), (r, b)
                fl = own[bx.flags_off + b * G * 4:bx.flags_off + (b + 1) * G * 4].view(torch.int32)
                assert fl.tolist() == [bx.epoch] * G
    assert [bx.epoch for bx in bxs] == [6] * G
    with pytest.raises(ValueError):
        bxs[0].begin(2, bxs[0].MAX_QUERY_ROWS)


def test_bounds_exchange_max_over_ranks_is_push_then_wait(knn):
    """With one rank, max_over_ranks (push + wait) is the identity clamped at -FLT_MAX."""
    import torch

    bufs, (bx,) = _virtual_exchanges(1)
    bx.begin(2, 300)
    gen = torch.Generator(device="cuda").manual_seed(5)
    for b in range(2):
        v = _bound_values(gen, 2, 600, 0)
        out = v.clone()
        bx.max_over_ranks(b, out)
        torch.cuda.synchronize()
        assert torch.equal(out, v.clamp(min=-FLT_MAX))
    bx.check()


# ---- c. the batch-wise ABI on G shards, as _two_phase_pipelined runs it ------------------------------------------
# Queries placed near a given row get this much Gaussian noise per coordinate, per metric.  Inner product: little, so
# that the row (and its copies) scores ~|y|^2, far ahead of the rest.  L2: enough that the distance (~64 at d = 64) is
# not tiny against |x|^2 + |y|^2 (~250) while the row still leads every other candidate by far.  At a distance of ~0.1
# the oracle's fp32 |x|^2 + |y|^2 - 2<x,y> cancels to a few ulp of 250, more than the parity rule's tau/8 floor at
# d = 64 allows, and how many ulp depends on the host BLAS's summation order.
NEAR = {IP: 0.05, L2: 1.0}


def _data(n, d, nq, seed, metric, clump=None):
    """Clustered rows (many near-equal scores), a row duplicated around every shard boundary and queries on it."""
    rng = np.random.default_rng(seed)
    centers = rng.standard_normal((20, d)).astype(np.float32)
    xb = (centers[rng.integers(0, 20, n)] + 0.7 * rng.standard_normal((n, d))).astype(np.float32)
    xq = (centers[rng.integers(0, 20, nq)] + 0.7 * rng.standard_normal((nq, d))).astype(np.float32)
    if clump is not None:  # identical rows inside one shard, queries on them: their candidate lists overflow
        a, b = clump
        xb[a:b] = xb[a]
        xq[1::5] = xb[a] + NEAR[metric] * rng.standard_normal((len(xq[1::5]), d)).astype(np.float32)
    return xb, xq


def _shard_rows(mix, G, k):
    """Rows per shard and the path param per shard (0 automatic) for one shard mix."""
    big, small = 9000, 5000  # >= tensor_min_n (8192) and below it
    rows, path = [big] * G, [0] * G
    if mix.startswith("small@"):
        at = {"first": 0, "mid": G // 2, "last": G - 1}[mix[6:]]
        rows[at] = small
    elif mix == "lt_k":  # the tensor path forced everywhere: only ntotal < k sends that shard to the exact scan
        rows[G // 2] = max(0, k - 37)
        path = [2] * G
    elif mix == "empty":
        rows[G - 1 if G == 2 else 1] = 0
    elif mix == "path1":
        path[0] = 1
    elif mix == "clump":
        rows[1] = 12000
    return rows, path


def _pipelined(knn, shards, starts, xq, k, combine):
    """ShardedIndexFlat._two_phase_pipelined with the G ranks as G shards of one process: filter of batch b on a
    high-priority main stream, combine + finish on a low-priority side stream, end, then the merge.  Like the real
    code, the BoundsExchange combine lays out every rank's slots from that rank's own (nbatches, rows); only the
    number of batches must agree (a wait for a batch that is never pushed would spin).  Returns (D, I, geometries)."""
    import torch

    G = len(shards)
    caller = torch.cuda.current_stream()
    side, main = torch.cuda.Stream(priority=0), torch.cuda.Stream(priority=-1)
    nq = xq.shape[0]
    main.wait_stream(caller)
    with torch.cuda.stream(main):
        geo = [sh.search_begin(xq, k) for sh in shards]
        assert len({g[0] for g in geo}) == 1, "shards report different numbers of batches: %s" % (geo,)
        if combine == "torch":
            assert len(set(geo)) == 1, "shards report different batch geometry (nbatches, rows): %s" % (geo,)
        nbatches = geo[0][0]
        bx = None
        if combine == "exchange":
            _, bx = _virtual_exchanges(G)
            for x, (_, rows) in zip(bx, geo):
                x.begin(nbatches, rows)
        bounds = [torch.zeros((nbatches, 2, rows), dtype=torch.float32, device="cuda") for _, rows in geo]
        D = [torch.empty((nq, k), dtype=torch.float32, device="cuda") for _ in shards]
        I = [torch.empty((nq, k), dtype=torch.int64, device="cuda") for _ in shards]
        j = -(-k // G)
        side.wait_stream(main)
        for b in range(nbatches):
            for sh, bd in zip(shards, bounds):
                sh.search_filter_batch(b, j, bd)
            filtered = torch.cuda.Event()
            filtered.record(main)
            with torch.cuda.stream(side):
                side.wait_event(filtered)
                if bx is None:
                    m = torch.stack([bd[b] for bd in bounds]).amax(0)
                    for bd in bounds:
                        bd[b].copy_(m)
                else:
                    for x, bd in zip(bx, bounds):
                        x.push(b, bd[b])
                    for x, bd in zip(bx, bounds):
                        x.wait_max(b, bd[b])
                for sh, bd, Ds, Is, a in zip(shards, bounds, D, I, starts):
                    sh.search_finish_batch(b, bd, Ds, Is, a)
        main.wait_stream(side)
        for sh, Ds, Is, a in zip(shards, D, I, starts):
            sh.search_end(Ds, Is, a)
    caller.wait_stream(main)
    Dm, Im = knn.merge_topk(torch.stack(D), torch.stack(I), shards[0].metric_type)
    torch.cuda.synchronize()
    if bx is not None:
        for x in bx:
            x.check()
    return Dm, Im, geo


# (metric, k, nq, query_batch (None: default), G, shard mix, operand format (None: automatic), d)
PIPE_CASES = [
    (IP, 10, 700, 256, 2, "tensor", None, 64),
    (L2, 10, 700, None, 2, "small@last", None, 64),     # one batch, rows 768 vs 700: the tensor shard read +FLT_MAX
    (IP, 100, 700, None, 3, "small@last", None, 64),    # [tensor, tensor, exact]
    (L2, 10, 700, None, 3, "small@first", None, 64),
    (IP, 10, 700, 256, 3, "small@first", None, 64),     # 3 batches against 1
    (L2, 100, 525, 256, 3, "small@mid", None, 64),
    (IP, 1, 1, None, 2, "small@last", None, 64),
    (L2, 10, 255, None, 3, "tensor", None, 64),
    (IP, 10, 256, None, 3, "small@mid", None, 64),      # nq a multiple of 256: same geometry on every path
    (L2, 10, 257, 256, 8, "small@first", None, 64),
    (IP, 1, 700, 256, 8, "small@last", None, 64),
    (IP, 1000, 700, 256, 2, "lt_k", None, 64),
    (L2, 2048, 257, None, 3, "lt_k", None, 64),
    (IP, 100, 700, 256, 3, "empty", None, 64),
    (L2, 10, 1, None, 8, "empty", None, 64),
    (IP, 10, 525, 256, 2, "path1", None, 64),
    (L2, 1000, 257, 256, 3, "path1", None, 64),
    (IP, 100, 525, 256, 8, "tensor", None, 64),
    (L2, 2048, 256, None, 2, "tensor", None, 64),
    (IP, 2048, 525, 256, 2, "small@first", None, 64),
    (IP, 100, 700, 256, 3, "small@mid", "bf16", 64),
    (L2, 10, 525, 256, 3, "small@last", "fp16", 64),
    (L2, 1000, 256, None, 2, "tensor", "fp16", 64),
    (IP, 10, 257, 256, 3, "clump", None, 64),
    (L2, 10, 700, None, 2, "clump", "bf16", 64),
    (IP, 100, 257, 256, 2, "small@last", None, 1024),
]


def _case_id(c):
    metric, k, nq, qb, G, mix, fmt, d = c
    return "%s-k%d-nq%d-qb%s-G%d-%s-%s-d%d" % ("ip" if metric == IP else "l2", k, nq, qb or "def", G, mix, fmt or "auto", d)


@pytest.mark.parametrize("combine", ["torch", "exchange"])
@pytest.mark.parametrize("case", PIPE_CASES, ids=[_case_id(c) for c in PIPE_CASES])
def test_batchwise_two_phase_on_mixed_shards_equals_unsharded(knn, case, combine):
    import torch

    metric, k, nq, qb, G, mix, fmt, d = case
    rows, path = _shard_rows(mix, G, k)
    starts = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    n = int(starts[-1])
    clump = (int(starts[1]) + 500, int(starts[1]) + 9500) if mix == "clump" else None
    xb, xq = _data(n, d, nq, seed=zlib.crc32(_case_id(case).encode()) % 1000, metric=metric, clump=clump)
    for a in starts[1:-1]:  # one row duplicated across every shard boundary (ties broken by global id)
        xb[max(0, a - 2):a + 2] = xb[3]
    xq[0] = xb[3] + NEAR[metric] * np.random.default_rng(1).standard_normal(d).astype(np.float32)

    def make(p, rows_):
        idx = knn.IndexFlat(d, metric, device=0)
        idx.set_param("path", p)
        if qb:
            idx.set_param("query_batch", qb)
        if fmt:
            idx.set_param("shadow_fmt", {"bf16": 1, "fp16": 2}[fmt])
        if rows_.shape[0]:
            idx.add(torch.from_numpy(rows_).cuda())
        return idx

    tq = torch.from_numpy(xq).cuda()
    full = make(2, xb)
    D1, I1 = full.search(tq, k)
    assert int(full.stat("path")) == 2
    exact = make(1, xb)
    De, Ie = exact.search(tq, k)
    assert torch.equal(I1, Ie) and torch.equal(D1, De), "unsharded tensor path differs from the exact scan"
    expect_path = [1 if p == 1 or r < k or (p == 0 and r < 8192) else 2 for p, r in zip(path, rows)]
    sample = np.unique(np.concatenate([[0, nq // 2, nq - 1], np.random.default_rng(nq).integers(0, nq, 24)]))
    shards = [make(p, xb[a:a + r]) for p, a, r in zip(path, starts, rows)]
    Dm, Im, geo = _pipelined(knn, shards, [int(a) for a in starts[:-1]], tq, k, combine)
    assert [int(sh.stat("path")) for sh in shards] == expect_path, "the case does not mix the paths it names"
    if mix == "clump":
        assert shards[1].stat("overflow_queries") > 0, "no candidate list overflowed: the repair went untested"
    bad = (Im != I1).any(1) | (Dm != D1).any(1)
    assert not bad.any(), "%d of %d queries differ from the unsharded index, first %d last %d (geometry %s)" % (
        int(bad.sum()), nq, int(bad.nonzero()[0, 0]), int(bad.nonzero()[-1, 0]), geo)
    assert len(set(geo)) == 1, geo
    D_ref, I_ref = fo.knn_flat(xq[sample], xb, k, metric, want=k + 4)
    check_parity(Dm.cpu().numpy()[sample], Im.cpu().numpy()[sample], D_ref, I_ref, xq[sample], xb, metric)


@pytest.mark.parametrize("path,ntotal", [(0, 0), (0, 5000), (0, 9000), (1, 9000), (2, 9000), (2, 7)])
def test_batch_geometry_depends_only_on_nq_and_query_batch(knn, path, ntotal):
    """Every shard of a search must report the same (nbatches, batch_rows), whichever path it takes: the callers lay
    out the bound slots of all shards from it."""
    import torch

    idx = knn.IndexFlat(16, L2, device=0)
    idx.set_param("path", path)
    if ntotal:
        idx.add(np.random.default_rng(ntotal).standard_normal((ntotal, 16)).astype(np.float32))
    xq = torch.randn(700, 16, device="cuda")
    for qb in (256, 512, 16384):
        idx.set_param("query_batch", qb)
        for nq in (1, 255, 256, 257, 525, 700):
            rows = -(-min(qb, nq) // 256) * 256
            assert idx.search_begin(xq[:nq], 10) == (-(-nq // rows), rows), (qb, nq)
    idx.search_end(torch.empty((700, 10), device="cuda"), torch.empty((700, 10), dtype=torch.int64, device="cuda"))


# ---- d. misuse of the batch-wise ABI ------------------------------------------------------------------------------
@pytest.mark.parametrize("path", [1, 2])
def test_batchwise_abi_misuse_returns_an_error(knn, path):
    import torch

    lib = knn._lib.load()
    rng = np.random.default_rng(9)
    idx = knn.IndexFlat(32, IP, device=0)
    idx.set_param("path", path)
    idx.set_param("query_batch", 256)
    idx.add(rng.standard_normal((10000, 32)).astype(np.float32))
    h, s = idx._h, _stream()
    xq = torch.from_numpy(rng.standard_normal((300, 32)).astype(np.float32)).cuda()
    k = 10
    bounds = torch.zeros((2, 2, 256), device="cuda")
    D = torch.empty((300, k), device="cuda")
    I = torch.empty((300, k), dtype=torch.int64, device="cuda")
    # nothing begun
    assert lib.knn_index_search_filter_batch_dev(h, 0, 1, bounds.data_ptr(), s) == ERR_INVALID
    assert lib.knn_index_search_finish_batch_dev(h, 0, bounds.data_ptr(), D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID
    assert lib.knn_index_search_end_dev(h, D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID
    nb, rows = idx.search_begin(xq, k)
    for b in (-1, nb, 1 << 40):
        assert lib.knn_index_search_filter_batch_dev(h, b, 1, bounds.data_ptr(), s) == ERR_INVALID
        assert lib.knn_index_search_finish_batch_dev(h, b, bounds.data_ptr(), D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID
    assert lib.knn_index_search_filter_batch_dev(h, 0, k + 1, bounds.data_ptr(), s) == ERR_INVALID  # j > k
    assert lib.knn_index_search_filter_batch_dev(h, 0, 1, None, s) == ERR_INVALID
    assert lib.knn_index_search_finish_batch_dev(h, 0, bounds.data_ptr(), None, I.data_ptr(), 0, s) == ERR_INVALID
    # the search is still usable after the rejected calls
    for b in range(nb):
        idx.search_filter_batch(b, k, bounds)
        idx.search_finish_batch(b, bounds, D, I)
    idx.search_end(D, I)
    assert lib.knn_index_search_end_dev(h, D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID  # end twice
    assert lib.knn_index_search_filter_batch_dev(h, 0, 1, bounds.data_ptr(), s) == ERR_INVALID  # after end
    assert lib.knn_index_search_finish_batch_dev(h, 0, bounds.data_ptr(), D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID
    D1, I1 = idx.search(xq, k)
    assert torch.equal(I, I1) and torch.equal(D, D1)


# ---- e. the real ShardedIndexFlat._two_phase_pipelined, two processes on cuda:0 -------------------------------------
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
    rng = np.random.default_rng(21)
    d = 64
    # (n, weights, metric, k values): rank 1 below tensor_min_n on the automatic path, below k = 1000, empty
    for n, weights, metric, ks in [(16000, [1.15, 0.85], IP, (10, 1000)), (16000, [1.15, 0.85], L2, (10,)),
                                   (10000, [1.9, 0.1], L2, (10, 1000)), (10000, [1.0, 1e-9], IP, (10,))]:
        centers = rng.standard_normal((20, d)).astype(np.float32)
        xb = (centers[rng.integers(0, 20, n)] + 0.7 * rng.standard_normal((n, d))).astype(np.float32)
        xq = (centers[rng.integers(0, 20, 700)] + 0.7 * rng.standard_normal((700, d))).astype(np.float32)
        xb_d, xq_d = torch.from_numpy(xb).cuda(), torch.from_numpy(xq).cuda()
        index = ShardedIndexFlat(d, metric, device=0, exchange_bounds=True, peer_merge=True, shard_weights=weights)
        assert index.pipeline_batches and not index.peer_bounds  # gloo: the bounds go through all_reduce
        index.local.set_param("query_batch", 256)
        cut = [n // 3, n // 3 + 1]                      # three add() segments: local -> global id mapping
        index.add(xb_d[:cut[0]])
        index.add(xb_d[cut[0]:cut[1]])
        index.add(xb_d[cut[1]:])
        single = knn_b200.IndexFlat(d, metric, device=0)
        single.add(xb_d)
        for k in ks:
            for nq in (700, 200):
                D, I = index.search(xq_d[:nq], k)
                D1, I1 = single.search(xq_d[:nq].contiguous(), k)
                path = int(index.local.stat("path"))
                tag = (rank, n, weights, metric, k, nq, index.local.ntotal, path)
                assert torch.equal(I, I1), ("ids differ from the unsharded index",) + tag
                assert torch.equal(D, D1), ("distances differ from the unsharded index",) + tag
                done.append(tag)
        index.close()
        dist.barrier()
    (Path(out_dir) / ("rank%d" % rank)).write_text(repr(done))
    dist.destroy_process_group()


def test_sharded_pipelined_search_with_an_exact_shard_two_processes_one_gpu(tmp_path):
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=False)
    deadline = time.time() + 180  # a geometry mismatch between the ranks must fail the test, not hang it
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("two-process sharded search did not finish in 180 s")
    done = [eval((tmp_path / ("rank%d" % r)).read_text()) for r in range(2)]
    assert len(done[0]) == len(done[1]) == 12
    assert all(t[7] == 2 for t in done[0]) and all(t[7] == 1 for t in done[1]), \
        "rank 0 must take the tensor path, rank 1 the exact scan: %s" % (done,)
