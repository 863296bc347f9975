"""world_size-2 gloo test (CPU) of the multi-GPU host logic: row split, local->global id
mapping across several add() calls, all-gather, merge call.  The per-shard search and the merge
kernel are CUDA-only in the product, so this test injects the oracle as the shard engine and a
numpy merge with the same tie rule - it checks the plumbing, not the kernels (those are covered
by tests/test_gpu_parity.py::test_torch_device_api_and_merge)."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = Path(__file__).resolve().parent.parent


class _OracleShard:
    def __init__(self, d, metric):
        from oracle import flat_oracle as fo

        self.ix = fo.IndexFlat(d, metric)
        self.device = 0

    @property
    def ntotal(self):
        return self.ix.ntotal

    def add(self, x):
        self.ix.add(np.ascontiguousarray(x, dtype=np.float32))

    def search(self, x, k):
        return self.ix.search(np.ascontiguousarray(x, dtype=np.float32), k)


def _merge_numpy(Dg, Ig, metric):
    w, nq, k = Dg.shape
    D = Dg.permute(1, 0, 2).reshape(nq, w * k).numpy()
    I = Ig.permute(1, 0, 2).reshape(nq, w * k).numpy()
    key = np.where(I < 0, np.inf, -D if metric == 0 else D)
    outD = np.empty((nq, k), np.float32)
    outI = np.empty((nq, k), np.int64)
    for r in range(nq):
        order = np.lexsort((I[r], key[r]))[:k]
        outD[r], outI[r] = D[r, order], I[r, order]
    return torch.from_numpy(outD), torch.from_numpy(outI)


def _worker(rank, world, port, metric, weights, out):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from knn_b200.distributed import ShardedIndexFlat
    from oracle import flat_oracle as fo

    rng = np.random.default_rng(0)
    xb = rng.standard_normal((1001, 32)).astype(np.float32)
    xq = rng.standard_normal((17, 32)).astype(np.float32)
    index = ShardedIndexFlat(32, metric, index_factory=lambda: _OracleShard(32, metric), merge_fn=_merge_numpy,
                             shard_weights=weights)
    index.add(xb[:300])      # three adds: ids must stay positions in the concatenation
    index.add(xb[300:301])
    index.add(xb[301:])
    assert index.ntotal == 1001
    if weights is None:
        assert index.local.ntotal in (500, 501)
    else:  # speed-proportional shards: rank 0 keeps ~30 % of every add
        assert abs(index.local.ntotal - 1001 * weights[rank] / sum(weights)) <= 2
    for k in (5, 1001 // 2, 1200):  # last one: k > ntotal -> -1 padding survives the merge
        D, I = index.search(xq, k)
        D_ref, I_ref = fo.knn_flat(xq, xb, k, metric)
        assert np.array_equal(I, I_ref), (rank, k)
        assert np.array_equal(D, D_ref), (rank, k)
    # queries every rank holds are uploaded in slices and all-gathered: same matrix on every rank
    xq_all = index.upload_queries(xq)
    assert xq_all.shape == xq.shape and np.array_equal(xq_all.numpy(), xq)
    assert np.array_equal(index.upload_queries(xq[:1]).numpy(), xq[:1])  # fewer rows than ranks
    index.TWO_PHASE_MAX_QUERIES = 5  # more queries than one two-phase call holds: processed in chunks (17 = 5+5+5+2)
    D, I = index.search(xq, 7)
    D_ref, I_ref = fo.knn_flat(xq, xb, 7, metric)
    # (the oracle's sgemm rounds differently for a different batch shape: scores to fp32 noise, ids exact)
    assert np.array_equal(I, I_ref) and np.allclose(D, D_ref, rtol=1e-6, atol=1e-6)
    if rank == 0:
        Path(out).write_text("ok")
    dist.destroy_process_group()


@pytest.mark.parametrize("metric,weights", [(0, None), (1, None), (0, [0.6, 1.4])])
def test_sharded_index_world2_gloo(tmp_path, metric, weights):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = tmp_path / "ok"
    mp.spawn(_worker, args=(2, port, metric, weights, str(out)), nprocs=2, join=True)
    assert out.read_text() == "ok"


def test_shard_bounds_cover_everything():
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    from knn_b200.distributed import shard_bounds

    for n in (0, 1, 7, 10_000_000):
        for w in (1, 2, 4, 8):
            b = shard_bounds(n, w)
            assert b[0] == 0 and b[-1] == n and all(x <= y for x, y in zip(b, b[1:]))
            assert max(y - x for x, y in zip(b, b[1:])) - min(y - x for x, y in zip(b, b[1:])) <= 1


def test_weighted_shard_bounds():
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    from knn_b200.distributed import shard_bounds

    assert shard_bounds(1000, 4, [1, 1, 1, 1]) == [0, 250, 500, 750, 1000]
    b = shard_bounds(10_000_000, 8, [1.0, 0.92, 1.03, 1.0, 1.05, 0.97, 1.01, 1.02])
    sizes = [y - x for x, y in zip(b, b[1:])]
    assert b[0] == 0 and b[-1] == 10_000_000 and min(sizes) == sizes[1] and max(sizes) == sizes[4]
    assert abs(sizes[1] / sizes[4] - 0.92 / 1.05) < 1e-4
    assert shard_bounds(3, 4, [5, 1, 1, 1])[-1] == 3
    for bad in ([1, 1], [1, 0, 1, 1]):
        with pytest.raises(ValueError):
            shard_bounds(10, 4, bad)


def _grid_worker(rank, world, port, out):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from knn_b200.distributed import GridIndexFlat
    from oracle import flat_oracle as fo

    rng = np.random.default_rng(1)
    xb = rng.standard_normal((803, 24)).astype(np.float32)
    xq = rng.standard_normal((21, 24)).astype(np.float32)
    for metric in (0, 1):
        # 2 query groups x 2 row shards; unequal shards inside the groups
        index = GridIndexFlat(24, metric, query_groups=2, index_factory=lambda: _OracleShard(24, metric), merge_fn=_merge_numpy,
                              shard_weights=[1.0, 1.5, 0.8, 1.2])
        index.add(xb[:400])
        index.add(xb[400:])
        assert index.ntotal == 803 and (index.R, index.Q) == (2, 2)
        # the groups share the queries in proportion to their ranks' weights: (1.0 + 1.5) : (0.8 + 1.2)
        assert index.query_slice(21) == ((0, 12) if rank < 2 else (12, 21))
        for k in (7, 900):
            D, I = index.search(xq, k)
            D_ref, I_ref = fo.knn_flat(xq, xb, k, metric)
            assert D.shape == (21, k) and np.array_equal(I, I_ref), (rank, metric, k)
            assert np.allclose(D, D_ref, rtol=1e-6, atol=1e-6)  # the oracle's sgemm rounds differently per batch shape
        D, I = index.search(xq[:1], 5)  # fewer queries than groups: one group searches nothing
        assert np.array_equal(I, fo.knn_flat(xq[:1], xb, 5, metric)[1])
    if rank == 0:
        Path(out).write_text("ok")
    dist.destroy_process_group()


def test_grid_index_world4_gloo(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = tmp_path / "ok"
    mp.spawn(_grid_worker, args=(4, port, str(out)), nprocs=4, join=True)
    assert out.read_text() == "ok"


def test_choose_query_groups_by_memory_fit(monkeypatch):
    """Layout rule of the multi-GPU bench (DESIGN.md section 6): the largest number of query groups whose per-rank
    share of the rows fits 60 % of the GPU memory (180 GB assumed when no GPU is visible)."""
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    from knn_b200.distributed import choose_query_groups, shard_bounds

    def no_device(*_):
        raise RuntimeError("no CUDA device")

    monkeypatch.setattr(torch.cuda, "get_device_properties", no_device)  # the sizes below assume the 180 GB default
    assert choose_query_groups(8, 10_000_000, 1024, 6) == 8       # C4: 61 GB fit every GPU -> pure query sharding
    assert choose_query_groups(4, 10_000_000, 1024, 6) == 4
    assert choose_query_groups(8, 100_000_000, 1024, 2) == 4      # C5: 205 GB in bf16 -> two row shards per group
    assert choose_query_groups(8, 100_000_000, 1024, 6) == 1      # 614 GB with fp32 master rows -> all 8 GPUs per group
    assert choose_query_groups(6, 30_000_000, 1024, 6) == 3       # divisors of the world only
    assert choose_query_groups(1, 10, 8, 6) == 1
    # weighted bounds cover the range exactly and respect the order of the weights
    b = shard_bounds(100_000, 8, [0.1238, 0.1265, 0.1237, 0.1241, 0.1275, 0.1236, 0.1237, 0.127])
    assert b[0] == 0 and b[-1] == 100_000 and all(x <= y for x, y in zip(b, b[1:]))
    assert (b[5] - b[4]) > (b[6] - b[5])
