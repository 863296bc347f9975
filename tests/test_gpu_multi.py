"""The real multi-GPU path: one process per GPU, NCCL, NVLink peer memory (skipped on a box with fewer than 2 GPUs).

ShardedIndexFlat with the bound exchange (two-phase search, batch-wise over two streams) and the exchange-fused peer
merge must return, on every rank,
  * exactly what ONE unsharded index returns on the same rows (bit for bit: ids and distances), and
  * what the CPU oracle returns (oracle/parity.py rule, reference's next candidates included),
for ragged speed-weighted shards, several add() segments, both metrics, k = 10 and k = 1000, one and several query
batches, with and without the stream pipeline.  Mirrors /root/reference/tests/test_main.py:10-27 in spirit: known
answers through the real path."""
import os
import socket
import sys
import time
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = Path(__file__).resolve().parent.parent


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import knn_b200
    from knn_b200.distributed import ShardedIndexFlat
    from oracle import flat_oracle as fo
    from oracle.parity import check_parity

    log = []
    rng = np.random.default_rng(11)
    d, n, nq = 256, 60011, 700
    centers = rng.standard_normal((50, d)).astype(np.float32)
    xb = (centers[rng.integers(0, 50, n)] + 0.7 * rng.standard_normal((n, d))).astype(np.float32)  # clustered: many near-equal scores
    xb[1000:1040] = xb[3]                                    # exact duplicates: ties broken by id across shard boundaries
    xb[n - 30:] = xb[3]
    xq = (centers[rng.integers(0, 50, nq)] + 0.7 * rng.standard_normal((nq, d))).astype(np.float32)
    xq[5] = xb[3]
    weights = [0.8, 1.2] + [1.0] * (world - 2)               # ragged, speed-proportional shards
    xb_d, xq_d = torch.from_numpy(xb).to(dev), torch.from_numpy(xq).to(dev)
    for metric in (knn_b200.METRIC_INNER_PRODUCT, knn_b200.METRIC_L2):
        single = knn_b200.IndexFlat(d, metric, device=rank)
        single.set_param("path", 2)
        single.add(xb_d)
        for pipeline in (True, False):
            index = ShardedIndexFlat(d, metric, device=rank, exchange_bounds=True, peer_merge=True, shard_weights=weights)
            index.pipeline_batches = pipeline
            index.local.set_param("path", 2)                 # tensor-core filter + bound exchange even on these small shards
            index.local.set_param("query_batch", 256)        # 3 query batches: the batch-wise pipeline is exercised
            index.add(xb_d[:20000])                          # three add() segments: local -> global id mapping
            index.add(xb_d[20000:20001])
            index.add(xb_d[20001:])
            assert index.ntotal == n and 0 < index.local.ntotal < n
            for k in (10, 1000):
                D, I = index.search(xq_d, k)
                assert int(index.local.stat("path")) == 2
                D1, I1 = single.search(xq_d, k)
                assert torch.equal(I, I1), (rank, metric, k, pipeline, "ids differ from the unsharded index")
                assert torch.equal(D, D1), (rank, metric, k, pipeline, "distances differ from the unsharded index")
                if pipeline:
                    D_ref, I_ref = fo.knn_flat(xq, xb, k, metric, want=k + 4)
                    st = check_parity(D.cpu().numpy(), I.cpu().numpy(), D_ref, I_ref, xq, xb, metric, max_excused_frac=2e-2)
                    log.append((metric, k, st["excused"], st["max_rel_err_D"]))
            # numpy in / numpy out goes through the same path
            Dn, In = index.search(xq[:33], 10)
            D1, I1 = single.search(xq_d[:33].contiguous(), 10)
            assert np.array_equal(In, I1.cpu().numpy()) and np.array_equal(Dn, D1.cpu().numpy())
            index.close()
    # a larger, GEMM-shaped case: 3 default-size query batches, unit vectors at d = 1024, vs the unsharded index
    g = torch.Generator(device=dev).manual_seed(5)
    xb2 = torch.randn(300_000, 1024, device=dev, generator=g)
    xq2 = torch.randn(40_000, 1024, device=dev, generator=g)
    knn_b200.normalize_L2(xb2)
    knn_b200.normalize_L2(xq2)
    single = knn_b200.IndexFlat(1024, 0, device=rank)
    single.add(xb2)
    index = ShardedIndexFlat(1024, 0, device=rank, shard_weights=weights)
    index.add(xb2)
    index.profile_phases = True
    for k in (100,):
        D, I = index.search(xq2, k)
        D1, I1 = single.search(xq2, k)
        assert torch.equal(I, I1) and torch.equal(D, D1), (rank, "large case")
    assert "exchange_finish_exposed" in index.last_phases_ms
    index.close()
    # query groups x row shards (bench.py's default layout when the database fits): Q = world (pure query sharding) and,
    # with 4 GPUs, 2 x 2; speed-weighted query slices; CUDA, pinned-host and numpy queries
    from knn_b200.distributed import GridIndexFlat, choose_query_groups

    assert choose_query_groups(world, 10_000_000, 1024, 6, device=rank) == world  # C4 fits every B200
    assert choose_query_groups(8, 100_000_000, 1024, 2, device=rank) == 4         # C5 (205 GB in bf16) needs 2 row shards
    for Q in sorted({world, 2}):
        grid = GridIndexFlat(1024, 0, query_groups=Q, device=rank, shard_weights=weights)
        grid.add(xb2)
        assert grid.ntotal == 300_000
        D, I = grid.search(xq2, 100)
        assert torch.equal(I, I1) and torch.equal(D, D1), (rank, "grid", Q)
        xq_pinned = torch.empty(xq2.shape, dtype=torch.float32, pin_memory=True).copy_(xq2)
        D, I = grid.search(xq_pinned, 100)
        assert D.is_cuda and torch.equal(I, I1) and torch.equal(D, D1), (rank, "grid pinned", Q)
        Dn, In = grid.search(xq2[:5000].cpu().numpy(), 100)
        assert isinstance(Dn, np.ndarray) and np.array_equal(In, I1[:5000].cpu().numpy()) and np.array_equal(Dn, D1[:5000].cpu().numpy())
        grid.close()
    dist.barrier()
    if rank == 0:
        (Path(out_dir) / "ok").write_text(repr(log))
    dist.destroy_process_group()


def test_sharded_two_phase_search_over_nccl_equals_unsharded_and_oracle(tmp_path):
    import torch
    import torch.multiprocessing as mp

    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    ctx = mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=False)
    deadline = time.time() + 600
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("multi-GPU workers did not finish in 600 s")
    log = (tmp_path / "ok").read_text()
    print("oracle parity over NCCL (metric, k, excused, max_rel_err_D):", log)


def test_dev_entry_points_follow_their_pointers_not_the_current_device():
    """ADVICE r1 (medium): the stateless *_dev entry points (normalize, merge, post-processing) and an index created
    with device=1 must work while the CALLER's current device is 0 - they select the device that owns the memory they
    are handed; the SM count is cached per device."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    sys.path.insert(0, str(REPO))
    sys.path.insert(0, str(REPO / "knn-for-homology_b200"))
    import knn_b200
    from oracle import flat_oracle as fo

    torch.cuda.set_device(0)
    rng = np.random.default_rng(3)
    xb = rng.standard_normal((20000, 128)).astype(np.float32)
    xq = rng.standard_normal((300, 128)).astype(np.float32)
    ref_b, ref_q = xb.copy(), xq.copy()
    fo.normalize_L2(ref_b)
    fo.normalize_L2(ref_q)
    dev1 = torch.device("cuda", 1)
    tb, tq = torch.from_numpy(xb).to(dev1), torch.from_numpy(xq).to(dev1)
    knn_b200.normalize_L2(tb)           # knn_normalize_l2_dev on cuda:1 memory, current device 0
    knn_b200.normalize_L2(tq)
    assert torch.cuda.current_device() == 0
    np.testing.assert_allclose(tb.cpu().numpy(), ref_b, rtol=2e-6, atol=1e-7)
    index = knn_b200.IndexFlat(128, 0, device=1)
    index.set_param("path", 2)
    index.add(tb)
    D, I = index.search(tq, 10)
    single0 = knn_b200.IndexFlat(128, 0, device=0)
    single0.set_param("path", 2)
    single0.add(tb.to("cuda:0"))
    D0, I0 = single0.search(tq.to("cuda:0"), 10)
    assert D.device == dev1 and torch.equal(I.cpu(), I0.cpu()) and torch.equal(D.cpu(), D0.cpu())
    # merge of two half-results on cuda:1
    h = 10000
    a = knn_b200.IndexFlat(128, 0, device=1)
    b = knn_b200.IndexFlat(128, 0, device=1)
    a.add(tb[:h])
    b.add(tb[h:])
    Da, Ia = a.search(tq, 10)
    Db, Ib = b.search(tq, 10, id_base=h)
    Dm, Im = knn_b200.merge_topk(torch.stack([Da, Db]), torch.stack([Ia, Ib]), 0)
    assert torch.equal(Im.cpu(), I0.cpu()) and torch.equal(Dm.cpu(), D0.cpu())
    # post-processing on cuda:1
    fam_db = rng.integers(0, 40, 20000).astype(np.int32)
    fam_q = rng.integers(0, 40, 300).astype(np.int32)
    lead1, tp1, _ = knn_b200.evaluate_ids(I, fam_q, fam_db)
    lead0, tp0, _ = knn_b200.evaluate_ids(I0, fam_q, fam_db)
    assert torch.equal(lead1.cpu(), lead0.cpu()) and torch.equal(tp1.cpu(), tp0.cpu())
    assert torch.cuda.current_device() == 0
