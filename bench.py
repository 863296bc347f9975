#!/usr/bin/env python3
"""Benchmark of the flat-search hot path (BASELINE.json: queries/s at 1024-d, k=100).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config C4 of BASELINE.json / SURVEY.md section 8d): synthetic 10M x 1024 fp32
database of L2-normalised N(0,1) rows (seeded per 65536-row block, so any GPU count builds
the same database), 100k normalised queries, k = 100, inner product.  One "step" = one full
pass of index.search over all queries.  With N GPUs the database is row-sharded (strong
scaling: total work fixed; shard sizes proportional to each GPU's measured speed unless
--no-balance), every rank scores all queries against its shard, the shards exchange a per-query
bound on the k-th best score (one NCCL all-reduce) before the exact rescoring, and the per-shard
results are exchanged and merged in one kernel over NVLink peer memory.

Legs, all in one JSON line printed by rank 0:
  value     queries/s with the queries already resident in HBM (device-pointer C-ABI call)
  e2e       same from pinned host queries to (D, I) in pinned host memory: N = 1 the host-pointer C-ABI call
            (H2D -> search -> D2H inside it); N > 1 every rank uploads 1/N of the queries, all-gather, search,
            rank 0 reads the result back
  e2e_pageable  the call the reference's drivers make: pageable numpy queries in, numpy (D, I) out
  roofline  the tcgen05 GEMM kernel: 2*nq*N*d flop / CUDA-event time of its launches
  parity_vs_fp64  >= 256 sampled queries of the last timed step against an fp64 brute force done with plain torch on
            every rank's shard (regenerated rows, fp64 matmul, local top-(k+8), all-gather, merge on rank 0 with the
            lower-id tie rule) - nothing of the engine is on that side.  A mismatch beyond the fp32 tie tolerance or a
            distance off by more than 1e-5 relative makes the run exit non-zero.
  small_batch   N = 1: whole index.search calls with 1..256 queries on the resident database against the HBM roofline
  cpu_baseline  blocked sgemm + top-k on the host cores (bounded sample, scaled by N)
--impl reference times the CPU implementation only (see oracle/cpu_baseline.py).
--config c2|c3 selects the rescoring-heavy all-vs-all stand-ins of BASELINE.json's configs 2 and 3 (k = 1000).
--dump-outputs DIR writes the (D, I) of the last timed step as DIR/D.npy and DIR/I.npy (see dump_outputs); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
for p in (str(REPO), str(REPO / "knn-for-homology_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

D_DIM = 1024
BLOCK_ROWS = 65536


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nb", type=int, default=10_000_000, help="database rows (C4: 10M)")
    ap.add_argument("--nq", type=int, default=100_000, help="queries per step (C4: 100k)")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--cta-group", type=int, default=2, choices=[1, 2], help="tcgen05 cta_group of the GEMM kernel")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-phases", action="store_true", help="skip the extra untimed pass that times the phases of the sharded search")
    ap.add_argument("--bf16-storage", action="store_true", help="the bf16 values ARE the database (config C5): no fp32 master rows")
    ap.add_argument("--shadow-fmt", type=int, default=0, choices=[0, 1, 2], help="16-bit format of the tensor-core copy of the database: 0 automatic, 1 bf16, 2 fp16")
    ap.add_argument("--query-groups", type=int, default=0, help="N > 1: Q query groups x (N / Q) row shards (GridIndexFlat).  0 (default): "
                    "automatic - the largest Q whose row share fits 60 %% of the GPU memory (knn_b200.distributed.choose_query_groups); "
                    "1: plain row sharding over all N GPUs")
    ap.add_argument("--no-balance", action="store_true", help="N > 1: equal row shards instead of shards proportional to each GPU's measured speed")
    ap.add_argument("--mantissa-bits", type=int, default=0, help="mantissa bits kept in bf16 tensor-core operands: 0 automatic, 2..7")
    ap.add_argument("--config", default="c4", choices=["c4", "c2", "c3", "c5"],
                    help="c4 (default): 10M x 1024, 100k queries, k=100.  c2: CATH20 stand-in, 14433 all-vs-all, k=1000.  "
                         "c3: Pfam20 stand-in, 300k all-vs-all, k=1000.  c5: 100M bf16 rows, 1M queries, k=1000 (8 GPUs)")
    ap.add_argument("--no-small-batch", action="store_true", help="N = 1: skip the small-batch (HBM roofline) legs")
    ap.add_argument("--no-autotune", action="store_true", help="query groups: keep the calibrated query shares (no feedback from measured call times)")
    ap.add_argument("--no-overlap", action="store_true", help="finish phase of a batch on the main stream (no side stream)")
    ap.add_argument("--parity-queries", type=int, default=256)
    ap.add_argument("--param", action="append", default=[], metavar="NAME=VALUE",
                    help="knn_index_set_param on every rank's index (A/B experiments; results never depend on it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (D, I) of the last timed step as DIR/D.npy (float32) and DIR/I.npy (float64), "
                         "at most 64 MB together (a fixed, seeded sample of query rows when the whole result is larger)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm keeps only its timings)")
    if args.config == "c2":
        args.nb, args.nq, args.k, args.all_vs_all = 14_433, 14_433, 1000, True
    elif args.config == "c3":
        args.nb, args.nq, args.k, args.all_vs_all = 300_000, 300_000, 1000, True
    elif args.config == "c5":
        args.nb, args.nq, args.k, args.bf16_storage, args.all_vs_all = 100_000_000, 1_000_000, 1000, True, False
    else:
        args.all_vs_all = False
    return args


def measured_peaks():
    f = REPO / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"tflops_burst": d.get("bf16_tflops"), "tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic():
    """DRAM bytes per launch of the GEMM kernel from the committed `ncu --set full` capture (profiles/)."""
    f = REPO / "profiles" / "gemm_traffic.json"
    if not f.exists():
        return None, "no ncu capture committed"
    d = json.loads(f.read_text())
    return d["dram_bytes_per_launch"], d["note"]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def reference_arm(args, rank, world):
    """CPU implementation of the path on the host cores, bounded sample per step."""
    if rank != 0:
        return
    from oracle import cpu_baseline

    n_sample, nq_sample = min(args.nb, 400_000), min(args.nq, 2048)
    res = None
    times = []
    for i in range(args.warmup + args.steps):
        res = cpu_baseline.time_sample(args.nb, D_DIM, args.k, n_sample=n_sample, nq_sample=nq_sample, seed=99 + i)
        if i >= args.warmup:
            times.append(res)
    qps = statistics.mean(r["value"] for r in times)
    line = {
        "impl": "reference", "metric": "queries/s at 1024-d, k=%d, exact flat inner-product search" % args.k,
        "value": qps, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * statistics.mean(r["seconds"] for r in times), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample"]},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    name = "C4" if (args.nb, args.nq, args.k) == (10_000_000, 100_000, 100) else "custom"
    if (args.nb, args.nq, args.k, args.bf16_storage) == (100_000_000, 1_000_000, 1000, True):
        name = "C5"
    if getattr(args, "all_vs_all", False):
        name = {"c2": "C2 stand-in (CATH20 all-vs-all)", "c3": "C3 stand-in (Pfam20 all-vs-all)"}[args.config]
    store = "bf16" if args.bf16_storage else "fp32"
    return {"workload": f"{name}: synthetic normalised {args.nb}x{D_DIM} {store} database, {args.nq} queries, k={args.k}, "
                        f"inner product, exact (ids = fp32 IndexFlatIP on the stored values)",
            "database_rows": args.nb, "queries_per_step": args.nq, "k": args.k, "d": D_DIM,
            "sharding": f"{world} GPU(s) of one box (the engine's layout over them is reported in `layout`)",
            "l2": "inputs larger than L2 (bf16 database shard >> 126 MB)"}


def gen_block(blk, nb, dev):
    """Rows [blk * BLOCK_ROWS, ...) of the synthetic database: seeded per block, so any GPU count builds the same one."""
    import torch

    import knn_b200

    r0, r1 = blk * BLOCK_ROWS, min((blk + 1) * BLOCK_ROWS, nb)
    g = torch.Generator(device=dev).manual_seed(1234 + blk)
    rows = torch.randn(r1 - r0, D_DIM, device=dev, generator=g)
    knn_b200.normalize_L2(rows)
    return r0, r1, rows


def fp64_parity(args, dev, rank, world, lo, hi, contributes, xq_s, D_s, I_s):
    """Independent check of the engine's answer for the sampled queries xq_s (their (D, I) rows: D_s, I_s).

    Every contributing rank regenerates its rows [lo, hi) block by block and scores the sample against them with a
    plain torch fp64 matmul, keeping a running top-(k + 8) by (score desc, id asc).  The per-rank lists are
    all-gathered and merged on rank 0 with the same rule.  Only torch ops on this side: no kernel, id mapping, bound
    exchange or merge of the engine.  (With bf16 storage the rows are rounded to bf16 first: those values ARE the
    database.)  Returns the record for the JSON line (rank 0) or None."""
    import torch
    import torch.distributed as dist

    ns, k = xq_s.shape[0], args.k
    kk = k + 8
    q64 = xq_s.double()
    best_s = torch.full((ns, kk), -float("inf"), dtype=torch.float64, device=dev)
    best_i = torch.full((ns, kk), -1, dtype=torch.int64, device=dev)

    def fold(bs, bi, cs, ci):
        s_all, i_all = torch.cat([bs, cs], 1), torch.cat([bi, ci], 1)
        # (score desc, id asc): stable sort by id first, then by score
        o = torch.argsort(i_all, dim=1, stable=True)
        s_all, i_all = torch.gather(s_all, 1, o), torch.gather(i_all, 1, o)
        o = torch.argsort(s_all, dim=1, descending=True, stable=True)[:, :kk]
        return torch.gather(s_all, 1, o), torch.gather(i_all, 1, o)

    if contributes:
        for blk in range(lo // BLOCK_ROWS, (hi + BLOCK_ROWS - 1) // BLOCK_ROWS):
            r0, r1, rows = gen_block(blk, args.nb, dev)
            s0, s1 = max(lo, r0), min(hi, r1)
            rows = rows[s0 - r0:s1 - r0]
            if args.bf16_storage:
                rows = rows.bfloat16().float()
            sc = q64 @ rows.double().T
            top_s, top_p = torch.topk(sc, min(kk, sc.shape[1]), dim=1)
            best_s, best_i = fold(best_s, best_i, top_s, top_p + s0)
    if world > 1:
        gs = torch.empty((world, ns, kk), dtype=torch.float64, device=dev)
        gi = torch.empty((world, ns, kk), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(gs, best_s)
        dist.all_gather_into_tensor(gi, best_i)
        best_s = torch.full((ns, kk), -float("inf"), dtype=torch.float64, device=dev)
        best_i = torch.full((ns, kk), -1, dtype=torch.int64, device=dev)
        for r in range(world):
            best_s, best_i = fold(best_s, best_i, gs[r], gi[r])
    if rank != 0:
        return None
    rec = compare_with_fp64(D_s, I_s, best_s, best_i, k, D_DIM)
    rec["reference"] = (f"torch fp64 brute force over the regenerated rows of all {world} shard(s), top-(k+8) per shard, "
                        "all-gather, merge on rank 0 (score desc, id asc)")
    return rec


def compare_with_fp64(D_s, I_s, best_s, best_i, k, d):
    """The gate of `parity_vs_fp64`: the engine's (D_s, I_s) for the sampled queries against the fp64 reference lists
    best_s / best_i (top-(k + e) per query, score desc / id asc).  Pure torch, device-agnostic (CPU-tested in
    tests/test_bench_parity_gate.py).  ok <=> no id mismatch beyond the fp32 tie tolerance, no duplicate id in a row, and
    every distance within 1e-5 relative of the fp64 score of the id it is reported for."""
    import torch

    ns, kk = best_i.shape
    tau = 2.0 * (d ** 0.5) * 2.0 ** -24  # unit vectors: scale |x||y| = 1
    ref_s, ref_i = best_s[:, :k], best_i[:, :k]
    differ = I_s != ref_i
    # fp64 score of OUR id at every position: looked up in the reference's top-(k + e); an id that is not even there lies
    # beyond the (k + e)-th fp64 candidate and counts as a mismatch
    ids_sorted, order = torch.sort(best_i, dim=1)
    at = torch.searchsorted(ids_sorted, I_s.contiguous()).clamp_(max=kk - 1)
    found = torch.gather(ids_sorted, 1, at) == I_s
    ours64 = torch.gather(torch.gather(best_s, 1, order), 1, at)
    gap = (ours64 - ref_s).abs()
    excused = differ & found & (gap <= tau)
    beyond = differ & ~excused
    rows_sorted, _ = torch.sort(I_s, dim=1)
    dup = int((rows_sorted[:, 1:] == rows_sorted[:, :-1]).any(dim=1).sum().item())
    # distances are checked against the fp64 score of the id they belong to (at an excused position that is OUR id)
    rel = (D_s.double() - ours64).abs() / ours64.abs().clamp_min(1e-300)
    rel = torch.where(found, rel, torch.zeros_like(rel))
    n_beyond = int(beyond.sum().item())
    max_rel = float(rel.max().item()) if rel.numel() else 0.0
    return {"queries": int(ns), "k": int(k), "positions": int(ns * k), "id_mismatches_beyond_tau": n_beyond,
            "excused": int(excused.sum().item()), "rows_with_duplicate_ids": dup, "max_rel_err_D": max_rel,
            "tau": tau, "rtol_D": 1e-5, "ok": bool(n_beyond == 0 and dup == 0 and max_rel <= 1e-5)}


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, D, I, limit=DUMP_LIMIT_BYTES):
    """Writes the search result (D, I) as out_dir/D.npy (float32) and out_dir/I.npy (float64, exact for ids below
    2**53), at most `limit` bytes together.  A larger result is cut to a sample of query rows drawn with a fixed seed
    (sorted, the same rows in both files), so two builds given the same arguments write the same rows.  Returns the
    number of query rows written."""
    import numpy as np
    import torch

    nq, k = D.shape
    fit = max(1, (limit - 1024) // (k * (4 + 8)))  # 1024 bytes: room for the two .npy headers
    if fit < nq:
        rows = np.sort(np.random.default_rng(0).choice(nq, size=fit, replace=False))
        sel = torch.from_numpy(rows).to(D.device)
        D, I = D[sel], I[sel]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "D.npy", D.cpu().numpy().astype(np.float32, copy=False))
    np.save(out / "I.npy", I.cpu().numpy().astype(np.float64))
    return int(D.shape[0])


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import knn_b200
    from knn_b200.distributed import GridIndexFlat, ShardedIndexFlat, choose_query_groups, measured_rank_speeds, shard_bounds

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- build the database shard on the device (index build is reported, not timed as search) ----
    # A step ends when the slowest shard is done, and under the board power cap the GPUs of one box do not clock
    # alike: shards are sized in proportion to each GPU's measured speed on the engine's own GEMM (2 s, untimed, part
    # of the index build like any placement decision).
    weights = None
    if world > 1 and not args.no_balance:
        weights = measured_rank_speeds(D_DIM, local_rank, seconds=2.0)
    t_build = time.perf_counter()
    Q = args.query_groups if world > 1 else 1
    if Q == 0:  # automatic layout
        Q = choose_query_groups(world, args.nb, D_DIM, 2 if args.bf16_storage else 6, device=local_rank)
    args.query_groups = Q
    if Q > 1:  # R = world / Q row shards per query group; every group holds the whole database
        index = GridIndexFlat(D_DIM, knn_b200.METRIC_INNER_PRODUCT, query_groups=Q, device=local_rank,
                              bf16_storage=args.bf16_storage, shard_weights=weights)
        R = world // Q
        b = shard_bounds(args.nb, R, weights[(rank // R) * R:(rank // R + 1) * R] if weights else None)
        lo, hi = b[rank % R], b[rank % R + 1]
    else:
        index = ShardedIndexFlat(D_DIM, knn_b200.METRIC_INNER_PRODUCT, device=local_rank, bf16_storage=args.bf16_storage,
                                 shard_weights=weights)
        b = shard_bounds(args.nb, world, weights)
        lo, hi = b[rank], b[rank + 1]
    if Q > 1 and args.no_autotune:
        index.autotune = False
    index.local.set_param("cta_group", args.cta_group)
    if args.shadow_fmt and not args.bf16_storage:
        index.local.set_param("shadow_fmt", args.shadow_fmt)
    index.local.set_param("mantissa_bits", args.mantissa_bits)
    for kv in args.param:
        name, _, val = kv.partition("=")
        index.local.set_param(name, int(val))
    if args.no_overlap:
        index.local.set_param("overlap_finish", 0)
        if Q == 1:
            index.pipeline_batches = False
        else:
            index.inner.pipeline_batches = False
    index.local.reserve(hi - lo)
    for blk in range(lo // BLOCK_ROWS, (hi + BLOCK_ROWS - 1) // BLOCK_ROWS):
        r0, r1, rows = gen_block(blk, args.nb, dev)
        s0, s1 = max(lo, r0), min(hi, r1)
        index.local.add(rows[s0 - r0:s1 - r0])
    index.adopt_local(global_start=lo, n_global=args.nb)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t_build

    if args.all_vs_all:  # C2 / C3: the queries are the database rows themselves (cath/search.py:24, pfam/proteins_search.py:49)
        xq_dev = torch.cat([gen_block(blk, args.nb, dev)[2] for blk in range((args.nb + BLOCK_ROWS - 1) // BLOCK_ROWS)])[:args.nq].contiguous()
    else:
        g = torch.Generator(device=dev).manual_seed(4321)
        xq_dev = torch.randn(args.nq, D_DIM, device=dev, generator=g)
        knn_b200.normalize_L2(xq_dev)
    if not args.no_e2e:
        xq_host = torch.empty((args.nq, D_DIM), dtype=torch.float32, pin_memory=True)
        xq_host.copy_(xq_dev)
        D_host = torch.empty((args.nq, args.k), dtype=torch.float32, pin_memory=True)
        I_host = torch.empty((args.nq, args.k), dtype=torch.int64, pin_memory=True)
        xq_np = xq_dev.cpu().numpy()  # pageable, what the reference's drivers hold
    torch.cuda.synchronize()

    lib = knn_b200._lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step_device():
        last["DI"] = index.search(xq_dev, args.k)
        return last["DI"]

    def step_e2e():
        if world == 1:
            # the raw host-pointer C-ABI call: H2D of the queries, search, D2H of (D, I)
            index.local.search_into(xq_host.data_ptr(), args.nq, args.k, D_host.data_ptr(), I_host.data_ptr())
        else:
            # every rank holds the host queries: each uploads 1/N of them, one all-gather over NVLink does the rest
            D, I = index.search(xq_host, args.k)  # pinned host tensor in: each rank uploads only its share
            if rank == 0:
                D_host.copy_(D, non_blocking=True)
                I_host.copy_(I, non_blocking=True)
            torch.cuda.synchronize()

    def step_e2e_pageable():
        if world == 1:
            last["np"] = index.local.search(xq_np, args.k)  # IndexFlat.search(numpy) -> numpy: what `index.search` is to the drivers
        else:
            last["np"] = index.search(xq_np, args.k)  # numpy in, numpy out on every rank (sharded upload inside)

    by_rank = {}

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        index.local.set_param("profile", 1 if profile else 0)
        barrier()
        launches0 = lib.knn_kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gemm_ms, gemm_launches = 0.0, 0
        e0.record()
        for _ in range(steps):
            fn()
            if profile:
                gemm_ms += index.last_stats["gemm_ms"]
                gemm_launches += int(index.last_stats["gemm_launches"])
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = lib.knn_kernel_launches() - launches0
        index.local.set_param("profile", 0)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            per_rank = torch.zeros((world, 2), device=dev, dtype=torch.float64)
            dist.all_gather_into_tensor(per_rank, torch.tensor([ms, gemm_ms], device=dev, dtype=torch.float64))
            by_rank["step_ms"] = [round(v / steps, 3) for v in per_rank[:, 0].tolist()]
            by_rank["gemm_ms"] = [round(v / steps, 3) for v in per_rank[:, 1].tolist()]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, gemm_ms, gemm_launches

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches, gemm_ms, gemm_launches = timed(step_device, args.steps, args.warmup, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    value = args.nq * args.steps / (ms / 1e3)
    by_rank_value = dict(by_rank)  # per-rank step / GEMM time of the `value` leg (chip-to-chip spread under the power cap)
    D, I = last["DI"]  # result of the last timed step
    dumped_rows = dump_outputs(args.dump_outputs, D, I) if args.dump_outputs and rank == 0 else None
    search_path = int(index.local.stat("path"))
    fmt_names = {1: "bf16", 2: "fp16"}
    fmt = fmt_names[int(index.local.stat("shadow_fmt"))]
    mbits = int(index.local.stat("mantissa_bits"))

    e2e = e2e_pageable = None
    if not args.no_e2e:
        h2d = args.nq * D_DIM * 4
        d2h = args.nq * args.k * 12
        ms_e, _, _, _ = timed(step_e2e, args.steps, 1)
        e2e = {"value": args.nq * args.steps / (ms_e / 1e3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ms_e / args.steps, "host_memory": "pinned"}
        ms_p, _, _, _ = timed(step_e2e_pageable, args.steps, 2)  # 2 warm-ups: both result buffers of the pinned-memory cache exist
        e2e_pageable = {"value": args.nq * args.steps / (ms_p / 1e3), "unit": "queries/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": ms_p / args.steps,
                        "host_memory": "pageable numpy arrays in and out (the reference drivers' call)"}

    # ---- parity of the result of the last timed step against an fp64 brute force that shares nothing with the engine ----
    ns = min(args.parity_queries, args.nq)
    chk = torch.arange(ns, device=dev) * (args.nq // ns)
    contributes = Q == 1 or rank // (world // Q) == 0  # with query groups every group holds the whole database: group 0 answers
    parity = fp64_parity(args, dev, rank, world, lo, hi, contributes, xq_dev[chk].contiguous(), D[chk], I[chk])
    if e2e_pageable and rank == 0 and parity is not None:  # the host path must return the same bits
        Dn, In = last["np"]
        parity["host_path_identical"] = bool(np.array_equal(Dn, D.cpu().numpy()) and np.array_equal(In, I.cpu().numpy()))
        parity["ok"] = parity["ok"] and parity["host_path_identical"]
    # ... and the engine's own exact fp32 path on a few of them (bit-identical by construction of the rerank)
    chk2 = chk[:64]
    index.local.set_param("path", 1)
    D1, I1 = index.search(xq_dev[chk2].contiguous(), args.k)
    index.local.set_param("path", 0)
    parity_ok = bool(torch.equal(I[chk2], I1) and torch.equal(D[chk2], D1))

    phases = None
    if world > 1 and not args.no_phases:  # one extra, untimed step with CUDA events around the phases of the sharded search
        index.profile_phases = True
        step_device()
        index.profile_phases = False
        phases = index.last_phases_ms

    small = None
    if world == 1 and not args.no_small_batch and not args.all_vs_all:
        # Small query batches on the resident database: whole index.search calls (every launch of the call inside the
        # timed region) against the HBM roofline; algorithmic bytes per SURVEY.md 8(d): N*d*2 + nq*d*4 + nq*k*12.
        peaks_hbm = measured_peaks()["hbm_gbs"]
        small = []
        for nq_s in (1, 16, 64, 128, 256):
            xs = xq_dev[:nq_s].contiguous()
            search = index.local.search  # the product call (IndexFlat.search on a CUDA tensor)
            for _ in range(3):
                search(xs, args.k)
            reps = 20
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = lib.knn_kernel_launches()
            e0.record()
            for _ in range(reps):
                search(xs, args.k)
            e1.record()
            torch.cuda.synchronize()
            ms_call = e0.elapsed_time(e1) / reps
            nbytes = args.nb * D_DIM * 2 + nq_s * D_DIM * 4 + nq_s * args.k * 12
            gbs = nbytes / (ms_call / 1e3) / 1e9
            launches_per_call = (lib.knn_kernel_launches() - l0) // reps
            Ds, Is = search(xs, args.k)
            tfl = 2.0 * nq_s * args.nb * D_DIM / (ms_call / 1e3) / 1e12
            small.append({"nq": nq_s, "ms_per_call": ms_call, "gbs": gbs, "frac_of_hbm": gbs / peaks_hbm,
                          # 129..256 queries sit at the machine balance (2*256*d flop per 2*d bytes of a bf16 row): the
                          # call keeps the tensor pipe AND HBM busy and runs into the board power cap (ncu: SM clock
                          # 1.16 GHz, tensor pipe 98 % active, profiles/r01_gemm_main_ncu_nq256.md)
                          "tflops": tfl, "frac_of_tensor_sustained": tfl / measured_peaks()["tflops_sustained"],
                          "kernel": ("gemm_stream_kernel (queries resident in shared memory)" if nq_s <= 64 else
                                     "gemm_stream_kernel, CTA pair" if nq_s <= 128 else "gemm_filter_kernel, one 256-query tile pair"),
                          "launches_per_call": launches_per_call,
                          "identical_to_large_batch_result": bool(torch.equal(Is, I[:nq_s]) and torch.equal(Ds, D[:nq_s]))})

    if rank == 0:
        peaks = measured_peaks()
        n_shard = hi - lo
        nq_rank = args.nq
        if Q > 1:
            q_lo, q_hi = index.query_slice(args.nq)
            nq_rank = q_hi - q_lo
        flops_per_step = 2.0 * nq_rank * n_shard * D_DIM  # this rank's GEMM work: its rows x its query group's queries
        achieved = flops_per_step * args.steps / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None
        peak = peaks["tflops_sustained"]
        traffic, traffic_note = ncu_traffic()
        roofline = {"bound": "tensor", "kernel": "gemm_filter_kernel (tcgen05 kind::f16, fused threshold filter)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": (achieved / peak) if achieved else None, "peak_kind": "sustained, " + peaks["source"],
                    "frac_of_burst": (achieved / peaks["tflops_burst"]) if achieved else None,
                    "traffic": traffic, "traffic_note": traffic_note, "launches": gemm_launches, "kernel_ms_per_step": gemm_ms / args.steps,
                    "algorithmic_flop_per_launch_avg": flops_per_step * args.steps / max(1, gemm_launches),
                    "whole_step_frac_of_burst": 2.0 * args.nq * args.nb * D_DIM / world / (ms / args.steps / 1e3) / 1e12 / peaks["tflops_burst"]}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import cpu_baseline

            cpu = cpu_baseline.time_sample(args.nb, D_DIM, args.k, n_sample=min(args.nb, 400_000),
                                           nq_sample=min(args.nq, 4096))
            cpu = {k: cpu[k] for k in ["value", "unit", "cores", "kind", "sample"]}
        line = {
            "metric": "queries/s at 1024-d, k=%d, exact flat inner-product search" % args.k,
            "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": fmt, "dtype_note": f"{fmt} x {fmt} ({mbits} mantissa bits) -> f32 tensor-core filter (tcgen05 kind::f16), then exact f32 "
                                        "rescoring: results equal f32 IndexFlatIP",
            "data": "synthetic",
            "config": workload_config(args, world), "e2e": e2e, "e2e_pageable": e2e_pageable, "gpu_launches": launches, "roofline": roofline,
            "parity_vs_fp64": parity, "small_batch": small,
            "cpu_baseline": cpu, "clocks": clocks, "index_build_s": build_s, "parity_spot_check": parity_ok,
            "search_path": search_path, "cta_group": args.cta_group, "phases_ms_rank0": phases, "ms_per_step_by_rank": by_rank_value or None,
            "shard_rows_by_rank": [b[r + 1] - b[r] for r in range(len(b) - 1)], "query_groups": Q,
            "layout": {"query_groups": Q, "row_shards_per_group": world // Q,
                       "note": ("one GPU" if world == 1 else
                                f"{Q} query group(s) x {world // Q} row shard(s): every group holds the whole database row-sharded over its "
                                "ranks and answers 1/Q of the queries; chosen as the largest group count whose row share fits 60 % of the "
                                "GPU memory unless --query-groups says otherwise (1 = plain row sharding)")},
            "rank_speed_weights": [round(w, 4) for w in weights] if weights else None,
            "query_share_by_group": ([round(w / sum(index.group_weights), 4) for w in index.group_weights]
                                     if Q > 1 and getattr(index, "group_weights", None) else None),
            "overlap_finish": not args.no_overlap, "params": args.param or None, "autotune_query_shares": bool(Q > 1 and not args.no_autotune),
            "dumped_query_rows": dumped_rows,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        ok = torch.tensor([1 if (rank != 0 or (parity["ok"] and parity_ok)) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        dist.barrier()
        dist.destroy_process_group()
        if int(ok.item()) == 0:
            sys.exit(3)
    elif not (parity["ok"] and parity_ok):
        sys.exit(3)


if __name__ == "__main__":
    main()
