"""What 16-bit inputs save: fp16 / bf16 rows and queries handed to the index as they are, against the same values in
float32 (the results are bit-identical either way; see tests/test_gpu_h16_inputs.py).  Prints one JSON object.

  add_host      IndexFlat.add of --rows x 1024 rows from pageable and from pinned host memory, fp32 against fp16:
                seconds and GB/s of caller bytes
  ingest_dev    the ingest kernel alone (add of a device tensor into a reserved index, CUDA events), fp32 against bf16
                source rows, in GB/s of HBM traffic (source read + fp32 master + 16-bit shadow written), next to the
                measured device-to-device copy rate
  peak_add_dev  torch's peak allocation while adding a bf16 device tensor: the old path's x.to(float32) against the
                16-bit path (the index storage itself, cudaMalloc'ed by the library, is the same for both)
  c4_host       C4 (10M x 1024 normalised rows, 100k queries, k = 100) searched from pageable host queries, fp32
                against fp16 (--c4-rows to shrink the database)
  c2_driver     drivers.search_and_save on one 14,433 x 1024 .npy file (CATH20-sized, both metrics), fp16 file against
                the fp32 cast of it

    python tools/bench_h16_inputs.py [--rows 10000000] [--c4-rows 10000000] [--reps 3]
"""
import argparse
import json
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "knn-for-homology_b200")]


def _host_rows(n, d, dtype, pinned):
    """n x d rows of the given numpy dtype, tiled from one random block (the values do not matter for a copy)."""
    import torch

    block = np.random.default_rng(0).standard_normal((4096, d)).astype(dtype)
    if pinned:
        t = torch.empty((n, d), dtype=torch.from_numpy(block).dtype, pin_memory=True)
        x = t.numpy()
    else:
        x = np.empty((n, d), dtype)
    for i in range(0, n, 4096):
        m = min(4096, n - i)
        x[i:i + m] = block[:m]
    return x


def bench_add_host(knn, n, d, reps):
    out = {}
    for pinned in (False, True):
        for name, dt in (("fp32", np.float32), ("fp16", np.float16)):
            x = _host_rows(n, d, dt, pinned)
            idx = knn.IndexFlat(d, 0, device=0)
            idx.reserve(n)
            best = None
            for _ in range(reps):
                idx.reset()
                t0 = time.perf_counter()
                idx.add(x)
                t = time.perf_counter() - t0
                best = t if best is None else min(best, t)
            out["%s_%s" % ("pinned" if pinned else "pageable", name)] = {"s": round(best, 3), "GB/s": round(x.nbytes / best / 1e9, 2)}
            del idx, x
    return out


def bench_ingest_dev(knn, n, d, reps):
    import torch

    out = {}
    src = torch.randn(n, d, device="cuda")
    for name, dt in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        x = src.to(dt)
        idx = knn.IndexFlat(d, 0, device=0)
        idx.reserve(n)
        times = []
        for _ in range(reps + 1):
            idx.reset()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            idx.add(x)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1) / 1e3)
        t = min(times[1:])
        traffic = x.numel() * x.element_size() + n * d * (4 + 2) + n * 4
        out[name] = {"ms": round(t * 1e3, 2), "GB/s": round(traffic / t / 1e9, 1), "source_GB": round(x.numel() * x.element_size() / 1e9, 2)}
        del idx, x
    a = torch.empty(n * d, device="cuda")
    b = torch.empty_like(a)
    times = []
    for _ in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    out["d2d_copy_GB/s"] = round(2 * a.numel() * 4 / min(times[1:]) / 1e9, 1)
    return out


def bench_peak_add_dev(knn, n, d):
    import torch

    x = torch.randn(n, d, device="cuda").to(torch.bfloat16)
    out = {}
    for name, arg in (("old_path_fp32_copy", lambda: x.to(torch.float32)), ("bf16_as_is", lambda: x)):
        idx = knn.IndexFlat(d, 0, device=0)
        idx.reserve(n)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        idx.add(arg())
        torch.cuda.synchronize()
        out[name + "_GB"] = round((torch.cuda.max_memory_allocated() - base) / 1e9, 2)
        del idx
    out["index_storage_GB"] = round(n * d * 6 / 1e9, 2)
    return out


def bench_c4_host(knn, n, reps):
    import torch

    d, nq, k = 1024, 100_000, 100
    g = torch.Generator(device="cuda").manual_seed(1)
    idx = knn.IndexFlat(d, 0, device=0)
    idx.reserve(n)
    for i in range(0, n, 1 << 20):
        x = torch.randn(min(1 << 20, n - i), d, device="cuda", generator=g)
        knn.normalize_L2(x)
        idx.add(x)
    q = torch.randn(nq, d, device="cuda", generator=g)
    knn.normalize_L2(q)
    out, res = {}, {}
    for name, dt in (("fp32", torch.float32), ("fp16", torch.float16)):
        qh = q.to(dt).cpu().numpy()  # pageable
        res[name] = idx.search(qh, k)
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            idx.search(qh, k)
            times.append(time.perf_counter() - t0)
        out[name] = {"s": round(min(times), 4), "queries/s": round(nq / min(times))}
    # fp16 queries are a different (rounded) query set: same-bits holds against the fp32 call on float(fp16)
    D32, I32 = idx.search(q.to(torch.float16).float().cpu().numpy(), k)
    out["fp16_equals_fp32_call_on_upconverted"] = bool(np.array_equal(I32, res["fp16"][1]) and np.array_equal(D32, res["fp16"][0]))
    out["database_rows"] = n
    return out


def bench_c2_driver(reps):
    from knn_b200 import drivers

    x = (np.random.default_rng(2).standard_normal((14_433, 1024)) * 0.05).astype(np.float16)
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, arr in (("fp16", x), ("fp32", x.astype(np.float32))):
            dd = Path(tmp) / name
            dd.mkdir()
            np.save(dd / "emb.npy", arr)
            times = []
            for _ in range(reps + 1):
                t0 = time.perf_counter()
                drivers.search_and_save(dd, device=0)
                times.append(time.perf_counter() - t0)
            out[name + "_s"] = round(min(times[1:]), 3)
        same = all(np.array_equal(np.load(Path(tmp) / "fp16" / f)["emb"], np.load(Path(tmp) / "fp32" / f)["emb"])
                   for f in ("hits_cosine.npz", "scores_cosine.npz", "hits_euclidean.npz", "scores_euclidean.npz"))
        out["outputs_identical"] = bool(same)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rows", type=int, default=10_000_000, help="rows of the add measurements (d = 1024)")
    ap.add_argument("--c4-rows", type=int, default=10_000_000, help="database rows of the C4 search")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import contextlib
    import io

    import torch

    import knn_b200 as knn

    res = {"gpu": torch.cuda.get_device_name(0), "rows": args.rows}
    res["ingest_dev"] = bench_ingest_dev(knn, args.rows, 1024, args.reps)
    torch.cuda.empty_cache()
    res["peak_add_dev"] = bench_peak_add_dev(knn, args.rows, 1024)
    torch.cuda.empty_cache()
    res["add_host"] = bench_add_host(knn, args.rows, 1024, args.reps)
    res["c4_host"] = bench_c4_host(knn, args.c4_rows, args.reps)
    torch.cuda.empty_cache()
    with contextlib.redirect_stdout(io.StringIO()):  # search_and_save prints its progress
        res["c2_driver"] = bench_c2_driver(args.reps)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
