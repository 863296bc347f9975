"""What a filtered search costs (IndexFlat.search with params=SearchParameters(sel=...) and exclude=...) on one GPU.
Prints one JSON object (and writes it to --out when given).

  c4          C4 (10M x 1024 normalised rows, 100k resident queries, k = 100, inner product), queries/s of a whole
              search call: no params, a selector of all rows, 50 % and 1 % random selectors, and a selector that masks
              every query's unfiltered top-1 row (the rows each query batch would have ranked best).  Every leg also
              reports gemm_ms, rerank_ms and gemm_launches from a separate pass with profile = 1.
  all_vs_all  the database searched against its own first nq rows with exclude = arange(nq), against the search of
              k + 1 neighbours (the drop-column-0 workaround): C2 (14,433 x 1024, k = 1000) and the C3 stand-in
              (300,000 x 1024, the first 32,768 rows as queries, k = 1000).
The GPU name and power limit are read in the same run.

    python tools/bench_filtered.py [--c4-rows 10000000] [--reps 3] [--out profiles/filtered_1gpu.json]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(REPO), str(REPO / "knn-for-homology_b200")]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def rows(n, d, seed):
    """n x d L2-normalised N(0, 1) rows on the device (seeded)."""
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn((n, d), generator=g, device="cuda")
    return x / x.norm(dim=1, keepdim=True)


def timed(fn, reps):
    import torch

    fn()  # warm-up: every shape of the timed window
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return sorted(ts)[len(ts) // 2]


def profile_stats(idx, fn):
    import torch

    idx.set_param("profile", 1)
    fn()
    torch.cuda.synchronize()
    idx.set_param("profile", 0)
    return {s: idx.stat(s) for s in ("gemm_ms", "rerank_ms", "gemm_launches", "overflow_queries")}


def bench_c4(knn, n, reps):
    import torch

    d, nq, k = 1024, 100_000, 100
    idx = knn.IndexFlat(d, 0, device=0)
    idx.reserve(n)
    for i in range(0, n, 1 << 20):
        idx.add(rows(min(1 << 20, n - i), d, seed=i))
    xq = rows(nq, d, seed=12345)
    gen = torch.Generator(device="cuda").manual_seed(7)
    _, I0 = idx.search(xq, 1)
    best = torch.ones(n, dtype=torch.bool, device="cuda")
    best[I0.view(-1)] = False
    legs = {
        "no_params": None,
        "all_rows": knn.IDSelectorRange(0, n),
        "random_50pct": knn.IDSelectorBatch(torch.nonzero(torch.rand(n, generator=gen, device="cuda") < 0.5).view(-1)),
        "random_1pct": knn.IDSelectorBatch(torch.nonzero(torch.rand(n, generator=gen, device="cuda") < 0.01).view(-1)),
        "mask_top1_of_every_query": knn.IDSelectorBatch(torch.nonzero(best).view(-1)),
    }
    out = {"rows": n, "queries": nq, "k": k, "masked_rows": int((~best).sum())}
    for name, sel in legs.items():
        p = knn.SearchParameters(sel=sel) if sel is not None else None
        fn = (lambda p=p: idx.search(xq, k, params=p))
        t = timed(fn, reps)
        out[name] = dict(qps=nq / t, seconds=t, **profile_stats(idx, fn))
    base = out["no_params"]["qps"]
    for name in legs:
        out[name]["vs_no_params"] = out[name]["qps"] / base
    return out


def bench_all_vs_all(knn, n, nq, reps, seed):
    import torch

    d, k = 1024, 1000
    x = rows(n, d, seed)
    idx = knn.IndexFlat(d, 0, device=0)
    idx.add(x)
    xq = x[:nq].contiguous()
    ex = torch.arange(nq, device="cuda", dtype=torch.int64)
    t_ex = timed(lambda: idx.search(xq, k, exclude=ex), reps)
    st_ex = profile_stats(idx, lambda: idx.search(xq, k, exclude=ex))
    t_k1 = timed(lambda: idx.search(xq, k + 1), reps)
    st_k1 = profile_stats(idx, lambda: idx.search(xq, k + 1))
    return {"rows": n, "queries": nq, "k": k,
            "exclude_self": dict(seconds=t_ex, qps=nq / t_ex, **st_ex),
            "search_k_plus_1": dict(seconds=t_k1, qps=nq / t_k1, **st_k1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-rows", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import knn_b200 as knn

    if not torch.cuda.is_available():
        sys.exit("bench_filtered: no CUDA device")
    res = {"gpu": gpu_info()}
    res["all_vs_all_c2"] = bench_all_vs_all(knn, 14433, 14433, args.reps, seed=2)
    res["all_vs_all_c3"] = bench_all_vs_all(knn, 300_000, 32768, args.reps, seed=3)
    torch.cuda.empty_cache()
    res["c4"] = bench_c4(knn, args.c4_rows, args.reps)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
