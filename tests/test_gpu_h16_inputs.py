"""fp16 / bf16 rows and queries read as they are (no fp32 copy): every call must return exactly what the same call
returns on the up-converted float32 rows - the same D and I bits, the same stored rows, the same shadow format.

a. ingest from the device, host numpy and CPU torch tensors, vector and scalar loads, misaligned sources, bf16 storage,
   several adds and a reset;
b. search: both metrics, every path, k from 1 to 2048, nq selecting every GEMM kernel and several query batches, host
   (pinned and pageable) and device queries, mixed database / query dtypes;
c. overflow repair with 16-bit queries on the device and host paths;
d. the adversarial error-bound cases with 16-bit queries;
e. the batch-wise two-phase ABI on three shards and ShardedIndexFlat in two processes;
f. no fp32 temporary on the device;
g. the drivers on fp16 .npy files;
h. misuse of the typed ABI."""
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


def _tdt(name):
    import torch

    return {"fp16": torch.float16, "bf16": torch.bfloat16}[name]


def _rows16(n, d, dt, seed, clustered=False):
    """(n, d) 16-bit rows on the device (clustered: many near-equal scores)."""
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, d, device="cuda", generator=g)
    if clustered:
        c = torch.randn(20, d, device="cuda", generator=g)
        x = c[torch.randint(0, 20, (n,), device="cuda", generator=g)] + 0.7 * x
    return x.to(_tdt(dt))


def _misaligned(x):
    """The same values in a contiguous view whose first element sits one element past an aligned address."""
    import torch

    if isinstance(x, np.ndarray):
        buf = np.empty(x.size + 1, x.dtype)
        v = buf[1:].reshape(x.shape)
        v[...] = x
        assert v.ctypes.data % 8 != 0
        return v
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 8 != 0 and v.is_contiguous()
    return v


def _host(x16, kind):
    """A device 16-bit matrix as host input of the given kind."""
    import torch

    if kind == "dev":
        return x16
    if kind == "numpy":
        assert x16.dtype == torch.float16
        return x16.cpu().numpy()
    if kind == "torch":
        return x16.cpu()
    if kind == "pinned_torch":
        return x16.cpu().pin_memory()
    if kind == "pinned_numpy":
        return x16.cpu().pin_memory().numpy()
    raise ValueError(kind)


def _eq(a, b):
    import torch

    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    return torch.equal(a, b)


def _same(D, I, D1, I1, what):
    assert _eq(I, I1), "ids differ from the fp32 call: %s" % (what,)
    assert _eq(D, D1), "distances differ from the fp32 call: %s" % (what,)


# ---- a. ingest ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [64, 100, 1024, 1900])
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("src", ["dev", "dev_misaligned", "numpy", "torch", "numpy_misaligned"])
def test_ingest_equals_ingesting_the_fp32_rows(knn, d, dt, src):
    if "numpy" in src and dt == "bf16":
        pytest.skip("numpy has no bfloat16")
    n = 9000 if d <= 1024 else 3000
    metric = IP if d in (64, 1024) else L2
    x16 = _rows16(n, d, dt, seed=d)
    x32 = x16.float()
    inp = _host(x16, "numpy" if "numpy" in src else "torch" if src == "torch" else "dev")
    if src.endswith("misaligned"):
        inp = _misaligned(inp)
    a, b = knn.IndexFlat(d, metric, device=0), knn.IndexFlat(d, metric, device=0)
    a.add(inp)
    b.add(x32)
    assert a.ntotal == b.ntotal == n
    assert np.array_equal(a.reconstruct_n(0, n), x32.cpu().numpy()), "stored rows are not the up-converted rows"
    assert a.stat("shadow_fmt") == b.stat("shadow_fmt")
    q = _rows16(64, d, dt, seed=d + 1).float()
    for path in (1, 2):
        a.set_param("path", path)
        b.set_param("path", path)
        D, I = a.search(q, 10)
        D1, I1 = b.search(q, 10)
        _same(D, I, D1, I1, (d, dt, src, path))
        assert a.stat("shadow_fmt") == b.stat("shadow_fmt") and a.stat("path") == path


@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("metric", [IP, L2])
def test_bf16_storage_with_16bit_rows(knn, dt, metric):
    """bf16 rows are stored as they are, fp16 rows as bf16(float(x)) - exactly what the fp32 rows give."""
    import torch

    d, n = 256, 10000
    x16 = _rows16(n, d, dt, seed=5 + metric)
    a = knn.IndexFlat(d, metric, device=0, bf16_storage=True)
    b = knn.IndexFlat(d, metric, device=0, bf16_storage=True)
    a.add(x16)
    b.add(x16.float())
    ra, rb = a.reconstruct_n(), b.reconstruct_n()
    assert np.array_equal(ra, rb)
    if dt == "bf16":
        assert np.array_equal(ra, x16.float().cpu().numpy())
    else:
        assert np.array_equal(ra, x16.float().to(torch.bfloat16).float().cpu().numpy())
    q = _rows16(300, d, dt, seed=9)
    for path in (1, 2):
        a.set_param("path", path)
        b.set_param("path", path)
        D, I = a.search(q, 50)
        D1, I1 = b.search(q.float(), 50)
        _same(D, I, D1, I1, (dt, metric, path))


@pytest.mark.parametrize("dt", ["fp16", "bf16"])
def test_several_adds_and_add_after_reset(knn, dt):
    d = 128
    x16 = _rows16(20000, d, dt, seed=11, clustered=True)
    q16 = _rows16(500, d, dt, seed=12, clustered=True)
    a, b = knn.IndexFlat(d, L2, device=0), knn.IndexFlat(d, L2, device=0)
    cuts = [0, 7000, 7001, 15000, 20000]
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        part = x16[lo:hi]
        a.add(part if lo % 2 == 0 else _host(part, "torch"))
        b.add(part.float())
        D, I = a.search(q16, 20)
        D1, I1 = b.search(q16.float(), 20)
        _same(D, I, D1, I1, ("after add", hi))
    assert np.array_equal(a.reconstruct_n(), b.reconstruct_n())
    a.reset()
    b.reset()
    a.add(x16[:12000])
    b.add(x16[:12000].float())
    assert a.stat("shadow_fmt") == b.stat("shadow_fmt")
    D, I = a.search(q16, 20)
    D1, I1 = b.search(q16.float(), 20)
    _same(D, I, D1, I1, "after reset")


# ---- b. search ----------------------------------------------------------------------------------------------------
_DBS = {}


def _db_pair(knn, metric):
    """An index built from fp16 rows and its twin built from the up-converted rows (20,000 x 64, clustered)."""
    if metric not in _DBS:
        x16 = _rows16(20000, 64, "fp16", seed=100 + metric, clustered=True)
        a, b = knn.IndexFlat(64, metric, device=0), knn.IndexFlat(64, metric, device=0)
        a.add(x16)
        b.add(x16.float())
        _DBS[metric] = (a, b, x16)
    return _DBS[metric]


# query kinds: (query dtype, where) - device tensors, host numpy (pageable, pinned), CPU torch (pageable, pinned)
QUERY_KINDS = [("bf16", "dev"), ("fp16", "dev"), ("fp16", "numpy"), ("fp16", "pinned_numpy"), ("bf16", "torch"),
               ("bf16", "pinned_torch"), ("f32", "dev")]


@pytest.mark.parametrize("k", [1, 100, 1000, 2048])
@pytest.mark.parametrize("path", [0, 1, 2])
@pytest.mark.parametrize("metric", [IP, L2])
def test_search_with_16bit_queries_equals_fp32_call(knn, metric, path, k):
    a, b, x16 = _db_pair(knn, metric)
    a.set_param("path", path)
    b.set_param("path", path)
    for nq in (1, 64, 128, 256, 20000):
        if nq == 20000 and k > 100:
            continue  # several query batches at k <= 100 (result rows of 2048 are covered at nq <= 256)
        q = _rows16(nq, 64, "bf16", seed=nq + k, clustered=True)
        for qdt, where in QUERY_KINDS:
            if nq == 20000 and where not in ("dev", "numpy", "pinned_torch"):
                continue
            q16 = q.float() if qdt == "f32" else q.float().to(_tdt(qdt))
            inp = _host(q16, where) if qdt != "f32" else q16
            D, I = a.search(inp, k)
            D1, I1 = b.search(q16.float().cpu().numpy() if where != "dev" else q16.float(), k)
            if where != "dev":
                assert isinstance(D, np.ndarray)
            _same(D, I, D1, I1, (metric, path, k, nq, qdt, where))
            assert a.stat("path") == b.stat("path")
            if path:
                assert a.stat("path") == path or (path == 2 and a.ntotal < k)
        if nq == 256 and k in (1, 100):
            sample = np.arange(0, 256, 37)
            qs = q.float().cpu().numpy()[sample]
            D, I = a.search(q[sample.tolist()].contiguous(), k)
            xb = x16.float().cpu().numpy()
            D_ref, I_ref = fo.knn_flat(qs, xb, k, metric, want=k + 4)
            check_parity(D.cpu().numpy(), I.cpu().numpy(), D_ref, I_ref, qs, xb, metric)


def test_search_filter_and_finish_with_16bit_queries(knn):
    """The all-batches two-phase form (search_filter / search_finish) on one shard."""
    a, b, _ = _db_pair(knn, IP)
    a.set_param("path", 0)
    b.set_param("path", 0)
    q = _rows16(700, 64, "fp16", seed=3, clustered=True)
    lo, lo_j = a.search_filter(q, 100, 100)
    lo1, lo_j1 = b.search_filter(q.float(), 100, 100)
    assert _eq(lo, lo1) and _eq(lo_j, lo_j1)
    D1, I1 = b.search_finish(lo1, 100)
    D, I = a.search_finish(lo, 100)
    _same(D, I, D1, I1, "two-phase, one shard")


# ---- c. overflow repair -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("where", ["dev", "host"])
def test_overflow_repair_with_16bit_queries(knn, dt, where):
    """Massively duplicated rows: candidate lists overflow and the flagged queries are redone by the exact scan,
    whose query rows are gathered from the 16-bit input (device) or copied from it (host)."""
    d, n, k = 64, 60000, 20
    x16 = _rows16(n, d, dt, seed=21)
    x16[10000:40000] = x16[10000]
    q16 = _rows16(500, d, dt, seed=22)
    q16[[3, 77, 400]] = x16[10000]
    a = knn.IndexFlat(d, IP, device=0)
    a.set_param("path", 2)
    a.add(x16)
    b = knn.IndexFlat(d, IP, device=0)
    b.set_param("path", 2)
    b.add(x16.float())
    if where == "dev":
        D, I = a.search(q16, k)
        D1, I1 = b.search(q16.float(), k)
    else:
        D, I = a.search(q16.cpu() if dt == "bf16" else q16.cpu().numpy(), k)
        D1, I1 = b.search(q16.float().cpu().numpy(), k)
    assert a.stat("overflow_queries") > 0, "no candidate list overflowed: the repair went untested"
    assert a.stat("overflow_queries") == b.stat("overflow_queries")
    _same(D, I, D1, I1, (dt, where))
    I = I.cpu().numpy() if not isinstance(I, np.ndarray) else I
    assert np.array_equal(I[3], np.arange(10000, 10000 + k))


# ---- d. error bound --------------------------------------------------------------------------------------------
ADV_CASES = [
    ("bf16-ip-main", dict(nq=300, d=1024, k=10, fmt="bf16")),
    ("bf16-l2-stream", dict(nq=60, d=1024, k=10, fmt="bf16", metric=L2)),
    ("bf16-ip-pair", dict(nq=100, d=1024, k=10, fmt="bf16")),
    ("bf16-l2-d64", dict(nq=640, d=64, k=8, fmt="bf16", metric=L2)),
    ("fp16-ip-main", dict(nq=300, d=1024, k=10, fmt="fp16")),
    ("fp16-l2-pair", dict(nq=120, d=1024, k=10, fmt="fp16", metric=L2)),
    ("fp16-ip-d64", dict(nq=300, d=64, k=10, fmt="fp16")),
    ("fp16-l2-block-k300", dict(nq=8, d=1024, k=300, n_decoys=302, fmt="fp16", metric=L2)),
]


@pytest.mark.parametrize("name,kw", ADV_CASES, ids=[c[0] for c in ADV_CASES])
@pytest.mark.parametrize("where", ["dev", "host"])
def test_adversarial_cases_with_16bit_queries(knn, name, kw, where):
    """oracle/adversarial.py's dy-aligned cases (queries are +-a, exact in 16 bits) with the queries passed in the
    operand format's own dtype: every hidden row found, no overflow fallback, bit-identical to the fp32 call."""
    import torch

    kw = dict(kw)
    nq, d, k = kw.pop("nq"), kw.pop("d"), kw.pop("k")
    case = adv.dy_aligned(nq, d, k, seed=sum(map(ord, name)), **kw)
    q16 = torch.from_numpy(case.xq).cuda().to(_tdt(case.fmt))
    assert torch.equal(q16.float().cpu(), torch.from_numpy(case.xq)), "the case's queries are not 16-bit exact"
    idx = knn.IndexFlat(d, case.metric, device=0)
    idx.set_param("path", 2)
    idx.set_param("shadow_fmt", {"bf16": 1, "fp16": 2}[case.fmt])
    idx.add(case.xb)
    if where == "dev":
        D, I = idx.search(q16, k)
        D, I = D.cpu().numpy(), I.cpu().numpy()
    else:
        D, I = idx.search(q16.cpu() if case.fmt == "bf16" else q16.cpu().numpy(), k)
    assert idx.stat("path") == 2 and idx.stat("overflow_batches") == 0
    for q in range(case.hidden.shape[0]):
        missing = set(case.hidden[q].tolist()) - set(I[q].tolist())
        assert not missing, "query %d lost hidden rows %s" % (q, sorted(missing))
    D1, I1 = idx.search(case.xq, k)
    _same(D, I, D1, I1, name)
    D_ref, I_ref = fo.knn_flat(case.xq, case.xb, k, case.metric, want=k + 4)
    check_parity(D, I, D_ref, I_ref, case.xq, case.xb, case.metric)


# ---- e. two-phase ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", ["fp16", "bf16"])
@pytest.mark.parametrize("metric,k", [(IP, 10), (L2, 100), (IP, 1000)])
def test_batchwise_two_phase_three_shards_with_16bit_queries(knn, dt, metric, k):
    """Tensor-path, exact-path and empty shards, run step for step as ShardedIndexFlat._two_phase_pipelined runs them
    (tests/test_gpu_two_phase.py), with 16-bit queries: equal to one unsharded index searched with the fp32 queries."""
    from test_gpu_two_phase import _pipelined

    d, nq = 64, 700
    rows = [9000, 5000, 0]  # tensor path, below tensor_min_n (exact scan), empty
    starts = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    x16 = _rows16(int(starts[-1]), d, dt, seed=31 + k, clustered=True)
    q16 = _rows16(nq, d, dt, seed=32 + k, clustered=True)

    def make(rows_):
        idx = knn.IndexFlat(d, metric, device=0)
        idx.set_param("query_batch", 256)
        if rows_.shape[0]:
            idx.add(rows_)
        return idx

    full = make(x16.float())
    full.set_param("path", 2)
    D1, I1 = full.search(q16.float(), k)
    shards = [make(x16[a:a + r]) for a, r in zip(starts, rows)]
    Dm, Im, geo = _pipelined(knn, shards, [int(a) for a in starts[:-1]], q16, k, "torch")
    assert [int(sh.stat("path")) for sh in shards] == [2, 1, 1]
    _same(Dm, Im, D1, I1, (dt, metric, k, geo))
    sample = np.arange(0, nq, 61)
    xb, xq = x16.float().cpu().numpy(), q16.float().cpu().numpy()[sample]
    D_ref, I_ref = fo.knn_flat(xq, xb, k, metric, want=k + 4)
    check_parity(Dm.cpu().numpy()[sample], Im.cpu().numpy()[sample], D_ref, I_ref, xq, xb, metric)


def _sharded_worker(rank, world, port, out_dir):
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
    d, n = 64, 20000
    g = torch.Generator(device="cuda").manual_seed(5)  # every rank holds the same rows and queries
    xb = torch.randn(n, d, device="cuda", generator=g)
    xq = torch.randn(700, d, device="cuda", generator=g)
    for metric, dt in [(IP, torch.bfloat16), (L2, torch.float16)]:
        xb16, xq16 = xb.to(dt), xq.to(dt)
        index = ShardedIndexFlat(d, metric, device=0, exchange_bounds=True, peer_merge=True)
        index.local.set_param("query_batch", 256)
        index.add(xb16[:n // 3])
        index.add(xb16[n // 3:])
        single = knn_b200.IndexFlat(d, metric, device=0)
        single.add(xb16.float())
        for k in (10, 1000):
            D, I = index.search(xq16, k)
            D1, I1 = single.search(xq16.float(), k)
            assert torch.equal(I, I1) and torch.equal(D, D1), (rank, metric, dt, k, "device queries")
            if dt == torch.float16:  # host numpy queries of every rank
                Dh, Ih = index.search(xq16.cpu().numpy(), k)
                assert np.array_equal(Ih, I1.cpu().numpy()) and np.array_equal(Dh, D1.cpu().numpy()), (rank, k, "host")
            done.append((rank, metric, str(dt), k, int(index.local.stat("path"))))
        index.close()
        dist.barrier()
    (Path(out_dir) / ("rank%d" % rank)).write_text(repr(done))
    dist.destroy_process_group()


def test_sharded_index_with_16bit_rows_and_queries_two_processes_one_gpu(tmp_path):
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=False)
    deadline = time.time() + 180
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("two-process sharded search did not finish in 180 s")
    done = [eval((tmp_path / ("rank%d" % r)).read_text()) for r in range(2)]
    assert len(done[0]) == len(done[1]) == 4
    assert all(t[4] == 2 for t in done[0] + done[1])


# ---- f. no fp32 temporary ---------------------------------------------------------------------------------------
def test_bf16_add_and_search_make_no_fp32_copy(knn):
    """The library allocates with cudaMalloc, so torch's allocator sees exactly the transients of the Python layer: the
    old path's x.to(float32) showed up here as a full fp32 copy."""
    import torch

    n, d, nq = 1 << 20, 1024, 65536
    x = _rows16(n, d, "bf16", seed=41)
    q = _rows16(nq, d, "bf16", seed=42)
    idx = knn.IndexFlat(d, IP, device=0)
    idx.reserve(n)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    idx.add(x)
    torch.cuda.synchronize()
    transient = torch.cuda.max_memory_allocated() - max(base, torch.cuda.memory_allocated())
    assert transient < 0.01 * n * d * 4, "add allocated %d bytes on the side" % transient
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    D, I = idx.search(q, 10)
    torch.cuda.synchronize()
    transient = torch.cuda.max_memory_allocated() - max(base, torch.cuda.memory_allocated())
    assert transient < 0.01 * nq * d * 4, "search allocated %d bytes on the side" % transient
    D1, I1 = idx.search(q.float(), 10)
    _same(D, I, D1, I1, "large bf16 search")


# ---- g. drivers -------------------------------------------------------------------------------------------------
def test_search_and_save_on_fp16_files_equals_the_fp32_cast(knn, tmp_path):
    from knn_b200 import drivers

    rng = np.random.default_rng(51)
    d16, d32 = tmp_path / "fp16", tmp_path / "fp32"
    d16.mkdir()
    d32.mkdir()
    # "c" (134 MB in fp16) goes through the chunked upload over the pinned bounce buffers
    for name, shape in [("a", (3000, 128)), ("b", (2500, 1024)), ("c", (65600, 1024))]:
        x = (rng.standard_normal(shape) * 0.3).astype(np.float16)
        np.save(d16 / (name + ".npy"), x)
        np.save(d32 / (name + ".npy"), x.astype(np.float32))
    drivers.search_and_save(d16, device=0)
    drivers.search_and_save(d32, device=0)
    for metric in ("cosine", "euclidean"):
        for kind in ("hits", "scores"):
            a = np.load(d16 / ("%s_%s.npz" % (kind, metric)))
            b = np.load(d32 / ("%s_%s.npz" % (kind, metric)))
            assert sorted(a.files) == sorted(b.files) == ["a", "b", "c"]
            for f in a.files:
                assert a[f].dtype == b[f].dtype and np.array_equal(a[f], b[f]), (metric, kind, f)


def test_proteins_search_on_an_fp16_file_equals_the_fp32_cast(knn, tmp_path):
    from knn_b200 import drivers

    x = (np.random.default_rng(52).standard_normal((5000, 256))).astype(np.float16)
    out = {}
    for tag, arr in [("fp16", x), ("fp32", x.astype(np.float32))]:
        (tmp_path / tag).mkdir()
        np.save(tmp_path / tag / "full_sequences.npy", arr)
        out[tag] = drivers.proteins_search(tmp_path / tag, k=100, device=0)
        out[tag] += ((tmp_path / tag / "full_sequences_flat.index").read_bytes(),)
    assert np.array_equal(out["fp16"][0], out["fp32"][0]) and np.array_equal(out["fp16"][1], out["fp32"][1])
    assert out["fp16"][2] == out["fp32"][2]


# ---- h. misuse ---------------------------------------------------------------------------------------------------
def test_unknown_dtype_and_mismatched_finish_are_rejected(knn):
    import torch

    lib = knn._lib.load()
    idx = knn.IndexFlat(32, IP, device=0)
    x = torch.randn(10000, 32, device="cuda").to(torch.float16)
    idx.add(x)
    h, s = idx._h, torch.cuda.current_stream().cuda_stream
    xh = x.cpu().numpy()
    D = torch.empty((300, 10), device="cuda")
    I = torch.empty((300, 10), dtype=torch.int64, device="cuda")
    Dh, Ih = np.empty((300, 10), np.float32), np.empty((300, 10), np.int64)
    nb, rows = ctypes.c_int64(), ctypes.c_int64()
    lower = torch.empty(300, device="cuda")
    for bad in (-1, 3, 7):
        assert lib.knn_index_add_typed(h, 5, xh.ctypes.data, bad) == ERR_INVALID
        assert lib.knn_index_add_typed_dev(h, 5, x.data_ptr(), bad, s) == ERR_INVALID
        assert lib.knn_index_search_typed(h, 300, xh.ctypes.data, bad, 10, Dh.ctypes.data, Ih.ctypes.data) == ERR_INVALID
        assert lib.knn_index_search_typed_dev(h, 300, x.data_ptr(), bad, 10, D.data_ptr(), I.data_ptr(), 0, s) == ERR_INVALID
        assert lib.knn_index_search_begin_typed_dev(h, 300, x.data_ptr(), bad, 10, ctypes.byref(nb), ctypes.byref(rows),
                                                    s) == ERR_INVALID
        assert lib.knn_index_search_filter_typed_dev(h, 300, x.data_ptr(), bad, 10, lower.data_ptr(), 0, None, s) == ERR_INVALID
        assert "dtype" in lib.knn_last_error().decode()
    assert idx.ntotal == 10000  # nothing was added
    q = x[:300]
    assert lib.knn_index_search_filter_typed_dev(h, 300, q.data_ptr(), F16, 10, lower.data_ptr(), 0, None, s) == 0
    for other in (F32, BF16):
        assert lib.knn_index_search_finish_typed_dev(h, 300, q.data_ptr(), other, 10, lower.data_ptr(), D.data_ptr(),
                                                     I.data_ptr(), 0, s) == ERR_INVALID
    assert lib.knn_index_search_finish_typed_dev(h, 300, q.data_ptr(), F16, 10, lower.data_ptr(), D.data_ptr(),
                                                 I.data_ptr(), 0, s) == 0
    D1, I1 = idx.search(q.float(), 10)
    _same(D, I, D1, I1, "two-phase after a rejected finish")
