"""The tensor path's error bound eps against data that reaches it (oracle/adversarial.py; the data itself is checked
on the CPU by tests/test_adversarial_data.py).  Every query has hidden rows, rounded down by ~eps, that belong to
the exact top-k, and >= k decoys rounded up by ~eps above them: the filter keeps the hidden rows only if its margin
really is 2 eps.  Each case must be answered by the filter itself (no overflow fallback), contain every hidden row,
equal the exact fp32 scan bit for bit and pass the oracle parity check.  Covered: every GEMM kernel, hidden rows in
the dense first panel and in late panels, both tighten kernels, every operand format, the stats after a second add /
a format switch / a reset, the two-phase bounds and the sharded path, and L2 with rows ~4000 x longer than the
queries (where the bound is dominated by fp32 roundings of |y|^2)."""
import numpy as np
import pytest

from oracle import adversarial as adv
from oracle import flat_oracle as fo
from oracle.parity import check_parity

pytestmark = pytest.mark.gpu

IP, L2 = 0, 1
FMT_PARAM = {"bf16": 1, "fp16": 2}


@pytest.fixture(scope="module")
def knn():
    import knn_b200

    assert knn_b200._lib.load().knn_device_count() >= 1, "no CUDA device: the CUDA path cannot run"
    return knn_b200


def _index(knn, case, path, params):
    idx = knn.IndexFlat(case.xb.shape[1], case.metric, bf16_storage=case.bf16_storage)
    idx.set_param("path", path)
    if not case.bf16_storage:
        idx.set_param("shadow_fmt", FMT_PARAM[case.fmt])
        if case.fmt == "bf16" and case.mbits != 7:
            idx.set_param("mantissa_bits", case.mbits)
    for name, v in params.items():
        idx.set_param(name, v)
    return idx


def _exact(knn, case):
    idx = _index(knn, case, 1, {})
    idx.add(case.xb)
    D, I = idx.search(case.xq, case.k)
    assert idx.stat("path") == 1
    return D, I


def _check(knn, case, D, I, idx, exact=None):
    """The four things every case asserts."""
    assert idx.stat("path") == 2
    assert idx.stat("overflow_batches") == 0, "the exact-scan fallback answered: the case proves nothing"
    if case.fmt == "bf16" and not case.bf16_storage:
        assert idx.stat("mantissa_bits") == case.mbits
    for q in range(case.hidden.shape[0]):
        missing = set(case.hidden[q].tolist()) - set(I[q].tolist())
        assert not missing, "query %d lost hidden rows %s" % (q, sorted(missing))
    D1, I1 = exact if exact is not None else _exact(knn, case)
    assert np.array_equal(I, I1) and np.array_equal(D, D1), "tensor path differs from the exact fp32 scan"
    D_ref, I_ref = fo.knn_flat(case.xq, case.xb, case.k, case.metric, want=case.k + 4)
    # no cap on tie-excused positions: a query's hidden rows (and its decoys) are permutations of each other with
    # identical fp64 scores, which two fp32 summation orders rank differently
    check_parity(D, I, D_ref, I_ref, case.xq, case.xb, case.metric)


def _search(knn, case, params=None):
    idx = _index(knn, case, 2, params or {})
    idx.add(case.xb)
    D, I = idx.search(case.xq, case.k)
    _check(knn, case, D, I, idx)
    return idx


# ---- GEMM kernels, panels, tighten kernels, formats -------------------------------------------------------------
# (id, generator kwargs, index params).  nq selects the GEMM kernel: <= 64 the few-queries kernel, 65-128 its CTA-pair
# form, 129-256 the main kernel or (stream_quad) the two-pair form, >= 257 the main kernel (cta_group 1 or 2); the
# tighten is the warp-per-query kernel for k <= 256 with > 512 queries, the block-per-query kernel otherwise.
CASES = [
    ("main-cg2-ip-bf16", dict(nq=300, d=1024, k=10), {}),
    ("main-cg1-l2-bf16", dict(nq=300, d=1024, k=10, metric=L2), {"cta_group": 1}),
    ("main-cg2-l2-bf16-front", dict(nq=300, d=1024, k=10, metric=L2, layout="front"), {}),
    ("main-cg1-ip-bf16-front", dict(nq=300, d=1024, k=10, layout="front"), {"cta_group": 1}),
    ("stream32-ip-bf16", dict(nq=24, d=1024, k=10), {}),
    ("stream64-l2-bf16", dict(nq=60, d=1024, k=10, metric=L2), {}),
    ("stream-pair-ip-bf16", dict(nq=100, d=1024, k=10), {}),
    ("stream-pair-l2-fp16", dict(nq=120, d=1024, k=10, metric=L2, fmt="fp16"), {}),
    ("main-256-ip-bf16", dict(nq=200, d=1024, k=10), {}),
    ("stream-quad-ip-bf16", dict(nq=200, d=1024, k=10), {"stream_quad": 1}),
    ("stream-quad-l2-bf16", dict(nq=250, d=1024, k=10, metric=L2), {"stream_quad": 1}),
    ("warp-tighten-ip-bf16", dict(nq=600, d=1024, k=10), {}),
    ("warp-tighten-l2-bf16", dict(nq=600, d=1024, k=16, metric=L2, layout="shuffled"), {}),
    ("block-tighten-k300-ip-bf16", dict(nq=8, d=1024, k=300, n_decoys=302), {}),
    ("block-tighten-k300-l2-fp16", dict(nq=8, d=1024, k=300, n_decoys=302, metric=L2, fmt="fp16"), {}),
    ("mbits5-ip", dict(nq=300, d=1024, k=10, fmt="bf16", mbits=5), {}),
    ("mbits5-l2-stream", dict(nq=40, d=1024, k=10, fmt="bf16", mbits=5, metric=L2), {}),
    ("fp16-ip-main", dict(nq=300, d=1024, k=10, fmt="fp16"), {}),
    ("fp16-ip-d64", dict(nq=300, d=64, k=10, fmt="fp16"), {}),
    ("fp16-l2-d64-stream", dict(nq=48, d=64, k=10, fmt="fp16", metric=L2), {}),
    ("bf16-l2-d64-warp", dict(nq=640, d=64, k=8, metric=L2), {}),
]


@pytest.mark.parametrize("name,kw,params", CASES, ids=[c[0] for c in CASES])
def test_dy_aligned_hidden_rows_survive(knn, name, kw, params):
    kw = dict(kw)
    nq, d, k = kw.pop("nq"), kw.pop("d"), kw.pop("k")
    case = adv.dy_aligned(nq, d, k, seed=sum(map(ord, name)), **kw)
    _search(knn, case, params)


@pytest.mark.parametrize("metric", [IP, L2])
@pytest.mark.parametrize("nq", [48, 300])
def test_dx_aligned_queries_on_bf16_storage(knn, metric, nq):
    case = adv.dx_aligned(nq, 1024, 10, metric=metric, seed=7 * nq + metric)
    _search(knn, case)


# ---- stats lifecycle ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [IP, L2])
def test_adversarial_rows_in_a_second_add(knn, metric):
    """max|y| and max|dy| must grow with the rows of a later add: the first add holds only exact background rows
    (dy = 0), the adversarial rows arrive in the second."""
    case = adv.dy_aligned(300, 1024, 10, metric=metric, layout="bg_first", seed=31 + metric)
    n_adv = case.hidden.size + case.decoys.size
    split = case.xb.shape[0] - n_adv
    idx = _index(knn, case, 2, {})
    idx.add(case.xb[:split])
    idx.search(case.xq, case.k)  # a search between the two adds: the bound of the first part is in use
    idx.add(case.xb[split:])
    D, I = idx.search(case.xq, case.k)
    _check(knn, case, D, I, idx)


@pytest.mark.parametrize("metric", [IP, L2])
def test_shadow_format_switch_remeasures_stats(knn, metric):
    """bf16-adversarial rows first searched through fp16 shadow rows (whose rounding error is far smaller), then
    through bf16 ones: the conversion must re-measure max|dy|, else the bf16 bound is the fp16 one."""
    case = adv.dy_aligned(300, 1024, 10, metric=metric, seed=41 + metric)
    idx = _index(knn, case, 2, {"shadow_fmt": 2})
    idx.add(case.xb)
    D16, I16 = idx.search(case.xq, case.k)
    assert idx.stat("shadow_fmt") == 2
    exact = _exact(knn, case)
    assert np.array_equal(I16, exact[1]) and np.array_equal(D16, exact[0])
    idx.set_param("shadow_fmt", 1)
    D, I = idx.search(case.xq, case.k)
    assert idx.stat("shadow_fmt") == 1 and idx.stat("shadow_conversions") >= 1
    _check(knn, case, D, I, idx, exact)
    # and back (fp16 stats after bf16 ones)
    idx.set_param("shadow_fmt", 2)
    D, I = idx.search(case.xq, case.k)
    assert np.array_equal(I, exact[1]) and np.array_equal(D, exact[0])


@pytest.mark.parametrize("metric", [IP, L2])
def test_stats_after_reset(knn, metric):
    """After reset the bound is measured from the new rows: exact rows (max|dy| = 0) first, reset, then the
    adversarial rows - whose dy must be counted; and the reverse, checked against the exact scan."""
    case = adv.dy_aligned(300, 1024, 10, metric=metric, seed=51 + metric)
    idx = _index(knn, case, 2, {})
    rng = np.random.default_rng(5)
    idx.add((rng.choice([-1.0, 1.0], size=(9000, 1024)) * (1.0 + 2.0 ** -7)).astype(np.float32))  # max|dy| = 0
    idx.search(case.xq, case.k)
    idx.reset()
    idx.add(case.xb)
    D, I = idx.search(case.xq, case.k)
    _check(knn, case, D, I, idx)
    # the reverse: exact rows after adversarial ones keep nothing of them
    idx.reset()
    xb2 = (rng.standard_normal((9000, 1024)) * 0.01).astype(np.float32)
    idx.add(xb2)
    D2, I2 = idx.search(case.xq, case.k)
    ex = _index(knn, case, 1, {})
    ex.add(xb2)
    assert np.array_equal(I2, ex.search(case.xq, case.k)[1])


# ---- bound exports -----------------------------------------------------------------------------------------
def _kth_exact(case, xb, j):
    s = adv.exact_scores(case.xq, xb, case.metric)
    return -np.sort(-s, axis=1)[:, j - 1]


@pytest.mark.parametrize("metric", [IP, L2])
@pytest.mark.parametrize("fmt", ["bf16", "fp16"])
def test_search_filter_bounds_hold(knn, metric, fmt, capsys):
    """lower <= fp64 k-th best and lower_j <= fp64 j-th best, with no tolerance (L2: in key space
    2<x,y> - |y|^2, what the filter compares)."""
    import torch

    case = adv.dy_aligned(300, 1024, 10, metric=metric, fmt=fmt, seed=61 + metric)
    idx = _index(knn, case, 2, {})
    idx.add(case.xb)
    tq = torch.from_numpy(case.xq).cuda()
    j = 4
    lower, lower_j = idx.search_filter(tq, case.k, j)
    lower, lower_j = lower.double().cpu().numpy(), lower_j.double().cpu().numpy()
    ref_k, ref_j = _kth_exact(case, case.xb, case.k), _kth_exact(case, case.xb, j)
    eps = case.eps()
    with capsys.disabled():
        print("\n  %s %s: max (lower - k-th)/eps = %.3f, max (lower_j - j-th)/eps = %.3f"
              % (fmt, "L2" if metric else "IP", ((lower - ref_k) / eps).max(), ((lower_j - ref_j) / eps).max()))
    assert np.all(lower > -3e38) and np.all(lower_j > -3e38)
    assert np.all(lower <= ref_k), "lower above the true k-th best"
    assert np.all(lower_j <= ref_j), "lower_j above the true j-th best"
    D, I = idx.search_finish(torch.from_numpy(lower.astype(np.float32)).cuda(), case.k)
    _check(knn, case, D.cpu().numpy(), I.cpu().numpy(), idx)


@pytest.mark.parametrize("metric", [IP, L2])
def test_two_phase_sharded_hidden_rows_in_a_low_eps_shard(knn, metric):
    """Three shards with different eps: hidden rows (and background) in a low-eps shard, decoys in a shard whose
    long, coarsely rounded extra rows raise its eps, the third shard exact background.  The merged result must equal
    the single index bit for bit (pattern of test_gpu_parity.py::test_two_phase_sharded_search_equals_single_index)."""
    import torch

    case = adv.dy_aligned(300, 1024, 10, metric=metric, layout="front", seed=71 + metric)
    rng = np.random.default_rng(3)
    nh, nd = case.hidden.size, case.decoys.size
    n = case.xb.shape[0]
    # rows: [hidden | background | decoys] (layout "front"); the decoy shard gets 64 heavy rows with scores far
    # below the adversarial ones: magnitudes ~3 on the bf16 grid (step 2u there) plus 0.9 u, which rounds away -
    # 7 x the adversarial rows' |dy|, in random directions
    u = 2.0 ** -7
    mag = 2 * u * np.round((3.0 + 3 * u * rng.integers(2, 20, size=(64, 1024))) / (2 * u)) + 0.9 * u
    heavy = (rng.choice([-1.0, 1.0], size=(64, 1024)) * mag).astype(np.float32)
    xb = np.concatenate([case.xb, heavy])
    bounds = [0, nh + (n - nh - nd) // 2, n - nd, xb.shape[0]]
    # shard 0: hidden rows + background, shard 1: background, shard 2: decoys + heavy rows
    dev = torch.device("cuda:0")
    tq = torch.from_numpy(case.xq).to(dev)
    full = _index(knn, case, 2, {})
    full.add(xb)
    D, I = full.search(tq, case.k)
    shards, eps_shard = [], []
    for a, b in zip(bounds[:-1], bounds[1:]):
        sh = _index(knn, case, 2, {})
        sh.add(torch.from_numpy(xb[a:b]).to(dev))
        shards.append(sh)
        eps_shard.append(adv.eps_reference(case.xq, xb[a:b], case.fmt, case.mbits, metric).mean())
    assert eps_shard[2] > 1.5 * eps_shard[0], eps_shard
    j = -(-case.k // len(shards))
    both = [sh.search_filter(tq, case.k, j) for sh in shards]
    lower = torch.maximum(torch.stack([b[0] for b in both]).max(dim=0).values,
                          torch.stack([b[1] for b in both]).min(dim=0).values)
    ref_k = _kth_exact(case, xb, case.k)
    assert np.all(lower.double().cpu().numpy() <= ref_k)
    Ds, Is = zip(*[sh.search_finish(lower, case.k, id_base=a) for sh, a in zip(shards, bounds[:-1])])
    for sh in shards:
        assert sh.stat("overflow_batches") == 0
    Dm, Im = knn.merge_topk(torch.stack(Ds), torch.stack(Is), metric)
    assert torch.equal(Im, I) and torch.equal(Dm, D)
    Im = Im.cpu().numpy()
    for q in range(case.hidden.shape[0]):
        assert set(case.hidden[q].tolist()) <= set(Im[q].tolist())
    D1, I1 = fo.knn_flat(case.xq, xb, case.k, metric, want=case.k + 4)
    check_parity(Dm.cpu().numpy(), Im, D1, I1, case.xq, xb, metric)


# ---- L2 with rows far longer than the queries --------------------------------------------------------------
@pytest.mark.parametrize("nq", [40, 300])
def test_l2_extreme_norm_ratio(knn, nq, capsys):
    """16-bit-exact rows ~4000 x longer than the queries: the inner-product bound is only the fp32 slack, far below
    ulp(|y|^2); the filter must still be exact and `lower` a true lower bound of the k-th best key."""
    import torch

    case = adv.l2_extreme_ratio(nq, 64, 10, seed=nq)
    for fmt in ("bf16", "fp16"):
        case.fmt = fmt
        idx = _index(knn, case, 2, {})
        idx.add(case.xb)
        D, I = idx.search(case.xq, case.k)
        _check(knn, case, D, I, idx)
        lower = idx.search_filter(torch.from_numpy(case.xq).cuda(), case.k).double().cpu().numpy()
        ref_k = _kth_exact(case, case.xb, case.k)
        with capsys.disabled():
            print("\n  L2 extreme %s nq=%d: max (lower - k-th key) = %.3g, eps = %.3g"
                  % (fmt, nq, (lower - ref_k).max(), case.eps().max()))
        assert np.all(lower <= ref_k), "lower above the true k-th best key"
