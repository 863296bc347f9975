"""The adversarial data of oracle/adversarial.py is what it claims to be, proved on the CPU before any GPU sees it:
the realised 16-bit score error reaches the error bound eps (restated from query_eps_kernel), the hidden rows are in
the exact top-k, and >= k decoys outrank every hidden row in 16-bit score.  tests/test_gpu_error_bound.py then
requires the tensor path to find the hidden rows anyway."""
import numpy as np
import pytest

from oracle import adversarial as adv
from oracle import flat_oracle as fo

IP, L2 = adv.METRIC_INNER_PRODUCT, adv.METRIC_L2

# (fmt, mantissa bits, d) -> least realised |16-bit score - fp64 score| / eps over the adversarial rows
FLOORS = {("bf16", 7, 1024): 0.85, ("bf16", 5, 1024): 0.85, ("fp16", 10, 1024): 0.5,
          ("bf16", 7, 64): 0.9, ("bf16", 5, 64): 0.9, ("fp16", 10, 64): 0.9}


def _check_case(case, floor):
    nq = case.xq.shape[0]
    r = np.arange(nq)[:, None]
    ex, ap, eps = case.exact(), case.approx(), case.eps()
    assert np.all(eps > 0)
    err = np.abs(ap - ex) / eps[:, None]
    assert err.max() <= 1.0, "the bound must hold: %r" % err.max()
    adv_err = np.concatenate([err[r, case.hidden], err[r, case.decoys]], axis=1)
    assert adv_err.min() >= floor, "realised error / eps only %.3f" % adv_err.min()
    # hidden rows: in the fp64 top-k, and rounded DOWN
    kth = -np.sort(-ex, axis=1)[:, case.k - 1]
    assert np.all(ex[r, case.hidden] >= kth[:, None])
    assert np.all(ap[r, case.hidden] < ex[r, case.hidden])
    # every hidden row is below >= k decoys in 16-bit score, and above all of them in true score
    below = (ap[r, case.decoys][:, None, :] > ap[r, case.hidden][:, :, None]).sum(axis=2)
    assert below.min() >= case.k
    assert np.all(ex[r, case.hidden].min(axis=1) > ex[r, case.decoys].max(axis=1))
    # ... by less than the filter's margin: the tensor path keeps them only if its 2 eps are really 2 eps
    gap = ap[r, case.decoys].max(axis=1) - ap[r, case.hidden].min(axis=1)
    assert np.all(gap <= 2 * eps) and np.all(gap >= 1.8 * floor * eps)
    # background and other queries' rows: far below
    others = np.ones_like(ex, dtype=bool)
    others[r, case.hidden] = False
    others[r, case.decoys] = False
    assert np.all(ex[others].reshape(nq, -1).max(axis=1) < ex[r, case.decoys].min(axis=1) - 4 * eps)
    # the norms and rounding errors that set eps come from the adversarial rows
    rows = case.xb.astype(np.float64)
    n2 = (rows ** 2).sum(1)
    assert n2[others.any(axis=0) & ~np.isin(np.arange(len(rows)), np.r_[case.hidden.ravel(), case.decoys.ravel()])].max() \
        <= n2[np.r_[case.hidden.ravel(), case.decoys.ravel()]].max()
    return adv_err.min()


@pytest.mark.parametrize("metric", [IP, L2])
@pytest.mark.parametrize("fmt,mbits,d", sorted(FLOORS))
def test_dy_aligned_rows_reach_the_bound(fmt, mbits, d, metric):
    case = adv.dy_aligned(24, d, 10, fmt=fmt, mbits=mbits, metric=metric, n_total=4096, seed=d + mbits + metric)
    _check_case(case, FLOORS[(fmt, mbits, d)])
    # the 16-bit rows are what the rounding makes of them: dy is parallel to the query, dx = 0
    assert np.array_equal(adv.round16(case.xq, fmt, mbits), case.xq)


@pytest.mark.parametrize("metric", [IP, L2])
def test_dx_aligned_queries_reach_the_bound(metric):
    case = adv.dx_aligned(24, 1024, 10, metric=metric, n_total=4096, seed=5 + metric)
    assert np.array_equal(adv.round16(case.xb, "bf16"), case.xb)  # bf16 storage: the rows are exact, dy = 0
    _check_case(case, 0.8)


@pytest.mark.parametrize("layout", ["front", "back", "bg_first", "shuffled"])
def test_layouts_place_the_rows(layout):
    case = adv.dy_aligned(16, 64, 10, layout=layout, n_total=8192, seed=3)
    h, dcy = case.hidden.ravel(), case.decoys.ravel()
    assert case.xb.shape[0] >= 8192 and len(np.unique(np.r_[h, dcy])) == h.size + dcy.size
    if layout == "front":
        assert h.max() < 1024 and dcy.min() > 4096  # dense first panel; decoys in a later panel
    if layout == "back":
        assert h.min() >= 4 * 1024 and dcy.max() < h.min()
    if layout == "bg_first":
        assert min(h.min(), dcy.min()) >= case.xb.shape[0] - h.size - dcy.size
    _check_case(case, 0.9)


def test_hidden_rows_are_in_the_fp32_oracle_top_k():
    """The margin between hidden rows and decoys is far above fp32 evaluation noise: the fp32 oracle (another
    summation order than the CUDA kernels) ranks them first, too."""
    for metric in (IP, L2):
        case = adv.dy_aligned(16, 1024, 10, metric=metric, n_total=4096, seed=11)
        _, I = fo.knn_flat(case.xq, case.xb, case.k, metric)
        for q in range(case.xq.shape[0]):
            assert set(case.hidden[q]) <= set(I[q])


def test_round_mantissa_matches_the_kernel_rule():
    """round_mantissa (kernels_basic.cu): to nearest, ties to even, on the explicit mantissa bits; NaN/Inf pass."""
    x = np.array([1.0, 1 + 2 ** -6, 1 + 3 * 2 ** -6, 1 + 2 ** -6 + 2 ** -20, -1.5 - 2 ** -6, np.inf, -np.inf],
                 np.float32)
    got = adv.round_mantissa(x, 5)
    want = np.array([1.0, 1.0, 1 + 4 * 2 ** -6, 1 + 2 ** -5, -1.5, np.inf, -np.inf], np.float32)
    assert np.array_equal(got, want)
    assert np.isnan(adv.round_mantissa(np.array([np.nan], np.float32), 5)[0])
    # 7 bits + bf16 rounding = bf16 rounding; the generic rule agrees with torch's bf16 conversion
    torch = pytest.importorskip("torch")
    v = np.random.default_rng(0).standard_normal(4096).astype(np.float32) * 3
    ref = torch.from_numpy(v).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(adv.round16(v, "bf16", 7), ref)
    assert np.array_equal(adv.round_mantissa(v, 7), ref)
    ref16 = torch.from_numpy(v).to(torch.float16).to(torch.float32).numpy()
    assert np.array_equal(adv.round16(v, "fp16"), ref16)


def test_l2_extreme_ratio_is_dominated_by_fp32_rounding():
    """16-bit-exact rows ~4000 x longer than the queries: the inner-product part of eps is only the fp32 slack,
    smaller than half an ulp of |y|^2 - the roundings the L2 term of eps exists for."""
    case = adv.l2_extreme_ratio(8, 64, 10, seed=1)
    assert np.array_equal(adv.round16(case.xb, "bf16"), case.xb) and np.array_equal(adv.round16(case.xb, "fp16"), case.xb)
    assert np.array_equal(adv.round16(case.xq, "fp16"), case.xq)
    xn = np.sqrt((case.xq.astype(np.float64) ** 2).sum(1))
    yn2 = (case.xb.astype(np.float64) ** 2).sum(1)
    assert 1e3 <= np.sqrt(yn2.max()) / xn.max() <= 1e4
    slack_only = 2 * 1.001 * 64 * 2.0 ** -22 * xn * np.sqrt(yn2.max())
    half_ulp = np.spacing(np.float32(yn2.max())) / 2
    assert np.all(slack_only < half_ulp)
    assert np.all(case.eps() > 8 * half_ulp)  # the rounding term covers them
    # |y|^2 is exact in fp32, the keys 2<x,y> - |y|^2 are not: their rounding is what eps must cover here
    assert np.array_equal(yn2.astype(np.float32).astype(np.float64), yn2)
    key = case.exact()
    off = np.abs(key.astype(np.float32).astype(np.float64) - key)
    assert off.max() > 2 * slack_only.max()
