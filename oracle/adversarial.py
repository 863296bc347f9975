"""Data that drives the tensor path's error bound to its limit (CPU only, numpy).

The filter of the tensor path keeps every row whose 16-bit score is at least (k-th best approximate) - 2 eps, with
eps the per-query bound of query_eps_kernel (csrc/kernels_basic.cu, DESIGN.md section 4).  Random data cannot tell
whether eps is large enough: its rounding errors point in random directions, the realised score error is about
eps / sqrt(d), and a bound 10 x too small still passes.  The generators here make the rounding error point along the
other operand, so that the realised error reaches 0.9-0.99 of eps, and arrange every query's rows so that the result
is right only if the filter's margin really is 2 eps:

* hidden rows: rounding pushes their 16-bit score DOWN by ~eps; they belong to the exact top-k;
* >= k decoys: rounding pushes their 16-bit score UP by ~eps; their 16-bit scores lie above every hidden row's, their
  true scores below;
* background rows: exactly representable (no rounding error), scores far below, norms no larger than the adversarial
  rows' (so that max|y| and max|dy| come from the adversarial rows).

For L2 the same is done in key space, key = 2<x,y> - |y|^2 (what the filter compares), where the error doubles.

dy_aligned: queries in {+-1}^d (exact in every format, dx = 0); an adversarial row is g +- c x with g on the 16-bit
  grid and c just under half a grid step, so it rounds back to g and dy = -+c x is parallel to the query.
dx_aligned: for an index with bf16 storage (the bf16 rows ARE the database, dy = 0): the query's rounding error lies
  along the hidden rows and against the decoys.
l2_extreme_ratio: 16-bit-exact data with rows ~4000 x longer than the queries: eps is only the fp32 slack, and the
  fp32 rounding of |y|^2 and of the key 2<x,y> - |y|^2 (of order ulp(|y|^2)) is what a bound has to cover.

eps_reference restates query_eps_kernel in fp64 on quantities measured from the data as the kernels measure them.
"""
from dataclasses import dataclass, field

import numpy as np

METRIC_INNER_PRODUCT, METRIC_L2 = 0, 1
_F32_SLACK = 2.0 ** -22  # fp32-accumulation slack per padded dimension (query_eps_kernel)


# ---- the 16-bit roundings of the ingest kernel ----------------------------------------------------------------
def round_mantissa(v, mbits: int) -> np.ndarray:
    """numpy copy of round_mantissa (kernels_basic.cu): round to `mbits` explicit mantissa bits, ties to even;
    NaN / Inf pass through."""
    v = np.ascontiguousarray(v, dtype=np.float32)
    u = v.view(np.uint32).astype(np.uint64)
    drop = 23 - mbits
    special = (u & 0x7F800000) == 0x7F800000
    r = u + ((1 << (drop - 1)) - 1) + ((u >> drop) & 1)
    r &= ~np.uint64((1 << drop) - 1)
    r = (r & 0xFFFFFFFF).astype(np.uint32)
    out = r.view(np.float32).copy()
    out[special] = v[special]
    return out


def _bf16_rne(v: np.ndarray) -> np.ndarray:
    v = np.ascontiguousarray(v, dtype=np.float32)
    u = v.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).astype(np.uint32)
    out = r.view(np.float32).copy()
    special = (u & 0x7F800000) == 0x7F800000
    out[special] = v[special]
    return out


def round16(v, fmt: str, mbits: int = 7) -> np.ndarray:
    """The values the 16-bit shadow holds for fp32 values v (pack_shadow2 in kernels_basic.cu), as float32."""
    v = np.asarray(v, dtype=np.float32)
    if fmt == "fp16":
        a = np.abs(v)
        v = np.where((a > 65504.0) & (a <= np.finfo(np.float32).max), np.copysign(np.float32(65504.0), v), v)
        v = np.where(a < 6.103515625e-05, np.float32(0.0), v).astype(np.float32)
        return v.astype(np.float16).astype(np.float32)
    if fmt != "bf16":
        raise ValueError("fmt must be 'bf16' or 'fp16'")
    if mbits < 7:
        v = round_mantissa(v, mbits)
    return _bf16_rne(v)


def grid_step(fmt: str, mbits: int = 7) -> float:
    """Spacing of the 16-bit grid in [1, 2)."""
    return 2.0 ** -10 if fmt == "fp16" else 2.0 ** -mbits


# ---- scores -------------------------------------------------------------------------------------------------
def exact_scores(xq, xb, metric) -> np.ndarray:
    """fp64 scores the filter is about: <x,y> (IP) or the L2 key 2<x,y> - |y|^2 (larger = better)."""
    q = np.asarray(xq, np.float64)
    b = np.asarray(xb, np.float64)
    s = q @ b.T
    if metric == METRIC_L2:
        s = 2.0 * s - (b * b).sum(1)[None, :]
    return s


def approx_scores(xq, xb, fmt, mbits, metric, bf16_storage=False) -> np.ndarray:
    """fp64 value of what the tensor cores are asked for: 16-bit x 16-bit products (exact in fp64), minus the
    stored |y|^2 for L2.  bf16_storage: the rows are the database already (xb must be bf16-exact)."""
    qh = round16(xq, fmt, mbits).astype(np.float64)
    bh = round16(xb, fmt, mbits).astype(np.float64)
    s = qh @ bh.T
    if metric == METRIC_L2:
        b = bh if bf16_storage else np.asarray(xb, np.float64)
        s = 2.0 * s - (b * b).sum(1)[None, :]
    return s


def eps_reference(xq, xb, fmt, mbits, metric, bf16_storage=False) -> np.ndarray:
    """Per-query eps of query_eps_kernel in fp64:
    (|dx| max|y| + |x| max|dy| + |dx| max|dy| + d_pad 2^-22 |x| max|y|) * 1.001, doubled for L2.
    |x|, |dx| come from the query and its rounding, max|y|, max|dy| from the stored rows and theirs (with bf16
    storage the rounded rows are the rows: dy = 0)."""
    q = np.asarray(xq, np.float32)
    b = np.asarray(xb, np.float32)
    dp = -(-q.shape[1] // 64) * 64
    qh = round16(q, fmt, mbits).astype(np.float64)
    bh = round16(b, fmt, mbits).astype(np.float64)
    rows = bh if bf16_storage else b.astype(np.float64)
    xn = np.sqrt((q.astype(np.float64) ** 2).sum(1))
    dx = np.sqrt(((q - qh) ** 2).sum(1))
    ymax = np.sqrt((rows ** 2).sum(1).max())
    dymax = 0.0 if bf16_storage else np.sqrt(((bh - rows) ** 2).sum(1).max())
    e = (dx * ymax + xn * dymax + dx * dymax + dp * _F32_SLACK * xn * ymax) * 1.001
    if metric == METRIC_L2:
        e = e * 2.0 + l2_rounding_term(dp, xn ** 2, ymax ** 2)
    return e


def l2_rounding_term(dp, xnorm2, ymax2):
    """The L2 part of eps that covers fp32 roundings of order ulp(|y|^2) (see query_eps_kernel)."""
    return (dp / 32.0 + 16.0) * 2.0 ** -24 * (xnorm2 + ymax2)


# ---- cases --------------------------------------------------------------------------------------------------
@dataclass
class Case:
    xq: np.ndarray            # (nq, d) float32
    xb: np.ndarray            # (N, d) float32
    k: int
    metric: int
    fmt: str
    mbits: int
    bf16_storage: bool = False
    hidden: np.ndarray = field(default_factory=lambda: np.zeros((0, 0), np.int64))  # (nq, h) row ids
    decoys: np.ndarray = field(default_factory=lambda: np.zeros((0, 0), np.int64))  # (nq, n_decoys) row ids

    def eps(self):
        return eps_reference(self.xq, self.xb, self.fmt, self.mbits, self.metric, self.bf16_storage)

    def exact(self):
        return exact_scores(self.xq, self.xb, self.metric)

    def approx(self):
        return approx_scores(self.xq, self.xb, self.fmt, self.mbits, self.metric, self.bf16_storage)


def _fit(contrib, m, step, lo_m, hi_m, target_lo, target_hi, rng, max_iter=64):
    """Move coordinates of m by whole grid steps (each at most once per round) until contrib(m).sum() lies in
    [target_lo, target_hi].  contrib: per-coordinate contribution of a row to its score."""
    m = m.copy()
    for _ in range(max_iter):
        cur = contrib(m).sum()
        if target_lo <= cur <= target_hi:
            return m
        want = 0.5 * (target_lo + target_hi) - cur
        up = np.where(m + step <= hi_m, contrib(m + step) - contrib(m), 0.0)
        dn = np.where(m - step >= lo_m, contrib(m - step) - contrib(m), 0.0)
        eff = np.where(np.sign(up) == np.sign(want), up, 0.0)
        eff_dn = np.where(np.sign(dn) == np.sign(want), dn, 0.0)
        use_dn = np.abs(eff_dn) > np.abs(eff)
        eff = np.where(use_dn, eff_dn, eff)
        mv = np.where(use_dn, -step, step)
        order = rng.permutation(m.shape[0])
        order = order[eff[order] != 0]
        if order.size == 0:
            break
        cs = np.cumsum(np.abs(eff[order]))
        n = int(np.searchsorted(cs, abs(want), side="right"))
        if n == 0:  # one move overshoots: take the smallest one
            n = 1
            order = order[np.argsort(np.abs(eff[order]), kind="stable")]
        sel = order[:n]
        m[sel] += mv[sel]
    raise ValueError("could not place a row's score in [%r, %r]" % (target_lo, target_hi))


def _layout(rng, n_adv_hidden, n_adv_decoy, n_bg, layout):
    """Row positions of (hidden, decoy, background) blocks.
    front: hidden rows first (the dense first panel), decoys last; back: decoys first, hidden rows last (beyond the
    later panels' starts); bg_first: background, decoys, hidden rows; shuffled: anywhere."""
    n = n_adv_hidden + n_adv_decoy + n_bg
    if layout == "front":
        pos = np.concatenate([np.arange(n_adv_hidden), n - n_adv_decoy + np.arange(n_adv_decoy),
                              n_adv_hidden + np.arange(n_bg)])
    elif layout == "back":
        pos = np.concatenate([n - n_adv_hidden + np.arange(n_adv_hidden), np.arange(n_adv_decoy),
                              n_adv_decoy + np.arange(n_bg)])
    elif layout == "bg_first":  # background, then decoys, then hidden rows: a split add brings every adversarial row late
        pos = np.concatenate([n - n_adv_hidden + np.arange(n_adv_hidden), n_bg + np.arange(n_adv_decoy),
                              np.arange(n_bg)])
    elif layout == "shuffled":
        pos = rng.permutation(n)
    else:
        raise ValueError(layout)
    return pos[:n_adv_hidden], pos[n_adv_hidden:n_adv_hidden + n_adv_decoy], pos[n_adv_hidden + n_adv_decoy:]


def _margin(u, d, scale):
    # what separates a hidden row from a decoy in TRUE score: several grid steps, and well above the error of an
    # fp32 evaluation of the score (so that the exact path, too, ranks the hidden rows first)
    return max(4.0 * u, 2.0 ** -18 * np.sqrt(d) * scale)


def _assemble(rng, d, k, metric, fmt, mbits, hidden_rows, decoy_rows, background, layout, bf16_storage=False, xq=None):
    nq, h, _ = hidden_rows.shape
    nd = decoy_rows.shape[1]
    hid_pos, dec_pos, bg_pos = _layout(rng, nq * h, nq * nd, background.shape[0], layout)
    xb = np.empty((nq * h + nq * nd + background.shape[0], d), np.float32)
    xb[hid_pos] = hidden_rows.reshape(-1, d)
    xb[dec_pos] = decoy_rows.reshape(-1, d)
    xb[bg_pos] = background
    return Case(xq=xq, xb=xb, k=k, metric=metric, fmt=fmt, mbits=mbits, bf16_storage=bf16_storage,
                hidden=hid_pos.reshape(nq, h).astype(np.int64), decoys=dec_pos.reshape(nq, nd).astype(np.int64))


def dy_aligned(nq, d, k, *, fmt="bf16", mbits=7, metric=METRIC_INNER_PRODUCT, n_hidden=2, n_decoys=None,
               layout="back", n_total=8192, seed=0) -> Case:
    """Rows whose rounding error dy is parallel to their query (see the module docstring).

    Query q is x = a b, b in {+-1}^d, a = 1 (IP) or 1/2 (L2: keeps |x|^2 + |y|^2 - 2<x,y> clear of cancellation, so
    that fp32 evaluations of the distance agree to the parity rule's bound).  An adversarial row of q is
    y = b (1 + u p) + s c b with p >= 2 integer (1 + u p is on the grid, u = grid step in [1, 2)) and c = u/2 - 2^-22:
    y rounds to b (1 + u p) and its 16-bit score misses the true one by s a c d (IP) or 2 s a c d (L2 key), s = +1 for
    hidden rows, -1 for decoys.  Every score is a sum of per-coordinate terms, so a row is placed by moving single
    coordinates of p by one step.  Rows of a query that are permutations of each other tie exactly."""
    rng = np.random.default_rng(seed)
    if fmt == "fp16":
        mbits = 10
    u = grid_step(fmt, mbits)
    c = u / 2 - 2.0 ** -22
    nd = n_decoys if n_decoys is not None else k + 2
    l2 = metric == METRIC_L2
    kappa = 2.0 if l2 else 1.0
    a = 0.5 if l2 else 1.0
    e2 = 2.0 * kappa * a * c * d       # approx gap at which a decoy's true score meets a hidden row's
    margin = _margin(u, d, 1.3 * d)
    pmax = int(0.25 / u)               # magnitudes stay in [1 + 2u, 1.25]: far from the binade edges

    def contrib(s):
        if l2:
            return lambda p: 2.0 * a * (1.0 + u * p) - (1.0 + u * p + s * c) ** 2
        return lambda p: a * (1.0 + u * p)

    signs = rng.choice(np.array([-1.0, 1.0], np.float32), size=(nq, d))
    xq = (a * signs).astype(np.float32)
    hid = np.empty((nq, n_hidden, d), np.float32)
    dec = np.empty((nq, nd, d), np.float32)
    lo_m, hi_m = np.full(d, 2.0), np.full(d, float(pmax))
    for q in range(nq):
        x = signs[q].astype(np.float64)
        base = rng.integers(2, min(pmax // 2, 2 + 12), size=d).astype(np.float64)
        a_h = contrib(+1)(base).sum()
        for j in range(n_hidden):  # permutations: different rows, identical scores
            p = rng.permutation(base)
            hid[q, j] = (x * (1.0 + u * p + c)).astype(np.float32)
        for j in range(nd):
            hi = a_h + e2 - margin - (j % 4) * u
            p = _fit(contrib(-1), base, 1.0, lo_m, hi_m, hi - 2 * u, hi, rng)
            dec[q, j] = (x * (1.0 + u * rng.permutation(p) - c)).astype(np.float32)
    # background: exact grid values, random signs, magnitude 1 or 1 + u (never longer than an adversarial row)
    n_adv = nq * (n_hidden + nd)
    n_bg = max(n_total - n_adv, 1024)
    bg = (rng.choice(np.array([-1.0, 1.0]), size=(n_bg, d)) * (1.0 + u * rng.integers(0, 2, size=(n_bg, d))))
    return _assemble(rng, d, k, metric, fmt, mbits, hid, dec, bg.astype(np.float32), layout, xq=xq)


def dx_aligned(nq, d, k, *, metric=METRIC_INNER_PRODUCT, n_hidden=2, n_decoys=None, layout="back", n_total=8192,
               seed=0) -> Case:
    """For an index with bf16 storage (dy = 0): the QUERY's rounding error points along the hidden rows and against
    the decoys.

    Query x = b * (1.5 + c z), b in {+-1}^d, z = +1 on a random half S1 of the coordinates and -1 on the other half,
    c = u/2 - 2^-22: x rounds to 1.5 b, dx = -c b z.  A row y = b * m (bf16-exact) has 16-bit score 1.5 sum(m) and
    true score 1.5 sum(m) + c sum(z m).  Hidden rows: m ~ +1.25 on S1, ~ -0.75 on S2 (sum(z m) = |y|_1); decoys: the
    halves swapped (sum(z m) = -|y|_1).  Their 16-bit scores are then moved apart by single bf16 steps."""
    rng = np.random.default_rng(seed)
    fmt, mbits = "bf16", 7
    u = grid_step(fmt, mbits)
    c = u / 2 - 2.0 ** -22
    nd = n_decoys if n_decoys is not None else k + 2
    l2 = metric == METRIC_L2
    kappa = 2.0 if l2 else 1.0
    margin = _margin(u, d, 1.3 * d)
    half = d // 2

    def contrib_approx(m):
        return 2.0 * 1.5 * m - m * m if l2 else 1.5 * m

    def true_of(m, z):
        return (2.0 * (1.5 + c * z) * m - m * m).sum() if l2 else ((1.5 + c * z) * m).sum()

    xq = np.empty((nq, d), np.float32)
    hid = np.empty((nq, n_hidden, d), np.float32)
    dec = np.empty((nq, nd, d), np.float32)
    for q in range(nq):
        b = rng.choice(np.array([-1.0, 1.0]), size=d)
        z = np.ones(d)
        z[rng.permutation(d)[half:]] = -1.0
        xq[q] = (b * (1.5 + c * z)).astype(np.float32)
        s1, s2 = np.flatnonzero(z > 0), np.flatnonzero(z < 0)
        big = 1.0 + u * rng.integers(24, 40, size=half)           # [1.19, 1.31], grid step u
        small = 0.5 + (u / 2) * rng.integers(56, 72, size=d - half)  # [0.72, 0.78], grid step u/2
        m_h = np.empty(d)
        for j in range(n_hidden):
            m_h[s1] = rng.permutation(big)
            m_h[s2] = -rng.permutation(small)
            hid[q, j] = (b * m_h).astype(np.float32)
        a_h = contrib_approx(m_h).sum()
        err_h = true_of(m_h, z) - a_h
        for j in range(nd):
            m = np.empty(d)
            m[s1] = -rng.permutation(small)
            m[s2] = rng.permutation(big)
            # only the large (S2) magnitudes move: one bf16 step u there
            lo_m = np.where(z < 0, 1.0 + 4 * u, -1.0)
            hi_m = np.where(z < 0, 2.0 - 4 * u, -0.5)
            step = np.where(z < 0, u, 0.0)
            for _ in range(3):  # the decoy's own error changes a little with its magnitudes
                err_d = contrib_approx(m).sum() - true_of(m, z)
                hi = a_h + err_h + err_d - margin - (j % 4) * u
                m = _fit(contrib_approx, m, step, np.minimum(lo_m, m), np.maximum(hi_m, m), hi - 2 * u, hi, rng)
            dec[q, j] = (b * m).astype(np.float32)
    n_adv = nq * (n_hidden + nd)
    n_bg = max(n_total - n_adv, 1024)
    bg = rng.choice(np.array([-1.0, 1.0], np.float32), size=(n_bg, d))
    return _assemble(rng, d, k, metric, fmt, mbits, hid, dec, bg, layout, bf16_storage=True, xq=xq)


def l2_extreme_ratio(nq, d, k, *, rows_per_query=None, n_total=8192, seed=0) -> Case:
    """L2 with 16-bit-exact data (dx = dy = 0, eps = the fp32 slack only) and rows ~4000 x longer than the queries.

    Query entries are +-1/4 (|x| = d^0.5 / 4).  Query q owns rows whose first d - 4 coordinates are 1024 times its
    signs and whose last 4 are small even integers: |y|^2 < 2^26 is a multiple of 4 (exact in fp32), the keys
    2<x,y> - |y|^2 ~ -6e7 are integers, and fp32 holds them to multiples of 4 - the rounding of the key is several
    times eps, and the fp32 distances tie in bulk at the k-th position (in the same bits for every fp32 evaluation
    of |x|^2 + |y|^2 - 2<x,y>, whose terms are all exact)."""
    rng = np.random.default_rng(seed)
    rpq = rows_per_query if rows_per_query is not None else 4 * k
    nb = d - 4
    xq = (rng.choice(np.array([-0.25, 0.25]), size=(nq, d))).astype(np.float32)
    own = np.empty((nq, rpq, d), np.float32)
    for q in range(nq):
        sgn = np.sign(xq[q])
        own[q, :, :nb] = 1024.0 * sgn[:nb]
        own[q, :, nb:] = 2 * rng.integers(-8, 9, size=(rpq, 4))
    n_bg = max(n_total - nq * rpq, 1024)
    bg = np.empty((n_bg, d), np.float32)
    bg[:, :nb] = 1024.0 * rng.choice(np.array([-1.0, 1.0]), size=(n_bg, nb))
    bg[:, nb:] = 2 * rng.integers(-8, 9, size=(n_bg, 4))
    xb = np.concatenate([own.reshape(-1, d), bg])
    perm = rng.permutation(xb.shape[0])
    return Case(xq=xq, xb=xb[perm], k=k, metric=METRIC_L2, fmt="bf16", mbits=7)
