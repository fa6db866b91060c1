"""Host restatements of pooled adaptation (csrc/pooled.cuh), for exact tests of
the accumulation kernels and the shared factor.

Statistics are packed as the engine packs them: S = (count, sum x_i,
sum x_i x_j for j <= i at i(i+1)/2 + j), the lower triangle of Y^T Y with
y = (1, x) per accumulated point.

Grid inputs.  A point x = m 2^-6 with integer |m| <= 2^7 makes every product
y_a y_b a multiple of 2^-12 of at most 2^14 ulps of that grid, and fewer than
2^20 such terms sum to less than 2^34 grid steps: every partial sum is a double,
whatever the order.  So atomics, DMMA accumulation order and slicing cannot
change a bit of S, and the device must reproduce `grid_stats` exactly.

Everything after S is IEEE arithmetic in a fixed order (the library is built
with -fmad=false), restated here one operation at a time:
  mean_i = S1_i / count;  cov_ij = S2_ij / count - mean_i mean_j;
  trace = cov_00 + cov_11 + ... summed in order;
  U = the column-ordered Cholesky of kPoolFactorCta / warpCholesky.

Moving chains.  For arbitrary points S is not exact.  Each statistic is a sum of
N products, and for ANY order of the N multiplications (fused or not) and N - 1
additions,
    |S^ - S| <= gamma_N A,   A = sum |y_a y_b|,   gamma_N = N u / (1 - N u),  u = 2^-53
(Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., sec. 3.1).
Call that bound e_S.  The count is a sum of ones, exact.  Then, with every
operation rounding once (|delta| <= u):

  mean   m^_i = (S^1_i / c)(1 + d):
         |m^_i - m_i| <= e_S1_i / c + u (|S1_i| + e_S1_i) / c                 =: M_i
  cov    q^ = (S^2_ij / c)(1 + d1):  |q^ - S2_ij / c| <= e_S2_ij / c + u (|S2_ij| + e_S2_ij) / c  =: Q
         p^ = m^_i m^_j (1 + d2):    |p^ - m_i m_j| <= M_i (|m_j| + M_j) + |m_i| M_j
                                                       + u (|m_i| + M_i)(|m_j| + M_j)          =: P
         c^ = (q^ - p^)(1 + d3):     |c^ - cov_ij| <= Q + P + u (|cov_ij| + Q + P)

The reference S of `dd_stats` is a double-double sum whose own error is far
below this (a few N^2 u^2 A); `mean_cov_bounds` adds 8 N^2 u^2 A to e_S to cover
it, and the comparison itself is done in exact rational arithmetic.
"""
import fractions

import numpy as np

GRID_STEP = 2.0 ** -6
GRID_MAX = 2 ** 7
U_ROUND = 2.0 ** -53


def tri(n):
    return n * (n + 1) // 2


# --------------------------------------------------------------------------- grid inputs

def grid_points(rows, n, seed):
    """`rows` points of the grid, as (x, m) with x = m 2^-6; distinct where the
    grid has room for them (4 rows per grid point or fewer)."""
    rng = np.random.default_rng(seed)
    side = 2 * GRID_MAX + 1
    distinct = 4 * rows <= side ** n
    if distinct and side ** n <= 2 ** 40:          # few grid points: draw them without replacement
        idx = rng.choice(side ** n, rows, replace=False)
        m = np.stack([(idx // side ** d) % side for d in range(n)], axis=1).astype(np.int64) - GRID_MAX
        return m * GRID_STEP, m
    while True:
        m = rng.integers(-GRID_MAX, GRID_MAX + 1, (rows, n), dtype=np.int64)
        if not distinct or len(np.unique(m, axis=0)) == rows:
            return m * GRID_STEP, m


def grid_stats(m, repeats=1):
    """Exact S of the grid points m 2^-6, each accumulated `repeats` times, from
    integer sums of the m values."""
    m = np.asarray(m, dtype=np.int64)
    rows, n = m.shape
    assert np.abs(m).max(initial=0) <= GRID_MAX and rows * repeats < 2 ** 20
    ii, jj = np.tril_indices(n)
    s1 = m.sum(0) * repeats
    # integer products of at most 2^14, fewer than 2^20 of them: every partial sum of the
    # floating-point product is an integer below 2^34, so BLAS computes it exactly
    mf = m.astype(np.float64)
    s2 = (mf.T @ mf)[ii, jj].astype(np.int64) * repeats
    out = np.empty(1 + n + tri(n))
    out[0] = rows * repeats
    out[1:1 + n] = s1 * GRID_STEP                 # exact: integers < 2^53 scaled by a power of two
    out[1 + n:] = s2 * (GRID_STEP * GRID_STEP)
    return out


# --------------------------------------------------------------------------- restatements

def restate_mean_cov(stats, n):
    count = stats[0]
    mean = stats[1:1 + n] / count
    ii, jj = np.tril_indices(n)
    cov = stats[1 + n:] / count - mean[ii] * mean[jj]     # two roundings and a subtraction, no FMA
    return mean, cov


def restate_trace(cov, n):
    t = 0.0
    for i in range(n):
        t += float(cov[tri(i) + i])
    return t


def restate_cholesky(cov, n):
    """(True, U) with U upper triangular, zeros below, or (False, None) at the
    first pivot v <= 0 -- kPoolFactorCta and warpCholesky.  Entry (c, j), j >= c:
    v = A(j, c); v -= U(r, j) U(r, c) for r = 0 .. c-1 ascending; U(c, c) = sqrt(v),
    U(c, j) = v / U(c, c).  Restated right-looking: after row r is final, every
    later (c, j) subtracts its r-th product, so each entry sees the same
    subtractions in the same order."""
    ii, jj = np.tril_indices(n)
    w = np.zeros((n, n))
    w[jj, ii] = cov                               # w[c, j] = A(j, c) for j >= c
    u = np.zeros((n, n))
    for r in range(n):
        v = w[r, r:]
        if v[0] <= 0.0:
            return False, None
        piv = np.sqrt(v[0])
        u[r, r] = piv
        u[r, r + 1:] = v[1:] / piv
        row = u[r, r + 1:]
        w[r + 1:, r + 1:] -= row[:, None] * row[None, :]
    return True, u


def restate_factor(stats, n):
    """What an exchange computes from S: dict(mean, cov, ok, u, trace); mean and
    cov are None when count <= n + 1 (the kernel returns before writing them)."""
    count = stats[0]
    if not count > n + 1:
        return {"mean": None, "cov": None, "ok": False, "u": None, "trace": None}
    mean, cov = restate_mean_cov(stats, n)
    ok, u = restate_cholesky(cov, n)
    return {"mean": mean, "cov": cov, "ok": ok, "u": u, "trace": restate_trace(cov, n) if ok else None}


# --------------------------------------------------------------------------- arbitrary points

def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(a):
    c = 134217729.0 * a                           # 2^27 + 1: Veltkamp
    hi = c - (c - a)
    return hi, a - hi


def _two_prod(a, b):
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def dd_stats(points):
    """S of the rows of `points` as double-double (hi, lo): every product split
    exactly (TwoProduct), every sum carried (TwoSum); vectorised over the
    statistics, one accumulated point after another.  Also A = sum |y_a y_b|."""
    pts = np.asarray(points, dtype=np.float64)
    n = pts.shape[1]
    ii, jj = np.tril_indices(n)
    nstat = 1 + n + tri(n)
    hi = np.zeros(nstat)
    lo = np.zeros(nstat)
    mag = np.zeros(nstat)
    for x in pts:
        a = np.concatenate(([1.0], x, x[ii]))
        b = np.concatenate(([1.0], np.ones(n), x[jj]))
        p, e = _two_prod(a, b)
        hi, err = _two_sum(hi, p)
        lo += err + e
        mag += np.abs(p)
    hi, lo = _two_sum(hi, lo)
    return hi, lo, mag


def gamma(N):
    return N * U_ROUND / (1.0 - N * U_ROUND)


def stats_bound(mag, N):
    """|S^ - S| <= gamma_N A for any summation order of N products per statistic."""
    return gamma(N) * mag


def mean_cov_bounds(ref_hi, mag, N, n):
    """Bounds on |mean^ - mean| and |cov^ - cov| (packed) for a device that summed
    N products per statistic, derived in the module docstring.  The reference's
    own error (8 N^2 u^2 A) is added to e_S, and 1e-6 relative to the result
    covers the rounding of the bound's own evaluation."""
    u = U_ROUND
    eS = stats_bound(mag, N) + 8.0 * (N * u) ** 2 * mag
    count = ref_hi[0]
    s1, e1 = np.abs(ref_hi[1:1 + n]), eS[1:1 + n]
    s2, e2 = np.abs(ref_hi[1 + n:]), eS[1 + n:]
    m = s1 / count
    M = e1 / count + u * (s1 + e1) / count
    ii, jj = np.tril_indices(n)
    Q = e2 / count + u * (s2 + e2) / count
    P = M[ii] * (m[jj] + M[jj]) + m[ii] * M[jj] + u * (m[ii] + M[ii]) * (m[jj] + M[jj])
    cabs = np.abs(s2 / count) + m[ii] * m[jj]                 # >= |cov_ij|
    C = Q + P + u * (cabs + Q + P)
    return M * (1 + 1e-6), C * (1 + 1e-6)


def exact_mean_cov(ref_hi, ref_lo, n):
    """mean and packed cov of the double-double S as exact fractions."""
    F = fractions.Fraction
    count = F(ref_hi[0]) + F(ref_lo[0])
    mean = [(F(ref_hi[1 + i]) + F(ref_lo[1 + i])) / count for i in range(n)]
    cov = []
    for i in range(n):
        for j in range(i + 1):
            p = 1 + n + tri(i) + j
            cov.append((F(ref_hi[p]) + F(ref_lo[p])) / count - mean[i] * mean[j])
    return mean, cov


def worst_ratio(got, exact, bound):
    """max |got - exact| / bound, the difference taken exactly."""
    F = fractions.Fraction
    worst = 0.0
    for g, e, b in zip(np.asarray(got, dtype=np.float64).ravel(), exact, np.asarray(bound).ravel()):
        d = abs(F(float(g)) - e)
        if d == 0:
            continue
        worst = max(worst, float(d / F(float(b))) if b > 0 else float("inf"))
    return worst


def pooled_ratios(mean, cov, ref_hi, ref_lo, mag, N, n):
    """(mean ratio, cov ratio) of a device result against the exact reference,
    in units of the bound: both <= 1 for a correct accumulation of N terms."""
    M, C = mean_cov_bounds(ref_hi, mag, N, n)
    em, ec = exact_mean_cov(ref_hi, ref_lo, n)
    return worst_ratio(mean, em, M), worst_ratio(cov, ec, C)


def float_stats(points):
    """S summed in plain double arithmetic (BLAS order), as a device might."""
    pts = np.asarray(points, dtype=np.float64)
    n = pts.shape[1]
    ii, jj = np.tril_indices(n)
    out = np.empty(1 + n + tri(n))
    out[0] = pts.shape[0]
    out[1:1 + n] = pts.sum(0)
    out[1 + n:] = (pts.T @ pts)[ii, jj]
    return out


# --------------------------------------------------------------------------- shapes used on the GPU

# moving chains, checked against the bound: (n, chains, steps)
MOVING_SHAPES = [(50, 768, 12), (57, 768, 12), (129, 512, 10)]


def moving_like_points(n, chains, steps, seed):
    """Points of the same shape and scale as the traced points of a moving
    ensemble on the unit Gaussian: steps x chains rows."""
    rng = np.random.default_rng(seed)
    return rng.normal(0.0, 1.0, (steps * chains, n))
