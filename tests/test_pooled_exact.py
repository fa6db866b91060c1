"""The host restatements of pooled adaptation (pooled_exact_support.py) that the
GPU tests of test_gpu_pooled_exact.py compare with: the Cholesky restatement,
the double-double statistics, exactness of grid sums, and that the error bound
used on moving chains is tight enough to reject a dropped chain or FP32 inputs
at every shape it is used at."""
import fractions

import numpy as np
import pytest

import pooled_exact_support as pes


def packed(a):
    n = a.shape[0]
    return a[np.tril_indices(n)]


@pytest.mark.parametrize("n", [1, 2, 7, 57, 130])
def test_cholesky_restatement_matches_numpy(n):
    rng = np.random.default_rng(n)
    b = rng.normal(0, 1, (n, n))
    a = b @ b.T / n + 0.2 * np.eye(n)
    ok, u = pes.restate_cholesky(packed(a), n)
    assert ok
    assert np.array_equal(u, np.triu(u))
    want = np.linalg.cholesky(a).T
    assert np.max(np.abs(u - want)) <= 1e-13 * np.max(np.abs(want))


def test_cholesky_restatement_rejects_a_zero_variance():
    n = 6
    _, m = pes.grid_points(40, n, seed=4)
    m[:, 3] = 5                                   # the same value in every point
    mean, cov = pes.restate_mean_cov(pes.grid_stats(m, 3), n)
    assert cov[pes.tri(3) + 3] == 0.0
    ok, u = pes.restate_cholesky(cov, n)
    assert not ok and u is None
    assert pes.restate_factor(pes.grid_stats(m, 3), n)["ok"] is False
    # too few points: nothing is computed
    assert pes.restate_factor(pes.grid_stats(m[:3], 2), n)["mean"] is None


def test_double_double_statistics_are_exact_on_a_small_case():
    rng = np.random.default_rng(8)
    pts = rng.normal(0, 1, (37, 3)) * np.array([1.0, 1e6, 1e-5])
    hi, lo, mag = pes.dd_stats(pts)
    F = fractions.Fraction
    n = pts.shape[1]
    exact = [F(len(pts))] + [sum(F(x) for x in pts[:, i]) for i in range(n)]
    exact += [sum(F(a) * F(b) for a, b in zip(pts[:, i], pts[:, j])) for i in range(n) for j in range(i + 1)]
    for k, e in enumerate(exact):
        assert hi[k] == float(e)                                          # correctly rounded
        assert abs(F(hi[k]) + F(lo[k]) - e) <= F(2.0 ** -100) * F(mag[k])


@pytest.mark.parametrize("n,rows,repeats", [(7, 9, 3), (55, 57, 3), (129, 8209, 3)])
def test_grid_sums_are_exact_in_any_order(n, rows, repeats):
    x, m = pes.grid_points(rows, n, seed=n)
    exact = pes.grid_stats(m, repeats)
    pts = np.tile(x, (repeats, 1))
    rng = np.random.default_rng(1)
    ii, jj = np.tril_indices(n)
    for _ in range(3):
        p = pts[rng.permutation(len(pts))]
        s = np.zeros(1 + n + pes.tri(n))
        for lo in range(0, len(p), 1000):           # chunked partial sums, then added: another order
            blk = p[lo:lo + 1000]
            s[0] += len(blk)
            s[1:1 + n] += blk[::-1].sum(0)
            s[1 + n:] += (blk.T @ blk)[ii, jj]
        assert np.array_equal(s, exact)
        assert np.array_equal(pes.float_stats(p.astype(np.float32).astype(np.float64)), exact)


@pytest.mark.parametrize("n,chains,steps", pes.MOVING_SHAPES)
def test_the_bound_has_teeth(n, chains, steps):
    """At each shape the GPU test checks against the bound: a plain float sum
    passes, and the same sum without one chain, or of the points rounded to FP32,
    fails it."""
    pts = pes.moving_like_points(n, chains, steps, seed=n)
    N = chains * steps
    hi, lo, mag = pes.dd_stats(pts)
    mean, cov = pes.restate_mean_cov(pes.float_stats(pts), n)
    rm, rc = pes.pooled_ratios(mean, cov, hi, lo, mag, N, n)
    assert rm <= 1.0 and rc <= 1.0

    by_chain = pts.reshape(steps, chains, n)
    dropped = np.delete(by_chain, chains // 2, axis=1).reshape(-1, n)
    mean, cov = pes.restate_mean_cov(pes.float_stats(dropped), n)
    rm, rc = pes.pooled_ratios(mean, cov, hi, lo, mag, N, n)
    assert rm > 1.0 and rc > 1.0

    fp32 = pts.astype(np.float32).astype(np.float64)
    mean, cov = pes.restate_mean_cov(pes.float_stats(fp32), n)
    rm, rc = pes.pooled_ratios(mean, cov, hi, lo, mag, N, n)
    assert rm > 1.0 and rc > 1.0
