"""Pooled adaptation checked exactly: every accumulation kernel of S = Y^T Y
(kPoolAccumulate, kPoolAccumulateDmma<true/false>, kPoolGramDmma<true/false>)
and both factor kernels (kPoolFactorCta, kPoolFactor) against the host
restatements of pooled_exact_support.py.

Frozen grid: with PROP_SIGMA = 0 the pooled proposal is x + (0 z) U = x, and the
acceptance-driven update and the trace rescale only multiply sigma, so the chains
stay on their grid start points.  Then S is exact in any summation order and
count, mean, covariance, U and the pooled trace must equal the host bit for bit.
Moving chains are checked against an error-free S within a rigorous bound.

The environment switches choose the kernel (engine.cu poolAccumulateOn,
poolExchange) and are read when a step runs: they are set before the Engine is
created and stay for the whole test."""
import fractions

import numpy as np
import pytest

import pooled_exact_support as pes

pytestmark = pytest.mark.gpu

SWITCHES = ("SMCMC_POOL_ACC_SCALAR", "SMCMC_POOL_ACC_DIRECT", "SMCMC_POOL_GRAM_MIN", "SMCMC_POOL_FACTOR_WARP")
STEPS = 3                     # exchange at step 3, then one more step for the chains to adopt the pooled trace
BIG = 8209                    # > 4096: several liveness slices of kPoolGramDmma; 8209 = 1 mod 16
BIG_LIMIT = 3e8               # E n^2: the per-chain decomposition is still allocated in pooled mode

# (switch, dimensions): the kernel each row runs is checked by test_kernel_selection
SELECTION = [
    (None, [1, 2, 7, 55, 56, 57, 63, 64, 65, 127, 128, 129, 191, 500, 600]),
    ("SMCMC_POOL_ACC_DIRECT", [111, 130, 167]),         # n + 1 = 112, 168: multiples of 56, or just past one
    ("SMCMC_POOL_GRAM_MIN", [1, 8, 63]),
    ("SMCMC_POOL_ACC_SCALAR", [55, 130, 600]),          # n = 55: 1596 statistics, two passes of 1536
    ("SMCMC_POOL_FACTOR_WARP", [57, 129]),
]


def smallest_ensemble(n):
    """n + 1 affinely independent points make the covariance positive definite;
    odd, so that E is not a multiple of 4 or 16 chains."""
    return n + 1 if (n + 1) % 2 else n + 2


def ensembles(n):
    return [smallest_ensemble(n)] + ([BIG] if BIG * n * n <= BIG_LIMIT else [])


FROZEN_CASES = [pytest.param(sw, n, E, id="%s-n%d-E%d" % ((sw or "default").replace("SMCMC_POOL_", ""), n, E))
                for sw, ns in SELECTION for n in ns for E in ensembles(n)]


def select(monkeypatch, switch):
    for s in SWITCHES:
        monkeypatch.delenv(s, raising=False)
    if switch:
        monkeypatch.setenv(switch, "1")


def frozen_run(n, x0, steps=STEPS):
    """Grid chains held still by sigma = 0: the device's pooled results after an
    exchange at `steps`, plus U and sigma_trace from before the first step."""
    import smcmc_b200
    from smcmc_b200 import binding
    E = x0.shape[0]
    eng = smcmc_b200.Engine(smcmc_b200.LLH_UNIT_GAUSS, n, E, seed=7)
    eng.prop_set(binding.PROP_POOLED_EVERY, steps)
    live = eng.start(x0).astype(bool)
    eng.prop_set(binding.PROP_SIGMA, 0.0)
    out = {"live": live, "u0": eng.get("pooled_decomposition"), "trace0": eng.get("sigma_trace")}
    out["points"] = eng.step_trace(steps, want=("points",))["points"]
    eng.step(1)
    for k in ("pooled_count", "pooled_mean", "pooled_covariance", "pooled_decomposition", "sigma_trace"):
        out[k] = eng.get(k)
    eng.close()
    return out


def check_frozen(dev, x0, m, n, steps=STEPS):
    live = dev["live"]
    # the premise: the started chains did not move
    assert np.array_equal(dev["points"][:, live], np.broadcast_to(x0[live], dev["points"][:, live].shape))
    host = pes.restate_factor(pes.grid_stats(m[live], steps), n)
    assert host["ok"], "the grid ensemble must have a positive definite covariance"
    assert dev["pooled_count"][0] == steps * live.sum()
    assert np.array_equal(dev["pooled_mean"], host["mean"])
    assert np.array_equal(dev["pooled_covariance"], host["cov"])
    assert np.array_equal(dev["pooled_decomposition"], host["u"])
    assert np.all(dev["sigma_trace"][live] == host["trace"])


@pytest.mark.parametrize("switch,n,E", FROZEN_CASES)
def test_frozen_grid_bit_for_bit(monkeypatch, switch, n, E):
    select(monkeypatch, switch)
    x0, m = pes.grid_points(E, n, seed=1000 + n)
    dev = frozen_run(n, x0)
    assert dev["live"].all()
    check_frozen(dev, x0, m, n)


def gram_slice_chains(E, n, sms):
    """Chains per CTA slice of kPoolGramDmma (engine.cu poolAccumulateOn)."""
    cdiv = lambda a, b: -(-a // b)
    nb = cdiv(n + 1, 64)
    pairs = nb * (nb + 1) // 2
    slices = max(1, min(cdiv(E, 64), (3 * sms) // pairs))
    slices = max(slices, cdiv(E, 4096))
    return cdiv(cdiv(E, slices), 16) * 16


@pytest.mark.parametrize("switch,n", [(None, 7), (None, 57), (None, 64), (None, 65), ("SMCMC_POOL_ACC_SCALAR", 55),
                                      ("SMCMC_POOL_ACC_DIRECT", 130), ("SMCMC_POOL_GRAM_MIN", 8)])
def test_chains_that_are_not_running_are_left_out(monkeypatch, switch, n):
    """NaN start rows do not start; any leak of their values into S shows as NaN.
    They sit at chain 0, the last chain, a whole group of 4 (one DMMA k step), a
    whole 16-chain slice, and the first and last chain of a Gram liveness slice."""
    import torch
    select(monkeypatch, switch)
    E = BIG
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    per = gram_slice_chains(E, n, sms)
    assert per < E // 3
    dead = sorted({0, E - 1, *range(20, 24), *range(48, 64), 2 * per, 3 * per - 1})
    x0, m = pes.grid_points(E, n, seed=2000 + n)
    x0 = x0.copy()
    x0[dead] = np.nan
    dev = frozen_run(n, x0)
    assert not dev["live"][dead].any() and dev["live"].sum() == E - len(dead)
    check_frozen(dev, x0, m, n)


@pytest.mark.parametrize("switch,n,E", [(None, 7, 65), (None, 57, 101), (None, 65, 101),
                                        ("SMCMC_POOL_FACTOR_WARP", 57, 101), ("SMCMC_POOL_GRAM_MIN", 8, 33),
                                        (None, 57, 9), (None, 65, 9), ("SMCMC_POOL_FACTOR_WARP", 57, 9)])
def test_covariance_that_is_not_positive_definite_keeps_the_previous_factor(monkeypatch, switch, n, E):
    """A coordinate with the same value in every chain has variance exactly 0; with
    E = 9 the count (27) is <= n + 1.  Either way U and the trace stay as they were."""
    select(monkeypatch, switch)
    x0, m = pes.grid_points(E, n, seed=3000 + n)
    m[:, n // 2] = 3
    x0[:, n // 2] = 3 * pes.GRID_STEP
    dev = frozen_run(n, x0)
    assert dev["live"].all()
    assert np.array_equal(dev["points"], np.broadcast_to(x0, dev["points"].shape))
    host = pes.restate_factor(pes.grid_stats(m, STEPS), n)
    assert not host["ok"]
    assert dev["pooled_count"][0] == STEPS * E
    assert np.array_equal(dev["pooled_decomposition"], dev["u0"])
    assert np.array_equal(dev["sigma_trace"], dev["trace0"])
    if host["mean"] is not None:              # mean and covariance are written before the factorisation
        assert host["cov"][pes.tri(n // 2) + n // 2] == 0.0
        assert np.array_equal(dev["pooled_mean"], host["mean"])
        assert np.array_equal(dev["pooled_covariance"], host["cov"])


@pytest.mark.parametrize("switch", ["SMCMC_POOL_ACC_SCALAR", "SMCMC_POOL_ACC_DIRECT", "SMCMC_POOL_GRAM_MIN"])
@pytest.mark.parametrize("n,E,steps", pes.MOVING_SHAPES)
def test_moving_chains_within_the_bound(monkeypatch, switch, n, E, steps):
    """Chains that move: mean and covariance against the error-free statistics of
    the traced points within the bound of pooled_exact_support (which
    test_pooled_exact.py shows rejects a dropped chain and FP32 inputs at these
    shapes); U bit for bit against the restated factorisation of the device's own
    covariance."""
    import smcmc_b200
    from smcmc_b200 import binding
    select(monkeypatch, switch)
    eng = smcmc_b200.Engine(smcmc_b200.LLH_UNIT_GAUSS, n, E, seed=40 + n)
    eng.prop_set(binding.PROP_POOLED_EVERY, steps)
    x0 = np.random.default_rng(n).normal(0, 1, (E, n))
    assert eng.start(x0).all()
    tr = eng.step_trace(steps, want=("accepted", "points"))
    assert tr["accepted"].mean() > 0.05
    count, mean, cov, u = (eng.get(k) for k in ("pooled_count", "pooled_mean", "pooled_covariance",
                                                  "pooled_decomposition"))
    eng.close()
    N = E * steps
    assert count[0] == N
    hi, lo, mag = pes.dd_stats(tr["points"].reshape(-1, n))
    rm, rc = pes.pooled_ratios(mean, cov, hi, lo, mag, N, n)
    assert rm <= 1.0 and rc <= 1.0, (rm, rc)
    ok, uh = pes.restate_cholesky(cov, n)
    assert ok and np.array_equal(u, uh)


# (switch, n, kernels that must run, kernels that must not)
PROFILED = [
    (None, 50, ["kPoolAccumulateDmma<true>", "kPoolFactorCta"], ["kPoolAccumulateDmma<false>", "kPoolGramDmma"]),
    (None, 57, ["kPoolAccumulateDmma<true>", "kPoolAccumulateDmma<false>"], ["kPoolGramDmma"]),
    (None, 64, ["kPoolGramDmma<true>"], ["kPoolAccumulateDmma", "kPoolGramDmma<false>"]),
    (None, 65, ["kPoolGramDmma<false>"], ["kPoolAccumulateDmma", "kPoolGramDmma<true>"]),
    (None, 600, ["kPoolGramDmma<true>", "kPoolFactorCta"], ["kPoolAccumulateDmma"]),
    ("SMCMC_POOL_ACC_DIRECT", 130, ["kPoolAccumulateDmma<true>", "kPoolAccumulateDmma<false>"], ["kPoolGramDmma"]),
    ("SMCMC_POOL_GRAM_MIN", 8, ["kPoolGramDmma<true>"], ["kPoolAccumulateDmma"]),
    ("SMCMC_POOL_GRAM_MIN", 63, ["kPoolGramDmma<false>"], ["kPoolAccumulateDmma"]),
    ("SMCMC_POOL_ACC_SCALAR", 55, ["kPoolAccumulate("], ["kPoolAccumulateDmma", "kPoolGramDmma"]),
    ("SMCMC_POOL_FACTOR_WARP", 57, ["kPoolFactor("], ["kPoolFactorCta"]),
]


@pytest.mark.parametrize("switch,n,want,unwanted", PROFILED)
def test_kernel_selection(monkeypatch, switch, n, want, unwanted):
    """One profiled step with an exchange: the intended kernels launch, so a change
    of the dispatch cannot quietly move the cases above to another kernel."""
    import smcmc_b200
    import torch
    from smcmc_b200 import binding
    from torch.profiler import ProfilerActivity, profile
    select(monkeypatch, switch)
    E = 257
    eng = smcmc_b200.Engine(smcmc_b200.LLH_UNIT_GAUSS, n, E, seed=3)
    eng.prop_set(binding.PROP_POOLED_EVERY, 1)
    assert eng.start(np.random.default_rng(1).normal(0, 1, (E, n))).all()
    eng.step(1)
    eng.sync()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.step(1)
        eng.sync()
        torch.cuda.synchronize()
    eng.close()
    names = [e.key for e in prof.key_averages()]
    for k in want:
        assert any(k in s for s in names), (k, names)
    for k in unwanted:
        assert not any(k in s for s in names), (k, names)


@pytest.mark.parametrize("switch,n,E", [(None, 7, 9), (None, 65, 67), ("SMCMC_POOL_ACC_SCALAR", 7, 9)])
def test_diagnostics_on_the_frozen_grid(monkeypatch, switch, n, E):
    """diag mean is S1 / count bit for bit; diag covariance is S / count - m_i m_j,
    rounded separately or fused (a host compiler may contract it)."""
    import smcmc_b200
    from smcmc_b200 import binding
    select(monkeypatch, switch)
    steps = 5
    x0, m = pes.grid_points(E, n, seed=4000 + n)
    eng = smcmc_b200.Engine(smcmc_b200.LLH_UNIT_GAUSS, n, E, seed=7)
    eng.prop_set(binding.PROP_POOLED_EVERY, 100)
    assert eng.start(x0).all()
    eng.prop_set(binding.PROP_SIGMA, 0.0)
    eng.diag_enable(0)
    tr = eng.step_trace(steps, want=("points",))
    d = eng.diag_get()
    eng.close()
    assert np.array_equal(tr["points"], np.broadcast_to(x0, tr["points"].shape))
    S = pes.grid_stats(m, steps)
    count = S[0]
    assert d["samples"] == count
    mean = S[1:1 + n] / count
    assert np.array_equal(d["mean"], mean)
    F = fractions.Fraction
    for i in range(n):
        for j in range(n):
            q = S[1 + n + pes.tri(max(i, j)) + min(i, j)] / count
            separate = q - mean[i] * mean[j]
            fused = float(F(q) - F(mean[i]) * F(mean[j]))
            assert d["covariance"][i, j] in (separate, fused), (i, j)


def test_rhat_counts_a_running_chain_that_sits_at_zero():
    """Chains held at the origin by sigma = 0 are running chains: R-hat counts them
    like every other chain (they are what R-hat is meant to expose).  Pooled mode,
    so that a frozen chain is not stopped by a zero per-chain covariance trace."""
    import smcmc_b200
    from smcmc_b200 import binding
    from test_gpu_diagnostics import reference_diagnostics
    n, E, steps = 4, 64, 200
    frozen = [0, 5, 17, 63]
    eng = smcmc_b200.Engine(smcmc_b200.LLH_UNIT_GAUSS, n, E, seed=31)
    assert eng.start(np.random.default_rng(6).normal(0, 1, (E, n))).all()
    llh0 = eng.eval(np.zeros(n))[0]
    saved = eng.save_state()
    saved["accepted"][frozen] = 0.0
    saved["sigma"][frozen] = 0.0
    saved["log_likelihood"][frozen] = llh0
    eng.restore_state(saved)
    eng.prop_set(binding.PROP_POOLED_EVERY, 10)
    eng.diag_enable(0)
    tr = eng.step_trace(steps, want=("points",))
    d = eng.diag_get()
    status = eng.get("status")
    eng.close()
    assert np.all(status == 0)
    moving = np.setdiff1d(np.arange(E), frozen)
    assert np.all(tr["points"][:, frozen] == 0.0)
    assert np.all(tr["points"][:, moving].std(0) > 0)
    _, _, _, rhat, _ = reference_diagnostics(tr["points"], [])
    assert np.allclose(d["rhat"], rhat, rtol=1e-9), (d["rhat"], rhat)
