"""TSimpleHMC on finite-difference gradients (PotentialGradient, TSimpleHMC.H:417-444):
every likelihood without a gradient of its own -- the built-in event likelihoods, user
event functors, user functors without a gradient entry -- reaches HMC this way
(engine_hmc.inl: hmcGradient(kGradFinite); hmc.cuh: kHmcFdPoints, kHmcFdGradient).

  * An ensemble too large for one pass of finite-difference work points, against the
    port chain for chain, bit for bit, across the boundary between the passes.
  * The gradient kept from the previous step (DESIGN 4.5) is dropped when the event
    sample or the data histograms change: runs with and without the kept gradients are
    identical through such changes.
  * The built-in unbinned likelihood against its restatement as a user event functor
    (tests/cpp/user_events.cuh): two code paths, the same HMC chains.
"""
import time

import numpy as np
import pytest

import user_events_support as ues
from helpers import hmc_error_matrix
from test_gpu_hmc import check_against

pytestmark = pytest.mark.gpu

LEAPFROG = 4            # SetLeapFrog: a fixed trajectory of 4 leap-frog steps, 5 gradients per step


@pytest.fixture(scope="module")
def user_events_lib(tmp_path_factory):
    return ues.build_library(str(tmp_path_factory.mktemp("user_events")))


def set_cache(monkeypatch, on):
    if on:
        monkeypatch.delenv("SMCMC_HMC_NO_GRADIENT_CACHE", raising=False)
    else:
        monkeypatch.setenv("SMCMC_HMC_NO_GRADIENT_CACHE", "1")


# ------------------------------------------------------------------------ chunked passes
def test_chunked_finite_difference_passes_equal_the_port(monkeypatch, checkers):
    """n = 300, 400 chains, finite differences forced (type 3) on TDummyLogLikelihood in
    EXACT mode.  One pass of work points holds 372 chains, so the second pass (28 chains)
    reads its points and writes its gradients at chain offset 372.  Chains on both sides of
    the boundary, the first, the last and one in the middle of the first pass equal the
    port's chains bit for bit after every step, and so does their final state.  The
    per-chain E[xx^T] triangles take 144 MB, below the 256 MB at which the covariance would
    be pooled, so every chain keeps the reference's own estimate.  The same ensemble with
    every gradient computed afresh (no kept gradients) gives the same run."""
    import smcmc_b200
    from smcmc_b200 import binding as b
    cc = checkers
    n, E, steps, seed = 300, 400, 20, 41
    # kHmcFdWorkBytes (engine_hmc.inl): 512 MiB of work points per pass, 2 n points of n
    # coordinates per chain
    per_pass = (512 << 20) // (2 * n * n * 8)
    assert (per_pass, E - per_pass) == (372, 28)
    assert E * (n * (n + 1) // 2) * 8 < 256 << 20
    prec = hmc_error_matrix("spd%d" % n)
    x0 = np.random.default_rng(300).normal(0.0, 0.4, (E, n))
    runs = {}
    for cache in (True, False):
        set_cache(monkeypatch, cache)
        eng = smcmc_b200.Engine(smcmc_b200.LLH_DUMMY, n, E, seed=seed)
        eng.set_error_matrix(prec)
        eng.hmc_set(b.HMC_LEAPFROG, LEAPFROG)
        eng.hmc_start(x0)
        tr = eng.hmc_step_trace(steps, 3)
        runs[cache] = (eng, tr)
    eng, tr = runs[True]
    fresh = runs[False][1]
    for k in ("potential", "points", "mean_epsilon", "leapfrog", "accepted"):
        assert np.array_equal(tr[k], fresh[k]), k
    for k in ("scalars", "momentum"):
        assert np.array_equal(eng.hmc_get(k), runs[False][0].hmc_get(k)), k
    del runs
    assert tr["accepted"][:, :per_pass].any() and tr["accepted"][:, per_pass:].any()
    t = time.perf_counter()
    for c in (0, 185, per_pass - 1, per_pass, E - 1):
        o = cc.CpuHmc("orc", cc.LLH_DUMMY, n, False, seed, c)
        o.set_error_matrix(prec)
        o.set(cc.HMC_LEAPFROG, LEAPFROG)
        o.start(x0[c])
        want = o.step(steps, 3)
        st = o.state()
        check_against(eng, tr, c, want, np.array([st[k] for k in cc.HMC_STATE_FIELDS]), st, False)
    print("port: 5 chains x %d steps in %.1f s" % (steps, time.perf_counter() - t))


# ------------------------------------------------------------------------ kept gradients
def hmc_steps(eng, steps, gtype):
    """`steps` steps taken one at a time: each step's trace, and after it the proposed
    points and every scalar of every chain (proposed potential and counters among them).
    The proposal of the first step after a change shows a stale starting gradient even
    where the chain rejects it."""
    out = []
    for _ in range(steps):
        tr = eng.hmc_step_trace(1, gtype)
        tr["proposed"] = eng.hmc_get("proposed")
        tr["scalars"] = eng.hmc_get("scalars")
        out.append(tr)
    return out


def assert_same_runs(runs):
    for (name, a), (_, c) in zip(*runs):
        for s, (x, y) in enumerate(zip(a, c)):
            for k in x:
                assert np.array_equal(x[k], y[k]), (name, s, k)


def test_kept_gradients_are_dropped_when_the_unbinned_sample_changes(monkeypatch):
    """SMCMC_LLH_UNBINNED, 64 chains, finite differences (type 0: no gradient functor).
    Steps on one sample of 10^4 events, then on another of 9000: with kept gradients the run
    equals the one that computes every gradient afresh, bit for bit.  The second sample is
    smaller, so every point is more likely under it and the chains take the first
    trajectory after the change."""
    import smcmc_b200
    from smcmc_b200 import binding as b
    from smcmc_b200 import synth
    first, second = synth.make_mc_sample(4000, 6000, seed=9), synth.make_mc_sample(3600, 5400, seed=19)
    x0 = np.random.default_rng(64).normal(0.0, 0.1, (64, 9))
    runs = []
    for cache in (True, False):
        set_cache(monkeypatch, cache)
        eng = smcmc_b200.Engine(smcmc_b200.LLH_UNBINNED, 9, 64, seed=17)
        eng.set_unbinned_events(first)
        eng.hmc_set(b.HMC_LEAPFROG, LEAPFROG)
        eng.hmc_start(x0)
        eng.hmc_set(b.HMC_MEAN_EPSILON, -0.01)          # a fixed step size (SimpleAHMC.C)
        out = [("first sample", hmc_steps(eng, 4, 0))]
        eng.set_unbinned_events(second)
        out.append(("second sample", hmc_steps(eng, 4, 0)))
        runs.append(out)
    assert_same_runs(runs)
    after = runs[0][1][1]
    assert after[0]["accepted"].all()
    assert np.all(after[-1]["scalars"][:, b.HMC_SCALARS.index("gradient_count")] == 8 * (LEAPFROG + 1))


def test_kept_gradients_are_dropped_when_the_fake_events_or_data_change(monkeypatch):
    """SMCMC_LLH_FAKE, 64 chains, finite differences (type 3).  Steps on one MC sample, on
    another (SetEvents), then against other data histograms (set_fake_data): with kept
    gradients the run equals the one that computes every gradient afresh, bit for bit.  The
    new data are the second sample's own prediction at the nominal point, under which every
    point near it is more likely, so the chains take the first trajectory after that change
    (after the change of sample, those whose point became more likely take it)."""
    import smcmc_b200
    from smcmc_b200 import binding as b
    from smcmc_b200 import synth
    events, data = synth.fake_inputs(1000, 1000, 10, seed=31)              # 30 000 events
    events2 = synth.make_mc_sample(10000, 20000, seed=60)
    probe = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, 1)
    probe.set_fake_events(events)
    expo = synth.exposure_ratio(probe, data)
    probe.set_fake_events(events2)
    probe.set_fake_data(data, expo)
    data2 = probe.fake_histograms(np.zeros((1, 9)))[0]
    x0 = np.random.default_rng(65).normal(0.0, 0.1, (64, 9))
    runs = []
    for cache in (True, False):
        set_cache(monkeypatch, cache)
        eng = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, 64, seed=18)
        eng.set_fake_events(events)
        eng.set_fake_data(data, expo)
        eng.hmc_set(b.HMC_LEAPFROG, LEAPFROG)
        eng.hmc_start(x0)
        eng.hmc_set(b.HMC_MEAN_EPSILON, -0.01)
        out = [("first sample", hmc_steps(eng, 4, 3))]
        eng.set_fake_events(events2)
        out.append(("second sample", hmc_steps(eng, 4, 3)))
        eng.set_fake_data(data2, expo)
        out.append(("second data", hmc_steps(eng, 4, 3)))
        runs.append(out)
    assert_same_runs(runs)
    assert runs[0][1][1][0]["accepted"].any()
    assert runs[0][2][1][0]["accepted"].mean() > 0.9
    assert np.all(runs[0][-1][1][-1]["scalars"][:, b.HMC_SCALARS.index("gradient_count")] == 12 * (LEAPFROG + 1))


# ------------------------------------------------------------------------ built-in vs user functor
def test_builtin_unbinned_and_its_user_functor_run_the_same_chains(user_events_lib):
    """One sample of 10^4 events bound twice: to SMCMC_LLH_UNBINNED and to the user event
    functor UnbinnedEvents.  The built-in path keeps gradients between steps and picks its
    chunk length from the batch size; the user path computes every gradient, sums in
    chunks fixed by the sample size, and grows its partial-sum scratch from the 64 points
    of the start to the 2 x 9 x 64 of a gradient.  The likelihoods differ in the last bits
    (order of the sums) and finite differences magnify that by |L| / 0.02, so: the same
    accept decisions and trajectory lengths, potentials, points and step sizes within 1e-9
    relative, and the counters of 2 n potentials per gradient."""
    import smcmc_b200
    from smcmc_b200 import binding as b
    from smcmc_b200 import synth
    n, E, steps = 9, 64, 20
    events = synth.make_mc_sample(4000, 6000, seed=9)
    x0 = np.random.default_rng(66).normal(0.0, 0.1, (E, n))
    builtin = smcmc_b200.Engine(smcmc_b200.LLH_UNBINNED, n, E, seed=21)
    builtin.set_unbinned_events(events)
    user = smcmc_b200.Engine(smcmc_b200.LLH_USER, n, E, seed=21)
    user.bind_user_events(user_events_lib, "user_unbinned_bind", ues.unbinned_events(events))
    runs = []
    for eng in (builtin, user):
        eng.hmc_set(b.HMC_LEAPFROG, LEAPFROG)
        eng.hmc_start(x0)
        eng.hmc_set(b.HMC_MEAN_EPSILON, -0.01)
        tr = eng.hmc_step_trace(steps, 0)
        tr["scalars"] = eng.hmc_scalars()
        runs.append(tr)
    a, u = runs
    assert np.all(np.isfinite(u["potential"]))
    bad = np.argwhere(a["accepted"] != u["accepted"])
    assert len(bad) == 0, [(s, c, a["potential"][s, c], u["potential"][s, c]) for s, c in bad[:5]]
    assert np.array_equal(a["leapfrog"], u["leapfrog"])
    assert a["accepted"].sum() > 0
    dev = {
        "potential": np.max(np.abs(u["potential"] / a["potential"] - 1.0)),
        "mean_epsilon": np.max(np.abs(u["mean_epsilon"] / a["mean_epsilon"] - 1.0)),
        "points": np.max(np.abs(u["points"] - a["points"]).max(axis=2) / np.abs(a["points"]).max(axis=2)),
    }
    print("largest relative deviation, user functor against built-in:",
          ", ".join("%s %.2e" % kv for kv in dev.items()))
    for k, v in dev.items():
        assert v < 1e-9, (k, v)
    for k in ("gradient_count", "potential_count", "step_count", "cov_trials"):
        assert np.array_equal(a["scalars"][k], u["scalars"][k]), k
    sc = u["scalars"]
    assert np.all(sc["gradient_count"] == steps * (LEAPFROG + 1))
    # Start and every step evaluate one point each, a gradient 2 n; UpdateErrorMatrix evaluates the
    # running mean (:729) once the covariance has 2 n trials -- once within 20 steps
    updates = (sc["cov_trials"] >= 2 * n).astype(int)
    assert np.array_equal(sc["potential_count"], 1 + steps + 2 * n * sc["gradient_count"] + updates)
    assert updates.any()
