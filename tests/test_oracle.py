"""The CPU checkers against the golden vectors that the reference build
produced (tests/golden/make_golden.py), and against each other.

The oracle port (oracle/smcmc_oracle.cc) must reproduce the reference's own
code BIT FOR BIT on identical injected draws: same accept/reject sequence,
same points, same adaptive state.  Where the reference-backed library is
present (build container; or prebuilt on the GPU box) it is re-checked too.
"""
import numpy as np
import pytest

from helpers import GOLDEN_CHAINS, configure_golden, golden, golden_chain


def _set_field(c, name, value):
    from oracle import cpu_checkers as cc
    c.set({"acceptance_rigidity": cc.SET_ACCEPTANCE_RIGIDITY, "sigma": cc.SET_SIGMA}[name], value)


def _run(cc, which, name, err=None):
    kind, dim, seed, chain, nsteps, start = GOLDEN_CHAINS[name]
    c = cc.CpuChain(which, kind, dim, seed, chain)
    if kind == cc.LLH_DUMMY and which == "orc":
        c.set_error_matrix(err)
    configure_golden(name, c, _set_field)
    x0 = np.zeros(dim) if start is None else np.full(dim, start)
    ok = c.start(x0)
    tr = c.step(nsteps)
    return ok, tr, c.state()


@pytest.mark.parametrize("name", sorted(GOLDEN_CHAINS))
@pytest.mark.parametrize("which", ["orc", "ref"])
def test_chain_matches_golden_bit_for_bit(checkers, have_ref, which, name):
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("chains.npz")
    want = golden_chain(g, name)
    ok, tr, st = _run(checkers, which, name, g["dummy100_error"])
    assert ok == int(want["ok"][0])
    for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
        assert np.array_equal(tr[k], want[k]), k
    assert np.array_equal(st["cov"], want["final_cov"])
    assert np.array_equal(st["decomp"], want["final_decomp"])
    assert np.array_equal(st["center"], want["final_center"])
    scal = np.array([st[k] for k in checkers.STATE_FIELDS])
    assert np.array_equal(scal, want["final_scalars"])


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_fake_likelihood_matches_golden(checkers, have_ref, which):
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("fake_likelihood.npz")
    for tag in ("", "_irregular"):
        c = checkers.CpuChain(which, checkers.LLH_FAKE, 9, 1, 0)
        c.set_fake(g["events" + tag], g["data"], float(g["exposure"]))
        for p, llh, hist in zip(g["points"], g["llh" + tag], g["hist" + tag]):
            assert c.llh(p) == llh
            assert np.array_equal(c.fake_hist(p), hist)


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_fake_schedule_matches_golden(checkers, have_ref, which):
    """Burn-in, ResetProposal, burn-in, UpdateProposal, run: the call
    sequence of example/FakeMCMC.C:93-165."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("fake_likelihood.npz")
    for chain in (0, 7):
        c = checkers.CpuChain(which, checkers.LLH_FAKE, 9, 4242, chain)
        c.set_fake(g["events"], g["data"], float(g["exposure"]))
        c.start(g["chain%d_x0" % chain])
        parts = [c.step(60)]
        c.reset_proposal()
        parts.append(c.step(60))
        c.update_proposal()
        parts.append(c.step(120))
        for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
            got = np.concatenate([p[k] for p in parts])
            assert np.array_equal(got, g["chain%d_%s" % (chain, k)]), k
        st = c.state()
        assert np.array_equal(st["cov"], g["chain%d_cov" % chain])
        assert np.array_equal(st["decomp"], g["chain%d_decomp" % chain])


def test_port_equals_reference_on_fresh_inputs(checkers, have_ref):
    """Not just the committed chains: new seeds, every likelihood kind.  The port's traces must
    match tests/golden/fresh_seeds.npz bit for bit (a SHA-256 per array, a sample of steps for
    a readable failure; `source` there names the build that made it) and, where the
    reference-backed checker is built, the reference's own traces."""
    from golden.make_golden import FRESH_CHAINS, FRESH_CHAIN_IDS, digest, fresh_chain, fresh_sample
    g = golden("fresh_seeds.npz")
    for kind, dim, n in FRESH_CHAINS:
        for chain in FRESH_CHAIN_IDS:
            p = "k%d_d%d_c%d/" % (kind, dim, chain)
            ok, tb = fresh_chain("orc", kind, dim, n, chain)
            assert ok == int(g[p + "ok"])
            rows = fresh_sample(n, chain)
            for k in tb:
                assert np.array_equal(tb[k][rows], g[p + k + "_sample"]), (kind, dim, chain, k)
                assert np.array_equal(digest(tb[k]), g[p + k + "_sha256"]), (kind, dim, chain, k)
            if have_ref:
                ok_ref, ta = fresh_chain("ref", kind, dim, n, chain)
                assert ok_ref == ok
                for k in ta:
                    assert np.array_equal(ta[k], tb[k]), (kind, k)


def test_cholesky_identity(checkers):
    """TDecompChol restated: U upper triangular with U^T U = covariance."""
    c = checkers.CpuChain("orc", checkers.LLH_UNIT_GAUSS, 7, 3, 0)
    c.start(np.zeros(7))
    c.step(3000)
    c.update_proposal()
    st = c.state()
    u = st["decomp"]
    assert np.allclose(np.tril(u, -1), 0.0)
    assert np.allclose(u.T @ u, st["cov"], rtol=1e-12, atol=1e-14)


def test_gaussian_target_statistics(checkers):
    """Analytic known-answer test: the chain of the unit Gaussian target has
    mean 0 and unit variance (MakeCovariance.C:63-89 formulas)."""
    c = checkers.CpuChain("orc", checkers.LLH_UNIT_GAUSS, 4, 12, 0)
    c.start(np.zeros(4))
    c.step(3000)
    x = c.step(40000)["x"]
    assert np.all(np.abs(x.mean(0)) < 0.08)
    cov = np.cov(x.T)
    assert np.all(np.abs(np.diag(cov) - 1.0) < 0.1)
    assert np.all(np.abs(cov - np.diag(np.diag(cov))) < 0.08)


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_restore_matches_golden(checkers, have_ref, which):
    """Restore() into a fresh sampler continues the chain exactly as the
    reference build did (TSimpleMCMC.H:282-352, :1501-1610)."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    want = golden_chain(golden("chains.npz"), "restore7")
    cc = checkers
    a = cc.CpuChain(which, cc.LLH_UNIT_GAUSS, 7, 31, 2)
    a.start(np.full(7, 0.1))
    assert np.array_equal(a.step(250)["accepted"], want["before_accepted"])
    a.step_saved(50)
    a.save_step()
    b = cc.CpuChain(which, cc.LLH_UNIT_GAUSS, 7, 31, 2)
    b.start(np.zeros(7))
    b.restore(a)
    tr = b.step(200)
    for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
        assert np.array_equal(tr[k], want[k]), k
    assert np.array_equal(np.array([b.state()[k] for k in cc.STATE_FIELDS]), want["final_scalars"])


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_debug_modes_match_golden(checkers, have_ref, which):
    """ForceStep, SetScanDimension, SetEstimatedCenter (TSimpleMCMC.H:671-704,
    :733-739, :811-830): the port and the reference build reproduce the golden run."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    from helpers import configure_debug_modes, run_debug_modes
    want = golden_chain(golden("chains.npz"), "debug9")
    cc = checkers
    c = cc.CpuChain(which, cc.LLH_UNIT_GAUSS, 9, 61, 5)
    configure_debug_modes(c)
    c.start(np.full(9, 0.2))
    got = run_debug_modes(c)
    for k in got:
        assert np.array_equal(got[k], want[k]), k
    st = c.state()
    assert np.array_equal(np.array([st[k] for k in cc.STATE_FIELDS]), want["final_scalars"])
    assert np.array_equal(st["center"], want["final_center"])
    assert np.array_equal(st["cov"], want["final_cov"])
    # the forced point was taken (metropolis = 2), and scans only move their dimension
    assert np.array_equal(want["x"][60], np.linspace(-0.4, 0.4, 9))
    scan = want["x"][66:91]
    assert np.all(scan[:, [0, 1, 2, 4, 5, 6, 7, 8]] == scan[0, [0, 1, 2, 4, 5, 6, 7, 8]])


def test_constrained_posterior_closed_form(checkers):
    """example4's likelihood has a closed-form posterior (SURVEY.md section 4): precision
    diag(1/s_i^2) + 1 1^T / 16^2.  The restated likelihood must be that quadratic form."""
    cc = checkers
    c = cc.CpuChain("orc", cc.LLH_CONSTRAINED, 25, 1, 0)
    mu = np.array([76.0] * 24 + [80.0])
    sg = np.array([76.0 * 0.08] * 24 + [2.0])
    prec = np.diag(1.0 / sg ** 2) + np.ones((25, 25)) / 16.0 ** 2
    b = mu / sg ** 2 + 1902.0 / 16.0 ** 2
    mean = np.linalg.solve(prec, b)
    rng = np.random.default_rng(5)
    l0 = c.llh(mean)
    for _ in range(50):
        d = rng.normal(0, 3, 25)
        want = l0 - 0.5 * d @ prec @ d
        assert abs(c.llh(mean + d) - want) < 1e-9 * abs(want)


# ---------------------------------------------------------------------------
# TSimpleHMC (TSimpleHMC.H:119-973)
# ---------------------------------------------------------------------------
from helpers import HMC_GOLDEN, HMC_PORT_ONLY, hmc_error_matrix, hmc_scalar_mask  # noqa: E402


def run_cpu_hmc(cc, which, cfg, error):
    fields = {"alpha": cc.HMC_ALPHA, "mean_epsilon": cc.HMC_MEAN_EPSILON, "leapfrog": cc.HMC_LEAPFROG}
    c = cc.CpuHmc(which, cfg["kind"], cfg["dim"], cfg["grad"], cfg["seed"], cfg["chain"])
    if error is not None and which == "orc":
        c.set_error_matrix(error)
    for f, v in cfg.get("pre", ()):
        c.set(fields[f], v)
    c.start(np.full(cfg["dim"], cfg["x0"]))
    for f, v in cfg.get("post", ()):
        c.set(fields[f], v)
    tr = c.step(cfg["nsteps"], cfg["gtype"])
    return tr, c.state()


@pytest.mark.parametrize("name", sorted(HMC_GOLDEN))
@pytest.mark.parametrize("which", ["orc", "ref"])
def test_hmc_chain_matches_golden_bit_for_bit(checkers, have_ref, which, name):
    """Positions, potentials, the adapted step size and trajectory length of
    every step, and the final state (covariance estimate, its inverse, the
    counters) equal what the reference build produced."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("hmc.npz")
    want = golden_chain(g, name)
    cfg = HMC_GOLDEN[name]
    err = g["error_" + cfg["error"]] if "error" in cfg else None
    tr, st = run_cpu_hmc(checkers, which, cfg, err)
    for k in ("potential", "x", "epsilon", "leapfrog"):
        assert np.array_equal(tr[k], want[k]), k
    scal = np.array([st[k] for k in checkers.HMC_STATE_FIELDS])
    mask = hmc_scalar_mask(want["final_scalars"], cfg["dim"])
    assert np.array_equal(scal[mask], want["final_scalars"][mask])
    for k in ("accepted", "momentum", "central", "average", "covariance", "error"):
        assert np.array_equal(st[k], want["final_" + k], equal_nan=True), k


def test_hmc_samples_the_target(checkers):
    """Known-answer check of the restated sampler itself: the marginal
    variances of a correlated Gaussian target (precision matrix P) are the
    diagonal of P^-1."""
    n = 6
    prec = hmc_error_matrix("spd6")
    c = checkers.CpuHmc("orc", checkers.LLH_DUMMY, n, True, 77, 0)
    c.set_error_matrix(prec)
    c.start(np.zeros(n))
    c.step(500)
    x = c.step(6000)["x"]
    var = np.diag(np.linalg.inv(prec))
    assert np.all(np.abs(x.mean(0)) < 0.15)
    assert np.all(np.abs(x.var(0) / var - 1.0) < 0.2)


# ---------------------------------------------------------------------------
# The unbinned mixture likelihood (not in the reference; defined in
# include/smcmc_b200.h).  Its checker is the port only: pin the port against an
# independent numpy statement of the definition.
# ---------------------------------------------------------------------------
def numpy_unbinned(events, p):
    from math import erf, pi
    scale, width, skewc = p[2] / 10.0, np.exp(p[3] / 10.0), 0.3 * erf(p[4] / 10.0)
    fakes = np.arctan(np.tan(pi * (0.05 - 0.5)) + p[7]) / pi + 0.5
    eff = np.arctan(np.tan(pi * (0.5 - 0.5)) + p[8]) / pi + 0.5
    w_s, w_b = np.exp(p[0] / 10.0), np.exp(p[1] / 10.0)
    tag = events["MuDk"] > 0
    lws = np.where(tag, np.log(w_s * fakes / 0.05), np.log(w_s * (1 - fakes) / 0.95))
    lwb = np.where(tag, np.log(w_b * eff / 0.5), np.log(w_b * (1 - eff) / 0.5))
    nl = np.log(events["TrueMass"])
    d = np.log(events["Mass"]) - nl
    ls = d / (np.log(events["TrueMass"] + events["TrueMassSigma"]) - nl)
    lm = nl + d * np.exp(ls * skewc) * width + scale
    sig, tau = np.log(1.3), 500.0
    a = lws - np.log(sig * np.sqrt(2 * pi)) - 0.5 * ((lm - np.log(135.0)) / sig) ** 2 - lm
    b = lwb - np.log(tau) - np.exp(lm) / tau
    return float(np.sum(np.logaddexp(a, b)))


def test_unbinned_port_matches_its_definition(checkers):
    import smcmc_b200.synth as synth
    events = synth.make_mc_sample(700, 1300, seed=9)
    c = checkers.CpuChain("orc", checkers.LLH_UNBINNED, 9, 1, 0)
    c.set_fake(events, np.zeros(150), 1.0)
    rng = np.random.default_rng(4)
    for p in np.concatenate([np.zeros((1, 9)), rng.uniform(-2, 2, (12, 9))]):
        want = numpy_unbinned(events, p)
        assert abs(c.llh(p) / want - 1.0) < 1e-13
    # a sum over events: additive over any split of the sample
    a = checkers.CpuChain("orc", checkers.LLH_UNBINNED, 9, 1, 0)
    b = checkers.CpuChain("orc", checkers.LLH_UNBINNED, 9, 1, 0)
    a.set_fake(events[:900], np.zeros(150), 1.0)
    b.set_fake(events[900:], np.zeros(150), 1.0)
    p = rng.uniform(-1, 1, 9)
    assert abs((a.llh(p) + b.llh(p)) / c.llh(p) - 1.0) < 1e-13


# ---------------------------------------------------------------------------
# example2/FakeLikelihood.H (SURVEY.md 8f rank 2)
# ---------------------------------------------------------------------------
def _fake2_schedule(c, g, chain):
    c.set_fake(g["events"], g["data"], 1.0)
    c.set_gaussian(0, 15.0)
    c.set_gaussian(1, 15.0)
    c.start(g["chain%d_x0" % chain])
    parts = [c.step(80)]
    c.reset_proposal()
    parts.append(c.step(80))
    c.update_proposal()
    parts.append(c.step(140))
    return parts


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_fake2_likelihood_matches_golden(checkers, have_ref, which):
    """Signal / background histograms renormalised by their integrals and the
    penalty terms (example2/FakeLikelihood.H:58-118, 222-289): bit for bit."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("fake2_likelihood.npz")
    for tag in ("", "_irregular"):
        c = checkers.CpuChain(which, checkers.LLH_FAKE2, 9, 1, 0)
        c.set_fake(g["events" + tag], g["data"], 1.0)
        for p, llh, hist in zip(g["points"], g["llh" + tag], g["hist" + tag]):
            assert c.llh(p) == llh
            assert np.array_equal(c.fake_hist(p), hist)


@pytest.mark.parametrize("which", ["orc", "ref"])
def test_fake2_schedule_matches_golden(checkers, have_ref, which):
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("fake2_likelihood.npz")
    for chain in (0, 5):
        c = checkers.CpuChain(which, checkers.LLH_FAKE2, 9, 777, chain)
        parts = _fake2_schedule(c, g, chain)
        for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
            got = np.concatenate([p[k] for p in parts])
            assert np.array_equal(got, g["chain%d_%s" % (chain, k)]), k
        st = c.state()
        assert np.array_equal(st["cov"], g["chain%d_cov" % chain])
        assert np.array_equal(st["decomp"], g["chain%d_decomp" % chain])


def test_fake2_port_equals_reference_on_fresh_inputs(checkers, have_ref):
    """New events and points, including negative event counts (the penalty
    branches) and a point where every event is cut (x / 0 normalisation): the port
    against tests/golden/fresh_seeds.npz and, where it is built, the reference."""
    from golden.make_golden import digest, fresh_fake2
    g = golden("fresh_seeds.npz")
    llh, hist = fresh_fake2("orc")
    assert np.array_equal(llh, g["fake2/llh"], equal_nan=True)
    assert np.array_equal(hist[::7], g["fake2/hist_sample"], equal_nan=True)
    assert np.array_equal(digest(hist), g["fake2/hist_sha256"])
    if have_ref:
        llh_ref, hist_ref = fresh_fake2("ref")
        assert np.array_equal(llh, llh_ref, equal_nan=True)
        assert np.array_equal(hist, hist_ref, equal_nan=True)
    assert np.isnan(llh[0])


# ---------------------------------------------------------------------------
# TProposeVAATStep (SURVEY.md 8f rank 4)
# ---------------------------------------------------------------------------
def _vaat_run(checkers, which, name):
    from golden.make_golden import VAAT_CHAINS
    kind, dim, seed, chain, nsteps, configure = VAAT_CHAINS[name]
    c = checkers.CpuChain(which, kind, dim, seed, chain, vaat=True)
    if configure:
        configure(c)
    ok = c.start(np.zeros(dim))
    first = c.step(nsteps - 300)
    c.set(checkers.SET_ACCEPTANCE_WINDOW, 37.0)
    second = c.step(300)
    return ok, first, second, c


@pytest.mark.parametrize("which", ["orc", "ref"])
@pytest.mark.parametrize("name", ["vaat_unit5", "vaat_unit9_hints", "vaat_horrific75"])
def test_vaat_chain_matches_golden(checkers, have_ref, which, name):
    """TSimpleMCMC<L, TProposeVAATStep>: shuffled index queue, per-dimension step
    size and acceptance (TProposeVAATStep.H:40-80, 176-190, 216-254), bit for bit."""
    if which == "ref" and not have_ref:
        pytest.skip("reference-backed checker not built here")
    g = golden("vaat.npz")
    ok, first, second, c = _vaat_run(checkers, which, name)
    assert ok == int(g[name + "/ok"][0])
    for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
        assert np.array_equal(np.concatenate([first[k], second[k]]), g[name + "/" + k]), k
    v = c.vaat_state()
    for k in ("sigma", "acceptance", "acceptance_trials"):
        assert np.array_equal(np.asarray(v[k]), g[name + "/final_" + k]), k
    assert [v["trials"], v["successes"], v["last_index"], v["queue"]] == list(g[name + "/final_misc"])
    assert c.state()["step_rms"] == g[name + "/final_step_rms"][0]


@pytest.mark.parametrize("n", [2, 5, 50, 100])
def test_shim_linear_algebra_against_lapack(checkers, n):
    """ROOT is absent, so `oracle/_ref` runs the reference's headers on a restatement of the ROOT
    linear algebra they call (oracle/rootshim: TDecompChol, TMatrixD::Invert, TMatrixDSymEigen),
    here compiled on its own (oracle/shim_linalg.cc).
    Held here against LAPACK (numpy), an independent implementation, on random symmetric positive
    definite matrices of the sizes the golden chains use: the factor, the inverse and the spectrum
    are unique, so agreement to rounding pins what the shim computes, not how."""
    rng = np.random.default_rng(1000 + n)
    for trial in range(4):
        g = rng.normal(size=(n, 2 * n))
        a = g @ g.T / (2 * n) + 0.05 * np.eye(n)
        if trial == 3:                                   # strongly correlated, condition number ~1e6
            d = np.logspace(0, 3, n)
            a = d[:, None] * (0.98 + 0.02 * np.eye(n)) * d[None, :]
        cond = np.linalg.cond(a)
        u, _ = checkers.shim_linalg(0, a)
        assert np.array_equal(np.tril(u, -1), np.zeros((n, n)))
        assert np.allclose(u, np.linalg.cholesky(a).T, rtol=1e-13 * cond, atol=1e-15 * np.abs(a).max())
        inv, _ = checkers.shim_linalg(1, a)
        ref = np.linalg.inv(a)
        assert np.abs(inv - ref).max() <= 1e-14 * cond * np.abs(ref).max()
        vec, val = checkers.shim_linalg(2, a)
        w, v = np.linalg.eigh(a)
        w, v = w[::-1], v[:, ::-1]                       # the reference relies on DESCENDING eigenvalues
        assert np.all(np.diff(val) <= 0.0)
        assert np.allclose(val, w, rtol=0, atol=1e-13 * w[0])
        assert np.allclose(vec.T @ vec, np.eye(n), atol=1e-12)
        assert np.abs(a @ vec - vec * val[None, :]).max() <= 1e-12 * w[0]
        gap = np.min(np.abs(np.diff(w))) / w[0]
        if gap > 1e-6:                                   # simple spectrum: the eigenvectors themselves, up to sign
            sign = np.sign(np.sum(vec * v, axis=0))
            assert np.abs(vec * sign[None, :] - v).max() <= 1e-12 / gap
    # a matrix that is not positive definite: Decompose() fails (TSimpleMCMC.H:1100-1118 takes that branch)
    bad = np.eye(n)
    bad[n - 1, n - 1] = -1.0
    assert checkers.shim_linalg(0, bad)[0] is None
