"""User EVENT functors on the device (include/smcmc_device_functor.cuh: kEventPairs,
kEventFinish, EventBinding).  The functors (tests/cpp/user_events.cuh) are
compiled by nvcc in a user translation unit; libsmcmc_b200 has no kernel for
them.  Checks: the device value equals the host restatement of the documented
summation order bit for bit, whatever else is evaluated in the same call; the
unbinned mixture restated as a user functor agrees with the built-in kernel and
the oracle port, and its chains follow the port's; the ensemble finds the known
posterior of a Gaussian sample; the C++ mirror reproduces a Python-bound chain;
TSimpleHMC runs on finite differences; misuse raises."""
import os
import re
import subprocess

import numpy as np
import pytest

import user_events_support as ues

pytestmark = pytest.mark.gpu

NS = [0, 1, 127, 128, 129, 1023, 1024, 1025, 10 ** 6]     # 1024: the chunk length below 262 145 events


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    return ues.build_library(str(tmp_path_factory.mktemp("user_events")))


@pytest.fixture(scope="module")
def program(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "user_events")
    subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-o", exe, os.path.join(ues.CPP, "user_events.cu"), "-L", ues.LIBDIR,
                                                "-lsmcmc_b200", "-Xlinker", "-rpath," + ues.LIBDIR], check=True)
    return exe


def engine(lib, kind, events, dim, chains=4, seed=1, chain_offset=0):
    import smcmc_b200
    eng = smcmc_b200.Engine(smcmc_b200.LLH_USER, dim, chains, seed=seed, chain_offset=chain_offset)
    eng.bind_user_events(lib, "user_%s_bind" % kind, events)
    return eng


def gauss_points(m, seed=0):
    return np.random.default_rng(seed).uniform([2.0, 1.0], [4.0, 3.0], (m, 2))


@pytest.mark.parametrize("n", NS)
def test_gauss_equals_the_host_restatement_bit_for_bit(lib, n):
    ev = ues.gauss_events(n, seed=n + 1)
    eng = engine(lib, "gauss", ev, 2)
    for m in (1, 5, 128, 129, 1000):
        pts = gauss_points(m, seed=m)
        assert np.array_equal(eng.eval(pts), ues.host_values(lib, "gauss", ev, pts)), m


@pytest.mark.parametrize("kind", ["gauss12", "gauss128"])
@pytest.mark.parametrize("n", [1, 129, 5000])
def test_awkward_event_sizes_bit_for_bit(lib, kind, n):
    rng = np.random.default_rng(n)
    ev = np.zeros(n, ues.KINDS[kind][1])
    if kind == "gauss12":
        ev["v"] = rng.normal(3, 2, n)
        ev["w"] = rng.uniform(-1, 1, n)
        ev["k"] = rng.integers(-3, 4, n)
    else:
        ev["v"] = rng.normal(3, 2, (n, 16))
    eng = engine(lib, kind, ev, 2)
    for m in (1, 129):
        pts = gauss_points(m, seed=m)
        assert np.array_equal(eng.eval(pts), ues.host_values(lib, kind, ev, pts))


def test_a_points_value_does_not_depend_on_the_batch(lib):
    ev = ues.gauss_events(100000, seed=5)
    eng = engine(lib, "gauss", ev, 2)
    pts = gauss_points(1000, seed=6)
    full = eng.eval(pts)
    for i in (0, 1, 127, 128, 500, 999):
        assert eng.eval(pts[i:i + 1])[0] == full[i]
    assert np.array_equal(eng.eval(pts[::-1]), full[::-1])
    assert np.array_equal(eng.eval(pts), full)


def unbinned_setup(lib, n_sig, n_bkg, chains, seed=9):
    import smcmc_b200
    from smcmc_b200 import synth
    events = synth.make_mc_sample(n_sig, n_bkg, seed=seed)
    user = engine(lib, "unbinned", ues.unbinned_events(events), 9, chains, seed=12)
    builtin = smcmc_b200.Engine(smcmc_b200.LLH_UNBINNED, 9, chains, seed=12)
    builtin.set_unbinned_events(events)
    return user, builtin, events


def oracle_llh(events, pts):
    from oracle import cpu_checkers as cc
    c = cc.CpuChain("orc", cc.LLH_UNBINNED, 9, 12, 0)
    c.set_fake(events, np.zeros(150), 1.0)
    return np.array([c.llh(p) for p in pts])


def test_unbinned_functor_matches_the_builtin_and_the_port(lib):
    user, builtin, events = unbinned_setup(lib, 7000, 13000, 64)
    rng = np.random.default_rng(1)
    pts = np.concatenate([np.zeros((1, 9)), rng.uniform(-1, 1, (150, 9)), rng.normal(0, 4, (49, 9))])
    got = user.eval(pts)
    assert np.all(np.isfinite(got))
    assert np.max(np.abs(got / builtin.eval(pts) - 1.0)) < 1e-12
    assert np.max(np.abs(got / oracle_llh(events, pts) - 1.0)) < 1e-12
    # and the host restatement of the functor (glibc's exp/log against CUDA's)
    assert np.max(np.abs(got / ues.host_values(lib, "unbinned", ues.unbinned_events(events), pts) - 1.0)) < 1e-12


def test_unbinned_non_positive_mass_is_nan_and_rejected(lib):
    from smcmc_b200 import synth
    events = synth.make_mc_sample(50, 50, seed=9)
    bad = events.copy()
    bad["Mass"][7] = -1.0
    eng = engine(lib, "unbinned", ues.unbinned_events(bad), 9, 4)
    assert np.all(np.isnan(eng.eval(np.zeros((3, 9)))))
    assert not eng.start(np.zeros(9)).any()          # an unusable starting likelihood
    eng.bind_user_events(lib, "user_unbinned_bind", ues.unbinned_events(events))
    assert eng.start(np.zeros(9)).all()


def test_unbinned_metropolis_chains_follow_the_port(lib):
    from oracle import cpu_checkers as cc
    user, _, events = unbinned_setup(lib, 1500, 2500, 6)
    x0 = np.random.default_rng(8).uniform(-1, 1, (6, 9))
    assert user.start(x0).all()
    tr = user.step_trace(150)
    for c in range(6):
        o = cc.CpuChain("orc", cc.LLH_UNBINNED, 9, 12, c)
        o.set_fake(events, np.zeros(150), 1.0)
        o.start(x0[c])
        want = o.step(150)
        assert np.array_equal(tr["accepted"][:, c], want["accepted"])
        assert np.allclose(tr["llh_accepted"][:, c], want["llh_accepted"], rtol=1e-11)
        assert np.allclose(tr["points"][:, c], want["x"], rtol=1e-9, atol=1e-12)


def test_gaussian_sample_posterior(lib):
    """10^5 events from N(3, 2), 4096 chains with pooled adaptation: the posterior
    of (mu, sigma) under a flat prior is centred on the sample mean with standard
    deviations s/sqrt(N) and s/sqrt(2N)."""
    from smcmc_b200 import binding
    E, N = 4096, 100000
    ev = ues.gauss_events(N, 3.0, 2.0, seed=11)
    v = ev["v"]
    eng = engine(lib, "gauss", ev, 2, E, seed=9)
    eng.prop_set(binding.PROP_POOLED_EVERY, 20)
    assert eng.start(np.array([3.0, 2.0])).all()
    eng.step(1000)
    eng.reset_proposal()
    eng.step(1000)
    pts = []
    for _ in range(16):
        eng.step(40)
        pts.append(eng.get("accepted"))
    x = np.concatenate(pts)
    s = v.std()
    sd_mu, sd_sigma = s / np.sqrt(N), s / np.sqrt(2 * N)
    se = sd_mu / np.sqrt(E * 4)                       # generous: autocorrelated samples
    assert abs(x[:, 0].mean() - v.mean()) < 6 * se, (x[:, 0].mean() - v.mean()) / se
    assert abs(x[:, 0].std() / sd_mu - 1.0) < 0.1
    assert abs(x[:, 1].std() / sd_sigma - 1.0) < 0.1
    assert abs(x[:, 1].mean() - s) < 6 * sd_sigma
    assert np.all(eng.get("status") == 0)


def test_cpp_program_reproduces_the_python_chain(lib, program, tmp_path):
    """sMCMC::TSimpleMCMC<GaussEvents> with a TTree, events set before Start and
    again halfway: the chain of a Python-bound engine with the same seed and chain
    index, accept for accept and bit for bit."""
    ev = ues.gauss_events(5000, seed=21)
    path = str(tmp_path / "events.bin")
    ev["v"].tofile(path)
    steps = 200
    r = subprocess.run([program, "chain", path, "7", "3", str(steps)], capture_output=True, text=True, check=True)
    s = re.search(r"start llh (\S+) host (\S+)", r.stdout)
    assert s and float(s.group(1)) == float(s.group(2))
    rows = re.findall(r"step (\d+) acc (\d) llh (\S+) x (\S+) (\S+)", r.stdout)
    assert len(rows) == steps
    eng = engine(lib, "gauss", ev, 2, 1, seed=7, chain_offset=3)
    assert eng.start(np.array([2.5, 1.5])).all()
    assert eng.eval(np.array([[2.5, 1.5]]))[0] == float(s.group(1))
    tr = eng.step_trace(steps)
    assert np.array_equal(np.array([int(x[1]) for x in rows]), tr["accepted"][:, 0])
    assert np.array_equal(np.array([float(x[2]) for x in rows]), tr["llh_accepted"][:, 0])
    assert np.array_equal(np.array([[float(x[3]), float(x[4])] for x in rows]), tr["points"][:, 0])
    # the comparison covers accepted moves, not only a chain standing still (the start is
    # several posterior widths from the sample's mean, so the first proposals mostly fail)
    assert tr["accepted"][:, 0].sum() >= 5
    assert np.all(tr["points"][-1, 0] != np.array([2.5, 1.5]))
    m = re.search(r"entries (\d+) calls (\d+)", r.stdout)
    assert m and int(m.group(1)) == steps + 1 and int(m.group(2)) == steps + 1


def test_hmc_with_finite_differences(lib, program, tmp_path):
    """TSimpleHMC<GaussEvents>: no gradient entry, so finite differences of the
    likelihood (evaluated at 2 x dim x chains points per gradient, which grows the
    partial-sum scratch).  Potentials stay finite; the likelihood's central
    differences agree with the analytic gradient."""
    N = 5000
    ev = ues.gauss_events(N, seed=31)
    v = ev["v"]
    eng = engine(lib, "gauss", ev, 2, 64, seed=61)
    eng.hmc_start(np.array([2.8, 2.1]))
    eng.hmc_step(50, 1)
    sc = eng.hmc_scalars()
    assert np.all(sc["step_count"] == 50)
    assert np.all(np.isfinite(sc["accepted_potential"]))
    assert np.all(sc["potential_count"] > 50 * 4)     # finite differences: 2 x dim potentials per gradient
    mu, sigma, h = 2.8, 2.1, 1e-5
    probe = np.array([[mu + h, sigma], [mu - h, sigma], [mu, sigma + h], [mu, sigma - h]])
    f = eng.eval(probe)
    fd = np.array([(f[0] - f[1]) / (2 * h), (f[2] - f[3]) / (2 * h)])
    exact = np.array([np.sum(v - mu) / sigma ** 2, np.sum((v - mu) ** 2) / sigma ** 3 - N / sigma])
    assert np.allclose(fd, exact, rtol=1e-6)
    path = str(tmp_path / "events.bin")
    v.tofile(path)
    r = subprocess.run([program, "hmc", path, "64", "50"], capture_output=True, text=True, check=True)
    assert re.search(r"hmc finite 64 of 64 potentials (\d+) gradients", r.stdout), r.stdout


def test_misuse_raises(lib):
    import smcmc_b200
    eng = smcmc_b200.Engine(smcmc_b200.LLH_USER, 2, 4, seed=1)
    assert lib.user_gauss_bind_without_sample(eng.h) == 1
    assert b"no event sample" in lib.user_events_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        eng.bind_user_events(lib, "user_gauss_bind", np.zeros(10, np.float32))
    assert b"sizeof(Event)" in lib.user_events_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        eng.eval(np.zeros((1, 2)))                   # nothing registered
    eng.bind_user_events(lib, "user_gauss_bind", ues.gauss_events(0))
    assert np.array_equal(eng.eval(np.array([[1.0, 2.0]])), [0.0])   # empty sample: Finish(c, 0, 0)
