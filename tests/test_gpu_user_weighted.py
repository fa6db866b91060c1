"""User WEIGHTED binned event functors on the device (include/smcmc_device_functor.cuh:
kWeightedPairs, kWeightedFinish, WeightedBinnedBinding).  The functors
(tests/cpp/user_weighted.cuh) are compiled by nvcc in a user translation unit;
libsmcmc_b200 has no kernel for them.  Checks: device sums and values equal the
host restatement bit for bit, whatever else is evaluated in the same call; a Bin
outside [0, kBins) adds nothing, whatever its weight; the reference's FillFake and
EvalFake written as a weighted functor fill the oracle port's histograms and
follow the built-in's chains; a template fit with per-event weights finds the
sample's mean and width; the C++ mirror reproduces a Python-bound chain; data
changes reach the device; misuse raises."""
import os
import re
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import user_binned_support as ubs
import user_events_support as ues
import user_weighted_support as uws

pytestmark = pytest.mark.gpu

NS = [0, 1, 127, 128, 129, 1023, 1024, 1025, 32768, 32769, 10 ** 6]
MS = [1, 5, 128, 129, 1000]


@pytest.fixture(scope="module")
def data():
    return ubs.gauss_data(10000, seed=2)


@pytest.fixture(scope="module")
def lib(tmp_path_factory, data):
    lib = uws.build_library(str(tmp_path_factory.mktemp("user_weighted")))
    uws.set_gauss_data(lib, data[1])
    return lib


@pytest.fixture(scope="module")
def program(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "user_weighted")
    subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-o", exe, os.path.join(ues.CPP, "user_weighted.cu"), "-L",
                                                ues.LIBDIR, "-lsmcmc_b200", "-Xlinker", "-rpath," + ues.LIBDIR],
                   check=True)
    return exe


def engine(lib, symbol, events, dim, chains=4, seed=1, chain_offset=0):
    import smcmc_b200
    eng = smcmc_b200.Engine(smcmc_b200.LLH_USER, dim, chains, seed=seed, chain_offset=chain_offset)
    eng.bind_user_events(lib, symbol, events)
    return eng


def gauss_points(m, seed=0):
    return np.random.default_rng(seed).uniform([2.0, 1.0], [4.0, 3.0], (m, 2))


def raw_points(m):
    return np.linspace(-2.0, 3.0, m).reshape(m, 1)


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("kind", ["gauss", "raw"])
def test_device_equals_the_host_restatement_bit_for_bit(lib, kind, n):
    if kind == "gauss":
        ev, code, symbol, points = uws.gauss_template(n, seed=n + 1), uws.GAUSS, "user_gauss_weighted_bind", gauss_points
    else:
        ev, code, symbol, points = uws.raw_events(n, seed=n), uws.RAW, "user_raw_weighted_bind", raw_points
    eng = engine(lib, symbol, ev, 2 if kind == "gauss" else 1)
    for m in MS:
        pts = points(m) if kind == "raw" else points(m, seed=m)
        values, sums = uws.host(lib, code, ev, pts)
        assert uws.same_bits(uws.device_sums(lib, code, eng, pts), sums), m
        assert uws.same_bits(eng.eval(pts), values), m


def test_bins_outside_0_to_kbins_add_nothing(lib):
    """RawWeighted events with Bin -1, -5, INT_MIN, kBins, kBins + 1 and INT_MAX,
    each with a NaN, inf and -inf weight, then bins 0 and kBins - 1: only the last
    two are summed, at 1, 64 (one CTA) and 300 points."""
    ev = np.zeros(6 * 3 + 3, uws.RAW_DTYPE)
    ev["bin"][:18] = np.repeat(uws.RAW_OUTSIDE, 3)
    ev["w"][:18] = np.tile([np.nan, np.inf, -np.inf], 6)
    ev["bin"][18:] = [0, 59, 59]
    ev["w"][18:] = [0.25, 1.5, 2.0]
    eng = engine(lib, "user_raw_weighted_bind", ev, 1)
    for m in (1, 64, 300):
        pts = np.arange(1.0, m + 1.0).reshape(m, 1)
        want = np.zeros((m, 60))
        want[:, 0], want[:, 59] = 0.25 * pts[:, 0], 3.5 * pts[:, 0]
        got = uws.device_sums(lib, uws.RAW, eng, pts)
        assert uws.same_bits(got, want), m
        assert uws.same_bits(eng.eval(pts), uws.host(lib, uws.RAW, ev, pts)[0]), m
        assert np.all(np.isfinite(got))


def test_a_points_value_does_not_depend_on_the_batch(lib):
    ev = uws.gauss_template(300000, seed=5)
    eng = engine(lib, "user_gauss_weighted_bind", ev, 2)
    pts = gauss_points(1000, seed=6)
    full = eng.eval(pts)
    full_sums = uws.device_sums(lib, uws.GAUSS, eng, pts)
    for i in (0, 1, 63, 64, 127, 128, 500, 999):
        assert uws.same_bits(eng.eval(pts[i:i + 1]), full[i:i + 1])
        assert uws.same_bits(uws.device_sums(lib, uws.GAUSS, eng, pts[i:i + 1]), full_sums[i:i + 1])
        again = eng.eval(pts[max(i - 3, 0):i + 4])
        assert uws.same_bits(again[min(i, 3)], full[i])
    assert uws.same_bits(eng.eval(pts[::-1]), full[::-1])
    assert uws.same_bits(uws.device_sums(lib, uws.GAUSS, eng, pts[::-1]), full_sums[::-1])
    assert uws.same_bits(eng.eval(pts), full)


# ---------------------------------------------------------------------------
# FakeWeighted against the oracle port's FillFake / EvalFake and the built-in
# ---------------------------------------------------------------------------
def c2_sample():
    """bench.py's C2 sample: 10^6 MC events and the data histograms."""
    from smcmc_b200 import synth
    n = 10 ** 6
    signal = n // 3 + (1 if n % 3 else 0)
    return synth.make_mc_sample(signal, n - signal, seed=2), synth.make_data_histograms(33334, 33334, seed=2)


@pytest.fixture(scope="module")
def fake_setup(lib):
    import smcmc_b200
    from smcmc_b200 import synth
    events, data = c2_sample()
    chains = 256
    builtin = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, chains, seed=3)
    builtin.set_fake_events(events)
    exposure = synth.exposure_ratio(builtin, data)
    builtin.set_fake_data(data, exposure)
    uws.set_fake_data(lib, data, exposure)
    user = engine(lib, "user_fake_weighted_bind", uws.fake_events(lib, events), 9, chains, seed=3)
    return user, builtin, events, data, exposure


def fake_points():
    rng = np.random.default_rng(8)
    start = np.stack([np.random.default_rng([3, c]).uniform(-1.0, 1.0, 9) for c in range(64)])
    wide = rng.normal(0, 10, (64, 9))
    extreme = rng.normal(0, 60, (64, 9))
    bad = rng.uniform(-1, 1, (64, 9))
    bad[0, 2] = np.nan
    bad[1, 3] = np.inf
    bad[2, 3] = -np.inf
    bad[3, 4] = np.nan
    bad[4, 5] = np.inf
    bad[5, 6] = np.nan
    bad[6, 0] = np.inf
    bad[7, 8] = np.nan
    bad[8, 1] = -np.inf
    return np.concatenate([start, wide, extreme, bad])


@pytest.fixture(scope="module")
def port_results(fake_setup):
    """The port's fake_hist and llh at every fake point, one oracle chain per
    worker thread (the port runs with the GIL released)."""
    from oracle import cpu_checkers as cc
    _, _, events, data, exposure = fake_setup
    pts = fake_points()
    workers = max(1, min(32, os.cpu_count() or 1))

    def run(rows):
        orc = cc.CpuChain("orc", cc.LLH_FAKE, 9, 1, 0)
        orc.set_fake(events, data, exposure)
        return [(orc.fake_hist(pts[i]), orc.llh(pts[i])) for i in rows]

    with ThreadPoolExecutor(workers) as pool:
        parts = list(pool.map(run, np.array_split(np.arange(len(pts)), workers)))
    res = [r for part in parts for r in part]
    return np.array([h for h, _ in res]), np.array([v for _, v in res])


def bin_events(builtin, pts):
    """Events in each of the 150 histogram bins at every point: the built-in's
    per-class counts (equal to FakeBinned's and the port's) added over the classes."""
    k = builtin.fake_counts(pts).astype(np.int64)
    n = k[:, 300:450].copy()                         # data-typed events
    n[:, :100] += k[:, :100] + k[:, 150:250]         # Close and Separated: signal, background
    n[:, 100:] += k[:, 100:150] + k[:, 250:300]      # DecayTag
    return n


def test_fake_weighted_histograms_equal_the_port(lib, fake_setup, port_results):
    """Within 1e-12 relative, widened where a bin holds so many events that the
    rounding of the port's own sum can exceed it: the port adds a bin's n weights
    in one pass (relative error up to (n - 1) 2^-53 for positive weights), the
    device in chunks (less), so the bound is 1e-12 + 2 n 2^-53.  At the extreme
    points a bin holds up to 6.5e5 of the 10^6 events."""
    user, builtin = fake_setup[:2]
    pts = fake_points()
    assert pts.shape == (256, 9)
    got = uws.device_sums(lib, uws.FAKE, user, pts)
    want = port_results[0]
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(np.isposinf(got), np.isposinf(want))
    assert np.array_equal(np.isneginf(got), np.isneginf(want))
    assert np.array_equal(got == 0, want == 0)
    fin = np.isfinite(want) & (want != 0)
    tol = 1e-12 + 2.0 * bin_events(builtin, pts) * 2.0 ** -53
    assert np.all(np.abs(got[fin] / want[fin] - 1.0) <= tol[fin])
    start = fin[:64]
    assert np.max(np.abs(got[:64][start] / want[:64][start] - 1.0)) < 1e-12   # start points: 1e-12 throughout
    assert np.count_nonzero(fin[:64]) > 64 * 100
    assert (~np.isfinite(want)).any()


def test_fake_weighted_values_equal_the_port_and_the_builtin(fake_setup, port_results):
    user, builtin = fake_setup[:2]
    pts = fake_points()
    got, port, want = user.eval(pts), port_results[1], builtin.eval(pts)
    for ref in (port, want):
        assert np.array_equal(np.isfinite(got), np.isfinite(ref))
        fin = np.isfinite(ref)
        assert fin[:192].all()
        assert np.max(np.abs(got[fin] / ref[fin] - 1.0)) < 1e-10


def test_fake_weighted_metropolis_follows_the_builtin(fake_setup):
    user, builtin = fake_setup[:2]
    x0 = np.stack([np.random.default_rng([3, c]).uniform(-1.0, 1.0, 9) for c in range(256)])
    assert user.start(x0).all()
    assert builtin.start(x0).all()
    tu = user.step_trace(20)
    tb = builtin.step_trace(20)
    assert np.array_equal(tu["accepted"], tb["accepted"])
    assert tu["accepted"].sum() > 0
    assert np.allclose(tu["points"], tb["points"], rtol=1e-9, atol=1e-12)
    assert np.allclose(tu["llh_accepted"], tb["llh_accepted"], rtol=1e-9, atol=0)


# ---------------------------------------------------------------------------
def test_template_fit_posterior(lib, data):
    """10^4 data events from N(3, 2), a flat template of 10^6 events reweighted to
    N(mu, sigma) event by event, 4096 chains with pooled adaptation: the posterior
    of (mu, sigma) is centred on the sample's mean and width, with widths s/sqrt(N)
    and s/sqrt(2N)."""
    from smcmc_b200 import binding
    v, _ = data
    E, N = 4096, len(v)
    eng = engine(lib, "user_gauss_weighted_bind", uws.gauss_template(10 ** 6, seed=11), 2, E, seed=9)
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
    assert abs(x[:, 0].mean() - v.mean()) < 0.5 * sd_mu, (x[:, 0].mean() - v.mean()) / sd_mu
    assert abs(x[:, 1].mean() - s) < 0.5 * sd_sigma, (x[:, 1].mean() - s) / sd_sigma
    assert abs(x[:, 0].std() / sd_mu - 1.0) < 0.15
    assert abs(x[:, 1].std() / sd_sigma - 1.0) < 0.15
    assert np.all(eng.get("status") == 0)


def test_cpp_program_reproduces_the_python_chain(lib, program, data, tmp_path):
    """sMCMC::TSimpleMCMC<GaussWeighted> with a TTree and events set before Start:
    the chain of a Python-bound engine with the same seed and chain index, accept
    for accept and bit for bit; then a data change through SyncLikelihood."""
    ev = uws.gauss_template(20000, seed=21)
    tpath, dpath = str(tmp_path / "template.bin"), str(tmp_path / "data.bin")
    ev["u"].tofile(tpath)
    data[1].tofile(dpath)
    steps = 200
    r = subprocess.run([program, tpath, dpath, "7", "3", str(steps)], capture_output=True, text=True, check=True)
    s = re.search(r"start llh (\S+) host (\S+)", r.stdout)
    assert s and float(s.group(1)) == float(s.group(2))
    rows = re.findall(r"step (\d+) acc (\d) llh (\S+) x (\S+) (\S+)", r.stdout)
    assert len(rows) == steps
    eng = engine(lib, "user_gauss_weighted_bind", ev, 2, 1, seed=7, chain_offset=3)
    assert eng.start(np.array([2.5, 1.5])).all()
    assert eng.eval(np.array([[2.5, 1.5]]))[0] == float(s.group(1))
    tr = eng.step_trace(steps)
    assert np.array_equal(np.array([int(x[1]) for x in rows]), tr["accepted"][:, 0])
    assert np.array_equal(np.array([float(x[2]) for x in rows]), tr["llh_accepted"][:, 0])
    assert np.array_equal(np.array([[float(x[3]), float(x[4])] for x in rows]), tr["points"][:, 0])
    assert tr["accepted"][:, 0].sum() >= 5
    m = re.search(r"entries (\d+) calls (\d+)", r.stdout)
    assert m and int(m.group(1)) == steps + 1 and int(m.group(2)) == steps + 1
    y = re.search(r"sync before (\S+) stale (\S+) after (\S+) host (\S+)", r.stdout)
    assert y
    before, stale, after, host = (float(y.group(k)) for k in range(1, 5))
    assert stale == before                           # not uploaded yet
    assert after != before and after == host


def test_data_change_and_misuse(lib, data):
    import smcmc_b200
    ev = uws.gauss_template(50000, seed=4)
    eng = engine(lib, "user_gauss_weighted_bind", ev, 2)
    pts = gauss_points(7, seed=3)
    before = eng.eval(pts)
    new = data[1][::-1].copy()
    assert lib.user_weighted_sync(uws.GAUSS, eng.h, new.ctypes.data) == 0
    after = eng.eval(pts)
    assert np.all(after != before)
    uws.set_gauss_data(lib, new)
    assert np.array_equal(after, uws.host(lib, uws.GAUSS, ev, pts)[0])
    uws.set_gauss_data(lib, data[1])

    bare = smcmc_b200.Engine(smcmc_b200.LLH_USER, 2, 4, seed=1)
    assert lib.user_gauss_weighted_bind_without_sample(bare.h) == 1
    assert b"no event sample" in lib.user_weighted_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        bare.bind_user_events(lib, "user_gauss_weighted_bind", np.zeros(10, np.float32))
    assert b"sizeof(Event)" in lib.user_weighted_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        bare.eval(np.zeros((1, 2)))                  # nothing registered
    bare.bind_user_events(lib, "user_gauss_weighted_bind", uws.gauss_template(0))
    empty = np.zeros(40)
    assert uws.same_bits(uws.device_sums(lib, uws.GAUSS, bare, np.array([[1.0, 2.0]]))[0], empty)
    assert np.array_equal(bare.eval(np.array([[1.0, 2.0]])),
                          uws.host(lib, uws.GAUSS, uws.gauss_template(0), np.array([[1.0, 2.0]]))[0])
