"""User BINNED event functors on the device (include/smcmc_device_functor.cuh:
kBinnedPairs, kBinnedFinish, BinnedBinding).  The functors (tests/cpp/user_binned.cuh)
are compiled by nvcc in a user translation unit; libsmcmc_b200 has no kernel for
them.  Checks: device counts and values equal the host restatement bit for bit,
whatever else is evaluated in the same call; a Bin outside [0, kBins) is not
counted; no 16-bit counter overflows; the
FAKE likelihood restated as a binned functor counts exactly what the built-in
kernel counts and its chains follow the built-in's; a template fit finds the
sample's mean and width; the C++ mirror reproduces a Python-bound chain; data
changes reach the device; misuse raises."""
import os
import re
import subprocess

import numpy as np
import pytest

import user_binned_support as ubs
import user_events_support as ues

pytestmark = pytest.mark.gpu

NS = [0, 1, 127, 128, 129, 65535, 65536, 65537, 10 ** 6]
MS = [1, 5, 128, 129, 1000]


@pytest.fixture(scope="module")
def data():
    return ubs.gauss_data(10000, seed=2)


@pytest.fixture(scope="module")
def lib(tmp_path_factory, data):
    lib = ubs.build_library(str(tmp_path_factory.mktemp("user_binned")))
    ubs.set_gauss_data(lib, data[1])
    return lib


@pytest.fixture(scope="module")
def program(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("cpp") / "user_binned")
    subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-o", exe, os.path.join(ues.CPP, "user_binned.cu"), "-L", ues.LIBDIR,
                                                "-lsmcmc_b200", "-Xlinker", "-rpath," + ues.LIBDIR], check=True)
    return exe


def engine(lib, symbol, events, dim, chains=4, seed=1, chain_offset=0):
    import smcmc_b200
    eng = smcmc_b200.Engine(smcmc_b200.LLH_USER, dim, chains, seed=seed, chain_offset=chain_offset)
    eng.bind_user_events(lib, symbol, events)
    return eng


def gauss_points(m, seed=0):
    return np.random.default_rng(seed).uniform([2.0, 1.0], [4.0, 3.0], (m, 2))


@pytest.mark.parametrize("n", NS)
def test_gauss_equals_the_host_restatement_bit_for_bit(lib, n):
    ev = ubs.gauss_template(n, seed=n + 1)
    eng = engine(lib, "user_gauss_binned_bind", ev, 2)
    for m in MS:
        pts = gauss_points(m, seed=m)
        values, counts = ubs.host(lib, ubs.GAUSS, ev, pts)
        assert np.array_equal(ubs.device_counts(lib, ubs.GAUSS, eng, pts), counts), m
        assert np.array_equal(eng.eval(pts), values), m


@pytest.mark.parametrize("n", [9, 1000, 70000])
def test_bins_outside_0_to_kbins_are_not_counted(lib, n):
    """RawBinned's Bin is a value carried by the event: -1, -5, INT_MIN, kBins,
    kBins + 1 and INT_MAX must not reach a counter (the kernel's guard keeps them out
    of the shared-memory counters of other bins and points); bins 0 and kBins - 1 are
    counted.  Two threads per point in kBinnedPairs; 70 000 events are two chunks."""
    ev, want = ubs.raw_events(n, seed=n)
    if n == 9:
        ev["bin"] = ubs.RAW_OUTSIDE + [0, 99, 99]
        want = np.zeros(100, np.uint32)
        want[0], want[99] = 1, 2
    eng = engine(lib, "user_raw_binned_bind", ev, 1)
    for m in (1, 129, 300):
        pts = np.arange(1.0, m + 1.0).reshape(m, 1)
        values, counts = ubs.host(lib, ubs.RAW, ev, pts)
        assert np.array_equal(counts, np.tile(want, (m, 1)))
        assert np.array_equal(ubs.device_counts(lib, ubs.RAW, eng, pts), counts), m
        assert np.array_equal(eng.eval(pts), values), m


def test_no_16_bit_overflow(lib):
    """200 000 events in one bin at every point: chunks stay below 65536 events, so
    no half-word carries into its partner (points p and p + 64 share a word)."""
    ev = np.zeros(200000, ubs.GAUSS_DTYPE)           # z = 0: every event at mu
    eng = engine(lib, "user_gauss_binned_bind", ev, 2)
    pts = np.tile([3.0, 2.0], (200, 1))
    pts[100:] = [4.6, 1.0]                            # bin 23 for points 100..199
    counts = ubs.device_counts(lib, ubs.GAUSS, eng, pts)
    want = np.zeros((200, 40), np.uint32)
    want[:100, 20] = 200000
    want[100:, 23] = 200000
    assert np.array_equal(counts, want)
    assert np.array_equal(eng.eval(pts), ubs.host(lib, ubs.GAUSS, ev, pts)[0])


def test_a_points_value_does_not_depend_on_the_batch(lib):
    ev = ubs.gauss_template(300000, seed=5)
    eng = engine(lib, "user_gauss_binned_bind", ev, 2)
    pts = gauss_points(1000, seed=6)
    full = eng.eval(pts)
    full_counts = ubs.device_counts(lib, ubs.GAUSS, eng, pts)
    for i in (0, 1, 63, 64, 127, 128, 500, 999):
        assert eng.eval(pts[i:i + 1])[0] == full[i]
        assert np.array_equal(ubs.device_counts(lib, ubs.GAUSS, eng, pts[i:i + 1])[0], full_counts[i])
    assert np.array_equal(eng.eval(pts[::-1]), full[::-1])
    assert np.array_equal(ubs.device_counts(lib, ubs.GAUSS, eng, pts[::-1]), full_counts[::-1])


# ---------------------------------------------------------------------------
# FakeBinned against the built-in SMCMC_LLH_FAKE
# ---------------------------------------------------------------------------
def c2_sample():
    """bench.py's C2 sample: 10^6 MC events and the data histograms."""
    from smcmc_b200 import synth
    n = 10 ** 6
    signal = n // 3 + (1 if n % 3 else 0)
    return synth.make_mc_sample(signal, n - signal, seed=2), synth.make_data_histograms(33334, 33334, seed=2)


@pytest.fixture(scope="module")
def fake_pair(lib):
    import smcmc_b200
    from smcmc_b200 import synth
    events, data = c2_sample()
    chains = 256
    builtin = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, chains, seed=3)
    builtin.set_fake_events(events)
    exposure = synth.exposure_ratio(builtin, data)
    builtin.set_fake_data(data, exposure)
    ubs.set_fake_data(lib, data, exposure)
    user = engine(lib, "user_fake_binned_bind", ubs.fake_events(lib, events), 9, chains, seed=3)
    return user, builtin


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
    return np.concatenate([start, wide, extreme, bad])


def test_fake_binned_counts_equal_the_builtin(lib, fake_pair):
    user, builtin = fake_pair
    pts = fake_points()
    assert pts.shape == (256, 9)
    got = ubs.device_counts(lib, ubs.FAKE, user, pts)
    want = builtin.fake_counts(pts)[:, :300]
    assert np.array_equal(got, want)
    assert got[:64].sum() > 0


def test_fake_binned_values_match_the_builtin(fake_pair):
    user, builtin = fake_pair
    pts = fake_points()
    got, want = user.eval(pts), builtin.eval(pts)
    assert np.array_equal(np.isfinite(got), np.isfinite(want))
    fin = np.isfinite(want)
    assert fin[:192].all()
    assert np.max(np.abs(got[fin] / want[fin] - 1.0)) < 1e-9


def test_fake_binned_metropolis_follows_the_builtin(fake_pair):
    user, builtin = fake_pair
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
    """10^4 data events from N(3, 2), a template of 10^6 standard-normal events,
    4096 chains with pooled adaptation: the posterior of (mu, sigma) is centred on
    the sample's mean and width, with widths s/sqrt(N) and s/sqrt(2N)."""
    from smcmc_b200 import binding
    v, _ = data
    E, N = 4096, len(v)
    eng = engine(lib, "user_gauss_binned_bind", ubs.gauss_template(10 ** 6, seed=11), 2, E, seed=9)
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
    """sMCMC::TSimpleMCMC<GaussBinned> with a TTree and events set before Start: the
    chain of a Python-bound engine with the same seed and chain index, accept for
    accept and bit for bit; then a data change through SyncLikelihood."""
    ev = ubs.gauss_template(20000, seed=21)
    tpath, dpath = str(tmp_path / "template.bin"), str(tmp_path / "data.bin")
    ev["z"].tofile(tpath)
    data[1].tofile(dpath)
    steps = 200
    r = subprocess.run([program, tpath, dpath, "7", "3", str(steps)], capture_output=True, text=True, check=True)
    s = re.search(r"start llh (\S+) host (\S+)", r.stdout)
    assert s and float(s.group(1)) == float(s.group(2))
    rows = re.findall(r"step (\d+) acc (\d) llh (\S+) x (\S+) (\S+)", r.stdout)
    assert len(rows) == steps
    eng = engine(lib, "user_gauss_binned_bind", ev, 2, 1, seed=7, chain_offset=3)
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
    ev = ubs.gauss_template(50000, seed=4)
    eng = engine(lib, "user_gauss_binned_bind", ev, 2)
    pts = gauss_points(7, seed=3)
    before = eng.eval(pts)
    new = data[1][::-1].copy()
    assert lib.user_binned_sync(ubs.GAUSS, eng.h, new.ctypes.data) == 0
    after = eng.eval(pts)
    assert np.all(after != before)
    ubs.set_gauss_data(lib, new)
    assert np.array_equal(after, ubs.host(lib, ubs.GAUSS, ev, pts)[0])
    ubs.set_gauss_data(lib, data[1])

    bare = smcmc_b200.Engine(smcmc_b200.LLH_USER, 2, 4, seed=1)
    assert lib.user_gauss_binned_bind_without_sample(bare.h) == 1
    assert b"no event sample" in lib.user_binned_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        bare.bind_user_events(lib, "user_gauss_binned_bind", np.zeros(10, np.float32))
    assert b"sizeof(Event)" in lib.user_binned_error()
    with pytest.raises(smcmc_b200.SmcmcError):
        bare.eval(np.zeros((1, 2)))                  # nothing registered
    bare.bind_user_events(lib, "user_gauss_binned_bind", ubs.gauss_template(0))
    empty = np.zeros(40, np.uint32)
    assert np.array_equal(ubs.device_counts(lib, ubs.GAUSS, bare, np.array([[1.0, 2.0]]))[0], empty)
    assert np.array_equal(bare.eval(np.array([[1.0, 2.0]])), ubs.host(lib, ubs.GAUSS, ubs.gauss_template(0),
                                                                      np.array([[1.0, 2.0]]))[0])
