"""The pair kernel's tile skip (DESIGN.md section 4.1): a warp of 32 chains
skips an event tile when every event of it is above the mass cut for the whole
box of its chains' parameters.  A skipped pair must be one the FP64 arithmetic
cuts, and the counts must not depend on the skip or on the event order."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CHAINS, EVENTS = 4096, 1_000_000


def bench_sample(n):
    from smcmc_b200 import synth
    signal = n // 3 + (1 if n % 3 else 0)
    events = synth.make_mc_sample(signal, n - signal, seed=2)
    data = synth.make_data_histograms(33334, 33334, seed=2)
    return events, data


def make_engine(events, data, chains, monkeypatch=None, no_skip=False):
    import smcmc_b200
    from smcmc_b200 import synth
    if no_skip:
        monkeypatch.setenv("SMCMC_FAKE_NO_SKIP", "1")
    eng = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, chains, seed=3)
    if no_skip:
        monkeypatch.delenv("SMCMC_FAKE_NO_SKIP")
    eng.set_fake_events(events)
    eng.set_fake_data(data, synth.exposure_ratio(eng, data))
    return eng


def start_points(chains):
    """bench.py's start points: every parameter ~ U(-1, 1)."""
    return np.stack([np.random.default_rng([3, c]).uniform(-1.0, 1.0, 9) for c in range(chains)])


@pytest.fixture(scope="module")
def full():
    events, data = bench_sample(EVENTS)
    return make_engine(events, data, CHAINS)


def test_skip_never_drops_a_counted_pair(full):
    rng = np.random.default_rng(8)
    wide = rng.normal(0, 10, (CHAINS, 9))
    extreme = rng.normal(0, 60, (CHAINS, 9))
    extreme[5, 3] = -900.0
    extreme[70, 4] = 1e5
    extreme[100, 2] = np.nan
    extreme[200, 6] = np.inf
    extreme[300, 3] = np.inf
    for x in (start_points(CHAINS), wide, extreme):
        tested, skipped, bad = full.fake_skip_check(x)
        assert bad == 0
        assert skipped <= tested


def test_skip_is_effective_at_the_start_points(full):
    tested, skipped, bad = full.fake_skip_check(start_points(CHAINS))
    assert bad == 0
    # about a quarter of all pairs lie in tiles above the cut for a box of p in [-1, 1]
    assert skipped > 0.3 * tested
    assert skipped * 128 * 32 > 0.15 * CHAINS * EVENTS


@pytest.fixture(scope="module")
def sample():
    return bench_sample(200_000)


def ragged_points(chains):
    x = np.concatenate([start_points(chains - 40), np.random.default_rng(2).normal(0, 3, (40, 9))])
    x[7, 2] = 1e3            # out of the filter's range: force
    x[40, 4] = np.nan        # force
    x[chains - 3, 3] = -50.0
    return x


@pytest.mark.parametrize("chains", [300, 1000])
def test_counts_equal_without_skip(sample, chains, monkeypatch):
    events, data = sample
    x = ragged_points(chains)
    skip = make_engine(events, data, chains)
    plain = make_engine(events, data, chains, monkeypatch, no_skip=True)
    tested, skipped, bad = skip.fake_skip_check(x)
    assert skipped > 0 and bad == 0
    assert plain.fake_skip_check(x) == (0, 0, 0)
    assert np.array_equal(skip.fake_counts(x), plain.fake_counts(x))
    assert np.array_equal(skip.eval(x), plain.eval(x), equal_nan=True)


def test_event_order_does_not_change_the_counts(sample):
    events, data = sample
    chains = 300
    x = ragged_points(chains)
    a = make_engine(events, data, chains)
    b = make_engine(np.random.default_rng(4).permutation(events), data, chains)
    assert np.array_equal(a.fake_counts(x), b.fake_counts(x))
