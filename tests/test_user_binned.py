"""Binned event functors (include/smcmc_device_functor.cuh) without a GPU: the host
restatement of the counts, the bins that are not counted, the launcher's chunk
rule and the compile-time checks.  The functors are compiled by nvcc in a user
translation unit (tests/cpp/user_binned_lib.cu); only host code runs here."""
import os
import subprocess

import numpy as np
import pytest

import user_binned_support as ubs
import user_events_support as ues


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import smcmc_b200
    if not os.path.exists(smcmc_b200.library_path()):
        smcmc_b200.build_library()
    lib = ubs.build_library(str(tmp_path_factory.mktemp("user_binned")))
    ubs.set_gauss_data(lib, ubs.gauss_data(5000)[1])
    return lib


@pytest.mark.parametrize("n", [0, 1, 127, 129, 10 ** 5])
def test_gauss_counts_equal_a_numpy_histogram(lib, n):
    ev = ubs.gauss_template(n, seed=n)
    x = np.array([[3.0, 2.0], [2.9, 1.7], [-1.0, 5.5], [20.0, 1.0]])
    _, counts = ubs.host(lib, ubs.GAUSS, ev, x)
    for p, (mu, sigma) in enumerate(x):
        b = ubs.gauss_bins(ev["z"], mu, sigma)
        want = np.bincount(b[b >= 0], minlength=40)
        assert np.array_equal(counts[p], want)


def test_gauss_bin_maps_values_outside_its_range_to_minus_one(lib):
    """GaussBinned's own rule: a value below the range, at its upper edge, far above
    it, infinite or NaN gives Bin = -1, so only the value inside is counted."""
    ev = np.zeros(6, ubs.GAUSS_DTYPE)
    # at mu = 0, sigma = 1: u = (z + 7) / 0.5
    ev["z"] = [-7.5, 13.0, 1e300, np.inf, np.nan, 0.0]   # -1, 40, huge, inf, NaN, bin 14
    _, counts = ubs.host(lib, ubs.GAUSS, ev, np.array([[0.0, 1.0]]))
    want = np.zeros(40, np.uint32)
    want[14] = 1
    assert np.array_equal(counts[0], want)


@pytest.mark.parametrize("n", [1, 9, 1000, 70000])
def test_bins_outside_0_to_kbins_are_not_counted(lib, n):
    """RawBinned's Bin is a value carried by the event: -1, -5, INT_MIN, kBins,
    kBins + 1 and INT_MAX are not counted, bins 0 and kBins - 1 are."""
    ev, want = ubs.raw_events(n, seed=n)
    if n == 9:                                       # one of each, then the first and the last bin
        ev["bin"] = ubs.RAW_OUTSIDE + [0, 99, 99]
        want = np.zeros(100, np.uint32)
        want[0], want[99] = 1, 2
    assert n < 10 or want[0] > 0 and want[99] > 0 and want.sum() < n
    values, counts = ubs.host(lib, ubs.RAW, ev, np.array([[1.0], [2.0]]))
    assert np.array_equal(counts[0], want) and np.array_equal(counts[1], want)
    assert values[1] == 2.0 * values[0] == 2.0 * float(np.sum(np.arange(1, 101) * want.astype(float)))


def test_host_value_is_finish_over_the_counts(lib):
    ev = ubs.gauss_template(20000, seed=3)
    _, data = ubs.gauss_data(5000)
    x = np.array([[3.0, 2.0], [2.5, 1.5]])
    values, counts = ubs.host(lib, ubs.GAUSS, ev, x)
    for p in range(2):
        mu = np.maximum(counts[p] * (data.sum() / len(ev)), 0.001)
        want = np.sum(data * np.log(mu) - mu)
        assert abs(values[p] / want - 1.0) < 1e-13


def test_chunk_rule_stays_below_65536(lib):
    rng = np.random.default_rng(1)
    ns = [0, 1, 127, 128, 65535, 65536, 65537, 10 ** 6, 10 ** 8, 2 ** 40] + list(rng.integers(0, 10 ** 9, 200))
    for n in ns:
        for tiles in (1, 2, 8, 32, 1000, 100000):
            for slots in (1, 148, 296, 1184, 4736):
                c = lib.user_binned_chunk(int(n), tiles, slots)
                assert 128 <= c <= 65535 and c % 128 == 0, (n, tiles, slots, c)


def test_chunk_rule_fills_whole_waves(lib):
    """C2 at 4096 chains (32 point tiles) on 148 SMs x 2 CTAs: the grid is at most
    two waves, and the chunk is the shortest that fits them."""
    n, tiles, slots = 10 ** 6, 32, 296
    c = lib.user_binned_chunk(n, tiles, slots)
    grid = -(-n // c) * tiles
    assert grid <= 2 * slots
    assert -(-n // (c - 128)) * tiles > 2 * slots


def compile_error(tmp_path, body, name):
    src = tmp_path / (name + ".cu")
    src.write_text('#include "smcmc_device_functor.cuh"\n#include "TSimpleHMC.H"\n' + body)
    r = subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / (name + ".o")), str(src)],
                       capture_output=True, text=True)
    assert r.returncode != 0
    return r.stdout + r.stderr


BINNED = """
struct B {
    struct Event { %s };
    struct Chain { double mu; };
    static constexpr int kBins = %d;
    __host__ __device__ Chain Prepare(const double* x, int) const { Chain c; c.mu = x[0]; return c; }
    __host__ __device__ %s Bin(const Chain& c, const Event& e) const { return (int)(c.mu + e.v[0]); }
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinCounts& k, int64_t) const { return k[0]; }
};
"""
USE = "double f(const B::Event* e, const double* x) { return smcmc_user::BinnedLikelihoodHost(B(), e, 1, x, 1); }\n"


@pytest.mark.parametrize("bins", [0, 513])
def test_bad_bin_count_fails_to_compile(tmp_path, bins):
    out = compile_error(tmp_path, BINNED % ("double v[1];", bins, "int") + USE, "bins%d" % bins)
    assert "F::kBins must be between 1 and 512" in out


def test_oversized_binned_event_fails_to_compile(tmp_path):
    out = compile_error(tmp_path, BINNED % ("unsigned char v[129];", 40, "int") + USE, "big")
    assert "sizeof(F::Event) must be at most 128 bytes" in out


def test_bin_must_return_int(tmp_path):
    out = compile_error(tmp_path, BINNED % ("double v[1];", 40, "long") + USE, "long")
    assert "F::Bin(chain, event) must return int" in out


def test_hmc_refuses_a_binned_functor(tmp_path):
    src = '#include "user_binned.cuh"\n#include "TSimpleHMC.H"\nsMCMC::TSimpleHMC<GaussBinned, GaussBinned> hmc;\n'
    p = tmp_path / "hmc.cu"
    p.write_text(src)
    r = subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / "hmc.o"), str(p)],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "TSimpleHMC cannot sample a BINNED event functor" in r.stdout + r.stderr
