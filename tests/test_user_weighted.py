"""Weighted binned event functors (include/smcmc_device_functor.cuh) without a GPU:
the host restatement of the weighted sums against a numpy statement of the
documented order, cut events and non-finite weights, the chunk rule and the
compile-time checks.  The functors are compiled by nvcc in a user translation unit
(tests/cpp/user_weighted_lib.cu); only host code runs here."""
import subprocess

import numpy as np
import pytest

import user_weighted_support as uws
import user_events_support as ues


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import os
    import smcmc_b200
    if not os.path.exists(smcmc_b200.library_path()):
        smcmc_b200.build_library()
    return uws.build_library(str(tmp_path_factory.mktemp("user_weighted")))


def chunk_edges(lib):
    """N at, and one either side of, the first chunk boundaries and the point where
    the chunk starts to grow past its minimum."""
    c0 = lib.user_weighted_chunk(1)
    grow = 32 * c0                                   # the largest N of minimal chunks
    return sorted({k + d for k in (c0, 2 * c0, grow) for d in (-1, 0, 1)} |
                  {lib.user_weighted_chunk(grow + 1) + d for d in (-1, 0, 1)})


def test_chunk_rule_depends_on_n_only_and_covers_the_sample(lib):
    rng = np.random.default_rng(1)
    ns = [0, 1, 127, 128, 129, 1023, 1024, 1025, 32768, 32769, 10 ** 6, 10 ** 8, 2 ** 40] + \
        [int(v) for v in rng.integers(0, 10 ** 9, 300)]
    for n in ns:
        c = lib.user_weighted_chunk(n)
        assert c % 128 == 0 and c >= 1024, (n, c)
        chunks = -(-n // c)
        assert chunks <= 32, (n, c)
        assert chunks * c >= n and (chunks == 0 or (chunks - 1) * c < n), (n, c)
        assert lib.user_weighted_chunk(n) == c       # a function of n alone: no state, no device


@pytest.mark.parametrize("case", ["0", "1", "127", "128", "129", "edges", "1e6"])
def test_host_sums_follow_the_documented_order_bit_for_bit(lib, case):
    ns = chunk_edges(lib) if case == "edges" else [int(float(case))]
    x = np.array([[1.0], [3.0], [-0.5]])
    for n in ns:
        ev = uws.raw_events(n, seed=n)
        _, sums = uws.host(lib, uws.RAW, ev, x)
        chunk = lib.user_weighted_chunk(n)
        for p, scale in enumerate(x[:, 0]):
            want = uws.ordered_sums(ev["bin"].astype(np.int64), scale * ev["w"], 60, chunk)
            assert uws.same_bits(sums[p], want), (n, p)
            assert np.all(np.isfinite(sums[p])), (n, p)   # the NaN and inf weights are all on cut events
        if n == 10 ** 6:                              # the chunking shows: one pass in event order differs
            one = uws.ordered_sums(ev["bin"].astype(np.int64), ev["w"], 60, n)
            assert not uws.same_bits(sums[0], one)


def test_cut_weights_are_never_added(lib):
    """Every RawWeighted value outside [0, 60) with NaN, inf and -inf weights, then
    bins 0 and 59: only those two are summed."""
    ev = np.zeros(6 * 3 + 3, uws.RAW_DTYPE)
    ev["bin"][:18] = np.repeat(uws.RAW_OUTSIDE, 3)
    ev["w"][:18] = np.tile([np.nan, np.inf, -np.inf], 6)
    ev["bin"][18:] = [0, 59, 59]
    ev["w"][18:] = [0.25, 1.5, 2.0]
    values, sums = uws.host(lib, uws.RAW, ev, np.array([[1.0], [2.0]]))
    want = np.zeros(60)
    want[0], want[59] = 0.25, 3.5
    assert uws.same_bits(sums[0], want) and uws.same_bits(sums[1], 2 * want)
    assert values[0] == 0.25 + 60 * 3.5 and values[1] == 2 * values[0]


def test_an_in_range_nan_weight_poisons_only_its_bin(lib):
    ev = np.zeros(5, uws.RAW_DTYPE)
    ev["bin"] = [3, 3, 7, 7, 8]
    ev["w"] = [1.0, np.nan, 2.0, np.inf, -np.inf]
    values, sums = uws.host(lib, uws.RAW, ev, np.array([[1.0]]))
    assert np.isnan(sums[0, 3]) and sums[0, 7] == np.inf and sums[0, 8] == -np.inf
    others = np.delete(sums[0], [3, 7, 8])
    assert np.all(others == 0.0)
    assert np.isnan(values[0])


def test_gauss_weights_reproduce_the_normal_template(lib):
    """GaussWeighted's sums are an importance-sampled N(mu, sigma) histogram of the
    flat template: scaled by 1/N they approach the normal's bin probabilities."""
    from scipy.stats import norm
    n = 400000
    ev = uws.gauss_template(n, seed=3)
    x = np.array([[3.0, 2.0], [1.0, 0.7]])
    _, sums = uws.host(lib, uws.GAUSS, ev, x)
    edges = np.linspace(-7.0, 13.0, 41)
    for p, (mu, sigma) in enumerate(x):
        want = np.diff(norm.cdf(edges, mu, sigma))
        # the weights reach 20 / (sigma sqrt(2 pi)): a bin's sum / N scatters by up to 3e-3
        assert np.max(np.abs(sums[p] / n - want)) < 1.5e-2, p
        assert abs(sums[p].sum() / n - 1.0) < 2e-2


def test_gauss_host_value_is_finish_over_the_sums(lib):
    ev = uws.gauss_template(20000, seed=3)
    data = np.random.default_rng(2).poisson(200.0, 40).astype(np.float64)
    uws.set_gauss_data(lib, data)
    x = np.array([[3.0, 2.0], [2.5, 1.5]])
    values, sums = uws.host(lib, uws.GAUSS, ev, x)
    for p in range(2):
        mu = np.maximum(sums[p] * (data.sum() / len(ev)), 0.001)
        want = np.sum(data * np.log(mu) - mu)
        assert abs(values[p] / want - 1.0) < 1e-13


def test_fake_weighted_host_equals_the_port_fill(lib):
    """FakeWeighted's host sums and value against the oracle port's FillFake and
    EvalFake, on a small sample that also holds data-typed events (weight 1, bins
    that no parameter moves)."""
    from oracle import cpu_checkers as cc
    from smcmc_b200 import synth
    events, data = synth.fake_inputs(300, 300, 60, seed=4)
    events["Type"][::7] = -1                          # data-typed events mixed into the sample
    orc = cc.CpuChain("orc", cc.LLH_FAKE, 9, 1, 0)
    orc.set_fake(events, data, 1.7)
    uws.set_fake_data(lib, data, 1.7)
    prepared = uws.fake_events(lib, events)
    rng = np.random.default_rng(5)
    pts = np.concatenate([rng.uniform(-1, 1, (6, 9)), rng.normal(0, 10, (6, 9))])
    values, sums = uws.host(lib, uws.FAKE, prepared, pts)
    for p, x in enumerate(pts):
        want = orc.fake_hist(x)
        nz = want != 0
        assert np.array_equal(sums[p] != 0, nz), p
        assert np.max(np.abs(sums[p][nz] / want[nz] - 1.0), initial=0.0) < 1e-12, p
        assert abs(values[p] / orc.llh(x) - 1.0) < 1e-10, p


def compile_error(tmp_path, body, name):
    src = tmp_path / (name + ".cu")
    src.write_text('#include "smcmc_device_functor.cuh"\n#include "TSimpleHMC.H"\n' + body)
    r = subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / (name + ".o")), str(src)],
                       capture_output=True, text=True)
    assert r.returncode != 0
    return r.stdout + r.stderr


WEIGHTED = """
struct W {
    struct Event { double v[1]; };
    struct Chain { double mu; };
    static constexpr int kBins = %d;
    __host__ __device__ Chain Prepare(const double* x, int) const { Chain c; c.mu = x[0]; return c; }
    __host__ __device__ int Bin(const Chain& c, const Event& e) const { return (int)(c.mu + e.v[0]); }
    __host__ __device__ %s Weight(const Chain& c, const Event& e) const { return c.mu * e.v[0]; }
    __host__ __device__ double Finish(const Chain&, const smcmc_user::BinSums& s, int64_t) const { return s[0]; }
};
"""
USE = "double f(const W::Event* e, const double* x) { return smcmc_user::WeightedBinnedLikelihoodHost(W(), e, 1, x, 1); }\n"


def test_weighted_functor_compiles(tmp_path):
    src = tmp_path / "ok.cu"
    src.write_text('#include "smcmc_device_functor.cuh"\n' + WEIGHTED % (256, "double") + USE +
                   "static_assert(smcmc_user::IsWeightedBinnedFunctor<W>::value, \"\");\n")
    subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / "ok.o"), str(src)], check=True)


@pytest.mark.parametrize("bins", [0, 257])
def test_bad_weighted_bin_count_fails_to_compile(tmp_path, bins):
    out = compile_error(tmp_path, WEIGHTED % (bins, "double") + USE, "bins%d" % bins)
    assert "F::kBins of a weighted binned functor must be between 1 and 256" in out


def test_weight_must_return_double(tmp_path):
    out = compile_error(tmp_path, WEIGHTED % (40, "float") + USE, "float")
    assert "F::Weight(chain, event) must return double" in out


def test_hmc_refuses_a_weighted_functor(tmp_path):
    src = '#include "user_weighted.cuh"\n#include "TSimpleHMC.H"\nsMCMC::TSimpleHMC<GaussWeighted, GaussWeighted> hmc;\n'
    p = tmp_path / "hmc.cu"
    p.write_text(src)
    r = subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / "hmc.o"), str(p)],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "TSimpleHMC cannot sample a BINNED event functor" in r.stdout + r.stderr
