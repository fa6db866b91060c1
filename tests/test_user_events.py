"""Event functors (include/smcmc_device_functor.cuh) without a GPU: the host
restatement of the summation order, the chunk length, and the compile-time
checks on the Event record.  The functors are compiled by nvcc in a user
translation unit (tests/cpp/user_events_lib.cu); only host code runs here."""
import math
import os
import subprocess

import numpy as np
import pytest

import user_events_support as ues


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    import smcmc_b200
    if not os.path.exists(smcmc_b200.library_path()):
        smcmc_b200.build_library()
    return ues.build_library(str(tmp_path_factory.mktemp("user_events")))


def chunks(lib, n):
    """(first, count) of every chunk in the documented order."""
    c = lib.user_event_chunk(n)
    return [(f, min(c, n - f)) for f in range(0, n, c)]


def gauss_numpy(lib, v, x):
    """GaussEvents in numpy, in the documented order: per-chunk sequential sums
    (np.add.accumulate adds left to right), chunk sums added in order, then
    Finish with the functor's own logarithm."""
    mu, sigma = x
    k = -0.5 / (sigma * sigma)
    terms = k * ((v - mu) * (v - mu))
    s = 0.0
    for f, c in chunks(lib, len(v)):
        s += np.add.accumulate(terms[f:f + c])[-1]
    return s - float(len(v)) * lib.user_portable_log(sigma)


def test_chunk_length_depends_on_the_sample_size_only(lib):
    c = [lib.user_event_chunk(n) for n in (0, 1, 1000, 10 ** 5, 10 ** 6, 10 ** 7, 10 ** 9)]
    assert all(x % 128 == 0 for x in c)
    assert c[0] == c[1] == c[2] == 1024
    assert c[-1] == 32768
    assert c == sorted(c)


N_CMIN = 1024        # the chunk length of small samples


@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, N_CMIN - 1, N_CMIN, N_CMIN + 1, 10 ** 6])
def test_chunks_cover_every_event_once_in_order(lib, n):
    parts = chunks(lib, n)
    covered = np.concatenate([np.arange(f, f + c) for f, c in parts]) if parts else np.zeros(0, int)
    assert np.array_equal(covered, np.arange(n))
    assert all(c > 0 for _, c in parts)
    assert len(parts) == (n + lib.user_event_chunk(n) - 1) // lib.user_event_chunk(n)


@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, N_CMIN - 1, N_CMIN, N_CMIN + 1, 10 ** 6])
def test_host_restatement_equals_numpy(lib, n):
    ev = ues.gauss_events(n, seed=n)
    x = np.array([[3.0, 2.0], [2.9, 1.7], [-1.0, 5.5]])
    host = ues.host_values(lib, "gauss", ev, x)
    want = np.array([gauss_numpy(lib, ev["v"], p) for p in x])
    assert np.array_equal(host, want)


def test_order_is_not_sequential_for_large_samples(lib):
    """At 10^6 events the chunked order differs from one sequential sum in the last
    bits for some points -- the test above pins the chunked one."""
    ev = ues.gauss_events(10 ** 6, seed=4)
    x = np.random.default_rng(2).uniform([2.0, 1.0], [4.0, 3.0], (20, 2))
    host = ues.host_values(lib, "gauss", ev, x)
    seq = np.array([np.add.accumulate(-0.5 / (s * s) * ((ev["v"] - m) * (ev["v"] - m)))[-1]
                    - 1e6 * lib.user_portable_log(s) for m, s in x])
    assert np.allclose(host, seq, rtol=1e-13, atol=0)
    assert not np.array_equal(host, seq)


def test_portable_log(lib):
    xs = np.concatenate([np.geomspace(1e-300, 1e300, 4001), np.random.default_rng(1).uniform(0.1, 10, 4000)])
    got = np.array([lib.user_portable_log(x) for x in xs])
    want = np.log(xs)
    assert np.all(np.abs(got - want) <= 4e-16 * np.maximum(np.abs(want), 1e-300) + 1e-300)
    assert math.isnan(lib.user_portable_log(-1.0))
    assert lib.user_portable_log(0.0) == -math.inf
    assert lib.user_portable_log(1.0) == 0.0


def test_awkward_event_sizes_on_the_host(lib):
    sizes = ctypes_sizes(lib)
    assert sizes == [8, 12, 128, 32]
    ev = np.zeros(300, ues.EVENT12_DTYPE)
    ev["v"] = np.linspace(0, 6, 300)
    ev["w"] = 0.25
    ev["k"] = np.arange(300) % 3
    got = ues.host_values(lib, "gauss12", ev, np.array([[3.0, 2.0]]))[0]
    t = -0.5 / 4.0 * ((ev["v"].astype(float) - 3.0) ** 2) + 0.25 * ev["k"]
    assert math.isclose(got, math.fsum(t) - 300 * math.log(2.0), rel_tol=1e-13)


def ctypes_sizes(lib):
    import ctypes
    out = (ctypes.c_int64 * 4)()
    assert lib.user_event_sizes(out) == 4
    return list(out)


def test_oversized_event_fails_to_compile(tmp_path):
    src = tmp_path / "big_event.cu"
    src.write_text("""
#include "smcmc_device_functor.cuh"
struct Big {
    struct Event { double v[18]; };
    struct Chain { double mu; };
    __host__ __device__ Chain Prepare(const double* x, int) const { Chain c; c.mu = x[0]; return c; }
    __host__ __device__ double Term(const Chain& c, const Event& e) const { return e.v[0] - c.mu; }
};
double f(const Big::Event* e, const double* x) { return smcmc_user::EventLikelihoodHost(Big(), e, 1, x, 1); }
""")
    r = subprocess.run(["nvcc"] + ues.NVCC_FLAGS + ["-c", "-o", str(tmp_path / "big_event.o"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode != 0
    assert "sizeof(F::Event) must be at most 128 bytes" in r.stdout + r.stderr
