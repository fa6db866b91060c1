"""Shared by tests/test_user_weighted.py, tests/test_gpu_user_weighted.py and
scripts/user_weighted_bench.py: builds of the weighted binned functors of
tests/cpp/user_weighted.cuh, the numpy layouts of their Event records, and a
numpy statement of the documented summation order."""
import ctypes
import os
import subprocess

import numpy as np

from user_events_support import CPP, LIBDIR, NVCC_FLAGS

GAUSS, FAKE, RAW = 0, 1, 2           # kind argument of the library's entry points
BINS = {GAUSS: 40, FAKE: 150, RAW: 60}
GAUSS_DTYPE = np.dtype([("u", np.float64)])
RAW_DTYPE = np.dtype([("bin", np.int32), ("pad", np.int32), ("w", np.float64)])
FAKE_DTYPE = np.dtype([("logSigma", np.float64), ("dLog", np.float64), ("nomLog", np.float64),
                       ("sep", np.float64), ("cls", np.int32), ("dataBin", np.int32)])
GAUSS_LO, GAUSS_HI = -7.0, 13.0       # GaussWeighted's bins over [-7, 13)

_p = ctypes.c_void_p


def build_library(outdir):
    """tests/cpp/user_weighted_lib.cu -> outdir/libuser_weighted.so, loaded."""
    so = os.path.join(outdir, "libuser_weighted.so")
    subprocess.run(["nvcc"] + NVCC_FLAGS + ["-Xcompiler", "-fPIC", "-shared", "-o", so,
                                            os.path.join(CPP, "user_weighted_lib.cu"), "-L", LIBDIR, "-lsmcmc_b200",
                                            "-Xlinker", "-rpath," + LIBDIR], check=True)
    lib = ctypes.CDLL(so)
    lib.user_weighted_error.restype = ctypes.c_char_p
    lib.user_gauss_weighted_data.argtypes = [_p]
    lib.user_fake_weighted_data.argtypes = [_p, ctypes.c_double]
    lib.user_weighted_sync.argtypes = [ctypes.c_int, _p, _p]
    lib.user_weighted_sums.argtypes = [ctypes.c_int, _p, _p, ctypes.c_int, ctypes.c_int, _p]
    lib.user_weighted_host.argtypes = [ctypes.c_int, _p, ctypes.c_int64, _p, ctypes.c_int, ctypes.c_int, _p, _p]
    lib.user_fake_weighted_events.argtypes = [_p, ctypes.c_int64, _p]
    lib.user_weighted_chunk.restype = ctypes.c_int64
    lib.user_weighted_chunk.argtypes = [ctypes.c_int64]
    lib.user_weighted_shape.argtypes = [ctypes.c_int, _p, _p]
    lib.user_gauss_weighted_bind_without_sample.argtypes = [_p]
    return lib


def set_gauss_data(lib, data):
    d = np.ascontiguousarray(data, dtype=np.float64)
    assert d.shape == (40,)
    lib.user_gauss_weighted_data(d.ctypes.data)


def set_fake_data(lib, data150, exposure):
    d = np.ascontiguousarray(data150, dtype=np.float64)
    assert d.shape == (150,)
    lib.user_fake_weighted_data(d.ctypes.data, float(exposure))


def host(lib, kind, events, x):
    """(WeightedBinnedLikelihoodHost, WeightedSumsHost) at every row of x."""
    ev = np.ascontiguousarray(events)
    x = np.ascontiguousarray(x, dtype=np.float64)
    values = np.zeros(x.shape[0])
    sums = np.zeros((x.shape[0], BINS[kind]))
    assert lib.user_weighted_host(kind, ev.ctypes.data if len(ev) else None, len(ev), x.ctypes.data, x.shape[0],
                                  x.shape[1], values.ctypes.data, sums.ctypes.data) == 0
    return values, sums


def device_sums(lib, kind, eng, x):
    """WeightedBinnedBinding::Sums of the functor bound to eng."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros((x.shape[0], BINS[kind]))
    rc = lib.user_weighted_sums(kind, eng.h, x.ctypes.data, x.shape[0], x.shape[1], out.ctypes.data)
    assert rc == 0, lib.user_weighted_error()
    return out


def same_bits(a, b):
    """Equal bit for bit, -0.0 and 0.0 apart; any NaN equals any NaN (the host and
    the device need not produce the same NaN payload)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    return np.array_equal(np.where(np.isnan(a), 0.0, a).view(np.uint64), np.where(np.isnan(b), 0.0, b).view(np.uint64))


def ordered_sums(bins, weights, nbins, chunk):
    """The documented order in numpy: per chunk of `chunk` events, each bin's sum
    starts at 0.0 and adds the weights of its events in event order (np.bincount
    accumulates sequentially); the chunk sums are added in chunk order from 0.0.
    Events whose bin is outside [0, nbins) are dropped before their weight is
    looked at."""
    total = np.zeros(nbins)
    for first in range(0, len(bins), chunk):
        b, w = bins[first:first + chunk], weights[first:first + chunk]
        keep = (b >= 0) & (b < nbins)
        total = total + np.bincount(b[keep], weights=w[keep], minlength=nbins)
    return total


def gauss_template(n, seed=1):
    """n flat template values over GaussWeighted's range."""
    ev = np.zeros(n, GAUSS_DTYPE)
    ev["u"] = np.random.default_rng(seed).uniform(GAUSS_LO, GAUSS_HI, n)
    return ev


def fake_events(lib, events):
    """FakeWeighted::PrepareEvent of smcmc_event records, on the host."""
    ev = np.ascontiguousarray(events)
    out = np.zeros(len(ev), FAKE_DTYPE)
    lib.user_fake_weighted_events(ev.ctypes.data, len(ev), out.ctypes.data)
    return out


# Bin values outside RawWeighted's [0, 60): -1, -5, INT_MIN, kBins, kBins + 1, INT_MAX
RAW_OUTSIDE = [-1, -5, -2 ** 31, 60, 61, 2 ** 31 - 1]


def raw_events(n, seed=0):
    """n RawWeighted events: about a third carry a bin of RAW_OUTSIDE with a NaN,
    inf or -inf weight, which must never be added; the rest a bin in [0, 60), the
    first and the last over-represented, with finite weights over twelve orders of
    magnitude and both signs, so that the order of summation shows in the sums."""
    rng = np.random.default_rng(seed)
    ev = np.zeros(n, RAW_DTYPE)
    pick = rng.integers(0, 9, n)
    inside = np.where(pick == 6, 0, np.where(pick == 7, 59, rng.integers(0, 60, n)))
    outside = np.array(RAW_OUTSIDE, np.int64)[rng.integers(0, 6, n)]
    cut = pick < 3
    ev["bin"] = np.where(cut, outside, inside).astype(np.int32)
    w = rng.choice([-1.0, 1.0], n) * 10.0 ** rng.uniform(-6, 6, n)
    ev["w"] = np.where(cut, np.array([np.nan, np.inf, -np.inf])[rng.integers(0, 3, n)], w)
    return ev
