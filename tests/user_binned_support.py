"""Shared by tests/test_user_binned.py, tests/test_gpu_user_binned.py and
scripts/user_binned_bench.py: builds of the binned functors of
tests/cpp/user_binned.cuh and the numpy layouts of their Event records."""
import ctypes
import os
import subprocess

import numpy as np

from user_events_support import CPP, LIBDIR, NVCC_FLAGS

GAUSS, FAKE, RAW = 0, 1, 2           # kind argument of the library's entry points
BINS = {GAUSS: 40, FAKE: 300, RAW: 100}
RAW_DTYPE = np.dtype([("bin", np.int32), ("pad", np.int32)])
GAUSS_DTYPE = np.dtype([("z", np.float64)])
FAKE_DTYPE = np.dtype([("logSigma", np.float64), ("dLog", np.float64), ("nomLog", np.float64),
                       ("sep", np.float64), ("cls", np.int32), ("pad", np.int32)])
GAUSS_LO, GAUSS_WIDTH = -7.0, 0.5     # GaussBinned's bins over [-7, 13)

_p = ctypes.c_void_p


def build_library(outdir):
    """tests/cpp/user_binned_lib.cu -> outdir/libuser_binned.so, loaded."""
    so = os.path.join(outdir, "libuser_binned.so")
    subprocess.run(["nvcc"] + NVCC_FLAGS + ["-Xcompiler", "-fPIC", "-shared", "-o", so,
                                            os.path.join(CPP, "user_binned_lib.cu"), "-L", LIBDIR, "-lsmcmc_b200",
                                            "-Xlinker", "-rpath," + LIBDIR], check=True)
    lib = ctypes.CDLL(so)
    lib.user_binned_error.restype = ctypes.c_char_p
    lib.user_gauss_binned_data.argtypes = [_p]
    lib.user_fake_binned_data.argtypes = [_p, ctypes.c_double]
    lib.user_binned_sync.argtypes = [ctypes.c_int, _p, _p]
    lib.user_binned_counts.argtypes = [ctypes.c_int, _p, _p, ctypes.c_int, ctypes.c_int, _p]
    lib.user_binned_host.argtypes = [ctypes.c_int, _p, ctypes.c_int64, _p, ctypes.c_int, ctypes.c_int, _p, _p]
    lib.user_fake_binned_events.argtypes = [_p, ctypes.c_int64, _p]
    lib.user_binned_chunk.restype = ctypes.c_int64
    lib.user_binned_chunk.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.c_int64]
    lib.user_binned_shape.argtypes = [ctypes.c_int, _p, _p]
    lib.user_gauss_binned_bind_without_sample.argtypes = [_p]
    return lib


def set_gauss_data(lib, data):
    d = np.ascontiguousarray(data, dtype=np.float64)
    assert d.shape == (40,)
    lib.user_gauss_binned_data(d.ctypes.data)


def set_fake_data(lib, data150, exposure):
    d = np.ascontiguousarray(data150, dtype=np.float64)
    assert d.shape == (150,)
    lib.user_fake_binned_data(d.ctypes.data, float(exposure))


def host(lib, kind, events, x):
    """(BinnedLikelihoodHost, BinnedCountsHost) at every row of x."""
    ev = np.ascontiguousarray(events)
    x = np.ascontiguousarray(x, dtype=np.float64)
    values = np.zeros(x.shape[0])
    counts = np.zeros((x.shape[0], BINS[kind]), np.uint32)
    assert lib.user_binned_host(kind, ev.ctypes.data if len(ev) else None, len(ev), x.ctypes.data, x.shape[0],
                                x.shape[1], values.ctypes.data, counts.ctypes.data) == 0
    return values, counts


def device_counts(lib, kind, eng, x):
    """BinnedBinding::Counts of the functor bound to eng."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros((x.shape[0], BINS[kind]), np.uint32)
    rc = lib.user_binned_counts(kind, eng.h, x.ctypes.data, x.shape[0], x.shape[1], out.ctypes.data)
    assert rc == 0, lib.user_binned_error()
    return out


def gauss_template(n, seed=1):
    ev = np.zeros(n, GAUSS_DTYPE)
    ev["z"] = np.random.default_rng(seed).standard_normal(n)
    return ev


def gauss_bins(z, mu, sigma):
    """GaussBinned::Bin in numpy: the same operations, -1 outside the range."""
    u = (mu + sigma * z - GAUSS_LO) / GAUSS_WIDTH
    inside = (u >= 0.0) & (u < 40.0)
    return np.where(inside, np.floor(np.where(inside, u, 0.0)), -1).astype(np.int64)


def gauss_data(n, mean=3.0, sigma=2.0, seed=2):
    """A data sample and its histogram in GaussBinned's bins."""
    v = np.random.default_rng(seed).normal(mean, sigma, n)
    hist = np.histogram(v, bins=40, range=(GAUSS_LO, GAUSS_LO + 40 * GAUSS_WIDTH))[0].astype(np.float64)
    return v, hist


def fake_events(lib, events):
    """FakeBinned::PrepareEvent of smcmc_event records, on the host."""
    ev = np.ascontiguousarray(events)
    out = np.zeros(len(ev), FAKE_DTYPE)
    lib.user_fake_binned_events(ev.ctypes.data, len(ev), out.ctypes.data)
    return out


# Bin values outside RawBinned's [0, 100): -1, -5, INT_MIN, kBins, kBins + 1, INT_MAX
RAW_OUTSIDE = [-1, -5, -2 ** 31, 100, 101, 2 ** 31 - 1]


def raw_events(n, seed=0):
    """n RawBinned events: about two thirds carry a value of RAW_OUTSIDE, the rest a
    bin in [0, 100) with the first and the last bin over-represented.  Returns the
    events and the counts a correct Bin guard gives."""
    rng = np.random.default_rng(seed)
    ev = np.zeros(n, RAW_DTYPE)
    pick = rng.integers(0, 9, n)
    inside = np.where(pick == 6, 0, np.where(pick == 7, 99, rng.integers(0, 100, n)))
    outside = np.array(RAW_OUTSIDE, np.int64)[np.minimum(pick, 5)]
    ev["bin"] = np.where(pick >= 6, inside, outside).astype(np.int32)
    want = np.bincount(ev["bin"][(ev["bin"] >= 0) & (ev["bin"] < 100)], minlength=100).astype(np.uint32)
    return ev, want
