"""Shared by tests/test_user_events.py, tests/test_gpu_user_events.py and
scripts/user_event_bench.py: builds of the event functors of
tests/cpp/user_events.cuh and the numpy layouts of their Event records."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
CPP = os.path.join(ROOT, "tests", "cpp")
LIBDIR = os.path.join(ROOT, "root-simple-mcmc_b200", "smcmc_b200")
NVCC_FLAGS = ["-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false",
              "-Xcompiler", "-ffp-contract=off", "-I", INCLUDE, "-I", CPP]

GAUSS_DTYPE = np.dtype([("v", np.float64)])
EVENT12_DTYPE = np.dtype([("v", np.float32), ("w", np.float32), ("k", np.int32)])
EVENT128_DTYPE = np.dtype([("v", np.float64, 16)])
UNBINNED_DTYPE = np.dtype([("logSigma", np.float64), ("dLog", np.float64), ("nomLog", np.float64),
                           ("tag", np.int32), ("pad", np.int32)])
# kind argument of user_events_host, bind symbol
KINDS = {"gauss": (0, GAUSS_DTYPE), "gauss12": (1, EVENT12_DTYPE), "gauss128": (2, EVENT128_DTYPE),
         "unbinned": (3, UNBINNED_DTYPE)}


def build_library(outdir):
    """tests/cpp/user_events_lib.cu -> outdir/libuser_events.so, loaded."""
    so = os.path.join(outdir, "libuser_events.so")
    subprocess.run(["nvcc"] + NVCC_FLAGS + ["-Xcompiler", "-fPIC", "-shared", "-o", so,
                                            os.path.join(CPP, "user_events_lib.cu"), "-L", LIBDIR, "-lsmcmc_b200",
                                            "-Xlinker", "-rpath," + LIBDIR], check=True)
    lib = ctypes.CDLL(so)
    lib.user_events_host.restype = ctypes.c_int
    lib.user_events_host.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_void_p]
    lib.user_event_chunk.restype = ctypes.c_int64
    lib.user_event_chunk.argtypes = [ctypes.c_int64]
    lib.user_portable_log.restype = ctypes.c_double
    lib.user_portable_log.argtypes = [ctypes.c_double]
    lib.user_events_error.restype = ctypes.c_char_p
    lib.user_gauss_bind_without_sample.restype = ctypes.c_int
    lib.user_gauss_bind_without_sample.argtypes = [ctypes.c_void_p]
    return lib


def host_values(lib, kind, events, x):
    """EventLikelihoodHost at every row of x."""
    code, dtype = KINDS[kind]
    ev = np.ascontiguousarray(events, dtype=dtype)
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros(x.shape[0])
    rc = lib.user_events_host(code, ev.ctypes.data if len(ev) else None, len(ev), x.ctypes.data, x.shape[0],
                              x.shape[1], out.ctypes.data)
    assert rc == 0
    return out


def gauss_events(n, mean=3.0, sigma=2.0, seed=1):
    ev = np.zeros(n, GAUSS_DTYPE)
    ev["v"] = np.random.default_rng(seed).normal(mean, sigma, n)
    return ev


def unbinned_events(events):
    """The host preparation of UnbinnedEvents from smcmc_event records: the
    per-event corrections that SMCMC_LLH_UNBINNED computes at upload."""
    out = np.zeros(len(events), UNBINNED_DTYPE)
    with np.errstate(invalid="ignore", divide="ignore"):
        nom = np.log(events["TrueMass"])
        nom_sigma = np.log(events["TrueMass"] + events["TrueMassSigma"]) - nom
        out["dLog"] = np.log(events["Mass"]) - nom
        out["logSigma"] = out["dLog"] / nom_sigma
    out["nomLog"] = nom
    out["tag"] = events["MuDk"] > 0
    return out
