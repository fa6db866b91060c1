"""ctypes binding of the C ABI declared in include/smcmc_b200.h."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(os.path.dirname(HERE), "csrc")

LLH_UNIT_GAUSS, LLH_DUMMY, LLH_HORRIFIC, LLH_ASYM, LLH_FAKE, LLH_UNBINNED, LLH_HARD, LLH_FAKE2, LLH_USER = range(9)
DUMMY_EXACT, DUMMY_TENSOR = 0, 1

# smcmc_prop_field
(PROP_SIGMA, PROP_TARGET_ACCEPTANCE, PROP_ACCEPTANCE_WINDOW,
 PROP_ACCEPTANCE_RIGIDITY, PROP_ACCEPTANCE_DEWEIGHT, PROP_COVARIANCE_WINDOW,
 PROP_COVARIANCE_DEWEIGHT, PROP_COVARIANCE_FROZEN, PROP_COVARIANCE_TRIALS,
 PROP_CENTER_TRIALS, PROP_NEXT_UPDATE, PROP_MAX_CORRELATION,
 PROP_STEP_RMS_WINDOW, PROP_POOLED_EVERY, PROP_POOLED_TENSOR) = range(15)
PROP_KIND = 15
PROPOSAL_ADAPTIVE, PROPOSAL_VAAT = 0, 1

# smcmc_field: name -> (id, dtype, shape code)
_FIELDS = {
    "accepted": (0, np.float64, "En"), "proposed": (1, np.float64, "En"),
    "accepted_llh": (2, np.float64, "E"), "proposed_llh": (3, np.float64, "E"),
    "step_rms": (4, np.float64, "E"), "sigma": (5, np.float64, "E"),
    "acceptance": (6, np.float64, "E"), "acceptance_trials": (7, np.float64, "E"),
    "acceptance_rigidity": (8, np.float64, "E"), "trials": (9, np.int32, "E"),
    "successes": (10, np.int32, "E"), "next_update": (11, np.int32, "E"),
    "covariance_trials": (12, np.float64, "E"), "center_trials": (13, np.float64, "E"),
    "center": (14, np.float64, "En"), "covariance": (15, np.float64, "Et"),
    "covariance_trace": (16, np.float64, "E"), "decomposition": (17, np.float64, "Enn"),
    "total_steps": (18, np.int32, "E"), "llh_calls": (19, np.int32, "E"),
    "status": (20, np.int32, "E"), "sigma_trace": (21, np.float64, "E"),
    "covariance_window": (22, np.float64, "1"), "acceptance_window": (23, np.float64, "1"),
    "target_acceptance": (24, np.float64, "1"),
    "pooled_mean": (25, np.float64, "n"), "pooled_covariance": (26, np.float64, "t"),
    "pooled_decomposition": (27, np.float64, "nn"), "pooled_count": (28, np.float64, "1"),
    "vaat_sigma": (29, np.float64, "En"), "vaat_acceptance": (30, np.float64, "En"),
    "vaat_acceptance_trials": (31, np.int32, "En"), "vaat_last_index": (32, np.int32, "E"),
    "vaat_queue": (33, np.int32, "E"),
}

# The reference's MC event record (example/Simulated.H:7-14), 48 bytes.
EVENT_DTYPE = np.dtype([
    ("Mass", "<f8"), ("Type", "<i4"), ("pad0", "<i4"),
    ("Separation", "<f8"), ("MuDk", "<i4"), ("pad1", "<i4"),
    ("TrueMass", "<f8"), ("TrueMassSigma", "<f8"),
])
assert EVENT_DTYPE.itemsize == 48


class SmcmcError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("smcmc status %d: %s" % (status, message))
        self.status = status


class _Config(ctypes.Structure):
    _fields_ = [("struct_size", ctypes.c_uint32), ("device", ctypes.c_int32),
                ("dim", ctypes.c_int32), ("chains", ctypes.c_int32),
                ("chain_offset", ctypes.c_uint32), ("likelihood", ctypes.c_int32),
                ("seed", ctypes.c_uint64)]


_SAVED_FIELDS = [("accepted", np.float64, "En"), ("log_likelihood", np.float64, "E"), ("total_steps", np.int32, "E"),
                 ("step_rms", np.float64, "E"), ("trials", np.int32, "E"), ("successes", np.int32, "E"),
                 ("next_update", np.int32, "E"), ("acceptance", np.float64, "E"),
                 ("acceptance_trials", np.float64, "E"), ("sigma", np.float64, "E"),
                 ("central_point", np.float64, "En"), ("central_point_trials", np.float64, "E"),
                 ("covariance", np.float64, "Et"), ("covariance_trials", np.float64, "E"),
                 ("covariance_trace", np.float64, "E")]


class _SavedState(ctypes.Structure):
    _fields_ = [(name, ctypes.c_void_p) for name, _, _ in _SAVED_FIELDS]


# smcmc_hmc_setting / smcmc_hmc_field / scalar columns of SMCMC_HMC_F_SCALARS
HMC_ALPHA, HMC_MEAN_EPSILON, HMC_LEAPFROG, HMC_USER_GRADIENT, HMC_KEEP_ERROR_MATRIX, HMC_POOLED_COVARIANCE = range(6)
_HMC_FIELDS = {"accepted": (0, "En"), "momentum": (1, "En"), "proposed": (2, "En"), "central": (3, "En"),
               "average": (4, "En"), "covariance": (5, "Enn"), "error_matrix": (6, "Enn"), "scalars": (7, "Es"),
               "pooled_covariance": (8, "nn"), "pooled_average": (9, "n"), "pooled_scalars": (10, "ps")}
HMC_POOLED_SCALARS = ["trials", "est_cov_trace", "cur_cov_trace", "orbit_length", "max_scale", "min_scale",
                      "step_count", "updates", "repaired"]
HMC_SCALARS = ["acceptance", "mean_epsilon", "leapfrog", "reversal_len", "accepted_potential",
               "proposed_potential", "central_potential", "potential_count", "gradient_count", "step_count",
               "cov_trials", "average_trials", "est_cov_trace", "cur_cov_trace", "orbit_length",
               "steps_remaining", "steps_since_update"]


class _HmcTrace(ctypes.Structure):
    _fields_ = [("potential", ctypes.c_void_p), ("points", ctypes.c_void_p), ("mean_epsilon", ctypes.c_void_p),
                ("leapfrog", ctypes.c_void_p), ("accepted", ctypes.c_void_p)]


class _Trace(ctypes.Structure):
    _fields_ = [("accepted", ctypes.c_void_p), ("llh_accepted", ctypes.c_void_p),
                ("llh_proposed", ctypes.c_void_p), ("points", ctypes.c_void_p),
                ("sigma", ctypes.c_void_p), ("step_rms", ctypes.c_void_p)]


def library_path():
    # SMCMC_B200_LIB: an alternative build of the same library (kernel tuning experiments)
    return os.environ.get("SMCMC_B200_LIB") or os.path.join(HERE, "libsmcmc_b200.so")


def build_library(verbose=False):
    """Compile libsmcmc_b200.so for sm_100a with nvcc (csrc/Makefile)."""
    subprocess.run(["make", "-C", CSRC], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)


class _DiagResult(ctypes.Structure):
    """smcmc_diag_result"""
    _fields_ = [(name, ctypes.c_void_p) for name in
                ("samples", "steps", "mean", "covariance", "rhat", "lags", "autocorrelation", "tau", "ess")]


_LIB = None


def load_library():
    """Load the CUDA library.  Raises if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise ImportError("%s is missing: run __graft_entry__.build() (there is no "
                          "CPU fallback for the MCMC step path)" % path)
    lib = ctypes.CDLL(path)
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    sig = {
        "smcmc_abi_version": (ci, []),
        "smcmc_last_error": (ctypes.c_char_p, [vp]),
        "smcmc_create": (ci, [ctypes.POINTER(_Config), ctypes.POINTER(vp)]),
        "smcmc_destroy": (ci, [vp]),
        "smcmc_set_stream": (ci, [vp, vp]),
        "smcmc_comm_unique_id": (ci, [ctypes.c_char_p, ctypes.c_size_t]),
        "smcmc_comm_init": (ci, [vp, ctypes.c_char_p, ctypes.c_size_t, ci, ci, ci]),
        "smcmc_sync": (ci, [vp]),
        "smcmc_prop_set": (ci, [vp, ci, cd]),
        "smcmc_prop_set_gaussian": (ci, [vp, ci, cd]),
        "smcmc_prop_set_uniform": (ci, [vp, ci, cd, cd]),
        "smcmc_prop_set_correlation": (ci, [vp, ci, ci, cd]),
        "smcmc_prop_reset_correlations": (ci, [vp]),
        "smcmc_prop_update": (ci, [vp]),
        "smcmc_prop_reset": (ci, [vp]),
        "smcmc_prop_force_step": (ci, [vp, vp, ci]),
        "smcmc_prop_set_scan_dimension": (ci, [vp, ci]),
        "smcmc_prop_set_center": (ci, [vp, vp, ci]),
        "smcmc_user_set_ops": (ci, [vp, vp]),
        "smcmc_fake_set_events": (ci, [vp, vp, ctypes.c_int64]),
        "smcmc_fake_set_data": (ci, [vp, vp, cd]),
        "smcmc_unbinned_set_events": (ci, [vp, vp, ctypes.c_int64]),
        "smcmc_fake_histograms": (ci, [vp, vp, ci, vp]),
        "smcmc_fake_counts": (ci, [vp, vp, ci, vp]),
        "smcmc_fake_filter_check": (ci, [vp, vp, ci, vp]),
        "smcmc_fake_skip_check": (ci, [vp, vp, ci, vp]),
        "smcmc_dummy_set_error": (ci, [vp, vp, ci]),
        "smcmc_dummy_set_mode": (ci, [vp, ci]),
        "smcmc_eval": (ci, [vp, vp, ci, vp]),
        "smcmc_start": (ci, [vp, vp, vp]),
        "smcmc_step": (ci, [vp, ci, ci]),
        "smcmc_step_trace": (ci, [vp, ci, ci, ctypes.POINTER(_Trace)]),
        "smcmc_get": (ci, [vp, ci, vp, ctypes.c_size_t]),
        "smcmc_save_state": (ci, [vp, ctypes.POINTER(_SavedState)]),
        "smcmc_restore_state": (ci, [vp, ctypes.POINTER(_SavedState), vp]),
        "smcmc_get_step_index": (ci, [vp, ctypes.POINTER(ctypes.c_uint32)]),
        "smcmc_set_step_index": (ci, [vp, ctypes.c_uint32]),
        "smcmc_hmc_set": (ci, [vp, ci, cd]),
        "smcmc_hmc_start": (ci, [vp, vp]),
        "smcmc_hmc_set_position": (ci, [vp, vp]),
        "smcmc_hmc_step": (ci, [vp, ci, ci]),
        "smcmc_hmc_step_trace": (ci, [vp, ci, ci, ctypes.POINTER(_HmcTrace)]),
        "smcmc_hmc_get": (ci, [vp, ci, vp, ctypes.c_size_t]),
        "smcmc_launch_count": (ctypes.c_int64, [vp]),
        "smcmc_pair_kernel_stats": (ci, [vp, ctypes.POINTER(cd), ctypes.POINTER(ctypes.c_int64), ci]),
        "smcmc_enable_kernel_timing": (ci, [vp, ci]),
        "smcmc_measure_fp64_peak": (ci, [ci, ctypes.POINTER(cd)]),
        "smcmc_measure_sfu_peak": (ci, [ci, ctypes.POINTER(cd)]),
        "smcmc_measure_dmma_peak": (ci, [ci, ctypes.POINTER(cd)]),
        "smcmc_selftest_division": (ci, [ci, ctypes.c_int64, ctypes.c_uint64, ctypes.POINTER(ctypes.c_int64)]),
        "smcmc_diag_enable": (ci, [vp, ci]),
        "smcmc_diag_reset": (ci, [vp]),
        "smcmc_diag_lag_count": (ci, [vp, ctypes.POINTER(ctypes.c_int32)]),
        "smcmc_diag_get": (ci, [vp, ctypes.POINTER(_DiagResult)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib


EXPORTED_SYMBOLS = [
    "smcmc_abi_version", "smcmc_last_error", "smcmc_create", "smcmc_destroy",
    "smcmc_set_stream", "smcmc_sync", "smcmc_comm_unique_id", "smcmc_comm_init", "smcmc_prop_set", "smcmc_prop_set_gaussian",
    "smcmc_prop_set_uniform", "smcmc_prop_set_correlation",
    "smcmc_prop_reset_correlations", "smcmc_prop_update", "smcmc_prop_reset",
    "smcmc_prop_force_step", "smcmc_prop_set_scan_dimension", "smcmc_prop_set_center", "smcmc_user_set_ops",
    "smcmc_fake_set_events", "smcmc_fake_set_data", "smcmc_unbinned_set_events", "smcmc_fake_histograms",
    "smcmc_fake_counts", "smcmc_fake_filter_check", "smcmc_fake_skip_check",
    "smcmc_dummy_set_error", "smcmc_dummy_set_mode", "smcmc_eval", "smcmc_start", "smcmc_step",
    "smcmc_step_trace", "smcmc_get", "smcmc_save_state", "smcmc_restore_state",
    "smcmc_get_step_index", "smcmc_set_step_index", "smcmc_launch_count",
    "smcmc_hmc_set", "smcmc_hmc_start", "smcmc_hmc_set_position", "smcmc_hmc_step",
    "smcmc_hmc_step_trace", "smcmc_hmc_get",
    "smcmc_pair_kernel_stats", "smcmc_enable_kernel_timing",
    "smcmc_measure_fp64_peak", "smcmc_measure_sfu_peak", "smcmc_measure_dmma_peak", "smcmc_selftest_division",
    "smcmc_diag_enable", "smcmc_diag_reset", "smcmc_diag_lag_count", "smcmc_diag_get",
]


def comm_unique_id():
    """A fresh 128-byte NCCL unique id (create on rank 0, broadcast, pass to Engine.comm_init)."""
    lib = load_library()
    buf = ctypes.create_string_buffer(128)
    rc = lib.smcmc_comm_unique_id(buf, 128)
    if rc != 0:
        raise SmcmcError(rc, lib.smcmc_last_error(None).decode())
    return buf.raw


def measure_fp64_peak(device=0):
    """Measured DFMA throughput of the device, TFLOP/s."""
    lib = load_library()
    out = ctypes.c_double()
    rc = lib.smcmc_measure_fp64_peak(device, ctypes.byref(out))
    if rc != 0:
        raise SmcmcError(rc, lib.smcmc_last_error(None).decode())
    return out.value


def measure_dmma_peak(device=0):
    """Measured FP64 tensor-core (DMMA m8n8k4) throughput of the device, TFLOP/s."""
    lib = load_library()
    out = ctypes.c_double()
    rc = lib.smcmc_measure_dmma_peak(device, ctypes.byref(out))
    if rc != 0:
        raise SmcmcError(rc, lib.smcmc_last_error(None).decode())
    return out.value


def measure_sfu_peak(device=0):
    """Measured MUFU.EX2 throughput of the device, 1e9 evaluations per second."""
    lib = load_library()
    out = ctypes.c_double()
    rc = lib.smcmc_measure_sfu_peak(device, ctypes.byref(out))
    if rc != 0:
        raise SmcmcError(rc, lib.smcmc_last_error(None).decode())
    return out.value


def selftest_division(count, seed=1, device=0):
    """Number of quotients of the staged covariance update's shared-divisor division
    that differ from the IEEE quotient, over `count` random cases (must be 0)."""
    lib = load_library()
    out = ctypes.c_int64()
    rc = lib.smcmc_selftest_division(device, count, seed, ctypes.byref(out))
    if rc != 0:
        raise SmcmcError(rc, lib.smcmc_last_error(None).decode())
    return out.value


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class Engine:
    """E chains of an n-dimensional adaptive Metropolis sampler on one GPU.

    Mirrors sMCMC::TSimpleMCMC<L, TProposeAdaptiveStep> (TSimpleMCMC.H:185):
    Start / Step / GetProposeStep().Set* keep their names and meaning, applied
    to every chain of the ensemble.
    """

    def __init__(self, likelihood, dim, chains, seed=1, device=0, chain_offset=0, proposal=PROPOSAL_ADAPTIVE):
        """proposal=PROPOSAL_VAAT: sMCMC::TSimpleMCMC<L, TProposeVAATStep> (TProposeVAATStep.H)."""
        self.lib = load_library()
        self.dim, self.chains = int(dim), int(chains)
        cfg = _Config(ctypes.sizeof(_Config), device, dim, chains, chain_offset,
                      likelihood, seed)
        h = ctypes.c_void_p()
        rc = self.lib.smcmc_create(ctypes.byref(cfg), ctypes.byref(h))
        if rc != 0:
            raise SmcmcError(rc, self.lib.smcmc_last_error(None).decode())
        self.h = h
        if proposal != PROPOSAL_ADAPTIVE:
            self.prop_set(PROP_KIND, proposal)

    def close(self):
        if getattr(self, "h", None):
            self.lib.smcmc_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _check(self, rc):
        if rc != 0:
            raise SmcmcError(rc, self.lib.smcmc_last_error(self.h).decode())

    # -- plumbing ---------------------------------------------------------
    def set_stream(self, cuda_stream):
        self._check(self.lib.smcmc_set_stream(self.h, ctypes.c_void_p(cuda_stream)))

    def comm_init(self, unique_id, world, rank, event_group=1):
        """Join the NCCL communicator(s); see smcmc_comm_init."""
        self._check(self.lib.smcmc_comm_init(self.h, unique_id, len(unique_id), world, rank, event_group))

    def sync(self):
        self._check(self.lib.smcmc_sync(self.h))

    # -- GetProposeStep().Set*  (TSimpleMCMC.H:733-1003) ---------------------
    def prop_set(self, field, value):
        self._check(self.lib.smcmc_prop_set(self.h, field, float(value)))

    def set_gaussian(self, d, sigma):
        self._check(self.lib.smcmc_prop_set_gaussian(self.h, d, float(sigma)))

    def set_uniform(self, d, lo, hi):
        self._check(self.lib.smcmc_prop_set_uniform(self.h, d, float(lo), float(hi)))

    def set_correlation(self, d1, d2, c):
        self._check(self.lib.smcmc_prop_set_correlation(self.h, d1, d2, float(c)))

    def reset_correlations(self):
        self._check(self.lib.smcmc_prop_reset_correlations(self.h))

    def update_proposal(self):
        self._check(self.lib.smcmc_prop_update(self.h))

    def reset_proposal(self):
        self._check(self.lib.smcmc_prop_reset(self.h))

    def force_step(self, x):
        """ForceStep (TSimpleMCMC.H:811-818): x[dim] for every chain or x[chains, dim]."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        per_chain = 1 if x.ndim == 2 else 0
        if x.size != (self.chains * self.dim if per_chain else self.dim):
            raise SmcmcError(-1, "Invalid forced step point.")
        self._check(self.lib.smcmc_prop_force_step(self.h, _ptr(x), per_chain))

    def set_scan(self, dim):
        """SetScanDimension (:820-830); -1 = off."""
        self._check(self.lib.smcmc_prop_set_scan_dimension(self.h, int(dim)))

    def set_center(self, v):
        """SetEstimatedCenter (:733-739): v[dim] for every chain or v[chains, dim]."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        self._check(self.lib.smcmc_prop_set_center(self.h, _ptr(v), 1 if v.ndim == 2 else 0))

    def bind_user_library(self, lib, symbol):
        """SMCMC_LLH_USER: `symbol(engine)` of a user library compiled by nvcc with
        include/smcmc_device_functor.cuh registers the functor's launch table."""
        fn = getattr(lib, symbol)
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_void_p]
        if fn(self.h) != 0:
            raise SmcmcError(-3, "%s failed: %s" % (symbol, self.lib.smcmc_last_error(self.h).decode()))

    def bind_user_events(self, lib, symbol, events):
        """SMCMC_LLH_USER with an EVENT functor (include/smcmc_device_functor.cuh):
        `symbol(engine, events, n, itemsize)` of a user library uploads the sample
        and registers the functor.  `events` is an array of n records laid out as
        the functor's Event (a structured dtype, or rows of a plain one); the
        library rejects an itemsize other than sizeof(Event).  The sample is
        copied; the array may be dropped afterwards."""
        ev = np.ascontiguousarray(events)
        n = ev.shape[0] if ev.ndim else 1
        itemsize = ev.itemsize * (int(np.prod(ev.shape[1:])) if ev.ndim > 1 else 1)
        fn = getattr(lib, symbol)
        fn.restype = ctypes.c_int
        fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_size_t]
        if fn(self.h, ev.ctypes.data if n else None, n, itemsize) != 0:
            raise SmcmcError(-3, "%s failed (itemsize %d, %d events)" % (symbol, itemsize, n))

    # -- likelihood inputs ---------------------------------------------------
    def set_fake_events(self, events):
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        self._check(self.lib.smcmc_fake_set_events(self.h, _ptr(ev), len(ev)))

    def set_unbinned_events(self, events):
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        self._check(self.lib.smcmc_unbinned_set_events(self.h, _ptr(ev), len(ev)))

    def set_fake_data(self, data150, exposure):
        d = np.ascontiguousarray(data150, dtype=np.float64).reshape(150)
        self._check(self.lib.smcmc_fake_set_data(self.h, _ptr(d), float(exposure)))

    def fake_histograms(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros((x.shape[0], 150))
        self._check(self.lib.smcmc_fake_histograms(self.h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def fake_counts(self, x):
        """Exact event counts per (weight class, histogram, bin): (m, 450) uint32."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros((x.shape[0], 450), np.uint32)
        self._check(self.lib.smcmc_fake_counts(self.h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def fake_filter_check(self, x):
        """(pairs, pairs left to FP64, filter decisions that differ from FP64)."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros(3, np.uint64)
        self._check(self.lib.smcmc_fake_filter_check(self.h, _ptr(x), x.shape[0], _ptr(out)))
        return int(out[0]), int(out[1]), int(out[2])

    def fake_skip_check(self, x):
        """(tiles tested, tiles skipped, pairs of skipped tiles that FP64 counts) of the
        pair kernel's tile skip, one box per 32 consecutive points."""
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros(3, np.uint64)
        self._check(self.lib.smcmc_fake_skip_check(self.h, _ptr(x), x.shape[0], _ptr(out)))
        return int(out[0]), int(out[1]), int(out[2])

    def set_dummy_mode(self, mode):
        """DUMMY_EXACT (reference operation order, default) or DUMMY_TENSOR (FP64 tensor cores)."""
        self._check(self.lib.smcmc_dummy_set_mode(self.h, int(mode)))

    def set_error_matrix(self, e):
        e = np.ascontiguousarray(e, dtype=np.float64)
        self._check(self.lib.smcmc_dummy_set_error(self.h, _ptr(e), e.shape[0]))

    # -- sampler -----------------------------------------------------------------
    def eval(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, self.dim)
        out = np.zeros(x.shape[0])
        self._check(self.lib.smcmc_eval(self.h, _ptr(x), x.shape[0], _ptr(out)))
        return out

    def start(self, x0):
        x0 = np.ascontiguousarray(np.broadcast_to(np.asarray(x0, dtype=np.float64),
                                                  (self.chains, self.dim)))
        ok = np.zeros(self.chains, np.int32)
        self._check(self.lib.smcmc_start(self.h, _ptr(x0), _ptr(ok)))
        return ok

    def step(self, nsteps=1, metropolis=0):
        self._check(self.lib.smcmc_step(self.h, nsteps, metropolis))

    def step_trace(self, nsteps, metropolis=0, want=("accepted", "llh_accepted", "llh_proposed",
                                                      "points", "sigma", "step_rms"), out=None):
        """Step(save=true): returns the per-step record a TTree::Fill would hold."""
        E, n = self.chains, self.dim
        shapes = {"accepted": ((nsteps, E), np.int32), "llh_accepted": ((nsteps, E), np.float64),
                  "llh_proposed": ((nsteps, E), np.float64), "points": ((nsteps, E, n), np.float64),
                  "sigma": ((nsteps, E), np.float64), "step_rms": ((nsteps, E), np.float64)}
        out = {} if out is None else out
        tr = _Trace()
        for name in want:
            shape, dt = shapes[name]
            if name not in out:
                out[name] = np.zeros(shape, dt)
            setattr(tr, name, out[name].ctypes.data)
        self._check(self.lib.smcmc_step_trace(self.h, nsteps, metropolis, ctypes.byref(tr)))
        return out

    def get(self, name):
        fid, dt, code = _FIELDS[name]
        E, n = self.chains, self.dim
        shape = {"E": (E,), "En": (E, n), "Et": (E, n * (n + 1) // 2), "Enn": (E, n, n), "1": (1,),
                 "n": (n,), "t": (n * (n + 1) // 2,), "nn": (n, n)}[code]
        out = np.zeros(shape, dt)
        self._check(self.lib.smcmc_get(self.h, fid, _ptr(out), out.nbytes))
        return out

    # -- checkpoint / resume --------------------------------------------------------
    def _saved_arrays(self):
        E, n = self.chains, self.dim
        shapes = {"E": (E,), "En": (E, n), "Et": (E, n * (n + 1) // 2)}
        return {name: np.zeros(shapes[code], dt) for name, dt, code in _SAVED_FIELDS}

    def save_state(self):
        """SaveStep(true) for every chain: dict of the tree-branch values, plus
        the stream position ("step_index")."""
        arrays = self._saved_arrays()
        st = _SavedState(**{k: v.ctypes.data for k, v in arrays.items()})
        self._check(self.lib.smcmc_save_state(self.h, ctypes.byref(st)))
        step = ctypes.c_uint32()
        self._check(self.lib.smcmc_get_step_index(self.h, ctypes.byref(step)))
        arrays["step_index"] = np.array([step.value], np.uint32)
        return arrays

    def restore_state(self, saved):
        """Restore() + RestoreState() for every chain (call after start())."""
        arrays = self._saved_arrays()
        for k in arrays:
            if k in saved:          # (the covariance trace is written by save_state only)
                arrays[k][...] = np.asarray(saved[k]).reshape(arrays[k].shape)
        st = _SavedState(**{k: v.ctypes.data for k, v in arrays.items()})
        mismatch = np.zeros(self.chains, np.int32)
        self._check(self.lib.smcmc_restore_state(self.h, ctypes.byref(st), _ptr(mismatch)))
        if "step_index" in saved:
            self._check(self.lib.smcmc_set_step_index(self.h, int(np.asarray(saved["step_index"]).reshape(-1)[0])))
        return mismatch

    # -- sMCMC::TSimpleHMC (TSimpleHMC.H:119-973) -----------------------------------
    def hmc_set(self, setting, value):
        """SetAlpha / SetMeanEpsilon / SetLeapFrog, and the two template choices."""
        self._check(self.lib.smcmc_hmc_set(self.h, setting, float(value)))

    def hmc_start(self, x0):
        x0 = np.ascontiguousarray(np.broadcast_to(np.asarray(x0, dtype=np.float64), (self.chains, self.dim)))
        self._check(self.lib.smcmc_hmc_start(self.h, _ptr(x0)))

    def hmc_set_position(self, x):
        x = np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=np.float64), (self.chains, self.dim)))
        self._check(self.lib.smcmc_hmc_set_position(self.h, _ptr(x)))

    def hmc_step(self, nsteps=1, gradient_type=0):
        self._check(self.lib.smcmc_hmc_step(self.h, nsteps, gradient_type))

    def hmc_step_trace(self, nsteps, gradient_type=0,
                       want=("potential", "points", "mean_epsilon", "leapfrog", "accepted"), out=None):
        """Step(save=true): the per-step record of the output tree (:139-147)."""
        E, n = self.chains, self.dim
        shapes = {"potential": ((nsteps, E), np.float64), "points": ((nsteps, E, n), np.float64),
                  "mean_epsilon": ((nsteps, E), np.float64), "leapfrog": ((nsteps, E), np.int32),
                  "accepted": ((nsteps, E), np.int32)}
        out = {} if out is None else out
        tr = _HmcTrace()
        for name in want:
            shape, dt = shapes[name]
            if name not in out:
                out[name] = np.zeros(shape, dt)
            setattr(tr, name, out[name].ctypes.data)
        self._check(self.lib.smcmc_hmc_step_trace(self.h, nsteps, gradient_type, ctypes.byref(tr)))
        return out

    def hmc_get(self, name):
        fid, code = _HMC_FIELDS[name]
        E, n = self.chains, self.dim
        shape = {"En": (E, n), "Enn": (E, n, n), "Es": (E, len(HMC_SCALARS)), "nn": (n, n), "n": (n,),
                 "ps": (len(HMC_POOLED_SCALARS),)}[code]
        out = np.zeros(shape)
        self._check(self.lib.smcmc_hmc_get(self.h, fid, _ptr(out), out.nbytes))
        return out

    def hmc_scalars(self):
        """dict name -> array[chains] of the scalar members (HMC_SCALARS)."""
        s = self.hmc_get("scalars")
        return {k: s[:, i] for i, k in enumerate(HMC_SCALARS)}

    # -- instrumentation -----------------------------------------------------------
    # -- ensemble diagnostics --------------------------------------------------------
    def diag_enable(self, max_lag=0):
        """Accumulate mean / covariance / R-hat / autocorrelation of the accepted points on
        the device after every step (MakeCovariance.C, MakeAutocorrelation.C)."""
        self._check(self.lib.smcmc_diag_enable(self.h, max_lag))

    def diag_reset(self):
        self._check(self.lib.smcmc_diag_reset(self.h))

    def diag_get(self):
        n = self.dim
        nl = ctypes.c_int32()
        self._check(self.lib.smcmc_diag_lag_count(self.h, ctypes.byref(nl)))
        nl = nl.value
        out = {"samples": np.zeros(1, np.int64), "steps": np.zeros(1, np.int64), "mean": np.zeros(n),
               "covariance": np.zeros((n, n)), "rhat": np.zeros(n), "lags": np.zeros(nl, np.int32),
               "autocorrelation": np.zeros((nl, n)), "tau": np.zeros(n), "ess": np.zeros(n)}
        res = _DiagResult()
        for k, v in out.items():
            setattr(res, k, v.ctypes.data)
        self._check(self.lib.smcmc_diag_get(self.h, ctypes.byref(res)))
        out["samples"] = int(out["samples"][0])
        out["steps"] = int(out["steps"][0])
        return out

    def launch_count(self):
        return int(self.lib.smcmc_launch_count(self.h))

    def enable_kernel_timing(self, on=True):
        self._check(self.lib.smcmc_enable_kernel_timing(self.h, 1 if on else 0))

    def pair_kernel_stats(self, reset=False):
        ms = ctypes.c_double()
        n = ctypes.c_int64()
        self._check(self.lib.smcmc_pair_kernel_stats(self.h, ctypes.byref(ms), ctypes.byref(n),
                                                     1 if reset else 0))
        return ms.value, n.value
