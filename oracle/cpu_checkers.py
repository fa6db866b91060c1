"""ctypes bindings for the two CPU checkers (TEST INFRASTRUCTURE ONLY).

``load("ref")`` -> oracle/_ref/libsmcmc_ref.so, the reference's own headers
compiled unmodified against oracle/rootshim (prebuilt in the build container;
the reference tree is not present on the GPU box).
``load("orc")`` -> oracle/_build/libsmcmc_oracle.so, the stand-alone
restatement oracle/smcmc_oracle.cc.

Both export the single-chain interface of oracle/chain_api.h.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module; the product package never does.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

LLH_UNIT_GAUSS, LLH_DUMMY, LLH_HORRIFIC, LLH_ASYM, LLH_FAKE, LLH_UNBINNED, LLH_HARD, LLH_FAKE2, LLH_CONSTRAINED = range(9)

(SET_SIGMA, SET_TARGET_ACCEPTANCE, SET_ACCEPTANCE_WINDOW,
 SET_ACCEPTANCE_RIGIDITY, SET_ACCEPTANCE_DEWEIGHT, SET_COVARIANCE_WINDOW,
 SET_COVARIANCE_DEWEIGHT, SET_COVARIANCE_FROZEN, SET_COVARIANCE_TRIALS,
 SET_CENTER_TRIALS, SET_NEXT_UPDATE, SET_MAX_CORRELATION,
 SET_STEP_RMS_WINDOW) = range(13)

STATE_FIELDS = [
    "sigma", "acceptance", "acceptance_trials", "acceptance_window",
    "acceptance_rigidity", "target_acceptance", "trials", "successes",
    "next_update", "covariance_trials", "covariance_window", "center_trials",
    "covariance_trace", "sigma_trace", "step_rms", "accepted_llh",
    "proposed_llh", "total_steps", "llh_calls",
]

EVENT_DTYPE = np.dtype([
    ("Mass", "<f8"), ("Type", "<i4"), ("pad0", "<i4"),
    ("Separation", "<f8"), ("MuDk", "<i4"), ("pad1", "<i4"),
    ("TrueMass", "<f8"), ("TrueMassSigma", "<f8"),
])
assert EVENT_DTYPE.itemsize == 48

_PATHS = {
    "ref": os.path.join(HERE, "_ref", "libsmcmc_ref.so"),
    "orc": os.path.join(HERE, "_build", "libsmcmc_oracle.so"),
}
_LIBS = {}


def build(which=("orc", "ref")):
    """Compile the checkers (make decides what is stale; `ref` needs the
    reference tree and is skipped with the prebuilt file kept otherwise)."""
    targets = ["oracle" if w == "orc" else "ref" for w in which]
    subprocess.run(["make", "-C", HERE] + targets, check=True,
                   stdout=subprocess.DEVNULL)


def available(which):
    return os.path.exists(_PATHS[which])


def load(which):
    if which in _LIBS:
        return _LIBS[which]
    path = _PATHS[which]
    if not os.path.exists(path):
        build((which,))
    lib = ctypes.CDLL(path)
    p = which + "_"
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    sig = {
        "chain_create": (vp, [ci, ci, ctypes.c_uint64, ctypes.c_uint32]),
        "chain_create_vaat": (vp, [ci, ci, ctypes.c_uint64, ctypes.c_uint32]),
        "chain_get_vaat": (ci, [vp, vp, vp, vp, vp]),
        "chain_destroy": (None, [vp]),
        "chain_set_fake": (ci, [vp, vp, ctypes.c_long, vp, cd]),
        "chain_set_error_matrix": (ci, [vp, vp, ci]),
        "chain_set": (ci, [vp, ci, cd]),
        "chain_set_gaussian": (ci, [vp, ci, cd]),
        "chain_set_uniform": (ci, [vp, ci, cd, cd]),
        "chain_set_correlation": (ci, [vp, ci, ci, cd]),
        "chain_start": (ci, [vp, vp]),
        "chain_step": (ci, [vp, ci, ci, vp, vp, vp, vp, vp]),
        "chain_update_proposal": (ci, [vp]),
        "chain_reset_proposal": (ci, [vp]),
        "chain_get_state": (ci, [vp, vp, vp, vp, vp, vp]),
        "chain_llh": (cd, [vp, vp]),
        "chain_fake_hist": (ci, [vp, vp, vp]),
        "last_error": (ctypes.c_char_p, []),
        "chain_step_saved": (ci, [vp, ci, vp]),
        "chain_save_step": (ci, [vp]),
        "chain_restore": (ci, [vp, vp]),
        "chain_force_step": (ci, [vp, vp]),
        "chain_set_scan": (ci, [vp, ci]),
        "chain_set_center": (ci, [vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, p + name)
        fn.restype = res
        fn.argtypes = args
    hsig = {
        "hmc_create": (vp, [ci, ci, ci, ctypes.c_uint64, ctypes.c_uint32]),
        "hmc_destroy": (None, [vp]),
        "hmc_set_error_matrix": (ci, [vp, vp, ci]),
        "hmc_set": (ci, [vp, ci, cd]),
        "hmc_start": (ci, [vp, vp]),
        "hmc_step": (ci, [vp, ci, ci, vp, vp, vp, vp]),
        "hmc_get_state": (ci, [vp] * 8),
    }
    for name, (res, args) in hsig.items():
        fn = getattr(lib, p + name)
        fn.restype = res
        fn.argtypes = args
    if which == "orc":
        lib.orc_chain_fake_counts.restype = ci
        lib.orc_chain_fake_counts.argtypes = [vp, vp, vp]
    if which == "ref":
        lib.ref_fake_generate.restype = ctypes.c_long
        lib.ref_fake_generate.argtypes = [ctypes.c_ulong, ci, ci, cd, vp,
                                          ctypes.c_long, vp, vp]
        lib.ref_dummy_matrices.restype = ci
        lib.ref_dummy_matrices.argtypes = [vp, vp]
        lib.ref_ex2_generate.restype = ctypes.c_long
        lib.ref_ex2_generate.argtypes = [ctypes.c_ulong, ci, ci, cd, vp, ctypes.c_long, vp]
        lib.ref_chain_restore_random.restype = ci
        lib.ref_chain_restore_random.argtypes = [vp, vp, vp]
    _LIBS[which] = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class CpuChain:
    """One chain of one checker (``which`` = "ref" or "orc")."""

    def __init__(self, which, kind, dim, seed, chain, vaat=False):
        """vaat=True: TSimpleMCMC<L, TProposeVAATStep> (TProposeVAATStep.H)."""
        self.lib = load(which)
        self.p = which + "_"
        self.dim = dim
        self.vaat = vaat
        self.h = self._f("chain_create_vaat" if vaat else "chain_create")(kind, dim, seed, chain)
        if not self.h:
            raise RuntimeError(self._f("last_error")().decode())
        self._keep = []

    def _f(self, name):
        return getattr(self.lib, self.p + name)

    def _check(self, rc):
        if rc < 0:
            raise RuntimeError(self._f("last_error")().decode())
        return rc

    def close(self):
        if self.h:
            self._f("chain_destroy")(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def set_fake(self, events, data150, exposure):
        ev = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        d = np.ascontiguousarray(data150, dtype=np.float64).reshape(150)
        self._check(self._f("chain_set_fake")(self.h, _ptr(ev), len(ev), _ptr(d), float(exposure)))

    def set_error_matrix(self, e):
        e = np.ascontiguousarray(e, dtype=np.float64)
        self._check(self._f("chain_set_error_matrix")(self.h, _ptr(e), e.shape[0]))

    def set(self, field, value):
        self._check(self._f("chain_set")(self.h, field, float(value)))

    def set_gaussian(self, d, sigma):
        self._check(self._f("chain_set_gaussian")(self.h, d, float(sigma)))

    def set_uniform(self, d, lo, hi):
        self._check(self._f("chain_set_uniform")(self.h, d, float(lo), float(hi)))

    def set_correlation(self, d1, d2, c):
        self._check(self._f("chain_set_correlation")(self.h, d1, d2, float(c)))

    def start(self, x0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        return self._check(self._f("chain_start")(self.h, _ptr(x0)))

    def step(self, nsteps, metropolis=0, want_x=True):
        acc = np.zeros(nsteps, np.int32)
        la = np.zeros(nsteps)
        lp = np.zeros(nsteps)
        sg = np.zeros(nsteps)
        x = np.zeros((nsteps, self.dim)) if want_x else None
        self._check(self._f("chain_step")(self.h, nsteps, metropolis, _ptr(acc),
                                          _ptr(la), _ptr(lp), _ptr(x), _ptr(sg)))
        return {"accepted": acc, "llh_accepted": la, "llh_proposed": lp,
                "x": x, "sigma": sg}

    def step_saved(self, nsteps):
        """Step(true): every step is written to the chain's tree."""
        acc = np.zeros(nsteps, np.int32)
        self._check(self._f("chain_step_saved")(self.h, nsteps, _ptr(acc)))
        return acc

    def save_step(self):
        """SaveStep(): the full proposal state goes to the tree."""
        self._check(self._f("chain_save_step")(self.h))

    def restore(self, source):
        """Restore() from the tree of `source` (call after start())."""
        self._check(self._f("chain_restore")(self.h, source.h))

    def restore_random(self, source):
        """Reference build only: Restore(tree, randomize=true); returns the
        TotalSteps of the adopted entry."""
        out = np.zeros(1, np.int32)
        self._check(self.lib.ref_chain_restore_random(self.h, source.h, _ptr(out)))
        return int(out[0])

    def force_step(self, x):
        """ForceStep (TSimpleMCMC.H:811-818): the next proposal is x."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        self._check(self._f("chain_force_step")(self.h, _ptr(x)))

    def set_scan(self, dim):
        """SetScanDimension (:820-830)."""
        self._check(self._f("chain_set_scan")(self.h, int(dim)))

    def set_center(self, v):
        """SetEstimatedCenter (:733-739)."""
        v = np.ascontiguousarray(v, dtype=np.float64)
        self._check(self._f("chain_set_center")(self.h, _ptr(v)))

    def update_proposal(self):
        self._check(self._f("chain_update_proposal")(self.h))

    def reset_proposal(self):
        self._check(self._f("chain_reset_proposal")(self.h))

    def state(self):
        n = self.dim
        s = np.zeros(len(STATE_FIELDS))
        acc = np.zeros(n)
        cen = np.zeros(n)
        cov = np.zeros((n, n))
        dec = np.zeros((n, n))
        self._f("chain_get_state")(self.h, _ptr(s), _ptr(acc), _ptr(cen), _ptr(cov), _ptr(dec))
        out = dict(zip(STATE_FIELDS, s))
        out.update(accepted=acc, center=cen, cov=cov, decomp=dec)
        return out

    def vaat_state(self):
        """The proposal's own state: per-dimension step size, acceptance, trial
        counts; trials, successes, last index, indices left in the queue."""
        n = self.dim
        sigma, acc = np.zeros(n), np.zeros(n)
        trials, misc = np.zeros(n, np.int32), np.zeros(4, np.int32)
        self._check(self._f("chain_get_vaat")(self.h, _ptr(sigma), _ptr(acc), _ptr(trials), _ptr(misc)))
        return {"sigma": sigma, "acceptance": acc, "acceptance_trials": trials, "trials": int(misc[0]),
                "successes": int(misc[1]), "last_index": int(misc[2]), "queue": int(misc[3])}

    def llh(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        return self._f("chain_llh")(self.h, _ptr(x))

    def fake_hist(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.zeros(150)
        self._check(self._f("chain_fake_hist")(self.h, _ptr(x), _ptr(out)))
        return out

    def fake_counts(self, x):
        """Oracle port only: exact event counts per (class, histogram, bin)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.zeros(450, np.uint32)
        self._check(self.lib.orc_chain_fake_counts(self.h, _ptr(x), _ptr(out)))
        return out


HMC_ALPHA, HMC_MEAN_EPSILON, HMC_LEAPFROG = range(3)
HMC_STATE_FIELDS = ["acceptance", "mean_epsilon", "leapfrog", "reversal_len", "accepted_potential",
                    "proposed_potential", "central_potential", "potential_count", "gradient_count",
                    "step_count", "cov_trials", "average_trials", "est_cov_trace", "cur_cov_trace",
                    "orbit_length", "steps_remaining", "steps_since_update"]


class CpuHmc:
    """One TSimpleHMC chain of one checker."""

    def __init__(self, which, kind, dim, with_gradient, seed, chain):
        self.lib = load(which)
        self.p = which + "_"
        self.dim = dim
        self.h = self._f("hmc_create")(kind, dim, 1 if with_gradient else 0, seed, chain)
        if not self.h:
            raise RuntimeError(self._f("last_error")().decode())

    def _f(self, name):
        return getattr(self.lib, self.p + name)

    def _check(self, rc):
        if rc < 0:
            raise RuntimeError(self._f("last_error")().decode())
        return rc

    def close(self):
        if getattr(self, "h", None):
            self._f("hmc_destroy")(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def set_error_matrix(self, e):
        e = np.ascontiguousarray(e, dtype=np.float64)
        self._check(self._f("hmc_set_error_matrix")(self.h, _ptr(e), e.shape[0]))

    def set(self, field, value):
        self._check(self._f("hmc_set")(self.h, field, float(value)))

    def start(self, x0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        return self._check(self._f("hmc_start")(self.h, _ptr(x0)))

    def step(self, nsteps, gradient_type=0):
        pot = np.zeros(nsteps)
        x = np.zeros((nsteps, self.dim))
        eps = np.zeros(nsteps)
        lf = np.zeros(nsteps, np.int32)
        self._check(self._f("hmc_step")(self.h, nsteps, gradient_type, _ptr(pot), _ptr(x), _ptr(eps), _ptr(lf)))
        return {"potential": pot, "x": x, "epsilon": eps, "leapfrog": lf}

    def state(self):
        n = self.dim
        s = np.zeros(len(HMC_STATE_FIELDS))
        acc, mom, cen, avg = np.zeros(n), np.zeros(n), np.zeros(n), np.zeros(n)
        cov, err = np.zeros((n, n)), np.zeros((n, n))
        self._f("hmc_get_state")(self.h, _ptr(s), _ptr(acc), _ptr(mom), _ptr(cen), _ptr(avg), _ptr(cov), _ptr(err))
        out = dict(zip(HMC_STATE_FIELDS, s))
        out.update(accepted=acc, momentum=mom, central=cen, average=avg, covariance=cov, error=err)
        return out


def ref_generate(seed, data_signal, data_background, oversample):
    """Run the reference's own FakeLikelihood::Init() (example/
    FakeLikelihood.H:86-179) under a seeded shim generator."""
    lib = load("ref")
    n = int(oversample * data_signal) + int(2 * oversample * data_background)
    ev = np.zeros(n, EVENT_DTYPE)
    data = np.zeros(150)
    expo = np.zeros(1)
    got = lib.ref_fake_generate(seed, data_signal, data_background, float(oversample),
                                _ptr(ev), n, _ptr(data), _ptr(expo))
    return ev[:got], data, float(expo[0])


def ref2_generate(seed, data_signal, data_background, oversample):
    """Run example2's own FakeLikelihood::Init() (example2/FakeLikelihood.H:123-199)
    under a seeded shim generator: (events, data150)."""
    lib = load("ref")
    cap = 8 * (int(oversample * max(data_signal, 1000)) + int(2 * oversample * max(data_background, 1000))) + 4096
    ev = np.zeros(cap, EVENT_DTYPE)
    data = np.zeros(150)
    got = lib.ref_ex2_generate(seed, data_signal, data_background, float(oversample), _ptr(ev), cap, _ptr(data))
    assert got <= cap
    return ev[:got], data


def ref_dummy_matrices():
    """(Covariance, Error) of the reference's TDummyLogLikelihood::Init()
    (TDummyLogLikelihood.H:44-142), 100 x 100."""
    lib = load("ref")
    cov = np.zeros((100, 100))
    err = np.zeros((100, 100))
    lib.ref_dummy_matrices(_ptr(cov), _ptr(err))
    return cov, err


def shim_linalg(which, a):
    """The shim's TDecompChol (0), TMatrixD::Invert (1) or TMatrixDSymEigen (2) on a square matrix:
    (matrix, values) as the reference's code receives them (oracle/shim_linalg.cc)."""
    if "shim" not in _LIBS:
        path = os.path.join(HERE, "_build", "libsmcmc_shim.so")
        if not os.path.exists(path):
            build(("orc",))
        lib = ctypes.CDLL(path)
        lib.shim_linalg.restype = ctypes.c_int
        lib.shim_linalg.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
        lib.shim_last_error.restype = ctypes.c_char_p
        _LIBS["shim"] = lib
    lib = _LIBS["shim"]
    a = np.ascontiguousarray(a, dtype=np.float64)
    n = a.shape[0]
    out = np.zeros((n, n))
    values = np.zeros(n)
    rc = lib.shim_linalg(which, n, _ptr(a), _ptr(out), _ptr(values))
    if rc < 0:
        raise RuntimeError(lib.shim_last_error().decode())
    return (out, values) if rc == 0 else (None, None)
