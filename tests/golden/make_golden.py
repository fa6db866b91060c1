"""Generate the golden vectors under tests/golden/ by running the REFERENCE's
own code (oracle/_ref/libsmcmc_ref.so = the reference's headers compiled
unmodified against oracle/rootshim) on seeded inputs.

Needs a checkout of the reference:
    REFERENCE=<checkout> python tests/golden/make_golden.py
The reference ships no golden vectors of its own (SURVEY.md section 4), so these
files are how its behaviour is pinned for the machines where the reference
tree is absent.  `python tests/golden/make_golden.py fresh` also runs without
the reference: fresh_seeds.npz then comes from the oracle port and says so in
its `source` entry.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, ROOT)

from oracle import cpu_checkers as cc  # noqa: E402
import smcmc_b200.synth as synth       # noqa: E402

# The parameter excursions of example/TestLikelihood.C:36-207 (nominal, then
# each of the 9 parameters at +delta and -delta).
GRID_DELTAS = [1.0, 1.0, 1.0, 1.0, 5.0, 5.0, 5.0, 10.0, 10.0]


def likelihood_grid():
    pts = [np.zeros(9)]
    for i, d in enumerate(GRID_DELTAS):
        for s in (+1.0, -1.0):
            p = np.zeros(9)
            p[i] = s * d
            pts.append(p)
    return np.array(pts)


def make_fake():
    events, data = synth.fake_inputs(200, 200, 10, seed=17)      # 6000 events
    # a few irregular records: data-typed, negative separation, zero mass
    extra = np.zeros(4, cc.EVENT_DTYPE)
    extra["Mass"] = [120.0, 80.0, 0.0, 250.0]
    extra["Type"] = [-1, 0, 1, -2]
    extra["Separation"] = [30.0, -5.0, 20.0, 150.0]
    extra["MuDk"] = [0, 0, 1, 1]
    extra["TrueMass"] = [135.0, 135.0, 300.0, 200.0]
    extra["TrueMassSigma"] = [40.5, 40.5, 90.0, 60.0]
    events_irregular = np.concatenate([events, extra])
    c = cc.CpuChain("ref", cc.LLH_FAKE, 9, 1, 0)
    c.set_fake(events, data, 1.0)
    sim0 = c.fake_hist(np.zeros(9))
    exposure = float(sum(data)) / float(sum(sim0))
    rng = np.random.default_rng(23)
    points = np.concatenate([likelihood_grid(), rng.uniform(-3, 3, (13, 9)),
                             rng.normal(0, 8, (6, 9))])
    out = {"events": events, "events_irregular": events_irregular, "data": data,
           "exposure": exposure, "points": points}
    for tag, ev in (("", events), ("_irregular", events_irregular)):
        c = cc.CpuChain("ref", cc.LLH_FAKE, 9, 1, 0)
        c.set_fake(ev, data, exposure)
        out["llh" + tag] = np.array([c.llh(p) for p in points])
        out["hist" + tag] = np.array([c.fake_hist(p) for p in points])
    # the FakeMCMC.C schedule (:93-165) in miniature, two chains
    for chain in (0, 7):
        x0 = np.random.default_rng(100 + chain).uniform(-1, 1, 9)
        c = cc.CpuChain("ref", cc.LLH_FAKE, 9, 4242, chain)
        c.set_fake(events, data, exposure)
        c.start(x0)
        parts = [c.step(60)]
        c.reset_proposal()
        parts.append(c.step(60))
        c.update_proposal()
        parts.append(c.step(120))
        for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
            out["chain%d_%s" % (chain, k)] = np.concatenate([p[k] for p in parts])
        out["chain%d_x0" % chain] = x0
        st = c.state()
        out["chain%d_cov" % chain] = st["cov"]
        out["chain%d_decomp" % chain] = st["decomp"]
        out["chain%d_center" % chain] = st["center"]
    np.savez_compressed(os.path.join(HERE, "fake_likelihood.npz"), **out)
    print("fake_likelihood.npz: %d events, %d points" % (len(events), len(points)))


def make_fake2():
    """example2/FakeLikelihood.H through the reference build: the parameter
    excursions of example2/TestLikelihood.C around the true event counts, random
    points (negative event counts and empty histograms included), and a chain
    with the example2/FakeMCMC.C schedule in miniature."""
    events, data = synth.fake2_inputs(150, 150, 10, seed=29)     # ~7 000 events
    extra = np.zeros(3, cc.EVENT_DTYPE)                          # data-typed records: background histograms, weight 1
    extra["Mass"] = [120.0, 250.0, 40.0]
    extra["Type"] = [-1, -2, -1]
    extra["Separation"] = [30.0, 150.0, 80.0]
    extra["MuDk"] = [0, 1, 0]
    extra["TrueMass"] = [135.0, 200.0, 135.0]
    extra["TrueMassSigma"] = [40.5, 60.0, 40.5]
    events_irregular = np.concatenate([events, extra])
    nominal = np.zeros(9)
    nominal[0], nominal[1] = 150.0, 150.0
    pts = [nominal.copy()]
    for i, d in enumerate([15.0, 15.0, 1.0, 1.0, 5.0, 5.0, 5.0, 2.0, 2.0]):
        for sgn in (+1.0, -1.0):
            q = nominal.copy()
            q[i] += sgn * d
            pts.append(q)
    rng = np.random.default_rng(31)
    rnd = rng.normal(0, 3, (14, 9))
    rnd[:, 0] = rng.uniform(-100, 900, 14)
    rnd[:, 1] = rng.uniform(-100, 900, 14)
    far = rng.normal(0, 40, (3, 9))
    far[0, 2] = 100.0                      # every event cut: empty histograms, x/0 normalisation
    points = np.concatenate([np.array(pts), rnd, far])
    out = {"events": events, "events_irregular": events_irregular, "data": data, "points": points}
    for tag, ev in (("", events), ("_irregular", events_irregular)):
        c = cc.CpuChain("ref", cc.LLH_FAKE2, 9, 1, 0)
        c.set_fake(ev, data, 1.0)
        out["llh" + tag] = np.array([c.llh(q) for q in points])
        out["hist" + tag] = np.array([c.fake_hist(q) for q in points])
    for chain in (0, 5):
        x0 = nominal + np.random.default_rng(200 + chain).uniform(-1, 1, 9)
        c = cc.CpuChain("ref", cc.LLH_FAKE2, 9, 777, chain)
        c.set_fake(events, data, 1.0)
        c.set_gaussian(0, 15.0)            # the event counts move on their own scale
        c.set_gaussian(1, 15.0)
        c.start(x0)
        parts = [c.step(80)]
        c.reset_proposal()
        parts.append(c.step(80))
        c.update_proposal()
        parts.append(c.step(140))
        for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
            out["chain%d_%s" % (chain, k)] = np.concatenate([q[k] for q in parts])
        out["chain%d_x0" % chain] = x0
        st = c.state()
        out["chain%d_cov" % chain] = st["cov"]
        out["chain%d_decomp" % chain] = st["decomp"]
    np.savez_compressed(os.path.join(HERE, "fake2_likelihood.npz"), **out)
    print("fake2_likelihood.npz: %d events, %d points, accepted %s" % (
        len(events), len(points), [int(out["chain%d_accepted" % c].sum()) for c in (0, 5)]))


# TSimpleMCMC<L, TProposeVAATStep> (SimpleVAAT.C:31): name -> (kind, dim, seed, chain, steps, configure)
def _vaat_hints(c):
    c.set_uniform(2, -1.5, 2.0)
    c.set_gaussian(4, 0.5)
    c.set(cc.SET_ACCEPTANCE_RIGIDITY, 1.5)


VAAT_CHAINS = {
    "vaat_unit5": (cc.LLH_UNIT_GAUSS, 5, 7, 3, 1500, None),
    "vaat_unit9_hints": (cc.LLH_UNIT_GAUSS, 9, 11, 0, 1200, _vaat_hints),
    "vaat_horrific75": (cc.LLH_HORRIFIC, 75, 5, 9, 900, None),
}


def make_vaat():
    out = {}
    for name, (kind, dim, seed, chain, nsteps, configure) in VAAT_CHAINS.items():
        c = cc.CpuChain("ref", kind, dim, seed, chain, vaat=True)
        if configure:
            configure(c)
        out[name + "/ok"] = np.array([c.start(np.zeros(dim))])
        first = c.step(nsteps - 300)
        c.set(cc.SET_ACCEPTANCE_WINDOW, 37.0)        # honoured after Start (before, InitializeState overrides it)
        second = c.step(300)
        for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma"):
            out[name + "/" + k] = np.concatenate([first[k], second[k]])
        v = c.vaat_state()
        for k in ("sigma", "acceptance", "acceptance_trials"):
            out[name + "/final_" + k] = np.asarray(v[k])
        out[name + "/final_misc"] = np.array([v["trials"], v["successes"], v["last_index"], v["queue"]])
        st = c.state()
        out[name + "/final_step_rms"] = np.array([st["step_rms"]])
        print(name, "accepted", int(out[name + "/accepted"].sum()), "of", nsteps)
    np.savez_compressed(os.path.join(HERE, "vaat.npz"), **out)


def run_chain(kind, dim, seed, chain, nsteps, configure=None, x0=None):
    c = cc.CpuChain("ref", kind, dim, seed, chain)
    if configure:
        configure(c)
    x0 = np.zeros(dim) if x0 is None else x0
    ok = c.start(x0)
    tr = c.step(nsteps)
    st = c.state()
    rec = {k: tr[k] for k in ("accepted", "llh_accepted", "llh_proposed", "x", "sigma")}
    rec["ok"] = np.array([ok])
    for k in ("cov", "decomp", "center", "accepted"):
        rec["final_" + k] = st[k]
    rec["final_scalars"] = np.array([st[k] for k in cc.STATE_FIELDS])
    return rec


def make_chains():
    out = {}

    def put(name, rec):
        for k, v in rec.items():
            out[name + "__" + k] = v

    # C1: the documentation example (TSimpleMCMC.H:111-157), 5 dimensions,
    # with its proposal hints, default adaptive proposal.
    def readme(c):
        c.set_gaussian(3, 2.0)
        c.set_uniform(4, -5, 5)
        c.set_correlation(3, 4, 0.3)
    put("unit5_hints", run_chain(cc.LLH_UNIT_GAUSS, 5, 1, 0, 4000, readme))
    put("unit5_plain", run_chain(cc.LLH_UNIT_GAUSS, 5, 1, 2, 4000))
    put("unit9", run_chain(cc.LLH_UNIT_GAUSS, 9, 5, 1, 2500))
    # step size frozen (SetAcceptanceRigidity(-1), TSimpleMCMC.H:995-1002):
    # no pow() in the loop, so every device must reproduce this bit for bit.
    def frozen(c):
        c.set(cc.SET_ACCEPTANCE_RIGIDITY, -1.0)
        c.set(cc.SET_SIGMA, 0.4)
    put("unit9_frozen_sigma", run_chain(cc.LLH_UNIT_GAUSS, 9, 5, 3, 2500, frozen))
    # as-shipped test likelihoods
    put("horrific75", run_chain(cc.LLH_HORRIFIC, 75, 4, 11, 2500))
    put("asym100", run_chain(cc.LLH_ASYM, 100, 4, 12, 1500, x0=np.full(100, 0.01)))
    cov, err = cc.ref_dummy_matrices()
    out["dummy100_error"] = err
    out["dummy100_covariance"] = cov
    put("dummy100", run_chain(cc.LLH_DUMMY, 100, 9, 0, 1200))
    # correlation hints that are out of range / nearly singular: drives the
    # conditioning ladder (SimpleMCMC.C:107-115, TSimpleMCMC.H:1124-1239)
    def nasty(c):
        rng = np.random.default_rng(8)
        for i in range(6):
            for j in range(i + 1, 6):
                c.set_correlation(i, j, float(rng.uniform(-0.2, 0.2)))
        c.set_correlation(2, 3, 2.0)     # clamped to the maximum correlation
    put("unit6_clamped", run_chain(cc.LLH_UNIT_GAUSS, 6, 3, 4, 1500, nasty))
    # ... and with the reference's own fault injection, c = 1.0/0.0 (SimpleMCMC.C:111)
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import configure_golden
    put("unit6_infinite", run_chain(cc.LLH_UNIT_GAUSS, 6, 3, 5, 1500,
                                    lambda c: configure_golden("unit6_infinite", c, None)))
    # SimpleMCMC.C -DUSE_HARD_LIKELIHOOD: the 6-dimensional Rosenbrock valley
    put("hard6", run_chain(cc.LLH_HARD, 6, 13, 2, 2500, x0=np.full(6, 0.5)))
    # example4: the constrained 25-dimensional Gaussian, started near its priors
    put("constrained25", run_chain(cc.LLH_CONSTRAINED, 25, 51, 3, 3000, x0=np.full(25, 70.0)))
    # the debugging modes of the proposal: ForceStep, SetScanDimension, SetEstimatedCenter
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import configure_debug_modes, run_debug_modes
    d = cc.CpuChain("ref", cc.LLH_UNIT_GAUSS, 9, 61, 5)
    configure_debug_modes(d)
    d.start(np.full(9, 0.2))
    rec = run_debug_modes(d)
    sd = d.state()
    rec["final_scalars"] = np.array([sd[k] for k in cc.STATE_FIELDS])
    rec["final_center"] = sd["center"]
    rec["final_cov"] = sd["cov"]
    put("debug9", rec)
    # Restore(tree, randomize = true): which entry of a 400-entry tree each of 6 chains adopts
    picks = []
    for chain in range(6):
        a = cc.CpuChain("ref", cc.LLH_UNIT_GAUSS, 4, 71, chain)
        a.start(np.full(4, 0.1))
        a.step_saved(400)
        a.save_step()
        b = cc.CpuChain("ref", cc.LLH_UNIT_GAUSS, 4, 71, chain)
        b.start(np.zeros(4))
        total = b.restore_random(a)
        picks.append(np.concatenate([[total], b.state()["accepted"], [b.state()["accepted_llh"]]]))
    out["restore_random__picks"] = np.array(picks)
    # checkpoint / resume: 250 unsaved + 50 saved steps, SaveStep(), then a NEW
    # sampler is started, Restore()d from that tree and run on (TSimpleMCMC.H:282-352)
    a = cc.CpuChain("ref", cc.LLH_UNIT_GAUSS, 7, 31, 2)
    a.start(np.full(7, 0.1))
    first = a.step(250)
    a.step_saved(50)
    a.save_step()
    sa = a.state()
    b = cc.CpuChain("ref", cc.LLH_UNIT_GAUSS, 7, 31, 2)
    b.start(np.zeros(7))
    b.restore(a)
    put("restore7", dict(b.step(200), before_accepted=first["accepted"],
                         saved_scalars=np.array([sa[k] for k in cc.STATE_FIELDS]), saved_accepted=sa["accepted"],
                         saved_center=sa["center"], saved_cov=sa["cov"],
                         final_scalars=np.array([b.state()[k] for k in cc.STATE_FIELDS])))
    np.savez_compressed(os.path.join(HERE, "chains.npz"), **out)
    print("chains.npz: %d arrays" % len(out))


def make_hmc():
    """TSimpleHMC chains of the reference build (TSimpleHMC.H:119-973)."""
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import HMC_GOLDEN, hmc_error_matrix
    fields = {"alpha": cc.HMC_ALPHA, "mean_epsilon": cc.HMC_MEAN_EPSILON, "leapfrog": cc.HMC_LEAPFROG}
    out = {}
    _, err100 = cc.ref_dummy_matrices()
    for name, cfg in HMC_GOLDEN.items():
        c = cc.CpuHmc("ref", cfg["kind"], cfg["dim"], cfg["grad"], cfg["seed"], cfg["chain"])
        if "error" in cfg:
            key = "error_" + cfg["error"]
            if key not in out:
                out[key] = err100 if cfg["error"] == "dummy100" else hmc_error_matrix(cfg["error"])
            # (the reference build keeps its own static matrix; the file carries it for the others)
        for f, v in cfg.get("pre", ()):
            c.set(fields[f], v)
        c.start(np.full(cfg["dim"], cfg["x0"]))
        for f, v in cfg.get("post", ()):
            c.set(fields[f], v)
        tr = c.step(cfg["nsteps"], cfg["gtype"])
        st = c.state()
        for k in ("potential", "x", "epsilon", "leapfrog"):
            out[name + "__" + k] = tr[k]
        out[name + "__final_scalars"] = np.array([st[k] for k in cc.HMC_STATE_FIELDS])
        for k in ("accepted", "momentum", "central", "average", "covariance", "error"):
            out[name + "__final_" + k] = st[k]
        print("  %-20s acceptance %.3f  leapfrog %d  epsilon %.4g  gradients %d" % (
            name, st["acceptance"], st["leapfrog"], st["mean_epsilon"], st["gradient_count"]))
    np.savez_compressed(os.path.join(HERE, "hmc.npz"), **out)
    print("hmc.npz: %d arrays" % len(out))


# ---------------------------------------------------------------------------
# Fresh seeds (tests/test_oracle.py::test_port_equals_reference_on_fresh_inputs and
# ::test_fake2_port_equals_reference_on_fresh_inputs): seeds and points that no other
# golden file uses.  The full traces are too large to commit, so fresh_seeds.npz holds a
# SHA-256 of every array (bit-for-bit comparison) and a seeded sample of steps (readable
# failures).  `source` names the build that produced the file: "reference" when
# oracle/_ref was built, otherwise "port" (the oracle port, itself pinned to the reference
# by the other golden files).
# ---------------------------------------------------------------------------
FRESH_CHAINS = [(0, 5, 1500), (0, 3, 800), (2, 75, 1200), (3, 100, 800)]
FRESH_CHAIN_IDS = (1, 9)
FRESH_SAMPLE_STEPS = 24


def digest(a):
    """SHA-256 of an array's dtype, shape and bytes (NaNs made canonical) as 32 uint8."""
    import hashlib
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def fresh_chain(which, kind, dim, n, chain):
    """(Start() result, trace of n steps) of one fresh-seed chain."""
    c = cc.CpuChain(which, kind, dim, 77, chain)
    ok = c.start(np.random.default_rng(chain).uniform(-0.2, 0.2, dim))
    return ok, c.step(n)


def fresh_sample(n, chain):
    return np.sort(np.random.default_rng(100 + chain).choice(n, FRESH_SAMPLE_STEPS, replace=False))


def fresh_fake2(which):
    """example2's likelihood and histograms at 30 new points on new events, including negative
    event counts (the penalty branches) and a point where every event is cut."""
    events, data = synth.fake2_inputs(120, 90, 10, seed=77)
    c = cc.CpuChain(which, cc.LLH_FAKE2, 9, 1, 0)
    c.set_fake(events, data, 1.0)
    rng = np.random.default_rng(5)
    pts = rng.normal(0, 2, (30, 9))
    pts[:, 0] = rng.uniform(-60, 400, 30)
    pts[:, 1] = rng.uniform(-60, 400, 30)
    pts[0, 2] = 2000.0      # exp overflows: every mass is inf, every event cut
    return np.array([c.llh(p) for p in pts]), np.array([c.fake_hist(p) for p in pts])


def make_fresh():
    which = "ref" if cc.available("ref") else "orc"
    out = {"source": np.array("reference" if which == "ref" else "port")}
    for kind, dim, n in FRESH_CHAINS:
        for chain in FRESH_CHAIN_IDS:
            ok, tr = fresh_chain(which, kind, dim, n, chain)
            p = "k%d_d%d_c%d/" % (kind, dim, chain)
            out[p + "ok"] = np.array(ok)
            rows = fresh_sample(n, chain)
            for k, v in tr.items():
                out[p + k + "_sha256"] = digest(v)
                out[p + k + "_sample"] = v[rows]
    llh, hist = fresh_fake2(which)
    out["fake2/llh"] = llh
    out["fake2/hist_sha256"] = digest(hist)
    out["fake2/hist_sample"] = hist[::7]
    np.savez_compressed(os.path.join(HERE, "fresh_seeds.npz"), **out)
    print("fresh_seeds.npz: %d arrays from the %s build" % (len(out), out["source"]))


if __name__ == "__main__":
    cc.build()
    which = sys.argv[1:] or ["fake", "fake2", "chains", "hmc", "vaat", "fresh"]
    if "vaat" in which:
        make_vaat()
    if "fake" in which:
        make_fake()
    if "fake2" in which:
        make_fake2()
    if "chains" in which:
        make_chains()
    if "hmc" in which:
        make_hmc()
    if "fresh" in which:
        make_fresh()
