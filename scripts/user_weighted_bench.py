"""A weighted binned user functor against the other FAKE paths at 4096 chains x
10^6 events (C2): FakeWeighted (tests/cpp/user_weighted.cuh) through
kWeightedPairs<F> / kWeightedFinish<F>, FakeBinned (tests/cpp/user_binned.cuh)
through kBinnedPairs<F> / kBinnedFinish<F>, the built-in SMCMC_LLH_FAKE (kFakePairs,
FP32 filter and tile skip), and the built-in with SMCMC_FAKE_EXACT=1 (every pair in
FP64 with one exp).  The four are alternated in one process, `--rounds` times; each
evaluation is timed with CUDA events on the default stream, which the engines use,
and includes the copy of the 4096 x 9 points in and of the values out.  GaussWeighted
(40 bins, 10^6 flat template events) is timed in the same rounds.  Then one
evaluation of each weighted functor under torch.profiler (CUDA activity), for the
split between the pair and the finish kernel, and the shapes of kWeightedPairs
(points per CTA, dynamic shared memory, resident CTAs per SM from the occupancy
query).  The user libraries are compiled into a temporary directory.  Prints one
JSON document (and writes it to --out)."""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, ROOT)

from user_binned_bench import gpu_info, time_eval  # noqa: E402


def kernel_times(fn):
    """Device time per kernel name of one call of fn, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0 and ("Weighted" in e.key or "Binned" in e.key):
            out[e.key] = t / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--events", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=10, help="evaluations per timed block")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import ctypes
    import torch
    import smcmc_b200
    from smcmc_b200 import synth
    import user_binned_support as ubs
    import user_weighted_support as uws

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark times the device")
    E, N = args.chains, args.events
    tmp = tempfile.mkdtemp(prefix="user_weighted_bench_")
    wlib = uws.build_library(tmp)
    blib = ubs.build_library(tmp)
    signal = N // 3 + (1 if N % 3 else 0)
    events = synth.make_mc_sample(signal, N - signal, seed=2)
    data = synth.make_data_histograms(33334, 33334, seed=2)
    x = np.stack([np.random.default_rng([3, c]).uniform(-1.0, 1.0, 9) for c in range(E)])

    builtin = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, E, seed=3)
    builtin.set_fake_events(events)
    exposure = synth.exposure_ratio(builtin, data)
    builtin.set_fake_data(data, exposure)
    os.environ["SMCMC_FAKE_EXACT"] = "1"                 # read when the engine is created
    exact = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, 9, E, seed=3)
    del os.environ["SMCMC_FAKE_EXACT"]
    exact.set_fake_events(events)
    exact.set_fake_data(data, exposure)
    ubs.set_fake_data(blib, data, exposure)
    binned = smcmc_b200.Engine(smcmc_b200.LLH_USER, 9, E, seed=3)
    binned.bind_user_events(blib, "user_fake_binned_bind", ubs.fake_events(blib, events))
    uws.set_fake_data(wlib, data, exposure)
    weighted = smcmc_b200.Engine(smcmc_b200.LLH_USER, 9, E, seed=3)
    weighted.bind_user_events(wlib, "user_fake_weighted_bind", uws.fake_events(wlib, events))
    v, hist = ubs.gauss_data(10000, seed=2)
    uws.set_gauss_data(wlib, hist)
    gauss = smcmc_b200.Engine(smcmc_b200.LLH_USER, 2, E, seed=3)
    gauss.bind_user_events(wlib, "user_gauss_weighted_bind", uws.gauss_template(N, seed=11))
    xg = np.random.default_rng(4).uniform([2.0, 1.0], [4.0, 3.0], (E, 2))

    paths = (("weighted", weighted, x), ("binned", binned, x), ("builtin", builtin, x), ("exact", exact, x),
             ("gauss_weighted", gauss, xg))
    res = dict(gpu_info(), chains=E, events=N, pairs=E * N, reps=args.reps, rounds=[])
    values = {}
    for _ in range(args.rounds):
        r = {}
        for name, eng, pts in paths:
            r[name + "_ms"], values[name] = time_eval(eng, pts, args.reps)
        res["rounds"].append(r)
    for name, _, _ in paths:
        times = [r[name + "_ms"] for r in res["rounds"]]
        res[name + "_ms"] = min(times)
        res[name + "_spread_ms"] = [min(times), max(times)]
        res[name + "_pairs_per_s"] = E * N / (min(times) * 1e-3)
    res["weighted_over_exact"] = res["weighted_ms"] / res["exact_ms"]
    res["weighted_over_binned"] = res["weighted_ms"] / res["binned_ms"]
    res["weighted_over_builtin"] = res["weighted_ms"] / res["builtin_ms"]
    res["max_rel_diff_weighted_builtin"] = float(np.max(np.abs(values["weighted"] / values["builtin"] - 1.0)))

    res["kernels_ms_fake_weighted"] = kernel_times(lambda: weighted.eval(x))
    res["kernels_ms_gauss_weighted"] = kernel_times(lambda: gauss.eval(xg))
    res["kernels_ms_fake_binned"] = kernel_times(lambda: binned.eval(x))
    for name, kind, eng in (("fake", uws.FAKE, weighted), ("gauss", uws.GAUSS, gauss)):
        shape = (ctypes.c_int64 * 3)()
        wlib.user_weighted_shape(kind, eng.h, shape)
        res[name + "_weighted_shape"] = {"points_per_cta": int(shape[0]), "dynamic_smem_bytes": int(shape[1]),
                                         "resident_ctas_per_sm": int(shape[2]),
                                         "chunks": -(-N // int(wlib.user_weighted_chunk(N))),
                                         "ctas": -(-N // int(wlib.user_weighted_chunk(N))) * -(-E // int(shape[0]))}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
