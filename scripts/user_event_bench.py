"""User event functors against the built-in kernel at 4096 chains x 10^6 events:
UnbinnedEvents (tests/cpp/user_events.cuh) through kEventPairs<F> / kEventFinish<F>
against SMCMC_LLH_UNBINNED (kUnbinnedPairs), alternating, then Metropolis steps of
both, and the chain-local functor that loops over a device pointer to the events
(UnbinnedLoop) as a contrast.  The user library is compiled into a temporary
directory.  Prints one JSON document (and writes it to --out).

Times are host clocks around synchronous calls: an evaluation includes the copy of
the 4096 x 9 points in and of the 4096 values out.  The prepared events (32 MB for
both paths) fit in the 126 MB L2."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def time_eval(eng, x, reps):
    eng.eval(x)
    t0 = time.perf_counter()
    for _ in range(reps):
        out = eng.eval(x)
    return (time.perf_counter() - t0) / reps * 1e3, out


def time_steps(eng, x0, warm, steps):
    assert eng.start(x0).all()
    eng.step(warm)
    eng.sync()
    t0 = time.perf_counter()
    eng.step(steps)
    eng.sync()
    return (time.perf_counter() - t0) / steps * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--events", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=10, help="evaluations per timed block")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--loop-reps", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()

    import smcmc_b200
    from smcmc_b200 import synth
    import user_events_support as ues

    E, N = args.chains, args.events
    tmp = tempfile.mkdtemp(prefix="user_event_bench_")
    lib = ues.build_library(tmp)
    events = synth.make_mc_sample(N // 3 + 1, N - N // 3 - 1, 2)
    prepared = ues.unbinned_events(events)
    x = np.random.default_rng(0).uniform(-1, 1, (E, 9))

    builtin = smcmc_b200.Engine(smcmc_b200.LLH_UNBINNED, 9, E, seed=3)
    builtin.set_unbinned_events(events)
    user = smcmc_b200.Engine(smcmc_b200.LLH_USER, 9, E, seed=3)
    user.bind_user_events(lib, "user_unbinned_bind", prepared)
    loop = smcmc_b200.Engine(smcmc_b200.LLH_USER, 9, E, seed=3)
    loop.bind_user_events(lib, "user_unbinned_loop_bind", prepared)

    res = dict(gpu_info(), chains=E, events=N, pairs=E * N, reps=args.reps, rounds=[])
    for _ in range(args.rounds):
        tb, vb = time_eval(builtin, x, args.reps)
        tu, vu = time_eval(user, x, args.reps)
        res["rounds"].append({"builtin_ms": tb, "user_ms": tu})
    res["builtin_ms"] = min(r["builtin_ms"] for r in res["rounds"])
    res["user_ms"] = min(r["user_ms"] for r in res["rounds"])
    res["user_over_builtin"] = res["user_ms"] / res["builtin_ms"]
    res["builtin_pairs_per_s"] = E * N / (res["builtin_ms"] * 1e-3)
    res["user_pairs_per_s"] = E * N / (res["user_ms"] * 1e-3)
    res["max_rel_diff_user_builtin"] = float(np.max(np.abs(vu / vb - 1.0)))

    tl, vl = time_eval(loop, x, args.loop_reps)
    res["loop_ms"] = tl
    res["loop_pairs_per_s"] = E * N / (tl * 1e-3)
    res["max_rel_diff_loop_builtin"] = float(np.max(np.abs(vl / vb - 1.0)))

    for name, eng, steps in (("builtin", builtin, args.steps), ("user", user, args.steps), ("loop", loop, 2)):
        ms = time_steps(eng, x, 2, steps)
        res[name + "_step_ms"] = ms
        res[name + "_chain_steps_per_s"] = E / (ms * 1e-3)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
