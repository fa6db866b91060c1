"""A binned user functor against the built-in kernel at 4096 chains x 10^6 events
(C2): FakeBinned (tests/cpp/user_binned.cuh) through kBinnedPairs<F> /
kBinnedFinish<F>, the built-in SMCMC_LLH_FAKE (kFakePairs, FP32 filter and tile
skip), and the built-in with SMCMC_FAKE_EXACT=1 (every pair in FP64 with one exp,
as the user functor does).  The three are alternated in one process; each
evaluation is timed with CUDA events on the default stream, which the engines use,
and includes the copy of the 4096 x 9 points in and of the values out.  Then the
flush's share of kBinnedPairs: the kernel, and a kernel of the same shape and grid
that only sets every counter half to 1 and runs the same flush (the most work a
flush can have), alternated.  The user library is compiled into a temporary
directory.  Prints one JSON document (and writes it to --out).  The events (32 MB built-in, 40 MB user) fit in
the 126 MB L2."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

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
    """ms per evaluation, CUDA events around `reps` synchronous evaluations."""
    import torch
    eng.eval(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = eng.eval(x)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=4096)
    ap.add_argument("--events", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=20, help="evaluations per timed block")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()

    import torch
    import smcmc_b200
    from smcmc_b200 import synth
    import user_binned_support as ubs

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this benchmark times the device")
    E, N = args.chains, args.events
    lib = ubs.build_library(tempfile.mkdtemp(prefix="user_binned_bench_"))
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
    ubs.set_fake_data(lib, data, exposure)
    prepared = ubs.fake_events(lib, events)
    user = smcmc_b200.Engine(smcmc_b200.LLH_USER, 9, E, seed=3)
    user.bind_user_events(lib, "user_fake_binned_bind", prepared)

    res = dict(gpu_info(), chains=E, events=N, pairs=E * N, reps=args.reps, rounds=[])
    for _ in range(args.rounds):
        r = {}
        for name, eng in (("user", user), ("builtin", builtin), ("exact", exact)):
            r[name + "_ms"], out = time_eval(eng, x, args.reps)
            r[name + "_values"] = out
        res["rounds"].append({k: v for k, v in r.items() if k.endswith("_ms")})
    for name in ("user", "builtin", "exact"):
        res[name + "_ms"] = min(r[name + "_ms"] for r in res["rounds"])
        res[name + "_pairs_per_s"] = E * N / (res[name + "_ms"] * 1e-3)
    res["user_over_exact"] = res["user_ms"] / res["exact_ms"]
    res["user_over_builtin"] = res["user_ms"] / res["builtin_ms"]
    res["max_rel_diff_user_builtin"] = float(np.max(np.abs(r["user_values"] / r["builtin_values"] - 1.0)))
    res["counts_equal_on_64_points"] = bool(np.array_equal(ubs.device_counts(lib, ubs.FAKE, user, x[:64]),
                                                           builtin.fake_counts(x[:64])[:, :300]))

    out = (ctypes.c_double * 4)()
    lib.user_fake_binned_flush_time.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_void_p]
    xc = np.ascontiguousarray(x)
    assert lib.user_fake_binned_flush_time(prepared.ctypes.data, len(prepared), xc.ctypes.data, E, args.reps,
                                           out) == 0, lib.user_binned_error()
    res["pairs_kernel_ms"], res["flush_only_worst_case_ms"] = out[0], out[1]
    res["flush_share_of_pairs_kernel_at_most"] = out[1] / out[0]
    res["resident_ctas_per_sm"], res["pairs_kernel_ctas"] = int(out[2]), int(out[3])
    shape = (ctypes.c_int64 * 3)()
    lib.user_binned_shape(ubs.FAKE, user.h, shape)
    res["cta_threads"], res["dynamic_smem_bytes"] = int(shape[0]), int(shape[1])
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
