#!/usr/bin/env python
"""bench.py -- the reference's headline metric on the reference's headline
config, on N B200s of one node.

Metric  : MH steps/s = chains x steps / time              (BASELINE.json)
Workload: example/FakeMCMC.C -- binned Poisson likelihood with
          SystematicCorrection reweighting, 4096 chains x 1 000 000 synthetic
          events PER GPU (BASELINE.json configs[1]); chains shard over GPUs
          with no data-path collective, so scaling is "weak".
A step  : one TSimpleMCMC::Step() of every chain = adaptive proposal, one
          likelihood evaluation over all events, Metropolis accept/reject.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU code

At N > 1 the line carries a second leg, "multi_gpu": the ensemble-sweep shape
(BASELINE.json configs[4], scaled to a bounded size) with the EVENTS sharded
over the GPUs -- integer event counts reduce-scattered / log-likelihoods
all-gathered over NCCL every step -- next to the same work chain-sharded, after
checking that the sharded chains are bit-identical to unsharded ones.

--config c1 | c3 | c4 print the same contract for the other BASELINE.json
configs (default c2 = the headline one):
  c1  SimpleMCMC.C / mcmc.exe schedule, 1 chain (latency-bound; steps/s only)
  c3  THorrificLogLikelihood 50-dim, 65 536 chains, per-chain adaptation (HBM-bound)
      + pooled adaptation as a sub-object
  c4  TSimpleHMC, 500-dim dense Gaussian, analytic gradient, 16 384 chains,
      contractions on the FP64 tensor cores (DMMA-bound)

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "root-simple-mcmc_b200"))
sys.path.insert(0, ROOT)

CHAINS_PER_GPU = 4096
EVENTS = 1_000_000
DIM = 9
SEED = 3
# SURVEY.md 8(d): algorithmic work of one (chain, event) pair and bytes of one
# ensemble step of the event likelihood.
FLOP_PER_PAIR = 120.0
BYTES_PER_EVENT = 32.0            # PreparedEvent, the record the pair kernel streams
BYTES_PER_CHAIN = (9 + 150) * 8.0 # parameters in, 150 bin contents out


def workload_inputs(events_n):
    """SURVEY.md 8(d) C2 inputs: 1:2 signal:background MC sample, the toy
    data of FakeData::FillData(33334, 33334); generator seed 2."""
    from smcmc_b200 import synth
    signal = events_n // 3 + (1 if events_n % 3 else 0)
    events = synth.make_mc_sample(signal, events_n - signal, seed=2)
    data = synth.make_data_histograms(33334, 33334, seed=2)
    return events, data


def start_points(chains, offset):
    """FakeMCMC.C:67: every parameter ~ U(-1, 1); chain seed 3."""
    x0 = np.zeros((chains, DIM))
    for c in range(chains):
        x0[c] = np.random.default_rng([SEED, offset + c]).uniform(-1.0, 1.0, DIM)
    return x0


# --------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML,
    the same counters as the nvidia-smi line of B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {
                pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self._stop_evt.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as exc:                      # NVML missing: report that
            self.reasons.add("nvml_unavailable:%s" % type(exc).__name__)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# --------------------------------------------------------------------------
# CPU arms (the reference's own code on the host cores)
# --------------------------------------------------------------------------
_worker = {}


def _cpu_worker_init(which, events, data, exposure, seed):
    from oracle import cpu_checkers as cc
    _worker["cc"] = cc
    _worker["which"] = which
    _worker["inputs"] = (events, data, exposure)
    _worker["seed"] = seed


def _cpu_worker_start(chain):
    cc = _worker["cc"]
    c = cc.CpuChain(_worker["which"], cc.LLH_FAKE, DIM, _worker["seed"], chain)
    c.set_fake(*_worker["inputs"])
    c.start(start_points(1, chain)[0])
    _worker["chain"] = c
    return chain


def _cpu_worker_step(nsteps):
    t = time.perf_counter()
    _worker["chain"].step(nsteps, want_x=False)
    return time.perf_counter() - t


def cpu_arm(events, data, exposure, steps, warmup, cores=None):
    """`cores` independent single-chain processes (the reference is single
    threaded and non-reentrant; independent processes are its own scale-out
    model, continue-chain.sh) each doing `steps` Metropolis steps over ALL
    events.  Returns (MH steps/s, description)."""
    from oracle import cpu_checkers as cc
    which = "ref" if cc.available("ref") else "orc"
    if which == "orc":
        cc.build(("orc",))
    cores = cores or len(os.sched_getaffinity(0))
    ctx = mp.get_context("fork")
    pools = [ctx.Pool(1, _cpu_worker_init, (which, events, data, exposure, SEED)) for _ in range(cores)]
    try:
        for r in [p.apply_async(_cpu_worker_start, (i,)) for i, p in enumerate(pools)]:
            r.get()
        if warmup:
            for r in [p.apply_async(_cpu_worker_step, (warmup,)) for p in pools]:
                r.get()
        t0 = time.perf_counter()
        for r in [p.apply_async(_cpu_worker_step, (steps,)) for p in pools]:
            r.get()
        wall = time.perf_counter() - t0
    finally:
        for p in pools:
            p.terminate()
    kind = "reference" if which == "ref" else "port"
    sample = ("%d chains (one process per host core) x %d steps x %d events of the same workload; "
              "per-chain rate is independent of the ensemble size" % (cores, steps, len(events)))
    return cores * steps / wall, {"kind": kind, "cores": cores, "sample": sample}


# --------------------------------------------------------------------------
# main arms
# --------------------------------------------------------------------------
def dist_setup(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def run_reference(args):
    rank, world, local = dist_setup(args)
    if rank != 0:
        return
    events, data = workload_inputs(args.events)
    # exposure ratio (FakeLikelihood.H:107-138) computed by the CPU code itself
    from oracle import cpu_checkers as cc
    which = "ref" if cc.available("ref") else "orc"
    if which == "orc":
        cc.build(("orc",))
    c = cc.CpuChain(which, cc.LLH_FAKE, DIM, SEED, 0)
    c.set_fake(events, data, 1.0)
    sim = c.fake_hist(np.zeros(DIM))
    exposure = float(data.sum()) / float(sim.sum())
    c.close()
    steps = max(1, args.steps)
    value, desc = cpu_arm(events, data, exposure, steps, min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": "MH steps/sec (chains x steps)", "value": value,
        "unit": "steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
        "ms_per_step": 1e3 * desc["cores"] / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "example/FakeMCMC.C binned Poisson likelihood, %d events; CPU arm runs %d "
                               "chains (one per core) instead of %d" % (args.events, desc["cores"], args.chains),
                   "events": args.events, "chains": desc["cores"], "dim": DIM},
        "cpu_baseline": dict(desc, value=value, unit="steps/s"),
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_b200(args):
    import torch
    import torch.distributed as dist
    import smcmc_b200
    from smcmc_b200 import binding, synth

    rank, world, local = dist_setup(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the MCMC step path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from smcmc_b200 import shard
    offset, chains = shard.chain_shard(world * args.chains, world, rank)     # weak scaling: args.chains per GPU
    events, data = workload_inputs(args.events)
    x0 = start_points(chains, offset)

    stream = torch.cuda.current_stream().cuda_stream
    eng = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, chains, seed=SEED, device=local, chain_offset=offset)
    eng.set_stream(stream)
    eng.set_fake_events(events)
    exposure = synth.exposure_ratio(eng, data)
    eng.set_fake_data(data, exposure)
    ok = eng.start(x0)
    assert ok.all()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def one_step():
        flush.zero_()
        eng.step(1)

    for _ in range(max(args.warmup, 3)):
        one_step()
    eng.sync()
    eng.enable_kernel_timing(True)
    eng.pair_kernel_stats(reset=True)
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin.record()
    for _ in range(args.steps):
        one_step()
    t_end.record()
    barrier()
    ms = t_begin.elapsed_time(t_end)
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0 + args.steps            # + the L2 flush memsets
    eng.sync()
    pair_ms, pair_n = eng.pair_kernel_stats(reset=True)
    eng.enable_kernel_timing(False)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * chains * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)

    # ---- end to end through the public API with host buffers -----------------
    pinned_events = torch.empty(len(events) * 48, dtype=torch.uint8, pin_memory=True)
    pinned_events.numpy()[:] = events.view(np.uint8)
    ev_host = pinned_events.numpy().view(binding.EVENT_DTYPE)
    e2e_steps = args.steps
    out = {"points": torch.empty((1, chains, DIM), dtype=torch.float64, pin_memory=True).numpy(),
           "llh_accepted": torch.empty((1, chains), dtype=torch.float64, pin_memory=True).numpy(),
           "accepted": torch.empty((1, chains), dtype=torch.int32, pin_memory=True).numpy()}
    def e2e_pass(steps):
        e = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, chains, seed=SEED, device=local, chain_offset=offset)
        e.set_stream(stream)
        barrier()
        t0 = time.perf_counter()
        e.set_fake_events(ev_host)                      # H2D 48 B/event
        ta = time.perf_counter()
        e.set_fake_data(data, exposure)
        e.start(x0)                                     # H2D chains*dim*8
        t1 = time.perf_counter()
        if os.environ.get("SMCMC_BENCH_VERBOSE"):
            sys.stderr.write("   upload %.1f ms, data+start %.1f ms\n" % ((ta - t0) * 1e3, (t1 - ta) * 1e3))
        for _ in range(steps):
            e.step_trace(1, want=("points", "llh_accepted", "accepted"), out=out)   # D2H every step
        barrier()
        t2 = time.perf_counter()
        e.close()
        return t2 - t0, t1 - t0

    for _ in range(2):                                  # untimed: first use of the upload / trace kernels,
        e2e_pass(max(args.warmup, 3))                   # allocator warm-up of a fresh process
    e2e_s, upload_s = e2e_pass(e2e_steps)
    sys.stderr.write("e2e: upload+start %.1f ms, %d traced steps %.1f ms\n"
                     % (upload_s * 1e3, e2e_steps, (e2e_s - upload_s) * 1e3))
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    h2d = (len(events) * 48 + 150 * 8 + chains * DIM * 8) / e2e_steps
    d2h = chains * (DIM * 8 + 8 + 4) + chains * 4 / e2e_steps
    e2e = {"value": world * chains * e2e_steps / e2e_s, "unit": "steps/s",
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "includes": "event upload + re-layout, Start, %d x Step(save=true) with the accepted points, "
                       "likelihoods and accept flags copied to pinned host memory every step" % e2e_steps}

    multi_gpu = None
    if world > 1 and not args.no_multi_leg:
        eng.close()
        del flush
        multi_gpu = multi_gpu_leg(args, rank, world, local, dist, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if world == 1 and not args.no_cpp_tree:
        e2e["via_cpp_tree"] = cpp_tree_leg(chains, len(events))

    # ---- roofline of the dominant kernel ------------------------------------------
    # kFakePairs is neither HBM- nor tensor-bound: every event is re-used by all
    # chains (hundreds of pair evaluations per byte of HBM traffic) and the
    # per-pair work is two exponentials plus a dozen FP32 / integer
    # instructions.  The binding resource is the special-function unit: the
    # reference's formula needs TWO exponentials per (chain, event) pair
    # (example/SystematicCorrection.H:68-74, DESIGN.md section 4.1), MUFU.EX2
    # issues 16 lanes per clock per SM, and every other pipe has headroom.
    pairs_per_launch = float(chains) * float(len(events))
    pair_warps = pairs_per_launch / 32.0
    pair_s = (pair_ms / max(pair_n, 1)) * 1e-3
    peaks, prof = {}, {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "pair_kernel_profile.json")))
    except Exception:
        pass
    props = torch.cuda.get_device_properties(local)
    sm_hz = (clocks.get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)) * 1e6
    sfu_peak = binding.measure_sfu_peak(local)                                   # G ex2/s, measured now
    sfu_nominal = props.multi_processor_count * 16 * sm_hz / 1e9                 # 16 lanes / clock / SM
    achieved = 2.0 * pairs_per_launch / pair_s / 1e9
    issue_peak = props.multi_processor_count * 4 * sm_hz / 1e9                  # G warp-inst/s
    executed = None
    if prof.get("warp_instructions_per_pair_warp"):
        executed = prof["warp_instructions_per_pair_warp"] * pair_warps / pair_s / 1e9
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    alg_bytes = len(events) * BYTES_PER_EVENT + chains * BYTES_PER_CHAIN
    traffic = None
    if prof.get("dram_bytes_per_launch") and prof.get("workload", {}).get("chains") == chains \
            and prof.get("workload", {}).get("events") == len(events):
        traffic = prof["dram_bytes_per_launch"]
    fp64_peak = binding.measure_fp64_peak(local)
    roofline = {
        "kernel": "smcmc::kFakePairs (event x chain pair kernel)",
        "bound": "sfu",
        "bound_note": "neither hbm nor tensor: %.0f pair evaluations per HBM byte; bound by the special-function "
                      "unit (2 exponentials per pair, MUFU.EX2 = 16 lanes/clock/SM)" % (pairs_per_launch / alg_bytes),
        "achieved": achieved, "peak": sfu_peak, "unit": "G ex2/s", "frac": achieved / sfu_peak,
        "algorithmic": "2 exponentials per (chain,event) pair (SystematicCorrection.H:68-74) x %.4g pairs per launch"
                       % pairs_per_launch,
        "peak_source": "measured in this run: register-resident MUFU.EX2 chains on every SM "
                       "(nominal %d SMs x 16 lanes x %.0f MHz = %.0f G/s)"
                       % (props.multi_processor_count, sm_hz / 1e6, sfu_nominal),
        "launch_ms": pair_ms / max(pair_n, 1), "launches_timed": int(pair_n),
        "kernel_share_of_step": (pair_ms / max(pair_n, 1)) / (ms / args.steps),
        "pairs_per_s": pairs_per_launch / pair_s,
        "traffic": traffic,
        "issue": {"note": "executed warp-instructions per 32 pairs from profiles/pair_kernel_profile.json "
                          "(ncu smsp__inst_executed.sum) against 1 warp-instruction/clock/SM sub-partition",
                  "executed_per_pair_warp": prof.get("warp_instructions_per_pair_warp"),
                  "achieved": executed, "peak": issue_peak, "unit": "G warp-inst/s",
                  "frac": (executed / issue_peak) if executed else None},
        "hbm": {"achieved": alg_bytes / pair_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": alg_bytes / pair_s / 1e9 / hbm_peak, "peak_source": hbm_src,
                "algorithmic_bytes": alg_bytes},
        "fp64_survey_8d": {
            "note": "SURVEY.md 8(d)'s own figure: 120 flop per (chain,event) pair against the FP64 peak.  NOT the "
                    "binding unit of this kernel: 99.94 % of the pairs are decided by an FP32 interval filter and "
                    "never reach the FP64 pipe (counts checked identical on every pair, tests/test_gpu_fullsize.py), "
                    "so the figure exceeds 1",
            "achieved": FLOP_PER_PAIR * pairs_per_launch / pair_s / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": FLOP_PER_PAIR * pairs_per_launch / pair_s / 1e12 / fp64_peak,
            "peak_source": "measured in this run (DFMA chain micro-benchmark)"},
        "fp64_of_unfiltered_algorithm": {
            "note": "the FP64 work the same counts cost WITHOUT the FP32 interval filter: 25 FP64 instructions "
                    "(50 flop) per pair, first version of this kernel; above 1.0 = faster than that roofline allows",
            "achieved": 50.0 * pairs_per_launch / pair_s / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": 50.0 * pairs_per_launch / pair_s / 1e12 / fp64_peak,
            "peak_source": "measured in this run (DFMA chain micro-benchmark)"},
    }

    # ---- the same likelihood in its streaming regime (SURVEY.md 8d): ONE chain, every event
    # read once per evaluation by kFakeStream -- the HBM-bound face of the event likelihood.
    # 16.8 M events = 268 MB of FP32 tile records: larger than the 126 MB L2.
    if world == 1 and not args.no_streaming:
        n_stream = 16777216
        sig = n_stream // 3 + 1
        ev_stream = synth.make_mc_sample(sig, n_stream - sig, seed=2)
        eng_s = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, 1, seed=SEED, device=local)
        eng_s.set_stream(stream)
        eng_s.set_fake_events(ev_stream)
        eng_s.set_fake_data(data, exposure * len(events) / float(n_stream))
        eng_s.start(start_points(1, 0))
        eng_s.step(3)
        eng_s.enable_kernel_timing(True)
        eng_s.pair_kernel_stats(reset=True)
        eng_s.step(20)
        eng_s.sync()
        s_ms, s_n = eng_s.pair_kernel_stats()
        s_sec = s_ms / max(s_n, 1) * 1e-3
        roofline["hbm_streaming"] = {
            "kernel": "smcmc::kFakeStream (the same likelihood with 1 chain: every event is read once per evaluation)",
            "bound": "hbm", "achieved": 16.0 * n_stream / s_sec / 1e9, "peak": hbm_peak, "unit": "GB/s",
            "frac": 16.0 * n_stream / s_sec / 1e9 / hbm_peak, "peak_source": hbm_src,
            "algorithmic": "16 B per event (FP32 tile record: logSigma, dLog, nomLog, separation) x %d events per launch"
                           % n_stream,
            "launch_ms": s_ms / max(s_n, 1), "launches_timed": int(s_n), "chains": 1, "events": n_stream,
            "inputs": "larger than L2 (268 MB)"}
        eng_s.close()
        del ev_stream

    cpu_value, cpu_desc = (None, None)
    if world == 1 and not args.no_cpu_baseline:
        cpu_value, cpu_desc = cpu_arm(events, data, exposure, args.cpu_steps, 1)

    line = {
        "metric": "MH steps/sec (chains x steps)", "value": value, "unit": "steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "example/FakeMCMC.C: binned Poisson likelihood with SystematicCorrection "
                               "reweighting, %d chains x %d events per GPU (BASELINE.json configs[1])"
                               % (chains, len(events)),
                   "chains_per_gpu": chains, "events": len(events), "dim": DIM, "parallelism": "chains/%d" % world,
                   "l2": "256 MiB memset between steps (inside the timed region) flushes the 126 MB L2"},
        "likelihood_evals_per_s": value,
        "event_pair_evals_per_s": value * len(events),
        "roofline": roofline,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if cpu_desc:
        line["cpu_baseline"] = dict(cpu_desc, value=cpu_value, unit="steps/s")
        line["cpu_baseline"]["gpu_over_cpu_per_core"] = value / (cpu_value / cpu_desc["cores"])
    if multi_gpu:
        line["multi_gpu"] = multi_gpu
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------
# N > 1: the ensemble-sweep shape with the events sharded over the GPUs
# --------------------------------------------------------------------------
def multi_gpu_leg(args, rank, world, local, dist, barrier):
    """BASELINE.json configs[4] ("chains and events sharded over 1/2/4/8 B200") at a bounded
    size: MG_CHAINS chains x MG_EVENTS events in total.
      event-sharded  1 x G: every rank holds ALL chains and 1/G of the events; each likelihood
                     evaluation reduce-scatters the integer count table over NCCL, each rank
                     finishes its block of chains, the log-likelihoods are all-gathered;
      chain-sharded  G x 1: every rank holds 1/G of the chains and all events, no exchange.
    Both do chains x events / G pair evaluations per rank and step.  Before timing, the first
    MG_SAMPLE chains of the sharded ensemble are compared bit for bit (likelihoods and two traced
    steps) with an unsharded engine on rank 0."""
    import torch
    import smcmc_b200
    from smcmc_b200 import binding, synth
    chains_total, events_total, sample, steps = args.mg_chains, args.mg_events, args.mg_sample, args.mg_steps
    signal = events_total // 3 + 1
    events = synth.make_mc_sample(signal, events_total - signal, seed=2)
    data = synth.make_data_histograms(33334, 33334, seed=2)
    exposure = 0.1 * 1e6 / events_total
    x0 = start_points(chains_total, 0)
    stream = torch.cuda.current_stream().cuda_stream
    dev = torch.device("cuda", local)

    def timed_steps(eng, n):
        eng.step(2)
        eng.sync()
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        eng.step(n)
        t1.record()
        barrier()
        eng.sync()
        t = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) * 1e-3 / n

    # ---- event-sharded: one event group of all ranks
    uid = [binding.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    eng = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, chains_total, seed=SEED, device=local, chain_offset=0)
    eng.set_stream(stream)
    eng.comm_init(uid[0], world, rank, event_group=world)
    eng.set_fake_events(events[rank::world])
    eng.set_fake_data(data, exposure)
    sharded_llh = eng.eval(x0[:sample])                  # collective: every rank of the group calls it
    assert eng.start(x0).all()
    tr = eng.step_trace(2, want=("accepted", "llh_accepted"))
    identical = None
    if rank == 0:
        full = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, sample, seed=SEED, device=local, chain_offset=0)
        full.set_stream(stream)
        full.set_fake_events(events)
        full.set_fake_data(data, exposure)
        full_llh = full.eval(x0[:sample])
        full.start(x0[:sample])
        ftr = full.step_trace(2, want=("accepted", "llh_accepted"))
        full.close()
        identical = bool(np.array_equal(full_llh, sharded_llh)
                         and np.array_equal(ftr["accepted"], tr["accepted"][:, :sample])
                         and np.array_equal(ftr["llh_accepted"], tr["llh_accepted"][:, :sample]))
    flag = torch.tensor([1 if (identical or rank != 0) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag.item()) != 1:
        raise SystemExit("bench.py: event-sharded chains differ from the unsharded evaluation")
    t_event = timed_steps(eng, steps)
    eng.close()

    # ---- chain-sharded: the same total work, no exchange
    per = chains_total // world
    eng = smcmc_b200.Engine(smcmc_b200.LLH_FAKE, DIM, per, seed=SEED, device=local, chain_offset=rank * per)
    eng.set_stream(stream)
    eng.set_fake_events(events)
    eng.set_fake_data(data, exposure)
    assert eng.start(x0[rank * per:(rank + 1) * per]).all()
    t_chain = timed_steps(eng, steps)
    eng.close()
    pairs = float(chains_total) * float(events_total)
    per_rank = -(-chains_total // world)
    block = -(-per_rank // 256) * 256              # chains per reduce-scatter block
    return {
        "workload": "ensemble sweep of the event likelihood (BASELINE.json configs[4] shape, bounded): %d chains x %d "
                    "events in total over %d GPUs" % (chains_total, events_total, world),
        "nccl_ranks": world,
        "bit_identical_to_unsharded": True,
        "checked": "likelihoods of %d chains and two traced Metropolis steps (accept flags, accepted likelihoods) "
                   "against an unsharded engine on rank 0" % sample,
        "event_sharded": {"layout": "1 x %d (every rank: all chains, 1/%d of the events)" % (world, world),
                          "s_per_step": t_event, "pair_evals_per_s": pairs / t_event, "steps_per_s": chains_total / t_event,
                          "exchange": "ncclReduceScatter of 450 x %d uint32 event counts + ncclAllGather of %d f64 "
                                      "log-likelihoods per evaluation" % (block * world, block * world),
                          "bytes_reduce_scattered_per_step": 450 * block * world * 4,
                          "bytes_all_gathered_per_step": block * world * 8},
        "chain_sharded": {"layout": "%d x 1 (every rank: 1/%d of the chains, all events)" % (world, world),
                          "s_per_step": t_chain, "pair_evals_per_s": pairs / t_chain, "steps_per_s": chains_total / t_chain,
                          "exchange": "none"},
        "event_vs_chain_sharded": t_chain / t_event,
        "steps_timed": steps,
    }


def cpp_tree_leg(chains, events_n):
    """"Accepted points written to the user's TTree" at the benchmark's size, through the C++
    mirror of the reference API (include/TSimpleMCMC.H): tests/cpp/simple_mcmc.cc `tree` mode runs
    Step(true) with a tree attached -- one synchronous device read of the step's record and one
    TTree::Fill per chain -- and StepMany() without one."""
    import re
    import subprocess
    import tempfile
    libdir = os.path.join(ROOT, "root-simple-mcmc_b200", "smcmc_b200")
    src = os.path.join(ROOT, "tests", "cpp", "simple_mcmc.cc")
    try:
        # compiled outside the source tree, which may be read-only
        with tempfile.TemporaryDirectory(prefix="smcmc_bench_") as tmp:
            exe = os.path.join(tmp, "simple_mcmc")
            subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-o", exe, src,
                            "-L", libdir, "-lsmcmc_b200", "-Wl,-rpath," + libdir], check=True)
            r = subprocess.run([exe, "tree", str(chains), "10", str(max(1, events_n // 30))], capture_output=True,
                               text=True, check=True, timeout=600)
        m = re.search(r"events (\d+) ms_per_step_plain (\S+) ms_per_step_tree (\S+) full_save_ms (\S+) entries (\d+)", r.stdout)
        plain, tree = float(m.group(2)), float(m.group(3))
        return {"value": chains / (tree * 1e-3), "unit": "steps/s", "ms_per_step_with_tree": tree,
                "ms_per_step_without_tree": plain, "events": int(m.group(1)), "tree_entries": int(m.group(5)),
                "full_state_save_ms": float(m.group(4)),
                "note": "sMCMC::TSimpleMCMC<FakeLikelihood>::Step(true) with a TTree attached (in-memory TTree of "
                        "include/smcmc_tree.h; ROOT is not installed): one TTree::Fill per chain and step on the host"}
    except Exception as exc:                          # reported, never fatal for the headline line
        return {"unavailable": "%s: %s" % (type(exc).__name__, exc)}


DUMP_MAX_CHAINS = 262144          # x (2 x 9 + 3) float64 per chain = 44 MB


def dump_outputs(out_dir, eng):
    """What the last timed step left for a caller of the step path, one .npy per array: every
    chain's accepted point and likelihood, the point it proposed and its likelihood, and its
    proposal step size (4096 chains: 0.7 MB in float64).  Above DUMP_MAX_CHAINS chains a fixed
    seeded sample of them is written, with their indices in chain_index.npy.  At a fixed
    --steps and --warmup the inputs and the number of steps taken (max(--warmup, 3) + --steps)
    are the same on every run, so two builds can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    eng.sync()
    keep = slice(None)
    if eng.chains > DUMP_MAX_CHAINS:
        keep = np.sort(np.random.default_rng(0).choice(eng.chains, DUMP_MAX_CHAINS, replace=False))
        np.save(os.path.join(out_dir, "chain_index.npy"), keep.astype(np.float64))
    for name, field in (("accepted_points", "accepted"), ("accepted_llh", "accepted_llh"),
                        ("proposed_points", "proposed"), ("proposed_llh", "proposed_llh"),
                        ("sigma", "sigma")):
        np.save(os.path.join(out_dir, name + ".npy"), eng.get(field)[keep].astype(np.float64))


_RESULT_OUT = None


def emit(line):
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU, help="chains per GPU")
    ap.add_argument("--events", type=int, default=EVENTS)
    ap.add_argument("--cpu-steps", type=int, default=12, help="steps of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-streaming", action="store_true",
                    help="skip the 1-chain x 16.8M-event streaming measurement (roofline.hbm_streaming)")
    ap.add_argument("--no-cpp-tree", action="store_true", help="skip e2e.via_cpp_tree (the compiled C++ program)")
    ap.add_argument("--no-multi-leg", action="store_true", help="N > 1: skip the event-sharded leg (multi_gpu)")
    ap.add_argument("--mg-chains", type=int, default=32768, help="multi_gpu leg: chains in total")
    ap.add_argument("--mg-events", type=int, default=8388608, help="multi_gpu leg: events in total")
    ap.add_argument("--mg-sample", type=int, default=4096, help="multi_gpu leg: chains compared with the unsharded engine")
    ap.add_argument("--mg-steps", type=int, default=5)
    ap.add_argument("--c4-chains", type=int, default=16384, help="--config c4: chains per GPU")
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4"],
                    help="which BASELINE.json config to measure (default c2, the headline one)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the chains' state after the last step as DIR/<name>.npy "
                         "(default config, rank 0's chains); fixed by --steps and --warmup, where any --warmup "
                         "below 3 runs 3 warm-up steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != "c2" or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for the default config of the b200 arm")
    # stdout carries exactly ONE line, the JSON result: anything else that writes to file
    # descriptor 1 (NCCL prints its version banner there when the first communicator is
    # made, child processes inherit it) is sent to stderr; emit() writes to the saved descriptor
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.config != "c2":
        import bench_configs
        bench_configs.run(args, emit, ClockSampler)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
