"""bench.py's output contract: `--impl reference` (no GPU needed) prints exactly ONE line on
stdout, a JSON object with the result's keys; `--dump-outputs` (GPU) writes the same arrays on
every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    from oracle import cpu_checkers as cc
    assert cc.available("ref") or cc.available("orc")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--events", "20000"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["metric"].startswith("MH steps/sec") and d["unit"] == "steps/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["data"] == "synthetic" and d["dtype"] == "f64"


def test_reference_arm_of_the_other_configs():
    """`bench.py --impl reference --config c1|c3|c4`: one JSON line each with the contract's keys."""
    for config, metric in (("c1", "MH steps/sec"), ("c3", "MH steps/sec"), ("c4", "HMC steps/sec")):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", config,
                            "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = [l for l in r.stdout.splitlines() if l.strip()]
        assert len(lines) == 1, r.stdout
        d = json.loads(lines[0])
        assert d["impl"] == "reference" and d["metric"].startswith(metric) and d["value"] > 0
        assert d["cpu_baseline"]["cores"] >= 1 and d["e2e"]["d2h_bytes_per_step"] == 0
        assert "workload" in d["config"] and d["vs_baseline"] is None


@pytest.mark.gpu
def test_dump_outputs_are_the_same_on_every_run(tmp_path):
    """`--dump-outputs DIR`: the chains' state after the last timed step as float .npy files,
    identical for two runs with the same arguments, and different after one more timed step."""
    dumps = []
    for run, steps in (("a", 2), ("b", 2), ("c", 3)):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                            "--chains", "256", "--events", "30000", "--no-cpu-baseline", "--no-streaming",
                            "--no-cpp-tree", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == steps
        dumps.append({f: np.load(out / f) for f in sorted(os.listdir(out))})
    a, b, c = dumps
    assert sorted(a) == ["accepted_llh.npy", "accepted_points.npy", "proposed_llh.npy", "proposed_points.npy",
                         "sigma.npy"]
    assert a["accepted_points.npy"].shape == (256, 9) and a["accepted_llh.npy"].shape == (256,)
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name], equal_nan=True), name
    assert np.all(np.isfinite(a["accepted_points.npy"])) and np.all(np.isfinite(a["accepted_llh.npy"]))
    # the third timed step proposes a new point for every chain, and some of the 256 chains accept it
    assert not np.any(np.all(c["proposed_points.npy"] == a["proposed_points.npy"], axis=1))
    assert not np.array_equal(c["accepted_llh.npy"], a["accepted_llh.npy"])


def test_bench_refuses_to_run_the_gpu_arm_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    for extra in ([], ["--config", "c3"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"] + extra,
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
