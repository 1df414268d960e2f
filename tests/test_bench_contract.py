"""bench.py's contract on CPU: the reference arm (`--impl reference`, the reference's CPU
path = the oracle port on the host cores) prints ONE JSON line with the keys the driver
reads; our arm has no CPU fallback and must fail without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=300, env=dict(os.environ, **(env or {})))


def test_reference_arm_prints_the_contract_line():
    out = _bench("--impl", "reference", "--n", "128", "--iters", "5", "--steps", "2", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["dtype"] == "f64"
    assert line["metric"].startswith("instance-EP-iterations/s") and line["unit"] == "instance-iterations/s"
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 1 and line["vs_baseline"] is None
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["gpu_launches"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]
    base = line["cpu_baseline"]
    assert base["kind"] == "port" and base["cores"] >= 1 and base["value"] == line["value"] and base["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    # the line describes what was timed: `steps` steps of the winning mode, ms_per_step their mean
    # (the rate follows from the units of one step), and the same arm with the SVD counted
    procs = os.cpu_count() or 1
    units = 5 * (procs if "one process" in base["sample"] else 1)       # instance-iterations of one step
    assert abs(line["value"] - units / (line["ms_per_step"] / 1e3)) <= 1e-6 * line["value"]
    assert 0 < line["incl_setup"]["value"] < line["value"]


def test_reference_arm_runs_on_rank_zero_only():
    """Under torchrun the other ranks exit 0 without work and without output."""
    out = _bench("--impl", "reference", "--gpus", "2", "--iters", "5", "--steps", "1", "--warmup", "0",
                 env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_our_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = _bench("--steps", "1", "--warmup", "0", "--instances", "1", "--n", "64", "--iters", "2")
    assert out.returncode != 0
    assert not any(ln.startswith("{") for ln in out.stdout.splitlines())


def test_arguments_that_would_not_time_or_dump_what_they_say_are_rejected(tmp_path):
    out = _bench("--impl", "reference", "--steps", "0")
    assert out.returncode == 2 and "--steps" in out.stderr
    out = _bench("--impl", "reference", "--dump-outputs", str(tmp_path / "out"))
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
    assert not (tmp_path / "out").exists()


def test_dump_outputs_writes_float64_and_a_fixed_sample_over_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.RandomState(1)
    arrays = {"x_r": rng.rand(40, 30), "x_v": rng.rand(40), "mse_per_iter": rng.rand(40, 5).astype(np.float32)}
    bench.dump_outputs(np, str(tmp_path / "all"), arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / (name + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * 36 * 8)         # 10 of the 40 instances (36 values each)
    for d in ("s1", "s2"):
        bench.dump_outputs(np, str(tmp_path / d), arrays)
    x_r = np.load(tmp_path / "s1" / "x_r.npy")
    keep = [int(np.flatnonzero((arrays["x_r"] == row).all(axis=1))[0]) for row in x_r]
    assert len(keep) == 10 and keep == sorted(keep)
    for name, a in arrays.items():
        s1, s2 = np.load(tmp_path / "s1" / (name + ".npy")), np.load(tmp_path / "s2" / (name + ".npy"))
        assert np.array_equal(s1, np.asarray(a, dtype=np.float64)[keep]) and np.array_equal(s1, s2)
