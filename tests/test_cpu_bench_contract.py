"""bench.py without a GPU: the reference arm (the reference's CPU torch program, oracle/torch_port.py) prints ONE JSON
line with the contract's keys on a tiny configuration, times the requested number of steps and dumps what its last
step returned; the argument checks and the sampling of --dump-outputs.  (The hitgeom arm needs a CUDA device.)"""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--points", "256", *extra], capture_output=True, text=True, timeout=600,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    d = _run()
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["metric"] == "point-pair distance evals/sec (fwd+bwd)" and d["unit"] == "pair-evals/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_is_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr, out.stderr[-2000:]


def test_reference_arm_dumps_its_last_step(tmp_path):
    d = _run("--dump-outputs", str(tmp_path))
    loss, grad = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "grad.npy")
    assert d["steps"] == 1 and loss.dtype == grad.dtype == np.float32
    assert grad.shape[1:] == (256, 3) and np.isfinite(grad).all() and np.isfinite(loss).all()


def test_reference_hitadv_arm_times_the_requested_steps_and_dumps(tmp_path):
    d = _run("--workload", "hitadv", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 1 and "1 iterations" in d["cpu_baseline"]["sample"]
    adv, succ = np.load(tmp_path / "adv.npy"), np.load(tmp_path / "success.npy")
    assert adv.dtype == np.float64 and adv.shape == (8, 256, 3) and succ.shape == () and 0 <= succ <= 8


def test_dump_outputs_samples_whole_clouds_with_a_fixed_seed(tmp_path, monkeypatch):
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    B, N = 50, 8
    grad = np.arange(B * N * 3, dtype=np.float32).reshape(B, N, 3)
    monkeypatch.setattr(bench, "DUMP_ARRAY_BYTES", 10 * N * 3 * 4)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), grad=torch.from_numpy(grad), loss=np.float64(1.5), idx=np.arange(3))
    a, b = np.load(tmp_path / "a" / "grad.npy"), np.load(tmp_path / "b" / "grad.npy")
    assert a.shape == (10, N, 3) and a.nbytes <= bench.DUMP_ARRAY_BYTES and np.array_equal(a, b)
    clouds = (a[:, 0, 0] // (N * 3)).astype(int)
    assert len(set(clouds)) == 10 and np.array_equal(a, grad[clouds])  # whole clouds, each once, in order
    assert np.load(tmp_path / "a" / "loss.npy").dtype == np.float64
    assert np.load(tmp_path / "a" / "idx.npy").dtype == np.float32
