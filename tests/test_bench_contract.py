"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the required keys,
and the own arm refuses to run (non-zero exit, no JSON) when there is no B200 -- it never falls back to the CPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "matrices/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_own_arm_needs_a_gpu():
    import ctypes

    from linalg_b200 import _native

    n = ctypes.c_int(0)
    if _native.load_library().lq_device_count(ctypes.byref(n)) == 0 and n.value > 0:
        pytest.skip("a GPU is visible here")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3", "--no-cpu"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert out.stdout.strip() == ""          # no JSON line from a machine without the device
    assert "no CPU fallback" in out.stderr


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and out.stdout.strip() == "" and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_steps_factors(tmp_path):
    """--dump-outputs writes Q and R of the timed path for a seeded sample of the batch; they factor the seeded inputs."""
    import numpy as np

    batch = 4096
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", str(batch),
                          "--no-extras", "--no-cpu", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout)
    assert line["steps"] == 2 and line["gpu_launches"] == 2
    assert sorted(os.listdir(tmp_path)) == ["Q.npy", "R.npy"]
    Q, R = np.load(tmp_path / "Q.npy"), np.load(tmp_path / "R.npy")
    assert Q.dtype == R.dtype == np.float64 and Q.shape == R.shape == (2048, 32, 32)
    assert Q.nbytes + R.nbytes <= 64 << 20
    idx = np.sort(np.random.default_rng(0).choice(batch, size=2048, replace=False))
    A = np.random.default_rng(2).standard_normal((batch, 32, 32))[idx]
    assert np.max(np.linalg.norm(A - Q @ R, axis=(1, 2)) / np.linalg.norm(A, axis=(1, 2))) <= 1e-12
    assert np.all(np.tril(R, -1) == 0.0)
