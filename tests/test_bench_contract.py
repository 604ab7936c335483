"""bench.py contract checks that need no GPU: the reference arm runs on the host cores, prints exactly one JSON line on stdout
with the keys the driver reads, and the GPU arm's argument surface exists."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    env = dict(os.environ, SO_BENCH_CACHE="")                       # no cache side effects from the test suite
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0",
                          "--ref-scans", "1", "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "scans/s" and d["higher_is_better"] is True and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]
    # --dump-outputs: the last step's per-scan results, float64, one row per scan
    pose, status = np.load(tmp_path / "out" / "pose.npy"), np.load(tmp_path / "out" / "status.npy")
    assert pose.dtype == np.float64 and pose.shape == (1, 7) and abs(np.linalg.norm(pose[0, 3:]) - 1) < 1e-9
    assert status.tolist() == [0.0] and np.load(tmp_path / "out" / "cov.npy").shape == (1, 36)


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", SO_BENCH_CACHE="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_cli_surface():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl"):
        assert flag in out.stdout
