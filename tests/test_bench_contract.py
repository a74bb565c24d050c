"""bench.py's output contract, on the arm that runs without a GPU (--impl reference: the oracle port timed on the host
cores): stdout is exactly ONE JSON line carrying the result's keys; everything else goes to stderr.  On the GPU:
--dump-outputs writes what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--cpu-sample", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert res.returncode == 0, res.stderr[-2000:]
    assert res.stdout.strip() == ""


def test_steps_and_dump_outputs_are_checked():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"],
                  ["--workload", "large-n", "--dump-outputs", "unused"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=600, cwd=ROOT)
        assert res.returncode == 2 and res.stdout.strip() == "", (extra, res.stderr[-2000:])


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_steps_outputs(tvf, tmp_path):
    """--dump-outputs writes the outputs of the timed path's last step; with fewer trials than the sample size that is
    every trial, and each equals what the pose API returns for the same (seeded) inputs."""
    from tft_vs_fund_b200 import scene
    B = 3000
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--trials", str(B),
                          "--legs", "headline", "--no-cpu-baseline", "--large-n-scenes", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout)["steps"] == 2
    out = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    shapes = {"trial": (B,), "R_t_2": (B, 12), "R_t_3": (B, 12), "Reconst": (B, 60), "T": (B, 27), "repr_err": (B,), "status": (B,)}
    assert {k: v.shape for k, v in out.items()} == shapes and all(v.dtype == np.float64 for v in out.values())
    assert sum(v.nbytes for v in out.values()) <= 64 * 10 ** 6
    assert np.array_equal(out["trial"], np.arange(B))
    d = scene.sweep_batch(B, 20)
    ref = tvf.LinearTFTPoseEstimation(d["Corresp"], d["CalM"], device=0)
    assert np.array_equal(out["repr_err"], ref.repr_err) and np.array_equal(out["status"], ref.status)
