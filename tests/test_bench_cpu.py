"""CPU: the reference arm of bench.py (`--impl reference`, the oracle port on the host cores) prints one JSON line
with the contract's keys; run on a tiny sample (vits, one frame) so the whole test takes seconds."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--encoder", "vits",
                          "--steps", "1", "--warmup", "0", "--cpu-frames", "1"], capture_output=True, text=True,
                         timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "frames/s" and d["unit"] == "frames/s" and d["higher_is_better"]
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env={**os.environ, "RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_sample_fits_the_budget_and_config_matches_the_gpu_arm():
    sys.path.insert(0, ROOT)
    import bench
    # 25 passes in 200 s at 0.9 frames/s -> 7 frames per pass; never more than the window, never less than one frame
    assert bench.reference_sample_frames("vitl", 20, 5, 200.0, 0.9) == 7
    assert bench.reference_sample_frames("vits", 1, 0, 200.0, 30.0) == 32
    assert bench.reference_sample_frames("vitl", 200, 50, 60.0, 0.5) == 1
    # the driver compares the two arms' config objects
    assert bench.workload_config("vitl", 4) == bench.workload_config("vitl", 4)
    assert "1x32x518x518" in bench.workload_config("vitl", 1)["workload"]


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=120, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]


def test_reference_arm_honours_steps_and_warmup():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--encoder", "vits",
                          "--steps", "2", "--warmup", "1", "--cpu-frames", "1"], capture_output=True, text=True,
                         timeout=600, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    sys.path.insert(0, ROOT)
    import bench
    assert d["steps"] == 2 and d["warmup"] == 1 and d["config"] == bench.workload_config("vits", 1)
