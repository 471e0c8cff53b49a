"""GPU: `bench.py --dump-outputs` writes exactly what the timed calls return -- the last timed window's depth map and a
seeded sample of the long-video result -- as float32 .npy files, bit-identical to the public API run on the same
seeded weights and inputs; `--steps` is the step count of every per-step arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_timed_results(tmp_path):
    from e2e_checks import build_model
    n_video = 40
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--encoder", "vits", "--steps", "2",
                          "--warmup", "1", "--video-frames", str(n_video), "--no-e2e",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2           # --steps sets every per-step arm, the extra configurations included
    assert {k: (v.get("steps"), v.get("error")) for k, v in line["other_configs"].items()} == \
        {"metric924": (2, None), "vits8clips": (2, None)}
    assert sorted(os.listdir(tmp_path)) == ["depth.npy", "video_depth.npy"]
    depth, video = np.load(tmp_path / "depth.npy"), np.load(tmp_path / "video_depth.npy")
    assert depth.dtype == video.dtype == np.float32 and depth.nbytes + video.nbytes <= 64 << 20
    assert depth.shape == (1, 32, 518, 518) and video.shape == (8, 518, 518)

    m, _ = build_model("vits", 0, torch.bfloat16)
    x = torch.randn(1, 32, 3, 518, 518, generator=torch.Generator().manual_seed(1234))
    assert np.array_equal(depth, m.forward(x.cuda()).cpu().numpy())
    base = np.random.default_rng(0).integers(0, 256, (64, 518, 518, 3), dtype=np.uint8)
    full, _ = m.infer_video_depth(base[np.arange(n_video) % 64], 24, device="cuda")
    pick = np.sort(np.random.default_rng(0).choice(n_video, 8, replace=False))
    assert np.array_equal(video, full[pick])
