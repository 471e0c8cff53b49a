"""N-GPU bit-identity of the window-sharded long-video driver as a pytest (driver-visible): launches
tests/multi_gpu_check.py under torchrun on every GPU of the box and requires both exchange forms (two-phase with the
fused alignment chain, to rank 0 and to the last rank; the gather of ranks on several hosts) to reproduce the
single-GPU `infer_video_depth` bit for bit.  30 frames are two windows: with 3 or more GPUs some ranks hold none.
Skips on boxes with fewer than two GPUs; the world-2/3/4 gloo tests in test_parallel_cpu.py cover the host logic
everywhere."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("frames", [30, 100, 230])
def test_sharded_video_is_bit_identical_to_one_gpu(frames):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(n, 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env={**os.environ, "VDA_FRAMES": str(frames)})
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-3000:])
    assert out.stdout.count("bit-identical") == 3, out.stdout[-2000:]
