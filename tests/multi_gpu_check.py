#!/usr/bin/env python
"""N-GPU check of the window-sharded driver (run under torchrun on a multi-GPU box):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \\
        tests/multi_gpu_check.py

Every rank computes its block of windows of a synthetic video; the sharded result is compared with the single-GPU
result of the same model on the rank that receives it: windows are independent in model compute and the kernels are
batch-invariant, so the two must be bit-identical.  Three runs: the two-phase form to rank 0 and to the last rank, and
the gather form of ranks on several hosts, forced on this one host by replacing `parallel._same_host`."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, synth_state_dict  # noqa: E402
from video_depth_anything_b200 import parallel  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    enc = os.environ.get("VDA_ENCODER", "vits")
    m = VideoDepthAnything(**MODEL_CONFIGS[enc], dtype=torch.bfloat16)
    m.load_state_dict(synth_state_dict(**MODEL_CONFIGS[enc], seed=0))
    m.to(f"cuda:{local}")
    n = int(os.environ.get("VDA_FRAMES", "100"))
    frames = np.random.default_rng(0).integers(0, 256, (n, 98, 126, 3), dtype=np.uint8)
    world = dist.get_world_size()
    ref = m.infer_video_depth(frames, 24, input_size=98, device=f"cuda:{local}")[0] if rank in (0, world - 1) else None
    for form, dst in (("two_phase", 0), ("two_phase", world - 1), ("gather", 0)):
        if form == "gather":
            parallel._same_host = lambda group: False
        out, _ = parallel.infer_video_depth_sharded(m, frames, 24, input_size=98, dst=dst)
        if rank == dst:
            same = np.array_equal(out, ref)
            print(f"multi_gpu_check[{form} -> rank {dst}]: world {world} frames {n} windows {-(-n // 22)}: "
                  f"{'bit-identical' if same else 'MISMATCH max abs ' + str(np.abs(out - ref).max())}", flush=True)
            assert same
        else:
            assert out is None
        dist.barrier()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
