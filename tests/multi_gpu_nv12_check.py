#!/usr/bin/env python
"""N-GPU check of the window-sharded driver on NV12 frames (run under torchrun on a multi-GPU box, as
tests/multi_gpu_check.py): the sharded result of an NV12 video must be bit-identical to the single-GPU
`infer_video_depth` of the same frames, in both exchange forms."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import yuv_oracle as Y  # noqa: E402
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, synth_state_dict  # noqa: E402
from video_depth_anything_b200 import parallel  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    m = VideoDepthAnything(**MODEL_CONFIGS["vits"], dtype=torch.bfloat16)
    m.load_state_dict(synth_state_dict(**MODEL_CONFIGS["vits"], seed=0))
    m.to(f"cuda:{local}")
    n = int(os.environ.get("VDA_FRAMES", "100"))
    frames = Y.random_video(n, 98, 126, "nv12", seed=0)
    world = dist.get_world_size()
    ref = m.infer_video_depth(frames, 24, input_size=98, device=f"cuda:{local}", pixel_format="nv12")[0] \
        if rank in (0, world - 1) else None
    for form, dst in (("two_phase", 0), ("two_phase", world - 1), ("gather", 0)):
        if form == "gather":
            parallel._same_host = lambda group: False
        out, _ = parallel.infer_video_depth_sharded(m, frames, 24, input_size=98, dst=dst, pixel_format="nv12")
        if rank == dst:
            same = np.array_equal(out, ref)
            print(f"multi_gpu_nv12_check[{form} -> rank {dst}]: world {world} frames {n}: "
                  f"{'bit-identical' if same else 'MISMATCH max abs ' + str(np.abs(out - ref).max())}", flush=True)
            assert same
        else:
            assert out is None
        dist.barrier()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
