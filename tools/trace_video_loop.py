#!/usr/bin/env python
"""Host-side time per phase of the long-video loop (debug): monkeypatches the phases of infer_video_depth with wall-clock
accumulators for a block of windows computed with raw_only (the sharded driver's per-rank path) or aligned by the
driver's own WindowAligner."""
import os
import sys
import time
from collections import defaultdict

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, synth_state_dict, video_depth  # noqa: E402

acc = defaultdict(float)


def timed(obj, name, label):
    fn = getattr(obj, name)

    def wrapper(*a, **k):
        t = time.perf_counter()
        r = fn(*a, **k)
        acc[label] += time.perf_counter() - t
        return r
    setattr(obj, name, wrapper)


timed(video_depth.FrameUploader, "ensure", "upload.ensure")
timed(video_depth.FeatureCache, "window", "cache.window")
timed(video_depth.WindowAligner, "push", "aligner.push")
timed(torch.Tensor, "clone", "clone")

m = VideoDepthAnything(**MODEL_CONFIGS["vitl"], dtype=torch.bfloat16)
m.load_state_dict(synth_state_dict(**MODEL_CONFIGS["vitl"], seed=0))
m.to("cuda")
base = np.random.default_rng(0).integers(0, 256, (64, 518, 518, 3), dtype=np.uint8)
frames = base[np.arange(2048) % 64]
m.infer_video_depth(frames[:66], 24)
for ids, raw in ((range(0, 47), True), (range(47, 94), True), (range(47, 94), False)):
    acc.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = m.infer_video_depth(frames, 24, window_ids=list(ids), raw_only=raw)
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    print(f"windows {ids.start}..{ids.stop - 1} raw_only={raw}: enqueue {1e3 * (t1 - t0):.0f} ms, +sync {1e3 * (t2 - t0):.0f} ms; " +
          ", ".join(f"{k} {1e3 * v:.0f}" for k, v in acc.items()), flush=True)
    out = None
