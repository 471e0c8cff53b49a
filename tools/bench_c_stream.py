#!/usr/bin/env python
"""Stream groups through the C library (cmodel.CStreamGroup: the C planner and vda_stream_step, one CUDA graph per
(bucket, causal)) against the Python DepthStreamGroup on the same weights, in one run; prints one JSON line and writes it
to --out.

Arms (ViT-L, bf16, 518x518 uint8 CUDA frames, depths returned as CUDA tensors on both sides, so both paths do the same
copies and run the same kernels and only the host work differs):
  * 1 stream, one frame per push;
  * 8 streams, every push names every stream (bucket 8);
  * 1 stream pushing stacks of 8 consecutive frames (causal step, bucket 8).
Per arm: --warmup pushes on each path (captures the graphs; the context is full after 31 frames), then --pushes timed
pushes per path, alternating which path goes first, host clock around each push (a push synchronises).  Reported: push
p50 / p99 per path and the C path's p50 difference.
Launches per step: the Python group's count of its captured graph (Engine.run_graphed), and the kernels torch.profiler lists
for one eager step of each path (graphs off; copies and memsets not counted).
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, synth_state_dict  # noqa: E402
from video_depth_anything_b200.cmodel import CModel, CStreamGroup  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"card": q.split(",")[0].strip() if q else torch.cuda.get_device_name(0),
            "power_limit": q.split(",")[1].strip() if "," in q else "unknown"}


def pct(xs, p):
    return float(np.percentile(np.asarray(xs), p))


class Arm:
    """One group on one path with its own streams and a frame cursor per stream."""

    def __init__(self, group, frames, S, k, python):
        self.g, self.frames, self.k, self.python = group, frames, k, python
        self.hs = [group.open() for _ in range(S)]
        self.t = 0

    def push(self):
        n = self.frames.shape[0]
        if self.k > 1:
            a = self.t % (n - self.k)
            push = {self.hs[0]: self.frames[a:a + self.k]}
        else:
            push = {h: self.frames[(self.t + i) % n] for i, h in enumerate(self.hs)}
        self.t += self.k
        return self.g.push(push, to_host=False) if self.python else self.g.push(push)


def kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return len([n for n in names if not n.startswith(("Memcpy", "Memset"))])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--pushes", type=int, default=300)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "c_stream_b200.json"))
    args = ap.parse_args()
    enc, dtype = "vitl", torch.bfloat16
    sd = synth_state_dict(**MODEL_CONFIGS[enc], seed=0)
    m = VideoDepthAnything(**MODEL_CONFIGS[enc], dtype=dtype)
    m.load_state_dict(sd)
    m.to("cuda")
    cm = CModel(**MODEL_CONFIGS[enc], dtype=dtype)
    cm.load_state_dict(sd)
    frames = torch.from_numpy(np.random.default_rng(0).integers(0, 256, (64, 518, 518, 3), dtype=np.uint8)).cuda()
    res = {"tool": "bench_c_stream", "encoder": enc, "dtype": "bf16", "frame": [518, 518], **card(), "arms": []}
    for name, S, k in (("1 stream", 1, 1), ("8 streams", 8, 1), ("1 stream, stacks of 8", 1, 8)):
        py = Arm(m.stream_group(S), frames, S, k, True)
        cs = Arm(CStreamGroup(cm, S), frames, S, k, False)
        for _ in range(args.warmup):
            py.push()
            cs.push()
        times = {"python": [], "c": []}
        for i in range(args.pushes):
            for arm, key in ((py, "python"), (cs, "c")) if i % 2 else ((cs, "c"), (py, "python")):
                t0 = time.perf_counter()
                arm.push()
                times[key].append(time.perf_counter() - t0)
        bk, causal = (8 if S == 8 or k == 8 else 1), k > 1
        graph_launches = (py.g.causal_graphs if causal else py.g.graphs)[bk][3]
        # eager steps under the profiler: every kernel is listed (the groups' first steps ran above, so no lazy state)
        py.g.engine.use_graphs = False
        try:
            py_kernels = kernels_of(py.push)
        finally:
            py.g.engine.use_graphs = True
        cs.g.use_graphs = False
        c_kernels = kernels_of(cs.push)
        row = {"arm": name, "streams": S, "frames_per_push": S * k, "bucket": bk, "causal": causal,
               "push_ms_p50": {p: 1e3 * pct(v, 50) for p, v in times.items()},
               "push_ms_p99": {p: 1e3 * pct(v, 99) for p, v in times.items()},
               "c_minus_python_p50_ms": 1e3 * (pct(times["c"], 50) - pct(times["python"], 50)),
               "frames_per_s_p50": {p: S * k / pct(v, 50) for p, v in times.items()},
               "launches": {"python_graph": graph_launches, "python_eager_kernels": py_kernels, "c_eager_kernels": c_kernels}}
        res["arms"].append(row)
        print(json.dumps(row), file=sys.stderr)
        py.g.close()
        cs.g.close()
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
