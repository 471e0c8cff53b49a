#!/usr/bin/env python
"""YUV 4:2:0 ingest (NV12 / I420 frames as video decoders give them) against packed RGB, in one run; writes
profiles/ingest_b200.json (or --out) and prints one JSON line.

  1. The ingest kernel alone: 8 frames of 1920x1080 and of 1280x720 -> 518x924 (the network size of both), RGB
     (vda_preprocess_frames), NV12 and I420 (vda_preprocess_frames_yuv); CUDA events around --launches back-to-back
     launches, the three formats alternated over --rounds rounds, median per launch.  The source frames (8 x 3 or
     8 x 1.5 bytes per pixel: 12-50 MB) stay in the 126 MB L2 across launches.
  2. Stream-group pushes (ViT-S, bf16, --encoder): 8 and 16 cameras, half 1280x720 and half 1920x1080, every push names
     every camera; host frames (numpy) and CUDA frames, RGB groups against NV12 groups, the two alternated push by push
     after --warmup pushes each; host clock around each push (a push synchronises), p50 / p99 over --pushes pushes.
  3. infer_video_depth on a 1280x720 video of --video-frames frames (ViT-S, bf16): RGB frames against NV12 frames (host
     arrays), alternated, best of --video-reps calls each; video frames per second.  The two results must be
     bit-identical (checked).
Frames are random (NV12 noise; the RGB arms get cv2.cvtColor of the same frames).  The card's name and power limit are
read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, ops, synth_state_dict  # noqa: E402

SIZES = {"720p": (720, 1280), "1080p": (1080, 1920)}
NET = (518, 924)


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"card": q.split(",")[0].strip() if q else torch.cuda.get_device_name(0),
            "power_limit": q.split(",")[1].strip() if "," in q else "unknown"}


def nv12_frames(n, h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (n, 3 * h // 2, w), dtype=np.uint8)


def to_rgb(frames, fmt="nv12"):
    code = cv2.COLOR_YUV2RGB_NV12 if fmt == "nv12" else cv2.COLOR_YUV2RGB_I420
    return np.stack([cv2.cvtColor(f, code) for f in frames])


def kernel_arm(launches, rounds):
    out = {}
    for name, (h, w) in SIZES.items():
        yuv = nv12_frames(8, h, w, seed=1)
        rgb = torch.from_numpy(to_rgb(yuv)).cuda()
        dev = torch.from_numpy(yuv).cuda()
        idx = torch.arange(8, dtype=torch.int32, device="cuda")
        calls = {"rgb": lambda: ops.preprocess_frames(rgb, idx, *NET),
                 "nv12": lambda: ops.preprocess_frames_yuv(dev, idx, 1, *NET),
                 "i420": lambda: ops.preprocess_frames_yuv(dev, idx, 2, *NET)}   # (same bytes read as I420)
        times = {k: [] for k in calls}
        for f in calls.values():
            for _ in range(5):
                f()
        for _ in range(rounds):
            for k, f in calls.items():
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(launches):
                    f()
                e.record()
                e.synchronize()
                times[k].append(s.elapsed_time(e) / launches)
        out[f"8x{name}"] = {k: round(float(np.median(v)), 4) for k, v in times.items()}
        out[f"8x{name}"]["bytes_in_per_launch"] = {"rgb": 8 * h * w * 3, "yuv": 8 * h * w * 3 // 2}
    return out


def push_arm(model, cams, cuda, warmup, pushes):
    """p50 / p99 push time (ms) of an RGB group and an NV12 group on the same frames, alternated push by push."""
    sizes = [SIZES["720p"] if i % 2 == 0 else SIZES["1080p"] for i in range(cams)]
    yuv = [nv12_frames(4, h, w, seed=10 + i) for i, (h, w) in enumerate(sizes)]
    rgb = [to_rgb(v) for v in yuv]
    if cuda:
        yuv = [torch.from_numpy(v).cuda() for v in yuv]
        rgb = [torch.from_numpy(v).cuda() for v in rgb]
    groups = {"rgb": model.stream_group(cams, pixel_format="rgb"), "nv12": model.stream_group(cams, pixel_format="nv12")}
    frames = {"rgb": rgb, "nv12": yuv}
    hs = {k: [g.open() for _ in range(cams)] for k, g in groups.items()}
    times = {k: [] for k in groups}
    for p in range(warmup + pushes):
        order = list(groups) if p % 2 == 0 else list(groups)[::-1]
        for k in order:
            push = {h: frames[k][i][p % 4] for i, h in enumerate(hs[k])}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            groups[k].push(push, to_host=not cuda)
            if p >= warmup:
                times[k].append((time.perf_counter() - t0) * 1e3)
    for g in groups.values():
        g.close()
    res = {k: {"p50_ms": round(float(np.percentile(v, 50)), 3), "p99_ms": round(float(np.percentile(v, 99)), 3)}
           for k, v in times.items()}
    res["nv12_minus_rgb_p50_ms"] = round(res["nv12"]["p50_ms"] - res["rgb"]["p50_ms"], 3)
    return res


def video_arm(model, n, reps):
    yuv = nv12_frames(n, 720, 1280, seed=30)
    rgb = to_rgb(yuv)
    best = {"rgb": float("inf"), "nv12": float("inf")}
    outs = {}
    for r in range(reps):
        order = ["rgb", "nv12"] if r % 2 == 0 else ["nv12", "rgb"]
        for k in order:
            frames = rgb if k == "rgb" else yuv
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            d, _ = model.infer_video_depth(frames, 24, device="cuda", pixel_format=k)
            best[k] = min(best[k], time.perf_counter() - t0)
            outs[k] = d
    same = bool(np.array_equal(outs["rgb"], outs["nv12"]))
    return {"frames": n, "size": "1280x720", "rgb_fps": round(n / best["rgb"], 1), "nv12_fps": round(n / best["nv12"], 1),
            "nv12_over_rgb": round(best["rgb"] / best["nv12"], 3), "bit_identical": same,
            "host_bytes_per_frame": {"rgb": 720 * 1280 * 3, "nv12": 720 * 1280 * 3 // 2}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--encoder", default="vits")
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--pushes", type=int, default=60)
    ap.add_argument("--video-frames", type=int, default=500)
    ap.add_argument("--video-reps", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ingest_b200.json"))
    a = ap.parse_args()
    res = {"tool": "tools/bench_ingest.py", **card(), "encoder": a.encoder, "dtype": "bf16"}
    res["kernel_ms"] = kernel_arm(a.launches, a.rounds)
    print(json.dumps(res["kernel_ms"]), file=sys.stderr)
    m = VideoDepthAnything(**MODEL_CONFIGS[a.encoder], dtype=torch.bfloat16)
    m.load_state_dict(synth_state_dict(**MODEL_CONFIGS[a.encoder], seed=0))
    m.to("cuda")
    res["push"] = {}
    for cams in (8, 16):
        for cuda in (False, True):
            key = f"{cams}cams_{'cuda' if cuda else 'host'}"
            res["push"][key] = push_arm(m, cams, cuda, a.warmup, a.pushes)
            print(key, json.dumps(res["push"][key]), file=sys.stderr)
    res["video"] = video_arm(m, a.video_frames, a.video_reps)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
