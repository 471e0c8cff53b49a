#!/usr/bin/env python
"""Colour-mapped depth frames (vda_depth_range + vda_colorize_depth) in one run; writes profiles/colorize_b200.json (or
--out) and prints one JSON line.

  1. The kernels alone: per-frame range (2 launches) + colour (1 launch) per output format, for 16 x 1920x1080 and for
     8 x 1280x720 + 8 x 1920x1080 depth frames.  Cold: a 256 MB buffer is written between timed passes, which evicts
     the 126 MB L2.  Warm: the depths are rewritten just before each pass, as a push's resize kernel leaves them.  CUDA
     events around each pass, median over --rounds; bytes = two reads of the fp32 depths (range, colour) + the frames.
  2. Stream-group pushes (ViT-S, bf16): 8 and 16 cameras, half 720p and half 1080p, every push names every camera;
     output "depth" against "nv12", "rgb" and "gray", the arms alternated push by push after --warmup pushes each;
     host clock around each push, p50 / p99 over --pushes.  Host outputs, and CUDA outputs (to_host=False) for depth
     and nv12.
  3. colorize() of host depths (2048 x 518x518 and 500 x 1280x720, "video" range, RGB) against the reference's NumPy
     frame loop with the same table (writer excluded), best of --reps; the two outputs must be equal (checked).
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
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, colorize, ops, synth_state_dict  # noqa: E402
from video_depth_anything_b200.windows import INFERNO, OUT_DESC, color_descriptors, color_frame_shape  # noqa: E402

SIZES = {"720p": (720, 1280), "1080p": (1080, 1920)}
FMTS = {"rgb": 0, "nv12": 1, "gray": 3, "i420": 2}


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"card": q.split(",")[0].strip() if q else torch.cuda.get_device_name(0),
            "power_limit": q.split(",")[1].strip() if "," in q else "unknown"}


def _dev(a):
    return torch.from_numpy(a.view(np.uint8).copy()).cuda()


def kernel_arm(rounds):
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    table = torch.from_numpy(INFERNO.copy()).cuda()
    for name, sizes in {"16x1080p": [SIZES["1080p"]] * 16, "8x720p+8x1080p": [SIZES["720p"], SIZES["1080p"]] * 8}.items():
        n = len(sizes)
        px = [h * w for h, w in sizes]
        depth = torch.rand(sum(px), device="cuda") * 10
        src = depth.clone()
        offs = np.cumsum([0] + px)
        od = np.zeros(n, OUT_DESC)
        for i, (h, w) in enumerate(sizes):
            od[i] = (depth.data_ptr() + 4 * int(offs[i]), h, w)
        od_d = _dev(od)
        rng = torch.empty(n, 2, device="cuda")
        scratch = ops.depth_range_scratch(n, "cuda")
        res = {}
        for fmt, code in FMTS.items():
            fb = [int(np.prod(color_frame_shape(h, w, code))) for h, w in sizes]
            dst = torch.empty(sum(fb), dtype=torch.uint8, device="cuda")
            fo = np.cumsum([0] + fb)
            cd_d = _dev(color_descriptors(n, [(dst.data_ptr() + int(fo[i]), h, w) for i, (h, w) in enumerate(sizes)], code))
            tab = None if code == 3 else table

            def run():
                ops.depth_range(od_d, False, rng, scratch)
                ops.colorize_depth(od_d, cd_d, rng, True, tab)
            for _ in range(3):
                run()
            times = {"cold": [], "warm": []}
            for _ in range(rounds):
                for mode in ("cold", "warm"):
                    if mode == "cold":
                        flush.fill_(1)
                    else:
                        depth.copy_(src)
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    run()
                    e.record()
                    e.synchronize()
                    times[mode].append(s.elapsed_time(e))
            nbytes = 2 * 4 * sum(px) + sum(fb)
            res[fmt] = {m: {"ms": round(float(np.median(v)), 4), "GB_per_s": round(nbytes / np.median(v) / 1e6, 1)}
                        for m, v in times.items()}
            res[fmt]["bytes"] = nbytes
        out[name] = res
    return out


def push_arm(model, cams, warmup, pushes, to_host):
    sizes = [SIZES["720p"] if i % 2 == 0 else SIZES["1080p"] for i in range(cams)]
    frames = [np.random.default_rng(10 + i).integers(0, 256, (4, h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(sizes)]
    arms = ("depth", "nv12", "rgb", "gray") if to_host else ("depth", "nv12")
    groups = {k: model.stream_group(cams, output_format=k) for k in arms}
    hs = {k: [g.open() for _ in range(cams)] for k, g in groups.items()}
    times = {k: [] for k in groups}
    for p in range(warmup + pushes):
        order = list(groups) if p % 2 == 0 else list(groups)[::-1]
        for k in order:
            push = {h: frames[i][p % 4] for i, h in enumerate(hs[k])}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            groups[k].push(push, to_host=to_host)
            if p >= warmup:
                times[k].append((time.perf_counter() - t0) * 1e3)
    for g in groups.values():
        g.close()
    res = {k: {"p50_ms": round(float(np.percentile(v, 50)), 3), "p99_ms": round(float(np.percentile(v, 99)), 3)}
           for k, v in times.items()}
    res["out_bytes_per_push"] = {k: sum(h * w for h, w in sizes) * b for k, b in
                                 {"depth": 4, "nv12": 1.5, "rgb": 3, "gray": 1}.items() if k in arms}
    return res


def reference_loop(frames, table):
    """utils/dc_utils.py:76-85 without the writer (the table stands for (colormap * 255).astype(np.uint8))."""
    out = np.empty(frames.shape + (3,), np.uint8)
    d_min, d_max = frames.min(), frames.max()
    for i in range(frames.shape[0]):
        depth_norm = ((frames[i] - d_min) / (d_max - d_min) * 255).astype(np.uint8)
        out[i] = table[depth_norm]
    return out


def colorize_arm(n, h, w, reps):
    d = (np.random.default_rng(n).random((n, h, w), dtype=np.float32) * 20 + 0.5).astype(np.float32)
    best = {"colorize": float("inf"), "numpy": float("inf")}
    outs = {}
    for r in range(reps):
        for k in (("colorize", "numpy") if r % 2 == 0 else ("numpy", "colorize")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[k] = colorize(d, colormap=INFERNO) if k == "colorize" else reference_loop(d, INFERNO)
            best[k] = min(best[k], time.perf_counter() - t0)
    return {"frames": n, "size": f"{w}x{h}", "colorize_s": round(best["colorize"], 3), "numpy_s": round(best["numpy"], 3),
            "speedup": round(best["numpy"] / best["colorize"], 2), "equal": bool(np.array_equal(outs["colorize"], outs["numpy"])),
            "colorize_mpx_per_s": round(n * h * w / best["colorize"] / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--pushes", type=int, default=40)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--long-frames", type=int, default=2048)
    ap.add_argument("--hd-frames", type=int, default=500)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "colorize_b200.json"))
    a = ap.parse_args()
    res = {"tool": "tools/bench_colorize.py", **card(), "encoder": "vits", "dtype": "bf16"}
    res["kernel_ms"] = kernel_arm(a.rounds)
    print(json.dumps(res["kernel_ms"]), file=sys.stderr)
    m = VideoDepthAnything(**MODEL_CONFIGS["vits"], dtype=torch.bfloat16)
    m.load_state_dict(synth_state_dict(**MODEL_CONFIGS["vits"], seed=0))
    m.to("cuda")
    res["push"] = {}
    for cams in (8, 16):
        for to_host in (True, False):
            key = f"{cams}cams_{'host' if to_host else 'cuda'}"
            res["push"][key] = push_arm(m, cams, a.warmup, a.pushes, to_host)
            print(key, json.dumps(res["push"][key]), file=sys.stderr)
    res["colorize"] = [colorize_arm(a.long_frames, 518, 518, a.reps), colorize_arm(a.hd_frames, 720, 1280, a.reps)]
    print(json.dumps(res["colorize"]), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
