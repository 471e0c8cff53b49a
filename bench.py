#!/usr/bin/env python
"""bench.py — frames/s of the Video-Depth-Anything hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--encoder vitl] [--dtype bf16]
                    [--dump-outputs DIR]

A "step" is one forward pass of one 1x32x518x518 window (BASELINE.json configs[1]) per GPU.  N>1 is launched by
torchrun (one rank per GPU, NCCL); windows are independent in model compute (SURVEY.md §3.2), so ranks process
their own windows with no data-path collective and the aggregate is reported as weak scaling.

Printed JSON (rank 0, one line):
  value        model frames/s, inputs resident in HBM, timed with CUDA events, max over ranks
  e2e          same metric through the public API with HOST buffers: every step's pinned H2D of its window, forward
               and D2H of its depth map inside the timed region (double-buffered by the caller, host wall clock)
  video        BASELINE.json configs[2]: infer_video_depth on a 2048-frame uint8 video, host frames -> host depths
  roofline     dominant kernel family = the tcgen05 GEMM/implicit-conv kernel; achieved = algorithmic FLOPs of
               those launches / their CUDA-event time, measured in the timed region; peak = MEASURED_PEAKS.json
  cpu_baseline the oracle port (oracle/vda_oracle.py, torch fp32 on the host cores) on a bounded sample
`--impl reference` times that CPU port alone (the reference itself is Python/PyTorch on CPU; /root/reference does
not exist on the GPU box, the oracle is its pinned restatement).

`--dump-outputs DIR` (GPU arm, rank 0) writes what the timed calls returned in their last step, so that two builds can be
compared output for output on the same seeded inputs (weights and inputs depend on the arguments only):
  depth.npy        the whole float32 [1, 32, 518, 518] depth map of the last timed window (34 MB)
  video_depth.npy  8 frames of the long-video result, picked with a fixed seed, in frame order: float32 [8, 518, 518]
                   (9 MB; every frame of a video shorter than 8 frames; absent with --video-frames 0, and with a
                   note on stderr if that arm failed)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_TFLOP_PER_WINDOW = {"vitl": 44.950, "vits": 3.881}     # SURVEY.md §6 / BASELINE.md §2 (32x518x518)
BASELINE_A100_FP16_FPS = {"vitl": 1000.0 / 14.0, "vits": 1000.0 / 7.5}   # BASELINE.md §1 (reference README.md:49-64)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"], src="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.05)   # (one nvidia-smi query takes ~50-100 ms itself: a few samples per second of load)

    def stop(self):
        self._stop_ev.set()
        self.join(timeout=3)
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(encoder: str, world: int) -> dict:
    """`config` of the JSON line: identical for the GPU arm and the reference arm (the driver compares them)."""
    return {"workload": f"{encoder} 1x32x518x518 window per GPU per step, random-init weights",
            "encoder": encoder, "frames_per_window": 32, "l2": "256 MB flush between steps",
            "launch": "CUDA graph replay per window", "parallelism": f"window-sharded replicas x{world}"}


def cpu_port_frames_per_s(encoder: str, frames: int, steps: int = 1, warmup: int = 0):
    """The reference's fp32 CPU path (oracle port) on a bounded sample: `frames` frames at 518x518."""
    from oracle import vda_oracle as O
    from video_depth_anything_b200.synth import MODEL_CONFIGS, synth_state_dict
    torch.set_num_threads(os.cpu_count())
    sd = synth_state_dict(**MODEL_CONFIGS[encoder], seed=0)
    x = torch.randn(1, frames, 3, 518, 518, generator=torch.Generator().manual_seed(1234))
    for _ in range(warmup):
        O.forward(sd, x, encoder)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        O.forward(sd, x, encoder)
        ts.append(time.perf_counter() - t0)
    return frames / (sum(ts) / len(ts)), ts


def reference_sample_frames(encoder: str, steps: int, warmup: int, budget_s: float, frames_per_s: float) -> int:
    """Frames per step of the reference arm: the largest T <= 32 for which (steps + warmup) passes fit `budget_s`
    at `frames_per_s` (a calibration pass measures it).  Pure function (tests/test_bench_cpu.py)."""
    per_step = budget_s / max(steps + warmup, 1)
    return int(max(1, min(32, per_step * frames_per_s)))


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path (the pinned oracle port: the reference
    is Python/PyTorch and /root/reference does not exist on the GPU box), all host threads, same metric / unit /
    config as the GPU arm, EXACTLY `--steps` timed and `--warmup` untimed passes.  A full ViT-L window is ~40 s of CPU
    work, so each pass runs a bounded sample of the window: T frames of the 32, T chosen from a one-frame calibration
    pass so that the whole run ends within `--cpu-budget` seconds (stated in cpu_baseline.sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W, K = args.warmup, args.steps
    frames = args.cpu_frames
    if frames <= 0:
        fps4, _ = cpu_port_frames_per_s(args.encoder, 4, steps=1, warmup=0)       # calibration pass (also warms the allocator)
        frames = reference_sample_frames(args.encoder, K, W, args.cpu_budget, fps4)
    fps, ts = cpu_port_frames_per_s(args.encoder, frames, steps=K, warmup=W)
    ms = 1e3 * sum(ts) / len(ts)
    sample = (f"{frames} of 32 frames (T={frames}) at 518x518 per step, {args.encoder} fp32, torch CPU oracle port, "
              f"{K} timed + {W} warm-up passes")
    line = {
        "impl": "reference", "metric": "frames/s", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.encoder, args.gpus),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--encoder", default="vitl", choices=["vitl", "vits"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"])
    ap.add_argument("--cpu-frames", type=int, default=0,
                    help="frames per pass of the CPU port (0: GPU arm = a full 32-frame window once, ~40 s on 16 cores for "
                         "vitl; reference arm = sized to --cpu-budget)")
    ap.add_argument("--cpu-budget", type=float, default=200.0, help="seconds the whole reference arm may take")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer arm (profiling runs only)")
    ap.add_argument("--video-frames", type=int, default=2048, help="length of the long-video arm (0 = skip)")
    ap.add_argument("--no-other-configs", dest="other_configs", action="store_false",
                    help="skip the BASELINE configs[3]/[4] arms (metric 518x924, vits clips)")
    ap.add_argument("--profile-out", default=None, help="write the per-kernel-family time table (JSON) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, ops, synth_state_dict

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    dt = torch.bfloat16 if args.dtype == "bf16" else torch.float16

    model = VideoDepthAnything(**MODEL_CONFIGS[args.encoder], dtype=dt)
    model.load_state_dict(synth_state_dict(**MODEL_CONFIGS[args.encoder], seed=0))
    model.to(dev)
    B, T, H, Wd = 1, 32, 518, 518
    g = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(B, T, 3, H, Wd, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    out_host = torch.empty(B, T, H, Wd, dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident arm ----------------
    for _ in range(W):
        d = model.forward(x_dev)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    launches0 = ops.LAUNCHES
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for i in range(K):
        flush.zero_()                      # evict L2 between steps (256 MB > 126 MB L2)
        ev[i][0].record()
        d = model.forward(x_dev)           # CUDA-graph replay of the ~330 libvda launches of one window
        ev[i][1].record()
    t_end.record()
    barrier()
    dumps = {}
    if args.dump_outputs and rank == 0:    # the last timed step's depth map
        dumps["depth"] = d.float().cpu().numpy()
    launches = ops.LAUNCHES - launches0
    clocks = sampler.stop() if sampler else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = t_start.elapsed_time(t_end)
    # per-kernel table: the same K steps once more, launched eagerly with a CUDA-event pair around every libvda
    # launch (events cannot be recorded per kernel inside a graph replay); shares are relative to these steps
    ops.PROFILE = []
    pev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for i in range(K):
        flush.zero_()
        pev[i][0].record()
        model.forward(x_dev)
        pev[i][1].record()
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    prof_step_ms = [a.elapsed_time(b) for a, b in pev]
    tmax = torch.tensor([total_ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = tmax.item()
    frames_total = world * K * B * T
    value = frames_total / (total_ms * 1e-3)
    assert (d > 0).float().mean().item() > 0.99, "degenerate output"

    # per-kernel-family table from the CUDA events recorded inside the timed region
    fam, shapes = {}, {}
    for name, info, s, e in prof:
        key = info.get("kind", name)
        if "M" in info:
            sh = shapes.setdefault((key, info["M"], info["N"], info["K"]), {"ms": 0.0, "flops": 0.0, "launches": 0})
            sh["ms"] += s.elapsed_time(e)
            sh["flops"] += info["flops"]
            sh["launches"] += 1
        f = fam.setdefault(key, {"ms": 0.0, "flops": 0.0, "launches": 0})
        f["ms"] += s.elapsed_time(e)
        f["flops"] += info.get("flops", 0.0)
        f["bytes"] = f.get("bytes", 0.0) + info.get("bytes", 0.0)
        f["launches"] += 1
    pk = peaks()
    tc = [v for k, v in fam.items() if k.startswith("gemm") or k.startswith("conv3x3")]
    tc_ms, tc_flops, tc_n = sum(v["ms"] for v in tc), sum(v["flops"] for v in tc), sum(v["launches"] for v in tc)
    achieved = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    roofline = {"bound": "tensor", "kernel": "gemm_kernel (tcgen05 GEMM + implicit 3x3 conv, all epilogues)",
                "achieved": achieved, "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved / pk["sustained"],
                "peak_kind": f"bf16_tflops_sustained of {pk['src']} (kernel timed inside a long step)",
                "flops_per_launch": tc_flops / max(tc_n, 1), "avg_launch_ms": tc_ms / max(tc_n, 1),
                "launches_per_step": tc_n / K, "share_of_step": tc_ms / sum(step_ms),
                "share_of_eager_profiled_step": tc_ms / sum(prof_step_ms),
                "measured": "CUDA events around every launch, eager replay of the timed steps; share_of_step = kernel "
                            "time / the timed graph-replay steps", "traffic": None}
    # DRAM traffic per launch from the committed `ncu --set full` capture of the four hot encoder GEMMs (proj, fc1,
    # fc2, qkv at M=43840: 96 of the family's launches per window), next to their algorithmic operand bytes
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if args.encoder == "vitl" and os.path.exists(tpath):
        t = json.load(open(tpath))
        # algorithmic bytes per launch with the LayerNorm fold: proj / fc2 also write the 16-bit copy of the rows and
        # 8 (mean, M2) partials per row; qkv / fc1 read those partials
        M_, st = 43840, 43840 * 8 * 8
        algo = {"proj": M_ * 1024 * 2 + 1024 * 1024 * 2 + 2 * M_ * 1024 * 4 + M_ * 1024 * 2 + st,
                "fc1": M_ * 1024 * 2 + 4096 * 1024 * 2 + M_ * 4096 * 2 + st,
                "fc2": M_ * 4096 * 2 + 4096 * 1024 * 2 + 2 * M_ * 1024 * 4 + M_ * 1024 * 2 + st,
                "qkv": M_ * 1024 * 2 + 3072 * 1024 * 2 + M_ * 3072 * 2 + st}
        det = {n: {"dram_bytes": t[f"gemm_prof.ncu-rep:{i}"]["dram_bytes"], "algorithmic_bytes": algo[n]}
               for i, n in enumerate(("proj", "fc1", "fc2", "qkv")) if f"gemm_prof.ncu-rep:{i}" in t}
        if len(det) == 4:
            roofline["traffic"] = sum(v["dram_bytes"] for v in det.values()) / 4
            roofline["traffic_unit"] = "bytes per launch, mean of the 4 hot encoder GEMM shapes (ncu dram__bytes_read+write)"
            roofline["traffic_detail"] = det
    whole = ALGO_TFLOP_PER_WINDOW[args.encoder] * K * B / (sum(step_ms) * 1e-3)
    # secondary kernels, same measurement: fused attention (tensor work 4*N^2*d per (frame, head); exp-bound, d = 64)
    # and LayerNorm (HBM-bound: fp32 rows in, 16-bit rows out)
    others = {}
    if "attention_spatial" in fam and fam["attention_spatial"]["ms"] > 0:
        a = fam["attention_spatial"]
        others["attention_spatial"] = {"bound": "tensor (exp-limited)", "achieved": a["flops"] / (a["ms"] * 1e-3) / 1e12,
                                       "peak": pk["sustained"], "unit": "TFLOP/s",
                                       "frac": a["flops"] / (a["ms"] * 1e-3) / 1e12 / pk["sustained"],
                                       "share_of_step": a["ms"] / sum(step_ms)}
    if "layernorm" in fam and fam["layernorm"]["ms"] > 0 and fam["layernorm"].get("bytes", 0) > 0:
        a = fam["layernorm"]
        gbs = a["bytes"] / (a["ms"] * 1e-3) / 1e9
        others["layernorm"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
                               "frac": gbs / pk["hbm"], "share_of_step": a["ms"] / sum(step_ms)}
    roofline["other_kernels"] = others

    # ---------------- end-to-end arm (host buffers, copies in the timed region) ----------------
    # Every step uploads its own window from pinned host memory, runs VideoDepthAnything.forward and reads the depth map
    # back to pinned host memory.  The caller double-buffers: the upload of step i+1 and the download of step i run on
    # copy streams next to the forward of step i+1 / i (a serving loop's normal shape); the host consumes each result
    # one step later, and all K uploads, forwards and downloads lie inside the timed region.
    e2e = None
    if not args.no_e2e:
        up, down = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream()
        xbuf = [torch.empty_like(x_dev) for _ in range(2)]
        out_hosts = [out_host, torch.empty_like(out_host).pin_memory()]

        def e2e_loop(n):
            ev_up = [torch.cuda.Event(), torch.cuda.Event()]
            ev_free = [None, None]                     # forward that last read xbuf[b] has finished
            ev_down = [None, None]
            with torch.cuda.stream(up):
                xbuf[0].copy_(x_host, non_blocking=True)
                ev_up[0].record(up)
            for i in range(n):
                b = i & 1
                main.wait_event(ev_up[b])
                dd = model.forward(xbuf[b])
                done = torch.cuda.Event()
                done.record(main)
                ev_free[b] = done
                if i + 1 < n:                          # upload of the next window overlaps this forward
                    with torch.cuda.stream(up):
                        if ev_free[1 - b] is not None:
                            up.wait_event(ev_free[1 - b])
                        xbuf[1 - b].copy_(x_host, non_blocking=True)
                        ev_up[1 - b].record(up)
                if ev_down[b] is not None:
                    ev_down[b].synchronize()           # the caller consumes result i-2 before its buffer is reused
                with torch.cuda.stream(down):
                    down.wait_event(done)
                    out_hosts[b].copy_(dd, non_blocking=True)
                    dd.record_stream(down)
                    ev_down[b] = torch.cuda.Event()
                    ev_down[b].record(down)
            for e in ev_down:
                if e is not None:
                    e.synchronize()

        e2e_loop(2)
        barrier()
        t0 = time.perf_counter()
        e2e_loop(K)
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        tm = torch.tensor([e2e_ms], device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e = {"value": frames_total / (tm.item() * 1e-3), "unit": "frames/s",
               "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
               "pipeline": "double-buffered: H2D of step i+1 and D2H of step i overlap the forward; host wall clock"}

    # ---------------- long-video arm (BASELINE.json configs[2]): infer_video_depth from host frames to host depths ---
    video = None

    def video_arm():
        import numpy as np
        from video_depth_anything_b200.parallel import infer_video_depth_sharded
        from video_depth_anything_b200.windows import num_windows
        base = np.random.default_rng(0).integers(0, 256, (64, H, Wd, 3), dtype=np.uint8)
        frames = base[np.arange(args.video_frames) % 64]
        # (measured scaling of this arm, 2048 frames: 1 GPU 3.9 s, 2 GPUs 2.10 s, 8 GPUs 0.64 s; DESIGN.md §8)
        # warm-up on the same video: graphs for the 32/22-frame encodes, allocator blocks, pinned staging / NCCL buffers of
        # the sizes the timed call uses (a short warm-up video left an unexplained ~25 ms in the 8-GPU exchange)
        infer_video_depth_sharded(model, frames, 24, device=dev)
        # the sharded driver releases the page lock of the warm-up call's result half a second after that call, in a
        # background thread (cudaHostUnregister holds the context lock for tens of ms per 100 MB): let it finish outside the
        # timed call instead of 0.5 s into it (seen once in four 2-GPU runs: 2.59 s instead of 2.01 s)
        time.sleep(1.0 if world > 1 else 0.0)
        barrier()
        l0 = ops.LAUNCHES
        t0 = time.perf_counter()
        depths, _ = infer_video_depth_sharded(model, frames, 24, device=dev)
        torch.cuda.synchronize()
        dt_s = time.perf_counter() - t0
        tv = torch.tensor([dt_s], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        nwin = num_windows(args.video_frames)
        if rank == 0:
            import zlib
            assert depths.shape == (args.video_frames, H, Wd) and np.isfinite(depths[::97]).all()
            # the result is bit-reproducible across GPU counts (fixed-order reductions, batch-invariant kernels): the
            # CRC of the depth bytes must be the same number in the N = 1, 2, 4, 8 lines (computed after the timed region)
            crc = zlib.crc32(memoryview(np.ascontiguousarray(depths)).cast("B")) & 0xFFFFFFFF
            if args.dump_outputs:
                pick = np.random.default_rng(0).choice(args.video_frames, min(8, args.video_frames), replace=False)
                dumps["video_depth"] = np.ascontiguousarray(depths[np.sort(pick)], dtype=np.float32)
            return {"workload": f"{args.encoder} {args.video_frames}x518x518 uint8 video, 32-frame windows, overlap 10, "
                                 f"host frames -> host depths (upload, device preprocessing, feature reuse, alignment, "
                                 f"download all inside the timed region)",
                     "video_frames_per_s": args.video_frames / tv.item(), "windows": nwin,
                     "window_slots_per_s": nwin * 32 / tv.item(), "seconds": tv.item(), "crc32": f"{crc:08x}",
                     "shard_mode": os.environ.get("VDA_SHARD_MODE", "two_phase") if world > 1 else "single process",
                     "gpu_launches_rank0": ops.LAUNCHES - l0, "timing": "host wall clock, max over ranks"}
        return None

    if args.video_frames > 0:
        if world > 1:
            video = video_arm()
        else:
            try:                                     # the headline line must survive a failure of this extra arm
                video = video_arm()
            except Exception as exc:                 # noqa: BLE001
                video = {"error": f"{type(exc).__name__}: {exc}"}

    # ---------------- BASELINE.json configs[3] / configs[4]: one clip per GPU per step, replicas (weak scaling) -------
    #   metric924   metric_depth vitl, 1x32x518x924 (2443 tokens per frame)      [metric_depth/.../video_depth.py:132 path]
    #   vits8clips  vits, one 32x518x518 clip per GPU (8 clips on 8 GPUs), bf16
    other = None
    if args.other_configs:
        other = {}
        model = x_dev = flush = None       # free the headline model's weights, buffers and graphs
        torch.cuda.empty_cache()
        for name, enc, (hh, ww), metric in (("metric924", "vitl", (518, 924), True), ("vits8clips", "vits", (518, 518), False)):
            try:
                m2 = VideoDepthAnything(**MODEL_CONFIGS[enc], dtype=dt, metric=metric)
                m2.load_state_dict(synth_state_dict(**MODEL_CONFIGS[enc], seed=0))
                m2.to(dev)
                xx = torch.randn(1, 32, 3, hh, ww, generator=torch.Generator().manual_seed(77 + rank)).to(dev)
                fl = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
                for _ in range(3):
                    m2.forward(xx)
                barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                tsum = 0.0
                for _ in range(K):
                    fl.zero_()
                    a.record()
                    dd = m2.forward(xx)
                    b.record()
                    torch.cuda.synchronize()
                    tsum += a.elapsed_time(b)
                tt = torch.tensor([tsum], device=dev)
                if world > 1:
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                ms2 = tt.item() / K
                tfl = {"metric924": 88.4, "vits8clips": ALGO_TFLOP_PER_WINDOW["vits"]}[name]
                other[name] = {"workload": f"{enc}{' metric' if metric else ''} 1x32x{hh}x{ww} clip per GPU per step x{world} GPUs",
                               "frames_per_s": world * 32 / (ms2 * 1e-3), "ms_per_clip": ms2, "steps": K, "dtype": args.dtype,
                               "tflops_algorithmic_per_gpu": tfl / (ms2 * 1e-3), "timing": "CUDA events, max over ranks, L2 flushed"}
                assert (dd > 0).float().mean().item() > 0.99
                m2 = xx = fl = dd = None
                torch.cuda.empty_cache()
            except Exception as exc:                      # noqa: BLE001  (extra arm: never takes the headline line down)
                other[name] = {"error": f"{type(exc).__name__}: {exc}"}
                if world > 1:
                    raise

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cf = args.cpu_frames if args.cpu_frames > 0 else 32
            fps, ts = cpu_port_frames_per_s(args.encoder, cf)
            cpu = {"value": fps, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"{cf} of 32 frames (T={cf}) at 518x518, one pass, {args.encoder} fp32, "
                             f"torch CPU oracle port, {ts[0]:.1f}s"}
        line = {
            "metric": "frames/s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "p50_window_latency_ms": statistics.median(step_ms),
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (value / world / BASELINE_A100_FP16_FPS[args.encoder]) if world == 1 else None,
            "baseline": "BASELINE.md: reference README latency on 1x A100 fp16 (vitl 14 ms/frame = 71.4 frames/s, vits "
                        "7.5 ms = 133 frames/s), other hardware; 1 GPU only",
            "dtype": args.dtype, "data": "synthetic",
            "config": workload_config(args.encoder, world),
            "tflops_algorithmic": whole if world == 1 else None,
            "frac_of_bf16_sustained": (whole / pk["sustained"]) if world == 1 else None,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "video": video, "gpu_launches": launches,
            "clocks": clocks,
            # BASELINE.json configs[2] (long video sharded over the GPUs) at the top level too: strong scaling, same
            # video at every N, identical CRC expected
            "video_frames_per_s": (video or {}).get("video_frames_per_s"), "video_seconds": (video or {}).get("seconds"),
            "video_crc32": (video or {}).get("crc32"),
            "other_configs": other,
        }
        print(json.dumps(line), flush=True)
        if args.profile_out:
            tab = sorted(((k, v["ms"] / K, v["launches"] / K, v["flops"] / K / 1e12) for k, v in fam.items()),
                         key=lambda r: -r[1])
            json.dump({"per_step": [dict(kernel=k, ms=ms, launches=n, tflop=tf,
                                         tflops=(tf / (ms * 1e-3) if ms > 0 else 0)) for k, ms, n, tf in tab],
                       "gemm_shapes": [dict(kernel=k[0], M=k[1], N=k[2], K=k[3], ms_per_launch=v["ms"] / v["launches"],
                                            launches=v["launches"] / K,
                                            tflops=v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["ms"] > 0 else 0)
                                       for k, v in sorted(shapes.items(), key=lambda kv: -kv[1]["ms"])],
                       "step_ms": step_ms, "eager_profiled_step_ms": prof_step_ms}, open(args.profile_out, "w"), indent=1)
        if args.dump_outputs:
            import numpy as np
            assert sum(a.nbytes for a in dumps.values()) <= 64 << 20
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
            if args.video_frames > 0 and "video_depth" not in dumps:
                print(f"bench.py: {os.path.join(args.dump_outputs, 'video_depth.npy')} not written: the long-video arm "
                      f"failed ({(video or {}).get('error')})", file=sys.stderr, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
