#!/usr/bin/env python
"""Streaming inference on one GPU (VideoDepthAnything.stream / DepthStream.push); prints one JSON line and writes it to
--out.

Per config (vits 518x518, vitl 518x518, vitl 518x924 = a 1280x720 video, the metric config):
  * push latency p50 / p99: host clock around `push` (H2D of the frame, graph replay, D2H of the depth, synchronised),
    400 frames after 40 warm-up frames, so the context has been sliding for 8 frames before the first timed one;
  * step device time p50 / p99: CUDA events around a replay of the step graph alone;
  * the windowed forward of the same model (one 32-frame window, CUDA events) in frames/s, for comparison.
Then the step kernel alone at every block shape of the configs with a full context (31 cached frames, 32 slots):
median time over launches with the L2 overwritten in between, the bytes it must move (computed from shapes) over that
time, and that rate's share of the HBM bound (7.7 TB/s, the HGX B200 data sheet's per-GPU figure); for the ViT-L 518x518
shapes also the batched kernel at B = 8 (8 streams' frames in one launch).
Then stream groups (VideoDepthAnything.stream_group) of each --streams count for ViT-S and ViT-L at 518x518: every push
names every stream, push latency p50 / p99 over --group-pushes pushes after 40 warm-up pushes, and aggregate frames/s
(streams / p50 push).
With --mixed (ViT-L, bf16, each count of --mixed-streams): cameras of two frame sizes that share one network size
(1280x720 and 1920x1080 -> 518x924), push p50 / p99 (host clock, every push names every stream, --group-pushes pushes
after 40 warm-up pushes) and aggregate frames/s for
  (a) one group, every camera 1280x720 (host frames, host depths: the only form before per-stream sizes);
  (b) one group, half the cameras 1280x720 and half 1920x1080;
  (c) (b) with the frames as CUDA tensors and to_host=False (depths stay on the device);
  (d) the cameras of (b) as two groups, one per frame size, pushed one after the other (a push = both pushes);
then, in a run of its own under torch.profiler (graphs off, so every kernel is listed), the device time of the ragged
ingest and egress kernels within a push of (b) and (c).
With --chunks (e.g. 1,2,4,8,16): a lone stream pushing k consecutive frames per push (DepthStream.push of a stack) for
ViT-S 518x518, ViT-L 518x518 and ViT-L 1280x720 (host frames, and CUDA stacks with to_host=False): push p50 / p99 on the
host clock (push synchronises), frames/s = k / p50, over --chunk-pushes pushes after 6 warm-up pushes of the same k
(the first captures the bucket's graph); then the causal step kernel alone at the ViT-L 518x518 block shapes (one stream,
k = 8 rows, 31 context frames each, L2 overwritten between launches) next to the batched kernel at B = 8, and the cache
store kernel.
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
from video_depth_anything_b200 import MODEL_CONFIGS, VideoDepthAnything, ops, synth_state_dict  # noqa: E402
from video_depth_anything_b200.windows import get_resize_hw  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
CONFIGS = [("vits", 518, 518), ("vitl", 518, 518), ("vitl", 720, 1280)]


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip()
    return {"card": q.split(",")[0].strip() if q else torch.cuda.get_device_name(0),
            "power_limit": q.split(",")[1].strip() if "," in q else "unknown"}


def pct(xs, p):
    return float(np.percentile(np.asarray(xs), p))


def model(enc, dtype):
    m = VideoDepthAnything(**MODEL_CONFIGS[enc], dtype=dtype)
    m.load_state_dict(synth_state_dict(**MODEL_CONFIGS[enc], seed=0))
    return m.to("cuda")


def bench_config(enc, h0, w0, warmup, frames, dtype):
    m = model(enc, dtype)
    pool = np.random.default_rng(0).integers(0, 256, (16, h0, w0, 3), dtype=np.uint8)
    st = m.stream()
    for t in range(warmup):
        st.push(pool[t % 16])
    host = []
    for t in range(frames):
        f = pool[t % 16]
        t0 = time.perf_counter()
        st.push(f)
        host.append((time.perf_counter() - t0) * 1e3)
    dev = []
    for _ in range(100):                              # replays of the last step (idempotent: same inputs, same slot)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        st.group._step(1)
        e.record()
        e.synchronize()
        dev.append(s.elapsed_time(e))
    nh, nw = get_resize_hw(h0, w0)
    x = torch.randn(1, 32, 3, nh, nw, device="cuda")
    for _ in range(2):
        m.forward(x)
    win = []
    for _ in range(5):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        m.forward(x)
        e.record()
        e.synchronize()
        win.append(s.elapsed_time(e))
    eng = st.engine
    hp, wp = nh // 14, nw // 14
    shapes = [(c.shape[2], c.shape[3] // 2) for c in st.group.pool[::2]]   # (hw, C) of motion modules 0..3
    launches = st.group.graphs[1][3]
    st.close()
    del st, m
    torch.cuda.empty_cache()
    return {"encoder": enc, "frame": [h0, w0], "network": [nh, nw], "dtype": str(dtype).split(".")[-1],
            "push_ms_p50": round(pct(host, 50), 3), "push_ms_p99": round(pct(host, 99), 3),
            "step_device_ms_p50": round(pct(dev, 50), 3), "step_device_ms_p99": round(pct(dev, 99), 3),
            "push_fps_p50": round(1e3 / pct(host, 50), 1), "launches_per_step": launches,
            "window_forward_ms": round(pct(win, 50), 2), "window_forward_fps": round(32e3 / pct(win, 50), 1),
            "grid": [hp, wp]}, shapes


def bench_kernel(hw, C, dtype, B=1, iters=30):
    slots, n = 32, 31
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(B * hw, 3 * C, device="cuda", generator=g).to(dtype)
    cache = torch.randn(B, slots, hw, 2 * C, device="cuda", generator=g).to(dtype)
    pe = torch.randn(32, 3 * C, device="cuda", generator=g)
    ctx = torch.tensor([[n, 31] + list(range(31))] * B, dtype=torch.int32, device="cuda")
    rows = torch.arange(B, dtype=torch.int32, device="cuda")
    out = torch.empty(B * hw, C, dtype=dtype, device="cuda")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def launch():
        if B == 1:
            ops.attention_temporal_step(qkv, cache[0], pe, ctx[0], out)
        else:
            ops.attention_temporal_step(qkv, cache, pe, ctx, out, rows=rows)
    launch()
    ts = []
    for _ in range(iters):
        flush.zero_()                                  # 512 MB written: the cache rows come from HBM, not the 126 MB L2
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        launch()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e))
    ms = pct(ts, 50)
    nbytes = B * 2 * hw * (n * 2 * C + 3 * C + C + 2 * C)   # cached k'|v' read, q'|k'|v' read, out + write-slot row written
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"B": B, "hw": hw, "C": C, "head_dim": C // 8, "us": round(ms * 1e3, 2), "MB": round(nbytes / 1e6, 2),
            "GB_s": round(gbs, 1), "hbm_share": round(gbs * 1e9 / HBM_BYTES_PER_S, 3)}


def bench_chunks(enc, h0, w0, chunks, pushes, dtype, cuda=False):
    """A lone stream pushing k frames per push, for each k of `chunks` (module docstring)."""
    m = model(enc, dtype)
    pool = np.random.default_rng(0).integers(0, 256, (32, h0, w0, 3), dtype=np.uint8)
    src = torch.from_numpy(pool).cuda() if cuda else pool
    out = {"encoder": enc, "frame": [h0, w0], "network": list(get_resize_hw(h0, w0)), "dtype": str(dtype).split(".")[-1],
           "frames": "CUDA stacks, to_host=False" if cuda else "host stacks, host depths", "chunks": []}
    for k in chunks:
        st = m.stream()
        for t in range(2):                               # past frame 0: the context slides from push 6 on for k >= 8
            st.push(src[t], to_host=not cuda)
        ts = []
        for p in range(6 + pushes):
            a = (p * k) % (32 - k + 1)
            t0 = time.perf_counter()
            st.push(src[a:a + k] if k > 1 else src[a], to_host=not cuda)
            if p >= 6:
                ts.append((time.perf_counter() - t0) * 1e3)
        gr = st.group.causal_graphs if k > 1 else st.group.graphs
        (bk, entry), = gr.items()
        st.close()
        p50 = pct(ts, 50)
        out["chunks"].append({"k": k, "bucket": bk, "launches_per_push": entry[3], "push_ms_p50": round(p50, 3),
                              "push_ms_p99": round(pct(ts, 99), 3), "fps": round(k * 1e3 / p50, 1)})
    r1 = next((c for c in out["chunks"] if c["k"] == 1), None)
    if r1:
        for c in out["chunks"]:
            c["vs_k1"] = round(c["fps"] / r1["fps"], 3)
    del m
    torch.cuda.empty_cache()
    return out


def bench_causal_kernel(hw, C, dtype, k=8, iters=30):
    """The causal step kernel at one stream, k rows at t = 100.. (31 context frames each: row j reads j of them from
    the push's own rows), and the store kernel of the same rows; L2 overwritten before every launch."""
    from video_depth_anything_b200.windows import StreamGroupPlan, split_group_table
    L, slots = 31, 32
    plan = StreamGroupPlan(1, L)
    h = plan.open()
    plan.t[h] = 100
    bk, table = plan.step([h], counts=[k])
    rows, ctx, _ = split_group_table(torch.from_numpy(table).cuda(), bk, L)
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(bk * hw, 3 * C, device="cuda", generator=g).to(dtype)
    pool = torch.randn(1, slots, hw, 2 * C, device="cuda", generator=g).to(dtype)
    pe = torch.randn(32, 3 * C, device="cuda", generator=g)
    out = torch.empty(bk * hw, C, dtype=dtype, device="cuda")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")

    def timed(launch):
        launch()
        ts = []
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            launch()
            e.record()
            e.synchronize()
            ts.append(s.elapsed_time(e))
        return pct(ts, 50)
    ms_a = timed(lambda: ops.attention_temporal_step_causal(qkv, pool, pe, ctx, out, rows))
    ms_s = timed(lambda: ops.stream_cache_store(qkv, pool, rows, ctx))
    # bytes the causal kernel must move: pool rows of the context frames older than the push, q'|k'|v' of the k rows
    # (the in-push keys are these same rows), the output
    pool_rows = sum(L - j for j in range(k))
    nb_a = 2 * hw * (pool_rows * 2 * C + k * (3 * C + C))
    nb_s = 2 * hw * k * (2 * C + 2 * C)
    res = {}
    for name, ms, nb in (("causal", ms_a, nb_a), ("store", ms_s, nb_s)):
        gbs = nb / (ms * 1e-3) / 1e9
        res[name] = {"us": round(ms * 1e3, 2), "MB": round(nb / 1e6, 2), "GB_s": round(gbs, 1),
                     "hbm_share": round(gbs * 1e9 / HBM_BYTES_PER_S, 3)}
    return {"k": k, "hw": hw, "C": C, "head_dim": C // 8, **res}


def bench_group(enc, h0, w0, S, warmup, pushes, dtype):
    m = model(enc, dtype)
    pool = np.random.default_rng(0).integers(0, 256, (16, h0, w0, 3), dtype=np.uint8)
    g = m.stream_group(max_streams=S)
    hs = [g.open() for _ in range(S)]
    host = []
    for t in range(warmup + pushes):
        batch = {h: pool[(t + i) % 16] for i, h in enumerate(hs)}
        t0 = time.perf_counter()
        g.push(batch)
        if t >= warmup:
            host.append((time.perf_counter() - t0) * 1e3)
    (bk, entry), = g.graphs.items()
    g.close()
    del g, m
    torch.cuda.empty_cache()
    p50 = pct(host, 50)
    return {"encoder": enc, "frame": [h0, w0], "streams": S, "bucket": bk, "launches_per_push": entry[3],
            "push_ms_p50": round(p50, 3), "push_ms_p99": round(pct(host, 99), 3),
            "aggregate_fps": round(S * 1e3 / p50, 1)}


MIXED_SIZES = [(720, 1280), (1080, 1920)]


def bench_mixed(S, warmup, pushes, dtype):
    """Arms (a)-(d) of the module docstring at S cameras."""
    m = model("vitl", dtype)
    rng = np.random.default_rng(0)
    host = {hw: rng.integers(0, 256, (4, *hw, 3), dtype=np.uint8) for hw in MIXED_SIZES}
    dev = {hw: torch.from_numpy(f).cuda() for hw, f in host.items()}
    half = [MIXED_SIZES[0]] * (S // 2) + [MIXED_SIZES[1]] * (S - S // 2)

    def timed(push):
        ts = []
        for t in range(warmup + pushes):
            t0 = time.perf_counter()
            push(t)
            if t >= warmup:
                ts.append((time.perf_counter() - t0) * 1e3)
        return ts

    def one_group(sizes, frames, to_host):
        g = m.stream_group(max_streams=S)
        hs = [(g.open(), hw) for hw in sizes]
        ts = timed(lambda t: g.push({h: frames[hw][(t + i) % 4] for i, (h, hw) in enumerate(hs)}, to_host=to_host))
        g.close()
        return ts

    def two_groups():
        gs = []
        for hw in MIXED_SIZES:
            g = m.stream_group(max_streams=S // 2)
            gs.append((g, [g.open() for _ in range(S // 2)], hw))
        ts = timed(lambda t: [g.push({h: host[hw][(t + i) % 4] for i, h in enumerate(hs)}) for g, hs, hw in gs])
        for g, _, _ in gs:
            g.close()
        return ts

    arms = {"a_uniform_720p_host": lambda: one_group([MIXED_SIZES[0]] * S, host, True),
            "b_mixed_host": lambda: one_group(half, host, True),
            "c_mixed_cuda_frames_cuda_depth": lambda: one_group(half, dev, False),
            "d_two_groups_host": two_groups}
    out = {"streams": S, "frames": [list(hw) for hw in MIXED_SIZES], "network": list(get_resize_hw(*MIXED_SIZES[0]))}
    for name, run in arms.items():
        ts = run()
        torch.cuda.empty_cache()
        p50 = pct(ts, 50)
        out[name] = {"push_ms_p50": round(p50, 3), "push_ms_p99": round(pct(ts, 99), 3),
                     "aggregate_fps": round(S * 1e3 / p50, 1)}
    del m
    torch.cuda.empty_cache()
    return out


def profile_ragged(S, dtype, pushes=5):
    """Device time per push of the two ragged kernels and of all kernels, arms (b) and (c), from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    m = model("vitl", dtype)
    eng = m._ensure_engine()
    rng = np.random.default_rng(0)
    half = [MIXED_SIZES[0]] * (S // 2) + [MIXED_SIZES[1]] * (S - S // 2)
    host = [rng.integers(0, 256, (*hw, 3), dtype=np.uint8) for hw in half]
    res = {}
    for arm, frames, to_host in (("b_mixed_host", host, True),
                                 ("c_mixed_cuda_frames_cuda_depth", [torch.from_numpy(f).cuda() for f in host], False)):
        g = m.stream_group(max_streams=S)
        hs = [g.open() for _ in half]
        eng.use_graphs = False                        # eager: the same launches as the graph, each one traced
        for _ in range(2):
            g.push(dict(zip(hs, frames)), to_host=to_host)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(pushes):
                g.push(dict(zip(hs, frames)), to_host=to_host)
            torch.cuda.synchronize()
        eng.use_graphs = True
        g.close()
        kern = {"preprocess_ragged_kernel": 0.0, "bilinear_f32_ragged_kernel": 0.0}
        total = 0.0
        for e in prof.key_averages():
            us = e.device_time_total
            if e.device_type.name != "CUDA" or us <= 0:
                continue
            if "Memcpy" not in e.key and "Memset" not in e.key:
                total += us
            for k in kern:
                if k in e.key:
                    kern[k] += us
        res[arm] = {**{k + "_us_per_push": round(v / pushes, 1) for k, v in kern.items()},
                    "all_kernels_ms_per_push": round(total / pushes / 1e3, 3)}
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--streams", default="", help="comma-separated stream counts for the group sweep, e.g. 1,2,4,8,16")
    ap.add_argument("--group-pushes", type=int, default=100)
    ap.add_argument("--skip-single", action="store_true", help="only the group sweep and the batched kernel")
    ap.add_argument("--mixed", action="store_true", help="only the mixed frame size / CUDA frame arms (a)-(d)")
    ap.add_argument("--mixed-streams", default="8,16")
    ap.add_argument("--chunks", default="", help="only the multi-frame push sweep, k frames per push, e.g. 1,2,4,8,16")
    ap.add_argument("--chunk-pushes", type=int, default=40)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stream_b200.json"))
    a = ap.parse_args()
    counts = [int(x) for x in a.streams.split(",") if x]
    if not torch.cuda.is_available():
        sys.exit("bench_stream.py needs a GPU")
    if a.chunks:
        ks = [int(x) for x in a.chunks.split(",")]
        bf = torch.bfloat16
        res = {"what": "lone stream, k consecutive frames per push (DepthStream.push of a stack), bf16", **card(),
               "chunks": [bench_chunks("vits", 518, 518, ks, a.chunk_pushes, bf),
                          bench_chunks("vitl", 518, 518, ks, a.chunk_pushes, bf),
                          bench_chunks("vitl", 720, 1280, ks, a.chunk_pushes, bf),
                          bench_chunks("vitl", 720, 1280, ks, a.chunk_pushes, bf, cuda=True)]}
        hp = 518 // 14
        vitl = [(hp * hp, 1024), ((hp + 1) // 2 * ((hp + 1) // 2), 1024), (hp * hp, 256), (4 * hp * hp, 256)]
        res["causal_kernel_k8"] = [{"config": f"vitl 518x518 mm{mm}", **bench_causal_kernel(hw, C, bf)}
                                   for mm, (hw, C) in enumerate(vitl)]
        res["step_kernel_b8"] = [{"config": f"vitl 518x518 mm{mm}", **bench_kernel(hw, C, bf, B=8)}
                                 for mm, (hw, C) in enumerate(vitl)]
        return write(res, a.out)
    if a.mixed:
        res = {"what": "stream groups of mixed frame sizes, host vs CUDA frames (ViT-L bf16)", **card(),
               "mixed": [bench_mixed(int(S), a.warmup, a.group_pushes, torch.bfloat16) for S in a.mixed_streams.split(",")],
               "ragged_kernels_profiled": {S: profile_ragged(int(S), torch.bfloat16) for S in a.mixed_streams.split(",")}}
        return write(res, a.out)
    res = {"what": "streaming push latency / step device time / step kernel", **card(), "configs": [], "step_kernel": []}
    seen = set()
    for enc, h0, w0 in CONFIGS:
        if a.skip_single:
            break
        r, shapes = bench_config(enc, h0, w0, a.warmup, a.frames, torch.bfloat16)
        res["configs"].append(r)
        for mm, (hw, C) in enumerate(shapes):
            if (hw, C) not in seen:
                seen.add((hw, C))
                res["step_kernel"].append({"config": f"{enc} {r['network'][0]}x{r['network'][1]} mm{mm}",
                                           **bench_kernel(hw, C, torch.bfloat16)})
    if counts:
        res["what"] += " / stream groups / batched step kernel at B = 8"
        hp = 518 // 14
        vitl = [(hp * hp, 1024), ((hp + 1) // 2 * ((hp + 1) // 2), 1024), (hp * hp, 256), (4 * hp * hp, 256)]
        res["step_kernel_b8"] = [{"config": f"vitl 518x518 mm{mm}", **bench_kernel(hw, C, torch.bfloat16, B=8)}
                                 for mm, (hw, C) in enumerate(vitl)]
        res["groups"] = [bench_group(enc, 518, 518, S, a.warmup, a.group_pushes, torch.bfloat16)
                         for enc in ("vits", "vitl") for S in counts]
    write(res, a.out)


def write(res, path):
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
