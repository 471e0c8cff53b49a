#!/usr/bin/env python
"""Micro-benchmark + parity of the spatial attention kernel at the ViT-L window shape (CUDA events, L2 flushed)."""
import os
import sys
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_depth_anything_b200 import ops  # noqa: E402


def run(frames, N, heads, dt, iters=10, check=True):
    g = torch.Generator().manual_seed(0)
    qkv = (torch.randn(frames, N, 3, heads, 64, generator=g) * 1.5).cuda().to(dt)
    out = torch.zeros(frames, N, heads * 64, device="cuda", dtype=dt)
    ops.attention_spatial(qkv, out, frames, N, heads)
    torch.cuda.synchronize()
    msg = ""
    if check:
        fr = min(frames, 2)
        q, k, v = (qkv[:fr, :, i].float().permute(0, 2, 1, 3) for i in range(3))
        ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(fr, N, heads * 64)
        err = (out[:fr].float() - ref).abs().max().item()
        msg = f" max abs err {err:.3e} (ref max {ref.abs().max().item():.3f})"
        if frames > 2:   # last frame too (persistent schedule tail)
            q, k, v = (qkv[-1:, :, i].float().permute(0, 2, 1, 3) for i in range(3))
            ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(1, N, heads * 64)
            msg += f" last-frame err {(out[-1:].float() - ref).abs().max().item():.3e}"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(iters):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.attention_spatial(qkv, out, frames, N, heads)
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ms = sorted(ts)[len(ts) // 2]
    fl = 4.0 * frames * heads * N * N * 64
    print(f"attn {frames}x{N}x{heads} {dt}: {ms:.3f} ms  {fl / ms / 1e9:.1f} TFLOP/s{msg}", flush=True)


def run_temporal(T, hw, C, dt, iters=10):
    g = torch.Generator().manual_seed(0)
    qkv = torch.randn(T * hw, 3 * C, generator=g).cuda().to(dt)
    out = torch.zeros(T * hw, C, device="cuda", dtype=dt)
    ops.attention_temporal(qkv, out, T, hw, C)
    torch.cuda.synchronize()
    heads, dh = 8, C // 8
    q, k, v = (qkv[:, i * C:(i + 1) * C].float().reshape(T, hw, heads, dh).permute(1, 2, 0, 3) for i in range(3))
    ref = F.scaled_dot_product_attention(q, k, v).permute(2, 0, 1, 3).reshape(T * hw, C)
    err = (out.float() - ref).abs().max().item()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ts = []
    for _ in range(iters):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        ops.attention_temporal(qkv, out, T, hw, C)
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ms = sorted(ts)[len(ts) // 2]
    gb = 4.0 * T * hw * C * 2 / 1e9
    print(f"temporal attn T={T} hw={hw} C={C} {dt}: {ms * 1e3:.1f} us  {gb / ms * 1e3:.0f} GB/s (q,k,v,o)  max abs err {err:.3e}", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "temporal":
        for hw, C in ((1369, 1024), (361, 1024), (1369, 256), (5476, 256), (1369, 192), (361, 384), (5476, 64)):
            run_temporal(32, hw, C, torch.bfloat16)
        run_temporal(8, 100, 256, torch.float16)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "prof32":    # the benchmarked shape, one warm-up + one launch (ncu -s 1 -c 1)
        run(32, 1370, 16, torch.bfloat16, iters=1, check=False)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "prof":      # short run for ncu
        run(8, 1370, 16, torch.bfloat16, iters=2, check=False)
        sys.exit(0)
    run(1, 21, 2, torch.float16)
    run(1, 128, 1, torch.bfloat16)
    run(1, 300, 2, torch.bfloat16)
    run(2, 1370, 16, torch.bfloat16)
    run(1, 2443, 4, torch.float16)
    run(32, 1370, 16, torch.bfloat16)
    run(32, 1370, 6, torch.float16)
