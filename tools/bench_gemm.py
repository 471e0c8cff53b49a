#!/usr/bin/env python
"""Micro-benchmark of the tcgen05 GEMM / implicit-conv kernel on the shapes of the ViT-L window (CUDA events, L2
flushed between launches, median of `iters`)."""
import os
import sys
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from video_depth_anything_b200 import ops  # noqa: E402
from video_depth_anything_b200._lib import ACT_GELU, ACT_NONE, ACT_RELU, EPI_TAIL  # noqa: E402

DT = torch.bfloat16
flush = None


def timeit(fn, iters=7):
    global flush
    if flush is None:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    return sorted(ts)[len(ts) // 2]


def plain(name, M, N, K, **kw):
    a = torch.randn(M, K, device="cuda").to(DT)
    w = (torch.randn(N, K, device="cuda") / K ** 0.5).to(DT)
    bias = torch.randn(N, device="cuda")
    out_f32 = kw.pop("out_f32", False)
    res_f32 = kw.pop("res_f32", False)
    out = torch.zeros(M, N, device="cuda", dtype=torch.float32 if out_f32 else DT)
    extra = {}
    if res_f32:
        extra = dict(res1=out, gamma=torch.ones(N, device="cuda"))
    ms = timeit(lambda: ops.gemm(a, w, out, bias=bias, **extra, **kw))
    print(f"{name:34s} M={M:8d} N={N:5d} K={K:5d}  {ms * 1e3:8.1f} us  {2.0 * M * N * K / ms / 1e9:7.1f} TF/s", flush=True)


def conv(name, n, H, W, ci, co, **kw):
    x = torch.randn(n * H * W, ci, device="cuda").to(DT)
    w = (torch.randn(co, 9 * ci, device="cuda") / (9 * ci) ** 0.5).to(DT)
    bias = torch.randn(co, device="cuda")
    tail = kw.pop("tail", False)
    if tail:
        out = torch.zeros(n * H * W, device="cuda")
        tw = torch.randn(32, device="cuda")
        fn = lambda: ops.gemm(x, w, out, bias=bias, epilogue=EPI_TAIL, tail_w=tw, tail_b=0.1, conv_shape=(n, H, W, ci))
    else:
        out = torch.zeros(n * H * W, co, device="cuda", dtype=DT)
        res = torch.randn(n * H * W, co, device="cuda").to(DT) if kw.pop("res", False) else None
        fn = lambda: ops.gemm(x, w, out, bias=bias, res1=res, conv_shape=(n, H, W, ci), **kw)
    ms = timeit(fn)
    M = n * H * W
    print(f"{name:34s} M={M:8d} N={co:5d} K={9 * ci:5d}  {ms * 1e3:8.1f} us  {2.0 * M * co * 9 * ci / ms / 1e9:7.1f} TF/s", flush=True)


def fold_set(M=43840, D=1024, once=False):
    """The four encoder GEMMs as the engine launches them with the LayerNorm fold: proj / fc2 with the 16-bit copy + row
    statistics (SPEC 4), qkv / fc1 with the fold epilogue (SPEC 5 / 6).  `once`: one launch each (ncu)."""
    parts, cols = ops.rowstat_layout(M, D)
    tok = torch.randn(M, D, device="cuda")
    x16 = torch.empty(M, D, device="cuda", dtype=DT)
    stats = torch.empty(M, parts, 2, device="cuda")
    ops.rowstats_cast(tok, x16, stats)
    ones, bias_d = torch.ones(D, device="cuda"), torch.randn(D, device="cuda")

    def run(name, fn, flops):
        if once:
            fn()
            torch.cuda.synchronize()
            return
        ms = timeit(fn)
        print(f"{name:44s} {ms * 1e3:8.1f} us  {flops / ms / 1e9:7.1f} TF/s", flush=True)

    att = torch.randn(M, D, device="cuda").to(DT)
    wp = (torch.randn(D, D, device="cuda") / D ** 0.5).to(DT)
    run("proj + ls + residual + x16 + stats (SPEC 4)",
        lambda: ops.gemm(att, wp, tok, bias=bias_d, gamma=ones, res1=tok, out16=x16, row_stats_out=stats), 2.0 * M * D * D)
    w1 = (torch.randn(4 * D, D, device="cuda") / D ** 0.5).to(DT)
    hid = torch.empty(M, 4 * D, device="cuda", dtype=DT)
    c1, c2 = w1.float().sum(1).contiguous(), torch.randn(4 * D, device="cuda")
    run("fc1 + GELU, LayerNorm folded (SPEC 6)",
        lambda: ops.gemm(x16, w1, hid, bias=c2, act=ACT_GELU, ln_fold=(stats, c1, 1e-6)), 2.0 * M * 4 * D * D)
    w2 = (torch.randn(D, 4 * D, device="cuda") / (4 * D) ** 0.5).to(DT)
    run("fc2 + ls + residual + x16 + stats (SPEC 4)",
        lambda: ops.gemm(hid, w2, tok, bias=bias_d, gamma=ones, res1=tok, out16=x16, row_stats_out=stats), 2.0 * M * 4 * D * D)
    wq = (torch.randn(3 * D, D, device="cuda") / D ** 0.5).to(DT)
    qkv = torch.empty(M, 3 * D, device="cuda", dtype=DT)
    cq1, cq2 = wq.float().sum(1).contiguous(), torch.randn(3 * D, device="cuda")
    run("qkv, LayerNorm folded (SPEC 5)",
        lambda: ops.gemm(x16, wq, qkv, bias=cq2, ln_fold=(stats, cq1, 1e-6)), 2.0 * M * 3 * D * D)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] in ("fold", "foldprof"):
    fold_set(once=sys.argv[1] == "foldprof")
    sys.exit(0)

if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] in ("smallk", "smallkprof"):
    # the head's small-K GEMMs (K = 256: AI 128 FLOP/B): timed, or one launch each for ncu
    if sys.argv[1] == "smallkprof":
        def once(fn, iters=1):
            fn()
            torch.cuda.synchronize()
            return 1.0
        timeit = once
    plain("out_conv 1x1 256->256 @74^2", 175232, 256, 256)
    plain("mm qkv 256->768 @74^2", 175232, 768, 256)
    plain("mm proj_in 256->256 f32 out", 175232, 256, 256, out_f32=True)
    plain("mm to_out 256->256 (+res f32)", 175232, 256, 256, out_f32=True, res_f32=True)
    plain("projects 1024->256", 43808, 256, 1024)
    conv("RCU conv 256->256 @37^2 +res", 32, 37, 37, 256, 256, res=True)
    sys.exit(0)

if __name__ == "__main__" and not (len(sys.argv) > 1 and sys.argv[1] in ("tail", "ln")):
    M = 43840
    if len(sys.argv) > 1 and sys.argv[1] == "prof":     # one launch per shape, for ncu
        def once(fn, iters=1):
            fn()
            torch.cuda.synchronize()
            return 1.0
        timeit = once
        plain("proj (+ls, fp32 residual in place)", M, 1024, 1024, out_f32=True, res_f32=True)
        plain("fc1 + GELU", M, 4096, 1024, act=ACT_GELU)
        plain("fc2 (+ls, fp32 residual in place)", M, 1024, 4096, out_f32=True, res_f32=True)
        plain("qkv", M, 3072, 1024)
        sys.exit(0)
    plain("qkv", M, 3072, 1024)
    plain("proj (+ls, fp32 residual in place)", M, 1024, 1024, out_f32=True, res_f32=True)
    plain("fc1 + GELU", M, 4096, 1024, act=ACT_GELU)
    plain("fc2 (+ls, fp32 residual in place)", M, 1024, 4096, out_f32=True, res_f32=True)
    plain("projects 1024->256", 43808, 256, 1024)
    plain("out_conv 1x1 256->256 @74^2", 175232, 256, 256)
    plain("out_conv 1x1 256->256 @148^2", 700928, 256, 256)
    conv("RCU conv 256->256 @148^2 +res", 32, 148, 148, 256, 256, res=True)
    conv("RCU conv 256->256 @148^2 relu", 32, 148, 148, 256, 256, act=ACT_RELU)
    conv("RCU conv 256->256 @74^2 +res", 32, 74, 74, 256, 256, res=True)
    conv("output_conv1 256->128 @296^2", 32, 296, 296, 256, 128)
    conv("output_conv2 tail 128->32->1 @518^2", 1, 518, 518, 128, 32, tail=True)


def tail(n=32, ih=296, iw=296, oh=518, ow=518, c=128):
    x = torch.randn(n * ih * iw, c, device="cuda").to(DT)
    w = (torch.randn(32, 9 * c, device="cuda") / (9 * c) ** 0.5).to(DT)
    b = torch.randn(32, device="cuda")
    w2 = torch.rand(32, device="cuda")
    out = torch.zeros(n, oh, ow, device="cuda")
    ms = timeit(lambda: ops.tail_fused(x, w, b, w2, 0.1, out, n, ih, iw, oh, ow, c))
    fl = 2.0 * n * oh * ow * 32 * 9 * c
    print(f"fused tail {n}x{ih}x{iw}->{oh}x{ow} C={c}: {ms * 1e3:8.1f} us  {fl / ms / 1e9:7.1f} TF/s", flush=True)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "tail":
    tail()
    tail(c=64)


def ln_bench(rows=43840, C=1024):
    x = torch.randn(rows, C, device="cuda")
    w = torch.randn(C, device="cuda"); b = torch.randn(C, device="cuda")
    out = torch.empty(rows, C, device="cuda", dtype=DT)
    ms = timeit(lambda: ops.layernorm(x, w, b, 1e-6, out))
    gb = rows * C * 6 / 1e9
    ref = torch.nn.functional.layer_norm(x, (C,), w, b, 1e-6)
    print(f"layernorm {rows}x{C} f32->bf16: {ms * 1e3:7.1f} us  {gb / ms * 1e3:6.0f} GB/s  max err {(out.float() - ref).abs().max().item():.3e}", flush=True)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "ln":
    ln_bench()
