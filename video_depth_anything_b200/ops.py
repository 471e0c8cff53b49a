"""Thin torch-tensor wrappers over the libvda C ABI.  torch is only used for device memory and streams; every
arithmetic operation below runs in the hand-written sm_100a kernels.  Each wrapper names the reference operator
it replaces."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import (A_CONV3, A_PLAIN, ACT_GELU, ACT_NONE, ACT_RELU, EPI_CONVT, EPI_GEGLU, EPI_LINEAR, EPI_TAIL,
                   GemmParams, VDA_BF16, VDA_FP16, check)

LSQ_MAX_PARTIALS = 592   # include/vda.h VDA_LSQ_MAX_PARTIALS
FRAME_DESC_BYTES, OUT_DESC_BYTES = 24, 16   # sizeof(vda_frame_desc), sizeof(vda_out_desc)
LAUNCHES = 0   # number of libvda kernel launches issued (bench.py reports it as gpu_launches)
PROFILE = None  # when a list: every op appends (name, info dict, start_event, end_event)   [bench.py / tools]
_INFO = {}


def dt_code(t: torch.dtype) -> int:
    if t == torch.bfloat16:
        return VDA_BF16
    if t == torch.float16:
        return VDA_FP16
    raise TypeError(f"16-bit operand type must be bfloat16 or float16, got {t}")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda, "libvda operates on CUDA tensors only (no CPU fallback)"
    return t.data_ptr()


def _count(n=1):
    global LAUNCHES
    LAUNCHES += n


def split_hi_lo(w: torch.Tensor, dtype) -> torch.Tensor:
    """fp32 weight matrix [N, K] -> h16 [N, 2 * round_up(K, 64)] = [h16(W) | h16(W - h16(W))] (zero padded): the operand
    format of the validation-precision GEMMs (vda_gemm_params.a_k)."""
    N, K = w.shape
    kp = (K + 63) // 64 * 64
    hi = w.to(dtype)
    lo = (w - hi.float()).to(dtype)
    out = torch.zeros(N, 2 * kp, dtype=dtype, device=w.device)
    out[:, :K] = hi
    out[:, kp:kp + K] = lo
    return out


def rowstat_layout(M: int, N: int):
    """(parts, part_cols) of the per-row partial statistics a residual GEMM with `row_stats` writes for an [M, N] output."""
    lib = _lib.load()
    a, b = C.c_int(0), C.c_int(0)
    check(lib.vda_gemm_rowstat_layout(M, N, C.byref(a), C.byref(b)))
    return a.value, b.value


def gemm(a: torch.Tensor, wt: torch.Tensor, out: torch.Tensor, *, bias=None, gamma=None, act=ACT_NONE,
         res1=None, res2=None, out_relu=None, row_group=0, epilogue=EPI_LINEAR,
         conv_shape=None, geglu_half=0, convt=None, tail_w=None, tail_b=0.0, M=None,
         out16=None, row_stats_out=None, ln_fold=None) -> torch.Tensor:
    """out = epilogue(a @ wt.T).  a: [M,K] h16 (row stride allowed) or NHWC [n,H,W,C] with conv_shape=(n,H,W,C);
    wt: [N,K] h16 contiguous.  Replaces F.linear / F.conv2d(1x1, 3x3 s1 p1) / F.conv_transpose2d(k == s)."""
    lib = _lib.load()
    p = GemmParams()
    N, K = wt.shape
    assert wt.is_contiguous() and wt.dtype == a.dtype
    p.N, p.K, p.dtype = N, K, dt_code(a.dtype)
    p.epilogue = epilogue
    if conv_shape is not None:
        n, H, W, Cc = conv_shape
        assert a.is_contiguous() and a.numel() == n * H * W * Cc
        p.a_mode, p.n_img, p.H, p.W, p.C = A_CONV3, n, H, W, Cc
        p.M, p.lda = n * H * W, Cc
        ka = 9 * Cc
    else:
        assert a.dim() == 2 and a.stride(1) == 1
        p.a_mode = A_PLAIN
        p.M, p.lda = (a.shape[0] if M is None else M), a.stride(0)
        ka = a.shape[1]
    if K != ka:      # weights packed as a hi | lo pair (split_hi_lo): A is walked twice
        assert K == 2 * ((ka + 63) // 64 * 64), (a.shape, wt.shape)
        p.a_k = ka
    p.A, p.Wt = _p(a), _p(wt)
    p.bias, p.gamma, p.act = _p(bias), _p(gamma), act
    if res1 is not None:
        p.res1, p.ldr1, p.res1_f32 = _p(res1), res1.stride(-2), int(res1.dtype == torch.float32)
        assert res1.stride(-1) == 1 and (res1.dtype == torch.float32 or res1.dtype == a.dtype)
    if res2 is not None:
        assert res2.dtype == a.dtype and res2.stride(-1) == 1
        p.res2 = _p(res2)
    p.out, p.out_f32 = _p(out), int(out.dtype == torch.float32)
    assert out.dtype == torch.float32 or out.dtype == a.dtype
    if epilogue == EPI_TAIL:
        p.ldo = 1
        p.tail_w, p.tail_b = _p(tail_w), float(tail_b)
    else:
        assert out.stride(-1) == 1
        p.ldo = out.stride(-2)
        if res2 is not None:
            assert res2.stride(-2) == p.ldo
        if out_relu is not None:
            assert out_relu.stride(-2) == p.ldo and out_relu.dtype == a.dtype
    p.out_relu = _p(out_relu)
    p.row_group = row_group
    p.geglu_half = geglu_half
    if convt is not None:
        p.convt_s, p.convt_co, p.in_h, p.in_w = convt
    if out16 is not None or row_stats_out is not None:
        # producer side of the LayerNorm fold: h16 copy of the new fp32 rows + per-row partial (mean, M2)
        if out16 is not None:
            assert out16.dtype == a.dtype and out16.stride(-2) == p.ldo and out16.stride(-1) == 1
            p.out16 = _p(out16)
        if row_stats_out is not None:
            assert row_stats_out.dtype == torch.float32 and row_stats_out.is_contiguous() and row_stats_out.shape[-1] == 2
            p.row_stats_out, p.stat_parts = _p(row_stats_out), row_stats_out.shape[-2]
    if ln_fold is not None:
        # consumer side: ln_fold = (row_stats [M, parts, 2] fp32, c1 [N] fp32, eps); `a` holds the un-normalised rows,
        # `wt` the LayerNorm-weight-scaled matrix, `bias` = W @ ln_bias + b
        stats, c1, eps = ln_fold
        assert stats.dtype == torch.float32 and stats.is_contiguous() and stats.shape[-1] == 2 and c1.dtype == torch.float32
        p.row_stats_in, p.ln_c1, p.ln_eps = _p(stats), _p(c1), float(eps)
        p.stat_parts = stats.shape[-2]
        assert K % p.stat_parts == 0
        p.stat_cols = K // p.stat_parts
    if PROFILE is not None:
        _INFO.update(kind=("conv3x3" if conv_shape is not None else "gemm") + f"/epi{epilogue}",
                     M=int(p.M), N=int(N), K=int(ka), flops=2.0 * p.M * N * ka)
    check(lib.vda_gemm(C.byref(p), _stream()))
    _count()
    return out


def layernorm(x: torch.Tensor, w, b, eps: float, out: torch.Tensor, *, drop_group=0, pe=None, pe_rows_per_frame=0,
              pe_frames=0):
    """nn.LayerNorm over the last dim; x fp32 or h16 [rows, C] -> out h16."""
    lib = _lib.load()
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    assert x.is_contiguous() and out.is_contiguous()
    if PROFILE is not None:
        _INFO.update(kind="layernorm", bytes=float(x.numel() * x.element_size() + out.numel() * out.element_size()))
    check(lib.vda_layernorm(_p(x), int(x.dtype == torch.float32), _p(out), _p(w), _p(b), eps, rows, Cc,
                            dt_code(out.dtype), drop_group, _p(pe), pe_rows_per_frame,
                            0 if pe is None else (pe_frames or pe.shape[0]), _stream()))
    _count()
    return out


def rowstats_cast(x: torch.Tensor, out16: torch.Tensor, stats: torch.Tensor):
    """fp32 rows [M, C] -> h16 copy + per-row partial statistics [M, parts, 2] (start of the LayerNorm-fold chain)."""
    lib = _lib.load()
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    parts = stats.shape[-2]
    assert x.is_contiguous() and x.dtype == torch.float32 and out16.is_contiguous() and stats.is_contiguous()
    assert stats.dtype == torch.float32 and Cc % parts == 0
    if PROFILE is not None:
        _INFO.update(kind="rowstats_cast", bytes=float(x.numel() * 4 + out16.numel() * 2))
    check(lib.vda_rowstats_cast(_p(x), _p(out16), _p(stats), rows, Cc, parts, Cc // parts, dt_code(out16.dtype), _stream()))
    _count()
    return out16


def groupnorm(x: torch.Tensor, w, b, eps: float, out: torch.Tensor, frames: int, hw: int, groups: int = 32):
    """nn.GroupNorm(groups, C) per frame over NHWC h16 [frames, hw, C]."""
    lib = _lib.load()
    Cc = x.shape[-1]
    stats = torch.empty((592 + 2 * frames) * groups * 2, dtype=torch.float32, device=x.device)   # VDA_GN_STATS_FLOATS
    check(lib.vda_groupnorm(_p(x), _p(out), _p(w), _p(b), eps, frames, hw, Cc, groups, _p(stats), dt_code(x.dtype),
                            _stream()))
    _count(3)
    return out


def attention_spatial(qkv: torch.Tensor, out: torch.Tensor, frames: int, N: int, heads: int):
    lib = _lib.load()
    assert qkv.is_contiguous() and out.is_contiguous()
    if PROFILE is not None:
        _INFO.update(kind="attention_spatial", flops=4.0 * frames * heads * N * N * 64)
    check(lib.vda_attention_spatial(_p(qkv), _p(out), frames, N, heads, dt_code(qkv.dtype), _stream()))
    _count()
    return out


def attention_temporal(qkv: torch.Tensor, out: torch.Tensor, T: int, hw: int, Cc: int, heads: int = 8):
    lib = _lib.load()
    assert qkv.is_contiguous() and out.is_contiguous()
    check(lib.vda_attention_temporal(_p(qkv), _p(out), T, hw, Cc, heads, dt_code(qkv.dtype), _stream()))
    _count()
    return out


def attention_temporal_step(qkv: torch.Tensor, cache: torch.Tensor, pe: torch.Tensor, ctx: torch.Tensor, out: torch.Tensor,
                            heads: int = 8, rows: Optional[torch.Tensor] = None):
    """Streaming temporal attention (vda.h vda_attention_temporal_step[_batched]).  One frame: qkv h16 [hw, 3C] (q'|k'|v',
    no positional encoding), cache h16 [slots, hw, 2C] (k'|v' rows of earlier frames), pe fp32 [32, 3C] (positional share
    of q|k|v), ctx device int32 [>= 2] = (n_ctx, write slot, context slots...) -> out h16 [hw, C].
    B frames of different streams (`rows` device int32 [B], pool index per batch row, -1 = pad row): qkv [B*hw, 3C],
    cache = the pool h16 [S, slots, hw, 2C], ctx [B, stride] one row as above per batch row -> out [B*hw, C]."""
    lib = _lib.load()
    C3 = qkv.shape[1]
    Cc = C3 // 3
    B = 1 if rows is None else rows.numel()
    hw = qkv.shape[0] // B
    assert qkv.is_contiguous() and cache.is_contiguous() and pe.is_contiguous() and out.is_contiguous()
    assert cache.shape[-2:] == (hw, 2 * Cc) and cache.dtype == qkv.dtype and out.dtype == qkv.dtype
    assert qkv.shape[0] == B * hw and out.shape == (B * hw, Cc)
    assert pe.dtype == torch.float32 and pe.shape[-1] == C3 and pe.shape[0] >= 32
    assert ctx.dtype == torch.int32 and ctx.is_contiguous() and ctx.numel() >= 2
    if PROFILE is not None:      # bytes of a full 31-frame context: cached k'|v' rows read, current q|k|v in, out + slot out
        _INFO.update(kind="attention_temporal_step",
                     bytes=float(qkv.element_size() * B * hw * (31 * 2 * Cc + 3 * Cc + Cc + 2 * Cc)))
    if rows is None:
        assert cache.dim() == 3
        check(lib.vda_attention_temporal_step(_p(qkv), _p(cache), _p(pe), _p(ctx), _p(out), hw, Cc, heads,
                                              cache.shape[0], dt_code(qkv.dtype), _stream()))
    else:
        assert cache.dim() == 4 and rows.dtype == torch.int32 and rows.is_contiguous() and ctx.dim() == 2
        assert ctx.shape[0] == B
        check(lib.vda_attention_temporal_step_batched(_p(qkv), _p(cache), _p(pe), _p(rows), _p(ctx), _p(out), B,
                                                      cache.shape[0], ctx.shape[1], hw, Cc, heads, cache.shape[1],
                                                      dt_code(qkv.dtype), _stream()))
    _count()
    return out


def attention_temporal_step_causal(qkv: torch.Tensor, pool: torch.Tensor, pe: torch.Tensor, ctx: torch.Tensor,
                                   out: torch.Tensor, rows: torch.Tensor, heads: int = 8):
    """Streaming temporal attention of several consecutive frames per stream in one launch (vda.h
    vda_attention_temporal_step_causal): as attention_temporal_step with `rows`, but a context entry e < 0 reads batch row
    -1 - e's k'|v' from `qkv`, and the pool is only read (stream_cache_store writes the new frames afterwards)."""
    lib = _lib.load()
    Cc = qkv.shape[1] // 3
    B = rows.numel()
    hw = qkv.shape[0] // B
    assert qkv.is_contiguous() and pool.is_contiguous() and pe.is_contiguous() and out.is_contiguous()
    assert pool.dim() == 4 and pool.shape[-2:] == (hw, 2 * Cc) and pool.dtype == qkv.dtype and out.dtype == qkv.dtype
    assert qkv.shape[0] == B * hw and out.shape == (B * hw, Cc)
    assert pe.dtype == torch.float32 and pe.shape[-1] == 3 * Cc and pe.shape[0] >= 32
    assert rows.dtype == torch.int32 and rows.is_contiguous()
    assert ctx.dtype == torch.int32 and ctx.is_contiguous() and ctx.dim() == 2 and ctx.shape[0] == B
    if PROFILE is not None:
        # no `bytes`: which context frames come from the pool and which from the push's own rows (already read as q'|k'|v')
        # is in the device table, so the HBM traffic is not known here (tools/bench_stream.py counts it per stack size);
        # key_row_bytes counts every k'|v' row read, wherever it comes from
        _INFO.update(kind="attention_temporal_step_causal",
                     key_row_bytes=float(qkv.element_size() * B * hw * 31 * 2 * Cc))
    check(lib.vda_attention_temporal_step_causal(_p(qkv), _p(pool), _p(pe), _p(rows), _p(ctx), _p(out), B, pool.shape[0],
                                                 ctx.shape[1], hw, Cc, heads, pool.shape[1], dt_code(qkv.dtype), _stream()))
    _count()
    return out


def stream_cache_store(qkv: torch.Tensor, pool: torch.Tensor, rows: torch.Tensor, ctx: torch.Tensor):
    """The cache write of a causal step (vda.h vda_stream_cache_store): every real row's k'|v' (qkv [B*hw, 3C], columns
    C..3C) -> pool[rows[b]] h16 [S, slots, hw, 2C], slot ctx[b, 1]."""
    lib = _lib.load()
    Cc = qkv.shape[1] // 3
    B = rows.numel()
    hw = qkv.shape[0] // B
    assert qkv.is_contiguous() and pool.is_contiguous() and pool.dim() == 4 and pool.dtype == qkv.dtype
    assert qkv.shape[0] == B * hw and pool.shape[-2:] == (hw, 2 * Cc)
    assert rows.dtype == torch.int32 and rows.is_contiguous()
    assert ctx.dtype == torch.int32 and ctx.is_contiguous() and ctx.dim() == 2 and ctx.shape[0] == B
    if PROFILE is not None:      # k'|v' rows read and written
        _INFO.update(kind="stream_cache_store", bytes=float(qkv.element_size() * B * hw * 4 * Cc))
    check(lib.vda_stream_cache_store(_p(qkv), _p(pool), _p(rows), _p(ctx), B, pool.shape[0], ctx.shape[1], hw, Cc,
                                     pool.shape[1], dt_code(qkv.dtype), _stream()))
    _count()
    return pool


def preprocess_frames(frames_u8: torch.Tensor, idx: torch.Tensor, nh: int, nw: int) -> torch.Tensor:
    """uint8 RGB [N,H0,W0,3] (device) + int32 frame indices [n] (device) -> normalised fp32 [n,3,nh,nw]
    (util/transform.py Resize(INTER_CUBIC) / NormalizeImage / PrepareForNet)."""
    lib = _lib.load()
    assert frames_u8.is_contiguous() and frames_u8.dtype == torch.uint8 and frames_u8.dim() == 4 and frames_u8.shape[3] == 3
    assert idx.dtype == torch.int32 and idx.is_contiguous()
    n = idx.numel()
    out = torch.empty(n, 3, nh, nw, dtype=torch.float32, device=frames_u8.device)
    check(lib.vda_preprocess_frames(_p(frames_u8), _p(idx), _p(out), n, frames_u8.shape[1], frames_u8.shape[2], nh, nw,
                                    _stream()))
    _count()
    return out


def preprocess_frames_ragged(rows: torch.Tensor, nh: int, nw: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One frame per batch row, each of its own size: rows = the vda_frame_desc array (device bytes [n * 24],
    windows.FRAME_DESC) -> fp32 [n,3,nh,nw], per row what preprocess_frames gives for that frame alone."""
    lib = _lib.load()
    assert rows.dtype == torch.uint8 and rows.is_contiguous() and rows.numel() % FRAME_DESC_BYTES == 0
    n = rows.numel() // FRAME_DESC_BYTES
    if out is None:
        out = torch.empty(n, 3, nh, nw, dtype=torch.float32, device=rows.device)
    assert out.is_contiguous() and out.dtype == torch.float32 and tuple(out.shape) == (n, 3, nh, nw)
    check(lib.vda_preprocess_frames_ragged(_p(rows), n, nh, nw, _p(out), _stream()))
    _count()
    return out


def copy_frames(src: torch.Tensor, src_idx: Optional[torch.Tensor], dst: torch.Tensor, dst_idx: Optional[torch.Tensor],
                n: int) -> torch.Tensor:
    """dst[dst_idx[i]] = src[src_idx[i]] for i < n over the leading (frame) axis; idx: device int32 or None (identity)."""
    lib = _lib.load()
    assert src.is_contiguous() and dst.is_contiguous() and src.dtype == dst.dtype
    fb = src[0].numel() * src.element_size()
    assert fb == dst[0].numel() * dst.element_size()
    for ix in (src_idx, dst_idx):
        assert ix is None or (ix.dtype == torch.int32 and ix.is_contiguous() and ix.numel() >= n)
    check(lib.vda_copy_frames(_p(src), _p(src_idx), _p(dst), _p(dst_idx), n, fb, _stream()))
    _count()
    return dst


def patch_im2col(x: torch.Tensor, out: torch.Tensor):
    """x fp32 [frames,3,H,W] -> out h16 [frames*hp*wp, kpad]"""
    lib = _lib.load()
    frames, _, H, W = x.shape
    assert x.is_contiguous() and x.dtype == torch.float32
    check(lib.vda_patch_im2col(_p(x), _p(out), frames, H, W, out.shape[1], dt_code(out.dtype), _stream()))
    _count()
    return out


def write_cls(tokens: torch.Tensor, cls_token: torch.Tensor, pos: torch.Tensor):
    lib = _lib.load()
    frames, tpf, D = tokens.shape
    check(lib.vda_write_cls(_p(tokens), _p(cls_token), _p(pos), frames, tpf, D, _stream()))
    _count()


def pos_embed_bicubic(pos_in: torch.Tensor, hp: int, wp: int) -> torch.Tensor:
    lib = _lib.load()
    n, D = pos_in.shape
    S = int(round((n - 1) ** 0.5))
    out = torch.empty(1 + hp * wp, D, dtype=torch.float32, device=pos_in.device)
    check(lib.vda_pos_embed_bicubic(_p(pos_in), _p(out), S, hp, wp, D, _stream()))
    _count()
    return out


def im2col3x3_s2(x: torch.Tensor, n: int, H: int, W: int, Cc: int) -> torch.Tensor:
    lib = _lib.load()
    oh, ow = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty(n * oh * ow, 9 * Cc, dtype=x.dtype, device=x.device)
    check(lib.vda_im2col3x3_s2(_p(x), _p(out), n, H, W, Cc, dt_code(x.dtype), _stream()))
    _count()
    return out


def bilinear_nhwc(x: torch.Tensor, out: torch.Tensor, n: int, ih: int, iw: int, oh: int, ow: int, Cc: int):
    lib = _lib.load()
    check(lib.vda_bilinear_nhwc(_p(x), _p(out), n, ih, iw, oh, ow, Cc, dt_code(x.dtype), _stream()))
    _count()
    return out


def tail_fused(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, w2: torch.Tensor, b2: float, out: torch.Tensor,
               n: int, ih: int, iw: int, oh: int, ow: int, Cc: int):
    """depth = relu(w2 . relu(conv3x3(bilinear(x -> oh x ow)) + bias) + b2); x h16 NHWC [n,ih,iw,Cc] -> out fp32 [n,oh,ow]."""
    lib = _lib.load()
    assert x.is_contiguous() and w.is_contiguous() and out.is_contiguous() and out.dtype == torch.float32
    assert w.shape == (32, 9 * Cc) and w.dtype == x.dtype
    if PROFILE is not None:
        _INFO.update(kind="tail_fused", flops=2.0 * n * oh * ow * 32 * 9 * Cc)
    check(lib.vda_tail_fused(_p(x), _p(w), _p(bias), _p(w2), float(b2), _p(out), n, ih, iw, oh, ow, Cc,
                             dt_code(x.dtype), _stream()))
    _count()
    return out


def bilinear_f32(x: torch.Tensor, oh: int, ow: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = _lib.load()
    n, ih, iw = x.shape
    assert x.is_contiguous() and x.dtype == torch.float32
    if out is None:
        out = torch.empty(n, oh, ow, dtype=torch.float32, device=x.device)
    assert out.is_contiguous() and out.dtype == torch.float32 and tuple(out.shape) == (n, oh, ow)
    check(lib.vda_bilinear_f32(_p(x), _p(out), n, ih, iw, oh, ow, _stream()))
    _count()
    return out


def bilinear_f32_ragged(x: torch.Tensor, rows: torch.Tensor) -> None:
    """x fp32 [n,ih,iw] -> row i resized (align_corners=True) into its vda_out_desc rows[i] (device bytes [n * 16],
    windows.OUT_DESC): dst [H0,W0], bit-identical to bilinear_f32 of that row alone; H0 = 0 writes nothing."""
    lib = _lib.load()
    n, ih, iw = x.shape
    assert x.is_contiguous() and x.dtype == torch.float32
    assert rows.dtype == torch.uint8 and rows.is_contiguous() and rows.numel() == n * OUT_DESC_BYTES
    check(lib.vda_bilinear_f32_ragged(_p(x), _p(rows), n, ih, iw, _stream()))
    _count()


def add_h16(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor):
    lib = _lib.load()
    check(lib.vda_add_h16(_p(a), _p(b), _p(out), a.numel(), dt_code(a.dtype), _stream()))
    _count()
    return out


def lsq_scale_shift(pred: torch.Tensor, target: torch.Tensor, scale_shift: torch.Tensor, scratch: torch.Tensor):
    lib = _lib.load()
    assert pred.is_contiguous() and target.is_contiguous() and pred.numel() == target.numel()
    assert scratch.dtype == torch.float64 and scratch.numel() >= 4 * LSQ_MAX_PARTIALS
    check(lib.vda_lsq_scale_shift(_p(pred), _p(target), pred.numel(), _p(scale_shift), _p(scratch), _stream()))
    _count(2)


def align_chain(anchors: torch.Tensor, table: torch.Tensor, scratch: torch.Tensor, affine: bool = True):
    """(scale, shift) of every window from the gathered anchor frames: anchors fp32 [K,3,h,w] (raw slots 0, 1, 12) ->
    table fp32 [K,2]; one cooperative kernel, bit-identical to WindowAligner's per-window recurrence."""
    lib = _lib.load()
    K = anchors.shape[0]
    assert anchors.is_contiguous() and anchors.dtype == torch.float32 and anchors.shape[1] == 3
    assert table.is_contiguous() and table.dtype == torch.float32 and table.numel() == 2 * K
    assert scratch.dtype == torch.float64 and scratch.numel() >= 8 * LSQ_MAX_PARTIALS
    check(lib.vda_align_chain(_p(anchors), K, anchors[0, 0].numel(), int(bool(affine)), _p(table), _p(scratch), _stream()))
    _count()
    return table


def affine_clamp_blend(x: torch.Tensor, scale_shift: torch.Tensor, out: torch.Tensor, prev=None, blend_w=None):
    lib = _lib.load()
    frames = x.shape[0]
    hw = x.numel() // frames
    assert x.is_contiguous() and out.is_contiguous()
    check(lib.vda_affine_clamp_blend(_p(x), _p(scale_shift), _p(prev), _p(blend_w), _p(out), frames, hw, _stream()))
    _count()
    return out


def _profiled(fn, name):
    import functools

    @functools.wraps(fn)
    def wrapper(*a, **k):
        if PROFILE is None:
            return fn(*a, **k)
        _INFO.clear()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r = fn(*a, **k)
        e.record()
        PROFILE.append((name, dict(_INFO), s, e))
        return r
    return wrapper


for _n in ("preprocess_frames", "preprocess_frames_ragged", "copy_frames", "gemm", "layernorm", "rowstats_cast", "groupnorm", "attention_spatial", "attention_temporal",
           "attention_temporal_step", "attention_temporal_step_causal", "stream_cache_store", "patch_im2col", "write_cls",
           "pos_embed_bicubic", "im2col3x3_s2", "bilinear_nhwc", "tail_fused", "bilinear_f32", "bilinear_f32_ragged", "add_h16", "lsq_scale_shift", "align_chain",
           "affine_clamp_blend"):
    globals()[_n] = _profiled(globals()[_n], _n)
