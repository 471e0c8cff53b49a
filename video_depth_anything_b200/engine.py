"""Host-side engine: packs a reference state dict (SURVEY.md App. C key set) into the layouts the sm_100a
kernels want and sequences the kernels of one forward pass.

Layout rules
  * activations are token-major / NHWC h16 (`[frames, h*w, C]`), so none of the reference's permutes exist;
  * the ViT residual stream is fp32 (as in the reference under autocast: cat with fp32 cls/pos promotes,
    SURVEY.md App. D); the motion-module residual stream is fp32 too;
  * GEMM weights are `[N, K]` row-major h16 (nn.Linear layout); 3x3 conv weights are `[Co, 9*Ci]` with
    K = (ky*3+kx)*Ci + ci; ConvTranspose weights are `[(ky*S+kx)*Co + co, ci]`; GEGLU weights are interleaved
    in blocks of 2*half rows `[a(half) | gate(half)]`;
  * channel counts consumed by the implicit-GEMM conv are zero-padded to a multiple of 64 at pack time
    (only ViT-S needs it: 48->64, 96->128, 32->64).

Reference call sites are cited next to each stage.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List

import torch

from . import ops
from ._lib import ACT_GELU, ACT_NONE, ACT_RELU, EPI_CONVT, EPI_GEGLU, EPI_LINEAR, EPI_TAIL
from .synth import ENCODER_DIMS

KPAD_PATCH = 592   # 3*14*14 = 588 padded to a 16-byte row pitch; the GEMM's TMA zero-fills the K tail


def _pad_to(n: int, m: int) -> int:
    return (n + m - 1) // m * m


# ------------------------------------------------------------------------------------------------
# weight packing helpers (pure tensor reshuffles; run once per load_state_dict)
# ------------------------------------------------------------------------------------------------
def pack_conv3x3(w: torch.Tensor, ci_pad: int, co_pad: int) -> torch.Tensor:
    """[Co,Ci,3,3] -> [co_pad, 9*ci_pad], K index = (ky*3+kx)*ci_pad + ci (matches the conv-mode TMA walk)."""
    co, ci = w.shape[:2]
    out = torch.zeros(co_pad, 3, 3, ci_pad, dtype=w.dtype, device=w.device)
    out[:co, :, :, :ci] = w.permute(0, 2, 3, 1)
    return out.reshape(co_pad, 9 * ci_pad).contiguous()


def pack_convt(w: torch.Tensor, b: torch.Tensor, co_pad: int):
    """ConvTranspose2d weight [Ci,Co,S,S] (kernel == stride) -> [(ky*S+kx)*co_pad + co, Ci]; bias -> [co_pad]."""
    ci, co, s, _ = w.shape
    out = torch.zeros(s, s, co_pad, ci, dtype=w.dtype, device=w.device)
    out[:, :, :co, :] = w.permute(2, 3, 1, 0)
    bp = torch.zeros(co_pad, dtype=torch.float32, device=w.device)
    bp[:co] = b.float()
    return out.reshape(s * s * co_pad, ci).contiguous(), bp


def pack_geglu(w: torch.Tensor, b: torch.Tensor, half: int):
    """GEGLU proj weight [2*inner, C] (rows: value | gate, motion_module/attention.py:382-384) -> row blocks
    [value(half) | gate(half)] so one GEMM tile holds both operands of a*gelu(g)."""
    inner = w.shape[0] // 2
    assert inner % half == 0
    a, g = w[:inner].reshape(inner // half, half, -1), w[inner:].reshape(inner // half, half, -1)
    wp = torch.cat([a, g], dim=1).reshape(2 * inner, -1).contiguous()
    ba, bg = b[:inner].reshape(inner // half, half), b[inner:].reshape(inner // half, half)
    bp = torch.cat([ba, bg], dim=1).reshape(2 * inner).contiguous().float()
    return wp, bp


class Engine:
    def __init__(self, encoder: str, features: int, out_channels: List[int], dtype=torch.bfloat16,
                 device="cuda", num_frames: int = 32, weight_split: bool = False):
        if encoder not in ENCODER_DIMS:
            raise ValueError(f"unknown encoder {encoder!r}")
        self.encoder = encoder
        e = ENCODER_DIMS[encoder]
        self.D, self.depth, self.heads, self.taps = e["embed_dim"], e["depth"], e["num_heads"], e["taps"]
        self.F = features
        self.oc = list(out_channels)
        self.dtype = dtype
        # The DPT head runs on fp16 operands even when the encoder uses bf16: its activations are bounded (post-ReLU
        # conv features; the reference runs the whole model under fp16 autocast), so it takes fp16's three extra
        # mantissa bits, while the encoder keeps bf16's range for the residual stream's large-magnitude channels.
        # Same tensor-core rate.  Measured on vits 2x518x518: the head took the bf16 error from 3.3e-3 (taps) to
        # 1.03e-2 (depth); the 1e-2 bar of BASELINE.json failed by one pixel.
        self.hdtype = torch.float16
        # LayerNorm folded into the consumer GEMMs of the encoder (proj / fc2 epilogues emit a 16-bit copy of the residual
        # stream and per-row statistics; qkv / fc1 apply mean / rstd in their epilogues): removes 2 of the 2.04 LayerNorm
        # launches per block.
        # Validation precision (`fp32=True`): every GEMM / conv weight is a hi | lo pair of 16-bit matrices (22 mantissa
        # bits; the GEMM walks A twice), activations stay 16-bit with fp32 accumulation / residuals / statistics.  Twice the
        # tensor work; the LayerNorm fold is off (one rounding less on the normalised rows).
        self.weight_split = weight_split
        self.ln_fold = not weight_split
        self.device = torch.device(device)
        self.num_frames = num_frames
        self.w: Dict[str, torch.Tensor] = {}
        self._pos_cache: Dict[tuple, torch.Tensor] = {}
        self.loaded = False
        self.generation = 0          # bumped by every load(): streams opened on older weights refuse to continue
        # One CUDA graph per input shape: a forward is ~330 back-to-back kernel launches with no host decisions,
        # so it is captured once and replayed (removes launch gaps and the host-side descriptor encoding).
        self.use_graphs = os.environ.get("VDA_NO_GRAPH", "0") != "1"
        self.launches_per_forward = 0
        self._graphs: Dict[tuple, tuple] = {}
        self._bufs: Dict[tuple, list] = {}
        # channel paddings (see module docstring)
        self.c_l1 = _pad_to(self.oc[0], 64)
        self.c_l2 = _pad_to(self.oc[1], 64)
        self.c_oc1 = _pad_to(self.F // 2, 64)
        assert self.oc[2] % 64 == 0 and self.oc[3] % 64 == 0 and self.F % 64 == 0

    # -------------------------------------------------------------------------------------------
    def load(self, sd: Dict[str, torch.Tensor]) -> None:
        dev, dt = self.device, self.dtype
        w = self.w = {}
        self._pos_cache = {}
        self._graphs = {}        # captured graphs hold pointers to the old packed weights
        self._bufs = {}

        def f32(k):
            return sd[k].detach().to(dev, torch.float32).contiguous()

        split = self.weight_split

        def h16(t):
            t = t.to(dev, torch.float32)
            return ops.split_hi_lo(t.reshape(t.shape[0], -1), dt) if split else t.to(dt).contiguous()

        def fold_ln(wk, bk, nk):
            """(h16(g * W), c1 = row sums of the ROUNDED folded matrix, c2 = W beta + b) for y = LN(x) W^T + b."""
            W = sd[wk].detach().to(dev, torch.float32)
            g, beta = f32(nk + ".weight"), f32(nk + ".bias")
            wf = (W * g[None, :]).to(dt).contiguous()
            # both vectors summed in double and rounded once: independent of the summation order, so the C engine
            # (csrc/model.cu, host loops) packs the same bits
            c1 = wf.double().sum(1).float().contiguous()
            c2 = (W.double() @ beta.double() + f32(bk).double()).float().contiguous()
            return wf, c1, c2

        D = self.D
        pw = sd["pretrained.patch_embed.proj.weight"].detach().to(dev, torch.float32).reshape(D, 588)
        pwp = torch.zeros(D, KPAD_PATCH, device=dev)
        pwp[:, :588] = pw
        w["pe.w"], w["pe.b"] = h16(pwp), f32("pretrained.patch_embed.proj.bias")
        w["cls"] = f32("pretrained.cls_token").reshape(D)
        w["pos"] = f32("pretrained.pos_embed").reshape(-1, D)
        for i in range(self.depth):
            p = f"pretrained.blocks.{i}."
            for n in ("norm1", "norm2"):
                w[f"b{i}.{n}.w"], w[f"b{i}.{n}.b"] = f32(p + n + ".weight"), f32(p + n + ".bias")
            for n, k in (("qkv", "attn.qkv"), ("proj", "attn.proj"), ("fc1", "mlp.fc1"), ("fc2", "mlp.fc2")):
                w[f"b{i}.{n}.w"], w[f"b{i}.{n}.b"] = h16(sd[p + k + ".weight"]), f32(p + k + ".bias")
            w[f"b{i}.ls1"], w[f"b{i}.ls2"] = f32(p + "ls1.gamma"), f32(p + "ls2.gamma")
            if self.ln_fold:
                w[f"b{i}.qkv.wf"], w[f"b{i}.qkv.c1"], w[f"b{i}.qkv.c2"] = fold_ln(p + "attn.qkv.weight", p + "attn.qkv.bias", p + "norm1")
                w[f"b{i}.fc1.wf"], w[f"b{i}.fc1.c1"], w[f"b{i}.fc1.c2"] = fold_ln(p + "mlp.fc1.weight", p + "mlp.fc1.bias", p + "norm2")
        w["norm.w"], w["norm.b"] = f32("pretrained.norm.weight"), f32("pretrained.norm.bias")

        h = "head."
        oc, F = self.oc, self.F
        hdt = self.hdtype

        def h16(t):                                    # head weights: head operand type  # noqa: F811
            t = t.to(dev, torch.float32)
            return ops.split_hi_lo(t.reshape(t.shape[0], -1), hdt) if split else t.to(hdt).contiguous()
        for i in range(4):
            w[f"proj{i}.w"] = h16(sd[f"{h}projects.{i}.weight"].reshape(oc[i], D))
            w[f"proj{i}.b"] = f32(f"{h}projects.{i}.bias")
        wt, bt = pack_convt(sd[h + "resize_layers.0.weight"].to(dev, torch.float32), sd[h + "resize_layers.0.bias"].to(dev), self.c_l1)
        w["rs0.w"], w["rs0.b"] = h16(wt), bt
        wt, bt = pack_convt(sd[h + "resize_layers.1.weight"].to(dev, torch.float32), sd[h + "resize_layers.1.bias"].to(dev), self.c_l2)
        w["rs1.w"], w["rs1.b"] = h16(wt), bt
        w["rs3.w"] = h16(pack_conv3x3(sd[h + "resize_layers.3.weight"].to(dev, torch.float32), oc[3], oc[3]))
        w["rs3.b"] = f32(h + "resize_layers.3.bias")
        cin = [self.c_l1, self.c_l2, oc[2], oc[3]]
        for i in range(4):
            w[f"rn{i + 1}.w"] = h16(pack_conv3x3(sd[f"{h}scratch.layer{i + 1}_rn.weight"].to(dev, torch.float32), cin[i], F))
        for r in (1, 2, 3, 4):
            rp = f"{h}scratch.refinenet{r}."
            w[f"rf{r}.out.w"] = h16(sd[rp + "out_conv.weight"].reshape(F, F))
            w[f"rf{r}.out.b"] = f32(rp + "out_conv.bias")
            for u in (1, 2):
                for c in (1, 2):
                    k = f"{rp}resConfUnit{u}.conv{c}."
                    w[f"rf{r}.u{u}.c{c}.w"] = h16(pack_conv3x3(sd[k + "weight"].to(dev, torch.float32), F, F))
                    w[f"rf{r}.u{u}.c{c}.b"] = f32(k + "bias")
        w["oc1.w"] = h16(pack_conv3x3(sd[h + "scratch.output_conv1.weight"].to(dev, torch.float32), F, self.c_oc1))
        b = torch.zeros(self.c_oc1, device=dev)
        b[:F // 2] = sd[h + "scratch.output_conv1.bias"].to(dev, torch.float32)
        w["oc1.b"] = b
        w["oc2.w"] = pack_conv3x3(sd[h + "scratch.output_conv2.0.weight"].to(dev, torch.float32), self.c_oc1, 32) \
            .to(hdt).contiguous()                      # (the fused tail kernel reads it directly: always a plain matrix)
        w["oc2.b"] = f32(h + "scratch.output_conv2.0.bias")
        w["oc3.w"] = f32(h + "scratch.output_conv2.2.weight").reshape(32)
        self.oc3_b = float(sd[h + "scratch.output_conv2.2.bias"].reshape(-1)[0])

        self.mm_c = [oc[2], oc[3], F, F]
        for m, C in enumerate(self.mm_c):
            t = f"{h}motion_modules.{m}.temporal_transformer."
            w[f"mm{m}.gn.w"], w[f"mm{m}.gn.b"] = f32(t + "norm.weight"), f32(t + "norm.bias")
            w[f"mm{m}.in.w"], w[f"mm{m}.in.b"] = h16(sd[t + "proj_in.weight"]), f32(t + "proj_in.bias")
            w[f"mm{m}.out.w"], w[f"mm{m}.out.b"] = h16(sd[t + "proj_out.weight"]), f32(t + "proj_out.bias")
            blk = t + "transformer_blocks.0."
            for a in (0, 1):
                ab = f"{blk}attention_blocks.{a}."
                w[f"mm{m}.a{a}.qkv.w"] = h16(torch.cat([sd[ab + "to_q.weight"], sd[ab + "to_k.weight"], sd[ab + "to_v.weight"]], 0))
                w[f"mm{m}.a{a}.o.w"], w[f"mm{m}.a{a}.o.b"] = h16(sd[ab + "to_out.0.weight"]), f32(ab + "to_out.0.bias")
                w[f"mm{m}.a{a}.pe"] = f32(ab + "pos_encoder.pe").reshape(-1, C)
                # streaming: q|k|v = (n + pe[p]) W^T = n W^T + pe[p] W^T, so cached frames keep n W_k^T | n W_v^T and the
                # step kernel adds this positional share (fp32, rounded once from double) at the position a frame has now
                wqkv = torch.cat([sd[ab + "to_q.weight"], sd[ab + "to_k.weight"], sd[ab + "to_v.weight"]], 0)
                pe32 = sd[ab + "pos_encoder.pe"].reshape(-1, C)[:32].double()
                w[f"mm{m}.a{a}.pet"] = (pe32 @ wqkv.double().t()).to(dev, torch.float32).contiguous()
                w[f"mm{m}.a{a}.ln.w"], w[f"mm{m}.a{a}.ln.b"] = f32(f"{blk}norms.{a}.weight"), f32(f"{blk}norms.{a}.bias")
            w[f"mm{m}.ffn.w"], w[f"mm{m}.ffn.b"] = f32(blk + "ff_norm.weight"), f32(blk + "ff_norm.bias")
            half = 128 if (4 * C) % 128 == 0 else 64
            wp, bp = pack_geglu(sd[blk + "ff.net.0.proj.weight"].to(dev, torch.float32),
                                sd[blk + "ff.net.0.proj.bias"].to(dev, torch.float32), half)
            w[f"mm{m}.ff0.w"], w[f"mm{m}.ff0.b"] = h16(wp), bp
            self.__dict__.setdefault("mm_half", {})[m] = half
            w[f"mm{m}.ff2.w"], w[f"mm{m}.ff2.b"] = h16(sd[blk + "ff.net.2.weight"]), f32(blk + "ff.net.2.bias")
        self.generation += 1
        self.loaded = True

    # -------------------------------------------------------------------------------------------
    def _pos(self, hp: int, wp: int) -> torch.Tensor:
        """dinov2.py:179-210; cached per grid (the reference recomputes it every call)."""
        key = (hp, wp)
        if key not in self._pos_cache:
            pos = self.w["pos"]
            S = int(round(math.sqrt(pos.shape[0] - 1)))
            if hp == S and wp == S:
                self._pos_cache[key] = pos
            else:
                self._pos_cache[key] = ops.pos_embed_bicubic(pos, hp, wp)
        return self._pos_cache[key]

    def _const(self, value: float, n: int) -> torch.Tensor:
        """Cached fp32 constant vector (zero bias / unit LayerScale that route a GEMM to a compile-time specialised
        epilogue; adding 0 and multiplying by 1 are exact)."""
        key = ("const", value, n)
        if key not in self._bufs:
            self._bufs[key] = [torch.full((n,), value, dtype=torch.float32, device=self.device)]
        return self._bufs[key][0]

    def _new(self, *shape, dtype=None):
        return torch.empty(*shape, dtype=dtype or self.dtype, device=self.device)

    def _hnew(self, *shape, dtype=None):
        """Head activation buffer (head operand type)."""
        return torch.empty(*shape, dtype=dtype or self.hdtype, device=self.device)

    # -------------------------------------------------------------------------------------------
    def encode(self, x: torch.Tensor, stages=None) -> List[torch.Tensor]:
        """DINOv2 get_intermediate_layers (dinov2.py:297-321).  x fp32 [BT,3,H,W] -> 4 x h16 [BT*P, D]."""
        w, D = self.w, self.D
        BT, _, H, W = x.shape
        hp, wp = H // 14, W // 14
        P, N = hp * wp, hp * wp + 1
        M = BT * N
        pos = self._pos(hp, wp)
        a = self._new(BT * P, KPAD_PATCH)
        ops.patch_im2col(x, a)                                                        # patch_embed.py:66,76
        tok = self._new(BT, N, D, dtype=torch.float32)
        tok2 = tok.view(M, D)
        ops.gemm(a, w["pe.w"], tok2, bias=w["pe.b"], res1=pos, row_group=P)            # + pos_embed (dinov2.py:219)
        ops.write_cls(tok, w["cls"], pos)                                              # dinov2.py:218
        del a
        if stages is not None:
            stages["tokens0"] = tok.clone()
        ln = self._new(M, D)
        qkv = self._new(M, 3 * D)
        att = self._new(M, D)
        hid = self._new(M, 4 * D)
        taps = []
        # LayerNorm fold: possible when the residual GEMM's tile geometry for [M, D] has a row-statistics layout
        layout = self._fold_layout(M, D) if self.ln_fold else None
        if layout is not None:
            stats = self._new(M, layout[0], 2, dtype=torch.float32)
            ops.rowstats_cast(tok2, ln, stats)            # `ln` holds the 16-bit copy of the residual stream from here on
        for i in range(self.depth):                                                   # block.py:82-107
            b = f"b{i}."
            if layout is not None:
                # norm1 / norm2 are applied inside the qkv / fc1 epilogues; proj / fc2 refresh the 16-bit rows + statistics
                ops.gemm(ln, w[b + "qkv.wf"], qkv, bias=w[b + "qkv.c2"], ln_fold=(stats, w[b + "qkv.c1"], 1e-6))
                ops.attention_spatial(qkv, att, BT, N, self.heads)
                ops.gemm(att, w[b + "proj.w"], tok2, bias=w[b + "proj.b"], gamma=w[b + "ls1"], res1=tok2, out16=ln,
                         row_stats_out=stats)
                ops.gemm(ln, w[b + "fc1.wf"], hid, bias=w[b + "fc1.c2"], act=ACT_GELU, ln_fold=(stats, w[b + "fc1.c1"], 1e-6))
                last = i == self.depth - 1            # nothing consumes the copy after the last block
                ops.gemm(hid, w[b + "fc2.w"], tok2, bias=w[b + "fc2.b"], gamma=w[b + "ls2"], res1=tok2,
                         out16=None if last else ln, row_stats_out=None if last else stats)
            else:
                ops.layernorm(tok2, w[b + "norm1.w"], w[b + "norm1.b"], 1e-6, ln)
                ops.gemm(ln, w[b + "qkv.w"], qkv, bias=w[b + "qkv.b"])                     # attention.py:51
                ops.attention_spatial(qkv, att, BT, N, self.heads)                         # attention.py:53-59
                ops.gemm(att, w[b + "proj.w"], tok2, bias=w[b + "proj.b"], gamma=w[b + "ls1"], res1=tok2)
                ops.layernorm(tok2, w[b + "norm2.w"], w[b + "norm2.b"], 1e-6, ln)
                ops.gemm(ln, w[b + "fc1.w"], hid, bias=w[b + "fc1.b"], act=ACT_GELU)       # mlp.py:36-37
                ops.gemm(hid, w[b + "fc2.w"], tok2, bias=w[b + "fc2.b"], gamma=w[b + "ls2"], res1=tok2)
            if stages is not None:
                stages[f"block{i}"] = tok.clone()
            if i in self.taps:                                                         # dinov2.py:309-312
                t = self._hnew(BT * P, D)
                ops.layernorm(tok2, w["norm.w"], w["norm.b"], 1e-6, t, drop_group=N)
                taps.append(t)
        return taps

    def _fold_layout(self, M: int, D: int):
        """(parts, part_cols) of the residual GEMMs' row statistics for an [M, D] token matrix, None if their tile
        geometry has none (tiny problems take narrower tiles)."""
        key = ("fold", M, D)
        if key not in self._pos_cache:
            try:
                self._pos_cache[key] = ops.rowstat_layout(M, D)
            except Exception:                       # noqa: BLE001  (VdaError: no layout)
                self._pos_cache[key] = None
        return self._pos_cache[key]

    # -------------------------------------------------------------------------------------------
    def _conv3(self, x, key, n, H, W, ci, co, **kw):
        out = kw.pop("out", None)
        if out is None:
            out = self._hnew(n * H * W, co)
        return ops.gemm(x, self.w[key + ".w"], out, bias=self.w.get(key + ".b"), conv_shape=(n, H, W, ci), **kw)

    def _rcu(self, r, u, x, x_relu, n, H, W, extra=None, want_relu=False):
        """ResidualConvUnit (util/blocks.py:68-91): conv2(relu(conv1(relu(x)))) + x [+ extra]."""
        F = self.F
        t = self._conv3(x_relu, f"rf{r}.u{u}.c1", n, H, W, F, F, act=ACT_RELU)
        out = self._hnew(n * H * W, F)
        out_relu = self._hnew(n * H * W, F) if want_relu else None
        self._conv3(t, f"rf{r}.u{u}.c2", n, H, W, F, F, out=out, res1=x, res2=extra, out_relu=out_relu)
        return out, out_relu

    def _fusion(self, r, x0, skip, skip_relu, n, H, W, oh, ow):
        """FeatureFusionBlock (util/blocks.py:135-162).  x0: upstream path (None for refinenet4),
        skip / skip_relu: layer_rn output and its relu'd copy.  The 1x1 out_conv is applied BEFORE the bilinear
        upsample: the two commute exactly in real arithmetic (interpolation weights sum to one) and it is 4x
        cheaper there (SURVEY.md App. H.2)."""
        F = self.F
        if x0 is None:
            cur, cur_relu = skip, skip_relu
        else:
            cur, cur_relu = self._rcu(r, 1, skip, skip_relu, n, H, W, extra=x0, want_relu=True)
        u, _ = self._rcu(r, 2, cur, cur_relu, n, H, W)
        o = self._hnew(n * H * W, F)
        ops.gemm(u, self.w[f"rf{r}.out.w"], o, bias=self.w[f"rf{r}.out.b"])
        up = self._hnew(n * oh * ow, F)
        ops.bilinear_nhwc(o, up, n, H, W, oh, ow, F)
        return up

    def _motion(self, m, x, B, T, hw, stream=None):
        """TemporalModule (motion_module.py:60-65, 102-126, 164-177).  x h16 [B*T*hw, C] rows (b, f, pos).
        `stream` = (pool, rows, ctx[, causal]): one streamed frame per batch row (T = 1) whose temporal attention reads its
        stream's cached frames (stream_group_step); `causal`: context entries may name earlier rows of the batch, and the
        rows' k'|v' go to the pool after the attention."""
        w, C = self.w, self.mm_c[m]
        M = B * T * hw
        p = f"mm{m}."
        gn = self._hnew(M, C)
        ops.groupnorm(x, w[p + "gn.w"], w[p + "gn.b"], 1e-6, gn, B * T, hw)              # :110
        h = self._hnew(M, C, dtype=torch.float32)
        ops.gemm(gn, w[p + "in.w"], h, bias=w[p + "in.b"])                              # :113
        n = gn                                                                          # reuse as LN output
        qkv = self._hnew(M, 3 * C)
        o = self._hnew(M, C)
        for a in (0, 1):                                                                # :165-172
            if stream is None:
                ops.layernorm(h, w[f"{p}a{a}.ln.w"], w[f"{p}a{a}.ln.b"], 1e-5, n, pe=w[f"{p}a{a}.pe"], pe_rows_per_frame=hw,
                              pe_frames=T)                 # rows are (clip, frame, position): frame = (r // hw) % T
                ops.gemm(n, w[f"{p}a{a}.qkv.w"], qkv, bias=self._const(0.0, 3 * C))   # zero bias: takes the specialised epilogue
                for b in range(B):
                    s = slice(b * T * hw, (b + 1) * T * hw)
                    ops.attention_temporal(qkv[s], o[s], T, hw, C)
            else:                                          # positional encoding enters through the `pet` table
                ops.layernorm(h, w[f"{p}a{a}.ln.w"], w[f"{p}a{a}.ln.b"], 1e-5, n)
                ops.gemm(n, w[f"{p}a{a}.qkv.w"], qkv, bias=self._const(0.0, 3 * C))
                if len(stream) > 3 and stream[3]:
                    ops.attention_temporal_step_causal(qkv, stream[0][2 * m + a], w[f"{p}a{a}.pet"], stream[2], o, stream[1])
                    ops.stream_cache_store(qkv, stream[0][2 * m + a], stream[1], stream[2])
                else:
                    ops.attention_temporal_step(qkv, stream[0][2 * m + a], w[f"{p}a{a}.pet"], stream[2], o, rows=stream[1])
            ops.gemm(o, w[f"{p}a{a}.o.w"], h, bias=w[f"{p}a{a}.o.b"], gamma=self._const(1.0, C), res1=h)   # unit LayerScale: ditto
        ops.layernorm(h, w[p + "ffn.w"], w[p + "ffn.b"], 1e-5, n)                        # :174
        g = self._hnew(M, 4 * C)
        ops.gemm(n, w[p + "ff0.w"], g, bias=w[p + "ff0.b"], epilogue=EPI_GEGLU, geglu_half=self.mm_half[m])
        h16 = o
        ops.gemm(g, w[p + "ff2.w"], h16, bias=w[p + "ff2.b"], res1=h)                    # ff + residual, h16 out
        out = self._hnew(M, C)
        ops.gemm(h16, w[p + "out.w"], out, bias=w[p + "out.b"], res1=x)                  # :120-125
        return out

    def head(self, taps, B, T, hp, wp, stages=None, stream=None) -> torch.Tensor:
        """DPTHeadTemporal.forward (dpt_temporal.py:53-114) -> fp32 [B*T, 14hp, 14wp].  `stream`: see _motion."""
        w, F, oc = self.w, self.F, self.oc
        BT = B * T
        P = hp * wp
        pr = []
        for i in range(4):                                                              # :66 projects[i]
            o = self._hnew(BT * P, oc[i])
            ops.gemm(taps[i], w[f"proj{i}.w"], o, bias=w[f"proj{i}.b"])
            pr.append(o)
        h1, w1, h2, w2 = 4 * hp, 4 * wp, 2 * hp, 2 * wp
        h4, w4 = (hp - 1) // 2 + 1, (wp - 1) // 2 + 1
        l1 = self._hnew(BT * h1 * w1, self.c_l1)                                          # :67 resize_layers
        ops.gemm(pr[0], w["rs0.w"], l1, bias=w["rs0.b"], epilogue=EPI_CONVT, convt=(4, self.c_l1, hp, wp))
        l2 = self._hnew(BT * h2 * w2, self.c_l2)
        ops.gemm(pr[1], w["rs1.w"], l2, bias=w["rs1.b"], epilogue=EPI_CONVT, convt=(2, self.c_l2, hp, wp))
        l3 = pr[2]
        col = ops.im2col3x3_s2(pr[3], BT, hp, wp, oc[3])
        l4 = self._hnew(BT * h4 * w4, oc[3])
        ops.gemm(col, w["rs3.w"], l4, bias=w["rs3.b"])
        del col
        if stages is not None:
            stages.update(layer_1=(l1, h1, w1), layer_2=(l2, h2, w2), layer_3=(l3, hp, wp), layer_4=(l4, h4, w4))
        l3 = self._motion(0, l3, B, T, P, stream)                                       # :75
        l4 = self._motion(1, l4, B, T, h4 * w4, stream)                                 # :76
        if stages is not None:
            stages.update(mm0=(l3, hp, wp), mm1=(l4, h4, w4))

        def rn(i, x, H, W, ci):                                                         # :78-81 layer{i}_rn (+ relu'd copy)
            o, orl = self._hnew(BT * H * W, F), self._hnew(BT * H * W, F)
            ops.gemm(x, w[f"rn{i}.w"], o, conv_shape=(BT, H, W, ci), out_relu=orl)
            return o, orl

        l1r, l1rr = rn(1, l1, h1, w1, self.c_l1)
        l2r, l2rr = rn(2, l2, h2, w2, self.c_l2)
        l3r, l3rr = rn(3, l3, hp, wp, oc[2])
        l4r, l4rr = rn(4, l4, h4, w4, oc[3])
        del l1, l2, l4
        if stages is not None:
            stages.update(layer_1_rn=(l1r, h1, w1), layer_2_rn=(l2r, h2, w2), layer_3_rn=(l3r, hp, wp), layer_4_rn=(l4r, h4, w4))
        p4 = self._fusion(4, None, l4r, l4rr, BT, h4, w4, hp, wp)                        # :83
        if stages is not None:
            stages["path_4_pre"] = (p4, hp, wp)
        p4 = self._motion(2, p4, B, T, P, stream)                                       # :84
        p3 = self._fusion(3, p4, l3r, l3rr, BT, hp, wp, h2, w2)                          # :85
        if stages is not None:
            stages.update(path_4=(p4, hp, wp), path_3_pre=(p3, h2, w2))
        p3 = self._motion(3, p3, B, T, h2 * w2, stream)                                 # :86
        p2 = self._fusion(2, p3, l2r, l2rr, BT, h2, w2, h1, w1)                          # :90/103
        p1 = self._fusion(1, p2, l1r, l1rr, BT, h1, w1, 2 * h1, 2 * w1)                  # :91/104
        if stages is not None:
            stages.update(path_3=(p3, h2, w2), path_2=(p2, h1, w1), path_1=(p1, 2 * h1, 2 * w1))
        del l1r, l1rr, l2r, l2rr, l3r, l3rr, l4r, l4rr, p2, p3, p4
        H8, W8 = 2 * h1, 2 * w1
        o1 = self._conv3(p1, "oc1", BT, H8, W8, F, self.c_oc1)                           # :92/105 output_conv1
        if stages is not None:
            stages["output_conv1"] = (o1, H8, W8)
        del p1
        H, W = 14 * hp, 14 * wp
        depth = self._hnew(BT, H, W, dtype=torch.float32)
        # :94-100 bilinear 296->518 + output_conv2 (3x3 -> ReLU -> 1x1 -> ReLU) in one kernel: the upsampled
        # 128-channel map (2.2 GB per window) is never materialised
        ops.tail_fused(o1, w["oc2.w"], w["oc2.b"], w["oc3.w"], self.oc3_b, depth, BT, H8, W8, H, W, self.c_oc1)
        return depth

    # -------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x: torch.Tensor, stages=None) -> torch.Tensor:
        """VideoDepthAnything.forward (video_depth.py:89-164): x [B,T,3,H,W] -> fp32 [B,T,H,W]."""
        if not self.loaded:
            raise RuntimeError("weights not loaded (call load_state_dict first)")
        if x.dim() != 5 or x.shape[2] != 3:
            raise ValueError(f"expected x of shape [B,T,3,H,W], got {tuple(x.shape)}")
        B, T, _, H, W = x.shape
        assert H % 14 == 0, f"Input image height {H} is not a multiple of patch height 14"    # patch_embed.py:73
        assert W % 14 == 0, f"Input image width {W} is not a multiple of patch width: 14"     # patch_embed.py:74
        if T > self.num_frames:
            raise ValueError(f"T={T} exceeds temporal_max_len={self.num_frames} (dpt_temporal.py:38)")
        if not x.is_cuda:
            raise RuntimeError("the engine has no CPU path; move the input to the B200")
        x = x.to(torch.float32).contiguous()
        if self.use_graphs and stages is None and ops.PROFILE is None:
            return self._forward_graph(x)
        return self._forward_eager(x, stages)

    def _graphed(self, key: tuple, fn, inputs: List[torch.Tensor], adopt: bool = False):
        """Run `fn(*inputs)` as a CUDA graph captured once per `key` in the engine's own bounded cache (run_graphed)."""
        if key not in self._graphs and len(self._graphs) >= 6:   # bound the memory held by private graph pools
            self._graphs.pop(next(iter(self._graphs)))
        return self.run_graphed(self._graphs, key, fn, inputs, adopt)

    @staticmethod
    def run_graphed(graphs: Dict[tuple, tuple], key: tuple, fn, inputs: List[torch.Tensor], adopt: bool = False):
        """Run `fn(*inputs)` (a fixed sequence of libvda launches, no host decisions) as a CUDA graph captured once
        per `key` into `graphs`; returns the graph's static outputs (valid until the next call with the same key).
        `adopt`: the caller's tensors are long-lived buffers and become the graph's inputs themselves (no staging copy)."""
        entry = graphs.get(key)
        if entry is None:
            static_in = list(inputs) if adopt else [t.clone() for t in inputs]
            n0 = ops.LAUNCHES
            fn(*static_in)                                  # warm-up: lazy caches, kernel attributes
            launches = ops.LAUNCHES - n0
            torch.cuda.current_stream().synchronize()
            graph = torch.cuda.CUDAGraph()
            # thread-local capture: the video driver's drain thread waits on copy-stream events (cudaEventSynchronize)
            # while a window's graph may be captured; in the default global mode that call from another thread
            # invalidates the capture, although it never touches the capturing stream
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                static_out = fn(*static_in)
            entry = graphs[key] = (graph, static_in, static_out, launches)
        graph, static_in, static_out, launches = entry
        for s, t in zip(static_in, inputs):
            if s.data_ptr() != t.data_ptr():
                s.copy_(t)
        graph.replay()
        ops.LAUNCHES += launches
        return static_out

    def _forward_graph(self, x: torch.Tensor) -> torch.Tensor:
        out = self._graphed(("fwd",) + tuple(x.shape), self._forward_eager, [x])
        self.launches_per_forward = self._graphs[("fwd",) + tuple(x.shape)][3]
        return out.clone()

    # ------------------------------------------------------------------------------------------- split forward
    def encode_frames(self, x: torch.Tensor) -> List[torch.Tensor]:
        """Encoder only, for the feature-reusing video driver: x fp32 [n,3,H,W] -> 4 x h16 [n*P, D] (static graph
        outputs when graphs are on: consume before the next call with the same n)."""
        # steady-state frame counts (a full window, or the 22 new frames of a follow-up window) replay a graph; the odd
        # counts at the ends of a video run eagerly once instead of paying a capture
        if self.use_graphs and ops.PROFILE is None and x.shape[0] in (32, 22):
            return self._graphed(("enc",) + tuple(x.shape), lambda t: self.encode(t), [x])
        return self.encode(x)

    def head_static_inputs(self, T: int, hp: int, wp: int) -> List[torch.Tensor]:
        """The head graph's own input buffers (4 x h16 [T*P, D]); the video driver gathers cached features straight
        into them, so `head_frames` does no extra copy."""
        key = ("head_in", T, hp, wp)
        if key not in self._bufs:
            self._bufs[key] = [self._hnew(T * hp * wp, self.D) for _ in range(4)]
        return self._bufs[key]

    def head_frames(self, taps: List[torch.Tensor], T: int, hp: int, wp: int) -> torch.Tensor:
        """Head only: 4 x h16 [T*P, D] -> fp32 [T, 14hp, 14wp] (one clip)."""
        if self.use_graphs and ops.PROFILE is None:
            own = self.head_static_inputs(T, hp, wp)
            adopt = all(a.data_ptr() == b.data_ptr() for a, b in zip(taps, own))
            return self._graphed(("head", T, hp, wp, adopt), lambda *t: self.head(list(t), 1, T, hp, wp), list(taps), adopt)
        return self.head(list(taps), 1, T, hp, wp)

    def _forward_eager(self, x: torch.Tensor, stages=None) -> torch.Tensor:
        B, T, _, H, W = x.shape
        x = x.flatten(0, 1)
        hp, wp = H // 14, W // 14
        taps = self.encode(x, stages)
        if stages is not None:
            for i, t in enumerate(taps):
                stages[f"tap{i}"] = t
        depth = self.head(taps, B, T, hp, wp, stages)
        # video_depth.py:162-163: bilinear to (H,W) is the identity (14*hp == H) and the ReLU is already applied
        return depth.view(B, T, H, W)

    # ------------------------------------------------------------------------------------------- streaming
    def stream_pool(self, S: int, hp: int, wp: int, slots: int) -> List[torch.Tensor]:
        """Temporal context of S streams.  Per temporal-attention block (index 2 * motion module + attention block) the
        k'|v' rows of `slots` frames of every stream: head dtype [S, slots, hw, 2C], row = k' (C) | v' (C) of one
        position, so one head's keys and values are contiguous 16-byte runs."""
        hws = [hp * wp, ((hp - 1) // 2 + 1) * ((wp - 1) // 2 + 1), hp * wp, 4 * hp * wp]
        return [self._hnew(S, slots, hws[m], 2 * self.mm_c[m]) for m in range(4) for _ in (0, 1)]

    def stream_group_step(self, frame_desc: torch.Tensor, out_desc: torch.Tensor, rows: torch.Tensor, ctx: torch.Tensor,
                          pool: List[torch.Tensor], nh: int, nw: int, causal: bool = False) -> None:
        """One streamed frame of each of B streams, every frame of its own size: batch row b reads the frame frame_desc[b]
        and writes its depth fp32 [H0,W0] (>= 0) to out_desc[b] (vda_frame_desc / vda_out_desc arrays, device bytes,
        windows.group_descriptors), takes pool entry rows[b] (int32 [B], -1: pad row) and context row ctx[b] (int32
        [B, stride], see vda_attention_temporal_step_batched).  Preprocessing to (nh, nw) as in infer_video_depth,
        encoder and head on the B frames at T = 1 with every temporal attention against the rows' pool entries, bilinear
        resize to each row's frame size.  The launches depend on neither B nor the sizes.  No host decisions:
        graph-capturable, and every frame-dependent address is read from the descriptors at run time.
        `causal`: rows may be consecutive frames of one stream (ctx entries < 0 name earlier rows of the batch,
        vda_attention_temporal_step_causal); each temporal attention is then followed by the pool write of the rows'
        k'|v' (vda_stream_cache_store): 8 more launches, nothing else differs."""
        x = ops.preprocess_frames_ragged(frame_desc, nh, nw)
        d = self.head(self.encode(x), rows.numel(), 1, nh // 14, nw // 14, stream=(pool, rows, ctx, causal))
        ops.bilinear_f32_ragged(d, out_desc)
