"""Streaming oracle (test infrastructure only): the definition of video_depth.DepthStream in fp32 torch.

There is no reference code for streaming, so this module defines the semantics, built from the pieces of
oracle/vda_oracle.py (pinned to the reference by tests/test_oracle_golden.py):

  * frame t is preprocessed as in infer_video_depth, encoded, and run through the DPT head with T = 1;
  * in each temporal-attention block (motion module m, attention block a) the sequence is
    [n_j for j in ctx(t)] + [n_t], n_j = the block's LayerNorm output for frame j before the positional encoding,
    pe[p] added at position p; the query is the current frame (last position), keys / values the whole sequence;
  * ctx(0) = [], ctx(t) = [0] + [max(1, t - L + 1) .. t - 1], L = 31;
  * the depth is bilinear (align_corners) resized to the frame size and ReLU'd; no alignment between frames.

`forward(causal=True)` is the windowed forward with a causal temporal mask: for t <= 31 streaming frames 0..t equals
it.  `forward(causal=False)` is oracle.forward restated through this module's head, which ties the restatement to the
pinned oracle (tests/test_stream_cpu.py).
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import vda_oracle as O

L_DEFAULT = O.INFER_LEN - 1


def stream_context_ids(t: int, L: int = L_DEFAULT):
    """Context frames of streamed frame t, in position order: frame 0, then the most recent earlier frames."""
    return [] if t == 0 else [0] + list(range(max(1, t - L + 1), t))


def _attend(sd, ab: str, seq: torch.Tensor, q_rows: slice, mask=None, heads: int = 8) -> torch.Tensor:
    """motion_module/attention.py:182-211 on sequences seq [d, S, C] (PE already added): queries seq[:, q_rows], keys
    and values the whole sequence, optional boolean mask [Sq, S] (True = masked); returns to_out(...) [d, Sq, C]."""
    d, S, C = seq.shape
    dh = C // heads
    q = F.linear(seq[:, q_rows], sd[ab + "to_q.weight"])
    Sq = q.shape[1]
    q = q.reshape(d, Sq, heads, dh).transpose(1, 2)
    k = F.linear(seq, sd[ab + "to_k.weight"]).reshape(d, S, heads, dh).transpose(1, 2)
    v = F.linear(seq, sd[ab + "to_v.weight"]).reshape(d, S, heads, dh).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * dh ** -0.5
    if mask is not None:
        s = s.masked_fill(mask, float("-inf"))
    o = (s.softmax(dim=-1) @ v).transpose(1, 2).reshape(d, Sq, C)
    return F.linear(o, sd[ab + "to_out.0.weight"], sd[ab + "to_out.0.bias"])


def _temporal_module(sd, m: int, x: torch.Tensor, T: int, attention) -> torch.Tensor:
    """oracle.temporal_module with the attention of block a given by attention(a, ab, n [T, d, C]) -> [T, d, C]."""
    p = f"head.motion_modules.{m}.temporal_transformer."
    BF, C, hh, ww = x.shape
    res = x
    h = F.group_norm(x, 32, sd[p + "norm.weight"], sd[p + "norm.bias"], 1e-6)
    h = h.permute(0, 2, 3, 1).reshape(BF, hh * ww, C)
    h = F.linear(h, sd[p + "proj_in.weight"], sd[p + "proj_in.bias"])
    blk = p + "transformer_blocks.0."
    for a in (0, 1):
        n = F.layer_norm(h, (C,), sd[f"{blk}norms.{a}.weight"], sd[f"{blk}norms.{a}.bias"], 1e-5)
        h = attention(a, f"{blk}attention_blocks.{a}.", n) + h
    n = F.layer_norm(h, (C,), sd[blk + "ff_norm.weight"], sd[blk + "ff_norm.bias"], 1e-5)
    g = F.linear(n, sd[blk + "ff.net.0.proj.weight"], sd[blk + "ff.net.0.proj.bias"])
    a_, gate = g.chunk(2, dim=-1)
    h = F.linear(a_ * F.gelu(gate), sd[blk + "ff.net.2.weight"], sd[blk + "ff.net.2.bias"]) + h
    h = F.linear(h, sd[p + "proj_out.weight"], sd[p + "proj_out.bias"])
    return h.reshape(BF, hh, ww, C).permute(0, 3, 1, 2) + res


def _dpt_head(sd, taps, hp: int, wp: int, temporal) -> torch.Tensor:
    """oracle.dpt_head with motion module m applied as temporal(m, x)."""
    h = "head."
    out = []
    for i, x in enumerate(taps):
        BT, _, D = x.shape
        x = F.conv2d(x.permute(0, 2, 1).reshape(BT, D, hp, wp), sd[f"{h}projects.{i}.weight"], sd[f"{h}projects.{i}.bias"])
        if i == 0:
            x = F.conv_transpose2d(x, sd[h + "resize_layers.0.weight"], sd[h + "resize_layers.0.bias"], stride=4)
        elif i == 1:
            x = F.conv_transpose2d(x, sd[h + "resize_layers.1.weight"], sd[h + "resize_layers.1.bias"], stride=2)
        elif i == 3:
            x = F.conv2d(x, sd[h + "resize_layers.3.weight"], sd[h + "resize_layers.3.bias"], stride=2, padding=1)
        out.append(x)
    l1, l2, l3, l4 = out
    l3, l4 = temporal(0, l3), temporal(1, l4)
    l1r = F.conv2d(l1, sd[h + "scratch.layer1_rn.weight"], padding=1)
    l2r = F.conv2d(l2, sd[h + "scratch.layer2_rn.weight"], padding=1)
    l3r = F.conv2d(l3, sd[h + "scratch.layer3_rn.weight"], padding=1)
    l4r = F.conv2d(l4, sd[h + "scratch.layer4_rn.weight"], padding=1)
    p4 = temporal(2, O.fusion(sd, 4, l4r, None, size=l3r.shape[2:]))
    p3 = temporal(3, O.fusion(sd, 3, p4, l3r, size=l2r.shape[2:]))
    p2 = O.fusion(sd, 2, p3, l2r, size=l1r.shape[2:])
    p1 = O.fusion(sd, 1, p2, l1r, None)
    o = F.conv2d(p1, sd[h + "scratch.output_conv1.weight"], sd[h + "scratch.output_conv1.bias"], padding=1)
    o = F.interpolate(o, (hp * 14, wp * 14), mode="bilinear", align_corners=True)
    o = F.relu(F.conv2d(o, sd[h + "scratch.output_conv2.0.weight"], sd[h + "scratch.output_conv2.0.bias"], padding=1))
    return F.relu(F.conv2d(o, sd[h + "scratch.output_conv2.2.weight"], sd[h + "scratch.output_conv2.2.bias"]))


@torch.no_grad()
def forward(sd, x: torch.Tensor, encoder: str, causal: bool = True) -> torch.Tensor:
    """oracle.forward of one clip x [1,T,3,H,W] -> [1,T,H,W]; `causal`: frame f's temporal attention sees frames <= f."""
    _, T, _, H, W = x.shape
    hp, wp = H // 14, W // 14
    taps = O.encoder_taps(sd, x.flatten(0, 1), encoder)
    mask = torch.ones(T, T, dtype=torch.bool, device=x.device).triu(1) if causal else None

    def attention(a, ab, n):                                            # n [(f), d, C] -> sequences over f per position
        seq = n.permute(1, 0, 2) + sd[ab + "pos_encoder.pe"][0, :T]
        return _attend(sd, ab, seq, slice(None), mask).permute(1, 0, 2)

    d = _dpt_head(sd, taps, hp, wp, lambda m, y: _temporal_module(sd, m, y, T, attention))
    d = F.relu(F.interpolate(d, size=(H, W), mode="bilinear", align_corners=True))
    return d.squeeze(1)[None]


@torch.no_grad()
def stream_depths(sd, frames_u8: np.ndarray, encoder: str, input_size: int = 518, L: int = L_DEFAULT) -> np.ndarray:
    """Streaming inference frame by frame (module docstring): frames uint8 [N,H0,W0,3] -> float32 [N,H0,W0]."""
    dev = sd["pretrained.cls_token"].device
    h0, w0 = frames_u8.shape[1:3]
    cache, out = {}, []                                 # cache[(m, a)][j] = n_j [hw, C] (fp32)
    for t in range(frames_u8.shape[0]):
        x = torch.from_numpy(O.preprocess_frame(frames_u8[t], input_size))[None].to(dev)
        hp, wp = x.shape[2] // 14, x.shape[3] // 14
        taps = O.encoder_taps(sd, x, encoder)
        ctx = stream_context_ids(t, L)

        def temporal(m, y):
            def attention(a, ab, n):                    # n [1, hw, C]
                c = cache.setdefault((m, a), {})
                c[t] = n[0]
                seq = torch.stack([c[j] for j in ctx] + [n[0]], dim=1)          # [hw, S, C]
                seq = seq + sd[ab + "pos_encoder.pe"][0, :seq.shape[1]]
                return _attend(sd, ab, seq, slice(-1, None)).permute(1, 0, 2)   # [1, hw, C]
            return _temporal_module(sd, m, y, 1, attention)

        d = _dpt_head(sd, taps, hp, wp, temporal)
        d = F.relu(F.interpolate(d, size=(h0, w0), mode="bilinear", align_corners=True))
        out.append(d[0, 0].float().cpu().numpy())
        keep = set(stream_context_ids(t + 1, L))
        for c in cache.values():                        # frames no later step reads
            for j in [j for j in c if j not in keep]:
                del c[j]
    return np.stack(out)
