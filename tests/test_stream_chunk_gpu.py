"""GPU: pushes that give a stream several consecutive frames (DepthStream.push / DepthStreamGroup.push with stacks,
vda_attention_temporal_step_causal + vda_stream_cache_store): the kernels against the one-frame kernel run frame by
frame, stacks against one-frame pushes (bit-identical with fp32=True) and the streaming oracle, bounded cost, errors."""
import gc

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import stream_oracle as SO  # noqa: E402
from e2e_checks import build_model  # noqa: E402
from oracle import vda_oracle as O  # noqa: E402
from video_depth_anything_b200 import ops  # noqa: E402
from video_depth_anything_b200.windows import STREAM_CONTEXT, StreamGroupPlan, split_group_table, stream_context  # noqa: E402

TOL = 1e-2


def _frames(n, h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (n, h, w, 3), dtype=np.uint8)


def _chunks(total, sizes):
    out, t = [], 0
    for k in sizes * (total // max(sum(sizes), 1) + 1):
        k = min(k, total - t)
        if k <= 0:
            break
        out.append((t, t + k))
        t += k
    return out


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("dh", [8, 24, 32, 48, 128])
def test_causal_kernel_and_store_vs_one_frame_kernel(dtype, dh):
    """One causal launch + the store against the same rows run one by one through the one-frame batched kernel: a
    stream with 5 frames across the ring wrap (t = 29..33), one with 1 frame at t = 0, one whose push starts at frame 0
    with 3 frames, pool rows out of order, 7 pad rows.  Outputs and the whole pool must be bit-identical."""
    g = torch.Generator(device="cuda").manual_seed(300 + dh)
    L, S, slots, hw, C = STREAM_CONTEXT, 6, 32, 37, 8 * dh
    plan = StreamGroupPlan(S, L)
    hs = [plan.open() for _ in range(S)]
    plan.t[hs[4]] = 29
    handles, counts = [hs[4], hs[1], hs[5]], [5, 1, 3]
    bk, table = plan.step(handles, counts=counts)
    assert bk == 16
    rows, ctx, _ = split_group_table(table, bk, L)
    ctx = ctx.copy()
    ctx[9:, 0], ctx[9:, 2:] = 7, -3                           # pad rows: whatever their context says is ignored
    starts = [(4, 29 + j) for j in range(5)] + [(1, 0)] + [(5, j) for j in range(3)]
    for scale in (1.0, 12.0):
        qkv = (torch.randn(bk * hw, 3 * C, device="cuda", generator=g) * scale).to(dtype)
        pool = (torch.randn(S, slots, hw, 2 * C, device="cuda", generator=g) * scale).to(dtype)
        pe = torch.randn(32, 3 * C, device="cuda", generator=g)
        ref_pool = pool.clone()
        out = torch.empty(bk * hw, C, dtype=dtype, device="cuda")
        rows_d, ctx_d = torch.from_numpy(rows.copy()).cuda(), torch.from_numpy(ctx).cuda()
        ops.attention_temporal_step_causal(qkv, pool, pe, ctx_d, out, rows_d)
        ops.stream_cache_store(qkv, pool, rows_d, ctx_d)
        ref = torch.empty_like(out)
        for b in range(bk):
            s = slice(b * hw, (b + 1) * hw)
            if b < len(starts):
                r, f = starts[b]
                _, sl, write = stream_context(f, L)
                one = torch.tensor([[len(sl), write] + sl + [0] * (L - len(sl))], dtype=torch.int32, device="cuda")
            else:
                r, one = -1, torch.zeros(1, 2 + L, dtype=torch.int32, device="cuda")
            ops.attention_temporal_step(qkv[s], ref_pool, pe, one, ref[s],
                                        rows=torch.tensor([r], dtype=torch.int32, device="cuda"))
        assert torch.equal(out, ref), "rows bit-identical to the one-frame kernel run frame by frame"
        assert torch.equal(pool, ref_pool), "the whole pool, entries no row names included"


def test_causal_kernels_reject_bad_arguments():
    from video_depth_anything_b200._lib import VdaError
    qkv = torch.zeros(2 * 10, 3 * 64, dtype=torch.bfloat16, device="cuda")
    pool = torch.zeros(2, 4, 10, 128, dtype=torch.bfloat16, device="cuda")
    out = torch.empty(20, 64, dtype=torch.bfloat16, device="cuda")
    pe = torch.zeros(32, 192, device="cuda")
    rows = torch.zeros(2, dtype=torch.int32, device="cuda")
    short = torch.zeros(2, 1, dtype=torch.int32, device="cuda")
    ctx3 = torch.zeros(2, 3, dtype=torch.int32, device="cuda")
    with pytest.raises(VdaError):                           # a context row needs {n_ctx, write slot}
        ops.attention_temporal_step_causal(qkv, pool, pe, short, out, rows)
    with pytest.raises(VdaError):                           # one slot
        ops.attention_temporal_step_causal(qkv, pool[:, :1].contiguous(), pe, ctx3, out, rows)
    with pytest.raises(VdaError):
        ops.stream_cache_store(qkv, pool, rows, short)
    with pytest.raises(VdaError):
        ops.stream_cache_store(qkv, pool[:, :1].contiguous(), rows, ctx3)


# ---------------------------------------------------------------------------------------------- end to end, fp32=True
def _stacked(stream, frames, chunks, **kw):
    outs = [stream.push(frames[a:b] if b - a > 1 or a % 2 else frames[a], **kw) for a, b in chunks]
    outs = [o if o.ndim == 3 else o[None] for o in outs]
    return torch.from_numpy(np.concatenate(outs)) if isinstance(outs[0], np.ndarray) else torch.cat(outs).cpu()


def test_vits_stacks_bit_identical_to_one_frame_pushes():
    m, _ = build_model("vits", 0, torch.bfloat16)
    x = _frames(70, 50, 70, seed=90)
    lone = m.stream(56, fp32=True)
    ref = torch.from_numpy(np.stack([lone.push(f) for f in x]))
    got = _stacked(m.stream(56, fp32=True), x, _chunks(70, [1, 4, 7, 16, 2, 13, 5, 9, 3, 10]))
    assert torch.equal(got, ref)


def test_vitl_518_stacks_of_8_vs_one_frame_pushes():
    """ViT-L 518x518, fp32=True, 40 frames in stacks of 8 (bucket 8).  Bit-identical to the same stream pushed one frame
    at a time in a group whose every push runs at bucket 8 (7 other streams alongside), and within 1e-3 of one-frame
    pushes of a lone stream (bucket 1): at ViT-L 518x518 some kernels of the validation engine change their summation
    order with the batch size (DESIGN.md 4.3c), so its last bits depend on the bucket, with or without stacks."""
    m, _ = build_model("vitl", 0, torch.bfloat16)
    x = _frames(40, 518, 518, seed=91)
    others = _frames(8, 518, 518, seed=96)
    g = m.stream_group(8, fp32=True)
    hs = [g.open() for _ in range(8)]
    at8 = torch.from_numpy(np.stack([g.push({hs[0]: f, **{h: others[i] for i, h in enumerate(hs[1:])}})[hs[0]]
                                     for f in x]))
    g.close()
    lone = m.stream(fp32=True)
    one = torch.from_numpy(np.stack([lone.push(f) for f in x]))
    lone.close()
    st = m.stream(fp32=True)
    got = torch.cat([st.push(torch.from_numpy(x[a:a + 8]).cuda(), to_host=False).cpu() for a in range(0, 40, 8)])
    assert torch.equal(got, at8)
    err = max(O.rel_err(got[t], one[t])[0] for t in range(40))
    print(f"vitl 518 fp32 stacks of 8 vs one-frame pushes at bucket 1: worst frame rel err {err:.3e}")
    assert err <= 1e-3


def test_group_mixed_sizes_and_stacks_bit_identical():
    """3 streams, frame sizes 50x70 and 100x140 (one network size), host and CUDA stacks and single frames mixed (the CUDA
    frames with pitched rows and a frame stride that is not H0 * pitch), random subsets and k per push, to_host on and
    off; each stream against a lone stream pushed frame by frame."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    sizes = [(50, 70), (100, 140), (50, 70)]
    videos = [_frames(160, h, w, seed=92 + i) for i, (h, w) in enumerate(sizes)]
    dev = []
    for v, (h, w) in zip(videos, sizes):
        buf = torch.zeros(160, 2, h, w + 3, 3, dtype=torch.uint8, device="cuda")
        buf[:, 0, :, :w] = torch.from_numpy(v).cuda()
        dev.append(buf[:, 0, :, :w])                                    # strides (2 * h * pitch, pitch, 3, 1)
    rng = np.random.default_rng(95)
    g = m.stream_group(3, 56, fp32=True)
    hs = [g.open() for _ in range(3)]
    t, outs = [0, 0, 0], [[], [], []]
    for p in range(26):
        sub = [i for i in range(3) if rng.random() < 0.8] or [0]
        push, ks = {}, {}
        for i in sub:
            k, a, form = int(rng.integers(1, 6)), t[i], int(rng.integers(4))
            push[hs[i]] = [videos[i][a:a + k], dev[i][a:a + k], videos[i][a], dev[i][a]][form]
            ks[i] = k if form < 2 else None
        got = g.push(push, to_host=bool(p % 2))
        for i in sub:
            o = got[hs[i]]
            o = o.cpu() if isinstance(o, torch.Tensor) else torch.from_numpy(o)
            assert tuple(o.shape) == ((ks[i],) if ks[i] else ()) + sizes[i]
            outs[i].append(o if ks[i] else o[None])
            t[i] += ks[i] or 1
    assert min(t) > 32
    for i in range(3):
        lone = m.stream(56, fp32=True)
        ref = torch.from_numpy(np.stack([lone.push(f) for f in videos[i][:t[i]]]))
        lone.close()
        assert torch.equal(torch.cat(outs[i]), ref), i


# ---------------------------------------------------------------------------------------------- default mode
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_vits_stacks_default_mode(dtype):
    m, sd = build_model("vits", 0, dtype)
    x = _frames(40, 50, 70, seed=97)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    oracle = torch.from_numpy(SO.stream_depths({k: v.cuda() for k, v in sd.items()}, x, "vits", input_size=56))
    lone = m.stream(56)
    one = torch.from_numpy(np.stack([lone.push(f) for f in x]))
    got = _stacked(m.stream(56), x, _chunks(40, [3, 8, 1, 16, 5, 2]))
    e_or = max(O.rel_err(got[t], oracle[t])[0] for t in range(40))
    e_one = max(O.rel_err(got[t], one[t])[0] for t in range(40))
    print(f"vits stacks {dtype}: worst frame rel err vs oracle {e_or:.3e}, vs one-frame pushes {e_one:.3e}")
    assert e_or <= TOL and e_one <= TOL
    assert (got >= 0).all()


# ---------------------------------------------------------------------------------------------- cost
def _profiled_push(g, pushes):
    ops.PROFILE = []
    try:
        g.push(pushes)
        torch.cuda.synchronize()
        return [n for n, *_ in ops.PROFILE]
    finally:
        ops.PROFILE = None


def test_causal_step_launches():
    m, _ = build_model("vits", 0, torch.bfloat16)
    f = _frames(8, 50, 70, seed=98)
    g = m.stream_group(4, 56)
    hs = [g.open() for _ in range(2)]
    g.push({hs[0]: f[0]})
    single = _profiled_push(g, {hs[0]: f[1], hs[1]: f[2]})                   # bucket 2
    causal = _profiled_push(g, {hs[0]: f[3:5]})                                 # bucket 2, k = 2
    expect = []
    for n in single:
        expect += ["attention_temporal_step_causal", "stream_cache_store"] if n == "attention_temporal_step" else [n]
    assert causal == expect and causal.count("stream_cache_store") == 8
    g.push({hs[0]: f[5]})                                                       # graphed: bucket 1 (single), then 2 of each
    g.push({hs[0]: f[6], hs[1]: f[7]})
    g.push({hs[1]: f[:2]})
    assert g.causal_graphs[2][3] == g.graphs[2][3] + 8


def test_cost_is_bounded():
    m, _ = build_model("vits", 0, torch.bfloat16)
    f = _frames(16, 50, 70, seed=99)
    g = m.stream_group(4, 56)
    hs = [g.open() for _ in range(4)]
    for k in (1, 2, 4):                                                         # first single-frame use of every bucket
        g.push({h: f[i] for i, h in enumerate(hs[:k])})
    for n in (2, 4, 8, 16):                                                     # first causal use of every bucket
        g.push({hs[0]: f[:n]} if n < 16 else {hs[0]: f[:8], hs[1]: f[8:16]})
    assert sorted(g.graphs) == [1, 2, 4] and sorted(g.causal_graphs) == [2, 4, 8, 16]
    graphs = {k: v[0] for k, v in g.graphs.items()}
    causal = {k: v[0] for k, v in g.causal_graphs.items()}
    gc.collect()
    mem0 = torch.cuda.memory_allocated()
    rng = np.random.default_rng(100)
    for p in range(200):
        if p % 25 == 7:
            i = int(rng.integers(4))
            g.close_stream(hs[i])
            hs[i] = g.open()
        sub = [hs[j] for j in rng.permutation(4)[:int(rng.integers(1, 5))]]
        push, room = {}, 16
        for j, h in enumerate(sub):
            k = int(rng.integers(1, min(8, room - (len(sub) - j - 1)) + 1)) if p % 3 else 1
            push[h] = f[:k] if k > 1 or rng.random() < 0.5 else f[p % 16]
            room -= k
        g.push(push)
    assert {k: v[0] for k, v in g.graphs.items()} == graphs, "no capture after a bucket's first use"
    assert {k: v[0] for k, v in g.causal_graphs.items()} == causal
    gc.collect()
    assert torch.cuda.memory_allocated() == mem0


# ---------------------------------------------------------------------------------------------- errors
def test_stack_errors():
    m, _ = build_model("vits", 0, torch.bfloat16)
    f = _frames(40, 50, 70, seed=101)
    g = m.stream_group(2, 56, max_frames=8)
    a, b = g.open(), g.open()
    g.push({a: f[:3]})
    before = dict(g.plan.t)
    bad = [{a: f[:0]},                                             # k = 0
           {a: np.concatenate([f, f])[:STREAM_CONTEXT + 1]},        # k > L
           {a: f[:5], b: f[:4]},                                    # more frames than max_frames
           {a: _frames(2, 60, 70)},                                 # another size than the stream's first frame
           {b: _frames(2, 60, 70)},                                 # another network size than the group's
           {a: f[:2].astype(np.float32)},
           {a: f[:2, :, :, :2]},
           {a: torch.from_numpy(f[:2]).cuda().permute(0, 2, 1, 3)},   # CUDA stack whose pixels are not contiguous
           {a: f[None, :2]}]                                        # 5-D
    for push in bad:
        with pytest.raises(ValueError):
            g.push(push)
        assert g.plan.t == before and g.plan.size.get(b) is None
    with pytest.raises(ValueError):
        m.stream_group(4, 56, max_frames=2)                         # max_frames below max_streams
    with pytest.raises(ValueError):
        m.infer_video_depth_one(f[:2], input_size=56)               # one frame per call
    assert g.push({a: f[3:5]})[a].shape == (2, 50, 70)
