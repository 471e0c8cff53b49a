"""GPU: batched streaming (VideoDepthAnything.stream_group / DepthStreamGroup, vda_attention_temporal_step_batched):
the batched kernel against its fp32 restatement, group streams against the streaming oracle and against lone streams,
isolation between the streams of a group, one batched step per push, bounded cost, errors."""
import gc

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import stream_oracle as SO  # noqa: E402
from e2e_checks import build_model  # noqa: E402
from oracle import vda_oracle as O  # noqa: E402
from test_stream_gpu import _step_reference  # noqa: E402
from video_depth_anything_b200 import ops  # noqa: E402

TOL = 1e-2
TOL_VALIDATION = 1e-3


def _frames(n, h, w, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (n, h, w, 3), dtype=np.uint8)


def _oracle(sd, frames, enc, size):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.from_numpy(SO.stream_depths({k: v.cuda() for k, v in sd.items()}, frames, enc, input_size=size))


# ---------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("dh", [8, 24, 32, 48, 128])
def test_batched_step_kernel_vs_fp32(dtype, dh):
    g = torch.Generator(device="cuda").manual_seed(100 + dh)
    C, hw, slots, S, stride = 8 * dh, 37, 32, 6, 33
    tol = 1e-2 if dtype == torch.bfloat16 else 2e-3
    ns = [17, 0, 31, None, 1]                               # None: pad row
    rows = [4, 1, 5, -1, 2]                                 # pool entries out of order; 0 and 3 are named by no row
    for scale in (1.0, 12.0):
        qkv = (torch.randn(5 * hw, 3 * C, device="cuda", generator=g) * scale).to(dtype)
        pool = (torch.randn(S, slots, hw, 2 * C, device="cuda", generator=g) * scale).to(dtype)
        pe = torch.randn(32, 3 * C, device="cuda", generator=g)
        ctx = torch.zeros(5, stride, dtype=torch.int32)
        plans = []
        for b, n in enumerate(ns):
            perm = torch.randperm(slots, generator=torch.Generator().manual_seed(b + dh)).tolist()
            write, ctx_slots = perm[0], perm[1:1 + (n or 0)]
            ctx[b, 0], ctx[b, 1] = (n if n is not None else 7), write   # a pad row's n_ctx is ignored
            ctx[b, 2:2 + len(ctx_slots)] = torch.tensor(ctx_slots, dtype=torch.int32)
            plans.append((write, ctx_slots))
        before = pool.clone()
        out = torch.empty(5 * hw, C, dtype=dtype, device="cuda")
        ops.attention_temporal_step(qkv, pool, pe, ctx.cuda(), out,
                                    rows=torch.tensor(rows, dtype=torch.int32, device="cuda"))
        expect = before.clone()
        for b, (n, r, (write, ctx_slots)) in enumerate(zip(ns, rows, plans)):
            q = qkv[b * hw:(b + 1) * hw]
            if n is None:
                ref = _step_reference(q, before[0], pe, 0, [])       # the pad row attends to itself only
            else:
                ref = _step_reference(q, before[r], pe, n, ctx_slots)
                expect[r, write] = q[:, C:]
            err = (out[b * hw:(b + 1) * hw].float() - ref).abs().max().item()
            assert err <= tol * ref.abs().max().item(), (b, n, scale, err)
        assert torch.equal(pool, expect), "only the write slots of the real rows change, with k'|v' as is"


def test_batched_step_kernel_rejects_bad_arguments():
    from video_depth_anything_b200._lib import VdaError
    qkv = torch.zeros(2 * 10, 3 * 64, dtype=torch.bfloat16, device="cuda")
    pool = torch.zeros(2, 4, 10, 128, dtype=torch.bfloat16, device="cuda")
    out = torch.empty(20, 64, dtype=torch.bfloat16, device="cuda")
    pe = torch.zeros(32, 192, device="cuda")
    rows = torch.zeros(2, dtype=torch.int32, device="cuda")
    with pytest.raises(VdaError):                           # a context row needs {n_ctx, write slot}
        ops.attention_temporal_step(qkv, pool, pe, torch.zeros(2, 1, dtype=torch.int32, device="cuda"), out, rows=rows)
    with pytest.raises(VdaError):                           # one slot
        ops.attention_temporal_step(qkv, pool[:, :1].contiguous(), pe, torch.zeros(2, 3, dtype=torch.int32,
                                    device="cuda"), out, rows=rows)


# ---------------------------------------------------------------------------------------------- against the oracle
def _schedule(n_push, opens, seed):
    """Per push, the streams (indices into `opens`, in a random order) it names: stream i is open from push opens[i]."""
    rng = np.random.default_rng(seed)
    out = []
    for p in range(n_push):
        live = [i for i, o in enumerate(opens) if o <= p]
        sub = [i for i in live if rng.random() < (0.95 if i == 0 else 0.7)] or [live[0]]
        out.append([sub[j] for j in rng.permutation(len(sub))])
    return out


def _run_group(group, videos, schedule, opens):
    handles, t, outs = {}, [0] * len(videos), [[] for _ in videos]
    for p, names in enumerate(schedule):
        for i, o in enumerate(opens):
            if o == p:
                handles[i] = group.open()
        got = group.push({handles[i]: videos[i][t[i]] for i in names})
        for i in names:
            outs[i].append(got[handles[i]])
            t[i] += 1
    return [torch.from_numpy(np.stack(o)) for o in outs]


@pytest.fixture(scope="module")
def vits_group_case():
    _, sd = build_model("vits", 0, torch.bfloat16)
    opens = [0, 4, 9]
    schedule = _schedule(44, opens, seed=11)
    counts = [sum(i in s for s in schedule) for i in range(3)]
    assert max(counts) > 32                                 # one stream's context slides
    videos = [_frames(c, 50, 70, seed=20 + i) for i, c in enumerate(counts)]
    refs = [_oracle(sd, v, "vits", 56) for v in videos]
    return videos, schedule, opens, refs


@pytest.mark.parametrize("mode", ["fp16", "bf16", "fp32"])
def test_group_vits_vs_oracle(vits_group_case, mode):
    videos, schedule, opens, refs = vits_group_case
    m, _ = build_model("vits", 0, torch.float16 if mode == "fp16" else torch.bfloat16)
    outs = _run_group(m.stream_group(max_streams=4, input_size=56, fp32=mode == "fp32"), videos, schedule, opens)
    tol = TOL_VALIDATION if mode == "fp32" else TOL
    for i, (got, ref) in enumerate(zip(outs, refs)):
        errs = [O.rel_err(got[t], ref[t])[0] for t in range(len(ref))]
        print(f"vits group {mode} stream {i}: {len(ref)} frames, worst frame rel err {max(errs):.3e}")
        assert max(errs) <= tol, (i, errs)
        assert (got >= 0).all()


def test_group_vitl_518_vs_oracle():
    m, sd = build_model("vitl", 0, torch.bfloat16)
    videos = [_frames(34, 518, 518, seed=30), _frames(34, 518, 518, seed=31)]
    outs = _run_group(m.stream_group(max_streams=2), videos, [[0, 1]] * 34, [0, 0])
    for i, got in enumerate(outs):
        ref = _oracle(sd, videos[i], "vitl", 518)
        errs = [O.rel_err(got[t], ref[t])[0] for t in range(34)]
        print(f"vitl 518x518 group bf16 stream {i}: worst frame rel err {max(errs):.3e}")
        assert max(errs) <= TOL, (i, errs)


# ---------------------------------------------------------------------------------------------- isolation
def test_group_streams_are_isolated():
    m, _ = build_model("vits", 0, torch.bfloat16)
    x, y = _frames(36, 50, 70, seed=40), _frames(36, 50, 70, seed=41)
    sched = _schedule(36, [0, 0, 0], seed=42)
    sched = [[0] + [i for i in s if i] for s in sched]      # stream 0 in every push, neighbours in random subsets
    a = _run_group(m.stream_group(4, 56), [x, x, x], sched, [0, 0, 0])[0]
    b = _run_group(m.stream_group(4, 56), [x, y, y[::-1].copy()], sched, [0, 0, 0])[0]
    assert torch.equal(a, b), "a stream's depths must not depend on what its neighbours push"
    # a closed and reopened handle (same pool row, stale cache contents) starts over like a fresh stream
    g = m.stream_group(2, 56)
    h0, h1 = g.open(), g.open()
    first = [g.push({h0: x[t], h1: y[t]})[h0] for t in range(34)]
    g.close_stream(h0)
    h2 = g.open()
    again = [g.push({h2: x[t], h1: y[t]})[h2] for t in range(34)]
    assert torch.equal(torch.from_numpy(np.stack(first)), torch.from_numpy(np.stack(again)))


# ---------------------------------------------------------------------------------------------- against lone streams
@pytest.mark.parametrize("fp32", [True, False], ids=["fp32", "default"])
def test_group_stream_vs_lone_stream(fp32):
    """Stream 0 pushes in every push, at buckets 1, 2, 4 and 8.  With fp32=True every kernel treats rows alone, so it
    is bit-identical to a lone DepthStream; in the default mode the encoder's LayerNorm fold lays its row statistics
    out by M (vda_gemm_rowstat_layout), so the bucket changes the last bits."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    x = _frames(40, 50, 70, seed=50)
    others = [_frames(40, 50, 70, seed=51 + i) for i in range(7)]
    sizes = [1, 2, 3, 5, 8, 4, 1, 6, 2, 7] * 4               # streams per push -> buckets 1, 2, 4, 8, 8, 4, 1, 8, ...
    sched = [list(range(k)) for k in sizes]
    got = _run_group(m.stream_group(8, 56, fp32=fp32), [x] + others, sched, [0] * 8)[0]
    lone = m.stream(input_size=56, fp32=fp32)
    ref = torch.from_numpy(np.stack([lone.push(f) for f in x]))
    if fp32:
        assert torch.equal(got, ref)
    else:
        errs = [O.rel_err(got[t], ref[t])[0] for t in range(40)]
        print(f"group vs lone stream, default mode: worst frame rel err {max(errs):.3e}")
        assert max(errs) <= TOL


# ---------------------------------------------------------------------------------------------- batched, bounded
def _profiled_push(g, pushes):
    ops.PROFILE = []
    try:
        g.push(pushes)
        torch.cuda.synchronize()
        return list(ops.PROFILE)
    finally:
        ops.PROFILE = None


def test_group_push_is_one_batched_step():
    m, _ = build_model("vits", 0, torch.bfloat16)
    f = _frames(3, 50, 70, seed=60)
    g = m.stream_group(8, 56)
    hs = [g.open() for _ in range(3)]
    g.push({hs[0]: f[0]})                                  # first call: the engine's per-grid caches fill once
    p1 = _profiled_push(g, {hs[0]: f[0]})                                    # bucket 1
    p4 = _profiled_push(g, {h: f[i] for i, h in enumerate(hs)})             # bucket 4 (3 streams + 1 pad row)
    names1, names4 = [n for n, *_ in p1], [n for n, *_ in p4]
    assert names4.count("attention_temporal_step") == 8 and "attention_temporal" not in names4
    assert names1 == names4                                                   # same launches whatever the bucket
    rows1 = [info["M"] for n, info, _, _ in p1 if n == "gemm"]
    rows4 = [info["M"] for n, info, _, _ in p4 if n == "gemm"]
    assert rows1 and rows4 == [4 * r for r in rows1]
    # graphed: the launch count of every bucket's graph is the same
    launches = {}
    for k in (1, 2, 3, 5, 8):
        g2 = m.stream_group(8, 56)
        g2.push({g2.open(): f[i % 3] for i in range(k)})
        (bk, entry), = g2.graphs.items()
        launches[bk] = entry[3]
    assert sorted(launches) == [1, 2, 4, 8] and len(set(launches.values())) == 1, launches


def test_group_cost_is_bounded():
    m, _ = build_model("vits", 0, torch.bfloat16)
    f = _frames(16, 50, 70, seed=70)
    g = m.stream_group(8, 56)
    hs = [g.open() for _ in range(8)]
    rng = np.random.default_rng(71)
    for k in (1, 2, 4, 8):                                    # first use of every bucket
        g.push({h: f[i] for i, h in enumerate(hs[:k])})
    assert sorted(g.graphs) == [1, 2, 4, 8]
    graphs = {k: v[0] for k, v in g.graphs.items()}
    gc.collect()
    mem0 = torch.cuda.memory_allocated()
    for p in range(150):
        if p % 10 == 5:                                        # close and reopen a stream now and then
            i = int(rng.integers(8))
            g.close_stream(hs[i])
            hs[i] = g.open()
        k = int(rng.integers(1, 9))
        sub = [hs[j] for j in rng.permutation(8)[:k]]
        g.push({h: f[(p + j) % 16] for j, h in enumerate(sub)})
    assert {k: v[0] for k, v in g.graphs.items()} == graphs, "no capture after a bucket's first use"
    gc.collect()
    assert torch.cuda.memory_allocated() == mem0


# ---------------------------------------------------------------------------------------------- errors
def test_group_errors():
    m, sd = build_model("vits", 0, torch.bfloat16)
    f = _frames(3, 50, 70, seed=80)
    g = m.stream_group(2, 56)
    a, b = g.open(), g.open()
    with pytest.raises(ValueError):
        g.open()                                              # more than max_streams
    g.push({a: f[0], b: f[1]})
    with pytest.raises(ValueError):
        g.push({a: _frames(1, 60, 70)[0]})                    # another size
    with pytest.raises(ValueError):
        g.push({a: f[0].astype(np.float32)})
    with pytest.raises(ValueError):
        g.push({a: f[0][..., :2]})
    with pytest.raises(ValueError):
        g.push({12345: f[0]})                                 # unknown handle
    with pytest.raises(ValueError):
        g.push([(a, f[0]), (a, f[1])])                        # named twice
    g.close_stream(b)
    with pytest.raises(ValueError):
        g.push({b: f[0]})                                     # closed handle
    with pytest.raises(ValueError):
        g.close_stream(b)
    g2 = m.stream_group(2, 56)
    with pytest.raises(ValueError):
        g2.push({g2.open(): f[0], g2.open(): f[1][:40]})      # sizes differ within the first push
    m.load_state_dict(sd)
    with pytest.raises(RuntimeError):
        g.push({a: f[2]})
    g3 = m.stream_group(2, 56)
    g3.push({g3.open(): f[2]})                                # a new group works
    g3.close()
    with pytest.raises(RuntimeError):
        g3.push({0: f[2]})
    with pytest.raises(RuntimeError):
        g3.open()
