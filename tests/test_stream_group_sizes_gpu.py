"""GPU: stream groups with a frame size per stream and frames / depths in device memory: the ragged ingest and egress
kernels (vda_preprocess_frames_ragged, vda_bilinear_f32_ragged) against their uniform siblings row by row, mixed-size
groups against the streaming oracle and against lone streams, CUDA frames and CUDA depths against the host path,
bounded cost, errors."""
import gc

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from e2e_checks import build_model  # noqa: E402
from oracle import vda_oracle as O  # noqa: E402
from test_stream_group_gpu import TOL, TOL_VALIDATION, _oracle, _schedule  # noqa: E402
from video_depth_anything_b200 import ops  # noqa: E402
from video_depth_anything_b200.windows import group_descriptors  # noqa: E402

SIZES = [(25, 35), (50, 70), (56, 84), (100, 140)]       # smaller, equal to and larger than the network size (56, 84)
NET = (56, 84)


def _frame(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _dev_bytes(arr):
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8)).cuda()


# ---------------------------------------------------------------------------------------------- kernels
def test_ragged_ingest_matches_uniform_kernel_per_row():
    frames = [torch.from_numpy(_frame(h, w, 10 + i)).cuda() for i, (h, w) in enumerate(SIZES)]
    big = torch.from_numpy(_frame(120, 160, 20)).cuda()
    frames.append(big[7:107, 11:151])                         # a pitched view: 100 x 140, row pitch 480 bytes
    assert frames[-1].stride() == (480, 3, 1) and not frames[-1].is_contiguous()
    idx0 = torch.zeros(1, dtype=torch.int32, device="cuda")
    expect = [ops.preprocess_frames(f.contiguous()[None], idx0, *NET)[0] for f in frames]
    descs = [(f.data_ptr(), f.stride(0), f.shape[0], f.shape[1]) for f in frames]
    for rows in ([0], [1], [2], [3], [4], [4, 0, 3, 2, 1, 4]):   # each kind alone, then a batch mixing all of them
        fd, _ = group_descriptors(len(rows), [descs[r] for r in rows], [0] * len(rows))
        got = ops.preprocess_frames_ragged(_dev_bytes(fd), *NET)
        for b, r in enumerate(rows):
            assert torch.equal(got[b], expect[r]), (rows, b)
    # pad rows (bucket larger than the push) read row 0's frame
    fd, _ = group_descriptors(4, [descs[1], descs[3]], [0, 0])
    got = ops.preprocess_frames_ragged(_dev_bytes(fd), *NET)
    assert torch.equal(got[2], expect[1]) and torch.equal(got[3], expect[1])


def test_ragged_egress_matches_uniform_kernel_per_row():
    g = torch.Generator(device="cuda").manual_seed(3)
    sizes = SIZES + [(1, 1), (518, 924), (0, 0)]               # ... a one-pixel row, a large one, an H0 = 0 row
    n = len(sizes)
    x = torch.rand(n, *NET, device="cuda", generator=g) * 10
    offs = np.cumsum([0] + [h * w for h, w in sizes]).tolist()
    arena = torch.empty(offs[-1] + 4096, dtype=torch.float32, device="cuda")
    arena.view(torch.int32).fill_(-1)                          # poison: NaN bit patterns
    poison = arena.clone()
    _, od = group_descriptors(n, [(1, 3 * max(w, 1), h, w) for h, w in sizes],
                              [arena.data_ptr() + 4 * o for o in offs[:-1]])
    od[-1]["dst"] = arena.data_ptr() + 4 * offs[-1]            # the H0 = 0 row points at poisoned bytes
    od[-1]["H0"], od[-1]["W0"] = 0, 77
    ops.bilinear_f32_ragged(x, _dev_bytes(od))
    for i, (h, w) in enumerate(sizes[:-1]):
        got = arena[offs[i]:offs[i + 1]].view(h, w)
        assert torch.equal(got, ops.bilinear_f32(x[i:i + 1].contiguous(), h, w)[0]), (h, w)
        if (h, w) == NET:
            assert torch.equal(got, x[i])
    assert torch.equal(arena[offs[-1]:].view(torch.int32), poison[offs[-1]:].view(torch.int32)), "H0 = 0 wrote bytes"


# ---------------------------------------------------------------------------------------------- end to end
OPENS = [0, 0, 3, 7]


@pytest.fixture(scope="module")
def mixed_case():
    _, sd = build_model("vits", 0, torch.bfloat16)
    schedule = _schedule(44, OPENS, seed=12)
    counts = [sum(i in s for s in schedule) for i in range(4)]
    assert max(counts) > 32                                    # one stream's context slides
    videos = [np.random.default_rng(60 + i).integers(0, 256, (c, h, w, 3), dtype=np.uint8)
              for i, (c, (h, w)) in enumerate(zip(counts, SIZES))]
    return sd, schedule, videos


def _run(group, videos, schedule, frame=lambda i, t, f: f, to_host=True):
    handles, t, outs = {}, [0] * len(videos), [[] for _ in videos]
    for p, names in enumerate(schedule):
        for i, o in enumerate(OPENS):
            if o == p:
                handles[i] = group.open()
        got = group.push({handles[i]: frame(i, t[i], videos[i][t[i]]) for i in names}, to_host=to_host)
        for i in names:
            d = got[handles[i]]
            if not to_host:
                assert d.is_cuda and d.dtype == torch.float32 and d.shape == videos[i].shape[1:3]
                d = d.cpu().numpy()
            outs[i].append(d)
            t[i] += 1
    return [torch.from_numpy(np.stack(o)) for o in outs]


@pytest.mark.parametrize("mode", ["fp16", "bf16", "fp32"])
def test_mixed_sizes_vs_oracle(mixed_case, mode):
    sd, schedule, videos = mixed_case
    m, _ = build_model("vits", 0, torch.float16 if mode == "fp16" else torch.bfloat16)
    outs = _run(m.stream_group(4, 56, fp32=mode == "fp32"), videos, schedule)
    tol = TOL_VALIDATION if mode == "fp32" else TOL
    for i, got in enumerate(outs):
        ref = _oracle(sd, videos[i], "vits", 56)
        errs = [O.rel_err(got[t], ref[t])[0] for t in range(len(ref))]
        print(f"mixed-size group {mode} stream {i} {SIZES[i]}: {len(ref)} frames, worst frame rel err {max(errs):.3e}")
        assert max(errs) <= tol, (i, errs)
        assert (got >= 0).all()


def test_mixed_sizes_fp32_bit_identical_to_lone_streams(mixed_case):
    _, schedule, videos = mixed_case
    m, _ = build_model("vits", 0, torch.bfloat16)
    outs = _run(m.stream_group(4, 56, fp32=True), videos, schedule)
    for i, got in enumerate(outs):
        lone = m.stream(input_size=56, fp32=True)
        assert torch.equal(got, torch.from_numpy(np.stack([lone.push(f) for f in videos[i]]))), i


def test_device_frames_and_depths_match_host_path(mixed_case):
    _, schedule, videos = mixed_case
    m, _ = build_model("vits", 0, torch.bfloat16)
    ref = _run(m.stream_group(4, 56), videos, schedule)

    def mixed(i, t, f):                  # streams 0 and 2: CUDA frames (stream 2 from a pitched view); 1 and 3 alternate
        if i == 2:
            h, w = f.shape[:2]
            pad = torch.zeros(h + 3, w + 9, 3, dtype=torch.uint8, device="cuda")
            pad[2:2 + h, 5:5 + w] = torch.from_numpy(f).cuda()
            return pad[2:2 + h, 5:5 + w]
        if i == 0 or t % 2:
            return torch.from_numpy(f).cuda()
        return f
    for to_host in (True, False):
        got = _run(m.stream_group(4, 56), videos, schedule, mixed, to_host=to_host)
        for i in range(4):
            assert torch.equal(got[i], ref[i]), (to_host, i)
    one = m.stream(input_size=56)                             # DepthStream / infer_video_depth_one take them too
    f = videos[1][0]
    a = one.push(torch.from_numpy(f).cuda(), to_host=False)
    assert a.is_cuda and torch.equal(a.cpu(), torch.from_numpy(m.stream(input_size=56).push(f)))
    b = m.infer_video_depth_one(torch.from_numpy(f).cuda(), input_size=56, to_host=False)
    assert b.is_cuda and torch.equal(b.cpu(), a.cpu())


# ---------------------------------------------------------------------------------------------- bounded cost
def test_mixed_cost_is_bounded():
    m, _ = build_model("vits", 0, torch.bfloat16)
    frames = {s: [_frame(*s, 100 + j) for j in range(3)] for s in SIZES}
    dev = {s: [torch.from_numpy(f).cuda() for f in fs] for s, fs in frames.items()}
    g = m.stream_group(8, 56)
    hs = [g.open() for _ in range(8)]
    g.push({h: frames[(100, 140)][0] for h in hs})            # the largest push: 8 host frames of the largest size
    for h in hs[1:]:                                          # start 7 streams over, at every size
        g.close_stream(h)
    hs[1:] = [g.open() for _ in hs[1:]]
    size = {h: SIZES[i % 4] for i, h in enumerate(hs)}
    size[hs[0]] = (100, 140)
    rng = np.random.default_rng(5)
    for k in (1, 2, 4):                                       # first use of every other bucket
        g.push({h: frames[size[h]][0] for h in hs[:k]})
    assert sorted(g.graphs) == [1, 2, 4, 8]
    graphs = {k: v[0] for k, v in g.graphs.items()}
    gc.collect()
    mem0 = torch.cuda.memory_allocated()
    per_push = {}                                             # bucket -> launches per push
    for p in range(200):
        if p % 10 == 5:                                        # reopen a stream at another size now and then
            i = int(rng.integers(1, 8))
            g.close_stream(hs[i])
            del size[hs[i]]
            hs[i] = g.open()
            size[hs[i]] = SIZES[int(rng.integers(4))]
        k = int(rng.integers(1, 9))
        sub = [hs[j] for j in rng.permutation(8)[:k]]
        push = {h: (dev if rng.random() < 0.5 else frames)[size[h]][p % 3] for h in sub}
        n0 = ops.LAUNCHES
        to_host = bool(rng.random() < 0.5)
        out = g.push(push, to_host=to_host)
        per_push.setdefault(g.plan.bucket(k), set()).add(ops.LAUNCHES - n0)
        del out                                                # CUDA depths dropped
    assert {k: v[0] for k, v in g.graphs.items()} == graphs, "no capture after a bucket's first use"
    assert all(len(v) == 1 for v in per_push.values()), per_push   # the launch count does not depend on the mix
    gc.collect()
    assert torch.cuda.memory_allocated() == mem0


# ---------------------------------------------------------------------------------------------- errors
def test_size_and_device_errors():
    m, _ = build_model("vits", 0, torch.bfloat16)
    g = m.stream_group(4, 56)
    a, b = g.open(), g.open()
    with pytest.raises(ValueError, match=r"\(56, 84\).*\(56, 98\)|\(56, 98\).*\(56, 84\)"):
        g.push({a: _frame(50, 70, 0), b: _frame(40, 70, 1)})      # network sizes differ within one push
    g.push({a: _frame(50, 70, 0), b: _frame(100, 140, 1)})       # two sizes, one network size
    with pytest.raises(ValueError, match="differs from its first"):
        g.push({a: _frame(25, 35, 2)})                           # another size of stream a
    with pytest.raises(ValueError, match=r"\(56, 98\).*\(56, 84\)"):
        g.push({g.open(): _frame(40, 70, 3)})                    # another network size than the group's
    c = g.open()
    with pytest.raises(ValueError):
        g.push({c: torch.from_numpy(_frame(50, 70, 4))})         # a CPU tensor
    with pytest.raises(ValueError):
        g.push({c: torch.zeros(50, 70, 3, dtype=torch.float32, device="cuda")})
    with pytest.raises(ValueError):
        g.push({c: torch.zeros(50, 140, 3, dtype=torch.uint8, device="cuda")[:, ::2]})   # pixels not contiguous
    with pytest.raises(ValueError):
        g.push({c: torch.zeros(50, 70, 4, dtype=torch.uint8, device="cuda")[..., :3]})   # pixel stride 4
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            g.push({c: torch.zeros(50, 70, 3, dtype=torch.uint8, device="cuda:1")})
    g.push({c: torch.from_numpy(_frame(25, 35, 5)).cuda()})     # the rejected pushes left c at t = 0, free to size
    assert g.plan.t[c] == 1 and g.plan.size[c] == (25, 35)
