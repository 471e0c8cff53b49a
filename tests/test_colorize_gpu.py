"""GPU: colour-mapped depth frames, bit-exact against colorize_oracle.  The kernels (every format x table x range mode,
ragged batches with pad rows and guard bytes, pitched and encoder-style surfaces, level boundaries), colorize() on
device and host depths, stream groups against the oracle applied to a "depth" group fed the same pushes (ViT-S bf16,
ViT-L, stacks, reopen, to_host both ways, RGB and NV12 input, graph replay and launch counts), CStreamGroup, and a
compiled C host writing NVENC-style NV12 surfaces."""
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import colorize_oracle as O  # noqa: E402
import yuv_oracle as Y  # noqa: E402
from e2e_checks import build_model  # noqa: E402
from video_depth_anything_b200 import MODEL_CONFIGS, colorize, display, ops  # noqa: E402
from video_depth_anything_b200.cmodel import CModel, CStreamGroup  # noqa: E402
from video_depth_anything_b200.windows import INFERNO, OUT_DESC, color_descriptors  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
FMTS = {"rgb": 0, "nv12": 1, "i420": 2, "gray": 3}
RAND_TABLE = np.random.default_rng(7).integers(0, 256, (256, 3), dtype=np.uint8)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda()


def _boundary_depths(h, w, lo, hi, seed):
    """Random depths in [lo, hi] with a quarter of them on the level boundaries lo + j (hi - lo) / 255 +- 1 ulp."""
    rng = np.random.default_rng(seed)
    d = (lo + rng.random((h, w)) * (hi - lo)).astype(np.float32)
    j = rng.integers(0, 256, (h, w)).astype(np.float32)
    b = (np.float32(lo) + j * (np.float32(hi) - np.float32(lo)) / np.float32(255)).astype(np.float32)
    b = np.nextafter(b, np.where(rng.random((h, w)) < 0.5, np.float32(-np.inf), np.float32(np.inf)).astype(np.float32))
    pick = rng.random((h, w)) < 0.25
    d[pick] = b[pick]
    d.flat[0], d.flat[-1] = lo, hi
    return np.clip(d, lo, hi).astype(np.float32)


def _kernel_run(depths, fmt, table, mode, pitch_pad=0, pad_rows=0, enc_align=0):
    """Run vda_depth_range + vda_colorize_depth on a ragged batch (depth frames of their own sizes, each in its own
    allocation; every output plane in a guarded buffer with pitch = row + pitch_pad, an NVENC-style UV plane at
    Y + pitch * align(H, enc_align) when enc_align) -> (frames packed in OpenCV's layout, guards intact)."""
    code = FMTS[fmt]
    dd = [torch.from_numpy(d).cuda() for d in depths]
    n = len(depths) + pad_rows
    od = np.zeros(n, OUT_DESC)
    for i, t in enumerate(dd):
        od[i] = (t.data_ptr(), *t.shape)
    bufs, rows = [], []
    for d in depths:
        h, w = d.shape
        rb = 3 * w if code == 0 else w
        p = rb + pitch_pad
        if code in (1, 2):
            hy = -(-h // enc_align) * enc_align if enc_align else h
            cp = p if code == 1 else (w // 2 + pitch_pad)
            size = p * hy + (cp * (h // 2) * (1 if code == 1 else 2))
        else:
            size = p * h
        buf = torch.full((size + 64,), 0xA5, dtype=torch.uint8, device="cuda")
        bufs.append(buf)
        base = buf.data_ptr() + 32
        if code in (0, 3):
            rows.append(((base, 0, 0), (p, 0, 0)))
        elif code == 1:
            rows.append(((base, base + p * hy, 0), (p, p, 0)))
        else:
            u = base + p * hy
            rows.append(((base, u, u + cp * (h // 2)), (p, cp, cp)))
    cd = np.zeros(n, color_descriptors(1, [(0, 2, 2)], 3).dtype)
    for i, (d, (pl, pi)) in enumerate(zip(depths, rows)):
        cd[i] = (pl, pi, d.shape[0], d.shape[1], code, 0)
    od_d, cd_d = _dev(od), _dev(cd)
    if mode == "video":
        rng = ops.depth_range(od_d, True)
        per_row = False
    elif mode == "frame":
        rng = ops.depth_range(od_d, False)
        per_row = True
    else:
        rng = torch.tensor(mode, dtype=torch.float32, device="cuda")
        per_row = False
    ops.colorize_depth(od_d, cd_d, rng, per_row, None if table is None else torch.from_numpy(table.copy()).cuda())
    torch.cuda.synchronize()
    outs = []
    for d, buf, (pl, pi) in zip(depths, bufs, rows):
        h, w = d.shape
        b = buf.cpu().numpy()
        assert (b[:32] == 0xA5).all() and (b[-32:] == 0xA5).all()
        base = buf.data_ptr()
        view = lambda a, rows_, cols, pitch: b[a - base:a - base + pitch * rows_].reshape(rows_, pitch)[:, :cols]  # noqa: E731
        if code in (0, 3):
            f = view(pl[0], h, 3 * w if code == 0 else w, pi[0])
            outs.append(f.reshape(h, w, 3) if code == 0 else f.copy())
        elif code == 1:
            outs.append(np.concatenate([view(pl[0], h, w, pi[0]), view(pl[1], h // 2, w, pi[1])]))
        else:
            u, v = view(pl[1], h // 2, w // 2, pi[1]), view(pl[2], h // 2, w // 2, pi[2])
            outs.append(np.concatenate([view(pl[0], h, w, pi[0]).ravel(), u.ravel(), v.ravel()]).reshape(3 * h // 2, w))
    return outs


def _oracle(depths, table, fmt, mode):
    if mode == "video":
        lo = min(d.min() for d in depths)
        hi = max(d.max() for d in depths)
        rngs = [(lo, hi)] * len(depths)
    elif mode == "frame":
        rngs = [(d.min(), d.max()) for d in depths]
    else:
        rngs = [mode] * len(depths)
    return [O.frames_of(O.level(d, lo, hi)[None], table, fmt)[0] for d, (lo, hi) in zip(depths, rngs)]


@pytest.mark.parametrize("fmt", ["rgb", "gray", "nv12", "i420"])
@pytest.mark.parametrize("tab", ["inferno", "random"])
@pytest.mark.parametrize("mode", ["video", "frame", (0.5, 3.0)])
def test_kernels_bit_exact(fmt, tab, mode):
    table = None if fmt == "gray" else (INFERNO if tab == "inferno" else RAND_TABLE)
    sizes = [(1080, 1920), (720, 1280), (518, 924)] + ([(37, 51), (1, 1), (3, 8)] if fmt in ("rgb", "gray") else [(2, 2)])
    depths = []
    for i, (h, w) in enumerate(sizes):
        lo, hi = 0.3 + i, 2.7 + 3 * i
        depths.append(_boundary_depths(h, w, lo, hi, seed=i + 10 * len(fmt)))
    if not isinstance(mode, str):
        depths[0] = depths[0] * np.float32(2) - np.float32(1)            # values below and above the fixed range
    depths.append(np.full((4, 6), 1.25, np.float32))                     # a constant frame
    got = _kernel_run(depths, fmt, table, mode, pitch_pad=0, pad_rows=0)
    for g, r in zip(got, _oracle(depths, table, fmt, mode)):
        assert g.shape == r.shape and np.array_equal(g, r)


@pytest.mark.parametrize("fmt", ["rgb", "gray", "nv12", "i420"])
def test_kernels_pitched_ragged_with_pad_rows(fmt):
    table = None if fmt == "gray" else RAND_TABLE
    sizes = [(64, 96), (130, 18), (2, 4)] if fmt in ("nv12", "i420") else [(63, 97), (130, 17), (1, 3)]
    depths = [_boundary_depths(h, w, 1.0, 9.0, seed=h) for h, w in sizes]
    got = _kernel_run(depths, fmt, table, "frame", pitch_pad=45 if fmt != "i420" else 22, pad_rows=3)
    for g, r in zip(got, _oracle(depths, table, fmt, "frame")):
        assert np.array_equal(g, r)


def test_encoder_style_nv12_surface():
    depths = [_boundary_depths(h, w, 0.0, 5.0, seed=h) for h, w in [(1080, 1920), (720, 1280), (518, 924)]]
    pitch_pad = 256 - 1920 % 256
    got = _kernel_run(depths, "nv12", INFERNO, "video", pitch_pad=pitch_pad, enc_align=16)
    for g, r in zip(got, _oracle(depths, INFERNO, "nv12", "video")):
        assert np.array_equal(g, r)


def test_range_kernel_fold_and_empty_rows():
    rng = np.random.default_rng(3)
    depths = [rng.standard_normal((h, w)).astype(np.float32) for h, w in [(1, 1), (5, 7), (300, 301), (1080, 1920)]]
    dd = [torch.from_numpy(d).cuda() for d in depths]
    od = np.zeros(6, OUT_DESC)
    for i, t in enumerate(dd):
        od[i] = (t.data_ptr() + (4 if i == 3 else 0), t.shape[0], t.shape[1] - (1 if i == 3 else 0))   # misaligned row
    per = ops.depth_range(_dev(od), False).cpu().numpy()
    for i in range(3):
        assert tuple(per[i]) == (depths[i].min(), depths[i].max())
    sub = depths[3].ravel()[1:1 + 1080 * 1919]
    assert tuple(per[3]) == (sub.min(), sub.max())
    assert per[4][0] == np.inf and per[4][1] == -np.inf
    all_ = ops.depth_range(_dev(od), True).cpu().numpy()
    assert tuple(all_) == (min(per[:4, 0]), max(per[:4, 1]))
    assert tuple(display._fold(torch.from_numpy(per[:4].copy()).cuda()).cpu().numpy()) == tuple(all_)


@pytest.mark.parametrize("fmt", ["rgb", "gray", "nv12", "i420"])
def test_colorize_device_and_host(fmt, monkeypatch):
    d = np.stack([_boundary_depths(96, 130, 0.2, 4.0 + i, seed=i) for i in range(11)])
    table = None if fmt == "gray" else RAND_TABLE
    for value_range in ("video", "frame", (1.0, 3.0)):
        ref = O.colorize(d, table if table is not None else INFERNO, value_range, fmt)
        kw = dict(colormap="inferno" if table is None else table, value_range=value_range, pixel_format=fmt)
        dev = colorize(torch.from_numpy(d).cuda(), **kw)
        assert dev.is_cuda and dev.dtype == torch.uint8 and np.array_equal(dev.cpu().numpy(), ref)
        monkeypatch.setattr(display, "STAGE_BYTES", 3 * 4 * 96 * 130)          # 4 chunks of 3 frames
        host = colorize(d, **kw)
        assert isinstance(host, np.ndarray) and np.array_equal(host, ref)
        monkeypatch.undo()
    one = colorize(d[3], pixel_format=fmt, value_range="frame")
    assert np.array_equal(one, O.colorize(d[3:4], INFERNO, "frame", fmt)[0])


def test_colorize_is_the_reference_loop(monkeypatch):
    """colorize(depths, colormap=reference-style table) equals save_video's loop over more frames than one chunk."""
    rng = np.random.default_rng(5)
    d = (rng.random((40, 518, 518)) * 7.0 + 0.5).astype(np.float32)
    d[3] += np.float32(2.0)
    ref_table = (np.linspace(0, 1, 768).reshape(256, 3) * 255).astype(np.uint8)     # truncating, as the reference's
    monkeypatch.setattr(display, "STAGE_BYTES", 16 << 20)                           # 15 frames per chunk
    got = colorize(d, colormap=ref_table)
    assert np.array_equal(got, O.save_video_frames(d, ref_table))
    assert np.array_equal(colorize(d, pixel_format="gray"), O.save_video_frames(d, grayscale=True))


# ---------------------------------------------------------------------------------------------------- stream groups
def _pushes(videos, n_push, seed, stacks=True):
    rng = np.random.default_rng(seed)
    sched, t = [], [0] * len(videos)
    for _ in range(n_push):
        items = []
        for i in range(len(videos)):
            if rng.random() < 0.8 or not items and i == len(videos) - 1:
                k = int(rng.integers(2, 4)) if stacks and rng.random() < 0.25 else 1
                if t[i] + k <= len(videos[i]):
                    items.append((i, k))
                    t[i] += k
        if items:
            sched.append(items)
    return sched


def _run_group(g, videos, sched, to_host=True, cuda_frames=False, close_at=None):
    hs = [g.open() for _ in videos]
    t = [0] * len(videos)
    outs = []
    for p, items in enumerate(sched):
        if close_at is not None and p == close_at:
            g.close_stream(hs[0])
            hs[0] = g.open()
        push = {}
        for i, k in items:
            f = videos[i][t[i]:t[i] + k] if k > 1 else videos[i][t[i]]
            push[hs[i]] = torch.from_numpy(np.ascontiguousarray(f)).cuda() if cuda_frames else f
            t[i] += k
        r = g.push(push, to_host=to_host)
        outs.append([r[hs[i]] if to_host else r[hs[i]].cpu().numpy() for i, _ in items])
    return outs


def _check_against_depth(depth_outs, color_outs, fmt, table, value_range):
    for dp, cp in zip(depth_outs, color_outs):
        for d, c in zip(dp, cp):
            d = d.reshape((-1,) + d.shape[-2:])
            ref = O.colorize(d, table, value_range, fmt)
            assert c.shape == (ref.shape if c.ndim == ref.ndim else ref.shape[1:])
            assert np.array_equal(c.reshape(ref.shape), ref)


@pytest.mark.parametrize("in_fmt", ["rgb", "nv12"])
def test_group_vits_720p_1080p(in_fmt):
    m, _ = build_model("vits", 0, torch.bfloat16)
    sizes = [(720, 1280), (1080, 1920), (720, 1280)]
    if in_fmt == "rgb":
        videos = [np.random.default_rng(i).integers(0, 256, (8, h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(sizes)]
    else:
        videos = [Y.random_video(8, h, w, "nv12", seed=i) for i, (h, w) in enumerate(sizes)]
    sched = _pushes(videos, 5, seed=1)
    dg = m.stream_group(3, pixel_format=in_fmt)
    depth = _run_group(dg, videos, sched, close_at=3)
    # the launch counts of a second depth group: the first capture at a network size also counts the one-off resampling
    # of the position embedding in its warm-up
    dg = m.stream_group(3, pixel_format=in_fmt)
    again = _run_group(dg, videos, sched, close_at=3)
    assert all(np.array_equal(x, y) for p, q in zip(depth, again) for x, y in zip(p, q))
    for fmt, table, vr, to_host in [("nv12", INFERNO, "frame", True), ("rgb", RAND_TABLE, (0.0, 0.6), False),
                                    ("gray", None, "frame", False), ("i420", INFERNO, "frame", True)]:
        cg = m.stream_group(3, pixel_format=in_fmt, output_format=fmt, colormap="inferno" if table is None else table,
                            value_range=vr)
        out = _run_group(cg, videos, sched, to_host=to_host, cuda_frames=not to_host, close_at=3)
        _check_against_depth(depth, out, fmt, INFERNO if table is None else table, vr)
        extra = 3 if vr == "frame" else 1
        for bk, entry in cg.graphs.items():
            assert entry[3] == dg.graphs[bk][3] + extra
        for bk, entry in cg.causal_graphs.items():
            assert entry[3] == dg.causal_graphs[bk][3] + extra
        cg.close()


def test_group_vitl_518():
    m, _ = build_model("vitl", 0, torch.bfloat16)
    videos = [np.random.default_rng(i).integers(0, 256, (3, 518, 518, 3), dtype=np.uint8) for i in range(2)]
    sched = [[(0, 1), (1, 1)], [(0, 2)], [(1, 1)]]
    depth = _run_group(m.stream_group(2), videos, sched)
    out = _run_group(m.stream_group(2, output_format="nv12"), videos, sched)
    _check_against_depth(depth, out, "nv12", INFERNO, "frame")


def test_group_replay_captures_nothing_new_and_grows_nothing():
    m, _ = build_model("vits", 0, torch.bfloat16)
    sizes = [(50, 70), (100, 140), (50, 70)]
    videos = [np.random.default_rng(i).integers(0, 256, (400, h, w, 3), dtype=np.uint8) for i, (h, w) in enumerate(sizes)]
    pattern = _pushes([v[:130] for v in videos], 25, seed=4)
    sched = pattern * 3                                  # the warm-up meets every (bucket, causal) the 50 later pushes do
    warm, rest = sched[:25], sched[25:]
    dg = m.stream_group(3, 56)
    cg = m.stream_group(3, 56, output_format="rgb")
    depth = _run_group(dg, videos, sched)
    hs = [cg.open() for _ in videos]
    t = [0] * len(videos)

    def run(part):
        outs = []
        for items in part:
            push = {}
            for i, k in items:
                push[hs[i]] = videos[i][t[i]:t[i] + k] if k > 1 else videos[i][t[i]]
                t[i] += k
            r = cg.push(push)
            outs.append([r[hs[i]] for i, _ in items])
        return outs
    out = run(warm)
    torch.cuda.synchronize()
    n_graphs = (len(cg.graphs), len(cg.causal_graphs))
    mem = torch.cuda.memory_allocated()
    arenas = {k: v.data_ptr() for k, v in cg.arenas.items()}
    out += run(rest)
    torch.cuda.synchronize()
    assert (len(cg.graphs), len(cg.causal_graphs)) == n_graphs
    assert torch.cuda.memory_allocated() == mem
    assert {k: v.data_ptr() for k, v in cg.arenas.items()} == arenas
    _check_against_depth(depth, out, "rgb", INFERNO, "frame")


def test_cstreamgroup_bit_identical_to_python():
    m, sd = build_model("vits", 0, torch.bfloat16)
    cm = CModel(**MODEL_CONFIGS["vits"], dtype=torch.bfloat16)
    cm.load_state_dict(sd)
    sizes = [(50, 70), (100, 140)]
    videos = [Y.random_video(20, h, w, "nv12", seed=30 + i) for i, (h, w) in enumerate(sizes)]
    sched = _pushes(videos, 10, seed=8)
    vids_cuda = [torch.from_numpy(v).cuda() for v in videos]
    for fmt, vr in [("nv12", "frame"), ("rgb", (0.0, 0.5)), ("gray", "frame")]:
        py = m.stream_group(2, 56, pixel_format="nv12", output_format=fmt, value_range=vr)
        cg = CStreamGroup(cm, 2, 56, pixel_format="nv12", output_format=fmt, value_range=vr)
        a = _run_group(py, videos, sched, to_host=False, cuda_frames=True)
        hs = [cg.open() for _ in videos]
        t = [0, 0]
        for p, items in enumerate(sched):
            push = {}
            for i, k in items:
                push[hs[i]] = vids_cuda[i][t[i]:t[i] + k] if k > 1 else vids_cuda[i][t[i]]
                t[i] += k
            r = cg.push(push)
            for (i, _), x in zip(items, a[p]):
                assert r[hs[i]].dtype == torch.uint8 and np.array_equal(r[hs[i]].cpu().numpy(), x), (fmt, p, i)
        cg.close()


def test_c_host_program_colorize_bit_identical_to_python(tmp_path):
    exe = str(tmp_path / "host_stream_colorize")
    from video_depth_anything_b200 import build
    libdir = os.path.dirname(build.build())
    subprocess.check_call(["gcc", "-O1", "-std=c99", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(CUDA, "include"),
                           os.path.join(ROOT, "tests", "c_host", "host_stream_colorize.c"), "-o", exe, "-L", libdir,
                           "-l:libvda.so", "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir,
                           "-Wl,-rpath," + os.path.join(CUDA, "lib64")])
    m, sd = build_model("vits", 0, torch.bfloat16)
    sizes = [(50, 70), (100, 140)]
    videos = [Y.random_video(60, h, w, "nv12", seed=22 + i) for i, (h, w) in enumerate(sizes)]
    sched = [[(i, k) for i, k in items] for items in _pushes(videos, 18, seed=23)]
    py = m.stream_group(2, 56, pixel_format="nv12", output_format="nv12")
    ref = [x.ravel() for p in _run_group(py, videos, sched) for x in p]
    wpath, ipath, opath, tpath = (str(tmp_path / n) for n in ("weights.bin", "input.bin", "output.bin", "table.bin"))
    with open(wpath, "wb") as f:
        f.write(struct.pack("<i", len(sd)))
        for k, v in sd.items():
            a = v.detach().to("cpu", torch.float32).contiguous().numpy()
            name = k.encode()
            f.write(struct.pack("<i", len(name)) + name + struct.pack("<i", a.ndim) + struct.pack(f"<{a.ndim}q", *a.shape))
            f.write(a.tobytes())
    with open(ipath, "wb") as f:
        f.write(struct.pack("<3i", 2, 56, len(sched)))
        for v, (h, w) in zip(videos, sizes):
            f.write(struct.pack("<3i", v.shape[0], h, w) + v.tobytes())
        for items in sched:
            f.write(struct.pack("<i", len(items)) + b"".join(struct.pack("<2i", i, k) for i, k in items))
    INFERNO.tofile(tpath)
    cfg = MODEL_CONFIGS["vits"]
    r = subprocess.run([exe, "vits", str(cfg["features"]), *map(str, cfg["out_channels"]), "0", wpath, ipath, opath, tpath],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    print(r.stdout.strip())
    out = np.fromfile(opath, dtype=np.uint8)
    flat = np.concatenate(ref)
    assert out.shape == flat.shape and np.array_equal(out, flat)
