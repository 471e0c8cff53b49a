"""GPU: YUV 4:2:0 input (NV12 / I420) through every ingest path.  The contract: for any NV12 or I420 frame F, each entry
point gives results bit-identical to the same entry point fed cv2.cvtColor(F, COLOR_YUV2RGB_*) as RGB -- the kernels
(all (Y, U, V) triples, resized, pitched, separate allocations, mixed sizes, pad rows), stream groups (host, CUDA and
plane-tuple frames, stacks, reopen, to_host=False, ViT-S bf16 / fp16, ViT-L, fp32=True), the long-video driver (upload
ring, feature reuse), the C stream step (ctypes and a compiled C host), graph replay and launch counts, and the sharded
driver on two or more GPUs."""
import gc
import os
import socket
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import yuv_oracle as Y  # noqa: E402
from e2e_checks import build_model  # noqa: E402
from video_depth_anything_b200 import MODEL_CONFIGS, ops  # noqa: E402
from video_depth_anything_b200.cmodel import CModel, CStreamGroup  # noqa: E402
from video_depth_anything_b200.windows import group_descriptors, yuv_planes  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
FMT_CODE = {"nv12": 1, "i420": 2}
NET = (56, 84)
SIZES = [(50, 70), (100, 140), (56, 84), (28, 42)]       # upscaled, downscaled, identity, upscaled: all at (56, 84)


def _dev_bytes(arr):
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8)).cuda()


def _rgb_ref(rgb_frames, nh, nw):
    """vda_preprocess_frames of uint8 RGB frames [n,H0,W0,3] (numpy): the RGB path every YUV result must equal."""
    t = torch.from_numpy(np.ascontiguousarray(rgb_frames)).cuda()
    return ops.preprocess_frames(t, torch.arange(len(rgb_frames), dtype=torch.int32, device="cuda"), nh, nw)


def _planes_of(packed, fmt, pitch_pad=0):
    """CUDA plane tensors of one packed frame: each plane in its own allocation with `pitch_pad` bytes of row padding."""
    y, u, v = Y.split_planes(packed, fmt)
    if fmt == "nv12":
        planes = [y, np.stack([u, v], -1).reshape(u.shape[0], -1)]
    else:
        planes = [y, u, v]
    out = []
    for p in planes:
        buf = torch.full((p.shape[0], p.shape[1] + pitch_pad), 77, dtype=torch.uint8, device="cuda")
        buf[:, :p.shape[1]] = torch.from_numpy(np.ascontiguousarray(p)).cuda()
        out.append(buf[:, :p.shape[1]])
    return tuple(out)


def _plane_src(planes):
    ptr = [t.data_ptr() for t in planes] + [0] * (3 - len(planes))
    pitch = [t.stride(0) for t in planes] + [0] * (3 - len(planes))
    return tuple(ptr), tuple(pitch)


# ---------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_all_triples_identity_size(fmt):
    """Every (Y, U, V) triple in one 4096 x 4096 frame, at identity size (no resize: each output is one converted pixel)."""
    frame = Y.all_triples(fmt)
    rgb = Y.to_rgb(frame, fmt)
    expect = _rgb_ref(rgb[None], 4096, 4096)
    dev = torch.from_numpy(frame).cuda()
    idx = torch.zeros(1, dtype=torch.int32, device="cuda")
    got = ops.preprocess_frames_yuv(dev[None], idx, FMT_CODE[fmt], 4096, 4096)
    assert torch.equal(got, expect)
    del got
    fd, _ = group_descriptors(1, [yuv_planes(dev.data_ptr(), 4096, 4096, 4096, fmt) + (4096, 4096)], [0], fmt)
    got = ops.preprocess_frames_planes(_dev_bytes(fd), 4096, 4096)
    assert torch.equal(got, expect)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_uniform_kernel_resized_frames(fmt):
    """The long-video form: a packed video, an index list with repeats and reordering, up- and downscaled."""
    for (h0, w0), (nh, nw) in [((50, 70), NET), ((100, 140), NET), ((56, 84), NET), ((720, 1280), (518, 924))]:
        video = Y.random_video(5, h0, w0, fmt, seed=h0)
        rgb = Y.video_to_rgb(video, fmt)
        order = [3, 0, 4, 4, 1]
        expect = _rgb_ref(rgb[order], nh, nw)
        idx = torch.tensor(order, dtype=torch.int32, device="cuda")
        got = ops.preprocess_frames_yuv(torch.from_numpy(video).cuda(), idx, FMT_CODE[fmt], nh, nw)
        assert torch.equal(got, expect), (h0, w0)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_ragged_kernel_pitched_separate_mixed_and_pad_rows(fmt):
    frames = [Y.random_video(1, h, w, fmt, seed=30 + i)[0] for i, (h, w) in enumerate(SIZES)]
    expect = [_rgb_ref(Y.to_rgb(f, fmt)[None], *NET)[0] for f in frames]
    keep = []
    srcs = []
    for i, f in enumerate(frames):
        h0, w0 = f.shape[0] * 2 // 3, f.shape[1]
        if i % 2:                                          # planes in separate allocations, pitched rows
            planes = _planes_of(f, fmt, pitch_pad=64 + 16 * i)
            keep.append(planes)
            src = _plane_src(planes)
        elif fmt == "nv12":                                # an NVDEC-like surface: UV at Y + pitch * aligned height
            pitch, rows = 256 * (-(-w0 // 256)), 32 * (-(-h0 // 32))
            surf = torch.zeros(pitch * (rows + h0 // 2), dtype=torch.uint8, device="cuda")
            surf[:h0 * pitch].view(h0, pitch)[:, :w0] = torch.from_numpy(f[:h0]).cuda()
            surf[rows * pitch:(rows + h0 // 2) * pitch].view(h0 // 2, pitch)[:, :w0] = torch.from_numpy(f[h0:]).cuda()
            keep.append(surf)
            src = ((surf.data_ptr(), surf.data_ptr() + rows * pitch, 0), (pitch, pitch, 0))
        else:                                              # a packed I420 frame
            t = torch.from_numpy(f).cuda()
            keep.append(t)
            src = yuv_planes(t.data_ptr(), w0, h0, w0, fmt)
        srcs.append(src + (h0, w0))
    for rows in ([0], [1], [2], [3], [3, 1, 0, 2, 1]):
        fd, _ = group_descriptors(len(rows), [srcs[r] for r in rows], [0] * len(rows), fmt)
        got = ops.preprocess_frames_planes(_dev_bytes(fd), *NET)
        for b, r in enumerate(rows):
            assert torch.equal(got[b], expect[r]), (rows, b)
    fd, _ = group_descriptors(4, [srcs[1], srcs[3]], [0, 0], fmt)       # pad rows read row 0's frame
    got = ops.preprocess_frames_planes(_dev_bytes(fd), *NET)
    assert torch.equal(got[2], expect[1]) and torch.equal(got[3], expect[1])


def test_launcher_rejects_bad_arguments():
    lib = ops._lib.load()
    buf = torch.zeros(3 * 50 * 70, dtype=torch.uint8, device="cuda")
    idx = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = torch.full((1, 3, 56, 84), -7.0, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for fmt, h0, w0, msg in [(1, 51, 70, "even size"), (2, 50, 71, "even size"), (0, 50, 70, "unknown pixel format"),
                             (3, 50, 70, "unknown pixel format")]:
        assert lib.vda_preprocess_frames_yuv(buf.data_ptr(), idx.data_ptr(), fmt, out.data_ptr(), 1, h0, w0, 56, 84, st) != 0
        assert msg in lib.vda_last_error().decode()
    torch.cuda.synchronize()
    assert (out == -7).all()


# ---------------------------------------------------------------------------------------------- streams
def _frame_forms(packed, fmt, form):
    """One packed frame (or stack) as `form`: "host" (numpy), "cuda" (packed CUDA tensor, NV12 rows pitched), "planes"."""
    if form == "host":
        return packed
    if form == "cuda":
        t = torch.from_numpy(np.ascontiguousarray(packed)).cuda()
        if fmt == "nv12":                                  # pitched rows
            pad = torch.zeros(*t.shape[:-1], t.shape[-1] + 32, dtype=torch.uint8, device="cuda")
            pad[..., :t.shape[-1]] = t
            t = pad[..., :t.shape[-1]]
        return t
    if packed.ndim == 2:
        return _planes_of(packed, fmt, pitch_pad=48)
    ps = [_planes_of(f, fmt, pitch_pad=48) for f in packed]
    return tuple(torch.stack([p[i] for p in ps]) for i in range(len(ps[0])))


def _run_pair(m, fmt, sizes, n_pushes, seed, fp32=False, input_size=56, reopen_at=7, max_k=4):
    """The same random push schedule through a YUV group and an RGB group fed cv2's RGB of the same frames; returns the
    two lists of depths."""
    rng = np.random.default_rng(seed)
    videos = [Y.random_video(n_pushes * max_k + 4, h, w, fmt, seed=seed + i) for i, (h, w) in enumerate(sizes)]
    rgbs = [Y.video_to_rgb(v, fmt) for v in videos]
    gy = m.stream_group(len(sizes), input_size, fp32=fp32, pixel_format=fmt)
    gr = m.stream_group(len(sizes), input_size, fp32=fp32)
    hy, hr = [gy.open() for _ in sizes], [gr.open() for _ in sizes]
    t = [0] * len(sizes)
    outs_y, outs_r = [], []
    forms = ("host", "cuda", "planes")
    for p in range(n_pushes):
        if p == reopen_at:
            gy.close_stream(hy[0]); gr.close_stream(hr[0])
            hy[0], hr[0] = gy.open(), gr.open()
        sub = [i for i in range(len(sizes)) if rng.random() < 0.8] or [0]
        py, pr = {}, {}
        for i in sub:
            k = int(rng.integers(2, max_k + 1)) if rng.random() < 0.3 else None
            sl = slice(t[i], t[i] + k) if k else t[i]
            form = forms[int(rng.integers(3))]
            py[hy[i]] = _frame_forms(videos[i][sl], fmt, form)
            rgb = rgbs[i][sl]
            pr[hr[i]] = rgb if form == "host" else torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
            t[i] += k or 1
        to_host = bool(rng.random() < 0.5)
        a, b = gy.push(py, to_host=to_host), gr.push(pr, to_host=to_host)
        for i in sub:
            x, y = a[hy[i]], b[hr[i]]
            outs_y.append(x.cpu() if isinstance(x, torch.Tensor) else torch.from_numpy(x))
            outs_r.append(y.cpu() if isinstance(y, torch.Tensor) else torch.from_numpy(y))
    gy.close(); gr.close()
    return outs_y, outs_r


def _assert_same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and torch.equal(x, y), f"output {i}: max abs diff {(x - y).abs().max().item():.3e}"


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_vits_groups_bit_identical_to_rgb(fmt, dtype):
    """Two frame sizes of one network size, stacks (causal steps), a close and reopen, host / CUDA / plane-tuple frames,
    to_host both ways."""
    m, _ = build_model("vits", 0, dtype)
    a, b = _run_pair(m, fmt, [(50, 70), (100, 140)], 16, seed=11)
    _assert_same(a, b)


def test_vits_fp32_and_vitl_518():
    m, _ = build_model("vits", 0, torch.bfloat16)
    a, b = _run_pair(m, "nv12", [(50, 70), (28, 42)], 6, seed=12, fp32=True, reopen_at=3)
    _assert_same(a, b)
    del m
    gc.collect()
    m, _ = build_model("vitl", 0, torch.bfloat16)
    a, b = _run_pair(m, "i420", [(518, 518)], 5, seed=13, input_size=518, reopen_at=-1, max_k=3)
    _assert_same(a, b)


def test_stream_and_infer_video_depth_one():
    m, _ = build_model("vits", 0, torch.bfloat16)
    video = Y.random_video(6, 50, 70, "nv12", seed=14)
    rgb = Y.video_to_rgb(video, "nv12")
    st_y, st_r = m.stream(56, pixel_format="nv12"), m.stream(56)
    for j in range(3):
        assert np.array_equal(st_y.push(video[j]), st_r.push(rgb[j]))
    assert np.array_equal(st_y.push(video[3:6]), st_r.push(rgb[3:6]))
    st_y.close(); st_r.close()
    ref = [m.infer_video_depth_one(rgb[j], 56) for j in range(3)]
    got = [m.infer_video_depth_one(video[j], 56, pixel_format="nv12") for j in range(3)]   # reopens: its own stream
    assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    with pytest.raises(ValueError):
        m.infer_video_depth_one(video[:2], 56, pixel_format="nv12")


# ---------------------------------------------------------------------------------------------- long video
@pytest.mark.parametrize("reuse", [True, False], ids=["feature-reuse", "per-window"])
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_infer_video_depth_bit_identical_to_rgb(fmt, reuse):
    """330 frames: the upload ring (4 x 64 frames + frame 0) wraps several times, at a resized size."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    video = Y.random_video(330, 46, 64, fmt, seed=15)
    a, _ = m.infer_video_depth(video, 24, input_size=56, device="cuda", reuse_features=reuse, pixel_format=fmt)
    b, _ = m.infer_video_depth(Y.video_to_rgb(video, fmt), 24, input_size=56, device="cuda", reuse_features=reuse)
    assert a.shape == (330, 46, 64) and np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------- C library
def _c_pair(enc="vits", dtype=torch.bfloat16):
    m, sd = build_model(enc, 0, dtype)
    cm = CModel(**MODEL_CONFIGS[enc], dtype=dtype)
    cm.load_state_dict(sd)
    return m, cm, sd


def test_cstreamgroup_nv12_bit_identical_to_python():
    m, cm, _ = _c_pair()
    fmt = "nv12"
    sizes = [(50, 70), (100, 140)]
    videos = [Y.random_video(60, h, w, fmt, seed=20 + i) for i, (h, w) in enumerate(sizes)]
    py = m.stream_group(2, 56, pixel_format=fmt)
    cg = CStreamGroup(cm, 2, 56, pixel_format=fmt)
    hp, hc = [py.open(), py.open()], [cg.open(), cg.open()]
    rng = np.random.default_rng(21)
    t = [0, 0]
    for p in range(24):
        if p == 9:
            py.close_stream(hp[1]); cg.close_stream(hc[1])
            hp[1], hc[1] = py.open(), cg.open()
        sub = [i for i in range(2) if rng.random() < 0.8] or [1]
        a, b = {}, {}
        for i in sub:
            k = int(rng.integers(2, 5)) if rng.random() < 0.3 else None
            sl = slice(t[i], t[i] + k) if k else t[i]
            f = _frame_forms(videos[i][sl], fmt, "planes" if rng.random() < 0.5 else "cuda")
            a[hp[i]], b[hc[i]] = f, f
            t[i] += k or 1
        x, y = py.push(a, to_host=False), cg.push(b)
        for i in sub:
            assert torch.equal(x[hp[i]], y[hc[i]]), (p, i)
    assert sorted(cg.graphs) == sorted([(k, False) for k in py.graphs] + [(k, True) for k in py.causal_graphs])


def test_c_host_program_nv12_bit_identical_to_python(tmp_path):
    exe = str(tmp_path / "host_stream_nv12")
    from video_depth_anything_b200 import build
    libdir = os.path.dirname(build.build())
    subprocess.check_call(["gcc", "-O1", "-std=c99", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(CUDA, "include"),
                           os.path.join(ROOT, "tests", "c_host", "host_stream_nv12.c"), "-o", exe, "-L", libdir,
                           "-l:libvda.so", "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir,
                           "-Wl,-rpath," + os.path.join(CUDA, "lib64")])
    m, sd = build_model("vits", 0, torch.bfloat16)
    sizes = [(50, 70), (100, 140)]                            # one network size, 56 x 84; surfaces of two sizes
    videos = [Y.random_video(80, h, w, "nv12", seed=22 + i) for i, (h, w) in enumerate(sizes)]
    rng = np.random.default_rng(23)
    sched = []
    t = [0, 0]
    for p in range(24):
        items = []
        for i in range(2):
            if rng.random() < 0.8 or i == 1 and not items:
                k = int(rng.integers(2, 5)) if rng.random() < 0.3 else 1
                items.append((i, k))
                t[i] += k
        sched.append(items)
    py = m.stream_group(2, 56, pixel_format="nv12")
    hs = [py.open(), py.open()]
    t = [0, 0]
    ref = []
    for items in sched:
        push = {}
        for i, k in items:
            push[hs[i]] = videos[i][t[i]:t[i] + k] if k > 1 else videos[i][t[i]]
            t[i] += k
        out = py.push(push, to_host=False)
        ref += [out[hs[i]].flatten().cpu() for i, _ in items]
    wpath, ipath, opath = (str(tmp_path / n) for n in ("weights.bin", "input.bin", "output.bin"))
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
    cfg = MODEL_CONFIGS["vits"]
    r = subprocess.run([exe, "vits", str(cfg["features"]), *map(str, cfg["out_channels"]), "0", wpath, ipath, opath],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    print(r.stdout.strip())
    out = torch.from_numpy(np.fromfile(opath, dtype=np.float32))
    flat = torch.cat(ref)
    assert out.shape == flat.shape and torch.equal(out, flat), f"max abs diff {(out - flat).abs().max().item():.3e}"


def test_rejected_planes_steps_launch_nothing():
    _, cm, _ = _c_pair()
    lib = cm.lib
    B, S, nh, nw = 2, 2, 56, 84
    frame = torch.randint(0, 256, (75, 70), dtype=torch.uint8, device="cuda")
    out = torch.full((B, 50, 70), -7.0, device="cuda")
    fd, od = group_descriptors(B, [yuv_planes(frame.data_ptr(), 70, 50, 70, "nv12") + (50, 70)] * B,
                               [out[b].data_ptr() for b in range(B)], "nv12")
    fd_d, od_d = _dev_bytes(fd), _dev_bytes(od)
    table = torch.from_numpy(np.concatenate([np.zeros(B, np.int32), np.zeros(B * 33, np.int32),
                                             np.arange(B, dtype=np.int32)])).cuda()
    pool = torch.full((lib.vda_stream_pool_bytes(cm.handle, S, nh, nw),), 3, dtype=torch.uint8, device="cuda")
    need = lib.vda_stream_workspace_bytes(cm.handle, B, nh, nw)
    ws = torch.empty(need + 1024, dtype=torch.uint8, device="cuda")
    wp = -(-ws.data_ptr() // 1024) * 1024
    st = torch.cuda.current_stream().cuda_stream
    ok = (cm.handle, fd_d.data_ptr(), od_d.data_ptr(), table.data_ptr(), B, 0, pool.data_ptr(), S, nh, nw, wp, need, st)
    for msg, i, v in [("workspace too small", 11, need - 1), ("null pointer", 1, None), ("bad batch", 4, 0),
                      ("multiples of the patch size", 8, 50)]:
        args = list(ok)
        args[i] = v
        assert lib.vda_stream_step_planes(*args) != 0, msg
        err = lib.vda_last_error().decode()
        assert msg in err and err.startswith("vda_stream_step_planes"), err
    torch.cuda.synchronize()
    assert (out == -7).all() and (pool == 3).all(), "a rejected call launched something"
    assert lib.vda_stream_step_planes(*ok) == 0
    torch.cuda.synchronize()
    assert (out >= 0).all()


# ---------------------------------------------------------------------------------------------- graphs
def test_graphs_replay_mixed_frame_forms_without_capture_or_growth():
    """100 pushes mixing host, CUDA and plane-tuple NV12 frames after every bucket's first use: no new capture, no growth
    of device memory in use, one launch count per bucket, and the RGB group's launch counts."""
    m, _ = build_model("vits", 0, torch.bfloat16)
    fmt = "nv12"
    sizes = [(50, 70), (100, 140), (56, 84), (28, 42)]
    frames = {s: Y.random_video(3, *s, fmt, seed=40 + i) for i, s in enumerate(sizes)}
    g = m.stream_group(4, 56, pixel_format=fmt)
    hs = [g.open() for _ in range(4)]
    size = dict(zip(hs, sizes))
    for k in (1, 2, 4):
        g.push({h: frames[size[h]][0] for h in hs[:k]})
    graphs = {k: v[0] for k, v in g.graphs.items()}
    forms = [{s: [_frame_forms(frames[s][j], fmt, f) for j in range(3)] for s in sizes} for f in ("host", "cuda", "planes")]
    rng = np.random.default_rng(41)
    gc.collect()
    torch.cuda.synchronize()
    mem0, free0 = torch.cuda.memory_allocated(), torch.cuda.mem_get_info()[0]
    per_push = {}
    for p in range(100):
        k = int(rng.integers(1, 5))
        sub = [hs[j] for j in rng.permutation(4)[:k]]
        push = {h: forms[int(rng.integers(3))][size[h]][p % 3] for h in sub}
        n0 = ops.LAUNCHES
        out = g.push(push, to_host=bool(rng.random() < 0.5))
        per_push.setdefault(g.plan.bucket(k), set()).add(ops.LAUNCHES - n0)
        del out
    assert {k: v[0] for k, v in g.graphs.items()} == graphs, "no capture after a bucket's first use"
    assert all(len(v) == 1 for v in per_push.values()), per_push
    gc.collect()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem0 and torch.cuda.mem_get_info()[0] >= free0
    # eager steps: the YUV and the RGB group issue the same number of launches per bucket
    eng = m._ensure_engine()
    counts = {}
    for fmt_ in ("nv12", "rgb"):
        eng.use_graphs = False
        try:
            gg = m.stream_group(4, 56, pixel_format=fmt_)
            hh = [gg.open() for _ in range(4)]
            for k in (1, 2, 4):
                n0 = ops.LAUNCHES
                gg.push({h: (frames[(50, 70)][0] if fmt_ == "nv12" else Y.to_rgb(frames[(50, 70)][0], "nv12"))
                         for h in hh[:k]})
                counts[(fmt_, k)] = ops.LAUNCHES - n0
            gg.close()
        finally:
            eng.use_graphs = True
    assert all(counts[("nv12", k)] == counts[("rgb", k)] for k in (1, 2, 4)), counts


# ---------------------------------------------------------------------------------------------- sharded
def test_sharded_nv12_is_bit_identical_to_one_gpu():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(n, 8)}", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "multi_gpu_nv12_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-3000:])
    assert out.stdout.count("bit-identical") == 3, out.stdout[-2000:]
