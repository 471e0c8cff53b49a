"""GPU: stream groups through the C library alone (the C planner + vda_stream_step, cmodel.CStreamGroup, and the compiled
tests/c_host/host_stream.c) against the Python DepthStreamGroup on the same weights and pushes.  Both issue the same
libvda operator calls with the same packed weights and the same tables, so the depths must be bit-identical."""
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from e2e_checks import build_model  # noqa: E402
from video_depth_anything_b200 import MODEL_CONFIGS  # noqa: E402
from video_depth_anything_b200.cmodel import CModel, CStreamGroup  # noqa: E402
from video_depth_anything_b200.windows import FRAME_DESC, OUT_DESC  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def _models(enc, dtype):
    m, sd = build_model(enc, 0, dtype)
    cm = CModel(**MODEL_CONFIGS[enc], dtype=dtype)
    cm.load_state_dict(sd)
    return m, cm, sd


def _videos(sizes, n, seed):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)).cuda() for h, w in sizes]


def _schedule(n_streams, n_pushes, seed, max_k=6, room=16, reopen=()):
    """[(op, arg)]: ("push", [(stream, k or None)]) with random subsets and stacks, ("reopen", stream)."""
    rng = np.random.default_rng(seed)
    out = []
    for p in range(n_pushes):
        if p in reopen:
            out.append(("reopen", int(rng.integers(n_streams))))
        sub = [i for i in range(n_streams) if rng.random() < 0.75] or [int(rng.integers(n_streams))]
        items, left = [], room
        for j, i in enumerate(sub):
            k = int(rng.integers(2, max_k + 1)) if rng.random() < 0.3 else None
            k = None if k is not None and k > left - (len(sub) - j - 1) else k
            left -= k or 1
            items.append((i, k))
        out.append(("push", items))
    return out


def _drive(group, videos, schedule):
    """Run a schedule on a group (DepthStreamGroup with to_host=False, or CStreamGroup); returns every depth in order."""
    hs = [group.open() for _ in videos]
    t = [0] * len(videos)
    outs = []
    for op, arg in schedule:
        if op == "reopen":
            group.close_stream(hs[arg])
            hs[arg] = group.open()
            continue
        push = {}
        for i, k in arg:
            push[hs[i]] = videos[i][t[i]:t[i] + k] if k else videos[i][t[i]]
            t[i] += k or 1
        got = group.push(push, to_host=False) if not isinstance(group, CStreamGroup) else group.push(push)
        outs += [got[hs[i]].clone() for i, _ in arg]
    return outs, t


def _assert_same(a, b):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and torch.equal(x, y), f"output {i}: max abs diff {(x - y).abs().max().item():.3e}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_vits_group_bit_identical_to_python(dtype):
    """Two frame sizes of one network size (56 x 84), 44 pushes past the slot-ring wrap, random subsets, stacks (causal
    steps) mixed with single frames, a close and reopen; the pool size of both groups."""
    m, cm, _ = _models("vits", dtype)
    videos = _videos([(50, 70), (100, 140), (50, 70)], 200, seed=1)
    sched = _schedule(3, 44, seed=2, reopen=(17,))
    py = m.stream_group(3, 56)
    ref, t = _drive(py, videos, sched)
    assert min(t) > 40
    g = CStreamGroup(cm, 3, 56)
    got, _ = _drive(g, videos, sched)
    _assert_same(got, ref)
    assert any(k for op, arg in sched if op == "push" for _, k in arg)
    assert cm.lib.vda_stream_pool_bytes(cm.handle, 3, 56, 84) == sum(p.numel() * p.element_size() for p in py.pool)
    assert g.pool.numel() == sum(p.numel() * p.element_size() for p in py.pool)
    assert sorted(g.graphs) == sorted([(b, False) for b in py.graphs] + [(b, True) for b in py.causal_graphs])


def test_vitl_518_two_streams_bit_identical_to_python():
    m, cm, _ = _models("vitl", torch.bfloat16)
    videos = _videos([(518, 518), (518, 518)], 52, seed=3)
    sched = [("push", [(0, None), (1, None)] if p % 3 else [(p % 2, None)]) for p in range(36)]
    sched.append(("push", [(0, 8)]))
    py = m.stream_group(2)
    ref, _ = _drive(py, videos, sched)
    py.close()
    got, _ = _drive(CStreamGroup(cm, 2), videos, sched)
    _assert_same(got, ref)


def test_single_stream_bit_identical_to_depth_stream():
    m, cm, _ = _models("vits", torch.bfloat16)
    video = _videos([(60, 80)], 60, seed=4)[0]
    st = m.stream(70)
    g = CStreamGroup(cm, 1, 70)
    h = g.open()
    t = 0
    for k in [1, 1, 4, 1, 8, 1, 3, 16, 1, 1, 5, 2, 1, 9]:
        x = video[t:t + k] if k > 1 else video[t]
        a, b = st.push(x, to_host=False), g.push({h: x})[h]
        assert torch.equal(a, b), t
        t += k
    assert t > 40


def test_graph_replay_equals_eager_and_steps_allocate_nothing():
    """Graph replay against eager steps over 30 pushes; then 50 pushes whose (bucket, causal) graphs all exist already
    leave the device's free memory unchanged (no capture, no allocation)."""
    m, cm, _ = _models("vits", torch.bfloat16)
    videos = _videos([(50, 70), (100, 140)], 500, seed=5)
    sched = _schedule(2, 80, seed=6, max_k=4)
    eager, _ = _drive(CStreamGroup(cm, 2, 56, graphs=False), videos, sched[:30])
    g = CStreamGroup(cm, 2, 56)
    hs = [g.open(), g.open()]
    t = [0, 0]

    def run(part, keep):
        outs = []
        for _, arg in part:
            push = {}
            for i, k in arg:
                push[hs[i]] = videos[i][t[i]:t[i] + k] if k else videos[i][t[i]]
                t[i] += k or 1
            got = g.push(push)
            if keep:
                outs.extend(got[hs[i]].clone() for i, _ in arg)
        return outs
    _assert_same(run(sched[:30], True), eager)
    run(sched[30:80], False)                             # warm-up: every graph the measured pushes replay
    keys = dict(g.graphs)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    run(sched[30:80], False)
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] == free0
    assert g.graphs == keys


def test_rejected_steps_launch_nothing():
    _, cm, _ = _models("vits", torch.bfloat16)
    lib = cm.lib
    B, S, nh, nw = 2, 2, 56, 84
    frame = torch.randint(0, 256, (50, 70, 3), dtype=torch.uint8, device="cuda")
    out = torch.full((B, 50, 70), -7.0, device="cuda")
    fd, od = np.zeros(B, FRAME_DESC), np.zeros(B, OUT_DESC)
    for b in range(B):
        fd[b] = (frame.data_ptr(), 210, 50, 70)
        od[b] = (out[b].data_ptr(), 50, 70)
    fd_d = torch.from_numpy(fd.view(np.uint8)).cuda()
    od_d = torch.from_numpy(od.view(np.uint8)).cuda()
    table = torch.from_numpy(np.concatenate([np.zeros(B, np.int32), np.zeros(B * 33, np.int32),
                                             np.arange(B, dtype=np.int32)])).cuda()
    pool = torch.full((lib.vda_stream_pool_bytes(cm.handle, S, nh, nw),), 3, dtype=torch.uint8, device="cuda")
    need = lib.vda_stream_workspace_bytes(cm.handle, B, nh, nw)
    assert need > 0 and lib.vda_stream_workspace_bytes(cm.handle, B, nh, nw + 1) == -1
    ws = torch.empty(need + 1024, dtype=torch.uint8, device="cuda")
    wp = -(-ws.data_ptr() // 1024) * 1024
    st = torch.cuda.current_stream().cuda_stream
    bare = CModel(**MODEL_CONFIGS["vits"])
    ok = (cm.handle, fd_d.data_ptr(), od_d.data_ptr(), table.data_ptr(), B, 0, pool.data_ptr(), S, nh, nw, wp, need, st)
    bad = {"workspace too small": dict(i=11, v=need - 1),
           "null pointer": dict(i=1, v=None),
           "not finalized": dict(i=0, v=bare.handle),
           "multiples of the patch size": dict(i=8, v=50),
           "multiples of the patch size ": dict(i=9, v=85),
           "bad batch": dict(i=4, v=0),
           "bad pool size": dict(i=7, v=0)}
    for msg, d in bad.items():
        args = list(ok)
        args[d["i"]] = d["v"]
        assert lib.vda_stream_step(*args) != 0, msg
        assert msg.strip() in lib.vda_last_error().decode(), (msg, lib.vda_last_error())
    torch.cuda.synchronize()
    assert (out == -7).all() and (pool == 3).all(), "a rejected call launched something"
    assert lib.vda_stream_step(*ok) == 0
    torch.cuda.synchronize()
    assert (out >= 0).all()
    bare.close()


def test_c_host_program_bit_identical_to_python(tmp_path):
    exe = str(tmp_path / "host_stream")
    from video_depth_anything_b200 import build
    libdir = os.path.dirname(build.build())
    subprocess.check_call(["gcc", "-O1", "-std=c99", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(CUDA, "include"),
                           os.path.join(ROOT, "tests", "c_host", "host_stream.c"), "-o", exe, "-L", libdir, "-l:libvda.so",
                           "-L", os.path.join(CUDA, "lib64"), "-lcudart", "-Wl,-rpath," + libdir,
                           "-Wl,-rpath," + os.path.join(CUDA, "lib64")])
    m, sd = build_model("vits", 0, torch.bfloat16)
    sizes = [(50, 70), (100, 140), (52, 72)]                # one network size, 56 x 84
    videos = _videos(sizes, 120, seed=7)
    sched = _schedule(3, 40, seed=8, max_k=5)
    py = m.stream_group(3, 56)
    ref, t = _drive(py, videos, sched)
    wpath, ipath, opath = (str(tmp_path / n) for n in ("weights.bin", "input.bin", "output.bin"))
    with open(wpath, "wb") as f:
        f.write(struct.pack("<i", len(sd)))
        for k, v in sd.items():
            a = v.detach().to("cpu", torch.float32).contiguous().numpy()
            name = k.encode()
            f.write(struct.pack("<i", len(name)) + name + struct.pack("<i", a.ndim) + struct.pack(f"<{a.ndim}q", *a.shape))
            f.write(a.tobytes())
    with open(ipath, "wb") as f:
        f.write(struct.pack("<3i", 3, 56, len(sched)))
        for v, (h, w) in zip(videos, sizes):
            f.write(struct.pack("<3i", v.shape[0], h, w) + v.cpu().numpy().tobytes())
        for _, arg in sched:
            f.write(struct.pack("<i", len(arg)) + b"".join(struct.pack("<2i", i, k or 1) for i, k in arg))
    cfg = MODEL_CONFIGS["vits"]
    r = subprocess.run([exe, "vits", str(cfg["features"]), *map(str, cfg["out_channels"]), "0", wpath, ipath, opath],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout
    print(r.stdout.strip())
    out = torch.from_numpy(np.fromfile(opath, dtype=np.float32))
    flat = torch.cat([d.flatten().cpu() for d in ref])
    assert out.shape == flat.shape and torch.equal(out, flat), f"max abs diff {(out - flat).abs().max().item():.3e}"
