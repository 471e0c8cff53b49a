"""CPU: the C host planner of a stream group (vda_stream_plan_*, vda_resize_hw; csrc/stream_plan.cu) against
windows.StreamGroupPlan / get_resize_hw: the same decisions, messages and table bytes over random operations, unchanged
state after a rejected push, the buckets; and the C streaming host compiles and links."""
import os
import subprocess

import numpy as np
import pytest

from video_depth_anything_b200.windows import StreamGroupPlan, get_resize_hw, stream_buckets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


@pytest.fixture(scope="module", autouse=True)
def lib():
    from video_depth_anything_b200 import build
    build.build()


def _both(fn_py, fn_c):
    """Run one operation on both planners: (accepted, result of the Python one, result of the C one); a rejection must
    be a ValueError on both sides with the same message."""
    try:
        rp = ("ok", fn_py())
    except ValueError as e:
        rp = ("err", str(e))
    try:
        rc = ("ok", fn_c())
    except ValueError as e:
        rc = ("err", str(e))
    assert rp[0] == rc[0], (rp, rc)
    if rp[0] == "err":
        assert rp[1] == rc[1]
    return rp[0] == "ok", rp[1], rc[1]


SIZES = [(50, 70), (100, 140), (52, 72), (60, 80), (40, 160), (70, 50), (0, 5)]   # 56: the first three share (56, 84)


@pytest.mark.parametrize("S,num_frames,max_frames,input_size", [(5, 32, 20, 56), (1, 32, None, 56), (3, 9, 6, 56),
                                                                (8, 32, None, 518)])
def test_planner_matches_python_over_random_operations(S, num_frames, max_frames, input_size):
    from video_depth_anything_b200.cmodel import CStreamPlan
    L = num_frames - 1
    py = StreamGroupPlan(S, L, input_size, max_frames)
    cp = CStreamPlan(S, num_frames, input_size, max_frames)
    assert cp.buckets == py.buckets
    rng = np.random.default_rng(S * 100 + num_frames)
    handles, seen_size = [], {}
    stats = dict(pushes=0, rejected=0, wraps=0, first_stacks=0, at_max=0, reopen=0)
    for op in range(400):
        r = rng.random()
        if r < 0.10:
            ok, hp, hc = _both(py.open, cp.open)
            if ok:
                assert hp == hc
                stats["reopen"] += bool(handles) and py.row[hp] < max(py.row.values())
                handles.append(hp)
            continue
        if r < 0.16:
            h = int(rng.choice(handles)) if handles and rng.random() < 0.8 else 1000 + op
            ok, _, _ = _both(lambda: py.close(h), lambda: cp.close(h))
            if ok:
                handles.remove(h)
                seen_size.pop(h, None)
            continue
        if not handles:
            continue
        k = int(rng.integers(1, len(handles) + 1))
        push = [int(h) for h in rng.permutation(handles)[:k]]
        if rng.random() < 0.05:
            push.append(push[0])                                   # named twice
        if rng.random() < 0.05:
            push.append(999)                                       # unknown
        if rng.random() < 0.03:
            push = []
        room = py.max_frames
        counts = []
        for i in range(len(push)):
            c = int(rng.integers(1, max(2, min(L, room - (len(push) - i - 1)) + 1)))
            counts.append(c)
            room -= c
        if rng.random() < 0.08 and counts:
            counts[int(rng.integers(len(counts)))] = int(rng.choice([0, L + 1, py.max_frames]))
        if rng.random() < 0.5:
            counts_arg = counts if any(c != 1 for c in counts) or rng.random() < 0.5 else None
        else:
            counts_arg = [1] * len(push)
        sizes = []
        for h in push:
            if h in seen_size and rng.random() < 0.95:
                sizes.append(seen_size[h])
            else:
                sizes.append(SIZES[int(rng.choice(len(SIZES), p=[.35, .25, .2, .06, .06, .05, .03]))])
        sizes_arg = sizes if rng.random() < 0.9 else None
        t_before = dict(py.t)
        ok, rp, rc = _both(lambda: py.step(push, sizes_arg, counts_arg), lambda: cp.step(push, sizes_arg, counts_arg))
        if not ok:
            stats["rejected"] += 1
            assert py.t == t_before
            continue
        stats["pushes"] += 1
        assert rp[0] == rc[0] and rp[1].dtype == rc[1].dtype == np.int32
        assert rp[1].tobytes() == rc[1].tobytes(), (op, push, counts_arg)
        assert cp.net == py.net
        cs = counts_arg or [1] * len(push)
        for h, c in zip(push, cs):
            stats["wraps"] += t_before[h] <= L < t_before[h] + c
            stats["first_stacks"] += t_before[h] == 0 and c > 1
        stats["at_max"] += sum(cs) == py.max_frames
        if sizes_arg:
            for h, hw in zip(push, sizes_arg):
                seen_size[h] = hw
    print(stats)
    assert stats["pushes"] >= 150 and stats["rejected"] >= 20 and stats["wraps"] >= 3
    if L > 1 and py.max_frames > 1:
        assert stats["first_stacks"] >= 3 and stats["at_max"] >= 1


def test_rejected_push_leaves_the_c_plan_unchanged():
    """After each rejected push the next push's table is the one the same push gives on a plan that never saw it."""
    from video_depth_anything_b200.cmodel import CStreamPlan
    L = 31
    bad = [([0], [(50, 70)], [L + 1]), ([0], [(50, 70)], [0]), ([0, 1], [(50, 70), (50, 70)], [12, 9]),
           ([0, 1], [(50, 70), (60, 70)], [2, 2]), ([0], [(50, 71)], [2]), ([0, 7], [(50, 70), (50, 70)], [1, 1]),
           ([0, 0], [(50, 70), (50, 70)], [1, 1]), ([1], [(0, 70)], [1])]
    a, b = CStreamPlan(2, 32, 56, 20), CStreamPlan(2, 32, 56, 20)
    for p in (a, b):
        assert (p.open(), p.open()) == (0, 1)
        p.step([0], [(50, 70)], [3])
    for handles, sizes, counts in bad:
        with pytest.raises(ValueError):
            a.step(handles, sizes, counts)
        ga, gb = a.step([1, 0], [(100, 140), (50, 70)], [2, 1]), b.step([1, 0], [(100, 140), (50, 70)], [2, 1])
        assert ga[0] == gb[0] and ga[1].tobytes() == gb[1].tobytes()
    with pytest.raises(ValueError, match="max_streams=2"):
        a.open()
    a.close(0)
    with pytest.raises(ValueError, match="unknown or closed"):
        a.close(0)
    assert a.open() == 2                                           # handles are never reused ...
    bk, table = a.step([2], [(10, 14)], [4])                       # ... its pool row is: the lowest free one
    assert bk == 4 and list(table[:4]) == [0, 0, 0, 0]


@pytest.mark.parametrize("S,F", [(1, None), (2, 12), (3, 5), (5, 16), (8, None), (16, 16), (20, None), (7, 40)])
def test_buckets(S, F):
    from video_depth_anything_b200.cmodel import CStreamPlan
    assert CStreamPlan(S, max_frames=F).buckets == StreamGroupPlan(S, max_frames=F).buckets == \
        stream_buckets(S, max(S, 16) if F is None else F)


def test_plan_create_errors():
    from video_depth_anything_b200.cmodel import CStreamPlan
    for args in ((0,), (4, 32, 518, 3), (4, 1), (4, 33), (4, 32, 0)):
        with pytest.raises(ValueError):
            CStreamPlan(*args)


def test_resize_hw_matches_python():
    from video_depth_anything_b200.cmodel import resize_hw
    grid = [(720, 1280), (1080, 1920), (480, 640), (768, 1024), (1280, 720), (1920, 1080), (640, 480), (518, 518),
            (480, 2000), (2000, 480), (100, 178), (100, 179), (1, 1), (1, 3), (3, 1), (14, 14), (7, 9), (50, 70),
            (60, 80), (40, 52), (100, 140), (1, 1000), (999, 1)]
    rng = np.random.default_rng(7)
    grid += [tuple(int(v) for v in rng.integers(1, 4000, 2)) for _ in range(400)]
    for input_size in (518, 56, 42, 70, 280, 364, 700, 1022, 14, 1):
        for h0, w0 in grid:
            assert resize_hw(h0, w0, input_size) == get_resize_hw(h0, w0, input_size), (h0, w0, input_size)


def test_host_stream_builds_and_links(tmp_path):
    from video_depth_anything_b200 import build
    lib = build.build()
    exe = str(tmp_path / "host_stream")
    libdir = os.path.dirname(lib)
    subprocess.check_call(["gcc", "-O1", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(CUDA, "include"), os.path.join(ROOT, "tests", "c_host", "host_stream.c"), "-o", exe,
                           "-L", libdir, "-l:libvda.so", "-L", os.path.join(CUDA, "lib64"), "-lcudart",
                           "-Wl,-rpath," + libdir, "-Wl,-rpath," + os.path.join(CUDA, "lib64")])
    assert subprocess.check_output([exe, "--version"]).decode().strip() == "100"
