"""CPU: frame sizes in a stream group (windows.StreamGroupPlan with sizes, windows.group_descriptors,
windows.group_block_layout): one network size per group, one frame size per stream, the per-row descriptors of a push."""
import numpy as np
import pytest

from video_depth_anything_b200.windows import (FRAME_DESC, OUT_DESC, STREAM_CONTEXT, StreamGroupPlan, get_resize_hw,
                                               group_block_layout, group_descriptors, split_group_table, stream_context)

SAME = [(25, 35), (50, 70), (56, 84), (100, 140), (75, 105)]     # all (56, 84) at input_size 56
OTHER = [(40, 70), (60, 70)]                                      # (56, 98), (56, 70)


def test_size_sets():
    assert {get_resize_hw(h, w, 56) for h, w in SAME} == {(56, 84)}
    assert all(get_resize_hw(h, w, 56) != (56, 84) for h, w in OTHER)
    assert get_resize_hw(720, 1280) == get_resize_hw(1080, 1920) == (518, 924)


def _expect_ok(plan_size, net, handles, sizes):
    """The rules, restated: a stream keeps its first size; every frame maps to the group's (or the push's) network size."""
    if any(h in plan_size and plan_size[h] != s for h, s in zip(handles, sizes)):
        return False
    nets = {get_resize_hw(h, w, 56) for h, w in sizes}
    return len(nets) == 1 and (net is None or nets == {net})


def test_plan_sizes_300_pushes():
    L, S = STREAM_CONTEXT, 8
    rng = np.random.default_rng(1)
    plan = StreamGroupPlan(S, L, input_size=56)
    t, size, net = {}, {}, None                       # the model
    accepted = rejected = 0
    for step in range(300):
        if rng.random() < 0.15 and t:
            h = list(t)[rng.integers(len(t))]
            plan.close(h)
            del t[h]
            size.pop(h, None)
        if rng.random() < 0.3 and len(t) < S:
            t[plan.open()] = 0
        if not t:
            continue
        k = int(rng.integers(1, len(t) + 1))
        handles = [list(t)[i] for i in rng.permutation(len(t))[:k]]
        # mostly each stream's own size, sometimes a random one (same network size or not)
        pool = SAME + OTHER if rng.random() < 0.2 else SAME
        sizes = [size[h] if h in size and rng.random() < 0.9 else pool[rng.integers(len(pool))] for h in handles]
        ok = _expect_ok(size, net, handles, sizes)
        before = (dict(plan.t), dict(plan.size), plan.net)
        if not ok:
            with pytest.raises(ValueError):
                plan.step(handles, sizes)
            assert (plan.t, plan.size, plan.net) == before, "a rejected push changes nothing"
            rejected += 1
            continue
        bk, table = plan.step(handles, sizes)
        accepted += 1
        net = get_resize_hw(*sizes[0], 56)
        assert plan.net == net
        for h, s in zip(handles, sizes):
            size.setdefault(h, s)
        assert plan.size == size
        rows, ctx, idx = split_group_table(table, bk, L)     # the table layout is unchanged
        assert table.size == bk * (L + 4)
        for i, h in enumerate(handles):
            _, slots, write = stream_context(t[h], L)
            assert rows[i] == plan.row[h] and idx[i] == i and ctx[i, 0] == len(slots) and ctx[i, 1] == write
            t[h] += 1
        assert (rows[k:] == -1).all() and (idx[k:] == 0).all()
        # descriptors: each row's own address, pitch and size; pad rows read row 0's frame and write nothing
        pitches = [3 * w + int(rng.integers(0, 3)) * 64 for _, w in sizes]
        srcs = [(0x10000 * (i + 1), p, h0, w0) for i, (p, (h0, w0)) in enumerate(zip(pitches, sizes))]
        dsts = [0x900000 + 0x1000 * i for i in range(k)]
        fd, od = group_descriptors(bk, srcs, dsts)
        assert fd.dtype == FRAME_DESC and od.dtype == OUT_DESC and len(fd) == len(od) == bk
        for i, (src, p, h0, w0) in enumerate(srcs):
            assert tuple(fd[i]) == (src, p, h0, w0) and tuple(od[i]) == (dsts[i], h0, w0)
        assert (fd[k:] == fd[0]).all() and (od[k:]["H0"] == 0).all() and (od[k:]["W0"] == 0).all()
    assert accepted > 150 and rejected > 10


def test_size_rules():
    plan = StreamGroupPlan(4, input_size=56)
    a, b = plan.open(), plan.open()
    with pytest.raises(ValueError, match=r"\(56, 84\).*\(56, 98\)|\(56, 98\).*\(56, 84\)"):
        plan.step([a, b], [(50, 70), (40, 70)])      # network sizes differ within the first push
    assert plan.net is None and plan.t[a] == 0
    plan.step([a, b], [(50, 70), (100, 140)])
    with pytest.raises(ValueError, match="differs from its first"):
        plan.step([a], [(25, 35)])                   # same network size, another size of this stream
    with pytest.raises(ValueError, match=r"\(56, 70\).*\(56, 84\)"):
        plan.step([plan.open()], [(60, 70)])          # the message names both network sizes
    c = plan.open()
    plan.step([c], [(56, 84)])                        # a new stream takes any size of the group's network size
    plan.close(a)
    d = plan.open()
    assert plan.row[d] == 0
    plan.step([d], [(25, 35)])                        # the reopened row starts over with a new size
    with pytest.raises(ValueError):
        plan.step([d], [(0, 35)])
    with pytest.raises(ValueError):
        plan.step([d, c], [(25, 35)])                 # one size per stream


def test_descriptor_errors_and_layout():
    with pytest.raises(ValueError):
        group_descriptors(2, [(1, 8, 2, 3)], [0])     # pitch < 3 * W0
    with pytest.raises(ValueError):
        group_descriptors(1, [(1, 9, 2, 3)] * 2, [0, 0])
    assert FRAME_DESC.itemsize == 24 and OUT_DESC.itemsize == 16   # sizeof(vda_frame_desc), sizeof(vda_out_desc)
    for bk in (1, 2, 3, 8):
        fs, os_, ts = group_block_layout(bk)
        assert fs.start == 0 and fs.stop == os_.start and os_.stop == ts.start and ts.stop - ts.start == 4 * bk * 35
        assert os_.start % 8 == 0 and ts.start % 8 == 0
