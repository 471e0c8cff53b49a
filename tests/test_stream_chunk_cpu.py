"""CPU: pushes that give a stream several consecutive frames (windows.StreamGroupPlan.step with `counts`): the bucket
rule, the causal context encoding of the table checked against a model of what the kernels do with it, and the
rejections."""
import numpy as np
import pytest

from video_depth_anything_b200.windows import (STREAM_CONTEXT, StreamGroupPlan, split_group_table, stream_buckets,
                                               stream_context)


def test_buckets_with_max_frames():
    assert stream_buckets(5, 16) == [1, 2, 4, 5, 8, 16]
    assert stream_buckets(8, 16) == [1, 2, 4, 8, 16]
    assert stream_buckets(1, 16) == [1, 2, 4, 8, 16]
    assert stream_buckets(16, 16) == stream_buckets(16) == [1, 2, 4, 8, 16]
    assert stream_buckets(3, 5) == [1, 2, 3, 4, 5]
    assert stream_buckets(2, 12) == [1, 2, 4, 8, 12]
    for s in (1, 2, 5, 8, 16):
        assert stream_buckets(s, None) == stream_buckets(s)
        assert stream_buckets(s, 32)[:len(stream_buckets(s))] == stream_buckets(s)   # single-frame pushes keep their bucket
    with pytest.raises(ValueError):
        stream_buckets(4, 3)
    assert StreamGroupPlan(8).max_frames == 16 and StreamGroupPlan(20).max_frames == 20   # default max(max_streams, 16)
    assert StreamGroupPlan(1).buckets == [1, 2, 4, 8, 16]
    with pytest.raises(ValueError):
        StreamGroupPlan(5, max_frames=4)


def _apply(table, bk, plan_rows, starts, L, pool):
    """What the causal kernel and the store read and write, on frame ids: every row reads its context (pool slots hold
    the frame ids written by earlier pushes, negative entries name a row of this push), then every row's frame goes to
    its write slot.  `starts`: batch row -> (pool row, frame id).  Returns the frame ids each row read."""
    rows, ctx, _ = split_group_table(table, bk, L)
    reads = {}
    for b in range(bk):
        if rows[b] < 0:
            continue
        r, f = starts[b]
        assert rows[b] == r
        got = []
        for e in ctx[b, 2:2 + ctx[b, 0]]:
            if e < 0:
                rb = -1 - e
                assert 0 <= rb < b, "a row reads only earlier rows of its push"
                assert rows[rb] == r, "an in-push reference names a frame of the same stream"
                got.append(starts[rb][1])
            else:
                got.append(pool[r][e])
        reads[b] = got
    for b in range(bk):
        if rows[b] >= 0:
            pool[rows[b]][ctx[b, 1]] = starts[b][1]
    return reads


def test_chunk_plan_300_random_pushes():
    L, S, F = STREAM_CONTEXT, 6, 24
    rng = np.random.default_rng(1)
    plan = StreamGroupPlan(S, L, max_frames=F)
    t, pool = {}, {r: {} for r in range(S)}              # model: handle -> frames pushed; pool row -> slot -> frame id
    wraps = first_stacks = multi = 0
    for step in range(300):
        if rng.random() < 0.12 and t:
            h = list(t)[rng.integers(len(t))]
            plan.close(h)
            del t[h]
        if rng.random() < 0.3 and len(t) < S:
            h = plan.open()
            pool[plan.row[h]] = {}                       # a reopened row's stale slots are never read (checked below)
            t[h] = 0
        if not t:
            continue
        live = list(t)
        handles = [live[i] for i in rng.permutation(len(live))[:int(rng.integers(1, len(live) + 1))]]
        counts, room = [], F
        for _ in handles:
            c = int(rng.integers(1, min(L, room - (len(handles) - len(counts) - 1)) + 1))
            counts.append(c)
            room -= c
        bk, table = plan.step(handles, counts=counts)
        assert bk == min(b for b in plan.buckets if b >= sum(counts))
        assert table.dtype == np.int32 and table.size == bk * (L + 4)
        rows, ctx, idx = split_group_table(table, bk, L)
        starts, b = {}, 0
        for h, c in zip(handles, counts):
            writes = []
            for j in range(c):
                starts[b] = (plan.row[h], t[h] + j)
                ids, _, write = stream_context(t[h] + j, L)
                assert ctx[b, 0] == len(ids) and ctx[b, 1] == write and idx[b] == b
                writes.append(write)
                b += 1
            assert len(set(writes)) == len(writes), "a stream's write slots in one push are distinct"
            wraps += t[h] < 32 <= t[h] + c
            first_stacks += t[h] == 0 and c > 1
            multi += c > 1
        assert (rows[b:] == -1).all() and (ctx[b:, 0] == 0).all()
        reads = _apply(table, bk, rows, starts, L, pool)
        for b, (r, f) in starts.items():
            ids, _, _ = stream_context(f, L)
            assert reads[b] == ids, (step, b, f)
            t0 = f - (b - min(bb for bb, (rr, _) in starts.items() if rr == r))
            rows_ctx = ctx[b, 2:2 + ctx[b, 0]]
            assert all((e < 0) == (fid >= t0) for e, fid in zip(rows_ctx, ids)), \
                "frames of this push come from its rows, never from a slot it writes"
        for h, c in zip(handles, counts):
            t[h] += c
        assert plan.t == t
    assert wraps > 5 and first_stacks > 5 and multi > 100


def test_single_frame_tables_unchanged():
    L = STREAM_CONTEXT
    a, b = StreamGroupPlan(4), StreamGroupPlan(4)
    ha, hb = [a.open() for _ in range(4)], [b.open() for _ in range(4)]
    rng = np.random.default_rng(2)
    for _ in range(80):
        k = int(rng.integers(1, 5))
        sub = [int(i) for i in rng.permutation(4)[:k]]
        bk1, t1 = a.step([ha[i] for i in sub])
        bk2, t2 = b.step([hb[i] for i in sub], counts=[1] * k)
        assert bk1 == bk2 and np.array_equal(t1, t2)
        rows, ctx, _ = split_group_table(t1, bk1, L)
        assert (ctx[:, 2:] >= 0).all(), "single-frame tables name no batch row"


def test_chunk_errors_leave_state_unchanged():
    L = STREAM_CONTEXT
    plan = StreamGroupPlan(2, L, input_size=56, max_frames=20)
    a, b = plan.open(), plan.open()
    plan.step([a], sizes=[(50, 70)], counts=[3])
    state = (dict(plan.t), dict(plan.size), plan.net)
    bad = [([a], [(50, 70)], [L + 1]),                   # more frames than the context length
           ([a], [(50, 70)], [0]),
           ([a, b], [(50, 70), (50, 70)], [12, 9]),     # more frames than max_frames
           ([a, b], [(50, 70), (50, 70)], [2]),         # one count per stream
           ([a, b], [(50, 70), (60, 70)], [2, 2]),      # b's first stack maps to another network size
           ([a], [(50, 71)], [2])]                      # a's stack differs from a's first frame
    for handles, sizes, counts in bad:
        with pytest.raises(ValueError):
            plan.step(handles, sizes, counts)
        assert (dict(plan.t), dict(plan.size), plan.net) == state
    bk, _ = plan.step([a, b], [(50, 70), (50, 70)], [16, 1])
    assert bk == 20 and plan.t == {a: 19, b: 1}


def test_binding_arity_of_the_causal_entry_points():
    """The ctypes prototypes of the two new entry points take as many arguments as include/vda.h declares."""
    import os
    import re
    from video_depth_anything_b200 import _lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "vda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for name in ("vda_attention_temporal_step_causal", "vda_stream_cache_store"):
        params = re.search(name + r"\s*\((.*?)\)\s*;", hdr, flags=re.S).group(1)
        assert len(_lib._SIGS[name][1]) == len(params.split(",")), name
