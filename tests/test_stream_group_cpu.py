"""CPU: the host plan of a stream group (windows.StreamGroupPlan): handles, pool rows, per-stream steps, buckets and the
rows | ctx | idx table of every push."""
import numpy as np
import pytest

from video_depth_anything_b200.windows import (STREAM_CONTEXT, StreamGroupPlan, split_group_table, stream_buckets,
                                               stream_context)


def test_buckets():
    assert stream_buckets(1) == [1]
    assert stream_buckets(2) == [1, 2]
    assert stream_buckets(5) == [1, 2, 4, 5]
    assert stream_buckets(8) == [1, 2, 4, 8]
    assert stream_buckets(16) == [1, 2, 4, 8, 16]
    with pytest.raises(ValueError):
        stream_buckets(0)


def test_group_plan_300_pushes_random_subsets_and_open_close():
    L, S = STREAM_CONTEXT, 8
    rng = np.random.default_rng(0)
    plan = StreamGroupPlan(S, L)
    t = {}                                          # the model: handle -> frames pushed so far
    used, reuses = set(), 0                          # pool rows ever handed out, opens that reuse one
    for step in range(300):
        if rng.random() < 0.15 and t:               # close a random stream
            h = list(t)[rng.integers(len(t))]
            plan.close(h)
            del t[h]
        if rng.random() < 0.3 and len(t) < S:       # open one
            free = set(range(S)) - set(plan.row.values())
            h = plan.open()
            assert plan.row[h] == min(free) and h not in t
            reuses += plan.row[h] in used
            used.add(plan.row[h])
            t[h] = 0
        rows_live = [plan.row[h] for h in t]
        assert len(set(rows_live)) == len(rows_live), "two live streams share a pool row"
        if not t:
            continue
        k = int(rng.integers(1, len(t) + 1))
        handles = [list(t)[i] for i in rng.permutation(len(t))[:k]]
        bk, table = plan.step(handles)
        assert bk == min(b for b in stream_buckets(S) if b >= k)
        assert table.dtype == np.int32 and table.size == bk * (L + 4)
        rows, ctx, idx = split_group_table(table, bk, L)
        for i, h in enumerate(handles):
            _, slots, write = stream_context(t[h], L)
            assert rows[i] == plan.row[h] and idx[i] == i
            assert ctx[i, 0] == len(slots) and ctx[i, 1] == write
            assert list(ctx[i, 2:2 + len(slots)]) == slots
            t[h] += 1
        assert (rows[k:] == -1).all() and (idx[k:] == 0).all() and (ctx[k:, 0] == 0).all()
        assert plan.t == t
    assert reuses > 0                               # reopened rows restarted at t = 0 (checked through `t`)


def test_reused_row_restarts_at_zero():
    plan = StreamGroupPlan(2)
    a, b = plan.open(), plan.open()
    for _ in range(40):
        plan.step([a, b])
    plan.close(a)
    c = plan.open()
    assert plan.row[c] == 0 and plan.t[c] == 0 and c != a
    bk, table = plan.step([c])
    rows, ctx, _ = split_group_table(table, bk)
    assert bk == 1 and rows[0] == 0 and ctx[0, 0] == 0 and ctx[0, 1] == 0       # t = 0: no context, writes slot 0


def test_plan_errors():
    plan = StreamGroupPlan(2)
    a, b = plan.open(), plan.open()
    with pytest.raises(ValueError):
        plan.open()                                  # more than max_streams
    with pytest.raises(ValueError):
        plan.step([a, a])                            # named twice
    with pytest.raises(ValueError):
        plan.step([a, 99])                           # unknown
    with pytest.raises(ValueError):
        plan.step([])
    plan.close(b)
    with pytest.raises(ValueError):
        plan.step([b])                               # closed
    with pytest.raises(ValueError):
        plan.close(b)
    assert plan.t[a] == 0                            # failed pushes advance nothing
