"""N>1 host logic on CPU (gloo, world sizes 1-4): window partition + gather of per-window depths to rank 0 reproduces
the single-process window stack bit-for-bit, and the sequential alignment (oracle restatement of
video_depth.py:216-252) gives the same video from the gathered stack; the two-phase exchange + finalisation gives it
too, also when some ranks hold no window."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from video_depth_anything_b200.parallel import gather_window_depths, partition_windows  # noqa: E402
from video_depth_anything_b200.windows import INFER_LEN, num_windows, window_source_indices  # noqa: E402


def fake_raw(window_id: int, h=6, w=5) -> torch.Tensor:
    """Deterministic stand-in for one window's raw depth: positive, window- and slot-dependent."""
    g = torch.Generator().manual_seed(1000 + window_id)
    return torch.rand(INFER_LEN, h, w, generator=g) * (1.0 + 0.1 * window_id) + 0.05 * window_id + 0.1


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n_frames, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        parts = partition_windows(num_windows(n_frames), world)
        mine = [fake_raw(k) for k in parts[rank]]
        local = torch.stack(mine) if mine else torch.empty(0, INFER_LEN, 6, 5)
        allraw = gather_window_depths(local, [len(p) for p in parts], dst=0)
        if rank == 0:
            np.save(out_path, allraw.numpy())
        else:
            assert allraw is None
    finally:
        dist.destroy_process_group()


def test_partition_is_contiguous_balanced_and_complete():
    for k in (0, 1, 2, 7, 8, 9, 94):
        for world in (1, 2, 3, 4, 8):
            parts = partition_windows(k, world)
            flat = [i for p in parts for i in p]
            assert flat == list(range(k))
            sizes = [len(p) for p in parts]
            assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
    with pytest.raises(ValueError):
        partition_windows(3, 0)


def test_windows_depend_on_input_frames_only():
    # closed form (SURVEY.md §3.2): slot 0 is always frame 0, slot 1 = 22k-10, then the natural run
    wins = window_source_indices(100)
    assert len(wins) == 5 and wins[0] == list(range(32))
    assert wins[2][:3] == [0, 34, 46] and wins[4][-1] == 99


@pytest.mark.parametrize("world,n_frames", [(2, 23), (2, 70), (2, 131), (3, 23)])
def test_gather_matches_single_process(tmp_path, world, n_frames):
    """The exchange of ranks on several hosts; (3, 23) has a rank with no window."""
    from oracle import vda_oracle as O
    port = _free_port()
    out = str(tmp_path / "gathered.npy")
    mp.spawn(_worker, args=(world, port, n_frames, out), nprocs=world, join=True)
    got = np.load(out)
    k = num_windows(n_frames)
    ref = torch.stack([fake_raw(i) for i in range(k)]).numpy()
    assert got.shape == ref.shape and np.array_equal(got, ref)
    # the alignment recurrence consumes the gathered stack exactly like the single-process list
    a = O.align_windows([w[i].copy() for w in got for i in range(INFER_LEN)], n_frames, "affine")
    b = O.align_windows([w[i].copy() for w in ref for i in range(INFER_LEN)], n_frames, "affine")
    assert np.array_equal(a, b) and a.shape[0] == n_frames


def test_frame_spans_tile_the_video():
    """Two-phase driver: the frames finalised by each rank's block of windows partition [0, n) in rank order."""
    from video_depth_anything_b200.parallel import frame_span
    for n in (1, 23, 45, 70, 100, 131, 2048):
        K = num_windows(n)
        for world in (1, 2, 3, 8):
            spans = [frame_span(p[0], p[-1] + 1, K, n) if len(p) else (0, 0) for p in partition_windows(K, world)]
            assert [f for lo, hi in spans for f in range(lo, hi)] == list(range(n)), (n, world, spans)


# ------------------------------------------------------------------------------------------------ two-phase driver
class _CpuKernels:
    """CPU stand-in for the libvda kernels two_phase_finalise sequences (numpy float32 arithmetic written like the
    reference's own lines, video_depth.py:227-250): the test exercises the product's exchange + sequencing code."""

    def __init__(self):
        from video_depth_anything_b200.windows import INTERP_LEN
        step = 1.0 / (INTERP_LEN - 1)
        self.w = [0.0] + [i * step for i in range(1, INTERP_LEN - 1)] + [1.0]

    def align_chain(self, anchors, affine):
        from oracle import vda_oracle as O
        a = anchors.numpy()
        K = a.shape[0]
        table = np.zeros((K, 2), np.float32)
        table[0] = (1.0, 0.0)
        ref0, ref1 = a[0, 0], a[0, 2].copy()
        for k in range(1, K):
            s, t = (1.0, 0.0)
            if affine:
                s, t = O.compute_scale_and_shift(np.concatenate([a[k, 0], a[k, 1]]), np.concatenate([ref0, ref1]))
            table[k] = (s, t)
            ref1 = a[k, 2] * np.float32(s) + np.float32(t)
            ref1[ref1 < 0] = 0
        return torch.from_numpy(table)

    def affine_clamp_blend(self, x, ss, out, prev=None, blend=False):
        s, t = np.float32(ss[0].item()), np.float32(ss[1].item())
        v = x.numpy() * s + t
        v[v < 0] = 0
        if blend:
            p = prev.numpy()
            v = np.stack([p[i] * (1 - self.w[i]) + v[i] * self.w[i] for i in range(v.shape[0])]).astype(np.float32)
        out.copy_(torch.from_numpy(v))
        return out


def _two_phase_worker(rank, world, port, n_frames, mode, out_dir):
    from video_depth_anything_b200.parallel import two_phase_finalise
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        K = num_windows(n_frames)
        parts = partition_windows(K, world)
        counts = [len(p) for p in parts]
        # (negative values too: the clamp must act exactly where the reference's does)
        raws = torch.stack([fake_raw(k) - 0.3 for k in parts[rank]]) if counts[rank] else torch.empty(0, INFER_LEN, 6, 5)
        got = []
        two_phase_finalise(raws, counts, K, n_frames, mode == "affine", _CpuKernels(),
                           lambda fr, f0: got.append((f0, fr.clone().numpy())))
        np.save(os.path.join(out_dir, f"r{rank}.npy"), np.array(got, dtype=object), allow_pickle=True)
    finally:
        if world > 1:
            dist.destroy_process_group()


@pytest.mark.parametrize("world,n_frames,mode", [(1, 70, "affine"), (2, 70, "affine"), (2, 131, "identity"),
                                                 (3, 200, "affine"), (3, 100, "affine"), (3, 23, "affine"),
                                                 (4, 50, "identity")])
def test_two_phase_finalise_matches_sequential_alignment(tmp_path, world, n_frames, mode):
    """The scalable driver's exchange (halo point-to-point, anchor all-gather) + per-rank finalisation, run with gloo on
    CPU tensors, emits every video frame exactly once and equals the reference's sequential alignment of the full
    window stack (oracle restatement of video_depth.py:216-252).  (3, 23) and (4, 50) have ranks with no window."""
    from oracle import vda_oracle as O
    port = _free_port()
    if world == 1:
        _two_phase_worker(0, 1, port, n_frames, mode, str(tmp_path))
    else:
        mp.spawn(_two_phase_worker, args=(world, port, n_frames, mode, str(tmp_path)), nprocs=world, join=True)
    K = num_windows(n_frames)
    full = [(fake_raw(k) - 0.3).numpy() for k in range(K)]
    ref = O.align_windows([w[i].copy() for w in full for i in range(INFER_LEN)], n_frames, mode)
    out = np.full_like(ref, np.nan)
    seen = np.zeros(n_frames, dtype=int)
    for r in range(world):
        for f0, fr in np.load(os.path.join(str(tmp_path), f"r{r}.npy"), allow_pickle=True):
            out[f0:f0 + fr.shape[0]] = fr
            seen[f0:f0 + fr.shape[0]] += 1
    assert (seen == 1).all(), seen
    np.testing.assert_allclose(out, ref, rtol=2e-6, atol=2e-6)


def test_rank_core_slices_are_disjoint_and_cover():
    from video_depth_anything_b200.parallel import rank_core_slice
    cores = list(range(3, 27))                       # 24 cores, ids not starting at 0
    for world in (1, 2, 3, 4, 8):
        sl = [rank_core_slice(r, world, cores) for r in range(world)]
        flat = [c for s in sl for c in s]
        assert len(set(flat)) == len(flat) and set(flat) <= set(cores)
        assert all(len(s) == len(cores) // world for s in sl)
    assert rank_core_slice(1, 8, list(range(12))) == list(range(12))      # < 2 cores per rank: no pinning
    with pytest.raises(ValueError):
        rank_core_slice(2, 2, cores)


# ---- bounded device buffers of the long-video driver (pure index logic in windows.py) -------------------------------
def test_aligner_ring_every_frame_leaves_once_and_is_never_overwritten_early():
    """Replay WindowAligner's push / _send bookkeeping on frame ids: each window's 22 new frames and its cross-fade tail are
    contiguous in the ring, a ring slot is only overwritten after its frame was handed to the D2H pipeline, and the
    frames leave in order, each exactly once."""
    from video_depth_anything_b200.windows import INFER_LEN, INTERP_LEN, OVERLAP, aligner_ring_len, aligner_ring_pos
    seg = INFER_LEN - OVERLAP
    for n in list(range(1, 300)) + [2048, 2049, 5000]:
        ring_len = aligner_ring_len(n)
        assert ring_len % seg == 0 and 2 * seg <= ring_len <= 4 * seg
        ring, out, sent, filled = [None] * ring_len, [], 0, 0

        def send(upto):
            nonlocal sent
            upto = min(upto, n)
            while upto > sent:
                r = aligner_ring_pos(sent, ring_len)
                m = min(upto - sent, ring_len - r)
                assert ring[r:r + m] == list(range(sent, sent + m))
                out.extend(range(sent, sent + m))
                sent += m

        for w in range(-(-n // seg)):
            if filled == 0:
                r = aligner_ring_pos(0, ring_len)
                assert r + INFER_LEN <= ring_len
                ring[r:r + INFER_LEN] = range(INFER_LEN)
                filled = INFER_LEN
            else:
                rt = aligner_ring_pos(filled - INTERP_LEN, ring_len)
                assert ring[rt:rt + INTERP_LEN] == list(range(filled - INTERP_LEN, filled))      # tail: contiguous, intact
                r = aligner_ring_pos(filled, ring_len)
                assert r % seg == 0 and r + seg <= ring_len
                assert all(o is None or o < sent for o in ring[r:r + seg])                          # old frames already sent
                ring[r:r + seg] = range(filled, filled + seg)
                filled += seg
            send(filled - INTERP_LEN)
        send(n)
        assert out == list(range(n))


def test_upload_ring_keeps_every_frame_a_window_reads_resident():
    """Replay FrameUploader.ensure on frame ids for whole videos and for contiguous rank blocks: when a window runs, every
    source frame it reads sits in the device slot the index tables point at."""
    from video_depth_anything_b200.windows import upload_ring_plan, window_source_indices
    for n, block in ((50, None), (300, None), (700, None), (2048, None), (2048, (40, 60)), (5000, (100, 228))):
        wins = window_source_indices(n)
        ids = list(range(len(wins))) if block is None else list(range(*block))
        needed = sorted({i for k in ids for i in wins[k]})
        pos = {f: j for j, f in enumerate(needed)}
        ring, n_slots, slots, chunks = upload_ring_plan(len(needed))
        assert ring == (len(needed) > 257) and n_slots == (257 if ring else len(needed))
        assert chunks[0][0] == 0 and chunks[-1][1] == len(needed) and all(a[1] == b[0] for a, b in zip(chunks, chunks[1:]))
        dev, uploaded, c = [None] * n_slots, 0, 0
        for k in ids:
            while uploaded < pos[max(wins[k])] + 1:
                lo, hi = chunks[c]
                d0 = slots[lo]
                assert slots[lo:hi] == list(range(d0, d0 + hi - lo))            # a chunk lands in consecutive slots
                dev[d0:d0 + hi - lo] = needed[lo:hi]
                uploaded, c = hi, c + 1
            assert all(dev[slots[pos[f]]] == f for f in wins[k])
