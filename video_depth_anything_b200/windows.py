"""Host-side logic of the long-video driver: window bookkeeping, resize geometry and frame preprocessing.

Reference: video_depth_anything/video_depth.py:166-201 and util/transform.py:62-158."""
from __future__ import annotations

from typing import Iterable, List

import numpy as np

# video_depth.py:29-33 — "infer settings, do not change"
INFER_LEN = 32
OVERLAP = 10
KEYFRAMES = [0, 12, 24, 25, 26, 27, 28, 29, 30, 31]
INTERP_LEN = 8
STEP = INFER_LEN - OVERLAP

_MEAN = np.array([0.485, 0.456, 0.406], dtype=np.float64)
_STD = np.array([0.229, 0.224, 0.225], dtype=np.float64)


def num_windows(n_frames: int) -> int:
    return -(-n_frames // STEP)


def window_source_indices(n_frames: int) -> List[List[int]]:
    """Source frame of every slot of every window.  The reference pads the frame list with copies of the last
    frame (video_depth.py:187-191), slices 32 frames every 22, and overwrites the first 10 slots with the
    previous window's KEYFRAMES slots (:200-201).  Unrolled, that recurrence has the closed form
        window 0 : 0..31
        window k : [0, 22k-10, 22k+2, ..., 22k+31]      (indices clipped to n-1)
    so windows depend on input frames only and can be computed in any order / on any GPU."""
    if n_frames <= 0:
        raise ValueError("empty video")
    out = []
    for k in range(num_windows(n_frames)):
        if k == 0:
            idx = list(range(INFER_LEN))
        else:
            idx = [0, STEP * k - OVERLAP] + [STEP * k + 2 + j for j in range(INFER_LEN - 2)]
        out.append([min(i, n_frames - 1) for i in idx])
    return out


def _constrain(x: float, min_val: int) -> int:
    y = int(np.round(x / 14) * 14)
    if y < min_val:
        y = int(np.ceil(x / 14) * 14)
    return y


def get_resize_hw(h0: int, w0: int, input_size: int = 518):
    """Network input size for an (h0, w0) video: aspect guard (video_depth.py:167-171) then Resize.get_size with
    keep_aspect_ratio / lower_bound / multiple of 14 (util/transform.py:62-107)."""
    ratio = max(h0, w0) / min(h0, w0)
    if ratio > 1.78:
        input_size = int(input_size * 1.777 / ratio)
        input_size = round(input_size / 14) * 14
    scale_h, scale_w = input_size / h0, input_size / w0
    if scale_w > scale_h:
        scale_h = scale_w
    else:
        scale_w = scale_h
    return _constrain(scale_h * h0, input_size), _constrain(scale_w * w0, input_size)


def preprocess_frames(frames: np.ndarray, indices: Iterable[int], input_size: int = 518) -> np.ndarray:
    """uint8 [N,H0,W0,3] RGB -> float32 [len(indices),3,nh,nw]: /255, cv2 INTER_CUBIC resize, ImageNet normalise in
    float64, CHW (util/transform.py:109-158 as composed at video_depth.py:173-185,198).  Each source frame is
    processed once (the reference redoes the overlap frames for every window)."""
    import cv2
    indices = list(indices)
    h0, w0 = frames.shape[1:3]
    nh, nw = get_resize_hw(h0, w0, input_size)
    out = np.empty((len(indices), 3, nh, nw), dtype=np.float32)
    for j, i in enumerate(indices):
        img = frames[i].astype(np.float32) / 255.0
        img = cv2.resize(img, (nw, nh), interpolation=cv2.INTER_CUBIC)
        img = (img - _MEAN) / _STD
        out[j] = np.transpose(img, (2, 0, 1))
    return out


def plan_feature_cache(windows, n_slots: int = INFER_LEN):
    """Slot bookkeeping of the encoder-feature cache for a sequence of windows (lists of source frames): frames the
    current window does not use are evicted (a window only ever reuses frames of its predecessor), frames not cached yet
    get free slots.  Returns, per window, (new_frames, their_slots, slot_of_each_window_position).  Pure host logic
    (the device side is video_depth.FeatureCache); at most `n_slots` frames are live because a window has 32 slots."""
    where, free, plan = {}, list(range(n_slots)), []
    for src in windows:
        need = set(src)
        for f in [f for f in where if f not in need]:
            free.append(where.pop(f))
        missing = sorted(need - where.keys())
        if len(missing) > len(free):
            raise ValueError("feature cache too small for this window")
        slots = [free.pop() for _ in missing]
        where.update(zip(missing, slots))
        plan.append((missing, slots, [where[f] for f in src]))
    return plan


# ------------------------------------------------------------------------------------------------
# bounded device buffers of the long-video driver (pure index logic; the device side is video_depth.FrameUploader /
# video_depth.WindowAligner, the property tests are tests/test_parallel_cpu.py::test_*_ring_*)
# ------------------------------------------------------------------------------------------------
def aligner_ring_len(n_frames: int, ring_segs: int = 4) -> int:
    """Length of the WindowAligner's ring of aligned frames: `ring_segs` segments of 22 frames, fewer for short videos
    (never less than the 44 frames window 0 needs behind the 12-frame shift)."""
    seg = INFER_LEN - OVERLAP
    k = -(-n_frames // seg)
    total = k * seg + OVERLAP
    return seg * min(ring_segs, (total + seg - OVERLAP) // seg)


def aligner_ring_pos(a: int, ring_len: int) -> int:
    """Ring position of aligned frame `a`: shifted by 12 so that window 0 (32 frames) ends, and every later window's 22
    new frames start, on a segment boundary -- a window's new frames and its 8-frame cross-fade tail never wrap."""
    return (a + INFER_LEN - 2 * OVERLAP) % ring_len


def upload_ring_plan(n_needed: int, chunk: int = 64, ring_chunks: int = 4):
    """Device slots and upload chunks of the FrameUploader for `n_needed` frames in upload order.  Returns
    (ring, n_slots, slot_of_position, chunks) with chunks = [(lo, hi)] in upload order.  With the ring on, position 0 (source
    frame 0, read by every window) owns slot 0 and is uploaded alone; positions >= 1 share `ring_chunks * chunk` slots and
    are uploaded in chunks aligned to the ring regions, so chunk m replaces chunk m - ring_chunks."""
    cap = chunk * ring_chunks
    ring = n_needed > 1 + cap
    if not ring:
        return False, n_needed, list(range(n_needed)), [(lo, min(lo + chunk, n_needed)) for lo in range(0, n_needed, chunk)]
    slots = [0] + [1 + (j - 1) % cap for j in range(1, n_needed)]
    chunks = [(0, 1)] + [(lo, min(lo + chunk, n_needed)) for lo in range(1, n_needed, chunk)]
    return True, 1 + cap, slots, chunks


# ------------------------------------------------------------------------------------------------
# streaming (video_depth.DepthStream): temporal context and cache slots of frame t
# ------------------------------------------------------------------------------------------------
STREAM_CONTEXT = INFER_LEN - 1          # L: cached frames a streamed frame attends to (32 positions with itself)


def stream_context(t: int, L: int = STREAM_CONTEXT):
    """Context of streamed frame t: (frame ids, their cache slots, slot frame t is written to).  Frame 0 is a permanent
    anchor at position 0 (as slot 0 of every offline window), followed by the most recent earlier frames:
    ctx(0) = [], ctx(t) = [0] + [max(1, t - L + 1) .. t - 1].  Frame 0 owns slot 0, frames j >= 1 share a ring of L slots
    (slot 1 + (j - 1) % L), so a stream holds at most L + 1 slots however long it runs.  The frame a write replaces
    (t - L) has just left the context, so the write slot is never read in the same step."""
    if t < 0 or L < 1:
        raise ValueError(f"bad stream step t={t} L={L}")

    def slot(j):
        return 0 if j == 0 else 1 + (j - 1) % L

    ids = [] if t == 0 else [0] + list(range(max(1, t - L + 1), t))
    return ids, [slot(j) for j in ids], slot(t)


# ------------------------------------------------------------------------------------------------
# stream groups (video_depth.DepthStreamGroup): handles, pool rows, per-stream steps, buckets and the per-push table
# ------------------------------------------------------------------------------------------------
def stream_buckets(max_streams: int, max_frames=None):
    """Batch sizes a group of at most `max_streams` streams runs at: the powers of two below it, then itself.  With
    `max_frames` (frames per push, >= max_streams; pushes that give a stream several frames), followed by the powers of two
    above max_streams and below max_frames, then max_frames: a push of <= max_streams single frames keeps its bucket."""
    if max_streams < 1:
        raise ValueError(f"a stream group needs max_streams >= 1, got {max_streams}")
    out = [1 << i for i in range(max_streams.bit_length()) if 1 << i < max_streams] + [max_streams]
    if max_frames is None or max_frames == max_streams:
        return out
    if max_frames < max_streams:
        raise ValueError(f"max_frames={max_frames} is below max_streams={max_streams}")
    return out + [1 << i for i in range(max_frames.bit_length()) if max_streams < 1 << i < max_frames] + [max_frames]


class StreamGroupPlan:
    """Host state of a stream group.  Every open stream has a handle (never reused), a pool row (the lowest free one;
    reused after close) and its own step counter t, which only a push that names it advances.  `step(handles)` returns
    the push's bucket and its int32 table rows [bucket] | ctx [bucket, 2 + L] | idx [bucket]: batch row i < len(handles)
    is stream handles[i] with pool row, stream_context(t, L) as {n_ctx, write slot, context slots...} and frame i;
    the pad rows behind it take pool row -1, n_ctx = 0 and frame 0.

    Frame sizes: `step(handles, sizes)` also checks the push's frame sizes [(H0, W0)] (batch-row order).  A stream's
    size is fixed by its first frame (a reopened pool row starts over with a new size); the group's network size
    get_resize_hw(H0, W0, input_size) is fixed by its first push, and every frame must map to it.  Nothing changes
    when a push is rejected.

    Several frames per stream: `step(handles, sizes, counts)` gives stream handles[i] counts[i] (1..L) consecutive
    frames t, t + 1, ... on consecutive batch rows, at most `max_frames` rows in all (default max(max_streams, 16)).  Row
    j of a stream at step t gets stream_context(t + j): a context frame >= t, produced by this push, is entered as
    -1 - (its batch row), an older one as its slot, and the write slot is slot(t + j).  The kernel reads the negative
    entries from the push's own rows and the pool writes follow the attention (vda_attention_temporal_step_causal,
    vda_stream_cache_store), so a slot the push overwrites is still read with its old frame.  Single-frame tables are
    unchanged."""

    def __init__(self, max_streams: int, L: int = STREAM_CONTEXT, input_size: int = 518, max_frames=None):
        max_frames = max(max_streams, 16) if max_frames is None else int(max_frames)
        self.buckets = stream_buckets(max_streams, max_frames)
        self.max_streams, self.max_frames, self.L = max_streams, max_frames, L
        self.stride = 2 + L
        self.input_size = input_size
        self.row, self.t = {}, {}                      # handle -> pool row, handle -> frames pushed so far
        self.size = {}                                 # handle -> (H0, W0) of its first frame
        self.net = None                                # (nh, nw) of the group, fixed by the first push
        self._next = 0

    def open(self) -> int:
        if len(self.row) >= self.max_streams:
            raise ValueError(f"the group already holds its max_streams={self.max_streams} streams")
        used = set(self.row.values())
        h = self._next
        self._next += 1
        self.row[h] = min(r for r in range(self.max_streams) if r not in used)
        self.t[h] = 0
        return h

    def check(self, h) -> None:
        if h not in self.row:
            raise ValueError(f"unknown or closed stream handle {h!r}")

    def close(self, h) -> None:
        self.check(h)
        del self.row[h], self.t[h]
        self.size.pop(h, None)

    def bucket(self, n: int) -> int:
        return next(b for b in self.buckets if b >= n)

    def _check_sizes(self, handles, sizes):
        """The group's network size after this push; ValueError if a frame breaks the size rules."""
        if len(sizes) != len(handles):
            raise ValueError("one frame size per stream of the push")
        net = self.net
        for h, (h0, w0) in zip(handles, sizes):
            if h0 < 1 or w0 < 1:
                raise ValueError(f"empty frame of size {(h0, w0)}")
            if h in self.size and self.size[h] != (h0, w0):
                raise ValueError(f"frame size {(h0, w0)} of stream {h!r} differs from its first frame's {self.size[h]}")
            nhw = get_resize_hw(h0, w0, self.input_size)
            if net is None:
                net = nhw
            elif nhw != net:
                what = "the group's" if self.net is not None else "that of another frame of this push,"
                raise ValueError(f"frame size {(h0, w0)} maps to network size {nhw}, {what} {net}; "
                                 f"streams of other network sizes need a group of their own")
        return net

    def step(self, handles, sizes=None, counts=None):
        """Table of one push of `handles` (distinct open streams, in batch-row order); advances their t by their frame
        counts (`counts`, default one each).  With `sizes`, the frame sizes of the push are checked and recorded too (see
        the class docstring)."""
        for h in handles:
            self.check(h)
        if len(set(handles)) != len(handles):
            raise ValueError("a stream is named more than once in one push")
        if not handles:
            raise ValueError("a push names at least one stream")
        counts = [1] * len(handles) if counts is None else [int(c) for c in counts]
        if len(counts) != len(handles):
            raise ValueError("one frame count per stream of the push")
        for h, c in zip(handles, counts):
            if not 1 <= c <= self.L:
                raise ValueError(f"stream {h!r}: {c} frames in one push; a push gives a stream 1..{self.L} frames")
        if sum(counts) > self.max_frames:
            raise ValueError(f"{sum(counts)} frames in one push, more than the group's max_frames={self.max_frames}")
        if sizes is not None:
            sizes = [(int(a), int(b)) for a, b in sizes]
            self.net = self._check_sizes(handles, sizes)
            for h, hw in zip(handles, sizes):
                self.size[h] = hw
        bk = self.bucket(sum(counts))
        rows = np.full(bk, -1, np.int32)
        ctx = np.zeros((bk, self.stride), np.int32)
        idx = np.zeros(bk, np.int32)
        i = 0
        for h, c in zip(handles, counts):
            t0 = self.t[h]
            for j in range(c):
                ids, slots, write = stream_context(t0 + j, self.L)
                rows[i], idx[i] = self.row[h], i
                ctx[i, 0], ctx[i, 1] = len(slots), write
                # frames of this push (ids >= t0) sit j' = f - t0 rows behind the stream's first row i - j
                ctx[i, 2:2 + len(slots)] = [-1 - (i - j + f - t0) if f >= t0 else s for f, s in zip(ids, slots)]
                i += 1
        for h, c in zip(handles, counts):
            self.t[h] += c
        return bk, np.concatenate([rows, ctx.ravel(), idx])


def split_group_table(table, bk: int, L: int = STREAM_CONTEXT):
    """Views (rows [bk], ctx [bk, 2 + L], idx [bk]) of a StreamGroupPlan table (numpy array or tensor)."""
    s = 2 + L
    return table[:bk], table[bk:bk + bk * s].reshape(bk, s), table[bk + bk * s:bk * (s + 2)]


# include/vda.h vda_frame_desc / vda_out_desc: what the ragged ingest and egress kernels read per batch row
FRAME_DESC = np.dtype([("src", "<u8"), ("pitch", "<i8"), ("H0", "<i4"), ("W0", "<i4")])
OUT_DESC = np.dtype([("dst", "<u8"), ("H0", "<i4"), ("W0", "<i4")])


def group_descriptors(bk: int, frames, dsts):
    """Descriptor arrays of one push: frames = [(device address, row pitch in bytes, H0, W0)] and dsts = [device address
    of the fp32 [H0, W0] output] of the real rows in batch-row order -> (FRAME_DESC [bk], OUT_DESC [bk]).  Pad rows read
    the first row's frame (any valid frame would do) and write nothing (H0 = W0 = 0)."""
    if not 1 <= len(frames) <= bk or len(dsts) != len(frames):
        raise ValueError(f"{len(frames)} frames / {len(dsts)} outputs for a bucket of {bk}")
    fd, od = np.zeros(bk, FRAME_DESC), np.zeros(bk, OUT_DESC)
    for i, ((src, pitch, h0, w0), dst) in enumerate(zip(frames, dsts)):
        if pitch < 3 * w0:
            raise ValueError(f"row pitch {pitch} < 3 * W0 = {3 * w0}")
        fd[i] = (src, pitch, h0, w0)
        od[i] = (dst, h0, w0)
    fd[len(frames):] = fd[0]
    return fd, od


def group_block_layout(bk: int, L: int = STREAM_CONTEXT):
    """Byte ranges (frame descriptors, output descriptors, int32 table) of a push's metadata block: everything a push
    uploads besides frame pixels, in one copy.  The descriptors come first, so every part is aligned to its type."""
    a = bk * FRAME_DESC.itemsize
    b = a + bk * OUT_DESC.itemsize
    return slice(0, a), slice(a, b), slice(b, b + 4 * bk * (L + 4))
