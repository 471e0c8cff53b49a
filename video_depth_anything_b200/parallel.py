"""Window-sharded multi-GPU driver for `infer_video_depth` (one process per GPU, torch.distributed).

The reference has no multi-GPU inference path at all (SURVEY.md §2.1).  Its long-video driver
(video_depth_anything/video_depth.py:166-254) computes K = ceil(N/22) overlapping 32-frame windows whose model
inputs depend on input frames only (closed form in windows.window_source_indices), followed by a cheap
*sequential* scale/shift alignment (:216-252).  So the windows are sharded in contiguous blocks over the ranks with
no data-path collective; what remains is the exchange that feeds the alignment:
  * ranks on one host: the two-phase form (`_infer_two_phase`): halo + anchor all-gather, every rank runs the
    alignment chain itself and downloads its own frames into a shared-memory result returned on rank `dst`;
  * ranks on several hosts: a gather of the raw per-window depths to rank `dst` (NCCL send/recv, 34 MB per
    32x518x518 fp32 window), which then runs the alignment recurrence on its GPU.

Host-side pieces (`partition_windows`, `gather_window_depths`, `two_phase_finalise`) work on CPU tensors with the
gloo backend too; that is how tests/test_parallel_cpu.py covers the N>1 logic without GPUs.
"""
from __future__ import annotations

import os
import time
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist

from .windows import INFER_LEN, INTERP_LEN, KEYFRAMES, OVERLAP, STEP, num_windows, video_frame_shape

KEYFRAME_REF = KEYFRAMES[1]           # slot 12: the frame whose aligned depth becomes the next window's reference


def partition_windows(n_windows: int, world: int) -> List[range]:
    """Contiguous, balanced blocks of window ids per rank (sizes differ by at most one; earlier ranks get the
    extra window).  Contiguity keeps overlapping neighbours on one GPU."""
    if world <= 0:
        raise ValueError("world size must be positive")
    base, extra = divmod(n_windows, world)
    out, start = [], 0
    for r in range(world):
        n = base + (1 if r < extra else 0)
        out.append(range(start, start + n))
        start += n
    return out


def _world(group) -> tuple:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def gather_window_depths(local: torch.Tensor, counts: Sequence[int], dst: int = 0, group=None) -> Optional[torch.Tensor]:
    """Gather per-rank raw window depths `[counts[rank], 32, H, W]` (fp32) to rank `dst`, in rank order (= window
    order for `partition_windows`).  Ranks are padded to the largest count so a single `gather` collective moves
    everything (NCCL: grouped ncclSend/ncclRecv over NVLink).  Returns `[sum(counts), 32, H, W]` on `dst`, None
    elsewhere."""
    rank, world = _world(group)
    if world == 1:
        return local
    assert len(counts) == world and local.shape[0] == counts[rank]
    kmax = max(counts)
    if kmax == 0:
        return local if rank == dst else None
    pad = local
    if local.shape[0] < kmax:
        pad = torch.zeros((kmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        pad[:local.shape[0]].copy_(local)
    pad = pad.contiguous()
    bufs = [torch.empty_like(pad) for _ in range(world)] if rank == dst else None
    dist.gather(pad, bufs, dst=dst, group=group)
    if rank != dst:
        return None
    return torch.cat([bufs[r][:counts[r]] for r in range(world)], dim=0)


def frame_span(k0: int, k1: int, n_windows: int, n_frames: int):
    """Video frames finalised by the rank that owns windows [k0, k1): window k's slots 2..9 are cross-faded with the
    previous window's slots 24..31 and become frames 22k+2..22k+9, its slots 10..31 become frames 22k+10..22k+31, of
    which the last 8 are re-blended (and finalised) by window k+1 (video_depth.py:216-252).  Returns [lo, hi)."""
    if k1 <= k0:
        return 0, 0
    lo = 0 if k0 == 0 else STEP * k0 + 2
    hi = STEP * k1 + 2 if k1 < n_windows else STEP * (n_windows - 1) + INFER_LEN
    return min(lo, n_frames), min(hi, n_frames)


_PINNED_CORES = [False]


def rank_core_slice(rank: int, world: int, cores: Sequence[int]) -> List[int]:
    """Disjoint, contiguous share of `cores` for local rank `rank` of `world` (pure function; tested on CPU).  Every
    rank of one host runs a launching thread, a drain thread, two copy threads and a page-touch thread: on a 24-core
    box with 8 ranks their 40+ runnable threads otherwise migrate over each other's cores and the window phase of
    every rank slows down (round 1: +100 ms of 500)."""
    cores = sorted(cores)
    if world <= 0 or rank < 0 or rank >= world:
        raise ValueError("bad rank / world")
    per = len(cores) // world
    if per < 2:                       # not enough cores to give every rank two: leave the scheduler alone
        return list(cores)
    return cores[rank * per:(rank + 1) * per]


def _pin_cores(rank: int, world: int) -> None:
    """Pin this process (all its threads, present and future) to its rank's core slice; once per process, Linux only,
    VDA_PIN_CORES=0 disables."""
    if _PINNED_CORES[0] or os.environ.get("VDA_PIN_CORES", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return
    _PINNED_CORES[0] = True
    try:
        mine = rank_core_slice(rank, world, sorted(os.sched_getaffinity(0)))
        os.sched_setaffinity(0, mine)
        torch.set_num_threads(max(1, min(torch.get_num_threads(), len(mine))))
    except OSError:
        pass


_SAME_HOST: dict = {}


def _same_host(group) -> bool:
    """All ranks of the group on one host? (one object all-gather per process group, then cached)"""
    key = id(group)
    if key not in _SAME_HOST:
        import socket
        names = [None] * dist.get_world_size(group)
        dist.all_gather_object(names, socket.gethostname(), group=group)
        _SAME_HOST[key] = len(set(names)) == 1
    return _SAME_HOST[key]


class _DeviceKernels:
    """The libvda kernels two_phase_finalise sequences (tests substitute a CPU stand-in with the same methods)."""

    def __init__(self, dev):
        from . import ops
        from .video_depth import make_blend_weights
        self.ops, self.dev = ops, dev
        self.blend_w = make_blend_weights(dev)

    def align_chain(self, anchors, affine):
        table = torch.empty(anchors.shape[0], 2, dtype=torch.float32, device=self.dev)
        scratch = torch.zeros(8 * self.ops.LSQ_MAX_PARTIALS, dtype=torch.float64, device=self.dev)
        return self.ops.align_chain(anchors, table, scratch, affine=affine)

    def affine_clamp_blend(self, x, ss, out, prev=None, blend=False):
        return self.ops.affine_clamp_blend(x, ss, out, prev=prev, blend_w=self.blend_w if blend else None)


def two_phase_finalise(raws: torch.Tensor, counts: Sequence[int], K: int, n: int, affine: bool, kern, emit, group=None,
                       stamp=lambda name: None) -> None:
    """Steps 1-4 of the two-phase driver for this rank's raw window stack `raws` [counts[rank],32,H,W] (windows
    partition_windows(K, world)[rank]); see _infer_two_phase.  `kern` supplies align_chain / affine_clamp_blend (libvda
    on the GPU), `emit(frames [m,H,W], first_video_frame)` receives every finished run of frames exactly once.
    Pure sequencing + torch.distributed: runs on CPU tensors with gloo too (tests/test_parallel_cpu.py)."""
    rank, world = _world(group)
    h0, w0 = raws.shape[-2:]
    dev = raws.device
    parts = partition_windows(K, world)
    k0, k1 = (parts[rank][0], parts[rank][-1] + 1) if counts[rank] else (0, 0)
    # ---- 1. halo: raw slots 24..31 of the window before my first one (no dependency on the table) ----
    reqs, halo = [], None
    owners = [r for r in range(world) if counts[r]]
    if counts[rank] and world > 1:
        i = owners.index(rank)
        if i + 1 < len(owners):
            reqs.append(dist.P2POp(dist.isend, raws[-1, INFER_LEN - INTERP_LEN:].contiguous(), owners[i + 1], group))
        if i > 0:
            halo = torch.empty(INTERP_LEN, h0, w0, dtype=torch.float32, device=dev)
            reqs.append(dist.P2POp(dist.irecv, halo, owners[i - 1], group))
    works = dist.batch_isend_irecv(reqs) if reqs else []
    stamp("halo posted")
    # ---- 2. anchors (slots 0, 1, 12) of every window on every rank ----
    kmax = max(counts)
    mine = torch.zeros(kmax, 3, h0, w0, dtype=torch.float32, device=dev)
    if counts[rank]:
        mine[:counts[rank]].copy_(raws[:, [0, 1, KEYFRAME_REF]])
    if world > 1:
        flat = torch.empty(world * kmax, 3, h0, w0, dtype=torch.float32, device=dev)   # (concatenated form: gloo too)
        dist.all_gather_into_tensor(flat, mine, group=group)
        gathered = flat.view(world, kmax, 3, h0, w0)
    else:
        gathered = mine.unsqueeze(0)
    if all(c == kmax for c in counts):
        anchors = gathered.view(world * kmax, 3, h0, w0)
    else:
        anchors = torch.cat([gathered[r, :counts[r]] for r in range(world)])                  # [K,3,h0,w0]
    stamp("anchors gathered")
    # ---- 3. (scale, shift) of every window: the whole recurrence in one cooperative kernel ----
    table = kern.align_chain(anchors, affine)                                                  # video_depth.py:227-250
    stamp("scale/shift table")
    for w in works:
        w.wait()
    stamp("halo received")
    # ---- 4. my frames: same kernel sequence as WindowAligner.push with the tabulated (scale, shift), in place in
    #      the raw stack (the kernels are elementwise): window j's slots 2..9 are cross-faded with the aligned slots
    #      24..31 of window j-1, slots 10..31 are aligned; its slots [2, 24) are then final video frames
    #      22k+2 .. 22k+23 and leave at once (the last window keeps its slots 24..31 too) ----
    for j in range(k1 - k0):
        k, d = k0 + j, raws[j]
        if k == 0:                                                   # window 0 is copied unclamped (:222-225)
            first = 0
        else:
            ssk = table[k]
            if j > 0:
                prev = raws[j - 1, INFER_LEN - INTERP_LEN:]          # already aligned in place
            elif k == 1:
                prev = halo                                          # window 0's frames: never scaled or clamped
            else:
                prev = kern.affine_clamp_blend(halo, table[k - 1], halo)
            head = d[OVERLAP - INTERP_LEN:OVERLAP]
            kern.affine_clamp_blend(head, ssk, head, prev=prev, blend=True)                        # :234-239
            kern.affine_clamp_blend(d[OVERLAP:], ssk, d[OVERLAP:])                                 # :241-244
            first = OVERLAP - INTERP_LEN
        last = INFER_LEN if k == K - 1 else INFER_LEN - INTERP_LEN
        f0 = STEP * k + first
        f1 = min(STEP * k + last, n)
        if f1 > f0:
            emit(d[first:first + f1 - f0], f0)
    stamp("frames blended")


@torch.no_grad()
def _infer_two_phase(model, frames, target_fps, input_size, device, dst, group, pixel_format="rgb"):
    """Scalable form for ranks on one host (SURVEY.md §8e option 2).  Every rank computes its block of windows
    with no data-path collective; then
      1. the last 8 raw slots of every block travel to the next rank (cross-fade halo; NCCL batch_isend_irecv),
      2. the three anchor frames of every window (slots 0, 1, 12) are all-gathered (NCCL over NVLink, 3.2 MB / window),
      3. every rank walks the sequential (scale, shift) recurrence itself in ONE cooperative kernel
         (ops.align_chain: bit-identical to WindowAligner.push's per-window kernels),
      4. each rank clamps / cross-fades ITS frames in place and downloads them into a POSIX shared-memory array owned
         by rank `dst` -- PCIe, host copies and page faults are spread over all ranks instead of funnelled through one.
    A rank without windows (more ranks than windows) takes part in every collective and downloads nothing.
    The result is bit-identical to the single-GPU `infer_video_depth`."""
    from multiprocessing import resource_tracker, shared_memory
    from .video_depth import HostDrain
    rank, world = _world(group)
    dev = torch.device(device)
    n, h0, w0 = video_frame_shape(frames, pixel_format)
    K = num_windows(n)
    parts = partition_windows(K, world)
    counts = [len(p) for p in parts]
    k0, k1 = (parts[rank][0], parts[rank][-1] + 1) if counts[rank] else (0, 0)
    lo, hi = frame_span(k0, k1, K, n)
    _pin_cores(rank, world)
    # shared result array: created by rank dst, attached by the others, first-touched per slice in the background
    nbytes = n * h0 * w0 * 4
    box = [None]
    if rank == dst:
        shm = shared_memory.SharedMemory(create=True, size=nbytes)
        box[0] = shm.name
    dist.broadcast_object_list(box, src=dst, group=group)
    if rank != dst:
        shm = shared_memory.SharedMemory(name=box[0])
        resource_tracker.unregister(shm._name, "shared_memory")     # rank dst owns the segment's lifetime
    host = np.ndarray((n, h0, w0), dtype=np.float32, buffer=shm.buf)
    trace = os.environ.get("VDA_TRACE_VIDEO") == "1"
    stamps = [("start", time.perf_counter())]

    def stamp(name):
        if trace:
            torch.cuda.synchronize(dev)
            stamps.append((name, time.perf_counter()))

    with torch.cuda.device(dev):
        stamp("shm ready")
        # one drain per rank on the same host: copy threads from this rank's share of the cores (2 at 8 ranks on 24
        # cores, up to 6 with fewer ranks) and 1 low-priority page-touch thread each.  All of a rank's frames leave in
        # the tail (they are final only once the table is known), so the host copies ARE the tail: 1.1 GB per rank took
        # 88 ms with 2 threads at 2 GPUs
        try:
            share = len(os.sched_getaffinity(0))
        except AttributeError:
            share = (os.cpu_count() or 8) // world
        # direct: the GPU writes into the page-locked result rows.  A rank without rows (lo == hi) has nothing to drain:
        # the staged path page-locks nothing and allocates its pinned buffers only on a first send, which never comes
        drain = HostDrain(host, dev, touch=slice(lo, hi), copy_threads=max(2, min(6, share - 1)), touch_threads=1,
                          direct=hi > lo)
        raws = model.infer_video_depth(frames, target_fps, input_size=input_size, device=dev,
                                       window_ids=list(parts[rank]), raw_only=True, pixel_format=pixel_format)   # [k_r,32,h0,w0]
        stamp("windows computed")
        two_phase_finalise(raws, counts, K, n, not model.metric, _DeviceKernels(dev), drain.send, group, stamp)
        drain.finish()
        stamp("downloaded")
        if trace:
            print(f"video trace rank {rank}: drain copied {drain.copied_bytes / 1e6:.0f} MB in {drain.copy_seconds * 1e3:.0f} ms "
                  f"of copy-thread time ({drain.COPY_THREADS} threads), waited {drain.touch_wait_seconds * 1e3:.0f} ms for the "
                  f"page touch, {drain.event_wait_seconds * 1e3:.0f} ms for D2H events; direct D2H "
                  f"{'on' if drain.direct and drain._reg_ok else 'off'} ({drain._reg_note})", flush=True)
    dist.barrier(group=group)
    stamp("barrier")
    if trace:
        print(f"video trace rank {rank}: " + ", ".join(f"{a} +{(t - stamps[0][1]) * 1e3:.0f} ms" for a, t in stamps[1:]), flush=True)
    if rank != dst:
        del host
        drain.unregister_later(close_after=shm)   # page lock released in the background, THEN the attachment is closed
        return None, target_fps
    drain.unregister_later()
    shm.unlink()                      # the name goes away now; the mapping lives as long as the returned array
    _LIVE_SEGMENTS.append(shm)
    return host, target_fps


_LIVE_SEGMENTS: list = []             # shared-memory segments backing arrays handed to the caller


@torch.no_grad()
def infer_video_depth_sharded(model, frames: np.ndarray, target_fps, input_size: int = 518, device=None,
                              dst: int = 0, group=None, pixel_format: str = "rgb"):
    """Drop-in for `model.infer_video_depth(frames, target_fps, input_size, device)` under torchrun: every rank
    passes the same `frames`; rank `dst` returns `(depths float32 [N,H0,W0], target_fps)`, the others `(None,
    target_fps)`.  With one process (no process group) it is exactly `model.infer_video_depth`.  Ranks on one host
    use the two-phase form (_infer_two_phase); ranks on several hosts, which cannot share one result array, send their
    raw window stacks to `dst` in one gather, and `dst` aligns them.  `pixel_format`: as for infer_video_depth (YUV 4:2:0
    frames [N,3*H0/2,W0] from a video decoder)."""
    from .video_depth import WindowAligner
    rank, world = _world(group)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if world == 1:
        return model.infer_video_depth(frames, target_fps, input_size=input_size, device=device, pixel_format=pixel_format)
    if _same_host(group):
        return _infer_two_phase(model, frames, target_fps, input_size, device, dst, group, pixel_format)
    n, h0, w0 = video_frame_shape(frames, pixel_format)
    parts = partition_windows(num_windows(n), world)
    counts = [len(p) for p in parts]
    raw = model.infer_video_depth(frames, target_fps, input_size=input_size, device=device,
                                  window_ids=list(parts[rank]), raw_only=True, pixel_format=pixel_format)   # [k_r,32,h0,w0]
    allraw = gather_window_depths(raw, counts, dst=dst, group=group)
    if rank != dst:
        return None, target_fps
    with torch.cuda.device(allraw.device):
        aligner = WindowAligner(n, h0, w0, allraw.device, "identity" if model.metric else "affine")
        for k in range(allraw.shape[0]):
            aligner.push(allraw[k])
        return aligner.result(), target_fps


__all__ = ["two_phase_finalise", "partition_windows", "gather_window_depths", "frame_span", "rank_core_slice",
           "infer_video_depth_sharded", "INFER_LEN"]
