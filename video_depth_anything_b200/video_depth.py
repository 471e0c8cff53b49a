"""Drop-in `VideoDepthAnything` (reference: video_depth_anything/video_depth.py:36-254 and its metric twin
metric_depth/video_depth_anything/video_depth.py:35-154): same constructor kwargs, same state-dict keys, same
`forward` / `infer_video_depth` signatures and error behaviour, with every operator executed by libvda's
sm_100a kernels.  There is no CPU path: calling `forward` without the CUDA extension or off-GPU raises.

The long-video driver does everything after the upload of the uint8 frames on the device: window gather + cv2-style
INTER_CUBIC resize + normalisation (util/transform.py), per-window forward, output resize, key-frame least-squares
alignment, clamp and 8-frame cross-fade; frames stream in and finished depths stream out through pinned staging
buffers while the windows compute.
"""
from __future__ import annotations

import os
import queue
import threading
import time
from collections import OrderedDict
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import ops
from .engine import Engine
from .synth import ENCODER_DIMS, synth_state_dict
from .windows import (INFER_LEN, INTERP_LEN, KEYFRAMES, OVERLAP, aligner_ring_len, aligner_ring_pos, get_resize_hw,
                      StreamGroupPlan, group_block_layout, group_descriptors, plan_feature_cache, split_group_table,
                      upload_ring_plan, window_source_indices)


VALIDATION_DTYPE = torch.float16     # operand type of the `fp32=True` path (see _ensure_engine)


class VideoDepthAnything(nn.Module):
    def __init__(self, encoder="vitl", features=256, out_channels=(256, 512, 1024, 1024), use_bn=False,
                 use_clstoken=False, num_frames=32, pe="ape", metric=False, dtype=torch.bfloat16, **ignored):
        """`metric=True` selects the metric_depth driver (identity alignment,
        metric_depth/video_depth_anything/video_depth.py:132).  The fork's dead kwargs
        (num_block/out_channel/conv, video_depth.py:47-49) are accepted and ignored."""
        super().__init__()
        if encoder not in ENCODER_DIMS:
            raise KeyError(encoder)                      # reference: KeyError from the model_zoo dict (dinov2.py:399-404)
        if use_bn or use_clstoken or pe != "ape":
            raise NotImplementedError("only the configurations the reference instantiates are supported: "
                                      "use_bn=False, use_clstoken=False, pe='ape' (run.py:40-43)")
        self.encoder = encoder
        self.intermediate_layer_idx = {"vits": [2, 5, 8, 11], "vitl": [4, 11, 17, 23]}
        self.features, self.out_channels, self.num_frames = features, list(out_channels), num_frames
        self.metric = metric
        self.dtype = dtype
        # parameters live in a plain fp32 state dict with the reference's key set; the engine owns packed copies
        self._sd = synth_state_dict(encoder, features, self.out_channels, num_frames, seed=0)
        self._engine: Optional[Engine] = None
        self._engine_val: Optional[Engine] = None        # fp32=True (validation precision), built on first use
        self._device = torch.device("cpu")
        self._stream_one: Optional["DepthStream"] = None   # infer_video_depth_one's stream

    # ---- nn.Module surface -------------------------------------------------------------------
    def state_dict(self, *a, **k):
        return OrderedDict((k_, v.clone()) for k_, v in self._sd.items())

    def load_state_dict(self, sd, strict=True):
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        bad = [k for k in self._sd if k in sd and tuple(sd[k].shape) != tuple(self._sd[k].shape)]
        if bad or (strict and (missing or unexpected)):
            raise RuntimeError(f"Error(s) in loading state_dict for VideoDepthAnything: missing {missing[:5]} "
                               f"unexpected {unexpected[:5]} size mismatch {bad[:5]}")
        for k in self._sd:
            if k in sd:
                self._sd[k] = sd[k].detach().to("cpu", torch.float32).clone()
        for eng in (self._engine, self._engine_val):
            if eng is not None:
                eng.load(self._sd)
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    def to(self, device=None, *a, **k):
        if device is not None and not isinstance(device, torch.dtype):
            dev = torch.device(device)
            if dev.type == "cuda" and dev.index is None:     # 'cuda' and 'cuda:<current>' are the same engine
                dev = torch.device("cuda", torch.cuda.current_device())
            self._device = dev
            if self._device.type == "cuda":
                self._ensure_engine()
        return self

    def cuda(self, device=None):
        return self.to("cuda" if device is None else device)

    def _ensure_engine(self, validation: bool = False) -> Engine:
        """The engine of the model's dtype; `validation=True`: the high-precision engine behind `fp32=True`: fp16
        activations (11 mantissa bits instead of bf16's 8), every weight matrix as a hi | lo pair of fp16 matrices (22
        bits; the GEMMs walk A twice), fp32 accumulation, residual streams, statistics and softmax.  Built lazily, holds
        its own packed copy of the weights, about twice the tensor work of the fast path."""
        if self._device.type != "cuda":
            raise RuntimeError("VideoDepthAnything (B200 engine) has no CPU path: call .to('cuda') first")
        if validation:
            if self._engine_val is None or self._engine_val.device != self._device:
                from . import _lib
                _lib.load()
                with torch.cuda.device(self._device):
                    self._engine_val = Engine(self.encoder, self.features, self.out_channels, VALIDATION_DTYPE,
                                              self._device, self.num_frames, weight_split=True)
                    self._engine_val.load(self._sd)
            return self._engine_val
        if self._engine is None or self._engine.device != self._device:
            from . import _lib
            _lib.load()                                  # raises if libvda.so is missing
            with torch.cuda.device(self._device):
                self._engine = Engine(self.encoder, self.features, self.out_channels, self.dtype, self._device,
                                      self.num_frames)
                self._engine.load(self._sd)
        return self._engine

    # ---- forward -----------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x: torch.Tensor, stages=None, fp32: bool = False) -> torch.Tensor:
        """x [B,T,3,H,W] -> depth [B,T,H,W] fp32, >= 0 (video_depth.py:89-164).  `fp32=True`: validation precision."""
        eng = self._ensure_engine(validation=bool(fp32))
        with torch.cuda.device(self._device):
            return eng.forward(x.to(self._device), stages)

    # ---- long-video driver -------------------------------------------------------------------
    @torch.no_grad()
    def infer_video_depth(self, frames: np.ndarray, target_fps, input_size=518, device="cuda", fp32=False,
                          window_ids: Optional[Sequence[int]] = None, raw_only=False, reuse_features: bool = True):
        """frames uint8 [N,H0,W0,3] -> (float32 [N,H0,W0], target_fps)   (video_depth.py:166-254).

        Everything after the upload of the uint8 frames runs on the device: per-window gather + cv2-style
        INTER_CUBIC resize + normalisation (one kernel), forward (CUDA-graph replay), output resize, key-frame
        least squares, clamp and cross-fade.  Frames are uploaded in chunks through pinned staging buffers while
        earlier windows compute, finished depth frames stream back the same way; the host never touches a pixel.
        `fp32=True` (the reference disables autocast, video_depth.py:203-205 / benchmark/infer/infer.py:58) selects the
        validation-precision engine: fp16 activations, weights as hi | lo fp16 pairs, fp32 accumulation, residual streams,
        statistics and softmax (<= 1e-3 of the fp32 reference on full vitl AND vits windows, tests/test_forward_gpu.py),
        whatever the model's own dtype; the flag is not silently ignored.
        `window_ids` / `raw_only` are the multi-GPU hooks (parallel.py): compute only those windows and return
        the raw, resized per-window depths [len(window_ids),32,H0,W0] on the device, skipping alignment.
        `reuse_features`: the DINOv2 encoder is per-frame and 10 of a window's 32 slots repeat frames of earlier
        windows (:200-201), so each source frame is encoded once and its four tap features are kept on the device
        until no later window needs them (FeatureCache); every kernel is batch-invariant, so the result is
        bit-identical to `reuse_features=False` (tests/test_forward_gpu.py)."""
        if torch.device(device).type != "cuda":
            raise RuntimeError("infer_video_depth: the B200 engine has no CPU path (device must be 'cuda')")
        if frames.ndim != 4 or frames.shape[3] != 3 or frames.dtype != np.uint8:
            raise ValueError("frames must be uint8 [N,H0,W0,3]")
        self.to(device)
        eng = self._ensure_engine(validation=bool(fp32))
        n = frames.shape[0]
        h0, w0 = frames.shape[1:3]
        nh, nw = get_resize_hw(h0, w0, input_size)
        wins = window_source_indices(n)
        ids = list(range(len(wins))) if window_ids is None else list(window_ids)
        with torch.cuda.device(self._device):
            if not ids:
                return torch.empty(0, INFER_LEN, h0, w0, device=self._device) if raw_only else \
                    (np.empty((0, h0, w0), np.float32), target_fps)
            needed = sorted({i for k in ids for i in wins[k]})
            # upload ring: windows in increasing order only; not for the two-phase sharded driver (raw_only), which keeps the
            # raw stacks of all its windows on the device anyway and whose per-rank share shrinks with the rank count
            up = FrameUploader(frames, needed, self._device, ring=not raw_only and all(a < b for a, b in zip(ids, ids[1:])))
            # raw stack allocated once: a fresh 34 MB block per window costs a cudaMalloc each (~10 ms at 518x518)
            raws = torch.empty(len(ids), INFER_LEN, h0, w0, dtype=torch.float32, device=self._device) if raw_only else None
            aligner = None if raw_only else WindowAligner(n, h0, w0, self._device, "identity" if self.metric else "affine")
            cache = FeatureCache(eng, up, nh, nw, [wins[k] for k in ids]) if reuse_features else None
            if cache is None:     # all index lists in one upload (a per-window pageable H2D would sync the stream)
                idx_all = torch.tensor([[up.slot[i] for i in wins[k]] for k in ids], dtype=torch.int32).pin_memory() \
                    .to(self._device, non_blocking=True)
            for j, k in enumerate(ids):
                up.ensure(max(wins[k]))                                      # H2D of the chunks this window needs
                if cache is not None:
                    d = cache.window(j)                                      # [32,nh,nw] fp32 (graph-owned buffer)
                else:
                    x = ops.preprocess_frames(up.dev, idx_all[j], nh, nw).unsqueeze(0)  # [1,32,3,nh,nw]   (:197-201)
                    up.reads_done(wins[k])
                    d = eng.forward(x)[0]                                    # [32,nh,nw] fp32   (:203-205)
                if (nh, nw) != (h0, w0):
                    d = ops.bilinear_f32(d, h0, w0, out=raws[j] if raw_only else None)   # video_depth.py:208
                elif raw_only:
                    raws[j].copy_(d)
                if not raw_only:
                    aligner.push(d)
            up.close()
            if raw_only:
                return raws
            return aligner.result(), target_fps

    # ---- streaming -----------------------------------------------------------------------------
    def stream(self, input_size: int = 518, fp32: bool = False, max_frames: int = 16) -> "DepthStream":
        """Open a depth stream on this model's device: `push` one uint8 frame, get its depth back at once, or push a stack
        of up to `max_frames` consecutive frames and get their depths as one step.  Each frame attends to frame 0 and the
        30 frames before it (DepthStream).  Streams are independent of each other and of `forward` /
        `infer_video_depth`; `fp32=True` selects the validation-precision engine as in infer_video_depth."""
        return DepthStream(self, self._ensure_engine(validation=bool(fp32)), input_size, max_frames)

    def stream_group(self, max_streams: int = 8, input_size: int = 518, fp32: bool = False,
                     max_frames: Optional[int] = None) -> "DepthStreamGroup":
        """Open a group of up to `max_streams` depth streams (several cameras) on this model's device: each `push` takes
        one frame, or a stack of consecutive frames, of any subset of the group's open streams and runs them as one
        batched step of at most `max_frames` frames (default max(max_streams, 16); DepthStreamGroup).  Every stream
        behaves as a DepthStream of its own; `fp32=True` selects the validation-precision engine."""
        return DepthStreamGroup(self, self._ensure_engine(validation=bool(fp32)), max_streams, input_size, max_frames)

    @torch.no_grad()
    def infer_video_depth_one(self, frame, input_size: int = 518, device="cuda", fp32: bool = False, to_host: bool = True):
        """Depth of the next frame of the model's own stream (the name of the upstream project's streaming entry
        point): frame uint8 [H0,W0,3] (numpy array or CUDA tensor) -> float32 [H0,W0] (numpy array, or with
        `to_host=False` a CUDA tensor; DepthStream.push).  The stream is opened on the first call and reopened (its
        temporal context starts over) when `input_size`, `fp32` or the device change or new weights were loaded."""
        if torch.device(device).type != "cuda":
            raise RuntimeError("infer_video_depth_one: the B200 engine has no CPU path (device must be 'cuda')")
        if getattr(frame, "ndim", None) != 3:
            raise ValueError("infer_video_depth_one takes one frame uint8 [H0,W0,3]; push stacks through model.stream()")
        self.to(device)
        eng = self._ensure_engine(validation=bool(fp32))
        st = self._stream_one
        if st is None or st.engine is not eng or st.input_size != input_size or st.generation != eng.generation:
            if st is not None:
                st.close()
            st = self._stream_one = self.stream(input_size, fp32)
        return st.push(frame, to_host)


class DepthStreamGroup:
    """Streaming inference for many live streams (cameras) on one model: every push runs the frames of all the streams
    it names as one batched step.

    Each stream follows DepthStream's semantics exactly, with its own step counter t and its own temporal context
    (windows.stream_context over its own row of a pooled k'|v' cache).  A push names any subset of the open streams,
    each at most once; a stream left out does not advance.  The batch is padded up to a bucket (the powers of two below
    `max_streams`, then `max_streams`; windows.stream_buckets): pad rows read the first row's frame, take pool row -1,
    which reads and writes no pool byte, and write no output.  One CUDA graph per bucket, captured on first use and
    owned by the group (the engine's forward / video graphs neither evict nor are evicted by them).

    Sizes: one network size per group, fixed by the first push (windows.get_resize_hw of its frames); every stream has
    its own frame size, fixed by its first frame (a closed stream's pool row starts over with a new size).  So 1280x720
    and 1920x1080 cameras (both 518x924) share a group; a 640x480 camera (518x686) needs a group of its own.

    Frames are uint8 RGB [H0, W0, 3], as numpy arrays or as CUDA tensors on the group's device (rows may be pitched:
    stride (pitch, 3, 1)), mixed freely.  Every frame-dependent address and size of a push is in a per-row descriptor
    block in device memory (windows.group_descriptors), so the graphs replay whatever mix of sizes and buffers later
    pushes bring.  A push is one H2D of the host frames (packed in a pinned arena, read from a device arena), one H2D
    of the descriptors and the int32 rows | ctx | idx table, a replay, and with to_host one D2H of the depths (packed in
    a device arena).  CUDA frames are read in place.  The arenas grow to the largest push seen; growing captures nothing.

    Device memory: the pool holds max_streams x (L + 1) = 32 frame slots per temporal-attention block, allocated at the
    first push: 903 MB per stream for ViT-L at 518x518 (214 MB for ViT-S), plus one graph's activations per bucket used
    and the arenas.

    Several frames per stream: a push may give a stream a stack of k consecutive frames uint8 [k, H0, W0, 3] (1 <= k <=
    L = num_frames - 1; a CUDA stack may have any frame stride, and its rows may be pitched), for at most `max_frames`
    frames in the push.  The stream advances by k and gets [k, H0, W0] back: the depths the k one-frame pushes would have
    returned, in order (bit-identical with fp32=True; in the default mode the encoder's LayerNorm fold depends on the
    bucket, as for groups).  Each frame takes a batch row of its own, and the buckets continue above max_streams up to
    max_frames (windows.stream_buckets).  A push that gives any stream k > 1 frames replays the bucket's causal graph
    (captured once per bucket, kept in `causal_graphs`): its temporal attention reads a frame's newer context from the
    push's own rows and writes the cache afterwards (Engine.stream_group_step(causal=True)); any other push replays
    today's graph."""

    def __init__(self, model: VideoDepthAnything, engine: Engine, max_streams: int = 8, input_size: int = 518,
                 max_frames: Optional[int] = None):
        self.engine, self.input_size = engine, int(input_size)
        self.device = engine.device
        self.generation = engine.generation
        L = model.num_frames - 1
        if not 1 <= L <= INFER_LEN - 1:
            raise ValueError(f"streaming needs num_frames in 2..{INFER_LEN}, got {model.num_frames}")
        self.plan = StreamGroupPlan(int(max_streams), L, self.input_size, max_frames)
        self.max_streams, self.max_frames = self.plan.max_streams, self.plan.max_frames
        self.pool = None
        self.graphs = {}                             # bucket -> captured step (Engine.run_graphed)
        self.causal_graphs = {}                      # bucket -> captured causal step (pushes with stacks)
        self.arenas = {}                             # name -> buffer, grown on demand (_arena)
        self.closed = False

    def open(self) -> int:
        """A new stream starting at t = 0; returns its handle.  ValueError beyond `max_streams` open streams."""
        if self.closed:
            raise RuntimeError("open on a closed DepthStreamGroup")
        return self.plan.open()

    def close_stream(self, handle: int) -> None:
        """Close one stream; its pool row is free for a later open (which starts over at t = 0)."""
        self.plan.close(handle)

    def _alloc(self) -> None:
        eng, S, L = self.engine, self.max_streams, self.plan.L
        self.nh, self.nw = self.plan.net
        nbytes = group_block_layout(self.plan.buckets[-1], L)[2].stop
        with torch.cuda.device(self.device):
            self.pool = eng.stream_pool(S, self.nh // 14, self.nw // 14, L + 1)
            self.meta_dev = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self.meta_host = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()

    def _arena(self, name: str, n: int, dtype, pinned: bool) -> torch.Tensor:
        """Buffer `name` with at least n elements; regrown (in 2 MiB steps) only when a push needs more."""
        t = self.arenas.get(name)
        if t is None or t.numel() < n:
            n = -(-max(n, 1) * dtype.itemsize // (2 << 20)) * (2 << 20) // dtype.itemsize
            t = torch.empty(n, dtype=dtype).pin_memory() if pinned else torch.empty(n, dtype=dtype, device=self.device)
            self.arenas[name] = t
        return t

    def _step(self, bk: int, causal: bool = False) -> None:
        eng = self.engine
        fs, os_, ts = group_block_layout(bk, self.plan.L)
        rows, ctx, _ = split_group_table(self.meta_dev[ts].view(torch.int32), bk, self.plan.L)
        inputs = [self.meta_dev[fs], self.meta_dev[os_], rows, ctx]

        def fn(frame_desc, out_desc, rows, ctx):
            return eng.stream_group_step(frame_desc, out_desc, rows, ctx, self.pool, self.nh, self.nw, causal)
        if eng.use_graphs and ops.PROFILE is None:
            return eng.run_graphed(self.causal_graphs if causal else self.graphs, bk, fn, inputs, adopt=True)
        return fn(*inputs)

    def _check_frame(self, f):
        """(k, H0, W0) of a frame (k = None) or of a stack of k frames; ValueError if it is neither."""
        if isinstance(f, torch.Tensor):
            if not f.is_cuda or f.device != self.device:
                raise ValueError(f"a tensor frame must be a CUDA tensor on the group's device {self.device}, got {f.device}")
            if f.dtype != torch.uint8 or f.dim() not in (3, 4) or f.shape[-1] != 3:
                raise ValueError(f"a CUDA frame must be a uint8 tensor [H0,W0,3] (or a stack [k,H0,W0,3]), "
                                 f"got {f.dtype} {tuple(f.shape)}")
            if f.stride(-1) != 1 or f.stride(-2) != 3 or f.stride(-3) < 3 * f.shape[-2]:
                raise ValueError(f"a CUDA frame's pixels must be contiguous, stride (pitch >= 3 * W0, 3, 1), "
                                 f"got {f.stride()}")
        elif not isinstance(f, np.ndarray) or f.ndim not in (3, 4) or f.shape[-1] != 3 or f.dtype != np.uint8:
            raise ValueError("a frame must be a uint8 numpy array [H0,W0,3] or a uint8 CUDA tensor [H0,W0,3] "
                             "(or a stack [k,H0,W0,3] of either)")
        k = int(f.shape[0]) if f.ndim == 4 else None
        if k is not None and not 1 <= k <= self.plan.L:
            raise ValueError(f"a stack holds 1..{self.plan.L} frames, got {k}")
        return k, int(f.shape[-3]), int(f.shape[-2])

    @torch.no_grad()
    def push(self, frames, to_host: bool = True) -> dict:
        """frames: {handle: uint8 RGB [H0,W0,3] numpy array or CUDA tensor, or a stack [k,H0,W0,3] of k consecutive
        frames} (or (handle, frame) pairs) -> {handle: depth [H0,W0] (>= 0), or [k,H0,W0] for a stack}: fresh float32
        numpy arrays, or with `to_host=False` fresh float32 CUDA tensors on the group's device (no device-to-host copy).
        Returns after the step has finished, so the caller may reuse its frame buffers at once."""
        if self.closed:
            raise RuntimeError("push on a closed DepthStreamGroup")
        if self.engine.generation != self.generation or not self.engine.loaded:
            raise RuntimeError("the model's weights changed since this stream group was opened; open a new one")
        items = list(frames.items()) if isinstance(frames, dict) else list(frames)
        shapes = [self._check_frame(f) for _, f in items]
        sizes = [(h0, w0) for _, h0, w0 in shapes]
        counts = [k or 1 for k, _, _ in shapes]
        handles = [h for h, _ in items]
        # ValueError: empty push, unknown / closed / repeated handle, a frame size the group cannot take, too many frames
        bk, table = self.plan.step(handles, sizes, counts)
        if self.pool is None:
            self._alloc()
        # batch rows: (item, frame of the item, H0, W0), the frames of a stack on consecutive rows
        rows = [(i, j, h0, w0) for i, (h0, w0) in enumerate(sizes) for j in range(counts[i])]
        host = [r for r, (i, _, _, _) in enumerate(rows) if isinstance(items[i][1], np.ndarray)]
        packed = np.cumsum([0] + [3 * rows[r][2] * rows[r][3] for r in host]).tolist()      # host frames, packed
        in_off, in_bytes = dict(zip(host, packed)), packed[-1]
        out_off = np.cumsum([0] + [h0 * w0 for _, _, h0, w0 in rows]).tolist()             # depths, packed
        out_elems = out_off[-1]
        first = np.cumsum([0] + counts).tolist()                                           # first batch row of item i
        with torch.cuda.device(self.device):
            if host:
                in_host = self._arena("in_host", in_bytes, torch.uint8, True)
                in_dev = self._arena("in_dev", in_bytes, torch.uint8, False)
                ih = in_host.numpy()
                for r in host:
                    i, j, h0, w0 = rows[r]
                    f = items[i][1]
                    np.copyto(ih[in_off[r]:in_off[r] + 3 * h0 * w0].reshape(h0, w0, 3), f[j] if f.ndim == 4 else f)
            srcs = []
            for r, (i, j, h0, w0) in enumerate(rows):
                f = items[i][1]
                if isinstance(f, torch.Tensor):
                    srcs.append((f[j].data_ptr(), f.stride(1), h0, w0) if f.dim() == 4 else (f.data_ptr(), f.stride(0), h0, w0))
                else:
                    srcs.append((in_dev.data_ptr() + in_off[r], 3 * w0, h0, w0))
            if to_host:
                out_dev = self._arena("out_dev", out_elems, torch.float32, False)
                dsts = [out_dev.data_ptr() + 4 * o for o in out_off[:-1]]
            else:
                # the kernel writes straight into the returned tensors (one allocation each from the caching allocator):
                # no device-to-device pass over the depths, and no arena a caller's tensor could alias
                outs = [torch.empty(*((k,) if k else ()), h0, w0, dtype=torch.float32, device=self.device)
                        for k, h0, w0 in shapes]
                dsts = [outs[i].data_ptr() + 4 * j * h0 * w0 for i, j, h0, w0 in rows]
            fd, od = group_descriptors(bk, srcs, dsts)
            fs, os_, ts = group_block_layout(bk, self.plan.L)
            mh = self.meta_host.numpy()
            mh[fs], mh[os_], mh[ts] = fd.view(np.uint8), od.view(np.uint8), table.view(np.uint8)
            if host:
                in_dev[:in_bytes].copy_(in_host[:in_bytes], non_blocking=True)
            self.meta_dev[:ts.stop].copy_(self.meta_host[:ts.stop], non_blocking=True)
            causal = max(counts) > 1
            if causal and bk not in self.causal_graphs and self.engine.use_graphs and ops.PROFILE is None:
                # capturing runs the step twice (warm-up, then the replay), and a causal step is not idempotent: its
                # cache store overwrites slots its earlier rows read.  So the capture runs with every row a pad row
                # (pool row -1: no pool byte read or written), then the push's own table replays the new graph.
                self.meta_dev[ts.start:ts.start + 4 * bk].fill_(255)
                self._step(bk, causal)
                self.meta_dev[:ts.stop].copy_(self.meta_host[:ts.stop], non_blocking=True)
            self._step(bk, causal)
            if to_host:
                out_host = self._arena("out_host", out_elems, torch.float32, True)
                out_host[:out_elems].copy_(out_dev[:out_elems], non_blocking=True)
            torch.cuda.current_stream().synchronize()   # (also: the pinned arenas are free for the next push)
        if not to_host:
            return dict(zip(handles, outs))
        oh = out_host.numpy()
        return {h: oh[out_off[first[i]]:out_off[first[i + 1]]].reshape(((k,) if k else ()) + sizes[i]).copy()
                for i, (h, (k, _, _)) in enumerate(zip(handles, shapes))}

    def close(self) -> None:
        """Release the group's graphs, pool and arenas (also done when the object is collected)."""
        self.graphs = {}
        self.causal_graphs = {}
        self.pool = None
        self.arenas = {}
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:                                # noqa: BLE001  (interpreter shutdown)
            pass


class DepthStream:
    """Streaming inference: one frame in, its depth out, with a cached temporal context.

    Frame t is preprocessed as in infer_video_depth, encoded and run through the head with T = 1; in each of the 8
    temporal-attention blocks its query attends to itself and to the context frames ctx(t) = [0] + the most recent
    earlier frames (at most L = num_frames - 1 = 31 of them, windows.stream_context), frame 0 at position 0 and the
    current frame last, each with the positional encoding of its position in that sequence.  So for t <= 31 the result is
    the windowed forward of frames 0..t under a causal temporal mask.  (The upstream streaming script pads the early
    context with copies of frame 0 instead; that breaks this equivalence and is not done here.)  No scale / shift
    alignment between frames.

    A cached frame is kept as its k'|v' = LayerNorm output @ [W_k | W_v]^T rows, without the positional encoding, whose
    share is added by the step kernel at the frame's current position: a step never re-projects old frames.  Device
    memory is bounded: L + 1 cache slots per block.  A DepthStream is a DepthStreamGroup of one stream: the whole step
    (preprocess, encoder, head, resize) is one CUDA graph; a push is one H2D of the frame (none for a CUDA frame) and of
    the context, a replay and one D2H of the depth (none with to_host=False).  Frame size (and so the network size) is
    fixed by the first frame.

    A push may also be a stack of k <= max_frames consecutive frames [k, H0, W0, 3] (k <= 31), e.g. when replaying a
    recording or draining a backlog: one batched step of k rows, returning the [k, H0, W0] depths the k one-frame pushes
    would have returned (DepthStreamGroup)."""

    def __init__(self, model: VideoDepthAnything, engine: Engine, input_size: int = 518, max_frames: int = 16):
        self.group = DepthStreamGroup(model, engine, 1, input_size, max_frames)
        self.engine, self.input_size, self.generation = engine, self.group.input_size, self.group.generation
        self.handle = self.group.open()

    def push(self, frame, to_host: bool = True):
        """frame uint8 RGB [H0,W0,3] (numpy array, or CUDA tensor on the stream's device, rows may be pitched) -> its
        depth float32 [H0,W0] (>= 0): a fresh numpy array on every call, or with `to_host=False` a fresh CUDA tensor.
        A stack [k,H0,W0,3] of the next k frames gives their depths [k,H0,W0]."""
        return self.group.push([(self.handle, frame)], to_host)[self.handle]

    def close(self) -> None:
        """Release the stream's graph and cache (also done when the object is collected)."""
        self.group.close()


class FeatureCache:
    """Per-frame encoder features shared by overlapping windows.  Window k's slots are source frames
    [0, 22k-10, 22k+2 .. 22k+31] (windows.window_source_indices): frame 0, one key frame and 8 overlap frames were
    already encoded for window k-1, and padded tails repeat the last frame, so only the frames not seen yet go
    through preprocessing + the encoder (22 of 32 in steady state = 31 % fewer encoder FLOPs).  Features live in
    32 device slots per tap ([slot, P, D] 16-bit); frames the current window does not use are evicted (later
    windows only ever reuse frames of their predecessor)."""

    def __init__(self, eng: Engine, up: "FrameUploader", nh: int, nw: int, windows: Sequence[Sequence[int]]):
        self.eng, self.up, self.nh, self.nw = eng, up, nh, nw
        self.hp, self.wp = nh // 14, nw // 14
        P = self.hp * self.wp
        self.store = [torch.empty(INFER_LEN, P, eng.D, dtype=eng.hdtype, device=eng.device) for _ in range(4)]   # taps: head operand type
        self.encoded = 0                                  # frames that went through the encoder (for reporting)
        # The slot bookkeeping depends on the window list only, so the index lists of ALL windows are planned on the
        # host now and uploaded once: per window [uploaded-frame index of each new frame | its cache slot | slot of
        # each of the 32 window positions].  (A per-window pageable H2D copy synchronises the stream and drains the
        # GPU between windows.)
        table = np.zeros((max(len(windows), 1), 3 * INFER_LEN), dtype=np.int32)
        self.n_new, self.missing = [], []
        for j, (missing, slots, positions) in enumerate(plan_feature_cache(windows)):
            n = len(missing)
            self.n_new.append(n)
            self.missing.append(list(missing))
            table[j, :n] = [up.slot[f] for f in missing]
            table[j, INFER_LEN:INFER_LEN + n] = slots
            table[j, 2 * INFER_LEN:] = positions
        self.table = torch.from_numpy(table).pin_memory().to(eng.device, non_blocking=True)

    def window(self, j: int) -> torch.Tensor:
        """Depths [32, nh, nw] of the j-th planned window (a graph-owned buffer: consume before the next call)."""
        eng, P, n = self.eng, self.hp * self.wp, self.n_new[j]
        row = self.table[j]
        if n:
            x = ops.preprocess_frames(self.up.dev, row[:n], self.nh, self.nw)          # [n,3,nh,nw]   (:197-198)
            self.up.reads_done(self.missing[j])
            taps = eng.encode_frames(x)
            for i in range(4):
                ops.copy_frames(taps[i].view(n, P, eng.D), None, self.store[i], row[INFER_LEN:INFER_LEN + n], n)
            self.encoded += n
        head_in = eng.head_static_inputs(INFER_LEN, self.hp, self.wp)
        for i in range(4):
            ops.copy_frames(self.store[i], row[2 * INFER_LEN:], head_in[i].view(INFER_LEN, P, eng.D), None, INFER_LEN)
        return eng.head_frames(head_in, INFER_LEN, self.hp, self.wp)


_PINNED: dict = {}
_PINNED_LOCK = threading.Lock()


def _pinned_acquire(key, count: int, shape, dtype):
    """Pinned host staging buffers, cached across calls (cudaHostAlloc of a few hundred MB costs tens of ms and
    synchronises the device; a serving loop calls infer_video_depth once per video).  One cached set per (purpose,
    frame size); a caller that finds the set taken by another live object (concurrent calls from several threads)
    gets a private allocation.  Returns (buffers, token); hand the token back with _pinned_release."""
    with _PINNED_LOCK:
        ent = _PINNED.get(key)
        if ent is not None and not ent["busy"] and len(ent["bufs"]) >= count and tuple(ent["bufs"][0].shape) == tuple(shape):
            ent["busy"] = True
            return ent["bufs"][:count], key
        if ent is not None and ent["busy"]:
            return [torch.empty(*shape, dtype=dtype).pin_memory() for _ in range(count)], None
        bufs = [torch.empty(*shape, dtype=dtype).pin_memory() for _ in range(count)]
        _PINNED[key] = {"bufs": bufs, "busy": True}
        return bufs, key


def _pinned_release(token) -> None:
    if token is not None:
        with _PINNED_LOCK:
            if token in _PINNED:
                _PINNED[token]["busy"] = False


class FrameUploader:
    """Chunked, asynchronous H2D of the uint8 frames a rank needs (pinned double buffer, copy stream); windows wait
    only for the chunks that hold their frames, so the upload overlaps the compute of earlier windows.

    Device memory is bounded: the first needed frame (source frame 0: slot 0 of every window, video_depth.py:200) keeps a
    slot of its own, all others go through a ring of RING_CHUNKS x CHUNK frames.  A window reads frame 0 and frames inside
    a span of 42 consecutive source frames, windows are visited in increasing order and a chunk is only uploaded when the
    current window needs it, so the chunk a new upload replaces (RING_CHUNKS chunks older) is never read again; the copy
    waits for the kernels that read it (`reads_done`).  `ring=False` (windows not in increasing order): everything stays."""

    CHUNK = 64
    RING_CHUNKS = 4

    def __init__(self, frames: np.ndarray, needed: List[int], device, ring: bool = True):
        self.frames, self.needed, self.device = frames, needed, device
        self.pos = {i: j for j, i in enumerate(needed)}            # position in upload order
        self.ring, n_slots, slots, self.chunks = upload_ring_plan(len(needed), self.CHUNK, self.RING_CHUNKS if ring else 1 << 30)
        self.slot = {i: slots[j] for i, j in self.pos.items()}     # device slot of every needed source frame
        h0, w0 = frames.shape[1:3]
        self.dev = torch.empty(n_slots, h0, w0, 3, dtype=torch.uint8, device=device)
        self.stage, self._stage_token = _pinned_acquire(("upload", h0, w0), 2, (self.CHUNK, h0, w0, 3), torch.uint8)
        self.stage_free = [None, None]           # event: staging buffer consumed by its H2D copy
        self.read_ev = [None] * (self.RING_CHUNKS if self.ring else 0)   # event: the kernels that read the chunk in this ring region are queued
        self.stream = torch.cuda.Stream(device=device)
        # `dev` comes from the caching allocator of the compute stream and may be a block that kernels of an earlier call
        # (still queued on that stream: the raw_only path returns without synchronising) are yet to read: the
        # copy stream starts after everything issued so far, and the block is not recycled before the copies are done
        self.stream.wait_stream(torch.cuda.current_stream(device))
        self.dev.record_stream(self.stream)
        self.uploaded = 0                        # number of `needed` entries issued so far
        self.chunk_no = 0

    def _region(self, p: int) -> int:
        """Ring region of upload position p >= 1."""
        return ((p - 1) // self.CHUNK) % self.RING_CHUNKS

    def ensure(self, max_frame: int) -> None:
        """Issue uploads until source frame `max_frame` is covered, then make the current stream wait for them."""
        target = self.pos[max_frame] + 1
        last_ev = None
        while self.uploaded < target:
            lo, hi = self.chunks[self.chunk_no]
            b = self.chunk_no & 1
            if self.stage_free[b] is not None:
                self.stage_free[b].synchronize()
            src_idx = self.needed[lo:hi]
            st = self.stage[b][:hi - lo]
            if src_idx[-1] - src_idx[0] == hi - lo - 1:                      # contiguous run: plain slice copy
                np.copyto(st.numpy(), self.frames[src_idx[0]:src_idx[-1] + 1])
            else:
                np.take(self.frames, src_idx, axis=0, out=st.numpy())
            d0 = self.slot[src_idx[0]]
            with torch.cuda.stream(self.stream):
                if self.ring and lo > 0 and self.read_ev[self._region(lo)] is not None:
                    self.stream.wait_event(self.read_ev[self._region(lo)])   # readers of the chunk this one replaces
                self.dev[d0:d0 + hi - lo].copy_(st, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.stream)
            self.stage_free[b] = ev
            last_ev = ev
            self.uploaded = hi
            self.chunk_no += 1
        if last_ev is not None:
            torch.cuda.current_stream().wait_event(last_ev)

    def reads_done(self, frame_ids: Sequence[int]) -> None:
        """The kernels that read these source frames from `dev` have been queued on the current stream."""
        if not self.ring:
            return
        regions = {self._region(self.pos[f]) for f in frame_ids if self.pos[f] > 0}
        if regions:
            ev = torch.cuda.Event()
            ev.record()
            for r in regions:
                self.read_ev[r] = ev

    def close(self) -> None:
        """All uploads have been issued: give the staging buffers back once their H2D copies are done."""
        for ev in self.stage_free:
            if ev is not None:
                ev.synchronize()
        _pinned_release(self._stage_token)
        self._stage_token = None


class HostDrain:
    """Device -> host streaming of finished fp32 frames: D2H into pinned staging buffers on a copy stream, and a drain
    thread (numpy copies release the GIL; every batch is split over a small pool) moves them into the result array,
    so the launching thread never waits for a host memcpy.  The result array is first-touched in the background (one
    write per page): the page faults of a fresh multi-GB allocation otherwise sit inside the drain copies and divide
    their bandwidth by ~5 (tools/microbench/host_touch.py)."""

    STAGES = 4
    COPY_THREADS = 6

    def __init__(self, host: np.ndarray, device, touch: Optional[slice] = None, copy_threads: Optional[int] = None,
                 touch_threads: Optional[int] = None, direct: bool = False):
        """`copy_threads` / `touch_threads`: host threads of the drain copies / of the background first-touch (default
        6 / 6 for a single process; the sharded driver runs one HostDrain per rank on the same host, see parallel.py).
        `direct`: page-lock the `touch` slice of the result array in the background (cudaHostRegister, started 50 ms
        after construction so that the first windows are already queued on the GPU) and let the GPU write finished
        frames straight into it -- no pinned staging, no host copy.  For the two-phase sharded driver, whose frames all
        leave in the tail: the staging -> result copies of all ranks share the host's memory bandwidth (measured: 2.2 GB in
        ~55 ms whatever the rank count).  Falls back to the staged path if the registration fails."""
        self.host, self.device = host, device
        self.direct, self._reg_ok, self._reg_done, self._reg_note = direct, False, threading.Event(), ""
        self._reg_slice = touch if touch is not None else slice(0, host.shape[0])
        if direct:
            threading.Thread(target=self._register, daemon=True).start()
            touch_threads = 1
            touch = slice(0, 0)                   # the registration faults the pages in itself
        self.COPY_THREADS = copy_threads or self.COPY_THREADS
        touch_threads = touch_threads or self.COPY_THREADS
        h0, w0 = host.shape[1:]
        self.stage, self._stage_token, self._stage_shape = None, None, (INFER_LEN, h0, w0)   # staging: on first staged send
        self.stage_free = [threading.Event() for _ in range(self.STAGES)]
        for e in self.stage_free:
            e.set()
        self.copy_stream = torch.cuda.Stream(device=device)
        self.batch_no = 0
        self.jobs: "queue.Queue" = queue.Queue()
        self.error = None
        self.copied_bytes, self.copy_seconds, self.touch_wait_seconds, self.event_wait_seconds = 0, 0.0, 0.0, 0.0   # trace
        self.pool = ThreadPoolExecutor(self.COPY_THREADS)
        flat = (host if touch is None else host[touch]).reshape(-1)
        cuts = np.linspace(0, flat.size, touch_threads + 1).astype(np.int64)
        self.touch_pool = ThreadPoolExecutor(touch_threads)

        def first_touch(a):
            try:     # background work: stay out of the way of the launching thread (Linux: per-thread nice value)
                os.setpriority(os.PRIO_PROCESS, threading.get_native_id(), 10)
            except (OSError, AttributeError):
                pass
            a[::1024].fill(0)

        self.touch = [self.touch_pool.submit(first_touch, flat[cuts[i]:cuts[i + 1]]) for i in range(touch_threads)]
        self.drainer = threading.Thread(target=self._drain_loop, daemon=True)
        self.drainer.start()

    def _register(self) -> None:
        try:
            torch.cuda.set_device(self.device)   # a new thread starts on device 0: register in THIS rank's context
            time.sleep(0.05)
            rt = torch.cuda.cudart()
            region = self.host[self._reg_slice]
            if region.size:
                ptr = region.ctypes.data
                rc = int(rt.cudaHostRegister(ptr, region.nbytes, 0))
                if rc == 712:                    # cudaErrorHostMemoryAlreadyRegistered: a stale entry for this address range
                    rt.cudaHostUnregister(ptr)
                    rc = int(rt.cudaHostRegister(ptr, region.nbytes, 0))
                self._reg_note = f"cudaHostRegister rc={rc}"
                if rc == 0:
                    self._host_t = torch.from_numpy(region)
                    self._reg_ok = True
        except Exception as exc:                 # noqa: BLE001  (no registration: staged copies)
            self._reg_ok = False
            self._reg_note = f"{type(exc).__name__}: {exc}"
        finally:
            if not self._reg_ok:
                # staged path after all: get its pinned buffers and fault the result pages in now, in the background,
                # not in the tail (first-touch page faults divide the copy bandwidth by 5)
                try:
                    self.stage, self._stage_token = _pinned_acquire(("drain",) + self._stage_shape[1:], self.STAGES,
                                                                    self._stage_shape, torch.float32)
                    self.host[self._reg_slice].reshape(-1)[::1024].fill(0)
                except Exception:                # noqa: BLE001
                    pass
            self._reg_done.set()

    def unregister_later(self, close_after=None) -> None:
        """Release the page lock in the background, half a second from now: the data is in place, but
        cudaHostUnregister holds the context lock for tens of ms per 100 MB -- right behind finish() it delayed the
        caller's next CUDA call (a dist.barrier waited 36 ms), and run back to back with the next call's registration it
        stalled that call's launches by 0.5 s.  The array is kept alive until then, and `close_after` (the rank's
        SharedMemory attachment) is closed only afterwards: NumPy does not hold a buffer export, so closing the mapping
        while it is page-locked leaves a stale registration behind that the next mapping at the same address trips
        over (cudaErrorHostMemoryAlreadyRegistered)."""
        if not (self.direct and self._reg_ok):
            if close_after is not None:
                try:
                    close_after.close()
                except BufferError:
                    pass
            return
        region = self.host[self._reg_slice]
        ptr, keep_ref, dev = region.ctypes.data, [self.host, close_after], self.device
        self.host = None

        def work():
            try:
                torch.cuda.set_device(dev)
                time.sleep(0.5)
                torch.cuda.cudart().cudaHostUnregister(ptr)
            finally:
                shm = keep_ref[1]
                del keep_ref[:]
                if shm is not None:
                    try:
                        shm.close()
                    except BufferError:
                        pass
        threading.Thread(target=work, daemon=True).start()

    def _drain_loop(self) -> None:
        while True:
            job = self.jobs.get()
            if job is None:
                self.jobs.task_done()
                return
            ev, b, lo, hi = job
            try:
                t0 = time.perf_counter()
                ev.synchronize()
                t1 = time.perf_counter()
                if self.touch:                   # a late page-touch write would zero a float of a drained frame
                    for f in self.touch:
                        f.result()
                    self.touch = []
                t2 = time.perf_counter()
                src = self.stage[b].numpy()
                cuts = np.linspace(0, hi - lo, self.COPY_THREADS + 1).astype(int)
                list(self.pool.map(lambda i: np.copyto(self.host[lo + cuts[i]:lo + cuts[i + 1]], src[cuts[i]:cuts[i + 1]]),
                                   range(self.COPY_THREADS)))
                self.event_wait_seconds += t1 - t0
                self.touch_wait_seconds += t2 - t1
                self.copy_seconds += time.perf_counter() - t2
                self.copied_bytes += (hi - lo) * src[0].nbytes
            except BaseException as e:       # surfaced by finish()
                self.error = e
            finally:
                self.stage_free[b].set()
                self.jobs.task_done()

    def send(self, frames: torch.Tensor, host_lo: int) -> "torch.cuda.Event":
        """Queue device frames [m,h0,w0] (final once the current stream gets here) for host rows [host_lo, host_lo+m).
        Returns an event on the copy stream behind the last D2H copy that reads `frames` (a caller that recycles the
        device memory makes its stream wait for it)."""
        if self.direct:
            self._reg_done.wait()
            if self._reg_ok:                     # DMA straight into the page-locked result rows
                lo0 = self._reg_slice.start or 0
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(self.copy_stream):
                    self.copy_stream.wait_event(ready)
                    self._host_t[host_lo - lo0:host_lo - lo0 + frames.shape[0]].copy_(frames, non_blocking=True)
                    done = torch.cuda.Event()
                    done.record(self.copy_stream)
                frames.record_stream(self.copy_stream)
                self.copied_bytes += frames.numel() * 4
                return done
        if self.stage is None:
            self.stage, self._stage_token = _pinned_acquire(("drain",) + self._stage_shape[1:], self.STAGES, self._stage_shape,
                                                            torch.float32)
        for off in range(0, frames.shape[0], INFER_LEN):
            part = frames[off:off + INFER_LEN]
            b = self.batch_no % self.STAGES
            self.stage_free[b].wait()
            self.stage_free[b].clear()
            ready = torch.cuda.Event()
            ready.record()
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(ready)
                self.stage[b][:part.shape[0]].copy_(part, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.copy_stream)
            self.jobs.put((ev, b, host_lo + off, host_lo + off + part.shape[0]))
            self.batch_no += 1
        return ev

    def finish(self) -> np.ndarray:
        if self.direct:
            self._reg_done.wait()
            if self._reg_ok:
                self.copy_stream.synchronize()   # (the caller releases the page lock: unregister_later)
        self.jobs.put(None)
        self.jobs.join()
        self.drainer.join()
        self.pool.shutdown()
        self.touch_pool.shutdown()
        _pinned_release(self._stage_token)       # every drain copy out of the staging buffers has completed
        self._stage_token = None
        if self.error is not None:
            raise self.error
        return self.host


def make_blend_weights(device) -> torch.Tensor:
    step = 1.0 / (INTERP_LEN - 1)                         # get_interpolate_frames (utils/util.py:65-74)
    return torch.tensor([0.0] + [i * step for i in range(1, INTERP_LEN - 1)] + [1.0], dtype=torch.float32, device=device)


class WindowAligner:
    """Sequential scale/shift alignment + cross-fade of consecutive windows on the device
    (video_depth.py:216-252, utils/util.py:40-74).  (scale, shift) never leave the GPU; frames that can no longer
    change (everything but the last 8) are streamed to the host (HostDrain) while the next windows compute.

    Device memory is bounded: the aligned frames live in a ring of RING_SEGS segments of 22 frames (a window adds 22
    frames and cross-fades into the last 8 of its predecessor; everything older has been handed to the D2H pipeline).
    Frame a sits at ring position (a + 12) % ring length, which puts the end of window 0 (32 frames) and every later
    window on segment boundaries, so each window's 22 new frames and its 8-frame cross-fade tail are contiguous; a
    segment is only overwritten after the D2H copies that read it have completed (events of HostDrain.send)."""

    SEG = INFER_LEN - OVERLAP          # 22 new frames per window
    RING_SEGS = 4

    def __init__(self, n_frames: int, h0: int, w0: int, device, mode: str = "affine"):
        self.n, self.h0, self.w0, self.device, self.mode = n_frames, h0, w0, device, mode
        self.ring_len = aligner_ring_len(n_frames, self.RING_SEGS)
        self.out = torch.empty(self.ring_len, h0, w0, dtype=torch.float32, device=device)
        self.seg_ev = [None] * (self.ring_len // self.SEG)               # last D2H copy that reads the segment
        self.filled = 0
        self.ref = None                      # [2,h0,w0]: (ref_align[0], ref_align[1])
        self.ss = torch.tensor([1.0, 0.0], dtype=torch.float32, device=device)
        self.scratch = torch.zeros(4 * ops.LSQ_MAX_PARTIALS, dtype=torch.float64, device=device)
        self.blend_w = make_blend_weights(device)
        self.drain = HostDrain(np.empty((n_frames, h0, w0), dtype=np.float32), device)
        self.sent = 0                        # frames already handed to the D2H pipeline

    def _pos(self, a: int) -> int:
        return aligner_ring_pos(a, self.ring_len)

    def _claim(self, r: int, m: int) -> torch.Tensor:
        """Ring frames [r, r+m) for writing: the D2H copies of what they held must have completed."""
        for g in range(r // self.SEG, (r + m - 1) // self.SEG + 1):
            if self.seg_ev[g] is not None:
                torch.cuda.current_stream().wait_event(self.seg_ev[g])
                self.seg_ev[g] = None
        return self.out[r:r + m]

    def _send(self, upto: int) -> None:
        """Stream frames [sent, upto) (final values) to the host."""
        upto = min(upto, self.n)
        while upto > self.sent:
            r = self._pos(self.sent)
            m = min(upto - self.sent, self.ring_len - r)                  # (split where the ring wraps)
            ev = self.drain.send(self.out[r:r + m], self.sent)
            for g in range(r // self.SEG, (r + m - 1) // self.SEG + 1):
                self.seg_ev[g] = ev
            self.sent += m

    def push(self, d: torch.Tensor) -> None:
        """d: raw depths of the next window, fp32 [32,h0,w0]."""
        d = d.contiguous()
        align_len = OVERLAP - INTERP_LEN                                  # 2; kf_align_list = [0, 12]
        if self.filled == 0:
            self._claim(self._pos(0), INFER_LEN).copy_(d)                 # window 0 copied unclamped (:222-225)
            self.ref = torch.stack([d[KEYFRAMES[0]], d[KEYFRAMES[1]]])
            self.filled = INFER_LEN
        else:
            if self.mode == "affine":
                ops.lsq_scale_shift(d[:align_len], self.ref, self.ss, self.scratch)      # :227-232
            rt = self._pos(self.filled - INTERP_LEN)                      # the last 8 frames of the previous segment
            tail = self.out[rt:rt + INTERP_LEN]
            ops.affine_clamp_blend(d[align_len:OVERLAP], self.ss, tail, prev=tail, blend_w=self.blend_w)   # :234-239
            new = self._claim(self._pos(self.filled), self.SEG)
            ops.affine_clamp_blend(d[OVERLAP:], self.ss, new)                                              # :241-244
            ref1 = self.ref[1:2]
            ops.affine_clamp_blend(d[KEYFRAMES[1]:KEYFRAMES[1] + 1], self.ss, ref1)                       # :246-250
            self.filled += self.SEG
        self._send(self.filled - INTERP_LEN)          # the last 8 frames are still cross-faded with the next window

    def result(self) -> np.ndarray:
        self._send(self.n)
        return self.drain.finish()
