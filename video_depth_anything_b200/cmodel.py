"""ctypes wrapper of libvda's handle-level API (vda_create / vda_set_weight / vda_finalize_weights / vda_workspace_bytes /
vda_forward, and the stream group's vda_stream_plan_* / vda_stream_step, include/vda.h): what a non-Python host binds.  The
Python package itself uses engine.py (same schedule, plus CUDA-graph replay and the encoder-feature cache) and its own
stream planner (windows.StreamGroupPlan); this wrapper exists so that tests can hold the C schedule and the C planner
against them bit for bit, and as the worked example of INTEGRATION.md §2b."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import check
from .ops import dt_code
from .video_depth import check_yuv_frame, yuv_source
from .windows import (color_args, color_descriptors, color_frame_shape, group_block_layout, group_color_layout,
                      group_descriptors, pixel_format_code)


class CModel:
    def __init__(self, encoder: str, features: int, out_channels: Sequence[int], num_frames: int = 32,
                 dtype=torch.bfloat16, device="cuda:0"):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.num_frames = num_frames
        oc = (C.c_int32 * 4)(*out_channels)
        self.handle = C.c_void_p()
        check(self.lib.vda_create(encoder.encode(), features, oc, num_frames, dt_code(dtype), self.device.index or 0,
                                  C.byref(self.handle)))
        self._ws = None

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for k, v in sd.items():
            t = v.detach().to("cpu", torch.float32).contiguous()
            shape = (C.c_int64 * t.dim())(*t.shape)
            check(self.lib.vda_set_weight(self.handle, k.encode(), t.data_ptr(), shape, t.dim()))
        with torch.cuda.device(self.device):
            check(self.lib.vda_finalize_weights(self.handle))

    def workspace_bytes(self, B: int, T: int, H: int, W: int) -> int:
        n = self.lib.vda_workspace_bytes(self.handle, B, T, H, W)
        if n < 0:
            raise _lib.VdaError("vda_workspace_bytes failed: " + self.lib.vda_last_error().decode(errors="replace"))
        return n

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x fp32 [B,T,3,H,W] on the model's device -> depth fp32 [B,T,H,W]."""
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
        x = x.contiguous()
        B, T, _, H, W = x.shape
        with torch.cuda.device(self.device):
            need = self.workspace_bytes(B, T, H, W)
            if self._ws is None or self._ws.numel() < need:
                self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
            out = torch.empty(B, T, H, W, dtype=torch.float32, device=self.device)
            check(self.lib.vda_forward(self.handle, x.data_ptr(), B, T, H, W, out.data_ptr(), self._ws.data_ptr(),
                                       self._ws.numel(), torch.cuda.current_stream().cuda_stream))
            return out

    def close(self) -> None:
        if self.handle:
            self.lib.vda_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:       # noqa: BLE001
            pass


def resize_hw(h0: int, w0: int, input_size: int = 518):
    """vda_resize_hw: the network size of an (h0, w0) frame (windows.get_resize_hw in C)."""
    lib = _lib.load()
    nh, nw = C.c_int(), C.c_int()
    check(lib.vda_resize_hw(int(h0), int(w0), int(input_size), C.byref(nh), C.byref(nw)))
    return nh.value, nw.value


class CStreamPlan:
    """The C host planner of a stream group (vda_stream_plan_*) with windows.StreamGroupPlan's methods: open / close /
    step(handles, sizes, counts) -> (bucket, int32 table), `net` = the group's network size.  A push the planner rejects
    raises ValueError with the library's message and changes nothing."""

    def __init__(self, max_streams: int, num_frames: int = 32, input_size: int = 518, max_frames: Optional[int] = None):
        self.lib = _lib.load()
        self.handle = C.c_void_p()
        self._call(self.lib.vda_stream_plan_create(int(max_streams), 0 if max_frames is None else int(max_frames),
                                                   int(num_frames), int(input_size), C.byref(self.handle)))
        self.L = num_frames - 1
        n = C.c_int()
        self._call(self.lib.vda_stream_plan_buckets(self.handle, None, 0, C.byref(n)))
        buckets = (C.c_int32 * n.value)()
        self._call(self.lib.vda_stream_plan_buckets(self.handle, buckets, n.value, C.byref(n)))
        self.buckets = list(buckets)
        self.net = None
        self._table = np.empty(self.buckets[-1] * (self.L + 4), np.int32)

    def _call(self, rc: int) -> None:
        if rc != 0:
            raise ValueError(self.lib.vda_last_error().decode(errors="replace"))

    def open(self) -> int:
        h = C.c_int64()
        self._call(self.lib.vda_stream_plan_open(self.handle, C.byref(h)))
        return h.value

    def close(self, h: int) -> None:
        self._call(self.lib.vda_stream_plan_close(self.handle, int(h)))

    def step(self, handles, sizes=None, counts=None):
        n = len(handles)
        hs = np.ascontiguousarray(handles, np.int64)
        sz = None if sizes is None else np.ascontiguousarray(np.asarray(sizes, np.int32).reshape(n, 2))
        ct = None if counts is None else np.ascontiguousarray(counts, np.int32)
        if ct is not None and ct.size != n:
            raise ValueError("one frame count per stream of the push")
        bk, nh, nw = C.c_int(), C.c_int(), C.c_int()
        self._call(self.lib.vda_stream_plan_step(self.handle, hs.ctypes.data, None if sz is None else sz.ctypes.data,
                                                 None if ct is None else ct.ctypes.data, n, self._table.ctypes.data,
                                                 self._table.size, C.byref(bk), C.byref(nh), C.byref(nw)))
        if nh.value:
            self.net = (nh.value, nw.value)
        return bk.value, self._table[:bk.value * (self.L + 4)].copy()

    def close_plan(self) -> None:
        if self.handle:
            self.lib.vda_stream_plan_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close_plan()
        except Exception:       # noqa: BLE001
            pass


class CStreamGroup:
    """A stream group run through the C library alone: the C planner (CStreamPlan) and vda_stream_step, with one CUDA
    graph per (bucket, causal) captured on first use.  The push contract of DepthStreamGroup.push(..., to_host=False) for
    uint8 CUDA frames: {handle: frame [H0,W0,3] or stack [k,H0,W0,3]} (or pairs) -> {handle: fresh fp32 CUDA depth [H0,W0]
    or [k,H0,W0]}.  Frames are read in place (rows may be pitched).  `graphs=False` runs every step eagerly.
    `pixel_format` "nv12" | "i420": YUV 4:2:0 CUDA frames (packed [3*H0/2, W0] or plane tuples, the CUDA forms of
    DepthStreamGroup.push) through vda_frame_planes descriptors and vda_stream_step_planes.
    `output_format` "rgb" | "gray" | "nv12" | "i420" (with `colormap`, `value_range`): fresh uint8 CUDA frames of that
    format instead of depths, the depths going to a device arena; vda_depth_range (for the "frame" range) and
    vda_colorize_depth run after the step inside the same graph."""

    def __init__(self, model: CModel, max_streams: int = 8, input_size: int = 518, max_frames: Optional[int] = None,
                 graphs: bool = True, pixel_format: str = "rgb", output_format: str = "depth", colormap="inferno",
                 value_range="frame"):
        pixel_format_code(pixel_format)
        self.color = color_args(output_format, colormap, value_range, allow_video=False)
        self.pixel_format = pixel_format
        self.model, self.lib, self.device = model, model.lib, model.device
        self.plan = CStreamPlan(max_streams, model.num_frames, input_size, max_frames)
        self.max_streams, self.L = int(max_streams), self.plan.L
        self.use_graphs = graphs
        self.graphs = {}                                 # (bucket, causal) -> torch.cuda.CUDAGraph
        self.pool = None

    def open(self) -> int:
        return self.plan.open()

    def close_stream(self, handle: int) -> None:
        self.plan.close(handle)

    def _alloc(self) -> None:
        h, (self.nh, self.nw) = self.model.handle, self.plan.net
        pool_bytes = self.lib.vda_stream_pool_bytes(h, self.max_streams, self.nh, self.nw)
        self.ws_bytes = self.lib.vda_stream_workspace_bytes(h, self.plan.buckets[-1], self.nh, self.nw)
        if pool_bytes < 0 or self.ws_bytes < 0:
            raise _lib.VdaError(self.lib.vda_last_error().decode(errors="replace"))
        bk_max = self.plan.buckets[-1]
        nbytes = group_block_layout(bk_max, self.L, self.pixel_format)[2].stop
        if self.color[0] is not None:
            nbytes = group_color_layout(bk_max, self.L, self.pixel_format).stop
        with torch.cuda.device(self.device):
            self.pool = torch.empty(pool_bytes, dtype=torch.uint8, device=self.device)
            self._ws = torch.empty(self.ws_bytes + 1024, dtype=torch.uint8, device=self.device)
            self.meta_dev = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
            self.meta_host = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
            if self.color[0] is not None:
                _, table, rng = self.color
                self.color_table = None if table is None else torch.from_numpy(table.copy()).to(self.device)
                self.range_scratch = torch.empty(self.lib.vda_depth_range_scratch_bytes(bk_max), dtype=torch.uint8,
                                                 device=self.device)
                self.color_range = torch.tensor([[float(rng[0]), float(rng[1])]] if rng != "frame" else
                                                [[0.0, 0.0]] * bk_max, dtype=torch.float32, device=self.device)
        self.ws = -(-self._ws.data_ptr() // 1024) * 1024          # vda_stream_step wants a 1024-byte aligned workspace

    def _launch(self, bk: int, causal: bool) -> None:
        fs, os_, ts = group_block_layout(bk, self.L, self.pixel_format)
        m = self.meta_dev.data_ptr()
        step = self.lib.vda_stream_step if self.pixel_format == "rgb" else self.lib.vda_stream_step_planes
        st = torch.cuda.current_stream().cuda_stream
        check(step(self.model.handle, m + fs.start, m + os_.start, m + ts.start, bk, int(causal),
                                       self.pool.data_ptr(), self.max_streams, self.nh, self.nw, self.ws, self.ws_bytes,
                                       st))
        if self.color[0] is not None:
            per_row = self.color[2] == "frame"
            if per_row:
                check(self.lib.vda_depth_range(m + os_.start, bk, 0, self.color_range.data_ptr(),
                                               self.range_scratch.data_ptr(), st))
            cs = group_color_layout(bk, self.L, self.pixel_format)
            check(self.lib.vda_colorize_depth(m + os_.start, m + cs.start, bk, self.color_range.data_ptr(), int(per_row),
                                              None if self.color_table is None else self.color_table.data_ptr(), st))

    def _step(self, bk: int, causal: bool) -> None:
        if not self.use_graphs:
            return self._launch(bk, causal)
        g = self.graphs.get((bk, causal))
        if g is None:
            # a step is not idempotent (it writes the pool), so the warm-up and the capture run on pad rows (pool row -1:
            # no pool byte read or written); the push's own table is restored for the replay
            ts = group_block_layout(bk, self.L, self.pixel_format)[2]
            end = group_color_layout(bk, self.L, self.pixel_format).stop if self.color[0] is not None else ts.stop
            self.meta_dev[ts.start:ts.start + 4 * bk].fill_(255)
            self._launch(bk, causal)                  # warm-up, outside the capture: a new network size's position table
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._launch(bk, causal)
            self.graphs[(bk, causal)] = g
            self.meta_dev[:end].copy_(self.meta_host[:end], non_blocking=True)
        g.replay()

    def _check_frame(self, f):
        if self.pixel_format != "rgb":
            return check_yuv_frame(f, self.pixel_format, self.device, self.L, host=False)
        if not isinstance(f, torch.Tensor) or not f.is_cuda or f.device != self.device:
            raise ValueError(f"a frame must be a CUDA tensor on the group's device {self.device}")
        if f.dtype != torch.uint8 or f.dim() not in (3, 4) or f.shape[-1] != 3:
            raise ValueError(f"a frame must be a uint8 tensor [H0,W0,3] (or a stack [k,H0,W0,3]), got {f.dtype} {tuple(f.shape)}")
        if f.stride(-1) != 1 or f.stride(-2) != 3 or f.stride(-3) < 3 * f.shape[-2]:
            raise ValueError(f"a frame's pixels must be contiguous, stride (pitch >= 3 * W0, 3, 1), got {f.stride()}")
        return (int(f.shape[0]) if f.dim() == 4 else None), int(f.shape[-3]), int(f.shape[-2])

    @torch.no_grad()
    def push(self, frames) -> dict:
        items = list(frames.items()) if isinstance(frames, dict) else list(frames)
        shapes = [self._check_frame(f) for _, f in items]
        handles = [h for h, _ in items]
        fmt = self.color[0]
        if fmt is not None:
            cshapes = [color_frame_shape(h0, w0, fmt) for _, h0, w0 in shapes]     # ValueError: odd size for YUV output
        bk, table = self.plan.step(handles, [(h0, w0) for _, h0, w0 in shapes], [k or 1 for k, _, _ in shapes])
        if self.pool is None:
            self._alloc()
        with torch.cuda.device(self.device):
            if fmt is not None:
                # depths to a device arena (grown on demand: its addresses are in the descriptors), colour frames returned
                n_px = sum((k or 1) * h0 * w0 for k, h0, w0 in shapes)
                if getattr(self, "depth_arena", None) is None or self.depth_arena.numel() < n_px:
                    self.depth_arena = torch.empty(n_px, dtype=torch.float32, device=self.device)
                depth_base = self.depth_arena.data_ptr()
                couts = [torch.empty(*((k,) if k else ()), *c, dtype=torch.uint8, device=self.device)
                         for (k, _, _), c in zip(shapes, cshapes)]
                cdst = []
            outs = [torch.empty(*((k,) if k else ()), h0, w0, dtype=torch.float32, device=self.device)
                    for k, h0, w0 in shapes] if fmt is None else [None] * len(shapes)
            srcs, dsts = [], []
            for (_, f), o, (k, h0, w0) in zip(items, outs, shapes):
                for j in range(k or 1):
                    if self.pixel_format != "rgb":
                        srcs.append(yuv_source(f, j if k else None, h0, w0, self.pixel_format) + (h0, w0))
                    else:
                        srcs.append((f[j].data_ptr(), f.stride(1), h0, w0) if k else (f.data_ptr(), f.stride(0), h0, w0))
                    if fmt is None:
                        dsts.append(o.data_ptr() + 4 * j * h0 * w0)
                    else:
                        dsts.append(depth_base)
                        depth_base += 4 * h0 * w0
            fd, od = group_descriptors(bk, srcs, dsts, self.pixel_format)
            fs, os_, ts = group_block_layout(bk, self.L, self.pixel_format)
            mh = self.meta_host.numpy()
            mh[fs], mh[os_], mh[ts] = fd.view(np.uint8), od.view(np.uint8), table.view(np.uint8)
            end = ts.stop
            if fmt is not None:
                cs = group_color_layout(bk, self.L, self.pixel_format)
                for c, (k, h0, w0) in zip(couts, shapes):
                    cdst += [(c.data_ptr() + j * c[0].numel() if k else c.data_ptr(), h0, w0) for j in range(k or 1)]
                mh[cs] = color_descriptors(bk, cdst, fmt).view(np.uint8)
                end = cs.stop
            self.meta_dev[:end].copy_(self.meta_host[:end], non_blocking=True)
            self._step(bk, max(k or 1 for k, _, _ in shapes) > 1)
            torch.cuda.current_stream().synchronize()
        return dict(zip(handles, outs if fmt is None else couts))

    def close(self) -> None:
        self.graphs = {}
        self.pool = None
        self.plan.close_plan()
