"""Depth frames for displays and encoders: `colorize` is the device-side replacement of save_video's frame loop
(utils/dc_utils.py:72-86): range, 8-bit level, colour table and pixel format in libvda's kernels (vda_depth_range,
vda_colorize_depth), for depths in device memory or on the host."""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .video_depth import _pinned_acquire, _pinned_release
from .windows import OUT_DESC, color_args, color_descriptors, color_frame_shape

STAGE_BYTES = 64 << 20          # fp32 depths per pinned staging buffer (two of them) for host input
MAX_ROWS = 4096                 # rows per launch for device input (a launch takes up to 65535)


def _out_desc(base: int, n: int, h: int, w: int) -> np.ndarray:
    od = np.zeros(n, OUT_DESC)
    od["dst"] = base + 4 * h * w * np.arange(n, dtype=np.uint64)
    od["H0"], od["W0"] = h, w
    return od


def _to_dev(a: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(a.view(np.uint8).copy()).to(device)


class _Colorizer:
    """Descriptors and launches for frames of one size: depth rows packed at a device address -> colour frames packed
    at another."""

    def __init__(self, h: int, w: int, fmt: int, table, device):
        self.h, self.w, self.fmt, self.device = h, w, fmt, device
        self.shape = color_frame_shape(h, w, fmt)
        self.frame_bytes = int(np.prod(self.shape))
        self.table = None if table is None else torch.from_numpy(np.array(table, order="C")).to(device)

    def descs(self, src: int, dst: int, n: int):
        cd = color_descriptors(n, [(dst + i * self.frame_bytes, self.h, self.w) for i in range(n)], self.fmt)
        return _to_dev(_out_desc(src, n, self.h, self.w), self.device), _to_dev(cd, self.device)

    def colorize(self, od, cd, rng: torch.Tensor, per_row: bool) -> None:
        ops.colorize_depth(od, cd, rng, per_row, self.table)


def _fold(ranges: torch.Tensor) -> torch.Tensor:
    """The combined range of k ranges fp32 [k, 2]: the all-rows range of the [k, 2] array itself (each lo <= its hi)."""
    od = _to_dev(_out_desc(ranges.data_ptr(), 1, ranges.shape[0], 2), ranges.device)
    return ops.depth_range(od, True)


@torch.no_grad()
def colorize(depths, colormap="inferno", value_range="video", pixel_format: str = "rgb"):
    """Colour-mapped uint8 frames of fp32 depths, the frame loop of the reference's save_video (utils/dc_utils.py:72-86):
    `for f in colorize(depths, colormap=table): writer.append_data(f)`.

    depths: float32 [N, H, W] or [H, W], a numpy array (frames come back as a numpy array) or a CUDA tensor (a fresh
    CUDA tensor on the same device).  Host depths go through two pinned staging buffers of STAGE_BYTES in chunks, so
    device memory stays bounded whatever the length of the video.
    colormap: "inferno" (OpenCV's table, windows.INFERNO) or a uint8 [256, 3] RGB table, e.g. the reference's
    (np.array(cm.get_cmap("inferno").colors) * 255).astype(np.uint8), which reproduces its frames exactly.
    value_range: "video" (save_video's frames.min(), frames.max() over all N frames), "frame" (each frame's own) or a
    fixed (lo, hi), e.g. metres for a metric model; values outside a fixed range clamp to levels 0 / 255.
    pixel_format: "rgb" -> [N, H, W, 3]; "gray" -> the 8-bit level [N, H, W] (save_video(grayscale=True)); "nv12" /
    "i420" -> YUV 4:2:0 [N, 3H/2, W] in OpenCV's packed layout (BT.601 limited range, cv2.cvtColor(COLOR_RGB2YUV_I420)
    of the RGB frame with top-left chroma), H and W even.
    Level of a depth d: min(255, max(0, trunc(((d - lo) / (hi - lo)) * 255))) in IEEE float32, bit-exact to the
    reference; 0 where hi <= lo.  ValueError for a bad argument, before anything is launched."""
    if pixel_format == "depth":
        raise ValueError("colorize writes uint8 frames: pixel_format is 'rgb', 'gray', 'nv12' or 'i420'")
    fmt, table, rng = color_args(pixel_format, colormap, value_range)
    host = isinstance(depths, np.ndarray)
    if host:
        ok = depths.dtype == np.float32 and depths.ndim in (2, 3)
    elif isinstance(depths, torch.Tensor):
        ok = depths.is_cuda and depths.dtype == torch.float32 and depths.dim() in (2, 3)
    else:
        ok = False
    if not ok:
        raise ValueError(f"depths must be float32 [N, H, W] or [H, W], a numpy array or a CUDA tensor, got "
                         f"{type(depths).__name__} {getattr(depths, 'dtype', '')} {tuple(getattr(depths, 'shape', ()))}")
    single = depths.ndim == 2
    n, h, w = (1,) + tuple(depths.shape) if single else tuple(depths.shape)
    if n < 1 or h < 1 or w < 1:
        raise ValueError(f"empty depths of shape {tuple(depths.shape)}")
    shape = color_frame_shape(h, w, fmt)                       # ValueError: odd size for YUV
    device = depths.device if not host else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(device):
        cz = _Colorizer(h, w, fmt, table, device)
        fixed = None if isinstance(rng, str) else torch.tensor([rng[0], rng[1]], dtype=torch.float32, device=device)
        if host:
            out = _colorize_host(cz, np.ascontiguousarray(depths.reshape(n, h, w)), rng, fixed)
        else:
            out = _colorize_device(cz, depths.reshape(n, h, w).contiguous(), rng, fixed)
    return out.reshape(shape) if single else out


def _colorize_device(cz: _Colorizer, d: torch.Tensor, rng, fixed) -> torch.Tensor:
    n = d.shape[0]
    out = torch.empty((n,) + cz.shape, dtype=torch.uint8, device=d.device)
    chunks = [(lo, min(lo + MAX_ROWS, n)) for lo in range(0, n, MAX_ROWS)]
    descs = [cz.descs(d[lo].data_ptr(), out[lo].data_ptr(), hi - lo) for lo, hi in chunks]
    if rng == "video":
        parts = torch.empty(len(chunks), 2, dtype=torch.float32, device=d.device)
        for c, (od, _) in enumerate(descs):
            ops.depth_range(od, True, parts[c])
        fixed = _fold(parts)
    for od, cd in descs:
        if rng == "frame":
            cz.colorize(od, cd, ops.depth_range(od, False), True)
        else:
            cz.colorize(od, cd, fixed, False)
    return out


def _colorize_host(cz: _Colorizer, d: np.ndarray, rng, fixed) -> np.ndarray:
    """Two passes over the chunks for the "video" range (its range, then its colours), one otherwise.  Each chunk: host
    copy into a pinned buffer, H2D, launches, D2H into a pinned buffer; the host copy of chunk c out of its buffer
    happens while chunk c + 1 is on the device."""
    n, h, w = d.shape
    dev = cz.device
    k = max(1, min(n, STAGE_BYTES // (4 * h * w)))
    chunks = [(lo, min(lo + k, n)) for lo in range(0, n, k)]
    out = np.empty((n,) + cz.shape, dtype=np.uint8)
    st_in, tok_in = _pinned_acquire(("colorize_in", h, w), 2, (k, h, w), torch.float32)
    st_out, tok_out = _pinned_acquire(("colorize_out", h, w, cz.fmt), 2, (k,) + cz.shape, torch.uint8)
    try:
        d_in = torch.empty(2, k, h, w, dtype=torch.float32, device=dev)
        d_out = torch.empty((2, k) + cz.shape, dtype=torch.uint8, device=dev)
        descs = [cz.descs(d_in[b].data_ptr(), d_out[b].data_ptr(), k) for b in range(2)]
        in_free = [None, None]

        def upload(c):
            lo, hi = chunks[c]
            b = c & 1
            if in_free[b] is not None:
                in_free[b].synchronize()
            np.copyto(st_in[b][:hi - lo].numpy(), d[lo:hi])
            d_in[b][:hi - lo].copy_(st_in[b][:hi - lo], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            in_free[b] = ev
            od, cd = descs[b]
            m = hi - lo
            return od[:m * OUT_DESC.itemsize], cd[:m * 64]

        if rng == "video":
            parts = torch.empty(len(chunks), 2, dtype=torch.float32, device=dev)
            for c in range(len(chunks)):
                od, _ = upload(c)
                ops.depth_range(od, True, parts[c])
            fixed = _fold(parts)
        pending = None          # (chunk, event of its D2H): drained after the next chunk is queued

        def drain(p):
            c, ev = p
            lo, hi = chunks[c]
            ev.synchronize()
            np.copyto(out[lo:hi], st_out[c & 1][:hi - lo].numpy())

        for c in range(len(chunks)):
            od, cd = upload(c)
            m = chunks[c][1] - chunks[c][0]
            if rng == "frame":
                cz.colorize(od, cd, ops.depth_range(od, False), True)
            else:
                cz.colorize(od, cd, fixed, False)
            st_out[c & 1][:m].copy_(d_out[c & 1][:m], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            if pending is not None:
                drain(pending)
            pending = (c, ev)
        if pending is not None:
            drain(pending)
        torch.cuda.current_stream().synchronize()
    finally:
        _pinned_release(tok_in)
        _pinned_release(tok_out)
    return out
