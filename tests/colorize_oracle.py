"""NumPy restatement of the colour-mapping contract of include/vda.h (vda_depth_range / vda_colorize_depth) and
display.colorize: the reference's save_video frame loop (utils/dc_utils.py:72-86), the clamped level for fixed
ranges, and the integer RGB -> YUV 4:2:0 form of cv2.cvtColor(COLOR_RGB2YUV_I420) with top-left chroma."""
import numpy as np


def save_video_frames(frames: np.ndarray, table=None, grayscale: bool = False):
    """The reference's loop, verbatim but for the writer and the table (a uint8 [256, 3] table T stands for
    (colormap * 255).astype(np.uint8), so T[depth_norm] is its depth_vis)."""
    out = []
    d_min, d_max = frames.min(), frames.max()
    for i in range(frames.shape[0]):
        depth = frames[i]
        depth_norm = ((depth - d_min) / (d_max - d_min) * 255).astype(np.uint8)
        depth_vis = table[depth_norm] if not grayscale else depth_norm
        out.append(depth_vis)
    return np.stack(out)


def level(d: np.ndarray, lo, hi) -> np.ndarray:
    """q = min(255, max(0, trunc(((d - lo) / (hi - lo)) * 255))) in float32; zeros when hi <= lo."""
    d = np.asarray(d, np.float32)
    lo, hi = np.float32(lo), np.float32(hi)
    if not hi > lo:
        return np.zeros(d.shape, np.uint8)
    with np.errstate(over="ignore", invalid="ignore"):
        t = ((d - lo) / (hi - lo)) * np.float32(255)
    return np.clip(np.trunc(t), 0, 255).astype(np.uint8)


def rgb_to_i420(rgb: np.ndarray) -> np.ndarray:
    """uint8 [H, W, 3] (H, W even) -> I420 [3H/2, W] in OpenCV's packed layout: Y, then U [H/2, W/2], then V."""
    h, w, _ = rgb.shape
    r, g, b = (rgb[..., c].astype(np.int64) for c in range(3))
    y = (269484 * r + 528482 * g + 102760 * b + (16 << 20) + (1 << 19)) >> 20
    r, g, b = r[::2, ::2], g[::2, ::2], b[::2, ::2]                    # chroma of the top-left pixel of each 2 x 2 block
    u = (-155188 * r - 305135 * g + 460324 * b + (128 << 20) + (1 << 19)) >> 20
    v = (460324 * r - 385875 * g - 74448 * b + (128 << 20) + (1 << 19)) >> 20
    return np.concatenate([y.ravel(), u.ravel(), v.ravel()]).astype(np.uint8).reshape(3 * h // 2, w)


def i420_to_nv12(yuv: np.ndarray) -> np.ndarray:
    """I420 [3H/2, W] -> NV12 [3H/2, W]: the same Y, then U and V interleaved."""
    h, w = 2 * yuv.shape[0] // 3, yuv.shape[1]
    flat = yuv.ravel()
    u = flat[h * w:h * w + h * w // 4]
    v = flat[h * w + h * w // 4:]
    uv = np.stack([u, v], axis=1).ravel()
    return np.concatenate([flat[:h * w], uv]).reshape(3 * h // 2, w)


def frames_of(q: np.ndarray, table, fmt: str) -> np.ndarray:
    """Frames [N, ...] of the levels q [N, H, W] in output format fmt ("rgb" | "gray" | "nv12" | "i420")."""
    if fmt == "gray":
        return q.copy()
    rgb = table[q]
    if fmt == "rgb":
        return rgb
    yuv = np.stack([rgb_to_i420(f) for f in rgb])
    return yuv if fmt == "i420" else np.stack([i420_to_nv12(f) for f in yuv])


def colorize(depths: np.ndarray, table, value_range="video", fmt: str = "rgb") -> np.ndarray:
    """What display.colorize returns for float32 depths [N, H, W]."""
    d = np.asarray(depths, np.float32)
    if isinstance(value_range, str):
        if value_range == "video":
            rngs = [(d.min(), d.max())] * d.shape[0]
        else:
            rngs = [(f.min(), f.max()) for f in d]
    else:
        rngs = [value_range] * d.shape[0]
    q = np.stack([level(f, lo, hi) for f, (lo, hi) in zip(d, rngs)])
    return frames_of(q, table, fmt)
