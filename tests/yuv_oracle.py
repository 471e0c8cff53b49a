"""NumPy restatement of the YUV 4:2:0 -> RGB conversion of the ingest kernels (include/vda.h, vda_frame_planes): BT.601
limited range, nearest chroma (pixel (y, x) takes chroma sample (y/2, x/2)), in the integer form of OpenCV's
cv2.cvtColor(COLOR_YUV2RGB_NV12 / COLOR_YUV2RGB_I420).  Tests hold it against cv2 on every (Y, U, V) triple and use it
to build the frames the GPU tests push."""
from __future__ import annotations

import numpy as np


def yuv_to_rgb(y: np.ndarray, u: np.ndarray, v: np.ndarray) -> np.ndarray:
    """uint8 Y, U, V of equal shapes -> uint8 RGB [..., 3]."""
    u = u.astype(np.int64) - 128
    v = v.astype(np.int64) - 128
    luma = np.maximum(0, y.astype(np.int64) - 16) * 1220542 + (1 << 19)
    rgb = [luma + 1673527 * v, luma - 852492 * v - 409993 * u, luma + 2116026 * u]
    return np.stack([np.clip(c >> 20, 0, 255) for c in rgb], -1).astype(np.uint8)


def split_planes(frame: np.ndarray, fmt: str):
    """(Y [H0,W0], U [H0/2,W0/2], V [H0/2,W0/2]) of one frame packed in OpenCV's layout [3*H0/2, W0]."""
    h0, w0 = frame.shape[0] * 2 // 3, frame.shape[1]
    y, c = frame[:h0], frame[h0:]
    if fmt == "nv12":
        uv = c.reshape(h0 // 2, w0 // 2, 2)
        return y, uv[..., 0], uv[..., 1]
    flat = c.reshape(-1)
    q = h0 * w0 // 4
    return y, flat[:q].reshape(h0 // 2, w0 // 2), flat[q:].reshape(h0 // 2, w0 // 2)


def to_rgb(frame: np.ndarray, fmt: str) -> np.ndarray:
    """uint8 RGB [H0,W0,3] of one packed NV12 / I420 frame (what cv2.cvtColor gives)."""
    y, u, v = split_planes(frame, fmt)
    up = lambda c: np.repeat(np.repeat(c, 2, 0), 2, 1)       # noqa: E731  (nearest chroma)
    return yuv_to_rgb(y, up(u), up(v))


def pack(y: np.ndarray, u: np.ndarray, v: np.ndarray, fmt: str) -> np.ndarray:
    """One frame packed in OpenCV's layout [3*H0/2, W0] from its planes Y [H0,W0], U and V [H0/2,W0/2]."""
    h0, w0 = y.shape
    if fmt == "nv12":
        c = np.stack([u, v], -1).reshape(h0 // 2, w0)
    else:
        c = np.concatenate([u.reshape(-1), v.reshape(-1)]).reshape(h0 // 2, w0)
    return np.concatenate([y, c], 0)


def all_triples(fmt: str) -> np.ndarray:
    """A 4096 x 4096 frame [6144, 4096] holding every (Y, U, V) triple once: each 2x2 luma block shares one chroma sample
    (U, V) and takes four of the 256 luma values; the 2048 x 2048 chroma samples cover the 2^16 (U, V) pairs 64 times,
    once for each group of four luma values."""
    b = np.arange(2048 * 2048)
    uv, yb = b // 64, b % 64
    u = (uv // 256).astype(np.uint8).reshape(2048, 2048)
    v = (uv % 256).astype(np.uint8).reshape(2048, 2048)
    y = np.zeros((4096, 4096), np.uint8)
    for k, (dy, dx) in enumerate([(0, 0), (0, 1), (1, 0), (1, 1)]):
        y[dy::2, dx::2] = (4 * yb + k).reshape(2048, 2048)
    return pack(y, u, v, fmt)


def random_video(n: int, h0: int, w0: int, fmt: str, seed: int) -> np.ndarray:
    """uint8 [n, 3*H0/2, W0] of random packed frames."""
    return np.random.default_rng(seed).integers(0, 256, (n, 3 * h0 // 2, w0), dtype=np.uint8)


def video_to_rgb(frames: np.ndarray, fmt: str) -> np.ndarray:
    return np.stack([to_rgb(f, fmt) for f in frames])
