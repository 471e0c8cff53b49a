"""CPU: YUV 4:2:0 input (NV12 / I420).  The NumPy restatement of the conversion against cv2 on every (Y, U, V) triple, the
vda_frame_planes descriptor and its C ABI, the descriptors of packed and plane-tuple frames, and the checks that reject a
frame before anything is planned or launched."""
import ctypes as C
import os
import shutil
import subprocess
import types

import numpy as np
import pytest
import torch

import yuv_oracle as Y
from video_depth_anything_b200 import _lib
from video_depth_anything_b200.video_depth import DepthStreamGroup, check_yuv_frame, yuv_source
from video_depth_anything_b200.windows import (FRAME_DESC, FRAME_PLANES, OUT_DESC, group_block_layout, group_descriptors,
                                               pixel_format_code, video_frame_shape, yuv_frame_hw, yuv_planes)

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODES = {"nv12": cv2.COLOR_YUV2RGB_NV12, "i420": cv2.COLOR_YUV2RGB_I420}


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_restatement_equals_cv2_on_all_triples(fmt):
    frame = Y.all_triples(fmt)
    y, u, v = Y.split_planes(frame, fmt)
    # every (Y, U, V) triple occurs: 2^16 chroma pairs x 256 luma values
    key = (np.repeat(np.repeat(u.astype(np.int64), 2, 0), 2, 1) << 16) | \
          (np.repeat(np.repeat(v.astype(np.int64), 2, 0), 2, 1) << 8) | y
    assert np.unique(key).size == 1 << 24
    assert np.array_equal(Y.to_rgb(frame, fmt), cv2.cvtColor(frame, CODES[fmt]))


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_pack_split_round_trip_and_random_frames(fmt):
    rng = np.random.default_rng(3)
    for h0, w0 in [(2, 2), (6, 10), (50, 70), (36, 64)]:
        y = rng.integers(0, 256, (h0, w0), dtype=np.uint8)
        u, v = (rng.integers(0, 256, (h0 // 2, w0 // 2), dtype=np.uint8) for _ in range(2))
        f = Y.pack(y, u, v, fmt)
        assert f.shape == (3 * h0 // 2, w0)
        assert all(np.array_equal(a, b) for a, b in zip(Y.split_planes(f, fmt), (y, u, v)))
        assert np.array_equal(Y.to_rgb(f, fmt), cv2.cvtColor(f, CODES[fmt]))


def test_descriptor_and_abi():
    assert FRAME_PLANES.itemsize == 64                       # sizeof(vda_frame_planes)
    assert [FRAME_PLANES.fields[n][1] for n in ("plane", "pitch", "H0", "W0", "format", "reserved")] == [0, 24, 48, 52, 56, 60]
    assert {n: pixel_format_code(n) for n in ("rgb", "nv12", "i420")} == {"rgb": 0, "nv12": 1, "i420": 2}
    assert (_lib.PIX_NV12, _lib.PIX_I420) == (1, 2)
    with pytest.raises(ValueError):
        pixel_format_code("bgr")
    sigs = _lib._SIGS
    assert sigs["vda_preprocess_frames_yuv"][0] is C.c_int and len(sigs["vda_preprocess_frames_yuv"][1]) == 10
    assert len(sigs["vda_preprocess_frames_planes"][1]) == 6
    assert len(sigs["vda_stream_step_planes"][1]) == len(sigs["vda_stream_step"][1]) == 13
    assert sigs["vda_stream_step_planes"][1] == sigs["vda_stream_step"][1]
    h = open(os.path.join(ROOT, "include", "vda.h")).read()
    for name in ("vda_preprocess_frames_yuv", "vda_preprocess_frames_planes", "vda_stream_step_planes"):
        assert f"int {name}(" in h
    assert "VDA_PIX_NV12 = 1, VDA_PIX_I420 = 2" in h


def test_packed_frame_descriptors():
    h0, w0 = 50, 70
    assert yuv_frame_hw(75, 70, "nv12") == (50, 70)
    for rows, cols in [(74, 70), (75, 71), (0, 70)]:
        with pytest.raises(ValueError):
            yuv_frame_hw(rows, cols, "nv12")
    base = 0x100000
    assert yuv_planes(base, 80, h0, w0, "nv12") == ((base, base + 50 * 80, 0), (80, 80, 0))
    assert yuv_planes(base, 70, h0, w0, "i420") == ((base, base + 3500, base + 3500 + 875), (70, 35, 35))
    with pytest.raises(ValueError, match="plane tuple"):
        yuv_planes(base, 80, h0, w0, "i420")                # pitched packed I420: its chroma rows have no one pitch
    for fmt, code in (("nv12", 1), ("i420", 2)):
        src = yuv_planes(base, w0, h0, w0, fmt)
        fd, od = group_descriptors(4, [src + (h0, w0)], [0x900000], fmt)
        assert fd.dtype == FRAME_PLANES and od.dtype == OUT_DESC and len(fd) == 4
        assert tuple(fd[0]["plane"]) == src[0] and tuple(fd[0]["pitch"]) == src[1]
        assert (fd[0]["H0"], fd[0]["W0"], fd[0]["format"], fd[0]["reserved"]) == (h0, w0, code, 0)
        assert (fd[1:] == fd[0]).all() and (od[1:]["H0"] == 0).all()
        fs, os_, ts = group_block_layout(4, 31, fmt)
        assert fs == slice(0, 256) and os_ == slice(256, 320) and ts == slice(320, 320 + 4 * 4 * 35)
    assert group_block_layout(4, 31, "rgb") == group_block_layout(4, 31)
    assert group_block_layout(4, 31)[0].stop == 4 * FRAME_DESC.itemsize


def test_plane_tuple_descriptors_pitched_uv_at_an_offset():
    """An NVDEC-like surface: Y rows 128 bytes apart, the UV plane at Y + 128 * 64 (the aligned height), not right after
    row H0 - 1; and an I420 frame in three separate buffers of their own pitches."""
    h0, w0, pitch, aligned = 50, 70, 128, 64
    surf = torch.zeros(pitch * (aligned + aligned // 2), dtype=torch.uint8)
    yp = surf[:h0 * pitch].view(h0, pitch)[:, :w0]
    uvp = surf[aligned * pitch:aligned * pitch + h0 // 2 * pitch].view(h0 // 2, pitch)[:, :w0]
    assert check_yuv_frame((yp, uvp), "nv12", torch.device("cpu"), 31) == (None, h0, w0)
    src = yuv_source((yp, uvp), None, h0, w0, "nv12")
    assert src == ((surf.data_ptr(), surf.data_ptr() + aligned * pitch, 0), (pitch, pitch, 0))
    fd, _ = group_descriptors(1, [src + (h0, w0)], [0], "nv12")
    assert fd[0]["plane"][1] - fd[0]["plane"][0] == aligned * pitch
    # I420 stack of k = 3 frames, planes in separate allocations
    ys, us, vs = (torch.zeros(3, h, p, dtype=torch.uint8)[..., :w] for h, w, p in ((h0, w0, 96), (h0 // 2, w0 // 2, 64),
                                                                                  (h0 // 2, w0 // 2, 48)))
    assert check_yuv_frame((ys, us, vs), "i420", torch.device("cpu"), 31) == (3, h0, w0)
    src = yuv_source((ys, us, vs), 2, h0, w0, "i420")
    assert src == ((ys[2].data_ptr(), us[2].data_ptr(), vs[2].data_ptr()), (96, 64, 48))
    fd, _ = group_descriptors(2, [src + (h0, w0)], [0], "i420")
    assert tuple(fd[0]["pitch"]) == (96, 64, 48) and fd[0]["format"] == 2


def test_descriptor_errors():
    ok = ((1, 2, 3), (70, 35, 35), 50, 70)
    group_descriptors(1, [ok], [0], "i420")
    for bad in [((1, 2, 3), (70, 34, 35), 50, 70),            # short U pitch
                ((1, 2, 3), (69, 35, 35), 50, 70),            # short Y pitch
                ((1, 2, 3), (70, 35, 35), 51, 70),            # odd height
                ((1, 2, 3), (70, 35, 35), 50, 69)]:           # odd width
        with pytest.raises(ValueError):
            group_descriptors(1, [bad], [0], "i420")
    with pytest.raises(ValueError):
        group_descriptors(1, [((1, 2, 0), (70, 69, 0), 50, 70)], [0], "nv12")   # short UV pitch


def test_video_frame_shape():
    assert video_frame_shape(np.zeros((4, 75, 70), np.uint8), "nv12") == (4, 50, 70)
    assert video_frame_shape(np.zeros((4, 50, 70, 3), np.uint8)) == (4, 50, 70)
    for frames, fmt in [(np.zeros((4, 75, 71), np.uint8), "i420"), (np.zeros((4, 74, 70), np.uint8), "nv12"),
                        (np.zeros((4, 50, 70, 3), np.uint8), "nv12"), (np.zeros((4, 75, 70), np.uint8), "rgb"),
                        (np.zeros((4, 75, 70), np.int16), "nv12")]:
        with pytest.raises(ValueError):
            video_frame_shape(frames, fmt)


def _stub_group(fmt, max_streams=2):
    """A DepthStreamGroup on a stand-in engine: push() checks frames and plans before it touches a device."""
    eng = types.SimpleNamespace(device=torch.device("cuda", 0), generation=0, loaded=True)
    model = types.SimpleNamespace(num_frames=32)
    return DepthStreamGroup(model, eng, max_streams, 56, pixel_format=fmt)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_rejected_pushes_change_nothing(fmt):
    g = _stub_group(fmt)
    a, b = g.open(), g.open()
    good = np.zeros((75, 70), np.uint8)
    bad = [np.zeros((50, 70, 3), np.uint8),                   # an RGB frame (W0 = 3 is odd)
           np.zeros((75, 71), np.uint8),                      # odd width
           np.zeros((74, 70), np.uint8),                      # rows not 3 * H0 / 2
           np.zeros((75, 70), np.float32),                    # dtype
           np.zeros((32, 75, 70), np.uint8),                  # a stack of more than L = 31 frames
           torch.zeros(75, 70, dtype=torch.uint8),            # a tensor not on the group's device
           (torch.zeros(50, 70, dtype=torch.uint8),),         # a plane tuple of the wrong length
           [np.zeros((50, 70), np.uint8)] * (2 if fmt == "nv12" else 3)]   # planes must be CUDA tensors
    for f in bad:
        before = (dict(g.plan.t), dict(g.plan.size), g.plan.net)
        with pytest.raises(ValueError):
            g.push({a: good, b: f})
        assert (dict(g.plan.t), dict(g.plan.size), g.plan.net) == before
        assert g.pool is None                                 # nothing allocated, nothing launched
    assert g.plan.t == {a: 0, b: 0}
    with pytest.raises(ValueError):
        _stub_group("yuv444")


def test_plane_shape_checks():
    dev = torch.device("cpu")
    y, uv = torch.zeros(50, 70, dtype=torch.uint8), torch.zeros(25, 70, dtype=torch.uint8)
    u, v = torch.zeros(25, 35, dtype=torch.uint8), torch.zeros(25, 35, dtype=torch.uint8)
    assert check_yuv_frame((y, uv), "nv12", dev, 31) == (None, 50, 70)
    assert check_yuv_frame((y, u, v), "i420", dev, 31) == (None, 50, 70)
    for f, fmt in [((y, u), "nv12"), ((y, uv, v), "i420"), ((y, u, u[:, :34]), "i420"),
                   ((y[:, :69], uv[:, :69]), "nv12"), ((y[:49], uv), "nv12"),
                   ((y.t(), uv), "nv12"),                                      # column-major: not a row pitch
                   ((y.unsqueeze(0), uv), "nv12"),                             # stack and single frame mixed
                   (torch.zeros(75, 140, dtype=torch.uint8)[:, :70], "i420"),   # pitched packed I420
                   (np.zeros((75, 70), np.uint8), "nv12")]:                   # host frames: Python group only
        with pytest.raises(ValueError):
            check_yuv_frame(f, fmt, dev, 31, host=False)
    assert check_yuv_frame(torch.zeros(3, 75, 140, dtype=torch.uint8)[..., :70], "nv12", dev, 31) == (3, 50, 70)


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no gcc")
def test_c_host_nv12_compiles(tmp_path):
    """tests/c_host/host_stream_nv12.c is C99 against include/vda.h alone (compiled, not linked: no GPU needed)."""
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(cuda, "include"), "-c",
                           os.path.join(ROOT, "tests", "c_host", "host_stream_nv12.c"), "-o", str(tmp_path / "h.o")])
