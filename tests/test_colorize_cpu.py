"""CPU: colour-mapped depth frames.  The NumPy restatement (colorize_oracle) against cv2 on every (R, G, B) triple and
against the reference expression at every level boundary, the built-in inferno table, the vda_color_planes layout,
the descriptors, and every argument check of colorize() and of stream groups, which all reject before anything is
planned or launched."""
import ctypes as C
import os
import shutil
import subprocess
import types

import numpy as np
import pytest
import torch

import colorize_oracle as O
from video_depth_anything_b200 import _lib, colorize, ops
from video_depth_anything_b200.video_depth import DepthStreamGroup
from video_depth_anything_b200.windows import (COLOR_PLANES, INFERNO, color_args, color_descriptors, color_frame_shape,
                                               group_block_layout, group_color_layout)

cv2 = pytest.importorskip("cv2")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_yuv_form_equals_cv2_on_all_triples():
    # every (R, G, B) triple as a uniform 2 x 2 block of an 8192 x 8192 image
    t = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([(t >> 16) & 255, (t >> 8) & 255, t & 255], axis=1).astype(np.uint8).reshape(4096, 4096, 3)
    img = np.repeat(np.repeat(rgb, 2, 0), 2, 1)
    assert np.array_equal(O.rgb_to_i420(img), cv2.cvtColor(img, cv2.COLOR_RGB2YUV_I420))


@pytest.mark.parametrize("hw", [(64, 96), (2, 2), (10, 6), (518, 924)])
def test_yuv_form_equals_cv2_on_random_images(hw):
    img = np.random.default_rng(hw[0]).integers(0, 256, hw + (3,), dtype=np.uint8)
    ref = cv2.cvtColor(img, cv2.COLOR_RGB2YUV_I420)
    assert np.array_equal(O.rgb_to_i420(img), ref)
    h, w = hw
    nv12 = O.i420_to_nv12(ref)
    assert np.array_equal(nv12[:h], ref[:h])
    assert np.array_equal(nv12[h:].reshape(h // 2, w // 2, 2)[..., 0].ravel(), ref.ravel()[h * w:h * w + h * w // 4])


def test_inferno_table_is_cv2s():
    t = cv2.applyColorMap(np.arange(256, dtype=np.uint8)[None], cv2.COLORMAP_INFERNO)[0, :, ::-1]
    assert INFERNO.dtype == np.uint8 and INFERNO.shape == (256, 3)
    assert np.array_equal(INFERNO, t) and tuple(INFERNO[0]) == (0, 0, 4)


def _reference_q(d, lo, hi):
    return ((d - lo) / (hi - lo) * 255).astype(np.uint8)


def test_level_equals_reference_on_random_data():
    rng = np.random.default_rng(0)
    for scale in (1e-3, 1.0, 37.5, 1e4):
        d = (rng.random((64, 257)) * scale).astype(np.float32) + np.float32(scale * 0.1)
        lo, hi = d.min(), d.max()
        assert np.array_equal(O.level(d, lo, hi), _reference_q(d, lo, hi))
        assert np.array_equal(O.save_video_frames(d[None], INFERNO)[0], INFERNO[_reference_q(d, lo, hi)])


def test_level_at_boundaries():
    for lo, hi in [(np.float32(0.1), np.float32(7.3)), (np.float32(-3.0), np.float32(1e-2)), (np.float32(2.0), np.float32(3.0))]:
        j = np.arange(256, dtype=np.float32)
        b = (lo + j * (hi - lo) / np.float32(255)).astype(np.float32)
        d = np.concatenate([b, np.nextafter(b, np.float32(np.inf)), np.nextafter(b, np.float32(-np.inf))])
        d = np.clip(d, lo, hi).astype(np.float32)
        assert np.array_equal(O.level(d, lo, hi), _reference_q(d, lo, hi))


def test_level_fixed_range_clamps_and_constant_is_zero():
    d = np.array([-1e30, -5.0, 0.0, 0.5, 1.0, 2.0, 1e30], np.float32)
    assert O.level(d, 0.0, 1.0).tolist() == [0, 0, 0, 127, 255, 255, 255]
    assert not O.level(np.full((4, 4), 3.0, np.float32), 3.0, 3.0).any()
    assert not O.colorize(np.full((2, 4, 4), 3.0, np.float32), INFERNO, "video", "gray").any()


def test_color_planes_struct_layout(tmp_path):
    """COLOR_PLANES (numpy) has the C layout of vda_color_planes (checked against a gcc probe)."""
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = ('#include "vda.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu %zu %zu %d %d", sizeof(vda_color_planes), '
           '__builtin_offsetof(vda_color_planes, pitch), __builtin_offsetof(vda_color_planes, H0), '
           '__builtin_offsetof(vda_color_planes, format), __builtin_offsetof(vda_color_planes, reserved), '
           'VDA_PIX_RGB, VDA_PIX_GRAY);return 0;}')
    (tmp_path / "p.c").write_text(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(tmp_path / "p.c"), "-o",
                           str(tmp_path / "p")])
    size, off_pitch, off_h, off_fmt, off_res, rgb, gray = map(int, subprocess.check_output([str(tmp_path / "p")]).split())
    assert size == COLOR_PLANES.itemsize == ops.COLOR_PLANES_BYTES == 64
    f = COLOR_PLANES.fields
    assert (f["pitch"][1], f["H0"][1], f["format"][1], f["reserved"][1]) == (off_pitch, off_h, off_fmt, off_res)
    assert (rgb, gray) == (_lib.PIX_RGB, _lib.PIX_GRAY)
    for name in ("vda_depth_range", "vda_colorize_depth", "vda_depth_range_scratch_bytes"):
        assert name in _lib.EXPORTS
    assert "#define VDA_RANGE_PARTIALS %d" % ops.RANGE_PARTIALS in open(os.path.join(ROOT, "include", "vda.h")).read()


def test_color_descriptors_and_layout():
    base = 1 << 40
    cd = color_descriptors(4, [(base, 6, 10), (base + 90, 4, 2)], 1)
    assert cd[0]["plane"].tolist() == [base, base + 60, 0] and cd[0]["pitch"].tolist() == [10, 10, 0]
    assert cd[1]["format"] == 1 and cd[2]["H0"] == 0 and not cd[3].tolist()[2]
    cd = color_descriptors(1, [(base, 6, 10)], 2)
    assert cd[0]["plane"].tolist() == [base, base + 60, base + 75] and cd[0]["pitch"].tolist() == [10, 5, 5]
    cd = color_descriptors(1, [(base, 5, 7)], 0)
    assert cd[0]["pitch"].tolist() == [21, 0, 0]
    assert color_descriptors(1, [(base, 5, 7)], 3)[0]["pitch"].tolist() == [7, 0, 0]
    with pytest.raises(ValueError):
        color_descriptors(1, [(base, 5, 8)], 1)
    with pytest.raises(ValueError):
        color_descriptors(1, [(base, 4, 8)] * 2, 1)
    assert color_frame_shape(4, 6, 0) == (4, 6, 3) and color_frame_shape(4, 6, 3) == (4, 6)
    assert color_frame_shape(4, 6, 1) == (6, 6) == color_frame_shape(4, 6, 2)
    for bk in (1, 2, 3, 16):
        for fmt in ("rgb", "nv12"):
            cs = group_color_layout(bk, 31, fmt)
            assert cs.start >= group_block_layout(bk, 31, fmt)[2].stop and cs.start % 64 == 0
            assert cs.stop - cs.start == 64 * bk


def test_color_args():
    assert color_args("depth", "inferno", "frame") == (None, None, "frame")
    fmt, table, rng = color_args("rgb", "inferno", (0, 2))
    assert fmt == 0 and table is INFERNO and rng == (0.0, 2.0)
    assert color_args("gray")[1] is None and color_args("gray", None)[1] is None
    t = np.zeros((256, 3), np.uint8)
    assert color_args("nv12", t, "video")[1] is not t and np.array_equal(color_args("nv12", t)[1], t)
    assert np.array_equal(color_args("i420", torch.zeros(256, 3, dtype=torch.uint8))[1], t)


BAD_ARGS = [dict(pixel_format="yuv444"), dict(pixel_format="depth"), dict(colormap="viridis"),
            dict(colormap=np.zeros((256, 3), np.float32)), dict(colormap=np.zeros((255, 3), np.uint8)),
            dict(colormap=np.zeros((256, 3), np.uint8), pixel_format="gray"), dict(value_range="clip"),
            dict(value_range=(1.0, 1.0)), dict(value_range=(2.0, 1.0)), dict(value_range=(0.0, np.inf)),
            dict(value_range=(0.0,)), dict(value_range=None)]


@pytest.mark.parametrize("kw", BAD_ARGS)
def test_colorize_rejects_bad_arguments(kw):
    d = np.random.default_rng(0).random((3, 8, 10)).astype(np.float32)
    before = d.copy()
    with pytest.raises(ValueError):
        colorize(d, **kw)
    assert np.array_equal(d, before)


@pytest.mark.parametrize("d, fmt", [(np.zeros((3, 8, 10), np.float64), "rgb"), (np.zeros((2, 3, 8, 10), np.float32), "rgb"),
                                    (np.zeros(10, np.float32), "rgb"), (np.zeros((0, 8, 10), np.float32), "rgb"),
                                    (np.zeros((3, 7, 10), np.float32), "nv12"), (np.zeros((9, 10), np.float32), "i420"),
                                    (np.zeros((8, 9), np.float32), "nv12"), (torch.zeros(3, 8, 10), "rgb"),
                                    ([[0.0, 1.0]], "rgb")])
def test_colorize_rejects_bad_depths(d, fmt):
    with pytest.raises(ValueError):
        colorize(d, pixel_format=fmt)


def _stub_group(max_streams=2, **kw):
    eng = types.SimpleNamespace(device=torch.device("cuda", 0), generation=0, loaded=True)
    model = types.SimpleNamespace(num_frames=32)
    return DepthStreamGroup(model, eng, max_streams, 56, **kw)


@pytest.mark.parametrize("kw", [dict(output_format="yuv"), dict(output_format="rgb", value_range="video"),
                                dict(output_format="nv12", value_range=(3.0, 3.0)), dict(output_format="gray",
                                colormap=np.zeros((256, 3), np.uint8)), dict(output_format="rgb", colormap="jet"),
                                dict(output_format="rgb", colormap=np.zeros((256, 4), np.uint8))])
def test_group_rejects_bad_color_arguments(kw):
    with pytest.raises(ValueError):
        _stub_group(**kw)


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_group_rejects_odd_frames_for_yuv_output_before_planning(fmt):
    g = _stub_group(output_format=fmt)
    a, b = g.open(), g.open()
    for bad in (np.zeros((51, 70, 3), np.uint8), np.zeros((50, 71, 3), np.uint8), np.zeros((2, 51, 70, 3), np.uint8)):
        before = (dict(g.plan.t), dict(g.plan.size), g.plan.net)
        with pytest.raises(ValueError):
            g.push({a: np.zeros((50, 70, 3), np.uint8), b: bad})
        assert (dict(g.plan.t), dict(g.plan.size), g.plan.net) == before
        assert g.pool is None


def test_depth_group_keeps_its_block_layout():
    g = _stub_group()
    assert g.color == (None, None, "frame") and g.output_format == "depth"
    assert group_block_layout(4, 31) == (slice(0, 96), slice(96, 160), slice(160, 720))


@pytest.mark.skipif(shutil.which("gcc") is None, reason="no gcc")
def test_c_host_colorize_compiles(tmp_path):
    """tests/c_host/host_stream_colorize.c is C99 against include/vda.h alone (compiled, not linked: no GPU needed)."""
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(cuda, "include"), "-c",
                           os.path.join(ROOT, "tests", "c_host", "host_stream_colorize.c"), "-o", str(tmp_path / "h.o")])


def test_colorize_cu_compiles_for_sm100a(tmp_path):
    """csrc/colorize.cu compiles for sm_100a with the library's flags, without spills."""
    from video_depth_anything_b200 import build
    nvcc = build._nvcc()
    if shutil.which(nvcc) is None and not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, "-Xptxas=-v", "-c", os.path.join(build.CSRC, "colorize.cu"), "-o",
                        str(tmp_path / "c.o")], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    assert "colorize_kernel" in r.stdout and "depth_range_partial_kernel" in r.stdout
    assert all(" 0 bytes spill stores, 0 bytes spill loads" in ln for ln in r.stdout.splitlines() if "spill" in ln)
