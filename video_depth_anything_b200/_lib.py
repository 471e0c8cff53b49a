"""ctypes binding of libvda.so (include/vda.h).  There is no fallback: if the shared library is missing the
import fails loudly, and every call that returns non-zero raises with the library's own message."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# VDA_LIB: debug hook (tools/build_variant.sh) -- another build of the same library, e.g. with different nvcc flags
LIB_PATH = os.environ.get("VDA_LIB") or os.path.join(HERE, "libvda.so")

VDA_BF16, VDA_FP16 = 0, 1
ACT_NONE, ACT_GELU, ACT_RELU = 0, 1, 2
EPI_LINEAR, EPI_GEGLU, EPI_CONVT, EPI_TAIL = 0, 1, 2, 3
A_PLAIN, A_CONV3 = 0, 1
PIX_RGB, PIX_NV12, PIX_I420, PIX_GRAY = 0, 1, 2, 3   # vda_frame_planes / vda_color_planes .format (VDA_PIX_*)


class VdaError(RuntimeError):
    pass


class GemmParams(C.Structure):
    _fields_ = [
        ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
        ("dtype", C.c_int32), ("a_mode", C.c_int32), ("epilogue", C.c_int32),
        ("A", C.c_void_p), ("lda", C.c_int64), ("Wt", C.c_void_p),
        ("n_img", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32),
        ("bias", C.c_void_p), ("gamma", C.c_void_p), ("act", C.c_int32),
        ("res1", C.c_void_p), ("ldr1", C.c_int64), ("res1_f32", C.c_int32),
        ("res2", C.c_void_p), ("out", C.c_void_p), ("ldo", C.c_int64), ("out_f32", C.c_int32),
        ("out_relu", C.c_void_p), ("row_group", C.c_int32), ("geglu_half", C.c_int32),
        ("convt_s", C.c_int32), ("convt_co", C.c_int32), ("in_h", C.c_int32), ("in_w", C.c_int32),
        ("tail_w", C.c_void_p), ("tail_b", C.c_float),
        ("out16", C.c_void_p), ("row_stats_out", C.c_void_p), ("row_stats_in", C.c_void_p), ("ln_c1", C.c_void_p),
        ("stat_parts", C.c_int32), ("stat_cols", C.c_int32), ("ln_eps", C.c_float),
        ("a_k", C.c_int32),
    ]


_SIGS = {
    "vda_version": (C.c_int, []),
    "vda_last_error": (C.c_char_p, []),
    "vda_device_query": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vda_gemm": (C.c_int, [C.POINTER(GemmParams), C.c_void_p]),
    "vda_gemm_rowstat_layout": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vda_layernorm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int64, C.c_int,
                                C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "vda_rowstats_cast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p]),
    "vda_groupnorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_int,
                                C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "vda_attention_spatial": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_attention_temporal": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_attention_temporal_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                              C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_attention_temporal_step_batched": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 8 + [C.c_void_p]),
    "vda_attention_temporal_step_causal": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 8 + [C.c_void_p]),
    "vda_stream_cache_store": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 7 + [C.c_void_p]),
    "vda_preprocess_frames": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p]),
    "vda_preprocess_frames_ragged": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vda_preprocess_frames_yuv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_void_p]),
    "vda_preprocess_frames_planes": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "vda_copy_frames": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]),
    "vda_eval_sequence": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "vda_eval_aligned_depth": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int64, C.c_void_p, C.c_void_p]),
    "vda_eval_tae": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vda_patch_im2col": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_write_cls": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_pos_embed_bicubic": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_im2col3x3_s2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_bilinear_nhwc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p]),
    "vda_tail_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_bilinear_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_bilinear_f32_ragged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "vda_add_h16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "vda_lsq_scale_shift": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vda_align_chain": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vda_create": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vda_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int]),
    "vda_finalize_weights": (C.c_int, [C.c_void_p]),
    "vda_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "vda_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_void_p]),
    "vda_destroy": (C.c_int, [C.c_void_p]),
    "vda_stream_plan_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "vda_stream_plan_buckets": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_int, C.POINTER(C.c_int)]),
    "vda_stream_plan_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "vda_stream_plan_close": (C.c_int, [C.c_void_p, C.c_int64]),
    "vda_stream_plan_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64,
                                       C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vda_stream_plan_destroy": (C.c_int, [C.c_void_p]),
    "vda_resize_hw": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vda_stream_pool_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "vda_stream_workspace_bytes": (C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "vda_stream_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                  C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "vda_stream_step_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                         C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "vda_depth_range_scratch_bytes": (C.c_int64, [C.c_int]),
    "vda_depth_range": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "vda_colorize_depth": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "vda_affine_clamp_blend": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64,
                                         C.c_void_p]),
}

EXPORTS = tuple(_SIGS)

_lib = None


def load() -> C.CDLL:
    """dlopen libvda.so (built in-tree by video_depth_anything_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise VdaError(f"{LIB_PATH} is missing: the CUDA extension has not been built "
                       f"(run `python -m video_depth_anything_b200.build`); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise VdaError(load().vda_last_error().decode(errors="replace") or f"libvda error {rc}")
