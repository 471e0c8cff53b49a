"""B200-native (sm_100a) inference engine for the Video-Depth-Anything hot path.

`VideoDepthAnything` mirrors the reference module (video_depth_anything/video_depth.py); all arithmetic runs in
libvda.so (hand-written CUDA: tcgen05/TMEM/TMA GEMMs and implicit-GEMM convs, fused attention, norms, resampling,
alignment) reached through the C ABI in include/vda.h."""
from .synth import MODEL_CONFIGS, synth_state_dict  # noqa: F401
from .video_depth import DepthStream, DepthStreamGroup, VideoDepthAnything  # noqa: F401

__all__ = ["VideoDepthAnything", "DepthStream", "DepthStreamGroup", "MODEL_CONFIGS", "synth_state_dict"]
