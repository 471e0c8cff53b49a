// Device-side frame preprocessing of the long-video driver (video_depth.py:173-185,197-198 with util/transform.py:109-158):
//
//   uint8 RGB frame -> float32 / 255 -> cv2.resize(INTER_CUBIC) to (nh, nw) -> (x - mean) / std in float64 -> CHW float32
//
// The reference does this on the host, frame by frame, 32 cv2 calls per window.  Here one kernel produces the whole
// [n, 3, nh, nw] window tensor from device-resident uint8 frames selected by an index list (the closed-form window
// gather of windows.window_source_indices), so a window costs one launch and no host work.
// The ragged form (stream groups) takes one frame per batch row, each of its own size and pitch, from per-row descriptors
// in device memory, so a captured graph replays it whatever frames a later push brings.
// cv2's INTER_CUBIC on float32 (A = -0.75): src coordinate fx = (dx + 0.5) * (src / dst) - 0.5, taps floor(fx)-1 ..
// floor(fx)+2 with replicated borders, horizontal pass then vertical pass in float32; a same-size resize is the
// identity (weights 0,1,0,0).  Differences to cv2 are last-bit (SIMD summation order): tests compare at 1e-5.
#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

__device__ __forceinline__ void cubic_coeffs(float x, float (&c)[4]) {
  const float A = -0.75f;
  c[0] = ((A * (x + 1.f) - 5.f * A) * (x + 1.f) + 8.f * A) * (x + 1.f) - 4.f * A;
  c[1] = ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f;
  c[2] = ((A + 2.f) * (1.f - x) - (A + 3.f)) * (1.f - x) * (1.f - x) + 1.f;
  c[3] = 1.f - c[0] - c[1] - c[2];
}

// One output pixel (dy, dx) of one frame: src row y starts at src + y * pitch, pixels are 3 bytes; writes the three
// channel planes of o (plane = nh * nw floats apart).  Shared by the uniform and the ragged kernel, so a frame gives the
// same bits through either.
__device__ __forceinline__ void preprocess_pixel(const uint8_t* __restrict__ src, long long pitch, int H0, int W0, int nh,
                                                 int nw, double scale_y, double scale_x, int dy, int dx,
                                                 float* __restrict__ o, long long plane) {
  const double mean[3] = {0.485, 0.456, 0.406}, stdv[3] = {0.229, 0.224, 0.225};
  float v[3];
  if (H0 == nh && W0 == nw) {
    const uint8_t* px = src + dy * pitch + dx * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) v[c] = __fdiv_rn(static_cast<float>(px[c]), 255.f);
  } else {
    float fx = static_cast<float>((dx + 0.5) * scale_x - 0.5);
    float fy = static_cast<float>((dy + 0.5) * scale_y - 0.5);
    const int sx = static_cast<int>(floorf(fx)), sy = static_cast<int>(floorf(fy));
    fx -= sx;
    fy -= sy;
    float cx[4], cy[4];
    cubic_coeffs(fx, cx);
    cubic_coeffs(fy, cy);
    v[0] = v[1] = v[2] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int yy = min(max(sy - 1 + j, 0), H0 - 1);
      float row[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int xx = min(max(sx - 1 + i, 0), W0 - 1);
        const uint8_t* px = src + yy * pitch + xx * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) row[c] = __fmaf_rn(__fdiv_rn(static_cast<float>(px[c]), 255.f), cx[i], row[c]);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = __fmaf_rn(row[c], cy[j], v[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c * plane] = static_cast<float>((static_cast<double>(v[c]) - mean[c]) / stdv[c]);
}

__global__ void __launch_bounds__(256)
preprocess_kernel(const uint8_t* __restrict__ frames, const int* __restrict__ idx, float* __restrict__ out, int n, int H0,
                  int W0, int nh, int nw, double scale_y, double scale_x) {
  const long long total = static_cast<long long>(n) * nh * nw;
  const long long plane = static_cast<long long>(nh) * nw;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int dx = static_cast<int>(t % nw);
    const int dy = static_cast<int>((t / nw) % nh);
    const int f = static_cast<int>(t / plane);
    const uint8_t* src = frames + static_cast<long long>(idx[f]) * H0 * W0 * 3;
    preprocess_pixel(src, static_cast<long long>(W0) * 3, H0, W0, nh, nw, scale_y, scale_x, dy, dx,
                     out + static_cast<long long>(f) * 3 * plane + static_cast<long long>(dy) * nw + dx, plane);
  }
}

// Ragged batch: row f has its own frame (rows[f]: address, row pitch, size), all rows go to one (nh, nw).  The scales
// are the uniform kernel's host divisions, done here in IEEE double (__ddiv_rn), so each row's bits equal the uniform
// kernel's on that frame alone.
__global__ void __launch_bounds__(256)
preprocess_ragged_kernel(const vda_frame_desc* __restrict__ rows, float* __restrict__ out, int n, int nh, int nw) {
  const long long total = static_cast<long long>(n) * nh * nw;
  const long long plane = static_cast<long long>(nh) * nw;
  for (long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int dx = static_cast<int>(t % nw);
    const int dy = static_cast<int>((t / nw) % nh);
    const int f = static_cast<int>(t / plane);
    const vda_frame_desc r = rows[f];
    preprocess_pixel(r.src, r.pitch, r.H0, r.W0, nh, nw, __ddiv_rn(r.H0, nh), __ddiv_rn(r.W0, nw), dy, dx,
                     out + static_cast<long long>(f) * 3 * plane + static_cast<long long>(dy) * nw + dx, plane);
  }
}

// Gather / scatter of whole per-frame slabs (encoder-feature cache of the long-video driver): frame i of the copy goes
// from src slab src_idx[i] to dst slab dst_idx[i] (a null index list = identity).  One 16-byte vector per thread.
__global__ void __launch_bounds__(256)
copy_frames_kernel(const uint4* __restrict__ src, const int* __restrict__ src_idx, uint4* __restrict__ dst,
                   const int* __restrict__ dst_idx, long long vec_per_frame) {
  const int f = blockIdx.y;
  const uint4* s = src + static_cast<long long>(src_idx ? src_idx[f] : f) * vec_per_frame;
  uint4* d = dst + static_cast<long long>(dst_idx ? dst_idx[f] : f) * vec_per_frame;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < vec_per_frame;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    d[i] = s[i];
}

}  // namespace vda

using namespace vda;

extern "C" int vda_copy_frames(const void* src, const int32_t* src_idx, void* dst, const int32_t* dst_idx, int n,
                               int64_t frame_bytes, void* stream) {
  VDA_CHECK(n > 0 && frame_bytes > 0 && frame_bytes % 16 == 0, "copy_frames: frame size must be a positive multiple of 16 B");
  VDA_CHECK((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) % 16 == 0, "copy_frames: unaligned pointer");
  const long long vec = frame_bytes / 16;
  long long gx = (vec + 256 * 4 - 1) / (256 * 4);
  if (gx < 1) gx = 1;
  if (gx > 148 * 8) gx = 148 * 8;
  copy_frames_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(n)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(src), src_idx, static_cast<uint4*>(dst), dst_idx, vec);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_preprocess_frames(const uint8_t* frames, const int32_t* idx, float* out, int n, int H0, int W0, int nh,
                                     int nw, void* stream) {
  VDA_CHECK(n > 0 && H0 > 0 && W0 > 0 && nh > 0 && nw > 0, "preprocess: bad shape");
  const long long total = static_cast<long long>(n) * nh * nw;
  long long g = (total + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  preprocess_kernel<<<static_cast<unsigned>(g), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      frames, idx, out, n, H0, W0, nh, nw, static_cast<double>(H0) / nh, static_cast<double>(W0) / nw);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_preprocess_frames_ragged(const vda_frame_desc* rows, int n, int nh, int nw, float* out, void* stream) {
  VDA_CHECK(n > 0 && nh > 0 && nw > 0, "preprocess_ragged: bad shape");
  const long long total = static_cast<long long>(n) * nh * nw;
  long long g = (total + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  preprocess_ragged_kernel<<<static_cast<unsigned>(g), 256, 0, static_cast<cudaStream_t>(stream)>>>(rows, out, n, nh, nw);
  VDA_CUDA(cudaGetLastError());
  return 0;
}
