// Depth frames for displays and encoders (utils/dc_utils.py:72-86 save_video): fp32 depth -> 8-bit level -> colour table
// -> packed RGB, 8-bit grey, or YUV 4:2:0 (NV12 / I420, BT.601 limited range, cv2.cvtColor(COLOR_RGB2YUV_I420)'s integer
// form with top-left chroma), written pitched into the caller's planes.
//
// The reference normalises by the video's min / max and colour-maps in NumPy on the host, frame by frame.  Here two
// launches do it for a ragged batch in device memory: depth_range_partial_kernel + depth_range_fold_kernel (per-row or
// all-rows min / max; exact and order-independent, so bit-reproducible) and colorize_kernel (level, table, format).
// Every per-row address and size is read from descriptors in device memory, so a captured graph replays any mix of
// frame sizes.  Levels use __fsub_rn / __fdiv_rn / __fmul_rn: the library is built with --use_fast_math, under which
// plain operators would not be IEEE, and the level must equal NumPy's float32 arithmetic at every boundary.
#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

static_assert(sizeof(vda_color_planes) == 64, "vda_color_planes is 64 bytes (include/vda.h)");

constexpr int kRangeThreads = 256;
constexpr int kColorThreads = 256;

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// (min, max) over the block: every thread passes its (lo, hi); thread 0 gets the result.
__device__ __forceinline__ void block_min_max(float& lo, float& hi) {
  __shared__ float s_lo[32], s_hi[32];
  lo = warp_min(lo);
  hi = warp_max(hi);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) {
    s_lo[w] = lo;
    s_hi[w] = hi;
  }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    lo = l < nw ? s_lo[l] : INFINITY;
    hi = l < nw ? s_hi[l] : -INFINITY;
    lo = warp_min(lo);
    hi = warp_max(hi);
  }
}

// Block (p, r) folds its strided share of row r's H0 * W0 depths into partial[r][p] = (min, max); an empty share (or a
// pad row, H0 == 0) gives (+inf, -inf), the identity of the fold.  16-byte loads when the row is 16-byte aligned.
__global__ void __launch_bounds__(kRangeThreads)
depth_range_partial_kernel(const vda_out_desc* __restrict__ rows, float2* __restrict__ partial) {
  const vda_out_desc r = rows[blockIdx.y];
  const long long n = static_cast<long long>(max(r.H0, 0)) * max(r.W0, 0);
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long nthr = static_cast<long long>(gridDim.x) * blockDim.x;
  float lo = INFINITY, hi = -INFINITY;
  if (n > 0) {
    const float* __restrict__ d = r.dst;
    long long head = 0;
    if ((reinterpret_cast<uintptr_t>(d) & 15) == 0) {
      const float4* __restrict__ d4 = reinterpret_cast<const float4*>(d);
      const long long n4 = n >> 2;
      for (long long i = tid; i < n4; i += nthr) {
        const float4 v = __ldcs(d4 + i);
        lo = fminf(lo, fminf(fminf(v.x, v.y), fminf(v.z, v.w)));
        hi = fmaxf(hi, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
      }
      head = n4 << 2;
    }
    for (long long i = head + tid; i < n; i += nthr) {
      const float v = __ldcs(d + i);
      lo = fminf(lo, v);
      hi = fmaxf(hi, v);
    }
  }
  block_min_max(lo, hi);
  if (threadIdx.x == 0) partial[static_cast<long long>(blockIdx.y) * gridDim.x + blockIdx.x] = make_float2(lo, hi);
}

// Block j folds `count` partials starting at partial[j * count] into range[j] = (min, max).
__global__ void __launch_bounds__(kRangeThreads)
depth_range_fold_kernel(const float2* __restrict__ partial, int count, float2* __restrict__ range) {
  const float2* p = partial + static_cast<long long>(blockIdx.x) * count;
  float lo = INFINITY, hi = -INFINITY;
  for (int i = threadIdx.x; i < count; i += blockDim.x) {
    const float2 v = p[i];
    lo = fminf(lo, v.x);
    hi = fmaxf(hi, v.y);
  }
  block_min_max(lo, hi);
  if (threadIdx.x == 0) range[blockIdx.x] = make_float2(lo, hi);
}

// The 8-bit level of one depth (include/vda.h vda_colorize_depth): trunc(((d - lo) / (hi - lo)) * 255) clamped to
// 0..255, each operation IEEE round-to-nearest in this order; 0 everywhere when hi <= lo.  (__float2int_rz saturates,
// so values far outside a fixed range clamp too.)
__device__ __forceinline__ int depth_level(float d, float lo, float hi) {
  if (!(hi > lo)) return 0;
  const float t = __fmul_rn(__fdiv_rn(__fsub_rn(d, lo), __fsub_rn(hi, lo)), 255.f);
  return min(255, max(0, __float2int_rz(t)));
}

// BT.601 limited range, cv2.cvtColor(COLOR_RGB2YUV_I420)'s integer form (equal to cv2 on every (R, G, B) triple).
// Every sum is in 0 .. 2^28, so int32 and >> are exact.
__device__ __forceinline__ uint8_t rgb_to_y(int r, int g, int b) {
  return static_cast<uint8_t>((269484 * r + 528482 * g + 102760 * b + (16 << 20) + (1 << 19)) >> 20);
}
__device__ __forceinline__ uint8_t rgb_to_u(int r, int g, int b) {
  return static_cast<uint8_t>((-155188 * r - 305135 * g + 460324 * b + (128 << 20) + (1 << 19)) >> 20);
}
__device__ __forceinline__ uint8_t rgb_to_v(int r, int g, int b) {
  return static_cast<uint8_t>((460324 * r - 385875 * g - 74448 * b + (128 << 20) + (1 << 19)) >> 20);
}

// One 2 x 2 block of one frame: pixels (y0 + i, x0 + j) for i, j < 2 that lie inside the H0 x W0 frame (RGB and grey
// frames may have an odd size; YUV frames are even).  Chroma of a YUV block is that of its top-left pixel.
template <int FMT>
__device__ __forceinline__ void colorize_block(const float* __restrict__ src, const vda_color_planes& o, int H0, int W0,
                                               int y0, int x0, float lo, float hi, const uint8_t* __restrict__ lut) {
  const bool two_x = x0 + 1 < W0;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int y = y0 + i;
    if (y >= H0) break;
    const float* s = src + static_cast<long long>(y) * W0 + x0;
    const int q0 = depth_level(__ldcs(s), lo, hi);
    const int q1 = two_x ? depth_level(__ldcs(s + 1), lo, hi) : 0;
    if (FMT == VDA_PIX_GRAY) {
      uint8_t* g = o.plane[0] + y * o.pitch[0] + x0;
      g[0] = static_cast<uint8_t>(q0);
      if (two_x) g[1] = static_cast<uint8_t>(q1);
    } else if (FMT == VDA_PIX_RGB) {
      uint8_t* p = o.plane[0] + y * o.pitch[0] + 3 * x0;
      p[0] = lut[3 * q0];
      p[1] = lut[3 * q0 + 1];
      p[2] = lut[3 * q0 + 2];
      if (two_x) {
        p[3] = lut[3 * q1];
        p[4] = lut[3 * q1 + 1];
        p[5] = lut[3 * q1 + 2];
      }
    } else {
      const int r0 = lut[3 * q0], g0 = lut[3 * q0 + 1], b0 = lut[3 * q0 + 2];
      const int r1 = lut[3 * q1], g1 = lut[3 * q1 + 1], b1 = lut[3 * q1 + 2];
      uchar2 yy;
      yy.x = rgb_to_y(r0, g0, b0);
      yy.y = rgb_to_y(r1, g1, b1);
      uint8_t* py = o.plane[0] + y * o.pitch[0] + x0;
      py[0] = yy.x;
      py[1] = yy.y;
      if (i == 0) {
        const int cy = y0 >> 1;
        const uint8_t u = rgb_to_u(r0, g0, b0), v = rgb_to_v(r0, g0, b0);
        if (FMT == VDA_PIX_NV12) {
          uint8_t* uv = o.plane[1] + cy * o.pitch[1] + x0;
          uv[0] = u;
          uv[1] = v;
        } else {
          o.plane[1][cy * o.pitch[1] + (x0 >> 1)] = u;
          o.plane[2][cy * o.pitch[2] + (x0 >> 1)] = v;
        }
      }
    }
  }
}

// Row blockIdx.y: the ceil(H0/2) x ceil(W0/2) blocks of 2 x 2 pixels, grid-strided over the gridDim.x blocks of the
// row.  The format is per row (a branch uniform over a row), the colour table is staged in shared memory.
__global__ void __launch_bounds__(kColorThreads)
colorize_kernel(const vda_out_desc* __restrict__ src, const vda_color_planes* __restrict__ dst, const float2* __restrict__ range,
                int range_per_row, const uint8_t* __restrict__ table) {
  __shared__ uint8_t lut[768];
  if (table != nullptr)
    for (int i = threadIdx.x; i < 768; i += blockDim.x) lut[i] = table[i];
  __syncthreads();
  const int row = blockIdx.y;
  const vda_color_planes o = dst[row];
  const int H0 = o.H0, W0 = o.W0;
  if (H0 <= 0 || W0 <= 0) return;
  const float* __restrict__ d = src[row].dst;
  const float2 rg = range[range_per_row ? row : 0];
  const int bw = (W0 + 1) >> 1;
  const long long nblk = static_cast<long long>((H0 + 1) >> 1) * bw;
  for (long long b = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; b < nblk;
       b += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int y0 = static_cast<int>(b / bw) * 2, x0 = static_cast<int>(b % bw) * 2;
    switch (o.format) {
      case VDA_PIX_GRAY: colorize_block<VDA_PIX_GRAY>(d, o, H0, W0, y0, x0, rg.x, rg.y, lut); break;
      case VDA_PIX_NV12: colorize_block<VDA_PIX_NV12>(d, o, H0, W0, y0, x0, rg.x, rg.y, lut); break;
      case VDA_PIX_I420: colorize_block<VDA_PIX_I420>(d, o, H0, W0, y0, x0, rg.x, rg.y, lut); break;
      default: colorize_block<VDA_PIX_RGB>(d, o, H0, W0, y0, x0, rg.x, rg.y, lut); break;
    }
  }
}

}  // namespace vda

using namespace vda;

extern "C" int64_t vda_depth_range_scratch_bytes(int n) {
  if (n <= 0) return -1;
  return static_cast<int64_t>(n) * VDA_RANGE_PARTIALS * 2 * sizeof(float);
}

extern "C" int vda_depth_range(const vda_out_desc* rows, int n, int all_rows, float* range, void* scratch, void* stream) {
  VDA_CHECK(n > 0 && n <= 65535, "depth_range: n = %d rows, want 1..65535", n);
  VDA_CHECK(rows != nullptr && range != nullptr && scratch != nullptr, "depth_range: null pointer");
  VDA_CHECK(reinterpret_cast<uintptr_t>(range) % 8 == 0 && reinterpret_cast<uintptr_t>(scratch) % 8 == 0,
            "depth_range: range and scratch must be 8-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float2* partial = static_cast<float2*>(scratch);
  depth_range_partial_kernel<<<dim3(VDA_RANGE_PARTIALS, n), kRangeThreads, 0, st>>>(rows, partial);
  VDA_CUDA(cudaGetLastError());
  if (all_rows)
    depth_range_fold_kernel<<<1, kRangeThreads, 0, st>>>(partial, n * VDA_RANGE_PARTIALS, reinterpret_cast<float2*>(range));
  else
    depth_range_fold_kernel<<<n, kRangeThreads, 0, st>>>(partial, VDA_RANGE_PARTIALS, reinterpret_cast<float2*>(range));
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_colorize_depth(const vda_out_desc* src, const vda_color_planes* dst, int n, const float* range,
                                  int range_per_row, const uint8_t* table, void* stream) {
  VDA_CHECK(n > 0 && n <= 65535, "colorize_depth: n = %d rows, want 1..65535", n);
  VDA_CHECK(src != nullptr && dst != nullptr && range != nullptr, "colorize_depth: null pointer");
  VDA_CHECK(reinterpret_cast<uintptr_t>(range) % 8 == 0, "colorize_depth: range must be 8-byte aligned");
  // ~8 resident blocks per SM over the batch; each block strides over its row
  const int gx = max(1, min(1024, (148 * 8 + n - 1) / n));
  colorize_kernel<<<dim3(gx, n), kColorThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      src, dst, reinterpret_cast<const float2*>(range), range_per_row, table);
  VDA_CUDA(cudaGetLastError());
  return 0;
}
