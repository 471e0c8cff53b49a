// Bandwidth-bound data-movement kernels: patch im2col, cls/pos-embed, bicubic pos-embed resampling,
// stride-2 im2col, bilinear (align_corners=True) resampling (also of a ragged batch), elementwise add.  All 128-bit
// vectorised along the contiguous (channel) dimension, grid-stride loops sized in multiples of the SM count.
#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

static inline unsigned grid_for(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  const long long cap = 148LL * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<unsigned>(g);
}

// ---- patch-embed im2col: x fp32 [F,3,H,W] -> A h16 [F*hp*wp, kpad]; column = c*196 + ky*14 + kx ----
template <typename T>
__global__ void patch_im2col_kernel(const float* __restrict__ x, T* __restrict__ A, int frames, int H, int W, int kpad) {
  const int hp = H / 14, wp = W / 14;
  const int kp2 = kpad / 2;
  const long long total = static_cast<long long>(frames) * hp * wp * kp2;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(idx % kp2) * 2;
    const long long row = idx / kp2;
    const int px = static_cast<int>(row % wp);
    const int py = static_cast<int>((row / wp) % hp);
    const int f = static_cast<int>(row / (static_cast<long long>(wp) * hp));
    float v0 = 0.f, v1 = 0.f;
    if (k < 588) {   // 14 is even, so (k, k+1) stay in one kernel row
      const int c = k / 196, rem = k - c * 196, ky = rem / 14, kx = rem - ky * 14;
      const float* src = x + ((static_cast<long long>(f) * 3 + c) * H + py * 14 + ky) * W + px * 14 + kx;
      const float2 v = *reinterpret_cast<const float2*>(src);
      v0 = v.x; v1 = v.y;
    }
    *reinterpret_cast<uint32_t*>(A + row * kpad + k) = H16<T>::pack2(v0, v1);
  }
}

__global__ void write_cls_kernel(float* __restrict__ tokens, const float* __restrict__ cls, const float* __restrict__ pos,
                                 int frames, int tpf, int D) {
  const int total = frames * D;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int f = idx / D, c = idx - f * D;
    tokens[static_cast<long long>(f) * tpf * D + c] = cls[c] + pos[c];
  }
}

// ---- bicubic (A = -0.75), PyTorch upsample_bicubic2d with explicit scale_factor, align_corners=False ----
__device__ __forceinline__ void cubic_coeffs(float t, float (&w)[4]) {
  const float A = -0.75f;
  float x = t + 1.f;
  w[0] = ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A;
  x = t;
  w[1] = ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f;
  x = 1.f - t;
  w[2] = ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f;
  x = 2.f - t;
  w[3] = ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A;
}

__global__ void pos_embed_bicubic_kernel(const float* __restrict__ pin, float* __restrict__ pout, int S, int hp, int wp,
                                         int D, float rscale_h, float rscale_w) {
  const long long total = static_cast<long long>(1 + hp * wp) * D;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % D);
    const int tok = static_cast<int>(idx / D);
    if (tok == 0) { pout[idx] = pin[c]; continue; }
    const int oy = (tok - 1) / wp, ox = (tok - 1) - oy * wp;
    // area_pixel_compute_source_index(scale, dst, align_corners=False, cubic=True): no clamp at 0
    const float sy = rscale_h * (oy + 0.5f) - 0.5f, sx = rscale_w * (ox + 0.5f) - 0.5f;
    const int iy = static_cast<int>(floorf(sy)), ix = static_cast<int>(floorf(sx));
    float wy[4], wx[4];
    cubic_coeffs(sy - iy, wy);
    cubic_coeffs(sx - ix, wx);
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int yy = min(max(iy - 1 + a, 0), S - 1);
      float r = 0.f;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int xx = min(max(ix - 1 + b, 0), S - 1);
        r += wx[b] * pin[static_cast<long long>(1 + yy * S + xx) * D + c];
      }
      acc += wy[a] * r;
    }
    pout[idx] = acc;
  }
}

// ---- im2col for 3x3 / stride 2 / pad 1 over NHWC: out [n*oh*ow, 9*C], column = (ky*3+kx)*C + ci ----
template <typename T>
__global__ void im2col3x3_s2_kernel(const T* __restrict__ in, T* __restrict__ out, int n, int H, int W, int C, int oh,
                                    int ow) {
  const int vecs = C / 8;
  const long long total = static_cast<long long>(n) * oh * ow * 9 * vecs;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int v = static_cast<int>(idx % vecs);
    long long r = idx / vecs;
    const int tap = static_cast<int>(r % 9);
    r /= 9;
    const int ox = static_cast<int>(r % ow);
    const int oy = static_cast<int>((r / ow) % oh);
    const int img = static_cast<int>(r / (static_cast<long long>(ow) * oh));
    const int iy = oy * 2 + tap / 3 - 1, ix = ox * 2 + tap % 3 - 1;
    uint4 val = make_uint4(0, 0, 0, 0);
    if (iy >= 0 && iy < H && ix >= 0 && ix < W)
      val = *reinterpret_cast<const uint4*>(in + ((static_cast<long long>(img) * H + iy) * W + ix) * C + v * 8);
    *reinterpret_cast<uint4*>(out + idx * 8) = val;
  }
}

// ---- bilinear, align_corners=True, NHWC h16 ----
// One CTA per output row: the vertical taps / weights are computed once per CTA, the threads walk the row's
// (pixel, 8-channel vector) units with 32-bit index math (a flat 64-bit div/mod version was ALU-bound at ~1 TB/s).
template <typename T>
__global__ void __launch_bounds__(256)
bilinear_nhwc_kernel(const T* __restrict__ in, T* __restrict__ out, int ih, int iw, int oh, int ow, int C, float sy,
                     float sx) {
  const int vecs = C >> 3;
  const int row = blockIdx.x;                 // img * oh + oy
  const int img = row / oh, oy = row - img * oh;
  const float fy = sy * oy;
  const int y0 = min(static_cast<int>(fy), ih - 1);
  const int y1 = min(y0 + 1, ih - 1);
  const float ly = fy - y0;
  const T* r0 = in + (static_cast<long long>(img) * ih + y0) * iw * C;
  const T* r1 = in + (static_cast<long long>(img) * ih + y1) * iw * C;
  T* o = out + static_cast<long long>(row) * ow * C;
  const int units = ow * vecs;
  for (int u = threadIdx.x; u < units; u += blockDim.x) {
    const int ox = u / vecs, v = u - ox * vecs;
    const float fx = sx * ox;
    const int x0 = min(static_cast<int>(fx), iw - 1), x1 = min(x0 + 1, iw - 1);
    const float lx = fx - x0;
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    const uint4 a00 = *reinterpret_cast<const uint4*>(r0 + x0 * C + v * 8);
    const uint4 a01 = *reinterpret_cast<const uint4*>(r0 + x1 * C + v * 8);
    const uint4 a10 = *reinterpret_cast<const uint4*>(r1 + x0 * C + v * 8);
    const uint4 a11 = *reinterpret_cast<const uint4*>(r1 + x1 * C + v * 8);
    const uint32_t p00[4] = {a00.x, a00.y, a00.z, a00.w}, p01[4] = {a01.x, a01.y, a01.z, a01.w};
    const uint32_t p10[4] = {a10.x, a10.y, a10.z, a10.w}, p11[4] = {a11.x, a11.y, a11.z, a11.w};
    uint32_t res[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f00 = H16<T>::unpack2(p00[i]), f01 = H16<T>::unpack2(p01[i]);
      const float2 f10 = H16<T>::unpack2(p10[i]), f11 = H16<T>::unpack2(p11[i]);
      res[i] = H16<T>::pack2(w00 * f00.x + w01 * f01.x + w10 * f10.x + w11 * f11.x,
                             w00 * f00.y + w01 * f01.y + w10 * f10.y + w11 * f11.y);
    }
    *reinterpret_cast<uint4*>(o + u * 8) = make_uint4(res[0], res[1], res[2], res[3]);
  }
}

__global__ void bilinear_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int n, int ih, int iw, int oh,
                                    int ow, float sy, float sx) {
  const long long total = static_cast<long long>(n) * oh * ow;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int ox = static_cast<int>(idx % ow);
    const int oy = static_cast<int>((idx / ow) % oh);
    const int img = static_cast<int>(idx / (static_cast<long long>(ow) * oh));
    const float fy = sy * oy, fx = sx * ox;
    const int y0 = min(static_cast<int>(fy), ih - 1), x0 = min(static_cast<int>(fx), iw - 1);
    const int y1 = min(y0 + 1, ih - 1), x1 = min(x0 + 1, iw - 1);
    const float ly = fy - y0, lx = fx - x0;
    const float* b = in + static_cast<long long>(img) * ih * iw;
    const float top = b[y0 * iw + x0] * (1.f - lx) + b[y0 * iw + x1] * lx;
    const float bot = b[y1 * iw + x0] * (1.f - lx) + b[y1 * iw + x1] * lx;
    out[idx] = top * (1.f - ly) + bot * ly;
  }
}

// Ragged batch: row f of in [n, ih, iw] goes to rows[f].dst at its own (H0, W0), grid (x, n) with a grid-stride loop
// over the row's pixels, so the launch does not depend on the sizes.  Same arithmetic as bilinear_f32_kernel; the
// scales are the host's IEEE divisions (__fdiv_rn: the library is built with --use_fast_math).  A row of the input's
// size is copied (the caller skipped the resize there before); H0 == 0 writes nothing (pad rows).
__global__ void __launch_bounds__(256)
bilinear_f32_ragged_kernel(const float* __restrict__ in, const vda_out_desc* __restrict__ rows, int ih, int iw) {
  const int img = blockIdx.y;
  const vda_out_desc r = rows[img];
  const int oh = r.H0, ow = r.W0;
  const long long total = static_cast<long long>(oh) * ow;
  const float* b = in + static_cast<long long>(img) * ih * iw;
  const bool same = oh == ih && ow == iw;
  const float sy = oh > 1 ? __fdiv_rn(static_cast<float>(ih - 1), static_cast<float>(oh - 1)) : 0.f;
  const float sx = ow > 1 ? __fdiv_rn(static_cast<float>(iw - 1), static_cast<float>(ow - 1)) : 0.f;
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (same) {
      r.dst[idx] = b[idx];
      continue;
    }
    const int ox = static_cast<int>(idx % ow);
    const int oy = static_cast<int>(idx / ow);
    const float fy = sy * oy, fx = sx * ox;
    const int y0 = min(static_cast<int>(fy), ih - 1), x0 = min(static_cast<int>(fx), iw - 1);
    const int y1 = min(y0 + 1, ih - 1), x1 = min(x0 + 1, iw - 1);
    const float ly = fy - y0, lx = fx - x0;
    const float top = b[y0 * iw + x0] * (1.f - lx) + b[y0 * iw + x1] * lx;
    const float bot = b[y1 * iw + x0] * (1.f - lx) + b[y1 * iw + x1] * lx;
    r.dst[idx] = top * (1.f - ly) + bot * ly;
  }
}

template <typename T>
__global__ void add_h16_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, long long nvec) {
  for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < nvec;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint4 x = reinterpret_cast<const uint4*>(a)[idx], y = reinterpret_cast<const uint4*>(b)[idx];
    const uint32_t xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
    uint32_t r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 p = H16<T>::unpack2(xs[i]), q = H16<T>::unpack2(ys[i]);
      r[i] = H16<T>::pack2(p.x + q.x, p.y + q.y);
    }
    reinterpret_cast<uint4*>(out)[idx] = make_uint4(r[0], r[1], r[2], r[3]);
  }
}

}  // namespace vda

using namespace vda;

extern "C" int vda_patch_im2col(const float* x, void* A, int frames, int H, int W, int kpad, int dtype, void* stream) {
  VDA_CHECK(H % 14 == 0 && W % 14 == 0, "Input image height %d / width %d is not a multiple of patch size 14", H, W);
  VDA_CHECK(kpad >= 588 && kpad % 8 == 0, "kpad must be >= 588 and a multiple of 8");
  VDA_CHECK(W % 2 == 0, "patch im2col needs an even width");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = static_cast<long long>(frames) * (H / 14) * (W / 14) * (kpad / 2);
  if (dtype == VDA_BF16)
    patch_im2col_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(x, static_cast<__nv_bfloat16*>(A), frames, H, W, kpad);
  else
    patch_im2col_kernel<__half><<<grid_for(total, 256), 256, 0, st>>>(x, static_cast<__half*>(A), frames, H, W, kpad);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_write_cls(float* tokens, const float* cls_token, const float* pos, int frames, int tokens_per_frame,
                             int D, void* stream) {
  write_cls_kernel<<<grid_for(static_cast<long long>(frames) * D, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      tokens, cls_token, pos, frames, tokens_per_frame, D);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_pos_embed_bicubic(const float* pos_in, float* pos_out, int S, int hp, int wp, int D, void* stream) {
  // scale_factor = ((hp+0.1)/S, (wp+0.1)/S) (dinov2.py:194-201); torch uses 1/scale_factor as the coordinate ratio
  const double sf_h = (hp + 0.1) / static_cast<double>(S), sf_w = (wp + 0.1) / static_cast<double>(S);
  const float rh = static_cast<float>(1.0 / sf_h), rw = static_cast<float>(1.0 / sf_w);
  const long long total = static_cast<long long>(1 + hp * wp) * D;
  pos_embed_bicubic_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(pos_in, pos_out, S, hp,
                                                                                                 wp, D, rh, rw);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_im2col3x3_s2(const void* in, void* out, int n, int H, int W, int C, int dtype, void* stream) {
  VDA_CHECK(C % 8 == 0, "im2col: C must be a multiple of 8");
  const int oh = (H + 2 - 3) / 2 + 1, ow = (W + 2 - 3) / 2 + 1;
  const long long total = static_cast<long long>(n) * oh * ow * 9 * (C / 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == VDA_BF16)
    im2col3x3_s2_kernel<__nv_bfloat16><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(in),
                                                                            static_cast<__nv_bfloat16*>(out), n, H, W, C, oh, ow);
  else
    im2col3x3_s2_kernel<__half><<<grid_for(total, 256), 256, 0, st>>>(static_cast<const __half*>(in), static_cast<__half*>(out),
                                                                     n, H, W, C, oh, ow);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_bilinear_nhwc(const void* in, void* out, int n, int ih, int iw, int oh, int ow, int C, int dtype,
                                 void* stream) {
  VDA_CHECK(C % 8 == 0, "bilinear: C must be a multiple of 8");
  const float sy = oh > 1 ? static_cast<float>(ih - 1) / (oh - 1) : 0.f;
  const float sx = ow > 1 ? static_cast<float>(iw - 1) / (ow - 1) : 0.f;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = static_cast<unsigned>(n) * oh;
  if (dtype == VDA_BF16)
    bilinear_nhwc_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(in),
                                                              static_cast<__nv_bfloat16*>(out), ih, iw, oh, ow, C, sy, sx);
  else
    bilinear_nhwc_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(in), static_cast<__half*>(out), ih, iw,
                                                       oh, ow, C, sy, sx);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_bilinear_f32(const float* in, float* out, int n, int ih, int iw, int oh, int ow, void* stream) {
  const float sy = oh > 1 ? static_cast<float>(ih - 1) / (oh - 1) : 0.f;
  const float sx = ow > 1 ? static_cast<float>(iw - 1) / (ow - 1) : 0.f;
  const long long total = static_cast<long long>(n) * oh * ow;
  bilinear_f32_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, n, ih, iw, oh, ow, sy, sx);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_bilinear_f32_ragged(const float* in, const vda_out_desc* rows, int n, int ih, int iw, void* stream) {
  VDA_CHECK(n > 0 && ih > 0 && iw > 0, "bilinear_f32_ragged: bad shape");
  // fixed grid (sizes live in device memory): about 8 CTAs per SM over the whole batch, at least one per row
  const unsigned gx = static_cast<unsigned>(n >= 148 * 8 ? 1 : (148 * 8) / n);
  bilinear_f32_ragged_kernel<<<dim3(gx, static_cast<unsigned>(n)), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, rows, ih,
                                                                                                             iw);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_add_h16(const void* a, const void* b, void* out, int64_t n, int dtype, void* stream) {
  VDA_CHECK(n % 8 == 0, "add: element count must be a multiple of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == VDA_BF16)
    add_h16_kernel<__nv_bfloat16><<<grid_for(n / 8, 256), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(a),
                                                                       static_cast<const __nv_bfloat16*>(b),
                                                                       static_cast<__nv_bfloat16*>(out), n / 8);
  else
    add_h16_kernel<__half><<<grid_for(n / 8, 256), 256, 0, st>>>(static_cast<const __half*>(a), static_cast<const __half*>(b),
                                                                static_cast<__half*>(out), n / 8);
  VDA_CUDA(cudaGetLastError());
  return 0;
}
