// Temporal attention (the spatial ViT attention lives in attention_spatial.cu).
//
// motion_module/motion_module.py:230-297 with motion_module/attention.py:182-211: at every spatial position an
// independent 32-frame sequence, 8 heads of d = C/8:  out = softmax(q k^T d^-1/2) v.
//
// The op is HBM-bound (4 * T*hw*C 16-bit elements moved for 4*T*T*d FLOP per (position, head): AI = T/2 = 16), so
// the kernel is organised around memory: one CTA per (position, group of heads), the q|k|v row segments of the
// 32 frames are copied with 16-byte cp.async into XOR-swizzled shared-memory tiles (512 B..1 KB contiguous per
// segment), several CTAs per SM keep the loads of the next CTA in flight while this one computes.  One warp per
// head: S = Q K^T (32x32) and O = P V on warp-level tensor-core MMAs (m16n8k16, fp32 accumulate; 32x32 tiles are
// far too small for a 128-row tcgen05 tile and the tensor work is < 10% of the HBM time either way), softmax in
// fp32 registers with quad shuffles, O staged through the (dead) Q tile so the global stores are 16-byte and
// row-contiguous.  Head dims that are not a multiple of 16 (ViT-S: 24, 48, 8) are zero-padded in shared memory.
#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

template <typename T>
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1);
template <>
__device__ __forceinline__ void mma16816<__nv_bfloat16>(float (&c)[4], const uint32_t (&a)[4], uint32_t b0,
                                                        uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <>
__device__ __forceinline__ void mma16816<__half>(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// One head tile: 32 rows (frames) x DHP columns of 16-bit, row pitch DHP*2 bytes, 16-byte chunks XOR-swizzled so
// that the 8 rows of an ldmatrix 8x8 block fall into 8 different bank groups for every pitch.
// ---------------------------------------------------------------------------------------------
template <int DHP>
__device__ __forceinline__ uint32_t ta_off(int row, int chunk) {
  constexpr int CH = DHP / 8;                       // chunks per row: 2, 4, 8 or 16
  constexpr int RPL = CH >= 8 ? 1 : 8 / CH;         // rows per 128-byte line
  constexpr int MASK = CH >= 8 ? 7 : CH - 1;
  return static_cast<uint32_t>(row * (DHP * 2) + ((chunk ^ ((row / RPL) & MASK)) << 4));
}

template <typename T, int DHP>
__global__ void __launch_bounds__(256)
temporal_attention_kernel(const T* __restrict__ qkv, T* __restrict__ out, int Tn, int hw, int C, int heads, int hpc) {
  extern __shared__ __align__(128) uint8_t sm_t[];   // [hpc][3 (q|k|v)][32][DHP] 16-bit
  constexpr int TILE = 32 * DHP * 2;
  constexpr int CH = DHP / 8;
  const int pos = blockIdx.x;
  const int dh = C / heads;
  const int h0 = blockIdx.y * hpc;
  const int dch = dh / 8;                            // valid 16-byte chunks per head row
  const uint32_t sbase = smem_u32(sm_t);

  // ---- cooperative load: (head, which, frame, chunk); rows >= Tn and pad chunks are zero-filled ----
  const int total = hpc * 3 * 32 * CH;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int c = idx % CH;
    int rest = idx / CH;
    const int h = rest % hpc;                        // consecutive threads: chunks, then heads (contiguous in global)
    rest /= hpc;
    const int f = rest % 32, which = rest / 32;
    const uint32_t dst = sbase + (h * 3 + which) * TILE + ta_off<DHP>(f, c);
    if (f < Tn && c < dch) {
      const T* src = qkv + (static_cast<long long>(f) * hw + pos) * (3LL * C) + which * C + (h0 + h) * dh + c * 8;
      cp_async16(dst, src);
    } else {
      asm volatile("st.shared.v4.b32 [%0], {%1,%1,%1,%1};" ::"r"(dst), "r"(0) : "memory");
    }
  }
  cp_async_wait_all();
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp >= hpc) return;
  const uint32_t sQ = sbase + (warp * 3 + 0) * TILE, sK = sQ + TILE, sV = sK + TILE;
  const int g = lane >> 2, t4 = lane & 3;

  // ---- S = Q K^T : 32 x 32, fp32 ----
  float s[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) s[mt][nt][e] = 0.f;
#pragma unroll
  for (int ks = 0; ks < DHP / 16; ++ks) {
    uint32_t a[2][4], b[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) ldsm_x4(a[mt], sQ + ta_off<DHP>(mt * 16 + (lane & 15), ks * 2 + (lane >> 4)));
#pragma unroll
    for (int np = 0; np < 2; ++np)
      ldsm_x4(b[np], sK + ta_off<DHP>(np * 16 + (lane & 7) + 8 * (lane >> 4), ks * 2 + ((lane >> 3) & 1)));
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int np = 0; np < 2; ++np) {
        mma16816<T>(s[mt][2 * np], a[mt], b[np][0], b[np][1]);
        mma16816<T>(s[mt][2 * np + 1], a[mt], b[np][2], b[np][3]);
      }
  }
  // ---- softmax over the key frames (columns); thread holds rows mt*16+g and mt*16+g+8, cols nt*8 + 2*t4 + {0,1} ----
  const float sc = rsqrtf(static_cast<float>(dh)) * 1.4426950408889634f;
  uint32_t pf[2][2][4];                               // P as A fragments: [m-tile][k-step of 16 keys]
  float inv[2][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {                  // hh = 0: row g, 1: row g + 8
      float mx = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int col = nt * 8 + 2 * t4 + e;
          float v = s[mt][nt][2 * hh + e];
          if (col >= Tn) v = -INFINITY;
          s[mt][nt][2 * hh + e] = v;
          mx = fmaxf(mx, v);
        }
      }
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float mb = mx * sc;
      float sum = 0.f;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float pv = exp2f(fmaf(s[mt][nt][2 * hh + e], sc, -mb));
          s[mt][nt][2 * hh + e] = pv;
          sum += pv;
        }
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      inv[mt][hh] = 1.f / sum;
    }
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      pf[mt][kk][0] = H16<T>::pack2(s[mt][2 * kk][0], s[mt][2 * kk][1]);
      pf[mt][kk][1] = H16<T>::pack2(s[mt][2 * kk][2], s[mt][2 * kk][3]);
      pf[mt][kk][2] = H16<T>::pack2(s[mt][2 * kk + 1][0], s[mt][2 * kk + 1][1]);
      pf[mt][kk][3] = H16<T>::pack2(s[mt][2 * kk + 1][2], s[mt][2 * kk + 1][3]);
    }
  }
  // ---- O = P V, 64 columns of d at a time; O -> (dead) Q tile ----
  constexpr int DSTEP = DHP < 64 ? DHP : 64;
#pragma unroll
  for (int d0 = 0; d0 < DHP; d0 += DSTEP) {
    float o[2][DSTEP / 8][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < DSTEP / 8; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) o[mt][nt][e] = 0.f;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
#pragma unroll
      for (int dp = 0; dp < DSTEP / 16; ++dp) {
        uint32_t vb[4];
        ldsm_x4_t(vb, sV + ta_off<DHP>(kk * 16 + (lane & 7) + 8 * ((lane >> 3) & 1), d0 / 8 + dp * 2 + (lane >> 4)));
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          mma16816<T>(o[mt][2 * dp], pf[mt][kk], vb[0], vb[1]);
          mma16816<T>(o[mt][2 * dp + 1], pf[mt][kk], vb[2], vb[3]);
        }
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < DSTEP / 8; ++nt) {
        const int r0 = mt * 16 + g, ch = d0 / 8 + nt;
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sQ + ta_off<DHP>(r0, ch) + t4 * 4),
                     "r"(H16<T>::pack2(o[mt][nt][0] * inv[mt][0], o[mt][nt][1] * inv[mt][0]))
                     : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(sQ + ta_off<DHP>(r0 + 8, ch) + t4 * 4),
                     "r"(H16<T>::pack2(o[mt][nt][2] * inv[mt][1], o[mt][nt][3] * inv[mt][1]))
                     : "memory");
      }
  }
  __syncwarp();
  // ---- coalesced 16-byte stores of the head's [Tn, dh] block ----
  for (int idx = lane; idx < Tn * dch; idx += 32) {
    const int f = idx / dch, c = idx - f * dch;
    uint4 u;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
                 : "r"(sQ + ta_off<DHP>(f, c)) : "memory");
    *reinterpret_cast<uint4*>(out + (static_cast<long long>(f) * hw + pos) * C + (h0 + warp) * dh + c * 8) = u;
  }
}

template <typename T, int DHP>
static int launch_temporal(const void* qkv, void* out, int T_, int hw, int C, int heads, cudaStream_t st) {
  // heads per CTA: largest divisor of `heads` whose q|k|v tiles stay <= 48 KB (>= 4 CTAs per SM)
  int hpc = heads;
  while (hpc > 1 && (heads % hpc != 0 || static_cast<size_t>(hpc) * 3 * 32 * DHP * 2 > 48 * 1024)) --hpc;
  const size_t smem = static_cast<size_t>(hpc) * 3 * 32 * DHP * 2;
  auto k = temporal_attention_kernel<T, DHP>;
  VDA_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(k), 64 * 1024));   // per (kernel, device)
  dim3 grid(hw, heads / hpc);
  const int threads = 32 * hpc < 128 ? 128 : 32 * hpc;    // >= 4 warps share the load loop
  k<<<grid, threads, smem, st>>>(static_cast<const T*>(qkv), static_cast<T*>(out), T_, hw, C, heads, hpc);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

template <typename T>
static int dispatch_temporal(const void* qkv, void* out, int T_, int hw, int C, int heads, cudaStream_t st) {
  const int dh = C / heads;
  if (dh <= 16) return launch_temporal<T, 16>(qkv, out, T_, hw, C, heads, st);
  if (dh <= 32) return launch_temporal<T, 32>(qkv, out, T_, hw, C, heads, st);
  if (dh <= 64) return launch_temporal<T, 64>(qkv, out, T_, hw, C, heads, st);
  return launch_temporal<T, 128>(qkv, out, T_, hw, C, heads, st);
}

// ---------------------------------------------------------------------------------------------
// Streaming step: each batch row's query (one new frame of one stream) against <= 31 cached frames of that stream's
// pool entry + itself (vda.h, vda_attention_temporal_step_batched; vda_attention_temporal_step is its B = 1 case).
//
// A CTA owns (batch row b, head h, 8 warps x PPT adjacent positions).  It first stages the k | v positional rows of
// head h at positions 0..n (fp32, n + 1 rows of 2 dh) in shared memory: they depend only on key position and column,
// so every warp of the CTA reads them from there instead of each lane loading 64 bytes of PE table per 32 bytes of
// cache from L2.  In a warp, lane = (key split ks, chunk c): c < G holds 16-byte chunk c of the head's dh columns
// (G = dh/8 rounded up to a power of two, the extra lanes hold zeros), and the KS = 32/G key splits take keys ks,
// ks + KS, ... of the sequence, so a lane walks at most 32/KS keys and a warp has all its loads in flight at once (the
// kernel is HBM-bound: the cached K'|V' rows are the traffic).  Scores are reduced over the G lanes of a split with
// xor shuffles; every split keeps an online softmax (fp32) and the splits are merged at the end (max, rescale, sum).
// A row whose pool index is outside 0..S-1 (-1: a pad row) attends to itself only and touches no pool byte.
//
// CAUSAL (vda_attention_temporal_step_causal: several consecutive frames of one stream in one launch): a context entry
// e < 0 names batch row -1 - e of the same launch, whose k'|v' are read from its q'|k'|v' block of `qkv` instead of a
// pool slot, and the kernel writes no pool byte (vda_stream_cache_store does, after it).  Everything else is the same
// code, so a row gives the bits the one-frame kernel gives against a pool that holds those frames.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 p = H16<T>::unpack2(w[e]);
    f[2 * e] = p.x;
    f[2 * e + 1] = p.y;
  }
}

__device__ __forceinline__ void load_pe8(const float* p, float (&f)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p));
  const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  f[0] = a.x, f[1] = a.y, f[2] = a.z, f[3] = a.w, f[4] = b.x, f[5] = b.y, f[6] = b.z, f[7] = b.w;
}

__device__ __forceinline__ void lds_pe8(const float* p, float (&f)[8]) {
  const float4 a = reinterpret_cast<const float4*>(p)[0];
  const float4 b = reinterpret_cast<const float4*>(p)[1];
  f[0] = a.x, f[1] = a.y, f[2] = a.z, f[3] = a.w, f[4] = b.x, f[5] = b.y, f[6] = b.z, f[7] = b.w;
}

constexpr int STEP_WARPS = 8;

// (min. 2 CTAs per SM: without it ptxas caps one instantiation at 64 registers and spills)
template <typename T, int G, int PPT, bool CAUSAL>
__global__ void __launch_bounds__(STEP_WARPS * 32, 2)
temporal_step_kernel(const T* __restrict__ qkv, T* __restrict__ pool, const float* __restrict__ pe,
                     const int32_t* __restrict__ rows, const int32_t* __restrict__ ctx, T* __restrict__ out, int hw,
                     int C, int heads, int S, int slots, int ctx_stride) {
  extern __shared__ float4 spe4[];                   // [n + 1][pe_k (dh) | pe_v (dh)] of head h
  float* spe = reinterpret_cast<float*>(spe4);
  constexpr int KS = 32 / G;
  const int b = blockIdx.y;
  const int h = static_cast<int>(blockIdx.x % heads);
  const int lane = threadIdx.x & 31, c = lane % G, ks = lane / G;
  const int dh = C / heads;
  // (no early exit for p0 >= hw: the shuffles need the whole warp, the staging the whole CTA)
  const long long p0 = (static_cast<long long>(blockIdx.x / heads) * STEP_WARPS + (threadIdx.x >> 5)) * PPT;
  const bool act = c * 8 < dh;                       // lane holds a real chunk of the head
  const int col = act ? h * dh + c * 8 : h * dh;
  const int sco = act ? c * 8 : 0;                   // the lane's column in a staged PE row
  const int32_t* cx = ctx + static_cast<long long>(b) * ctx_stride;
  const int r = rows ? __ldg(rows + b) : 0;
  const bool real = r >= 0 && r < S;                 // a pad row (r = -1) or a bad index reads / writes no pool byte
  const int n = real ? min(min(max(__ldg(cx), 0), 31), ctx_stride - 2) : 0;
  const int ws = min(max(__ldg(cx + 1), 0), slots - 1);
  const float sc = rsqrtf(static_cast<float>(dh)) * 1.4426950408889634f;
  const long long row2 = 2LL * C;
  const long long hwl = hw;
  T* cache = pool + (real ? static_cast<long long>(r) * slots * hwl * row2 : 0LL);
  const T* cq = qkv + static_cast<long long>(b) * hwl * 3 * C;
  T* co = out + static_cast<long long>(b) * hwl * C;

  for (int i = threadIdx.x; i < (n + 1) * dh / 2; i += blockDim.x) {   // float4 i of the staged rows
    const int j = i / (dh / 2), w = (i % (dh / 2)) * 4;
    const int src = w < dh ? C + h * dh + w : 2 * C + h * dh + (w - dh);
    spe4[i] = __ldg(reinterpret_cast<const float4*>(pe + static_cast<long long>(j) * 3 * C + src));
  }

  float q[PPT][8], o[PPT][8], m[PPT], l[PPT];
  {
    float pq[8];
    load_pe8(pe + static_cast<long long>(n) * 3 * C + col, pq);
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
      const long long pos = p0 + i;
      uint4 uq = make_uint4(0, 0, 0, 0);
      if (act && pos < hw) {
        const T* rq = cq + pos * 3 * C + col;
        uq = __ldg(reinterpret_cast<const uint4*>(rq));
        if (!CAUSAL && ks == 0 && real) {            // the current frame's k'|v' go to the write slot unchanged
          T* w = cache + (static_cast<long long>(ws) * hw + pos) * row2 + col;
          *reinterpret_cast<uint4*>(w) = __ldg(reinterpret_cast<const uint4*>(rq + C));
          *reinterpret_cast<uint4*>(w + C) = __ldg(reinterpret_cast<const uint4*>(rq + 2 * C));
        }
      }
      float fq[8];
      unpack8<T>(uq, fq);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        q[i][e] = act ? (fq[e] + pq[e]) * sc : 0.f;
        o[i][e] = 0.f;
      }
      m[i] = -INFINITY;
      l[i] = 0.f;
    }
  }
  __syncthreads();
  // ---- keys ks, ks + KS, ... of the sequence: context positions 0..n-1 (cache), then the current frame (position n) ----
#pragma unroll 2
  for (int jb = 0; jb <= n; jb += KS) {             // (warp-uniform trip count: the shuffles need every lane)
    const int j = min(jb + ks, n);
    const bool valid = jb + ks <= n, cur = j == n;
    const int slot = cur ? 0 : min(max(__ldg(cx + 2 + j), 0), slots - 1);
    float pk[8], pv[8];
    lds_pe8(spe + j * 2 * dh + sco, pk);
    lds_pe8(spe + j * 2 * dh + dh + sco, pv);
    uint4 uk[PPT], uv[PPT];
    if constexpr (CAUSAL) {
      // key row base and row pitch: the current frame, an earlier row of this launch (e < 0) or a pool slot
      const int e = cur ? 0 : __ldg(cx + 2 + j);
      const T* kb;
      long long kp;
      if (cur) {
        kb = cq + C + col, kp = 3LL * C;
      } else if (e < 0) {
        const int rb = min(-1 - e, static_cast<int>(gridDim.y) - 1);
        kb = qkv + static_cast<long long>(rb) * hwl * 3 * C + C + col, kp = 3LL * C;
      } else {
        kb = cache + static_cast<long long>(slot) * hw * row2 + col, kp = row2;
      }
#pragma unroll
      for (int i = 0; i < PPT; ++i) {
        const long long pos = p0 + i;
        uk[i] = uv[i] = make_uint4(0, 0, 0, 0);
        if (act && pos < hw) {
          const T* rk = kb + pos * kp;
          uk[i] = __ldg(reinterpret_cast<const uint4*>(rk));
          uv[i] = __ldg(reinterpret_cast<const uint4*>(rk + C));
        }
      }
    } else {
#pragma unroll
      for (int i = 0; i < PPT; ++i) {
        const long long pos = p0 + i;
        uk[i] = uv[i] = make_uint4(0, 0, 0, 0);
        if (act && pos < hw) {
          const T* rk = cur ? cq + pos * 3 * C + C + col : cache + (static_cast<long long>(slot) * hw + pos) * row2 + col;
          uk[i] = __ldg(reinterpret_cast<const uint4*>(rk));
          uv[i] = __ldg(reinterpret_cast<const uint4*>(rk + C));
        }
      }
    }
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
      float fk[8], fv[8];
      unpack8<T>(uk[i], fk);
      unpack8<T>(uv[i], fv);
      float s = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) s = fmaf(q[i][e], fk[e] + pk[e], s);
#pragma unroll
      for (int x = 1; x < G; x <<= 1) s += __shfl_xor_sync(0xffffffffu, s, x);
      if (valid) {
        const float mn = fmaxf(m[i], s);
        const float corr = exp2f(m[i] - mn), p = exp2f(s - mn);
        m[i] = mn;
        l[i] = fmaf(l[i], corr, p);
#pragma unroll
        for (int e = 0; e < 8; ++e) o[i][e] = fmaf(o[i][e], corr, p * (fv[e] + pv[e]));
      }
    }
  }
  // ---- merge the key splits (lanes c, c + G, c + 2G, ...); a split without keys has m = -inf, l = 0 ----
#pragma unroll
  for (int i = 0; i < PPT; ++i) {
    float mx = m[i];
#pragma unroll
    for (int x = G; x < 32; x <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, x));
    const float f = exp2f(m[i] - mx);
    float li = l[i] * f;
#pragma unroll
    for (int x = G; x < 32; x <<= 1) li += __shfl_xor_sync(0xffffffffu, li, x);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = o[i][e] * f;
#pragma unroll
      for (int x = G; x < 32; x <<= 1) v += __shfl_xor_sync(0xffffffffu, v, x);
      o[i][e] = v;
    }
    const long long pos = p0 + i;
    if (ks == 0 && act && pos < hw) {
      const float inv = 1.f / li;
      uint4 u;
      u.x = H16<T>::pack2(o[i][0] * inv, o[i][1] * inv);
      u.y = H16<T>::pack2(o[i][2] * inv, o[i][3] * inv);
      u.z = H16<T>::pack2(o[i][4] * inv, o[i][5] * inv);
      u.w = H16<T>::pack2(o[i][6] * inv, o[i][7] * inv);
      *reinterpret_cast<uint4*>(co + pos * C + col) = u;
    }
  }
}

struct StepArgs {
  const void* qkv;
  void* pool;
  const float* pe;
  const int32_t* rows;
  const int32_t* ctx;
  void* out;
  int B, S, ctx_stride, hw, C, heads, slots;
  bool causal;                                       // vda_attention_temporal_step_causal
};

template <typename T, int G, bool CAUSAL>
static int launch_step(const StepArgs& a, cudaStream_t st) {
  constexpr int PPT = 2;
  const int tiles = (a.hw + STEP_WARPS * PPT - 1) / (STEP_WARPS * PPT);
  const dim3 grid(static_cast<unsigned>(tiles * a.heads), static_cast<unsigned>(a.B));
  const size_t smem = static_cast<size_t>(32) * 2 * (a.C / a.heads) * sizeof(float);   // <= 32 KB (dh <= 128)
  temporal_step_kernel<T, G, PPT, CAUSAL><<<grid, STEP_WARPS * 32, smem, st>>>(
      static_cast<const T*>(a.qkv), static_cast<T*>(a.pool), a.pe, a.rows, a.ctx, static_cast<T*>(a.out), a.hw, a.C,
      a.heads, a.S, a.slots, a.ctx_stride);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

template <typename T, bool CAUSAL>
static int dispatch_step(const StepArgs& a, cudaStream_t st) {
  const int chunks = a.C / a.heads / 8;
  if (chunks <= 1) return launch_step<T, 1, CAUSAL>(a, st);
  if (chunks <= 2) return launch_step<T, 2, CAUSAL>(a, st);
  if (chunks <= 4) return launch_step<T, 4, CAUSAL>(a, st);
  if (chunks <= 8) return launch_step<T, 8, CAUSAL>(a, st);
  return launch_step<T, 16, CAUSAL>(a, st);
}

static int temporal_step(const StepArgs& a, int dtype, void* stream) {
  VDA_CHECK(dtype == VDA_BF16 || dtype == VDA_FP16, "bad dtype %d", dtype);
  VDA_CHECK(a.hw > 0, "temporal step: hw must be positive, got %d", a.hw);
  VDA_CHECK(a.C % 8 == 0 && a.C % a.heads == 0 && (a.C / a.heads) % 8 == 0 && a.heads <= 8 && a.C / a.heads <= 128,
            "bad channel/head split C=%d heads=%d (head dim must be a multiple of 8, <= 128; heads <= 8)", a.C, a.heads);
  VDA_CHECK(a.slots >= 2 && a.slots <= 32, "temporal step: the cache holds 2..32 frame slots, got %d", a.slots);
  VDA_CHECK(a.B >= 1 && a.B <= 65535, "temporal step: 1..65535 batch rows, got %d", a.B);
  VDA_CHECK(a.S >= 1, "temporal step: the pool needs at least one entry, got %d", a.S);
  VDA_CHECK(a.ctx_stride >= 2, "temporal step: a context row holds at least {n_ctx, write slot}, got stride %d",
            a.ctx_stride);
  VDA_CHECK(a.qkv && a.pool && a.pe && a.ctx && a.out, "temporal step: null pointer");
  VDA_CHECK(((reinterpret_cast<uintptr_t>(a.qkv) | reinterpret_cast<uintptr_t>(a.pool) |
              reinterpret_cast<uintptr_t>(a.pe) | reinterpret_cast<uintptr_t>(a.out)) & 15) == 0,
            "qkv/cache/pe/out must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (a.causal) {
    if (dtype == VDA_BF16) return dispatch_step<__nv_bfloat16, true>(a, st);
    return dispatch_step<__half, true>(a, st);
  }
  if (dtype == VDA_BF16) return dispatch_step<__nv_bfloat16, false>(a, st);
  return dispatch_step<__half, false>(a, st);
}

// ---------------------------------------------------------------------------------------------
// Deferred cache write of a causal step (vda_stream_cache_store): batch row b's k'|v' (columns C..3C of its q'|k'|v'
// rows) -> pool[rows[b]], slot ctx[b][1].  A pool slot is a contiguous [hw, 2C] block, so thread i of row b moves
// 16-byte chunk i of it; the source chunk sits at position i / (C/4), column C + 8 (i % (C/4)) of the row's block.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
stream_cache_store_kernel(const uint16_t* __restrict__ qkv, uint16_t* __restrict__ pool, const int32_t* __restrict__ rows,
                          const int32_t* __restrict__ ctx, int S, int ctx_stride, int hw, int C, int slots) {
  const int b = blockIdx.y;
  const int r = __ldg(rows + b);
  if (r < 0 || r >= S) return;                        // pad row
  const int ws = min(max(__ldg(ctx + static_cast<long long>(b) * ctx_stride + 1), 0), slots - 1);
  const int cpr = C / 4;                              // 16-byte chunks per k'|v' row
  const long long n = static_cast<long long>(hw) * cpr;
  const uint16_t* src = qkv + static_cast<long long>(b) * hw * 3 * C + C;
  uint4* dst = reinterpret_cast<uint4*>(pool + (static_cast<long long>(r) * slots + ws) * hw * 2 * C);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pos = i / cpr;
    const int c = static_cast<int>(i - pos * cpr);
    dst[i] = __ldg(reinterpret_cast<const uint4*>(src + pos * 3 * C + c * 8));
  }
}

}  // namespace vda

using namespace vda;

extern "C" int vda_attention_temporal_step_batched(const void* qkv, void* pool, const float* pe, const int32_t* rows,
                                                   const int32_t* ctx, void* out, int B, int S, int ctx_stride, int hw,
                                                   int C, int heads, int slots, int dtype, void* stream) {
  VDA_CHECK(rows, "temporal step: null row table");
  return temporal_step({qkv, pool, pe, rows, ctx, out, B, S, ctx_stride, hw, C, heads, slots}, dtype, stream);
}

extern "C" int vda_attention_temporal_step_causal(const void* qkv, const void* pool, const float* pe, const int32_t* rows,
                                                  const int32_t* ctx, void* out, int B, int S, int ctx_stride, int hw,
                                                  int C, int heads, int slots, int dtype, void* stream) {
  VDA_CHECK(rows, "temporal step: null row table");
  return temporal_step({qkv, const_cast<void*>(pool), pe, rows, ctx, out, B, S, ctx_stride, hw, C, heads, slots, true},
                       dtype, stream);
}

extern "C" int vda_stream_cache_store(const void* qkv, void* pool, const int32_t* rows, const int32_t* ctx, int B, int S,
                                      int ctx_stride, int hw, int C, int slots, int dtype, void* stream) {
  VDA_CHECK(dtype == VDA_BF16 || dtype == VDA_FP16, "bad dtype %d", dtype);
  VDA_CHECK(hw > 0 && C > 0 && C % 8 == 0, "cache store: need hw > 0 and C a positive multiple of 8, got hw=%d C=%d", hw, C);
  VDA_CHECK(slots >= 2 && slots <= 32, "cache store: the cache holds 2..32 frame slots, got %d", slots);
  VDA_CHECK(B >= 1 && B <= 65535, "cache store: 1..65535 batch rows, got %d", B);
  VDA_CHECK(S >= 1, "cache store: the pool needs at least one entry, got %d", S);
  VDA_CHECK(ctx_stride >= 2, "cache store: a context row holds at least {n_ctx, write slot}, got stride %d", ctx_stride);
  VDA_CHECK(qkv && pool && rows && ctx, "cache store: null pointer");
  VDA_CHECK(((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(pool)) & 15) == 0,
            "qkv/pool must be 16-byte aligned");
  const long long chunks = static_cast<long long>(hw) * (C / 4);
  const dim3 grid(static_cast<unsigned>((chunks + 255) / 256 < 4096 ? (chunks + 255) / 256 : 4096), static_cast<unsigned>(B));
  stream_cache_store_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(qkv), static_cast<uint16_t*>(pool), rows, ctx, S, ctx_stride, hw, C, slots);
  VDA_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int vda_attention_temporal_step(const void* qkv, void* cache, const float* pe, const int32_t* ctx, void* out,
                                           int hw, int C, int heads, int slots, int dtype, void* stream) {
  // one row, pool entry 0; a stride of 2 + 31 keeps n_ctx's clamp at 31
  return temporal_step({qkv, cache, pe, nullptr, ctx, out, 1, 1, 33, hw, C, heads, slots}, dtype, stream);
}

extern "C" int vda_attention_temporal(const void* qkv, void* out, int T, int hw, int C, int heads, int dtype,
                                      void* stream) {
  VDA_CHECK(T > 0 && T <= 32, "temporal attention supports 1..32 frames (temporal_max_len, dpt_temporal.py:38), got %d", T);
  VDA_CHECK(dtype == VDA_BF16 || dtype == VDA_FP16, "bad dtype %d", dtype);
  VDA_CHECK(C % 8 == 0 && C % heads == 0 && (C / heads) % 8 == 0 && heads <= 8 && C / heads <= 128,
            "bad channel/head split C=%d heads=%d (head dim must be a multiple of 8, <= 128; heads <= 8)", C, heads);
  VDA_CHECK((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
            "qkv/out must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == VDA_BF16) return dispatch_temporal<__nv_bfloat16>(qkv, out, T, hw, C, heads, st);
  return dispatch_temporal<__half>(qkv, out, T, hw, C, heads, st);
}
