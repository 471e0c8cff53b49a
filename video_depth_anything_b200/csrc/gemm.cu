// tcgen05 / TMEM / TMA GEMM for sm_100a with fused epilogues, also used as an implicit-GEMM
// 3x3 convolution (A tiles gathered by 4-D TMA boxes with out-of-bounds zero fill = padding).
//
//   out[M,N] = A[M,K] . Wt[N,K]^T      A, Wt: bf16|fp16, K-major;  fp32 accumulators in TMEM
//
// One persistent CTA per SM (or one CTA pair per TPC, cta_group::2), 320 threads, warp-specialised:
//   warp 0     : TMA producer (one elected lane)   smem ring of `stages` x {A 128x64, B rows x 64}, SWIZZLE_128B
//   warp 1     : TMEM allocator + tcgen05.mma issuer (one elected lane), UMMA 128|256 x block_n x 16
//   warps 2..9 : epilogue, two warps per TMEM lane quadrant (each drains half of the tile's columns): tcgen05.ld,
//                fused math, staged through a swizzled smem tile so that every global access is a row segment.
//                Two accumulator stages in TMEM overlap the epilogue of tile i with the MMAs of tile i+1.
// block_n (16..256, multiple of 16) is a run-time parameter: it only appears in the instruction
// descriptor, the B tensor map and loop bounds.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <mutex>
#include <unordered_map>

#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int kEpiWarps = 8;                 // two warps per TMEM lane quadrant, each takes half of the columns
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kMaxStages = 8;
constexpr uint32_t kABytes = BLOCK_M * BLOCK_K * 2;

struct GemmDev {
  int M, N, K;
  int block_n, num_k_blocks, tiles_m, tiles_n, num_tiles, stages;
  uint32_t stage_bytes, tx_bytes, tmem_cols, acc_stride;   // tx_bytes: TMA bytes per stage issued by one CTA
  // conv addressing
  int H, W, bw, bh, tiles_x, tiles_y, cblocks;
  // epilogue
  const float* bias;
  const float* gamma;
  int act;
  const void* res1;
  long long ldr1;
  int res1_f32;
  const void* res2;
  void* out;
  long long ldo;
  int out_f32;
  void* out_relu;
  int row_group;
  int geglu_half;
  int convt_s, convt_co, in_h, in_w;
  const float* tail_w;
  float tail_b;
  int staged;   // LINEAR: transpose the tile through shared memory (fp32 residual / fp32 output streams)
  // LayerNorm folding (see SPEC 4 / 5 / 6 in the kernel)
  void* out16;              // SPEC 4: 16-bit copy of the fp32 output rows [M, ldo]
  float2* stats_out;        // SPEC 4: per-row partial statistics [M][stat_parts] = (mean, M2) over stat_cols columns
  const float2* stats_in;   // SPEC 5/6: the producer's partial statistics of the A rows
  const float* ln_c1;       // SPEC 5/6: c1[n] = sum_k W'[n,k]  (W' = 16-bit(LayerNorm weight * W))
  int stat_parts, stat_cols;
  float ln_eps, ln_inv_d;
  int a_k_blocks;           // k-blocks of A (== num_k_blocks unless the weights are a hi | lo pair: A is then walked twice)
  int epi_nbuf;             // SPEC 4: residual boxes per epilogue warp (1 | 2)
  uint32_t epi_warp_bytes;  // SPEC 4: shared memory per epilogue warp
  int pair;     // host only: launch the cta_group::2 variant
  int prefetch_max_kb;   // residual L2 prefetch of the next tile only when the K loop has at most this many blocks
};

// 4 consecutive columns as two packed fp32 pairs (FFMA2 / FADD2 / FMUL2 process a pair per instruction)
struct F4 { float2 a, b; };

template <typename T>
__device__ __forceinline__ F4 load4h(const T* src) {
  const uint2 u = *reinterpret_cast<const uint2*>(src);
  F4 r;
  r.a = H16<T>::unpack2(u.x);
  r.b = H16<T>::unpack2(u.y);
  return r;
}
__device__ __forceinline__ F4 load4f(const float* src) {
  const float4 v = *reinterpret_cast<const float4*>(src);
  F4 r;
  r.a = make_float2(v.x, v.y);
  r.b = make_float2(v.z, v.w);
  return r;
}
template <typename T>
__device__ __forceinline__ void store4h(T* dst, const F4& v) {
  uint2 u;
  u.x = H16<T>::pack2(v.a.x, v.a.y);
  u.y = H16<T>::pack2(v.b.x, v.b.y);
  *reinterpret_cast<uint2*>(dst) = u;
}
__device__ __forceinline__ void store4f(float* dst, const F4& v) {
  *reinterpret_cast<float4*>(dst) = make_float4(v.a.x, v.a.y, v.b.x, v.b.y);
}
__device__ __forceinline__ F4 add4(const F4& x, const F4& y) {
  F4 r;
  r.a = __fadd2_rn(x.a, y.a);
  r.b = __fadd2_rn(x.b, y.b);
  return r;
}
__device__ __forceinline__ F4 mul4(const F4& x, const F4& y) {
  F4 r;
  r.a = __fmul2_rn(x.a, y.a);
  r.b = __fmul2_rn(x.b, y.b);
  return r;
}
__device__ __forceinline__ F4 relu4(const F4& x) {
  F4 r;
  r.a = make_float2(fmaxf(x.a.x, 0.f), fmaxf(x.a.y, 0.f));
  r.b = make_float2(fmaxf(x.b.x, 0.f), fmaxf(x.b.y, 0.f));
  return r;
}
template <typename T>
__device__ __forceinline__ F4 gelu4(const F4& x) {
  // (a one-MUFU variant through tanh.approx -- gelu_tanh2 in common.cuh -- was measured for bf16 outputs: fc1 274 -> 266 us
  // in step, but 1 + tanh(u) cancels for negative inputs and the 2^-11 error of MUFU.TANH raised the bf16 end-to-end
  // p99.9 error by up to 18 %; the sigmoid form keeps full relative accuracy in the tail and stays)
  F4 r;
  r.a = gelu_erf2(x.a);
  r.b = gelu_erf2(x.b);
  return r;
}

// byte offset of the 16-byte slot holding columns 4*c4..4*c4+3 of `row` in a warp's 32 x 32 fp32 staging tile
// (rows of 128 B, slots XOR-swizzled by row: conflict-free for row-per-thread writes and row-segment reads)
__device__ __forceinline__ uint32_t stg_off(int row, int c4) {
  return static_cast<uint32_t>(row * 128 + ((c4 ^ (row & 7)) << 4));
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ F4 lds128(uint32_t addr) {
  F4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.a.x), "=f"(r.a.y), "=f"(r.b.x), "=f"(r.b.y) : "r"(addr)
               : "memory");
  return r;
}

constexpr uint32_t kStageTile = 32 * 32 * 4;            // per-warp epilogue staging tile (bytes)
constexpr uint32_t kStagingBytes = kEpiWarps * kStageTile;

// CTA2: cta_group::2 -- the two CTAs of a cluster (one TPC) work on a 256-row tile pair with ONE stream of
// M = 256 UMMAs issued by the leader (rank 0).  Each CTA loads its own 128 rows of A and only HALF of the B tile
// (block_n/2 rows), so the L2 -> smem operand traffic and the smem writes per SM drop by a third and the smem
// reads of the tensor core from 96 to 64 B/clk/SM; accumulator rows 128r..128r+127 live in CTA r's TMEM and are
// drained by that CTA's own epilogue warps.
template <typename T, int EPI, bool CONV, bool STAGED, int SPEC, bool CTA2>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmD, const GemmDev p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t rfull_bar[kEpiWarps][2];   // SPEC 4: residual chunk landed (per epilogue warp)
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  __shared__ __align__(8) uint64_t tfull_bar[2];
  __shared__ __align__(8) uint64_t tempty_bar[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // 1024-byte aligned operand ring (SWIZZLE_128B atoms are 8 rows x 128 B), followed by the epilogue staging tiles
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], (CTA2 ? 2 : 1) * kEpiWarps);   // one arrival per epilogue warp; pair: both CTAs
    }
    if (SPEC == 4) {
      tma_prefetch_desc(&tmC);
      if (p.out16) tma_prefetch_desc(&tmD);
      for (int w = 0; w < kEpiWarps; ++w) { mbar_init(&rfull_bar[w][0], 1); mbar_init(&rfull_bar[w][1], 1); }
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    if (CTA2) tmem_alloc2(&tmem_base_s, p.tmem_cols);
    else tmem_alloc(&tmem_base_s, p.tmem_cols);
  }
  tc_fence_before();
  if (CTA2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  // PDL: everything above (barriers, TMEM, descriptor prefetch) may run under the tail of the previous kernel; nothing
  // below may start before its results are visible.  Our own successor may be scheduled as our CTAs retire.
  pdl_trigger();
  pdl_wait();
  const uint32_t tmem_base = tmem_base_s;
  const int rank = CTA2 ? static_cast<int>(cluster_ctarank()) : 0;
  // persistent tile loop: a CTA pair shares tile index, CTA r takes m block 2*pair + r
  const int tile0 = CTA2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = CTA2 ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);

  if (warp == 0) {
    // ================================ TMA producer ================================
    // warp-uniform control flow, one elected lane issues (see elect_one)
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = tile0; tile < p.num_tiles; tile += tile_step) {
      const int n_blk = tile % p.tiles_n;
      const int m_blk = CTA2 ? 2 * (tile / p.tiles_n) + rank : tile / p.tiles_n;
      int img = 0, x0 = 0, y0 = 0;
      if (CONV) {
        const int per_img = p.tiles_x * p.tiles_y;
        img = m_blk / per_img;
        const int rem = m_blk - img * per_img;
        y0 = (rem / p.tiles_x) * p.bh;
        x0 = (rem % p.tiles_x) * p.bw;
      }
      int tap = 0, cb = 0;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        if (elect_one()) {
          uint8_t* sA = smem_gen + static_cast<size_t>(stage) * p.stage_bytes;
          uint8_t* sB = sA + kABytes;
          if (CTA2) {
            // both CTAs load (A rows of their own m block, their half of the B rows); all bytes are credited to the
            // leader's full barrier, which expects the sum
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2u * p.tx_bytes);
            if (CONV) {
              const int dy = tap / 3 - 1, dx = tap % 3 - 1;
              tma_load_4d_pair(sA, &tmA, &full_bar[stage], cb * BLOCK_K, x0 + dx, y0 + dy, img);
            } else {
              tma_load_2d_pair(sA, &tmA, &full_bar[stage], (kb % p.a_k_blocks) * BLOCK_K, m_blk * BLOCK_M);
            }
            tma_load_2d_pair(sB, &tmB, &full_bar[stage], kb * BLOCK_K, n_blk * p.block_n + rank * (p.block_n >> 1));
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], p.tx_bytes);
            if (CONV) {
              const int dy = tap / 3 - 1, dx = tap % 3 - 1;
              tma_load_4d(sA, &tmA, &full_bar[stage], cb * BLOCK_K, x0 + dx, y0 + dy, img);
            } else {
              tma_load_2d(sA, &tmA, &full_bar[stage], (kb % p.a_k_blocks) * BLOCK_K, m_blk * BLOCK_M);
            }
            tma_load_2d(sB, &tmB, &full_bar[stage], kb * BLOCK_K, n_blk * p.block_n);
          }
        }
        __syncwarp();
        if (CONV && ++cb == p.cblocks) { cb = 0; if (++tap == 9) tap = 0; }   // (hi | lo weights: the taps are walked twice)
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    const uint32_t idesc = umma_idesc_m(H16<T>::kUmmaFmt, static_cast<uint32_t>(p.block_n), CTA2 ? 256u : 128u);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = tile0; tile < p.num_tiles && rank == 0; tile += tile_step) {   // pair: only the leader issues
      mbar_wait(&tempty_bar[as], aphase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + as * p.acc_stride;
      for (int kb = 0; kb < p.num_k_blocks; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sA = smem_base + stage * p.stage_bytes;
        const uint64_t da = umma_desc_sw128(sA);
        const uint64_t db = umma_desc_sw128(sA + kABytes);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) {
            // +32 bytes (16 elements) along K inside the 128-byte swizzle atom = +2 in the address field
            if (CTA2) umma_f16_pair(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
            else umma_f16(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          if (CTA2) {
            umma_commit_pair(&empty_bar[stage]);                                // frees the slot in both CTAs
            if (kb == p.num_k_blocks - 1) umma_commit_pair(&tfull_bar[as]);     // both epilogues may drain
          } else {
            umma_commit(&empty_bar[stage]);  // frees the smem slot once these MMAs retire
            if (kb == p.num_k_blocks - 1) umma_commit(&tfull_bar[as]);   // accumulator ready for the epilogue
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
      as ^= 1;
      if (as == 0) aphase ^= 1u;
    }
  } else {
    // ================================ epilogue ====================================
    const int ew = warp - 2;                // 0..7
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int eh = ew >> 2;                 // which half of the tile's columns this warp drains
    const uint32_t stg = smem_base + p.stages * p.stage_bytes + ew * kStageTile;
    // phase-2 mapping: 8 lanes per row (4 columns each), 4 rows per pass, 8 passes
    const int cg = lane & 7;
    const int rsub = lane >> 3;
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = tile0; tile < p.num_tiles; tile += tile_step) {
      const int n_blk = tile % p.tiles_n;
      const int m_blk = CTA2 ? 2 * (tile / p.tiles_n) + rank : tile / p.tiles_n;
      const int col_base = n_blk * p.block_n;
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * p.acc_stride;

      if (EPI == VDA_EPI_LINEAR && SPEC == 4) {
        // ---- fp32 residual stream updated in place, all global traffic of the tile by TMA (thread = row) ----
        //   out[r, n] = (acc + bias[n]) * gamma[n] + out[r, n]          (proj / fc2 + LayerScale + residual)
        // Each epilogue warp owns 32 rows x its half of the tile's columns, in chunks of 32 columns (a 32 x 32 fp32 box
        // = 4 KB, SWIZZLE_128B: row r's 16-byte slot j sits at slot j ^ (r & 7), conflict-free for row-per-thread
        // accesses).  The residual box of chunk k+2 is requested as soon as the result of chunk k has left its buffer
        // (two buffers per warp, flat over this CTA's tiles, so the first chunks of the NEXT tile are in flight a whole
        // tile ahead); results go back with TMA stores from the same buffer.  64 KB of loads in flight per SM without
        // a single address register: the register-staged version (SPEC 3) was bound by the 32 KB its 8 warps could
        // keep in flight (3.9 TB/s, tensor pipe 41 % active on proj).
        // Optional LayerNorm folding for the consumer GEMM (SPEC 5 / 6): a 16-bit copy of the new rows and, per row and
        // column half, (mean, M2) of the new values (shifted sums: M2 = sum d^2 - (sum d)^2 / n with d = v - v[first]).
        const int r = q * 32 + lane;
        const int nch32 = p.block_n >> 6;                       // 32-column chunks per warp (block_n % 64 == 0)
        const int c_begin = eh * (p.block_n >> 1);
        // per warp: epi_nbuf residual / result boxes (4 KB each) + one 2 KB box for the 16-bit copy.  epi_nbuf = 2 for
        // short K loops (the epilogue is the critical path: chunk k+2 is requested while chunk k+1 is processed), 1 for
        // long ones (fc2, K = 4096: the MMAs of a tile take 4x longer than its epilogue, the operand ring needs the
        // shared memory more)
        const uint32_t nbuf = static_cast<uint32_t>(p.epi_nbuf);
        const uint32_t buf0 = smem_base + p.stages * p.stage_bytes + ew * p.epi_warp_bytes;
        const uint32_t hbuf = buf0 + nbuf * 4096u;
        uint64_t* rfull = rfull_bar[ew];
        // flat chunk k of this warp: tile tile0 + (k / nch32) * tile_step, chunk k % nch32; buffer k % nbuf
        auto issue_load = [&](uint32_t k) {
          const int tl = tile0 + static_cast<int>(k / nch32) * tile_step;
          if (tl >= p.num_tiles) return;
          const int ci = static_cast<int>(k % nch32);
          const int nb = tl % p.tiles_n;
          const int mb = CTA2 ? 2 * (tl / p.tiles_n) + rank : tl / p.tiles_n;
          const uint32_t b = k % nbuf;
          mbar_arrive_expect_tx(&rfull[b], 4096u);
          tma_load_2d(reinterpret_cast<void*>(smem_gen + (buf0 - smem_base) + b * 4096u), &tmC, &rfull[b],
                      nb * p.block_n + c_begin + ci * 32, mb * BLOCK_M + q * 32);
        };
        if (tile == tile0) {                                    // first tile of this CTA: prime the buffer(s)
          if (elect_one()) { issue_load(0); if (nbuf > 1) issue_load(1); }
          __syncwarp();
        }
        const uint32_t kbase = static_cast<uint32_t>((tile - tile0) / tile_step) * nch32;
        const long long grow = static_cast<long long>(m_blk) * BLOCK_M + r;
        const bool row_ok = grow < p.M;
        float2 s1 = make_float2(0.f, 0.f), s2 = make_float2(0.f, 0.f);
        float shift = 0.f;
        for (int ci = 0; ci < nch32; ++ci) {
          const uint32_t k = kbase + ci;
          const uint32_t buf = buf0 + (k % nbuf) * 4096u;
          const int c0 = c_begin + ci * 32;
          const int col = col_base + c0;
          mbar_wait(&rfull[k % nbuf], (k / nbuf) & 1u);
          if (ci == 0) {
            mbar_wait(&tfull_bar[as], aphase);
            tc_fence_after();
          }
          uint32_t rr[32];
          tmem_ld32(t_row + c0, rr);
          tmem_ld_wait32(rr);
          uint32_t h16[16];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t a = buf + stg_off(lane, j);
            const F4 res = lds128(a);
            const F4 b4 = load4f(p.bias + col + 4 * j), g4 = load4f(p.gamma + col + 4 * j);   // warp-uniform addresses
            F4 v;
            v.a = __ffma2_rn(__fadd2_rn(make_float2(__uint_as_float(rr[4 * j]), __uint_as_float(rr[4 * j + 1])), b4.a), g4.a, res.a);
            v.b = __ffma2_rn(__fadd2_rn(make_float2(__uint_as_float(rr[4 * j + 2]), __uint_as_float(rr[4 * j + 3])), b4.b), g4.b, res.b);
            sts128(a, __float_as_uint(v.a.x), __float_as_uint(v.a.y), __float_as_uint(v.b.x), __float_as_uint(v.b.y));
            if (p.stats_out) {
              if (ci == 0 && j == 0) shift = v.a.x;
              const float2 sh2 = make_float2(shift, shift);
              const float2 da = __fadd2_rn(v.a, make_float2(-sh2.x, -sh2.y)), db = __fadd2_rn(v.b, make_float2(-sh2.x, -sh2.y));
              s1 = __fadd2_rn(s1, __fadd2_rn(da, db));
              s2 = __ffma2_rn(da, da, s2);
              s2 = __ffma2_rn(db, db, s2);
            }
            h16[2 * j] = H16<T>::pack2(v.a.x, v.a.y);
            h16[2 * j + 1] = H16<T>::pack2(v.b.x, v.b.y);
          }
          if (p.out16) {
            // 32 rows x 64 B box, SWIZZLE_64B: 16-byte slot j of row r sits at slot j ^ ((r >> 1) & 3)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              sts128(hbuf + static_cast<uint32_t>(lane * 64 + ((j ^ ((lane >> 1) & 3)) << 4)), h16[4 * j], h16[4 * j + 1],
                     h16[4 * j + 2], h16[4 * j + 3]);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_2d(&tmC, reinterpret_cast<const void*>(smem_gen + (buf - smem_base)), col, m_blk * BLOCK_M + q * 32);
            if (p.out16)
              tma_store_2d(&tmD, reinterpret_cast<const void*>(smem_gen + (hbuf - smem_base)), col, m_blk * BLOCK_M + q * 32);
            bulk_commit();
            bulk_wait_read<0>();          // the stores have read their boxes: the next residual chunk may land
            issue_load(k + nbuf);
          }
          __syncwarp();
        }
        if (p.stats_out && row_ok) {
          const float n = static_cast<float>(p.block_n >> 1);
          const float t1 = s1.x + s1.y, t2 = s2.x + s2.y;
          const float md = t1 / n;
          p.stats_out[grow * p.stat_parts + (n_blk * 2 + eh)] = make_float2(shift + md, fmaxf(t2 - t1 * md, 0.f));
        }
      } else if (EPI == VDA_EPI_TAIL) {   // block_n == N == 32: one dot product per row, thread = row (no staging)
        const int r = q * 32 + lane;
        bool valid;
        long long out_row;
        if (CONV) {
          const int per_img = p.tiles_x * p.tiles_y;
          const int img = m_blk / per_img;
          const int rem = m_blk - img * per_img;
          const int y = (rem / p.tiles_x) * p.bh + r / p.bw;
          const int x = (rem % p.tiles_x) * p.bw + r % p.bw;
          valid = (y < p.H) && (x < p.W) && (m_blk < p.tiles_m);
          out_row = (static_cast<long long>(img) * p.H + y) * p.W + x;
        } else {
          out_row = static_cast<long long>(m_blk) * BLOCK_M + r;
          valid = out_row < p.M;
        }
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        if (eh == 0) {
          float acc = p.tail_b;
          uint32_t rr[32];
          tmem_ld32(t_row, rr);
          tmem_ld_wait32(rr);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float h = fmaxf(__uint_as_float(rr[i]) + __ldg(p.bias + i), 0.f);
            acc = fmaf(h, __ldg(p.tail_w + i), acc);
          }
          if (valid) reinterpret_cast<float*>(p.out)[out_row] = fmaxf(acc, 0.f);
        }
      } else {
        // (output row, res1 row) of tile row r; output row -1 = outside the problem
        auto row_info = [&](int r, int& o, int& rr) {
          if (CONV) {
            const int per_img = p.tiles_x * p.tiles_y;
            const int img = m_blk / per_img;
            const int rem = m_blk - img * per_img;
            const int y = (rem / p.tiles_x) * p.bh + r / p.bw;
            const int x = (rem % p.tiles_x) * p.bw + r % p.bw;
            o = ((y < p.H) && (x < p.W) && (m_blk < p.tiles_m)) ? (img * p.H + y) * p.W + x : -1;
            rr = o;
          } else {
            const int m = m_blk * BLOCK_M + r;
            o = m < p.M ? m : -1;
            rr = m;
            if (p.row_group > 0) {
              o = m < p.M ? m + m / p.row_group + 1 : -1;
              rr = m % p.row_group + 1;
            }
            if (EPI == VDA_EPI_CONVT && m < p.M) {
              const int per_img = p.in_h * p.in_w;
              const int img = m / per_img;
              const int rem = m - img * per_img;
              const int y = rem / p.in_w, x = rem - y * p.in_w;
              // row index of output pixel (img, y*S, x*S) in the upsampled map
              o = (img * p.in_h * p.convt_s + y * p.convt_s) * (p.in_w * p.convt_s) + x * p.convt_s;
            }
          }
        };
        constexpr bool staged = STAGED;
        if (EPI == VDA_EPI_LINEAR && (p.res1 || p.res2) && p.num_k_blocks <= p.prefetch_max_kb) {
          // pull the residual rows of this CTA's NEXT tile towards L2 now: its epilogue then reads them at L2
          // latency instead of queueing behind HBM (the epilogue is a dependent load -> math -> store chain).
          // Only when the next epilogue is near (short K loop): with K = 4096 it is ~20 us away and the streaming
          // traffic of the kernel evicts most prefetched lines first (fc2: 185 MB of excess DRAM reads per launch)
          const int nxt = tile + tile_step;
          if (nxt < p.num_tiles) {
            const int n_blk2 = nxt % p.tiles_n;
            int o2, r2i;
            {
              const int m_blk2 = CTA2 ? 2 * (nxt / p.tiles_n) + rank : nxt / p.tiles_n;
              const int r = q * 32 + lane;
              if (CONV) {
                const int per_img = p.tiles_x * p.tiles_y;
                const int img = m_blk2 / per_img;
                const int rem = m_blk2 - img * per_img;
                const int y = (rem / p.tiles_x) * p.bh + r / p.bw;
                const int x = (rem % p.tiles_x) * p.bw + r % p.bw;
                o2 = ((y < p.H) && (x < p.W) && (m_blk2 < p.tiles_m)) ? (img * p.H + y) * p.W + x : -1;
                r2i = o2;
              } else {
                const int m = m_blk2 * BLOCK_M + r;
                o2 = m < p.M ? m : -1;
                r2i = m;
                if (p.row_group > 0) {
                  o2 = m < p.M ? m + m / p.row_group + 1 : -1;
                  r2i = m % p.row_group + 1;
                }
              }
            }
            if (o2 >= 0) {
              const int nch = p.block_n >> 4;
              const int c_lo = n_blk2 * p.block_n + (eh ? (nch + 1) / 2 : 0) * 16;
              int c_hi = n_blk2 * p.block_n + (eh ? nch : (nch + 1) / 2) * 16;
              if (c_hi > p.N) c_hi = p.N;
              if (p.res1) {
                const int esz = p.res1_f32 ? 4 : 2;
                const char* base = reinterpret_cast<const char*>(p.res1) + (r2i * p.ldr1 + c_lo) * esz;
                for (int off = 0; off < (c_hi - c_lo) * esz; off += 128) prefetch_l2(base + off);
              }
              if (p.res2) {
                const char* base = reinterpret_cast<const char*>(p.res2) + (o2 * p.ldo + c_lo) * 2;
                for (int off = 0; off < (c_hi - c_lo) * 2; off += 128) prefetch_l2(base + off);
              }
            }
          }
        }
        int orow[8], rrow[8];     // staged: rows of this lane in the transposed (phase 2) passes
        int o_row = -1, r_row = 0;   // direct: this thread's own row
        if (staged) {
#pragma unroll
          for (int it = 0; it < 8; ++it) row_info(q * 32 + it * 4 + rsub, orow[it], rrow[it]);
        } else {
          row_info(q * 32 + lane, o_row, r_row);
        }
        if (!(EPI == VDA_EPI_LINEAR && STAGED)) {   // (the staged LINEAR path first issues its residual loads)
          mbar_wait(&tfull_bar[as], aphase);
          tc_fence_after();
        }

        if ((EPI == VDA_EPI_LINEAR || EPI == VDA_EPI_CONVT) && !STAGED) {
          // ---- direct path (16-bit operands only): thread = row, 16 columns per step, no shared-memory traffic
          //      (the operand ring already uses ~3/4 of the smem bandwidth while the tensor pipe is busy) ----
          const int nch = p.block_n >> 4;
          const int ch_begin = eh ? (nch + 1) / 2 : 0, ch_end = eh ? nch : (nch + 1) / 2;
          auto process = [&](const uint32_t (&rr)[16], int c0) {
            const int col = col_base + c0;
            if (o_row < 0 || col >= p.N) return;
            const bool two = p.N - col > 8;      // N % 8 == 0: a 16-column chunk holds 8 or 16 valid columns
            F4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              v[i].a = make_float2(__uint_as_float(rr[4 * i]), __uint_as_float(rr[4 * i + 1]));
              v[i].b = make_float2(__uint_as_float(rr[4 * i + 2]), __uint_as_float(rr[4 * i + 3]));
            }
            int co = col;
            long long orow_l = o_row;
            if (EPI == VDA_EPI_CONVT) {
              const int kk = col / p.convt_co;
              co = col - kk * p.convt_co;
              const int ky = kk / p.convt_s, kx = kk - ky * p.convt_s;
              orow_l += static_cast<long long>(ky) * (p.in_w * p.convt_s) + kx;
            }
            F4 r1[4], r2[4];
            if (EPI == VDA_EPI_LINEAR) {   // all global loads before any store
              if (p.res1) {
                const T* r = reinterpret_cast<const T*>(p.res1) + r_row * p.ldr1 + col;
                r1[0] = load4h<T>(r); r1[1] = load4h<T>(r + 4);
                if (two) { r1[2] = load4h<T>(r + 8); r1[3] = load4h<T>(r + 12); }
              }
              if (p.res2) {
                const T* r = reinterpret_cast<const T*>(p.res2) + orow_l * p.ldo + col;
                r2[0] = load4h<T>(r); r2[1] = load4h<T>(r + 4);
                if (two) { r2[2] = load4h<T>(r + 8); r2[3] = load4h<T>(r + 12); }
              }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (i >= 2 && !two) break;
              if (p.bias) v[i] = add4(v[i], load4f(p.bias + co + 4 * i));
              if (EPI == VDA_EPI_LINEAR) {
                if (p.gamma) v[i] = mul4(v[i], load4f(p.gamma + col + 4 * i));
                if (p.act == VDA_ACT_GELU) v[i] = gelu4<T>(v[i]);
                else if (p.act == VDA_ACT_RELU) v[i] = relu4(v[i]);
                if (p.res1) v[i] = add4(v[i], r1[i]);
                if (p.res2) v[i] = add4(v[i], r2[i]);
              }
            }
            T* o = reinterpret_cast<T*>(p.out) + orow_l * p.ldo + co;
            auto st8 = [&](T* dst, const F4& x, const F4& y) {
              uint4 u;
              u.x = H16<T>::pack2(x.a.x, x.a.y); u.y = H16<T>::pack2(x.b.x, x.b.y);
              u.z = H16<T>::pack2(y.a.x, y.a.y); u.w = H16<T>::pack2(y.b.x, y.b.y);
              *reinterpret_cast<uint4*>(dst) = u;
            };
            st8(o, v[0], v[1]);
            if (two) st8(o + 8, v[2], v[3]);
            if (EPI == VDA_EPI_LINEAR && p.out_relu) {
              T* orl = reinterpret_cast<T*>(p.out_relu) + orow_l * p.ldo + co;
              st8(orl, relu4(v[0]), relu4(v[1]));
              if (two) st8(orl + 8, relu4(v[2]), relu4(v[3]));
            }
          };
          // software-pipelined TMEM drain: the load of chunk i+1 is in flight while chunk i is processed
          uint32_t ra[16], rb[16];
          if (ch_begin < ch_end) tmem_ld16(t_row + ch_begin * 16, ra);
          for (int ch = ch_begin; ch < ch_end; ch += 2) {
            tmem_ld_wait16(ra);
            if (ch + 1 < ch_end) tmem_ld16(t_row + (ch + 1) * 16, rb);
            process(ra, ch * 16);
            if (ch + 1 < ch_end) {
              tmem_ld_wait16(rb);
              if (ch + 2 < ch_end) tmem_ld16(t_row + (ch + 2) * 16, ra);
              process(rb, (ch + 1) * 16);
            }
          }
        } else if (EPI == VDA_EPI_LINEAR) {
          // ---- staged path: fp32 residual (optional) / fp32 or 16-bit output, no 16-bit residuals ----
          // SPEC folds the run-time epilogue flags of the three hot encoder GEMMs at compile time (the generic
          // version spends more instructions on flag tests, uniform loads and branches than on arithmetic):
          //   1: bias -> 16 bit (qkv)   2: bias, GELU -> 16 bit (fc1)   3: bias, LayerScale, fp32 residual -> fp32 (proj, fc2)
          //   5 / 6: as 1 / 2 with the preceding LayerNorm folded in (A holds the un-normalised 16-bit rows):
          //          out = rstd_r * (acc - mu_r * c1[n]) + c2[n], (mu_r, rstd_r) from the producer's row statistics
          constexpr bool fold = SPEC == 5 || SPEC == 6;
          const bool has_bias = SPEC != 0 ? true : p.bias != nullptr;
          const bool has_gamma = SPEC != 0 ? SPEC == 3 : p.gamma != nullptr;
          const int act = SPEC != 0 ? ((SPEC == 2 || SPEC == 6) ? VDA_ACT_GELU : VDA_ACT_NONE) : p.act;
          const bool has_res = SPEC != 0 ? SPEC == 3 : (p.res1 != nullptr && p.res1_f32);
          const bool out_f32 = SPEC != 0 ? SPEC == 3 : p.out_f32 != 0;
          const bool relu_copy = SPEC != 0 ? false : p.out_relu != nullptr;
          const bool has_r1h = SPEC != 0 ? false : (p.res1 != nullptr && !p.res1_f32);   // 16-bit residuals (RCU skips)
          const bool has_r2h = SPEC != 0 ? false : p.res2 != nullptr;
          const int nch = p.block_n >> 4;                                  // 16-column units in the tile
          const int c_begin = (eh ? (nch + 1) / 2 : 0) * 16;
          const int c_end = (eh ? nch : (nch + 1) / 2) * 16;
          // per-row base pointers (rows of this lane in the transposed passes), once per tile
          const float* rbase[8];
          char* obase[8];
          bool all_rows = true;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            rbase[it] = reinterpret_cast<const float*>(p.res1) + static_cast<long long>(rrow[it]) * p.ldr1;
            obase[it] = reinterpret_cast<char*>(p.out) + static_cast<long long>(orow[it]) * p.ldo * (out_f32 ? 4 : 2);
            all_rows = all_rows && orow[it] >= 0;
          }
          all_rows = __all_sync(0xffffffffu, all_rows);   // warp-uniform: the common full-tile case stores without row tests
          float rs_row[8], nm_row[8];                     // fold: rstd and -mu * rstd of the 8 rows of this lane
          if (fold) {
            // thread = row: Chan-merge the producer's partial (mean, M2) of row q*32 + lane, then hand the two scalars
            // to the lanes that hold the row in the transposed passes
            const long long grow = static_cast<long long>(m_blk) * BLOCK_M + q * 32 + lane;
            float mean = 0.f, m2 = 0.f, n = 0.f;
            if (grow < p.M) {
              const float nb = static_cast<float>(p.stat_cols);
              // all partials of the row are requested before the first one is used (the merge is a dependent chain: one
              // L2 round trip per partial sat in front of every tile -- 8.6 % of the epilogue warps' samples in fc1)
              constexpr int kMaxParts = 8;
              const float2* sp = p.stats_in + grow * p.stat_parts;
              for (int i0 = 0; i0 < p.stat_parts; i0 += kMaxParts) {
                float2 pm[kMaxParts];
#pragma unroll
                for (int i = 0; i < kMaxParts; ++i)
                  pm[i] = i0 + i < p.stat_parts ? sp[i0 + i] : make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < kMaxParts; ++i) {
                  if (i0 + i < p.stat_parts) {
                    const float delta = pm[i].x - mean;
                    const float nn = n + nb;
                    mean += delta * (nb / nn);
                    m2 += pm[i].y + delta * delta * (n * nb / nn);
                    n = nn;
                  }
                }
              }
            }
            const float rstd = rsqrtf(m2 * p.ln_inv_d + p.ln_eps);
            const float nm = -mean * rstd;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              rs_row[it] = __shfl_sync(0xffffffffu, rstd, it * 4 + rsub);
              nm_row[it] = __shfl_sync(0xffffffffu, nm, it * 4 + rsub);
            }
          }
          // residual row segments are loaded one chunk ahead (the first one before the accumulator is ready), so
          // their HBM/L2 latency hides behind the TMEM drain and the math of the previous chunk
          F4 rnxt[8];
          auto load_res = [&](int c0) {
            const int col = col_base + c0 + 4 * cg;
            const bool ok = col < p.N && (c0 + 32 <= c_end || cg < 4);
#pragma unroll
            for (int it = 0; it < 8; ++it)
              if (ok && orow[it] >= 0) rnxt[it] = load4f(rbase[it] + col);
          };
          // 16-bit residual row segments (4 columns = 8 bytes per lane and row), same one-chunk-ahead scheme
          uint2 r1h[8], r2h[8];
          auto load_resh = [&](int c0) {
            const int col = col_base + c0 + 4 * cg;
            const bool ok = col < p.N && (c0 + 32 <= c_end || cg < 4);
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              if (ok && orow[it] >= 0) {
                if (has_r1h)
                  r1h[it] = *reinterpret_cast<const uint2*>(reinterpret_cast<const T*>(p.res1) +
                                                            static_cast<long long>(rrow[it]) * p.ldr1 + col);
                if (has_r2h)
                  r2h[it] = *reinterpret_cast<const uint2*>(reinterpret_cast<const T*>(p.res2) +
                                                            static_cast<long long>(orow[it]) * p.ldo + col);
              }
            }
          };
          if (has_res && c_begin < c_end) load_res(c_begin);
          if ((has_r1h || has_r2h) && c_begin < c_end) load_resh(c_begin);
          // bias / LayerScale segments are fetched one chunk ahead as well (the first before the accumulator is
          // ready): loaded at their point of use, the L2 round trip sat in front of every chunk's math
          F4 bias_nxt = {}, gamma_nxt = {};
          auto load_bg = [&](int c0) {
            const int col = col_base + c0 + 4 * cg;
            if (col < p.N && (c0 + 32 <= c_end || cg < 4)) {
              if (has_bias) bias_nxt = load4f(p.bias + col);
              if (has_gamma) gamma_nxt = load4f(p.gamma + col);
              if (fold) gamma_nxt = load4f(p.ln_c1 + col);
            }
          };
          if (c_begin < c_end) load_bg(c_begin);
          mbar_wait(&tfull_bar[as], aphase);
          tc_fence_after();
          for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            const bool wide = c0 + 32 <= c_end;                            // 32 columns, else the last 16
            // ---- phase 1: accumulators (thread = row) -> swizzled staging tile ----
            // (issuing the tcgen05.ld of chunk c+1 before chunk c's math was tried: the 32 extra live registers push
            // the kernel over its 168-register cap and the spills cost more than the hidden latency: proj 115 -> 125 us)
            {
              uint32_t rr[32];
              if (wide) {
                tmem_ld32(t_row + c0, rr);
                tmem_ld_wait32(rr);
              } else {
                tmem_ld16(t_row + c0, *reinterpret_cast<uint32_t(*)[16]>(rr));
                tmem_ld_wait16(*reinterpret_cast<uint32_t(*)[16]>(rr));
              }
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4)
                if (wide || c4 < 4)
                  sts128(stg + stg_off(lane, c4), rr[4 * c4], rr[4 * c4 + 1], rr[4 * c4 + 2], rr[4 * c4 + 3]);
            }
            __syncwarp();
            // ---- phase 2: lane = 4 consecutive columns of 8 rows; coalesced row segments ----
            const int col = col_base + c0 + 4 * cg;
            const bool col_ok = col < p.N && (wide || cg < 4);
            F4 v[8];
            if (col_ok) {
              // loads, math and stores in separate unrolled passes: the 16 independent packed chains of a lane
              // are interleaved by the scheduler (the GELU chain alone is ~100 cycles deep)
#pragma unroll
              for (int it = 0; it < 8; ++it) v[it] = lds128(stg + stg_off(it * 4 + rsub, cg));
              const F4 bias4 = bias_nxt, gamma4 = gamma_nxt;
              if (c0 + 32 < c_end) load_bg(c0 + 32);
              if (fold) {
#pragma unroll
                for (int it = 0; it < 8; ++it) {   // rstd * acc + (-mu rstd * c1 + c2)
                  const float2 nm2 = make_float2(nm_row[it], nm_row[it]), rs2 = make_float2(rs_row[it], rs_row[it]);
                  v[it].a = __ffma2_rn(v[it].a, rs2, __ffma2_rn(nm2, gamma4.a, bias4.a));
                  v[it].b = __ffma2_rn(v[it].b, rs2, __ffma2_rn(nm2, gamma4.b, bias4.b));
                }
              } else if (has_bias) {
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = add4(v[it], bias4);
              }
              if (has_gamma) {
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = mul4(v[it], gamma4);
              }
              if (act == VDA_ACT_GELU) {
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = gelu4<T>(v[it]);
              } else if (act == VDA_ACT_RELU) {
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = relu4(v[it]);
              }
              if (has_res) {
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = add4(v[it], rnxt[it]);
              }
              if (has_r1h) {
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                  F4 r;
                  r.a = H16<T>::unpack2(r1h[it].x); r.b = H16<T>::unpack2(r1h[it].y);
                  v[it] = add4(v[it], r);
                }
              }
              if (has_r2h) {
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                  F4 r;
                  r.a = H16<T>::unpack2(r2h[it].x); r.b = H16<T>::unpack2(r2h[it].y);
                  v[it] = add4(v[it], r);
                }
              }
            }
            if (has_res && c0 + 32 < c_end) load_res(c0 + 32);   // next chunk's residual, consumed one iteration later
            if ((has_r1h || has_r2h) && c0 + 32 < c_end) load_resh(c0 + 32);
            if (col_ok) {
              const int cbyte = col * (out_f32 ? 4 : 2);
              auto store_row = [&](int it) {
                if (out_f32) store4f(reinterpret_cast<float*>(obase[it] + cbyte), v[it]);
                else store4h<T>(reinterpret_cast<T*>(obase[it] + cbyte), v[it]);
                if (relu_copy)
                  store4h<T>(reinterpret_cast<T*>(p.out_relu) + static_cast<long long>(orow[it]) * p.ldo + col, relu4(v[it]));
              };
              if (all_rows) {
#pragma unroll
                for (int it = 0; it < 8; ++it) store_row(it);
              } else {
#pragma unroll
                for (int it = 0; it < 8; ++it)
                  if (orow[it] >= 0) store_row(it);
              }
            }
            __syncwarp();
          }
        } else {  // VDA_EPI_GEGLU: tile columns are [a(half) | g(half)]; out[:, j] = (a + ba) * gelu(g + bg)
          const int half = p.geglu_half;
          const int nch = half >> 4;
          const int c_begin = (eh ? (nch + 1) / 2 : 0) * 16;
          const int c_end = (eh ? nch : (nch + 1) / 2) * 16;
          for (int c0 = c_begin; c0 < c_end; c0 += 32) {
            const bool wide = c0 + 32 <= c_end;
            const int pc = col_base + c0 + 4 * cg;                    // packed column of `a`
            const bool col_ok = pc < p.N && (wide || cg < 4);
            F4 gl[8];
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {                    // pass 0: gate columns, pass 1: value columns
              {
                uint32_t rr[32];
                const uint32_t ta = t_row + (pass == 0 ? half : 0) + c0;
                if (wide) {
                  tmem_ld32(ta, rr);
                  tmem_ld_wait32(rr);
                } else {
                  tmem_ld16(ta, *reinterpret_cast<uint32_t(*)[16]>(rr));
                  tmem_ld_wait16(*reinterpret_cast<uint32_t(*)[16]>(rr));
                }
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4)
                  if (wide || c4 < 4)
                    sts128(stg + stg_off(lane, c4), rr[4 * c4], rr[4 * c4 + 1], rr[4 * c4 + 2], rr[4 * c4 + 3]);
              }
              __syncwarp();
              if (col_ok) {
                const F4 b4 = load4f(p.bias + pc + (pass == 0 ? half : 0));
                F4 v[8];
#pragma unroll
                for (int it = 0; it < 8; ++it) v[it] = lds128(stg + stg_off(it * 4 + rsub, cg));
#pragma unroll
                for (int it = 0; it < 8; ++it) {
                  v[it] = add4(v[it], b4);
                  if (pass == 0) gl[it] = gelu4<T>(v[it]);
                  else v[it] = mul4(v[it], gl[it]);
                }
                if (pass == 1) {
                  const int oc = n_blk * half + c0 + 4 * cg;
#pragma unroll
                  for (int it = 0; it < 8; ++it)
                    if (orow[it] >= 0)
                      store4h<T>(reinterpret_cast<T*>(p.out) + static_cast<long long>(orow[it]) * p.ldo + oc, v[it]);
                }
              }
              __syncwarp();
            }
          }
        }
      }
      // one arrival per warp (a cluster-scope release per thread costs a fence each): every lane has waited for its
      // own tcgen05.ld, the warp converges, lane 0 signals the (leader's) issuer
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTA2 && rank != 0) mbar_arrive_leader(&tempty_bar[as]);
        else mbar_arrive(&tempty_bar[as]);
      }
      as ^= 1;
      if (as == 0) aphase ^= 1u;
    }
    if (EPI == VDA_EPI_LINEAR && SPEC == 4) {   // this lane's TMA stores have completed before the CTA retires
      if (elect_one()) bulk_wait<0>();
      __syncwarp();
    }
  }

  tc_fence_before();
  if (CTA2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (CTA2) tmem_dealloc2(tmem_base, p.tmem_cols);
    else tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(f);
  });
  return fn;
}

int make_tensor_map(CUtensorMap* m, int dtype, const void* base, int rank, const cuuint64_t* dims,
                    const cuuint64_t* strides_bytes, const cuuint32_t* box) {
  PFN_encodeTiled enc = get_encode();
  VDA_CHECK(enc != nullptr, "cuTensorMapEncodeTiled driver entry point not available");
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const bool sw64 = (dtype & kTmapSwizzle64) != 0;
  dtype &= ~kTmapSwizzle64;
  const CUtensorMapDataType cdt = dtype == kTmapF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                  : (dtype == VDA_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  CUresult r = enc(m, cdt,
                   static_cast<cuuint32_t>(rank), const_cast<void*>(base), dims, strides_bytes, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VDA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu %llu box %u %u)",
            static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)dims[1], box[0], box[1]);
  return 0;
}

int current_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  return dev;
}

// per-device caches: a process may drive several GPUs (one engine per device)
constexpr int kMaxDevices = 64;
int sm_count() {
  static int cached[kMaxDevices] = {};
  const int dev = current_device();
  if (dev >= 0 && dev < kMaxDevices && cached[dev] > 0) return cached[dev];
  int n = 0;
  if (dev < 0 || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  if (dev >= 0 && dev < kMaxDevices) cached[dev] = n;
  return n;
}

cudaError_t ensure_dynamic_smem(const void* kernel, size_t bytes) {
  static std::mutex mu;
  static std::unordered_map<const void*, size_t> opted[kMaxDevices];   // largest opt-in so far per (device, kernel)
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices)
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  std::lock_guard<std::mutex> lock(mu);
  auto it = opted[dev].find(kernel);
  if (it != opted[dev].end() && it->second >= bytes) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e == cudaSuccess) opted[dev][kernel] = bytes;
  return e;
}

static int pick_block_n(int N, int tiles_m) {
  int bn;
  if (N <= 256) {
    bn = (N + 15) / 16 * 16;
  } else {
    bn = 128;
    for (int c = 256; c >= 128; c -= 16)
      if (N % c == 0) { bn = c; break; }
  }
  // fill the machine: halve wide tiles while there are fewer tiles than SMs
  while (bn >= 128 && bn % 32 == 0 && tiles_m * ((N + bn - 1) / bn) < sm_count()) bn /= 2;
  return bn;
}

template <typename T, int EPI, bool CONV, bool STAGED, int SPEC, bool CTA2>
static int launch2(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmD,
                   const GemmDev& d, size_t smem, cudaStream_t st) {
  auto kfn = gemm_kernel<T, EPI, CONV, STAGED, SPEC, CTA2>;
  VDA_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(kfn), smem));   // per (kernel, device)
  const bool pdl = pdl_enabled();
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (!CTA2) {
    cfg.gridDim = dim3(d.num_tiles < sm_count() ? d.num_tiles : sm_count());
  } else {
    // CTA pairs: clusters of 2 (same TPC), one tile pair per cluster and round
    int pairs = sm_count() / 2;
    if (d.num_tiles < pairs) pairs = d.num_tiles;
    cfg.gridDim = dim3(2 * pairs);
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = 2;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {   // programmatic dependent launch: our prologue overlaps the predecessor's tail (see pdl_wait in the kernel)
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  VDA_CUDA(cudaLaunchKernelEx(&cfg, kfn, tmA, tmB, tmC, tmD, d));
  VDA_CUDA(cudaGetLastError());
  return 0;
}
struct Maps { CUtensorMap a, b, c, d; };   // c / d: fp32 residual-output and 16-bit copy tile maps (SPEC 4 only; else copies of a)
template <typename T, int EPI, bool CONV, bool STAGED, int SPEC = 0>
static int launch(const Maps& tm, const GemmDev& d, size_t smem, cudaStream_t st) {
  if (d.pair) return launch2<T, EPI, CONV, STAGED, SPEC, true>(tm.a, tm.b, tm.c, tm.d, d, smem, st);
  return launch2<T, EPI, CONV, STAGED, SPEC, false>(tm.a, tm.b, tm.c, tm.d, d, smem, st);
}

template <typename T>
static int dispatch(const vda_gemm_params* p, const Maps& tm, const GemmDev& d, int spec, size_t smem, cudaStream_t st) {
  const bool conv = p->a_mode == VDA_A_CONV3;
  switch (p->epilogue) {
    case VDA_EPI_LINEAR:
      // compile-time specialisations of the hot encoder epilogues (see SPEC in the kernel; chosen by pick_spec)
      switch (spec) {
        case 1: return launch<T, VDA_EPI_LINEAR, false, true, 1>(tm, d, smem, st);
        case 2: return launch<T, VDA_EPI_LINEAR, false, true, 2>(tm, d, smem, st);
        case 3: return launch<T, VDA_EPI_LINEAR, false, true, 3>(tm, d, smem, st);
        case 4: return launch<T, VDA_EPI_LINEAR, false, true, 4>(tm, d, smem, st);
        case 5: return launch<T, VDA_EPI_LINEAR, false, true, 5>(tm, d, smem, st);
        case 6: return launch<T, VDA_EPI_LINEAR, false, true, 6>(tm, d, smem, st);
        default: break;
      }
      return conv ? launch<T, VDA_EPI_LINEAR, true, true>(tm, d, smem, st)
                  : launch<T, VDA_EPI_LINEAR, false, true>(tm, d, smem, st);
    case VDA_EPI_GEGLU:
      VDA_CHECK(!conv, "GEGLU epilogue is only defined for plain GEMMs");
      return launch<T, VDA_EPI_GEGLU, false, true>(tm, d, smem, st);
    case VDA_EPI_CONVT:
      VDA_CHECK(!conv, "CONVT epilogue is only defined for plain GEMMs");
      return launch<T, VDA_EPI_CONVT, false, false>(tm, d, smem, st);
    case VDA_EPI_TAIL:
      return conv ? launch<T, VDA_EPI_TAIL, true, false>(tm, d, smem, st)
                  : launch<T, VDA_EPI_TAIL, false, false>(tm, d, smem, st);
  }
  set_error("unknown epilogue %d", p->epilogue);
  return 1;
}

// Which compile-time specialised epilogue serves this problem (0 = generic).  block_n is known.
static int pick_spec(const vda_gemm_params* p, const GemmDev& d) {
  if (p->epilogue != VDA_EPI_LINEAR || p->a_mode == VDA_A_CONV3) return 0;
  const bool plain16 = p->bias && !p->res1 && !p->res2 && !p->out_f32 && !p->out_relu && !p->gamma && p->row_group == 0;
  if (plain16 && p->row_stats_in) return p->act == VDA_ACT_GELU ? 6 : (p->act == VDA_ACT_NONE ? 5 : 0);
  if (plain16 && p->act == VDA_ACT_NONE) return 1;
  if (plain16 && p->act == VDA_ACT_GELU) return 2;
  if (p->bias && p->gamma && p->res1 && p->res1_f32 && !p->res2 && p->out_f32 && !p->out_relu && p->act == VDA_ACT_NONE &&
      p->row_group == 0) {
    // fp32 residual stream: all tile traffic by TMA when the residual is updated in place and the tile geometry allows
    // 32-column boxes (SPEC 4); otherwise the register-staged epilogue (SPEC 3)
    const bool tma_ok = p->res1 == p->out && p->ldr1 == p->ldo && d.block_n % 64 == 0 && p->N % d.block_n == 0 &&
                        (p->ldo % 4) == 0;
    if (tma_ok) return 4;
    return (p->out16 || p->row_stats_out) ? -1 : 3;
  }
  return 0;
}

}  // namespace vda

using namespace vda;

extern "C" int vda_gemm(const vda_gemm_params* p, void* stream) {
  VDA_CHECK(p != nullptr, "null params");
  VDA_CHECK(p->M > 0 && p->N > 0 && p->K > 0, "bad GEMM shape %d %d %d", p->M, p->N, p->K);
  VDA_CHECK(p->dtype == VDA_BF16 || p->dtype == VDA_FP16, "bad dtype %d", p->dtype);
  VDA_CHECK(p->N % 8 == 0, "N (%d) must be a multiple of 8", p->N);
  VDA_CHECK(p->K % 8 == 0, "K (%d) must be a multiple of 8", p->K);
  VDA_CHECK((reinterpret_cast<uintptr_t>(p->A) & 15) == 0 && (reinterpret_cast<uintptr_t>(p->Wt) & 15) == 0,
            "A / Wt must be 16-byte aligned");
  VDA_CHECK(p->out != nullptr && (reinterpret_cast<uintptr_t>(p->out) & 15) == 0, "out must be 16-byte aligned");
  const bool conv = p->a_mode == VDA_A_CONV3;

  GemmDev d = {};
  d.M = p->M; d.N = p->N; d.K = p->K;
  d.num_k_blocks = (p->K + BLOCK_K - 1) / BLOCK_K;
  d.prefetch_max_kb = 32;
  Maps tm;
  CUtensorMap& tmA = tm.a;
  CUtensorMap& tmB = tm.b;

  // Weights as a hi | lo pair of 16-bit matrices (validation precision): Wt is [N, 2 * Ka'] with Ka' = a_k rounded up to a
  // k-block, the second half holding the 16-bit rounding residue of the first; A ([M, a_k]) is walked twice.
  const int a_k = p->a_k > 0 ? p->a_k : p->K;
  const int a_kp = (a_k + BLOCK_K - 1) / BLOCK_K * BLOCK_K;
  VDA_CHECK(p->a_k <= 0 || p->K == 2 * a_kp, "hi|lo weights: K (%d) must be 2 * round_up(a_k = %d, 64)", p->K, p->a_k);
  d.a_k_blocks = a_kp / BLOCK_K;
  if (conv) {
    VDA_CHECK(p->C % 64 == 0 && a_k == 9 * p->C, "conv mode needs C %% 64 == 0 and K == 9*C (C=%d K=%d)", p->C, a_k);
    VDA_CHECK(p->M == p->n_img * p->H * p->W, "conv mode: M must be n_img*H*W");
    d.H = p->H; d.W = p->W;
    // pick the 128-pixel box shape (bw x bh) wasting the fewest out-of-image pixels
    const int cand[5][2] = {{16, 8}, {32, 4}, {8, 16}, {64, 2}, {128, 1}};
    long long best = -1;
    for (int i = 0; i < 5; ++i) {
      const long long tx = (p->W + cand[i][0] - 1) / cand[i][0], ty = (p->H + cand[i][1] - 1) / cand[i][1];
      if (best < 0 || tx * ty < best) { best = tx * ty; d.bw = cand[i][0]; d.bh = cand[i][1]; }
    }
    d.tiles_x = (p->W + d.bw - 1) / d.bw;
    d.tiles_y = (p->H + d.bh - 1) / d.bh;
    d.tiles_m = d.tiles_x * d.tiles_y * p->n_img;
    d.cblocks = p->C / 64;
    cuuint64_t dims[4] = {(cuuint64_t)p->C, (cuuint64_t)p->W, (cuuint64_t)p->H, (cuuint64_t)p->n_img};
    cuuint64_t strides[3] = {(cuuint64_t)p->C * 2, (cuuint64_t)p->C * 2 * p->W, (cuuint64_t)p->C * 2 * p->W * p->H};
    cuuint32_t box[4] = {64, (cuuint32_t)d.bw, (cuuint32_t)d.bh, 1};
    if (make_tensor_map(&tmA, p->dtype, p->A, 4, dims, strides, box)) return 1;
  } else {
    VDA_CHECK(p->lda >= a_k && p->lda % 8 == 0, "lda (%lld) must be >= K and a multiple of 8", (long long)p->lda);
    d.tiles_m = (p->M + BLOCK_M - 1) / BLOCK_M;
    cuuint64_t dims[2] = {(cuuint64_t)a_k, (cuuint64_t)p->M};
    cuuint64_t strides[1] = {(cuuint64_t)p->lda * 2};
    cuuint32_t box[2] = {64, 128};
    if (make_tensor_map(&tmA, p->dtype, p->A, 2, dims, strides, box)) return 1;
  }

  if (p->epilogue == VDA_EPI_GEGLU) {
    VDA_CHECK(p->geglu_half > 0 && p->geglu_half % 16 == 0 && p->geglu_half <= 128 &&
                  p->N % (2 * p->geglu_half) == 0,
              "GEGLU: N must be a multiple of 2*geglu_half (<=256)");
    d.block_n = 2 * p->geglu_half;
  } else if (p->epilogue == VDA_EPI_TAIL) {
    VDA_CHECK(p->N == 32 && p->tail_w && p->bias, "TAIL epilogue needs N == 32, bias and tail_w");
    d.block_n = 32;
  } else {
    d.block_n = pick_block_n(p->N, d.tiles_m);
  }
  if (p->epilogue == VDA_EPI_CONVT) {
    VDA_CHECK(p->convt_s > 0 && p->convt_co % 8 == 0 && p->N == p->convt_s * p->convt_s * p->convt_co && p->bias &&
                  p->M % (p->in_h * p->in_w) == 0,
              "CONVT: inconsistent shape");
  }
  if (p->epilogue == VDA_EPI_LINEAR) {
    VDA_CHECK(p->ldo % 8 == 0 && (!p->res1 || p->ldr1 % 8 == 0), "ldo / ldr1 must be multiples of 8");
  }
  d.tiles_n = (p->N + d.block_n - 1) / d.block_n;
  d.num_tiles = d.tiles_m * d.tiles_n;
  // CTA pairs (cta_group::2, M = 256): when there are enough 256-row tile pairs to fill the 74 TPCs; each CTA then
  // loads only block_n/2 rows of B per stage
  // (not for K <= 256: those GEMMs are bound by their output stream, measured slower in pair mode)
  d.pair = (p->epilogue != VDA_EPI_TAIL && d.block_n % 32 == 0 && d.tiles_m >= 2 && d.num_k_blocks >= 8 &&
            ((d.tiles_m + 1) / 2) * d.tiles_n >= sm_count() / 2) ? 1 : 0;
  if (d.pair) d.num_tiles = ((d.tiles_m + 1) / 2) * d.tiles_n;
  const uint32_t b_rows = d.pair ? d.block_n / 2 : d.block_n;   // B rows loaded (and stored) per CTA and stage
  {
    cuuint64_t dims[2] = {(cuuint64_t)p->K, (cuuint64_t)p->N};
    cuuint64_t strides[1] = {(cuuint64_t)p->K * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)b_rows};
    if (make_tensor_map(&tmB, p->dtype, p->Wt, 2, dims, strides, box)) return 1;
  }
  d.tx_bytes = kABytes + b_rows * BLOCK_K * 2;
  d.stage_bytes = d.tx_bytes;
  // block_n*128 is a multiple of 2048 only when block_n % 16 == 0 -> every stage stays 1024-byte aligned
  d.stage_bytes = (d.stage_bytes + 1023u) & ~1023u;
  // 227 KB per CTA: 1 KB alignment slack + static barriers, the epilogue staging tiles, the rest for the operand ring
  // LINEAR epilogue variant (measured with tools/bench_gemm.py): the shared-memory transpose (coalesced row segments
  // for every residual load and store) wins for all LINEAR epilogues, 16-bit residuals included (RCU conv @148^2:
  // 703 -> 627 us); the row-per-thread path remains for CONVT.
  d.staged = (p->epilogue == VDA_EPI_GEGLU || p->epilogue == VDA_EPI_LINEAR) ? 1 : 0;
  const int spec = pick_spec(p, d);
  VDA_CHECK(spec >= 0, "out16 / row_stats_out need the in-place fp32 residual epilogue with N %% block_n == 0 and "
                       "block_n %% 64 == 0 (N=%d block_n=%d)", p->N, d.block_n);
  VDA_CHECK(spec == 4 || (!p->out16 && !p->row_stats_out), "out16 / row_stats_out: unsupported epilogue combination");
  VDA_CHECK((spec == 5 || spec == 6) == (p->row_stats_in != nullptr), "row_stats_in: unsupported epilogue combination");
  // epilogue staging: 8 transposition tiles of 4 KB, or (SPEC 4) 8 x 2 TMA boxes of 4 KB
  d.epi_nbuf = d.num_k_blocks >= 32 ? 1 : 2;
  d.epi_warp_bytes = static_cast<uint32_t>(d.epi_nbuf) * 4096u + (p->out16 ? 2048u : 0u);
  const uint32_t staging = spec == 4 ? kEpiWarps * d.epi_warp_bytes : (d.staged ? kStagingBytes : 0u);
  int stages = static_cast<int>((227u * 1024u - 1024u - 512u - staging) / d.stage_bytes);
  if (stages > kMaxStages) stages = kMaxStages;
  d.stages = stages;
  const size_t smem = static_cast<size_t>(stages) * d.stage_bytes + staging + 1024;
  uint32_t cols = 32;
  while (cols < 2u * d.block_n) cols <<= 1;
  d.tmem_cols = cols;
  d.acc_stride = cols / 2;

  d.bias = p->bias; d.gamma = p->gamma; d.act = p->act;
  d.res1 = p->res1; d.ldr1 = p->ldr1; d.res1_f32 = p->res1_f32; d.res2 = p->res2;
  d.out = p->out; d.ldo = p->ldo; d.out_f32 = p->out_f32; d.out_relu = p->out_relu;
  d.row_group = p->row_group; d.geglu_half = p->geglu_half;
  d.convt_s = p->convt_s; d.convt_co = p->convt_co; d.in_h = p->in_h; d.in_w = p->in_w;
  d.tail_w = p->tail_w; d.tail_b = p->tail_b;

  tm.c = tm.a;
  tm.d = tm.a;
  if (spec == 4) {
    cuuint64_t dims[2] = {(cuuint64_t)p->N, (cuuint64_t)p->M};
    cuuint64_t strides[1] = {(cuuint64_t)p->ldo * 4};
    cuuint32_t box[2] = {32, 32};
    if (make_tensor_map(&tm.c, kTmapF32, p->out, 2, dims, strides, box)) return 1;
    if (p->out16) {
      VDA_CHECK((reinterpret_cast<uintptr_t>(p->out16) & 15) == 0, "out16 must be 16-byte aligned");
      cuuint64_t strides16[1] = {(cuuint64_t)p->ldo * 2};
      if (make_tensor_map(&tm.d, p->dtype | kTmapSwizzle64, p->out16, 2, dims, strides16, box)) return 1;
    }
    d.out16 = p->out16;
    d.stats_out = reinterpret_cast<float2*>(p->row_stats_out);
    d.stat_parts = 2 * d.tiles_n;
    d.stat_cols = d.block_n / 2;
    VDA_CHECK(!p->row_stats_out || p->stat_parts == d.stat_parts,
              "row_stats_out: caller expects %d parts, the kernel writes %d (see vda_gemm_rowstat_layout)", p->stat_parts,
              d.stat_parts);
  }
  if (spec == 5 || spec == 6) {
    VDA_CHECK(p->ln_c1 && p->stat_parts > 0 && p->stat_cols > 0 && p->stat_parts * p->stat_cols == p->K,
              "LayerNorm fold: need ln_c1 and a statistics layout covering K (parts %d x cols %d, K %d)", p->stat_parts,
              p->stat_cols, p->K);
    d.stats_in = reinterpret_cast<const float2*>(p->row_stats_in);
    d.ln_c1 = p->ln_c1;
    d.stat_parts = p->stat_parts;
    d.stat_cols = p->stat_cols;
    d.ln_eps = p->ln_eps;
    d.ln_inv_d = 1.f / static_cast<float>(p->K);
  }

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (p->dtype == VDA_BF16) return dispatch<__nv_bfloat16>(p, tm, d, spec, smem, st);
  return dispatch<__half>(p, tm, d, spec, smem, st);
}

// Layout of the per-row partial statistics a GEMM with row_stats_out writes for an [M, N] output: `parts` partials
// per row, each over `part_cols` consecutive columns (the column halves of the kernel's N tiles).
extern "C" int vda_gemm_rowstat_layout(int M, int N, int* parts, int* part_cols) {
  VDA_CHECK(M > 0 && N > 0 && parts && part_cols, "bad arguments");
  const int bn = pick_block_n(N, (M + BLOCK_M - 1) / BLOCK_M);
  VDA_CHECK(bn % 64 == 0 && N % bn == 0, "no row-statistics layout for N=%d (block_n=%d)", N, bn);
  *parts = 2 * (N / bn);
  *part_cols = bn / 2;
  return 0;
}
