// Spatial ViT attention (dinov2_layers/attention.py:49-62) as a tcgen05 / TMEM / TMA flash-attention kernel.
//
//   out[f, n, h, :] = softmax_n'( q[f,n,h,:] . k[f,n',h,:] / sqrt(64) ) v[f,n',h,:]       d = 64, N ~ 1370..2443
//
// Persistent kernel, one CTA (384 threads = 3 warpgroups) per SM.  A CTA runs TWO independent tile streams
// (t = 0 / 1), each made of one MMA-issuing warp and one softmax warpgroup that owns a 128-query tile:
//   warp 0      TMA producer: Q tiles once per item, K / V tiles (128 keys x 64) through two 3-slot rings
//   warp 1 / 2  tcgen05.mma issuer of stream 0 / 1:  S = Q K^T  (SS form, 128 x kv x 64)  and  O += P V  (TS form:
//               P is read from TMEM, V from smem as an MN-major operand -- no transpose of V anywhere).  S of step
//               j+1 is issued before P V of step j.  One issuer per stream: a stream never waits for the other
//               stream's softmax (round 1 had one issuer walking S0 S1 PV0 PV1 in a fixed order, which cost each
//               warpgroup ~500 cycles per step in front of its P store)
//   warp 3      idle (donates registers: setmaxnreg.dec on warpgroup 0, .inc on the softmax warpgroups)
//   warps 4-7   softmax warpgroup of stream 0      \  one thread per query row: the 128 scores of a row are read
//   warps 8-11  softmax warpgroup of stream 1      /  from TMEM straight into that thread's registers (no shuffles)
// Work items (one flat list per CTA; the K / V rings never drain between items, Q is double-buffered):
//   PAIR    two neighbouring query tiles of one (frame, head): both streams consume every K / V tile (one L2 -> smem
//           load serves 2 x 128 queries)
//   SPLIT   the odd last query tile of a (frame, head) (N = 1370: 11 tiles): ONE query tile whose key tiles are
//           divided between the streams (stream 0: tiles 0..ja-1, stream 1: ja..n_kv-1, loaded interleaved); the two
//           partial results (m, l, O) are merged through shared memory by warpgroup 0 (standard split-KV flash merge).
//           Round 1 ran these items on one stream with the other idle (8 % of the kernel's time)
//   SINGLE  the same odd tile on stream 0 only (when there is just one key tile)
// Every `empty` barrier (K / V slots, Q buffers) expects TWO arrivals per use: one tcgen05.commit from each stream that
// consumes the use; for a use only one stream consumes, the PRODUCER arrives in place of the other stream right after
// issuing the load.  A stream therefore never waits on, or acknowledges, a slot it does not read -- it only counts
// it (slot = use index mod ring depth).  (A first version let the non-owner acknowledge the slot when its cursor
// walked past it; the S look-ahead then waited for tiles the producer could only load after an acknowledgement
// that sat behind that very wait: a deadlock whenever a stream had two foreign uses in a row.)
// TMEM (512 columns): S_0 | S_1 (128 fp32 columns each), O_0 | O_1 (64), P_0 | P_1 (64: 128 packed 16-bit keys).
// Because a warpgroup copies S to registers before it starts the exponentials, the issuer refills S with the next
// key tile immediately (s_free); P has its own columns, so S(j+1) never waits for O += P(j) V(j).
// Online softmax in fp32 with lazy rescaling: O / l are only rescaled when the running row maximum grows by more
// than 2^8 (rare after the first key tiles), done by the owning warp through a TMEM round trip.
// The kernel is bound by the instruction issue of the softmax warps (MUFU.EX2: 16/clk/SM), see DESIGN.md.
#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

namespace sa {
constexpr int BM = 128;            // queries per tile
constexpr int BN = 128;            // keys per tile
constexpr int D = 64;              // head dim
constexpr int KS = 3, VS = 3;      // K / V ring depth
constexpr int THREADS = 384;
constexpr int REGS_CTRL = 56, REGS_SOFTMAX = 224;   // setmaxnreg budgets: 128*56 + 256*224 <= 64K
constexpr uint32_t TILE_BYTES = BM * D * 2;   // 16 KB: one Q, K or V tile
constexpr uint32_t XCH_FLOATS = (D + 2) * BM; // split-item exchange: O_1 [64][128], m_1 [128], l_1 [128]
constexpr uint32_t SMEM_BYTES = (4 + KS + VS) * TILE_BYTES + XCH_FLOATS * 4 + 1024;   // Q: 2 buffers x 2 tiles
// TMEM columns
constexpr uint32_t COL_S = 0, COL_O = 256, COL_P = 384;
constexpr float RESCALE_LOG2 = 8.0f;
constexpr int POLY_MASK = 3;       // pair p of a score row takes exp2_poly2 when (p & POLY_MASK) == POLY_MASK: 25 %
enum { PAIR = 0, SPLIT = 1, SINGLE = 2 };
enum { BAR_XCH_FULL = 1, BAR_XCH_EMPTY = 2 };   // named barriers (0 is __syncthreads)
}  // namespace sa

struct SaParams {
  int N, heads, frames;
  int n_qt;            // query tiles per (frame, head)
  int n_pairs;         // full pairs of query tiles per (frame, head)
  int n_items;         // FH * n_pairs + (n_qt odd ? FH : 0)
  int n_kv;            // key tiles
  int ja;              // split items: stream 0 takes key tiles [0, ja), stream 1 [ja, n_kv)
  int split;           // odd tiles are SPLIT items (else SINGLE)
  void* out;
};

struct SaItem {
  int frame, head, q0;   // q0: first query row of tile A
  int kind;
};

__device__ __forceinline__ SaItem sa_decode(const SaParams& p, int item) {
  SaItem it;
  const int fh_total = p.frames * p.heads;
  int fh, tile;
  if (item < fh_total * p.n_pairs) {
    fh = item / p.n_pairs;
    tile = 2 * (item - fh * p.n_pairs);
    it.kind = sa::PAIR;
  } else {
    fh = item - fh_total * p.n_pairs;
    tile = p.n_qt - 1;
    it.kind = p.split ? sa::SPLIT : sa::SINGLE;
  }
  it.frame = fh / p.heads;
  it.head = fh - it.frame * p.heads;
  it.q0 = tile * sa::BM;
  return it;
}
__device__ __forceinline__ int sa_kind(const SaParams& p, int item) {
  return item < p.frames * p.heads * p.n_pairs ? sa::PAIR : (p.split ? sa::SPLIT : sa::SINGLE);
}
// does stream t consume ring use u (the u-th K / V tile loaded for an item of this kind)?
__device__ __forceinline__ bool sa_mine(int kind, int t, int u) {
  return kind == sa::PAIR ? true : (kind == sa::SINGLE ? t == 0 : (u & 1) == t);
}
// key tile loaded by ring use u
__device__ __forceinline__ int sa_tile(const SaParams& p, int kind, int u) {
  return kind == sa::SPLIT ? ((u & 1) ? p.ja + (u >> 1) : (u >> 1)) : u;
}

__device__ __forceinline__ int sa_kv_cols(const SaParams& p, int j) {   // columns of key tile j, rounded up to 32
  const int valid = p.N - j * sa::BN;
  return valid >= sa::BN ? sa::BN : ((valid + 31) & ~31);
}

// exp2 on the FMA / ALU pipes for a pair of values (Cody-Waite: x = j + f, j = round(x), f in [-0.5, 0.5];
// 2^f by a degree-3 minimax polynomial, max rel. error 7.7e-5 -- below the 16-bit rounding of P; 2^j by adding j
// to the exponent field).  A quarter of the exponentials of a score tile take this path so that the MUFU (16 ex2/clk/SM)
// is no longer the only unit that can produce them.
__device__ __forceinline__ float2 exp2_poly2(float2 x) {
  x.x = fmaxf(x.x, -126.f);
  x.y = fmaxf(x.y, -126.f);
  const float2 t = __fadd2_rn(x, make_float2(12582912.f, 12582912.f));          // 1.5 * 2^23: integer part in the low bits
  const float2 j = __fadd2_rn(t, make_float2(-12582912.f, -12582912.f));
  const float2 f = __ffma2_rn(j, make_float2(-1.f, -1.f), x);   // x - j in one packed op (a negated operand costs two scalar FADDs)
  float2 q = __ffma2_rn(make_float2(5.508868381e-02f, 5.508868381e-02f), f, make_float2(2.426040515e-01f, 2.426040515e-01f));
  q = __ffma2_rn(q, f, make_float2(6.932762417e-01f, 6.932762417e-01f));
  q = __ffma2_rn(q, f, make_float2(9.999289404e-01f, 9.999289404e-01f));
  float2 r;
  r.x = __int_as_float(__float_as_int(q.x) + (__float_as_int(t.x) << 23));
  r.y = __int_as_float(__float_as_int(q.y) + (__float_as_int(t.y) << 23));
  return r;
}

template <int N>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }

template <typename T>
__global__ void __launch_bounds__(sa::THREADS, 1)
spatial_attention_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const SaParams p) {
  using namespace sa;
  pdl_trigger();   // the proj GEMM that follows (launched with the PDL attribute) may be scheduled as our CTAs retire
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t q_full[2], q_empty[2];
  __shared__ __align__(8) uint64_t k_full[KS], k_empty[KS], v_full[VS], v_empty[VS];
  __shared__ __align__(8) uint64_t s_ready[2], s_free[2], p_ready[2], o_done[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  // smem map: Q[buffer 0: A, B | buffer 1: A, B] | K[KS] | V[VS] | split-item exchange
  const uint32_t offQ = 0, offK = 4 * TILE_BYTES, offV = (4 + KS) * TILE_BYTES, offX = (4 + KS + VS) * TILE_BYTES;
  const int n_my = (p.n_items - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) /
                   static_cast<int>(gridDim.x);   // items of this CTA: blockIdx.x + i * gridDim.x

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQKV);
    for (int s = 0; s < 2; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 2); }
    for (int s = 0; s < KS; ++s) { mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 2); }
    for (int s = 0; s < VS; ++s) { mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 2); }
    for (int t = 0; t < 2; ++t) {
      mbar_init(&s_ready[t], 1);
      mbar_init(&s_free[t], 128);
      mbar_init(&p_ready[t], 128);
      mbar_init(&o_done[t], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp < 4) {
    reg_dec<REGS_CTRL>();
    if (warp == 0 && lane == 0) {
      // ===================================== TMA producer =====================================
      int ks = 0, vs = 0;
      uint32_t kph = 0, vph = 0;
      for (int i = 0; i < n_my; ++i) {
        const SaItem it = sa_decode(p, blockIdx.x + i * gridDim.x);
        const int qb = i & 1;
        uint8_t* sQ = smem_gen + offQ + qb * 2 * TILE_BYTES;
        mbar_wait(&q_empty[qb], ((i >> 1) & 1u) ^ 1u);
        mbar_arrive_expect_tx(&q_full[qb], it.kind == PAIR ? 2 * TILE_BYTES : TILE_BYTES);
        tma_load_4d(sQ, &tmQKV, &q_full[qb], 0, it.head, it.q0, it.frame);
        if (it.kind == PAIR) tma_load_4d(sQ + TILE_BYTES, &tmQKV, &q_full[qb], 0, it.head, it.q0 + BM, it.frame);
        if (it.kind == SINGLE) mbar_arrive(&q_empty[qb]);          // stream 1 never reads this Q buffer
        for (int u = 0; u < p.n_kv; ++u) {
          const int j = sa_tile(p, it.kind, u);
          const bool both = it.kind == PAIR;                      // else exactly one stream consumes this use
          mbar_wait(&k_empty[ks], kph ^ 1u);
          mbar_arrive_expect_tx(&k_full[ks], TILE_BYTES);
          tma_load_4d(smem_gen + offK + ks * TILE_BYTES, &tmQKV, &k_full[ks], 0, p.heads + it.head, j * BN, it.frame);
          if (!both) mbar_arrive(&k_empty[ks]);                   // (counts for the phase that has just begun)
          if (++ks == KS) { ks = 0; kph ^= 1u; }
          mbar_wait(&v_empty[vs], vph ^ 1u);
          mbar_arrive_expect_tx(&v_full[vs], TILE_BYTES);
          tma_load_4d(smem_gen + offV + vs * TILE_BYTES, &tmQKV, &v_full[vs], 0, 2 * p.heads + it.head, j * BN,
                      it.frame);
          if (!both) mbar_arrive(&v_empty[vs]);
          if (++vs == VS) { vs = 0; vph ^= 1u; }
        }
      }
    } else if (warp == 1 || warp == 2) {
      // ===================================== MMA issuer of stream t ============================
      // The whole warp runs the (warp-uniform) control flow; one elected lane issues the tcgen05 instructions.
      const int t = warp - 1;
      int ks = 0, vs = 0;
      uint32_t kph = 0, vph = 0;
      uint32_t n_s = 0, n_pv = 0;          // running counts of S / PV tiles issued by this stream
      int ki = 0, ku = 0, vi = 0, vu = 0;  // cursors over the flat (item, ring use) sequence of the K and V rings
      int s_item = -1, pv_item = -1;       // item of this stream's latest S / PV (first-use detection)
      const uint32_t idesc_pv = umma_idesc(H16<T>::kUmmaFmt, D) | kIdescBMnMajor;
      const int stride = static_cast<int>(gridDim.x);

      // Advance the K cursor to this stream's next own use and issue its S; uses of the other stream are only counted
      // (ring slot / phase follow from the use count).  false: the item list is exhausted.
      auto next_s = [&]() -> bool {
        while (ki < n_my) {
          const int kind = sa_kind(p, static_cast<int>(blockIdx.x) + ki * stride);
          const bool mine = sa_mine(kind, t, ku);
          const int qb = ki & 1;
          if (mine) {
            mbar_wait(&k_full[ks], kph);
            if (s_item != ki) {                         // first S of the item: its Q tile(s) must have landed
              mbar_wait(&q_full[qb], (ki >> 1) & 1u);
              s_item = ki;
            }
            const int cols = sa_kv_cols(p, sa_tile(p, kind, ku));
            const uint32_t idesc = umma_idesc(H16<T>::kUmmaFmt, static_cast<uint32_t>(cols));
            const uint64_t db = umma_desc_sw128(smem_base + offK + ks * TILE_BYTES);
            const uint64_t da = umma_desc_sw128(smem_base + offQ + (qb * 2 + (kind == PAIR ? t : 0)) * TILE_BYTES);
            mbar_wait(&s_free[t], (n_s & 1u) ^ 1u);     // the warpgroup has copied the previous S to registers
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < D / 16; ++k) umma_f16(tmem_base + COL_S + t * BN, da + 2u * k, db + 2u * k, idesc, k);
              umma_commit(&s_ready[t]);
              umma_commit(&k_empty[ks]);
            }
            __syncwarp();
            ++n_s;
          }
          if (ku == p.n_kv - 1 && s_item == ki) {       // end of an item this stream read Q for: release the Q buffer
            if (elect_one()) umma_commit(&q_empty[qb]); // ... once its S MMAs have retired
            __syncwarp();
          }
          if (++ks == KS) { ks = 0; kph ^= 1u; }
          if (++ku == p.n_kv) { ku = 0; ++ki; }
          if (mine) return true;
        }
        return false;
      };
      // Same walk over the V ring: O += P V of this stream's next own use.
      auto next_pv = [&]() -> bool {
        while (vi < n_my) {
          const int kind = sa_kind(p, static_cast<int>(blockIdx.x) + vi * stride);
          const bool mine = sa_mine(kind, t, vu);
          if (mine) {
            mbar_wait(&v_full[vs], vph);
            const int nk = sa_kv_cols(p, sa_tile(p, kind, vu)) >> 4;
            const uint64_t db = umma_desc_sw128_mn(smem_base + offV + vs * TILE_BYTES);
            const uint32_t acc0 = pv_item == vi ? 1u : 0u;   // first P V of an item overwrites O
            pv_item = vi;
            mbar_wait(&p_ready[t], n_pv & 1u);
            tc_fence_after();
            if (elect_one()) {
              for (int k = 0; k < nk; ++k)   // 16 keys per MMA: 8 TMEM columns of P, 16 rows (2048 B) of V
                umma_f16_ts(tmem_base + COL_O + t * D, tmem_base + COL_P + t * (BN / 2) + 8u * k, db + 128u * k,
                            idesc_pv, (acc0 | static_cast<uint32_t>(k)) != 0u ? 1u : 0u);
              umma_commit(&o_done[t]);
              umma_commit(&v_empty[vs]);
            }
            __syncwarp();
            ++n_pv;
          }
          if (++vs == VS) { vs = 0; vph ^= 1u; }
          if (++vu == p.n_kv) { vu = 0; ++vi; }
          if (mine) return true;
        }
        return false;
      };

      bool have = next_s();
      while (have) {
        const bool nxt = next_s();   // S of the next step of the flat stream (next key tile, or the next item's first)
        next_pv();                   // O += P V of the current step
        have = nxt;
      }
    }
  } else {
    // ===================================== softmax warpgroups ===============================
    reg_inc<REGS_SOFTMAX>();
    const int t = (warp - 4) >> 2;                    // stream / query tile handled by this warpgroup
    const int quad = warp & 3;                        // TMEM lane quadrant of this warp
    const int row = quad * 32 + lane;                 // query row inside the tile
    const uint32_t lane_base = static_cast<uint32_t>(quad * 32) << 16;
    const uint32_t tS = tmem_base + lane_base + COL_S + t * BN;
    const uint32_t tO = tmem_base + lane_base + COL_O + t * D;
    const uint32_t tP = tmem_base + lane_base + COL_P + t * (BN / 2);
    const float sc = 0.125f * 1.4426950408889634f;    // d^-0.5 * log2(e)
    const float2 sc2 = make_float2(sc, sc);
    uint32_t cnt = 0;                                 // running key-tile counter of this stream
    T* outp = reinterpret_cast<T*>(p.out);
    float* xch = reinterpret_cast<float*>(smem_gen + offX);

    for (int i = 0; i < n_my; ++i) {
      const SaItem it = sa_decode(p, blockIdx.x + i * gridDim.x);
      // key tiles of this stream: PAIR all, SPLIT [0, ja) / [ja, n_kv), SINGLE all / none
      const int j_begin = (it.kind == SPLIT && t == 1) ? p.ja : 0;
      const int j_end = it.kind == SPLIT ? (t == 0 ? p.ja : p.n_kv) : ((it.kind == SINGLE && t == 1) ? 0 : p.n_kv);
      if (j_begin >= j_end) continue;
      float m_run = 0.f, l_run = 0.f;
      for (int j = j_begin; j < j_end; ++j, ++cnt) {
        const bool first = j == j_begin;
        const int cols = sa_kv_cols(p, j);
        const int valid = p.N - j * BN;
        uint32_t s[BN];
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;
        mbar_wait(&s_ready[t], cnt & 1u);
        tc_fence_after();
        if (valid >= BN) {
          // full key tile: the row maximum of chunk c is computed while chunk c+1 is still in flight from TMEM
          tmem_ld32(tS, s);
          tmem_ld_wait32(s);
#pragma unroll
          for (int c = 0; c < BN; c += 32) {
            if (c + 32 < BN) tmem_ld32(tS + c + 32, s + c + 32);
#pragma unroll
            for (int k = 0; k < 32; k += 4) {
              mx0 = fmaxf(mx0, __uint_as_float(s[c + k]));
              mx1 = fmaxf(mx1, __uint_as_float(s[c + k + 1]));
              mx2 = fmaxf(mx2, __uint_as_float(s[c + k + 2]));
              mx3 = fmaxf(mx3, __uint_as_float(s[c + k + 3]));
            }
            if (c + 32 < BN) tmem_ld_wait32(s + c + 32);
          }
          tc_fence_before();
          mbar_arrive(&s_free[t]);
        } else {
          // last, partial key tile: mask the keys beyond N
#pragma unroll
          for (int c = 0; c < BN; c += 32)
            if (c < cols) tmem_ld32(tS + c, s + c);
          tmem_ld_wait();
          tc_fence_before();
          mbar_arrive(&s_free[t]);
#pragma unroll
          for (int c = 0; c < BN; ++c)
            if (c >= valid) s[c] = 0xff800000u;   // -inf
#pragma unroll
          for (int c = 0; c < BN; c += 32) {
            if (c < cols) {
#pragma unroll
              for (int k = 0; k < 32; k += 4) {
                mx0 = fmaxf(mx0, __uint_as_float(s[c + k]));
                mx1 = fmaxf(mx1, __uint_as_float(s[c + k + 1]));
                mx2 = fmaxf(mx2, __uint_as_float(s[c + k + 2]));
                mx3 = fmaxf(mx3, __uint_as_float(s[c + k + 3]));
              }
            }
          }
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        // O += P(j-1) V(j-1) was issued by this stream's own issuer as soon as P(j-1) was complete; P and O are ours
        // again once it has retired.  Normally that wait is taken as late as possible (in front of the first P store,
        // behind the first 32 exponentials); only a rescale needs O earlier.
        bool pv_done = first;
        if (first) {
          m_run = mx;
        } else {
          const float m_new = fmaxf(m_run, mx);
          const bool need = (m_new - m_run) * sc > RESCALE_LOG2;
          if (__any_sync(0xffffffffu, need)) {
            // rare: rescale O (TMEM round trip by the owning warp)
            mbar_wait(&o_done[t], (cnt - 1u) & 1u);
            tc_fence_after();
            pv_done = true;
            float alpha = 1.f;
            if (need) {
              alpha = exp2f((m_run - m_new) * sc);
              m_run = m_new;
              l_run *= alpha;
            }
#pragma unroll
            for (int c = 0; c < D; c += 16) {
              uint32_t o[16];
              tmem_ld16(tO + c, o);
              tmem_ld_wait16(o);
#pragma unroll
              for (int k = 0; k < 16; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * alpha);
              tmem_st16(tO + c, o);
            }
            tmem_st_wait();
          }
        }
        // ---- exp phase: P = exp2(s*sc - m*sc), row sum, pack to 16 bit, store to TMEM ----
        const float nmb = -m_run * sc;
        const float2 nmb2 = make_float2(nmb, nmb);
        float2 la = make_float2(0.f, 0.f), lb = make_float2(0.f, 0.f);
        auto exp_chunk = [&](int c, uint32_t (&pk)[16]) {
#pragma unroll
          for (int k = 0; k < 32; k += 4) {
            float2 x0 = __ffma2_rn(make_float2(__uint_as_float(s[c + k]), __uint_as_float(s[c + k + 1])), sc2, nmb2);
            float2 x1 =
                __ffma2_rn(make_float2(__uint_as_float(s[c + k + 2]), __uint_as_float(s[c + k + 3])), sc2, nmb2);
            if ((((c + k) >> 1) & POLY_MASK) == POLY_MASK) x0 = exp2_poly2(x0);
            else { x0.x = exp2f(x0.x); x0.y = exp2f(x0.y); }
            if (((((c + k) >> 1) + 1) & POLY_MASK) == POLY_MASK) x1 = exp2_poly2(x1);
            else { x1.x = exp2f(x1.x); x1.y = exp2f(x1.y); }
            la = __fadd2_rn(la, x0);
            lb = __fadd2_rn(lb, x1);
            pk[k >> 1] = H16<T>::pack2(x0.x, x0.y);
            pk[(k >> 1) + 1] = H16<T>::pack2(x1.x, x1.y);
          }
        };
        {
          uint32_t pk[16];
          exp_chunk(0, pk);                    // cols >= 32 always (N >= 1)
          if (!pv_done) {
            mbar_wait(&o_done[t], (cnt - 1u) & 1u);
            tc_fence_after();
          }
          tmem_st16(tP, pk);
        }
        if (cols == BN) {   // straight-line code for full key tiles: the scheduler hides the FMAs behind the MUFU
#pragma unroll
          for (int c = 32; c < BN; c += 32) {
            uint32_t pk[16];
            exp_chunk(c, pk);
            tmem_st16(tP + (c >> 1), pk);
          }
        } else {
#pragma unroll
          for (int c = 32; c < BN; c += 32) {
            if (c < cols) {
              uint32_t pk[16];
              exp_chunk(c, pk);
              tmem_st16(tP + (c >> 1), pk);
            }
          }
        }
        l_run += (la.x + la.y) + (lb.x + lb.y);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&p_ready[t]);
      }
      // ---- epilogue: O / l -> 16 bit -> global ----
      mbar_wait(&o_done[t], (cnt - 1u) & 1u);
      tc_fence_after();
      if (it.kind == SPLIT && t == 1) {
        // hand (O_1, m_1, l_1) to warpgroup 0 through shared memory ([value][row]: conflict-free)
        if (i > 0 && sa_kind(p, static_cast<int>(blockIdx.x) + (i - 1) * static_cast<int>(gridDim.x)) == SPLIT)
          named_bar_sync(BAR_XCH_EMPTY, 256);         // warpgroup 0 has consumed the previous hand-over
#pragma unroll
        for (int c = 0; c < D; c += 32) {
          uint32_t o[32];
          tmem_ld32(tO + c, o);
          tmem_ld_wait32(o);
#pragma unroll
          for (int k = 0; k < 32; ++k) xch[(c + k) * BM + row] = __uint_as_float(o[k]);
        }
        xch[D * BM + row] = m_run;
        xch[(D + 1) * BM + row] = l_run;
        tc_fence_before();   // the O reads above are ordered before this thread's next p_ready arrive
        named_bar_arrive(BAR_XCH_FULL, 256);
      } else {
        float fa = 1.f, fb = 0.f;
        if (it.kind == SPLIT) {
          // merge the two halves of the key range:  O = (O_0 2^(m_0-m) + O_1 2^(m_1-m)) / (l_0 2^(m_0-m) + l_1 2^(m_1-m))
          named_bar_sync(BAR_XCH_FULL, 256);
          const float mb = xch[D * BM + row], lbv = xch[(D + 1) * BM + row];
          const float m = fmaxf(m_run, mb);
          fa = exp2f((m_run - m) * sc);
          fb = exp2f((mb - m) * sc);
          const float inv = 1.f / (l_run * fa + lbv * fb);
          fa *= inv;
          fb *= inv;
        } else {
          fa = 1.f / l_run;
        }
        const int q = it.q0 + (it.kind == PAIR ? t * BM : 0) + row;
        T* orow = outp + (static_cast<long long>(it.frame) * p.N + q) * (static_cast<long long>(p.heads) * D) +
                  it.head * D;
#pragma unroll
        for (int c = 0; c < D; c += 32) {
          uint32_t o[32];
          tmem_ld32(tO + c, o);
          tmem_ld_wait32(o);
          float v[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(o[k]) * fa;
          if (it.kind == SPLIT) {
#pragma unroll
            for (int k = 0; k < 32; ++k) v[k] = fmaf(xch[(c + k) * BM + row], fb, v[k]);
          }
          if (q < p.N) {
#pragma unroll
            for (int k = 0; k < 32; k += 8) {
              uint4 u;
              u.x = H16<T>::pack2(v[k], v[k + 1]);
              u.y = H16<T>::pack2(v[k + 2], v[k + 3]);
              u.z = H16<T>::pack2(v[k + 4], v[k + 5]);
              u.w = H16<T>::pack2(v[k + 6], v[k + 7]);
              *reinterpret_cast<uint4*>(orow + c + k) = u;
            }
          }
        }
        tc_fence_before();   // the O reads above are ordered before this thread's next p_ready arrive
        if (it.kind == SPLIT && i + 1 < n_my) named_bar_arrive(BAR_XCH_EMPTY, 256);   // (split items are the tail of the list)
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace vda

using namespace vda;

extern "C" int vda_attention_spatial(const void* qkv, void* out, int frames, int N, int heads, int dtype,
                                     void* stream) {
  VDA_CHECK(frames > 0 && N > 0 && heads > 0, "bad attention shape");
  VDA_CHECK(dtype == VDA_BF16 || dtype == VDA_FP16, "bad dtype %d", dtype);
  VDA_CHECK((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
            "qkv/out must be 16-byte aligned");
  // qkv is [frames, N, 3, heads, 64]: a 4-D tensor (d, which*heads + head, token, frame); token rows beyond N are
  // zero-filled by TMA instead of running into the next frame
  CUtensorMap tm;
  const cuuint64_t row_bytes = static_cast<cuuint64_t>(3) * heads * sa::D * 2;
  cuuint64_t dims[4] = {sa::D, static_cast<cuuint64_t>(3 * heads), static_cast<cuuint64_t>(N),
                        static_cast<cuuint64_t>(frames)};
  cuuint64_t strides[3] = {sa::D * 2, row_bytes, row_bytes * N};
  cuuint32_t box[4] = {sa::D, 1, sa::BM, 1};
  if (make_tensor_map(&tm, dtype, qkv, 4, dims, strides, box)) return 1;

  SaParams p;
  p.N = N; p.heads = heads; p.frames = frames;
  p.n_qt = (N + sa::BM - 1) / sa::BM;
  p.n_pairs = p.n_qt / 2;
  p.n_items = frames * heads * p.n_pairs + ((p.n_qt & 1) ? frames * heads : 0);
  p.n_kv = (N + sa::BN - 1) / sa::BN;
  p.ja = (p.n_kv + 1) / 2;
  p.split = p.n_kv >= 2 ? 1 : 0;
  p.out = out;
  const int grid = p.n_items < sm_count() ? p.n_items : sm_count();
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == VDA_BF16) {
    auto k = spatial_attention_tc_kernel<__nv_bfloat16>;
    VDA_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(k), sa::SMEM_BYTES));
    k<<<grid, sa::THREADS, sa::SMEM_BYTES, st>>>(tm, p);
  } else {
    auto k = spatial_attention_tc_kernel<__half>;
    VDA_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(k), sa::SMEM_BYTES));
    k<<<grid, sa::THREADS, sa::SMEM_BYTES, st>>>(tm, p);
  }
  VDA_CUDA(cudaGetLastError());
  return 0;
}
