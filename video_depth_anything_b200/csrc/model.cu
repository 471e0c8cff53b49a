// Handle-level C ABI (SURVEY.md §8(b)): the whole forward of VideoDepthAnything (video_depth_anything/video_depth.py:89-164)
// behind   vda_create -> vda_set_weight* -> vda_finalize_weights -> vda_workspace_bytes -> vda_forward   so that a host that
// is not Python does not have to re-implement the engine's launch schedule; vda_stream_step is the streaming step of a
// stream group (engine.py Engine.stream_group_step) on the same schedule.  This file is that schedule (the same sequence
// of libvda operator calls as video_depth_anything_b200/engine.py: encode / head / motion module / fusion blocks) plus the
// weight packing (reference state-dict tensors -> kernel layouts), written against the operator-level entry points of
// include/vda.h.  tests/test_cmodel_gpu.py requires its output to be BIT-identical to the Python engine's.
//
// Memory: vda_forward does not allocate.  The caller passes one workspace (vda_workspace_bytes, a dry run of the schedule
// over a bump allocator); nothing synchronises, so the call can be captured in a CUDA graph.  The only lazily created device
// state is the bicubic-resampled position embedding of a new token grid (cached in the model, created on first use with
// cudaMalloc: do the first call of a new geometry outside a capture).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/vda.h"
#include "common.cuh"

namespace vda {

struct HostTensor {
  std::vector<float> v;
  std::vector<int64_t> shape;
  int64_t dim(int i) const { return shape[static_cast<size_t>(i)]; }
};

constexpr int KPAD_PATCH = 592;   // 3*14*14 = 588 padded to a 16-byte row pitch (engine.py)

}  // namespace vda

struct vda_model {
  std::string enc;
  int D = 0, depth = 0, heads = 0, taps[4] = {0, 0, 0, 0};
  int F = 0, oc[4] = {0, 0, 0, 0}, num_frames = 32;
  int dtype = VDA_BF16, hdtype = VDA_FP16, device = 0;
  bool ln_fold = true, finalized = false;
  int c_l1 = 0, c_l2 = 0, c_oc1 = 0, mm_c[4] = {0, 0, 0, 0}, mm_half[4] = {0, 0, 0, 0};
  float oc3_b = 0.f;
  std::map<std::string, vda::HostTensor> sd;          // reference state dict (fp32, host), until finalize
  std::map<std::string, void*> w;                     // packed device weights
  std::vector<void*> owned;                           // everything cudaMalloc'ed by the model
  std::map<std::pair<int, int>, float*> pos_cache;    // bicubic pos-embed per token grid
  int pos_S = 0;
};

namespace vda {

static int pad_to(int n, int m) { return (n + m - 1) / m * m; }

static uint16_t to_h16(float f, int dtype) {
  if (dtype == VDA_BF16) {
    const __nv_bfloat16 h = __float2bfloat16_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
  }
  const __half h = __float2half_rn(f);
  uint16_t u;
  memcpy(&u, &h, 2);
  return u;
}

// ---- device uploads -------------------------------------------------------------------------
static int dev_alloc(vda_model* m, size_t bytes, void** out) {
  VDA_CUDA(cudaMalloc(out, bytes ? bytes : 16));
  m->owned.push_back(*out);
  return 0;
}
static int up_f32(vda_model* m, const std::string& key, const float* src, size_t n) {
  void* d;
  if (dev_alloc(m, n * 4, &d)) return 1;
  VDA_CUDA(cudaMemcpy(d, src, n * 4, cudaMemcpyHostToDevice));
  m->w[key] = d;
  return 0;
}
static int up_h16(vda_model* m, const std::string& key, const std::vector<float>& src, int dtype) {
  std::vector<uint16_t> h(src.size());
  for (size_t i = 0; i < src.size(); ++i) h[i] = to_h16(src[i], dtype);
  void* d;
  if (dev_alloc(m, h.size() * 2, &d)) return 1;
  VDA_CUDA(cudaMemcpy(d, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  m->w[key] = d;
  return 0;
}

// ---- weight packing (engine.py pack_conv3x3 / pack_convt / pack_geglu) ------------------------
// [Co,Ci,3,3] -> [co_pad, 9*ci_pad], K index = (ky*3+kx)*ci_pad + ci
static std::vector<float> pack_conv3x3(const HostTensor& t, int ci_pad, int co_pad) {
  const int co = static_cast<int>(t.dim(0)), ci = static_cast<int>(t.dim(1));
  std::vector<float> out(static_cast<size_t>(co_pad) * 9 * ci_pad, 0.f);
  for (int o = 0; o < co; ++o)
    for (int c = 0; c < ci; ++c)
      for (int k = 0; k < 9; ++k)
        out[(static_cast<size_t>(o) * 9 + k) * ci_pad + c] = t.v[(static_cast<size_t>(o) * ci + c) * 9 + k];
  return out;
}
// ConvTranspose2d weight [Ci,Co,S,S] (kernel == stride) -> [(ky*S+kx)*co_pad + co, Ci]; bias -> [co_pad]
static void pack_convt(const HostTensor& t, const HostTensor& b, int co_pad, std::vector<float>& w, std::vector<float>& bp) {
  const int ci = static_cast<int>(t.dim(0)), co = static_cast<int>(t.dim(1)), s = static_cast<int>(t.dim(2));
  w.assign(static_cast<size_t>(s) * s * co_pad * ci, 0.f);
  for (int c = 0; c < ci; ++c)
    for (int o = 0; o < co; ++o)
      for (int k = 0; k < s * s; ++k)
        w[(static_cast<size_t>(k) * co_pad + o) * ci + c] = t.v[(static_cast<size_t>(c) * co + o) * s * s + k];
  bp.assign(static_cast<size_t>(co_pad), 0.f);
  for (int o = 0; o < co; ++o) bp[static_cast<size_t>(o)] = b.v[static_cast<size_t>(o)];
}
// GEGLU proj weight [2*inner, C] (rows: value | gate) -> row blocks [value(half) | gate(half)]
static void pack_geglu(const HostTensor& t, const HostTensor& b, int half, std::vector<float>& w, std::vector<float>& bp) {
  const int inner = static_cast<int>(t.dim(0)) / 2, C = static_cast<int>(t.dim(1));
  w.resize(t.v.size());
  bp.resize(b.v.size());
  for (int blk = 0; blk < inner / half; ++blk)
    for (int j = 0; j < 2 * half; ++j) {
      const int src = j < half ? blk * half + j : inner + blk * half + (j - half);
      const int dst = blk * 2 * half + j;
      memcpy(&w[static_cast<size_t>(dst) * C], &t.v[static_cast<size_t>(src) * C], static_cast<size_t>(C) * 4);
      bp[static_cast<size_t>(dst)] = b.v[static_cast<size_t>(src)];
    }
}

// ---- bump allocator over the caller's workspace ---------------------------------------------
struct Arena {
  char* base;
  size_t off, cap;
  void* get(size_t bytes) {
    const size_t a = (off + 1023) & ~static_cast<size_t>(1023);   // TMA boxes want 16 B, swizzled staging 1 KB: be generous
    off = a + bytes;
    return base ? base + a : reinterpret_cast<void*>(a + 4096);   // dry run: fake, never dereferenced
  }
};

struct Ctx {
  const vda_model* m;
  Arena a;
  void* st;
  bool dry;
  int rc;
  const void* W(const std::string& k) const {
    auto it = m->w.find(k);
    return it == m->w.end() ? nullptr : it->second;
  }
  const float* Wf(const std::string& k) const { return static_cast<const float*>(W(k)); }
};
#define RUN(c, expr)                  \
  do {                                \
    if (!(c).dry && (c).rc == 0) {    \
      const int _r = (expr);          \
      if (_r) (c).rc = _r;            \
    }                                 \
  } while (0)

struct G {   // options of one GEMM launch (mirrors ops.gemm)
  const float* bias = nullptr;
  const float* gamma = nullptr;
  int act = VDA_ACT_NONE;
  const void* res1 = nullptr;
  int64_t ldr1 = 0;
  int res1_f32 = 0;
  const void* res2 = nullptr;
  void* out_relu = nullptr;
  int row_group = 0, epilogue = VDA_EPI_LINEAR, geglu_half = 0;
  int convt_s = 0, convt_co = 0, in_h = 0, in_w = 0;
  int conv_n = 0, conv_h = 0, conv_w = 0, conv_c = 0;   // implicit 3x3 conv over NHWC [n,h,w,c]
  void* out16 = nullptr;
  float* stats_out = nullptr;
  const float* stats_in = nullptr;
  const float* ln_c1 = nullptr;
  int stat_parts = 0;
  int dtype = VDA_BF16;
  int out_f32 = 0;
};

// out[M,N] = epilogue(A[M,K] Wt[N,K]^T)
static void gemm(Ctx& c, const void* A, int M, int K, const void* Wt, int N, void* out, int64_t ldo, const G& o) {
  vda_gemm_params p;
  memset(&p, 0, sizeof(p));
  p.N = N;
  p.K = K;
  p.dtype = o.dtype;
  p.epilogue = o.epilogue;
  if (o.conv_n) {
    p.a_mode = VDA_A_CONV3;
    p.n_img = o.conv_n; p.H = o.conv_h; p.W = o.conv_w; p.C = o.conv_c;
    p.M = o.conv_n * o.conv_h * o.conv_w;
    p.lda = o.conv_c;
  } else {
    p.a_mode = VDA_A_PLAIN;
    p.M = M;
    p.lda = K;
  }
  p.A = A;
  p.Wt = Wt;
  p.bias = o.bias; p.gamma = o.gamma; p.act = o.act;
  p.res1 = o.res1; p.ldr1 = o.ldr1; p.res1_f32 = o.res1_f32; p.res2 = o.res2;
  p.out = out; p.ldo = ldo; p.out_f32 = o.out_f32; p.out_relu = o.out_relu;
  p.row_group = o.row_group; p.geglu_half = o.geglu_half;
  p.convt_s = o.convt_s; p.convt_co = o.convt_co; p.in_h = o.in_h; p.in_w = o.in_w;
  p.out16 = o.out16; p.row_stats_out = o.stats_out; p.row_stats_in = o.stats_in; p.ln_c1 = o.ln_c1;
  p.stat_parts = o.stat_parts;
  if (o.stats_in) { p.stat_cols = K / o.stat_parts; p.ln_eps = 1e-6f; }
  RUN(c, vda_gemm(&p, c.st));
}

static const float* const_vec(vda_model* m, float value, int n) {   // cached constant vectors (zero bias / unit LayerScale)
  const std::string key = "const." + std::to_string(value) + "." + std::to_string(n);
  auto it = m->w.find(key);
  if (it != m->w.end()) return static_cast<const float*>(it->second);
  std::vector<float> v(static_cast<size_t>(n), value);
  if (up_f32(m, key, v.data(), v.size())) return nullptr;
  return static_cast<const float*>(m->w[key]);
}

// ---- encoder (engine.py Engine.encode; dinov2.py:297-321) ------------------------------------
static void encode(Ctx& c, const float* x, int BT, int H, int W, const float* pos, void* taps[4]) {
  const vda_model* m = c.m;
  const int D = m->D, hp = H / 14, wp = W / 14, P = hp * wp, N = P + 1, M = BT * N;
  const int dt = m->dtype;
  void* a = c.a.get(static_cast<size_t>(BT) * P * KPAD_PATCH * 2);
  RUN(c, vda_patch_im2col(x, a, BT, H, W, KPAD_PATCH, dt, c.st));
  float* tok = static_cast<float*>(c.a.get(static_cast<size_t>(M) * D * 4));
  {
    G o; o.dtype = dt; o.bias = c.Wf("pe.b"); o.res1 = pos; o.ldr1 = D; o.res1_f32 = 1; o.row_group = P; o.out_f32 = 1;
    gemm(c, a, BT * P, KPAD_PATCH, c.W("pe.w"), D, tok, D, o);
  }
  RUN(c, vda_write_cls(tok, c.Wf("cls"), pos, BT, N, D, c.st));
  void* ln = c.a.get(static_cast<size_t>(M) * D * 2);
  void* qkv = c.a.get(static_cast<size_t>(M) * 3 * D * 2);
  void* att = c.a.get(static_cast<size_t>(M) * D * 2);
  void* hid = c.a.get(static_cast<size_t>(M) * 4 * D * 2);
  int parts = 0, cols = 0;
  const bool fold = m->ln_fold && vda_gemm_rowstat_layout(M, D, &parts, &cols) == 0;
  float* stats = nullptr;
  if (fold) {
    stats = static_cast<float*>(c.a.get(static_cast<size_t>(M) * parts * 2 * 4));
    RUN(c, vda_rowstats_cast(tok, ln, stats, M, D, parts, cols, dt, c.st));
  }
  int ntap = 0;
  for (int i = 0; i < m->depth; ++i) {
    const std::string b = "b" + std::to_string(i) + ".";
    if (fold) {
      { G o; o.dtype = dt; o.bias = c.Wf(b + "qkv.c2"); o.stats_in = stats; o.ln_c1 = c.Wf(b + "qkv.c1"); o.stat_parts = parts;
        gemm(c, ln, M, D, c.W(b + "qkv.wf"), 3 * D, qkv, 3 * D, o); }
      RUN(c, vda_attention_spatial(qkv, att, BT, N, m->heads, dt, c.st));
      { G o; o.dtype = dt; o.bias = c.Wf(b + "proj.b"); o.gamma = c.Wf(b + "ls1"); o.res1 = tok; o.ldr1 = D; o.res1_f32 = 1;
        o.out_f32 = 1; o.out16 = ln; o.stats_out = stats; o.stat_parts = parts;
        gemm(c, att, M, D, c.W(b + "proj.w"), D, tok, D, o); }
      { G o; o.dtype = dt; o.bias = c.Wf(b + "fc1.c2"); o.act = VDA_ACT_GELU; o.stats_in = stats; o.ln_c1 = c.Wf(b + "fc1.c1");
        o.stat_parts = parts;
        gemm(c, ln, M, D, c.W(b + "fc1.wf"), 4 * D, hid, 4 * D, o); }
      { const bool last = i == m->depth - 1;
        G o; o.dtype = dt; o.bias = c.Wf(b + "fc2.b"); o.gamma = c.Wf(b + "ls2"); o.res1 = tok; o.ldr1 = D; o.res1_f32 = 1;
        o.out_f32 = 1; o.out16 = last ? nullptr : ln; o.stats_out = last ? nullptr : stats; o.stat_parts = last ? 0 : parts;
        gemm(c, hid, M, 4 * D, c.W(b + "fc2.w"), D, tok, D, o); }
    } else {
      RUN(c, vda_layernorm(tok, 1, ln, c.Wf(b + "norm1.w"), c.Wf(b + "norm1.b"), 1e-6f, M, D, dt, 0, nullptr, 0, 0, c.st));
      { G o; o.dtype = dt; o.bias = c.Wf(b + "qkv.b"); gemm(c, ln, M, D, c.W(b + "qkv.w"), 3 * D, qkv, 3 * D, o); }
      RUN(c, vda_attention_spatial(qkv, att, BT, N, m->heads, dt, c.st));
      { G o; o.dtype = dt; o.bias = c.Wf(b + "proj.b"); o.gamma = c.Wf(b + "ls1"); o.res1 = tok; o.ldr1 = D; o.res1_f32 = 1; o.out_f32 = 1;
        gemm(c, att, M, D, c.W(b + "proj.w"), D, tok, D, o); }
      RUN(c, vda_layernorm(tok, 1, ln, c.Wf(b + "norm2.w"), c.Wf(b + "norm2.b"), 1e-6f, M, D, dt, 0, nullptr, 0, 0, c.st));
      { G o; o.dtype = dt; o.bias = c.Wf(b + "fc1.b"); o.act = VDA_ACT_GELU; gemm(c, ln, M, D, c.W(b + "fc1.w"), 4 * D, hid, 4 * D, o); }
      { G o; o.dtype = dt; o.bias = c.Wf(b + "fc2.b"); o.gamma = c.Wf(b + "ls2"); o.res1 = tok; o.ldr1 = D; o.res1_f32 = 1; o.out_f32 = 1;
        gemm(c, hid, M, 4 * D, c.W(b + "fc2.w"), D, tok, D, o); }
    }
    if (ntap < 4 && i == m->taps[ntap]) {     // dinov2.py:309-312: final norm, cls row dropped, head operand type
      void* t = c.a.get(static_cast<size_t>(BT) * P * D * 2);
      RUN(c, vda_layernorm(tok, 1, t, c.Wf("norm.w"), c.Wf("norm.b"), 1e-6f, M, D, m->hdtype, N, nullptr, 0, 0, c.st));
      taps[ntap++] = t;
    }
  }
}

// ---- head pieces (engine.py _conv3 / _rcu / _fusion / _motion / head) ------------------------
struct Map { void* p; void* relu; };   // NHWC h16 activation (+ its ReLU'd copy when a following RCU wants it)

static void* conv3(Ctx& c, const void* x, const std::string& key, int n, int H, int W, int ci, int co, G o, void* out = nullptr) {
  if (!out) out = c.a.get(static_cast<size_t>(n) * H * W * co * 2);
  o.dtype = c.m->hdtype;
  o.bias = c.Wf(key + ".b");
  o.conv_n = n; o.conv_h = H; o.conv_w = W; o.conv_c = ci;
  gemm(c, x, 0, 9 * ci, c.W(key + ".w"), co, out, co, o);
  return out;
}

// ResidualConvUnit (util/blocks.py:68-91): conv2(relu(conv1(relu(x)))) + x [+ extra]
static Map rcu(Ctx& c, int r, int u, const Map& x, int n, int H, int W, const void* extra, bool want_relu) {
  const int F = c.m->F;
  const std::string k = "rf" + std::to_string(r) + ".u" + std::to_string(u);
  G o1; o1.act = VDA_ACT_RELU;
  void* t = conv3(c, x.relu, k + ".c1", n, H, W, F, F, o1);
  Map out;
  out.p = c.a.get(static_cast<size_t>(n) * H * W * F * 2);
  out.relu = want_relu ? c.a.get(static_cast<size_t>(n) * H * W * F * 2) : nullptr;
  G o2; o2.res1 = x.p; o2.ldr1 = F; o2.res1_f32 = 0; o2.res2 = extra; o2.out_relu = out.relu;
  conv3(c, t, k + ".c2", n, H, W, F, F, o2, out.p);
  return out;
}

// FeatureFusionBlock (util/blocks.py:135-162); the 1x1 out_conv before the bilinear upsample (engine.py _fusion)
static void* fusion(Ctx& c, int r, const void* x0, const Map& skip, int n, int H, int W, int oh, int ow) {
  const int F = c.m->F, hdt = c.m->hdtype;
  Map cur = skip;
  if (x0) cur = rcu(c, r, 1, skip, n, H, W, x0, true);
  const Map u = rcu(c, r, 2, cur, n, H, W, nullptr, false);
  void* o = c.a.get(static_cast<size_t>(n) * H * W * F * 2);
  const std::string k = "rf" + std::to_string(r) + ".out";
  { G g; g.dtype = hdt; g.bias = c.Wf(k + ".b"); gemm(c, u.p, n * H * W, F, c.W(k + ".w"), F, o, F, g); }
  void* up = c.a.get(static_cast<size_t>(n) * oh * ow * F * 2);
  RUN(c, vda_bilinear_nhwc(o, up, n, H, W, oh, ow, F, hdt, c.st));
  return up;
}

// One streamed frame per batch row (T = 1) whose temporal attentions read the rows' pool entries (engine.py
// Engine.stream_group_step): the pool block of attention block a of motion module m starts at off[2 * m + a].
struct StreamStep {
  char* pool;
  size_t off[8];
  const int32_t* rows;   // [B]
  const int32_t* ctx;    // [B, stride]
  int S, slots, stride;
  bool causal;
};

// TemporalModule (motion_module.py:60-65, 102-126, 164-177).  x h16 [B*T*hw, C], rows (b, f, pos).
// `s`: the streaming branch of engine.py Engine._motion (LayerNorm without the positional encoding, whose share enters
// through the `pet` tables inside the step kernels)
static void* motion(Ctx& c, vda_model* mm, int mi, const void* x, int B, int T, int hw, const StreamStep* s) {
  const vda_model* m = c.m;
  const int C = m->mm_c[mi], M = B * T * hw, hdt = m->hdtype;
  const std::string p = "mm" + std::to_string(mi) + ".";
  void* gn = c.a.get(static_cast<size_t>(M) * C * 2);
  float* gstats = static_cast<float*>(c.a.get(static_cast<size_t>(592 + 2 * B * T) * 32 * 2 * 4));   // VDA_GN_STATS_FLOATS
  RUN(c, vda_groupnorm(x, gn, c.Wf(p + "gn.w"), c.Wf(p + "gn.b"), 1e-6f, B * T, hw, C, 32, gstats, hdt, c.st));
  float* h = static_cast<float*>(c.a.get(static_cast<size_t>(M) * C * 4));
  { G g; g.dtype = hdt; g.bias = c.Wf(p + "in.b"); g.out_f32 = 1; gemm(c, gn, M, C, c.W(p + "in.w"), C, h, C, g); }
  void* nrm = gn;                                          // reused as the LayerNorm output
  void* qkv = c.a.get(static_cast<size_t>(M) * 3 * C * 2);
  void* o = c.a.get(static_cast<size_t>(M) * C * 2);
  const float* zero3c = const_vec(mm, 0.f, 3 * C);
  const float* onec = const_vec(mm, 1.f, C);
  for (int a = 0; a < 2; ++a) {
    const std::string ab = p + "a" + std::to_string(a) + ".";
    RUN(c, vda_layernorm(h, 1, nrm, c.Wf(ab + "ln.w"), c.Wf(ab + "ln.b"), 1e-5f, M, C, hdt, 0, s ? nullptr : c.Wf(ab + "pe"),
                         s ? 0 : hw, s ? 0 : T, c.st));
    { G g; g.dtype = hdt; g.bias = zero3c; gemm(c, nrm, M, C, c.W(ab + "qkv.w"), 3 * C, qkv, 3 * C, g); }
    if (!s) {
      for (int b = 0; b < B; ++b) {
        const size_t off = static_cast<size_t>(b) * T * hw;
        RUN(c, vda_attention_temporal(static_cast<const char*>(qkv) + off * 3 * C * 2, static_cast<char*>(o) + off * C * 2, T, hw, C,
                                      8, hdt, c.st));
      }
    } else {
      void* blk = s->pool + s->off[2 * mi + a];
      if (s->causal) {
        RUN(c, vda_attention_temporal_step_causal(qkv, blk, c.Wf(ab + "pet"), s->rows, s->ctx, o, B, s->S, s->stride, hw, C, 8,
                                                  s->slots, hdt, c.st));
        RUN(c, vda_stream_cache_store(qkv, blk, s->rows, s->ctx, B, s->S, s->stride, hw, C, s->slots, hdt, c.st));
      } else {
        RUN(c, vda_attention_temporal_step_batched(qkv, blk, c.Wf(ab + "pet"), s->rows, s->ctx, o, B, s->S, s->stride, hw, C, 8,
                                                   s->slots, hdt, c.st));
      }
    }
    { G g; g.dtype = hdt; g.bias = c.Wf(ab + "o.b"); g.gamma = onec; g.res1 = h; g.ldr1 = C; g.res1_f32 = 1; g.out_f32 = 1;
      gemm(c, o, M, C, c.W(ab + "o.w"), C, h, C, g); }
  }
  RUN(c, vda_layernorm(h, 1, nrm, c.Wf(p + "ffn.w"), c.Wf(p + "ffn.b"), 1e-5f, M, C, hdt, 0, nullptr, 0, 0, c.st));
  void* gg = c.a.get(static_cast<size_t>(M) * 4 * C * 2);
  { G g; g.dtype = hdt; g.bias = c.Wf(p + "ff0.b"); g.epilogue = VDA_EPI_GEGLU; g.geglu_half = m->mm_half[mi];
    gemm(c, nrm, M, C, c.W(p + "ff0.w"), 8 * C, gg, 4 * C, g); }
  void* h16 = o;
  { G g; g.dtype = hdt; g.bias = c.Wf(p + "ff2.b"); g.res1 = h; g.ldr1 = C; g.res1_f32 = 1; gemm(c, gg, M, 4 * C, c.W(p + "ff2.w"), C, h16, C, g); }
  void* out = c.a.get(static_cast<size_t>(M) * C * 2);
  { G g; g.dtype = hdt; g.bias = c.Wf(p + "out.b"); g.res1 = x; g.ldr1 = C; g.res1_f32 = 0; gemm(c, h16, M, C, c.W(p + "out.w"), C, out, C, g); }
  return out;
}

// DPTHeadTemporal.forward (dpt_temporal.py:53-114) -> fp32 [B*T, 14hp, 14wp]; `s`: see motion
static void head(Ctx& c, vda_model* mm, void* taps[4], int B, int T, int hp, int wp, float* depth, const StreamStep* s) {
  const vda_model* m = c.m;
  const int F = m->F, D = m->D, BT = B * T, P = hp * wp, hdt = m->hdtype;
  const int* oc = m->oc;
  void* pr[4];
  for (int i = 0; i < 4; ++i) {
    pr[i] = c.a.get(static_cast<size_t>(BT) * P * oc[i] * 2);
    const std::string k = "proj" + std::to_string(i);
    G g; g.dtype = hdt; g.bias = c.Wf(k + ".b");
    gemm(c, taps[i], BT * P, D, c.W(k + ".w"), oc[i], pr[i], oc[i], g);
  }
  const int h1 = 4 * hp, w1 = 4 * wp, h2 = 2 * hp, w2 = 2 * wp, h4 = (hp - 1) / 2 + 1, w4 = (wp - 1) / 2 + 1;
  void* l1 = c.a.get(static_cast<size_t>(BT) * h1 * w1 * m->c_l1 * 2);
  { G g; g.dtype = hdt; g.bias = c.Wf("rs0.b"); g.epilogue = VDA_EPI_CONVT; g.convt_s = 4; g.convt_co = m->c_l1; g.in_h = hp; g.in_w = wp;
    gemm(c, pr[0], BT * P, oc[0], c.W("rs0.w"), 16 * m->c_l1, l1, m->c_l1, g); }
  void* l2 = c.a.get(static_cast<size_t>(BT) * h2 * w2 * m->c_l2 * 2);
  { G g; g.dtype = hdt; g.bias = c.Wf("rs1.b"); g.epilogue = VDA_EPI_CONVT; g.convt_s = 2; g.convt_co = m->c_l2; g.in_h = hp; g.in_w = wp;
    gemm(c, pr[1], BT * P, oc[1], c.W("rs1.w"), 4 * m->c_l2, l2, m->c_l2, g); }
  void* l3 = pr[2];
  void* col = c.a.get(static_cast<size_t>(BT) * h4 * w4 * 9 * oc[3] * 2);
  RUN(c, vda_im2col3x3_s2(pr[3], col, BT, hp, wp, oc[3], hdt, c.st));
  void* l4 = c.a.get(static_cast<size_t>(BT) * h4 * w4 * oc[3] * 2);
  { G g; g.dtype = hdt; g.bias = c.Wf("rs3.b"); gemm(c, col, BT * h4 * w4, 9 * oc[3], c.W("rs3.w"), oc[3], l4, oc[3], g); }
  l3 = motion(c, mm, 0, l3, B, T, P, s);
  l4 = motion(c, mm, 1, l4, B, T, h4 * w4, s);
  auto rn = [&](int i, const void* x, int H, int W, int ci) {   // layer{i}_rn (+ relu'd copy)
    Map o;
    o.p = c.a.get(static_cast<size_t>(BT) * H * W * F * 2);
    o.relu = c.a.get(static_cast<size_t>(BT) * H * W * F * 2);
    G g; g.dtype = hdt; g.out_relu = o.relu; g.conv_n = BT; g.conv_h = H; g.conv_w = W; g.conv_c = ci;
    gemm(c, x, 0, 9 * ci, c.W("rn" + std::to_string(i) + ".w"), F, o.p, F, g);
    return o;
  };
  const Map l1r = rn(1, l1, h1, w1, m->c_l1), l2r = rn(2, l2, h2, w2, m->c_l2), l3r = rn(3, l3, hp, wp, oc[2]),
            l4r = rn(4, l4, h4, w4, oc[3]);
  void* p4 = fusion(c, 4, nullptr, l4r, BT, h4, w4, hp, wp);
  p4 = motion(c, mm, 2, p4, B, T, P, s);
  void* p3 = fusion(c, 3, p4, l3r, BT, hp, wp, h2, w2);
  p3 = motion(c, mm, 3, p3, B, T, h2 * w2, s);
  void* p2 = fusion(c, 2, p3, l2r, BT, h2, w2, h1, w1);
  void* p1 = fusion(c, 1, p2, l1r, BT, h1, w1, 2 * h1, 2 * w1);
  const int H8 = 2 * h1, W8 = 2 * w1;
  G g1;
  void* o1 = conv3(c, p1, "oc1", BT, H8, W8, F, m->c_oc1, g1);
  RUN(c, vda_tail_fused(o1, c.W("oc2.w"), c.Wf("oc2.b"), c.Wf("oc3.w"), m->oc3_b, depth, BT, H8, W8, 14 * hp, 14 * wp, m->c_oc1, hdt,
                        c.st));
}

static int pos_for(vda_model* m, int hp, int wp, void* st, const float** out) {
  const auto key = std::make_pair(hp, wp);
  auto it = m->pos_cache.find(key);
  if (it != m->pos_cache.end()) { *out = it->second; return 0; }
  const float* pos = static_cast<const float*>(m->w["pos"]);
  if (hp == m->pos_S && wp == m->pos_S) { *out = pos; return 0; }
  void* d;
  if (dev_alloc(m, static_cast<size_t>(1 + hp * wp) * m->D * 4, &d)) return 1;
  if (vda_pos_embed_bicubic(pos, static_cast<float*>(d), m->pos_S, hp, wp, m->D, st)) return 1;
  m->pos_cache[key] = static_cast<float*>(d);
  *out = static_cast<float*>(d);
  return 0;
}

static int run_forward(vda_model* m, const float* x, int B, int T, int H, int W, float* depth, void* ws, size_t ws_bytes, void* st,
                       bool dry, size_t* need) {
  Ctx c;
  c.m = m;
  c.a.base = static_cast<char*>(ws);
  c.a.off = 0;
  c.a.cap = ws_bytes;
  c.st = st;
  c.dry = dry;
  c.rc = 0;
  const float* pos = nullptr;
  if (!dry && pos_for(m, H / 14, W / 14, st, &pos)) return 1;
  for (int mi = 0; mi < 4; ++mi) {             // constants the motion modules use: created outside the launch sequence
    if (!const_vec(m, 0.f, 3 * m->mm_c[mi]) || !const_vec(m, 1.f, m->mm_c[mi])) return 1;
  }
  void* taps[4] = {nullptr, nullptr, nullptr, nullptr};
  encode(c, x, B * T, H, W, pos, taps);
  head(c, m, taps, B, T, H / 14, W / 14, depth, nullptr);
  if (need) *need = c.a.off + 1024;
  return c.rc;
}

// Byte offsets of the 8 blocks of a stream pool (engine.py Engine.stream_pool order: block 2 * m + a is attention block a
// of motion module m, h16 [S, slots, hw_m, 2 C_m]); returns the total.  Every block is a multiple of 256 bytes (C_m is a
// multiple of 64), so each starts 256-byte aligned without padding.
static size_t pool_layout(const vda_model* m, int S, int hp, int wp, size_t off[8]) {
  const int hws[4] = {hp * wp, ((hp - 1) / 2 + 1) * ((wp - 1) / 2 + 1), hp * wp, 4 * hp * wp};
  size_t total = 0;
  for (int b = 0; b < 8; ++b) {
    off[b] = total;
    total += static_cast<size_t>(S) * m->num_frames * hws[b / 2] * 2 * m->mm_c[b / 2] * 2;
  }
  return total;
}

// engine.py Engine.stream_group_step: ragged preprocessing to (nh, nw), encoder and head on the B frames at T = 1 with
// every temporal attention against the rows' pool entries, ragged bilinear resize to each row's frame size.  `ingest` is
// the ragged preprocessing entry point of the frames' descriptor type: vda_preprocess_frames_ragged (RGB) or
// vda_preprocess_frames_planes (YUV 4:2:0); nothing else depends on the pixel format.
template <class Desc>
static int run_step(vda_model* m, int (*ingest)(const Desc*, int, int, int, float*, void*), const Desc* frames,
                    const vda_out_desc* outs, const int32_t* table, int B, bool causal, void* pool, int S, int nh, int nw,
                    void* ws, size_t ws_bytes, void* st, bool dry, size_t* need) {
  Ctx c;
  c.m = m;
  c.a.base = static_cast<char*>(ws);
  c.a.off = 0;
  c.a.cap = ws_bytes;
  c.st = st;
  c.dry = dry;
  c.rc = 0;
  const int hp = nh / 14, wp = nw / 14;
  const float* pos = nullptr;
  if (!dry && pos_for(m, hp, wp, st, &pos)) return 1;
  for (int mi = 0; mi < 4; ++mi) {
    if (!const_vec(m, 0.f, 3 * m->mm_c[mi]) || !const_vec(m, 1.f, m->mm_c[mi])) return 1;
  }
  StreamStep s;
  s.pool = static_cast<char*>(pool);
  pool_layout(m, S, hp, wp, s.off);
  s.rows = table;
  s.ctx = table ? table + B : nullptr;
  s.S = S;
  s.slots = m->num_frames;
  s.stride = m->num_frames + 1;
  s.causal = causal;
  float* x = static_cast<float*>(c.a.get(static_cast<size_t>(B) * 3 * nh * nw * 4));
  RUN(c, ingest(frames, B, nh, nw, x, st));
  void* taps[4] = {nullptr, nullptr, nullptr, nullptr};
  encode(c, x, B, nh, nw, pos, taps);
  float* depth = static_cast<float*>(c.a.get(static_cast<size_t>(B) * nh * nw * 4));
  head(c, m, taps, B, 1, hp, wp, depth, &s);
  RUN(c, vda_bilinear_f32_ragged(depth, outs, B, nh, nw, st));
  if (need) *need = c.a.off + 1024;
  return c.rc;
}

}  // namespace vda

using namespace vda;

extern "C" int vda_create(const char* encoder, int features, const int32_t* out_channels, int num_frames, int dtype, int device,
                          vda_model** out) {
  VDA_CHECK(encoder && out_channels && out, "vda_create: null argument");
  VDA_CHECK(dtype == VDA_BF16 || dtype == VDA_FP16, "vda_create: bad dtype %d", dtype);
  vda_model* m = new vda_model();
  m->enc = encoder;
  if (m->enc == "vits") { m->D = 384; m->depth = 12; m->heads = 6; const int t[4] = {2, 5, 8, 11}; memcpy(m->taps, t, sizeof(t)); }
  else if (m->enc == "vitl") { m->D = 1024; m->depth = 24; m->heads = 16; const int t[4] = {4, 11, 17, 23}; memcpy(m->taps, t, sizeof(t)); }
  else { delete m; set_error("vda_create: unknown encoder '%s' (vits | vitl)", encoder); return 1; }
  m->F = features;
  for (int i = 0; i < 4; ++i) m->oc[i] = out_channels[i];
  m->num_frames = num_frames;
  m->dtype = dtype;
  m->hdtype = VDA_FP16;          // the DPT head runs on fp16 operands (engine.py: Engine.hdtype)
  m->device = device;
  m->c_l1 = pad_to(m->oc[0], 64);
  m->c_l2 = pad_to(m->oc[1], 64);
  m->c_oc1 = pad_to(m->F / 2, 64);
  if (m->oc[2] % 64 || m->oc[3] % 64 || m->F % 64) { delete m; set_error("vda_create: out_channels[2..3] and features must be multiples of 64"); return 1; }
  m->mm_c[0] = m->oc[2]; m->mm_c[1] = m->oc[3]; m->mm_c[2] = m->F; m->mm_c[3] = m->F;
  for (int i = 0; i < 4; ++i) m->mm_half[i] = (4 * m->mm_c[i]) % 128 == 0 ? 128 : 64;
  *out = m;
  return 0;
}

extern "C" int vda_set_weight(vda_model* m, const char* name, const float* host_data, const int64_t* shape, int ndim) {
  VDA_CHECK(m && name && host_data && shape && ndim >= 0 && ndim <= 8, "vda_set_weight: bad argument");
  VDA_CHECK(!m->finalized, "vda_set_weight: weights already finalized");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= static_cast<size_t>(shape[i]); }
  t.v.assign(host_data, host_data + n);
  m->sd[name] = std::move(t);
  return 0;
}

extern "C" int vda_finalize_weights(vda_model* m) {
  VDA_CHECK(m && !m->finalized, "vda_finalize_weights: bad model");
  VDA_CUDA(cudaSetDevice(m->device));
  const int D = m->D, F = m->F, dt = m->dtype, hdt = m->hdtype;
  const int* oc = m->oc;
  auto has = [&](const std::string& k) { return m->sd.count(k) != 0; };
  auto T = [&](const std::string& k) -> const HostTensor& { return m->sd.at(k); };
  auto f32 = [&](const std::string& dst, const std::string& k) { return up_f32(m, dst, T(k).v.data(), T(k).v.size()); };
  auto h16 = [&](const std::string& dst, const std::string& k, int dtp) { return up_h16(m, dst, T(k).v, dtp); };
  // every key the engine consumes must be present (strict load, like load_state_dict(strict=True))
  std::vector<std::string> need = {"pretrained.patch_embed.proj.weight", "pretrained.patch_embed.proj.bias", "pretrained.cls_token",
                                   "pretrained.pos_embed", "pretrained.norm.weight", "pretrained.norm.bias"};
  for (const auto& k : need) VDA_CHECK(has(k), "vda_finalize_weights: missing key %s", k.c_str());
  try {
    {
      const HostTensor& pw = T("pretrained.patch_embed.proj.weight");       // [D,3,14,14] -> [D, 592]
      std::vector<float> p(static_cast<size_t>(D) * KPAD_PATCH, 0.f);
      for (int r = 0; r < D; ++r) memcpy(&p[static_cast<size_t>(r) * KPAD_PATCH], &pw.v[static_cast<size_t>(r) * 588], 588 * 4);
      if (up_h16(m, "pe.w", p, dt) || f32("pe.b", "pretrained.patch_embed.proj.bias") || f32("cls", "pretrained.cls_token") ||
          f32("pos", "pretrained.pos_embed"))
        return 1;
      const int64_t npos = static_cast<int64_t>(T("pretrained.pos_embed").v.size()) / D;
      m->pos_S = static_cast<int>(lround(sqrt(static_cast<double>(npos - 1))));
    }
    for (int i = 0; i < m->depth; ++i) {
      const std::string p = "pretrained.blocks." + std::to_string(i) + ".", b = "b" + std::to_string(i) + ".";
      for (const char* n : {"norm1", "norm2"})
        if (f32(b + n + ".w", p + n + ".weight") || f32(b + n + ".b", p + n + ".bias")) return 1;
      const char* pairs[4][2] = {{"qkv", "attn.qkv"}, {"proj", "attn.proj"}, {"fc1", "mlp.fc1"}, {"fc2", "mlp.fc2"}};
      for (auto& pr : pairs)
        if (h16(b + pr[0] + ".w", p + pr[1] + ".weight", dt) || f32(b + pr[0] + ".b", p + pr[1] + ".bias")) return 1;
      if (f32(b + "ls1", p + "ls1.gamma") || f32(b + "ls2", p + "ls2.gamma")) return 1;
      if (m->ln_fold) {
        // LayerNorm fold: W' = h16(g * W), c1 = row sums of the ROUNDED W' and c2 = W beta + b, both summed in double
        // and rounded once (engine.py fold_ln does the same, so the two packings agree bit for bit)
        const char* f[2][3] = {{"qkv", "attn.qkv", "norm1"}, {"fc1", "mlp.fc1", "norm2"}};
        for (auto& q : f) {
          const HostTensor& Wt = T(p + q[1] + ".weight");
          const std::vector<float>& g = T(p + q[2] + ".weight").v;
          const std::vector<float>& beta = T(p + q[2] + ".bias").v;
          const std::vector<float>& bias = T(p + q[1] + ".bias").v;
          const int N = static_cast<int>(Wt.dim(0)), K = static_cast<int>(Wt.dim(1));
          std::vector<float> wf(Wt.v.size()), c1(static_cast<size_t>(N)), c2(static_cast<size_t>(N));
          std::vector<uint16_t> wh(Wt.v.size());
          for (int n = 0; n < N; ++n) {
            double s1 = 0.0, s2 = 0.0;
            for (int k = 0; k < K; ++k) {
              const size_t ix = static_cast<size_t>(n) * K + k;
              const float prod = Wt.v[ix] * g[static_cast<size_t>(k)];
              wh[ix] = to_h16(prod, dt);
              float back;
              if (dt == VDA_BF16) { __nv_bfloat16 hh; memcpy(&hh, &wh[ix], 2); back = __bfloat162float(hh); }
              else { __half hh; memcpy(&hh, &wh[ix], 2); back = __half2float(hh); }
              s1 += static_cast<double>(back);
              s2 += static_cast<double>(Wt.v[ix]) * static_cast<double>(beta[static_cast<size_t>(k)]);
            }
            c1[static_cast<size_t>(n)] = static_cast<float>(s1);
            c2[static_cast<size_t>(n)] = static_cast<float>(s2 + static_cast<double>(bias[static_cast<size_t>(n)]));
          }
          void* d;
          if (dev_alloc(m, wh.size() * 2, &d)) return 1;
          VDA_CUDA(cudaMemcpy(d, wh.data(), wh.size() * 2, cudaMemcpyHostToDevice));
          m->w[b + q[0] + ".wf"] = d;
          if (up_f32(m, b + q[0] + ".c1", c1.data(), c1.size()) || up_f32(m, b + q[0] + ".c2", c2.data(), c2.size())) return 1;
        }
      }
    }
    if (f32("norm.w", "pretrained.norm.weight") || f32("norm.b", "pretrained.norm.bias")) return 1;

    const std::string h = "head.";
    for (int i = 0; i < 4; ++i) {
      const std::string k = h + "projects." + std::to_string(i);
      if (h16("proj" + std::to_string(i) + ".w", k + ".weight", hdt) || f32("proj" + std::to_string(i) + ".b", k + ".bias")) return 1;
    }
    {
      std::vector<float> w, bp;
      pack_convt(T(h + "resize_layers.0.weight"), T(h + "resize_layers.0.bias"), m->c_l1, w, bp);
      if (up_h16(m, "rs0.w", w, hdt) || up_f32(m, "rs0.b", bp.data(), bp.size())) return 1;
      pack_convt(T(h + "resize_layers.1.weight"), T(h + "resize_layers.1.bias"), m->c_l2, w, bp);
      if (up_h16(m, "rs1.w", w, hdt) || up_f32(m, "rs1.b", bp.data(), bp.size())) return 1;
      if (up_h16(m, "rs3.w", pack_conv3x3(T(h + "resize_layers.3.weight"), oc[3], oc[3]), hdt) || f32("rs3.b", h + "resize_layers.3.bias"))
        return 1;
    }
    const int cin[4] = {m->c_l1, m->c_l2, oc[2], oc[3]};
    for (int i = 0; i < 4; ++i)
      if (up_h16(m, "rn" + std::to_string(i + 1) + ".w", pack_conv3x3(T(h + "scratch.layer" + std::to_string(i + 1) + "_rn.weight"), cin[i], F), hdt))
        return 1;
    for (int r = 1; r <= 4; ++r) {
      const std::string rp = h + "scratch.refinenet" + std::to_string(r) + ".", k = "rf" + std::to_string(r);
      if (h16(k + ".out.w", rp + "out_conv.weight", hdt) || f32(k + ".out.b", rp + "out_conv.bias")) return 1;
      for (int u = 1; u <= 2; ++u)
        for (int cc = 1; cc <= 2; ++cc) {
          const std::string src = rp + "resConfUnit" + std::to_string(u) + ".conv" + std::to_string(cc) + ".";
          const std::string dst = k + ".u" + std::to_string(u) + ".c" + std::to_string(cc);
          if (up_h16(m, dst + ".w", pack_conv3x3(T(src + "weight"), F, F), hdt) || f32(dst + ".b", src + "bias")) return 1;
        }
    }
    {
      if (up_h16(m, "oc1.w", pack_conv3x3(T(h + "scratch.output_conv1.weight"), F, m->c_oc1), hdt)) return 1;
      std::vector<float> b(static_cast<size_t>(m->c_oc1), 0.f);
      const std::vector<float>& sb = T(h + "scratch.output_conv1.bias").v;
      for (size_t i = 0; i < sb.size(); ++i) b[i] = sb[i];
      if (up_f32(m, "oc1.b", b.data(), b.size())) return 1;
      if (up_h16(m, "oc2.w", pack_conv3x3(T(h + "scratch.output_conv2.0.weight"), m->c_oc1, 32), hdt) ||
          f32("oc2.b", h + "scratch.output_conv2.0.bias") || f32("oc3.w", h + "scratch.output_conv2.2.weight"))
        return 1;
      m->oc3_b = T(h + "scratch.output_conv2.2.bias").v[0];
    }
    for (int mi = 0; mi < 4; ++mi) {
      const std::string t = h + "motion_modules." + std::to_string(mi) + ".temporal_transformer.", p = "mm" + std::to_string(mi) + ".";
      if (f32(p + "gn.w", t + "norm.weight") || f32(p + "gn.b", t + "norm.bias") || h16(p + "in.w", t + "proj_in.weight", hdt) ||
          f32(p + "in.b", t + "proj_in.bias") || h16(p + "out.w", t + "proj_out.weight", hdt) || f32(p + "out.b", t + "proj_out.bias"))
        return 1;
      const std::string blk = t + "transformer_blocks.0.";
      for (int a = 0; a < 2; ++a) {
        const std::string ab = blk + "attention_blocks." + std::to_string(a) + ".", dst = p + "a" + std::to_string(a) + ".";
        std::vector<float> cat;
        for (const char* n : {"to_q.weight", "to_k.weight", "to_v.weight"}) cat.insert(cat.end(), T(ab + n).v.begin(), T(ab + n).v.end());
        if (up_h16(m, dst + "qkv.w", cat, hdt) || h16(dst + "o.w", ab + "to_out.0.weight", hdt) || f32(dst + "o.b", ab + "to_out.0.bias") ||
            f32(dst + "pe", ab + "pos_encoder.pe") || f32(dst + "ln.w", blk + "norms." + std::to_string(a) + ".weight") ||
            f32(dst + "ln.b", blk + "norms." + std::to_string(a) + ".bias"))
          return 1;
        // streaming: pet = pe[:32] [W_q | W_k | W_v]^T fp32 [32, 3C], summed in double and rounded once (engine.py load
        // does the same, so both tables hold the same bits); the step kernels add it at a frame's current position
        const int C = m->mm_c[mi];
        const std::vector<float>& pe = T(ab + "pos_encoder.pe").v;
        const int npe = static_cast<int>(pe.size() / static_cast<size_t>(C)) < 32 ? static_cast<int>(pe.size() / C) : 32;
        std::vector<float> pet(static_cast<size_t>(32) * 3 * C, 0.f);
        for (int r = 0; r < npe; ++r)
          for (int n = 0; n < 3 * C; ++n) {
            double acc = 0.0;
            for (int k = 0; k < C; ++k)
              acc += static_cast<double>(pe[static_cast<size_t>(r) * C + k]) * static_cast<double>(cat[static_cast<size_t>(n) * C + k]);
            pet[static_cast<size_t>(r) * 3 * C + n] = static_cast<float>(acc);
          }
        if (up_f32(m, dst + "pet", pet.data(), pet.size())) return 1;
      }
      if (f32(p + "ffn.w", blk + "ff_norm.weight") || f32(p + "ffn.b", blk + "ff_norm.bias")) return 1;
      std::vector<float> wp, bp;
      pack_geglu(T(blk + "ff.net.0.proj.weight"), T(blk + "ff.net.0.proj.bias"), m->mm_half[mi], wp, bp);
      if (up_h16(m, p + "ff0.w", wp, hdt) || up_f32(m, p + "ff0.b", bp.data(), bp.size()) || h16(p + "ff2.w", blk + "ff.net.2.weight", hdt) ||
          f32(p + "ff2.b", blk + "ff.net.2.bias"))
        return 1;
      if (!const_vec(m, 0.f, 3 * m->mm_c[mi]) || !const_vec(m, 1.f, m->mm_c[mi])) return 1;
    }
  } catch (const std::out_of_range&) {
    set_error("vda_finalize_weights: a state-dict key of the reference model is missing (strict load)");
    return 1;
  }
  m->sd.clear();
  m->finalized = true;
  return 0;
}

extern "C" int64_t vda_workspace_bytes(vda_model* m, int B, int T, int H, int W) {
  if (!m || !m->finalized || B <= 0 || T <= 0 || H % 14 || W % 14 || H <= 0 || W <= 0) return -1;
  size_t need = 0;
  if (run_forward(m, nullptr, B, T, H, W, nullptr, nullptr, 0, nullptr, true, &need)) return -1;
  return static_cast<int64_t>(need);
}

extern "C" int vda_forward(vda_model* m, const float* x, int B, int T, int H, int W, float* depth, void* workspace,
                           int64_t workspace_bytes, void* stream) {
  VDA_CHECK(m && m->finalized, "vda_forward: weights not finalized");
  VDA_CHECK(x && depth && workspace, "vda_forward: null pointer");
  VDA_CHECK(B > 0 && T > 0 && T <= m->num_frames, "vda_forward: bad clip shape B=%d T=%d (temporal_max_len %d)", B, T, m->num_frames);
  VDA_CHECK(H > 0 && W > 0 && H % 14 == 0 && W % 14 == 0, "vda_forward: H (%d) and W (%d) must be multiples of the patch size 14", H, W);
  VDA_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "vda_forward: workspace must be 1024-byte aligned");
  {
    // size check BEFORE anything is launched (a dry run of the schedule is host arithmetic only)
    size_t need = 0;
    if (run_forward(m, nullptr, B, T, H, W, nullptr, nullptr, 0, nullptr, true, &need)) return 1;
    VDA_CHECK(static_cast<size_t>(workspace_bytes) >= need, "vda_forward: workspace too small: %zu bytes needed, %lld given", need,
              static_cast<long long>(workspace_bytes));
  }
  return run_forward(m, x, B, T, H, W, depth, workspace, static_cast<size_t>(workspace_bytes), stream, false, nullptr);
}

extern "C" int64_t vda_stream_pool_bytes(vda_model* m, int S, int nh, int nw) {
  if (!m || S < 1 || nh <= 0 || nw <= 0 || nh % 14 || nw % 14) return -1;
  size_t off[8];
  return static_cast<int64_t>(pool_layout(m, S, nh / 14, nw / 14, off));
}

extern "C" int64_t vda_stream_workspace_bytes(vda_model* m, int B, int nh, int nw) {
  if (!m || !m->finalized || B < 1 || nh <= 0 || nw <= 0 || nh % 14 || nw % 14) return -1;
  size_t need = 0;
  if (run_step<vda_frame_desc>(m, vda_preprocess_frames_ragged, nullptr, nullptr, nullptr, B, false, nullptr, 1, nh, nw, nullptr,
                               0, nullptr, true, &need))
    return -1;
  return static_cast<int64_t>(need);
}

// vda_stream_step and vda_stream_step_planes: the checks, then the step with the frames' ingest
template <class Desc>
static int stream_step(const char* fn, vda_model* m, int (*ingest)(const Desc*, int, int, int, float*, void*),
                       const Desc* frames, const vda_out_desc* outs, const int32_t* table, int B, int causal, void* pool, int S,
                       int nh, int nw, void* workspace, int64_t workspace_bytes, void* stream) {
  VDA_CHECK(m && m->finalized, "%s: weights not finalized", fn);
  VDA_CHECK(frames && outs && table && pool && workspace, "%s: null pointer", fn);
  VDA_CHECK(B >= 1, "%s: bad batch B=%d", fn, B);
  VDA_CHECK(S >= 1, "%s: bad pool size S=%d", fn, S);
  VDA_CHECK(m->num_frames >= 2 && m->num_frames <= 32, "%s: streaming needs num_frames in 2..32, got %d", fn,
            m->num_frames);
  VDA_CHECK(nh > 0 && nw > 0 && nh % 14 == 0 && nw % 14 == 0,
            "%s: nh (%d) and nw (%d) must be multiples of the patch size 14", fn, nh, nw);
  VDA_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "%s: workspace must be 1024-byte aligned", fn);
  VDA_CHECK((reinterpret_cast<uintptr_t>(pool) & 255) == 0, "%s: pool must be 256-byte aligned", fn);
  {
    size_t need = 0;
    if (run_step(m, ingest, static_cast<const Desc*>(nullptr), nullptr, nullptr, B, false, nullptr, S, nh, nw, nullptr, 0,
                 nullptr, true, &need))
      return 1;
    VDA_CHECK(workspace_bytes >= 0 && static_cast<size_t>(workspace_bytes) >= need, "%s: workspace too small: %zu bytes needed, %lld given",
              fn, need, static_cast<long long>(workspace_bytes));
  }
  return run_step(m, ingest, frames, outs, table, B, causal != 0, pool, S, nh, nw, workspace, static_cast<size_t>(workspace_bytes),
                  stream, false, nullptr);
}

extern "C" int vda_stream_step(vda_model* m, const vda_frame_desc* frames, const vda_out_desc* outs, const int32_t* table, int B,
                               int causal, void* pool, int S, int nh, int nw, void* workspace, int64_t workspace_bytes,
                               void* stream) {
  return stream_step("vda_stream_step", m, vda_preprocess_frames_ragged, frames, outs, table, B, causal, pool, S, nh, nw,
                     workspace, workspace_bytes, stream);
}

extern "C" int vda_stream_step_planes(vda_model* m, const vda_frame_planes* frames, const vda_out_desc* outs,
                                      const int32_t* table, int B, int causal, void* pool, int S, int nh, int nw,
                                      void* workspace, int64_t workspace_bytes, void* stream) {
  return stream_step("vda_stream_step_planes", m, vda_preprocess_frames_planes, frames, outs, table, B, causal, pool, S, nh,
                     nw, workspace, workspace_bytes, stream);
}

extern "C" int vda_destroy(vda_model* m) {
  if (!m) return 0;
  for (void* p : m->owned) cudaFree(p);
  delete m;
  return 0;
}
