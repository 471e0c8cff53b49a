/* libvda — C ABI of the B200-native Video-Depth-Anything hot path.
 *
 * The reference has no FFI: its boundary is the Python nn.Module surface
 * (video_depth_anything/video_depth.py:38-63 ctor, :89-164 forward, :166-254 infer_video_depth).
 * Everything those functions delegate to torch.nn / ATen operators is replaced by the entry points
 * below (one per operator family); the Python mirror in video_depth_anything_b200/ binds them with
 * ctypes (see INTEGRATION.md).  Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error (message: vda_last_error()).
 *   - all pointers are DEVICE pointers unless named host_*; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*), no hidden synchronisation.
 *   - "h16" tensors hold 16-bit floats: bf16 when dtype == VDA_BF16, fp16 when VDA_FP16.
 *   - activations are token-major / NHWC:  [frames, h*w, C].
 */
#ifndef VDA_H_
#define VDA_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { VDA_BF16 = 0, VDA_FP16 = 1 };
enum { VDA_OUT_H16 = 0, VDA_OUT_F32 = 1 };
enum { VDA_ACT_NONE = 0, VDA_ACT_GELU = 1, VDA_ACT_RELU = 2 };

/* epilogue families of the tensor-core GEMM */
enum {
  VDA_EPI_LINEAR = 0, /* bias, layer-scale, activation, up to two residuals, optional relu'd copy        */
  VDA_EPI_GEGLU = 1,  /* out[m,j] = (a+ba) * gelu(g+bg); weight rows interleaved per 2*geglu_half block  */
  VDA_EPI_CONVT = 2,  /* ConvTranspose2d with kernel == stride: pixel-shuffle scatter store              */
  VDA_EPI_TAIL = 3    /* relu(acc+bias) . w2 + b2 -> relu -> fp32 scalar per row (output_conv2)          */
};

/* A-operand addressing */
enum {
  VDA_A_PLAIN = 0,  /* A is a row-major [M,K] h16 matrix with row stride lda                            */
  VDA_A_CONV3 = 1   /* implicit 3x3 / stride 1 / pad 1 convolution over an NHWC h16 tensor              */
};

typedef struct vda_gemm_params {
  /* problem: out[M,N] = A[M,K] . Wt[N,K]^T  (both K-major, h16), fp32 accumulation in TMEM */
  int32_t M, N, K;
  int32_t dtype;    /* VDA_BF16 | VDA_FP16 */
  int32_t a_mode;   /* VDA_A_PLAIN | VDA_A_CONV3 */
  int32_t epilogue; /* VDA_EPI_* */
  const void* A;    /* plain: [M,lda]; conv: NHWC [n_img,H,W,C] (C % 64 == 0, K == 9*C)        */
  int64_t lda;
  const void* Wt;   /* [N,K] row-major (nn.Linear layout); conv: K index = (ky*3+kx)*C + ci     */
  int32_t n_img, H, W, C;

  /* LINEAR epilogue: v = acc + bias[n]; v *= gamma[n]; v = act(v); v += res1[r,n]; v += res2[r,n] */
  const float* bias;   /* [N] or NULL */
  const float* gamma;  /* [N] or NULL (LayerScale, dinov2_layers/layer_scale.py:27-28) */
  int32_t act;         /* VDA_ACT_* */
  const void* res1;    /* NULL, or [rows,ldr1] fp32 (res1_f32 != 0) / h16 */
  int64_t ldr1;
  int32_t res1_f32;
  const void* res2;    /* NULL or h16 [rows,ldo] */
  void* out;           /* [rows,ldo] h16 or fp32 (out_f32) */
  int64_t ldo;
  int32_t out_f32;
  void* out_relu;      /* NULL or h16 [rows,ldo]: relu(v), the pre-activated copy an RCU conv1 consumes */
  /* row remap for the patch-embed GEMM (dinov2.py:212-219): with group = patches per frame,
     out row = m + m/group + 1 (skips each frame's cls row) and res1 row = m % group + 1 (pos_embed). */
  int32_t row_group;   /* 0 = identity mapping */

  /* GEGLU: N is the packed width (2*inner); out has N/2 columns */
  int32_t geglu_half;  /* columns of `a` per interleaved block (block = [a(half) | g(half)]) */

  /* CONVT: rows are input pixels (img,y,x) of an in_h x in_w map; column j = (ky*S+kx)*Co + co */
  int32_t convt_s, convt_co, in_h, in_w;

  /* TAIL: N == 32; out is fp32 [rows] */
  const float* tail_w; /* [32] */
  float tail_b;

  /* LayerNorm folding (dinov2_layers/block.py:82-107: x = x + ls1(attn(norm1(x))); x = x + ls2(mlp(norm2(x)))).
   * Producer (proj / fc2: bias, gamma, fp32 residual updated in place, res1 == out): besides the fp32 rows it writes
   *   out16          h16 copy of the new rows [rows, ldo]                                  (NULL: not wanted)
   *   row_stats_out  fp32 [rows, stat_parts, 2] = (mean, M2) of each row over consecutive column groups
   *                  (layout from vda_gemm_rowstat_layout; stat_parts must match)          (NULL: not wanted)
   * Consumer (qkv / fc1: bias, optional GELU, h16 out): with row_stats_in != NULL, A holds the UN-normalised h16 rows
   * and the LayerNorm is applied in the epilogue:  out = rstd_r (acc - mu_r ln_c1[n]) + bias[n],  where Wt holds
   * h16(ln_weight * W) row-wise, ln_c1[n] = sum_k Wt[n,k] (of the rounded values) and bias[n] = W ln_bias + b;
   * (mu_r, rstd_r) come from the stat_parts partials of stat_cols columns each (stat_parts * stat_cols == K). */
  void* out16;
  float* row_stats_out;
  const float* row_stats_in;
  const float* ln_c1;
  int32_t stat_parts, stat_cols;
  float ln_eps;

  /* Validation precision (`fp32=True`, reference video_depth.py:203-205): weights as a hi | lo pair of h16 matrices.
   * a_k > 0: A is [M, a_k] and Wt is [N, K] with K == 2 * round_up(a_k, 64): columns [0, a_k) hold h16(W), columns
   * [K/2, K/2 + a_k) hold h16(W - h16(W)), the rest zeros; A is walked twice, so out = A (Wh + Wl)^T with the weights'
   * rounding error squared.  0: plain (A is [M, K]). */
  int32_t a_k;
} vda_gemm_params;

int vda_version(void);
const char* vda_last_error(void);
/* fills sm count and compute capability of `device`; returns non-zero if it is not sm_100 */
int vda_device_query(int device, int* sm_count, int* cc_major, int* cc_minor);

/* tcgen05/TMEM/TMA GEMM + implicit-GEMM conv (replaces nn.Linear / nn.Conv2d / nn.ConvTranspose2d call sites:
 * dinov2_layers/attention.py:44-46, mlp.py:30-32, patch_embed.py:66, dpt.py:60-90,117-124, util/blocks.py:20-32,52-58,
 * 124-126, motion_module/motion_module.py:85,100, motion_module/attention.py:81-83,90,335-338,382-384) */
int vda_gemm(const vda_gemm_params* p, void* stream);
/* layout of row_stats_out for an [M, N] output: `parts` partials per row over `part_cols` consecutive columns each */
int vda_gemm_rowstat_layout(int M, int N, int* parts, int* part_cols);

/* nn.LayerNorm over the last dim (block.py:56,68; dinov2.py:165,309-310; motion_module.py:156-163).
 * in: fp32 (in_f32) or h16 [rows, C]; out: h16 [rows_out, C].
 * drop_group > 0: input rows are frames of drop_group tokens whose first (cls) token is dropped
 * (dinov2.py:312), out row = r - r/drop_group - 1.
 * pe != NULL: adds pe[(r / pe_rows_per_frame) % pe_frames, :] after the affine (PositionalEncoding,
 * motion_module.py:196-198, applied to the normed states at :234-235). */
int vda_layernorm(const void* in, int in_f32, void* out, const float* w, const float* b, float eps, int64_t rows,
                  int C, int dtype, int drop_group, const float* pe, int pe_rows_per_frame, int pe_frames,
                  void* stream);

/* LayerNorm folding, start of the chain (see vda_gemm_params.row_stats_in): h16 copy of the fp32 rows `in` [rows, C]
 * and their per-row partial statistics fp32 [rows, parts, 2] = (mean, M2) over part_cols consecutive columns each
 * (parts * part_cols == C), the format a residual GEMM with row_stats_out writes. */
int vda_rowstats_cast(const float* in, void* out16, float* stats, int64_t rows, int C, int parts, int part_cols, int dtype,
                      void* stream);

/* GroupNorm(32, C, eps) per frame over an NHWC h16 tensor [frames, hw, C] (motion_module.py:84,110).
 * stats: fp32 scratch of VDA_GN_STATS_FLOATS(frames, groups) floats (per-slab partial sums + per-frame totals;
 * no atomics, so the result is bit-reproducible). */
#define VDA_GN_STATS_FLOATS(frames, groups) ((592 + 2 * (frames)) * (groups) * 2)
int vda_groupnorm(const void* in, void* out, const float* w, const float* b, float eps, int frames, int hw, int C,
                  int groups, float* stats, int dtype, void* stream);

/* fused softmax(q k^T / sqrt(64)) v for the spatial ViT attention (dinov2_layers/attention.py:49-62).
 * qkv: h16 [frames, N, 3, heads, 64] (the qkv Linear's output), out: h16 [frames, N, heads*64]. */
int vda_attention_spatial(const void* qkv, void* out, int frames, int N, int heads, int dtype, void* stream);

/* temporal attention core over the frame axis at every spatial position (motion_module.py:230-297 with
 * motion_module/attention.py:182-211).  qkv: h16 [T*hw, 3*C] rows ordered (frame, position), columns
 * [q | k | v], each split in `heads` heads of C/heads.  out: h16 [T*hw, C]. */
int vda_attention_temporal(const void* qkv, void* out, int T, int hw, int C, int heads, int dtype, void* stream);

/* Streaming temporal attention: the current frame's query against the cached frames of the stream and itself.
 *   qkv:   h16 [hw, 3*C], the current frame's q'|k'|v' (the q|k|v Linear applied to the LayerNorm output WITHOUT the
 *          positional encoding);
 *   cache: h16 [slots, hw, 2*C], per slot and position the row k'|v' of an earlier frame;
 *   pe:    fp32 [32, 3*C], pe[p] @ [W_q | W_k | W_v]^T, the positional encoding's share of q|k|v at position p;
 *   ctx:   device int32 [2 + n_ctx] = {n_ctx, write_slot, slot of context position 0, ..., n_ctx - 1}, n_ctx <= 31
 *          (larger values are clamped to 31, slot indices to slots - 1).
 * Keys / values are the n_ctx cached rows (position p: k' + pe_k[p], v' + pe_v[p]) followed by the current frame at
 * position n_ctx, whose query is q' + pe_q[n_ctx]; out: h16 [hw, C] = softmax(q k^T / sqrt(C/heads)) v per head, fp32
 * inside.  The current frame's k'|v' rows are also copied, unchanged, into slot `write_slot` of the cache, which must
 * not be one of the slots read.  Everything that changes from step to step is in `ctx`, so a captured CUDA graph
 * replays it.  The B = 1 case of vda_attention_temporal_step_batched on pool entry 0. */
int vda_attention_temporal_step(const void* qkv, void* cache, const float* pe, const int32_t* ctx, void* out, int hw,
                                int C, int heads, int slots, int dtype, void* stream);

/* The streaming step of B frames of different streams in one launch (a group of streams pushing together):
 *   qkv:  h16 [B*hw, 3*C], row block b = batch row b's q'|k'|v';
 *   pool: h16 [S, slots, hw, 2*C], one cache as above per stream;
 *   rows: device int32 [B], the pool entry of batch row b; -1 marks a pad row;
 *   ctx:  device int32 [B, ctx_stride], row b laid out as ctx above (n_ctx is also clamped to ctx_stride - 2).
 * A real row does exactly what vda_attention_temporal_step does against pool[rows[b]], including the write of its k'|v'
 * into its write slot.  A row whose pool index is outside 0..S-1 (a pad row) attends to itself only (n_ctx = 0) and
 * reads and writes no pool byte; pool entries no row names are not touched.  out: h16 [B*hw, C]. */
int vda_attention_temporal_step_batched(const void* qkv, void* pool, const float* pe, const int32_t* rows,
                                        const int32_t* ctx, void* out, int B, int S, int ctx_stride, int hw, int C,
                                        int heads, int slots, int dtype, void* stream);

/* The streaming step of several consecutive frames of one stream (and of other streams) in one launch.  Arguments as
 * for vda_attention_temporal_step_batched, with two differences:
 *   ctx:  a context entry e >= 0 is a slot of the row's pool entry, as there; an entry e < 0 names batch row -1 - e of
 *         this launch (clamped to 0..B-1): that key's k'|v' are read from the row's block of `qkv` (columns C..3C) at
 *         the same position, with the positional share of its place in this row's sequence.  So frame t + j of a push
 *         reads its context frames >= t from the push's own rows and the older ones from the pool.
 *   pool: only read.  The kernel writes no cache slot: with k >= 2 frames of one stream in a launch, the slot frame
 *         t + j overwrites (that of frame t + j - L) is still a context slot of the push's earlier rows, so the writes
 *         are deferred to vda_stream_cache_store, launched after this kernel on the same stream.
 * Per row, the key order, key-split assignment and arithmetic are those of vda_attention_temporal_step_batched, so a
 * row is bit-identical to that kernel run with the same keys in the pool.  Pad rows as there. */
int vda_attention_temporal_step_causal(const void* qkv, const void* pool, const float* pe, const int32_t* rows,
                                       const int32_t* ctx, void* out, int B, int S, int ctx_stride, int hw, int C,
                                       int heads, int slots, int dtype, void* stream);

/* The deferred cache write of a causal step: for every real batch row b (0 <= rows[b] < S), its k'|v' (columns C..3C of
 * its rows of qkv h16 [B*hw, 3*C]) are copied unchanged to pool[rows[b]], slot ctx[b][1] (clamped to 0..slots-1); no
 * other pool byte is touched.  Bandwidth-bound, 16-byte accesses. */
int vda_stream_cache_store(const void* qkv, void* pool, const int32_t* rows, const int32_t* ctx, int B, int S,
                           int ctx_stride, int hw, int C, int slots, int dtype, void* stream);

/* Frame preprocessing of infer_video_depth (video_depth.py:173-185,197-198; util/transform.py:109-158): for every
 * i < n, frame idx[i] of the device-resident uint8 RGB video frames [*, H0, W0, 3] -> /255 -> cv2-style INTER_CUBIC
 * resize to (nh, nw) -> (x - mean) / std (float64) -> out fp32 [n, 3, nh, nw].  idx: device int32 [n]. */
int vda_preprocess_frames(const uint8_t* frames, const int32_t* idx, float* out, int n, int H0, int W0, int nh, int nw,
                          void* stream);

/* Frame preprocessing of a ragged batch (util/transform.py:109-158): batch row i < n is its own frame, described by
 * rows[i] (device memory, read by the kernel); every row is resized to the same (nh, nw) -> out fp32 [n, 3, nh, nw].
 * Per row bit-identical to vda_preprocess_frames of that frame alone (same per-pixel code).  Pixels are 3 contiguous
 * bytes (RGB), row y of a frame starts at src + y * pitch, pitch >= 3 * W0. */
typedef struct vda_frame_desc {
  const uint8_t* src;
  int64_t pitch;
  int32_t H0, W0;
} vda_frame_desc;
int vda_preprocess_frames_ragged(const vda_frame_desc* rows, int n, int nh, int nw, float* out, void* stream);

/* YUV 4:2:0 frames, as video decoders hand them over: NVDEC / GStreamer / DeepStream give NV12 (a Y plane, then one
 * interleaved U,V plane), FFmpeg's software decoders I420 = yuv420p (a Y plane, then a U and a V plane).  Chroma planes
 * are [H0/2, W0/2] samples; H0 and W0 must be even.  Each pixel is converted to RGB as it is fetched, then goes through
 * the RGB path above unchanged.  The conversion is BT.601 limited range with nearest chroma -- pixel (y, x) takes chroma
 * sample (y/2, x/2) -- in the integer form of OpenCV's cv2.cvtColor(COLOR_YUV2RGB_NV12 / COLOR_YUV2RGB_I420), which it
 * equals on every (Y, U, V) triple:
 *   u' = U - 128, v' = V - 128, y' = max(0, Y - 16) * 1220542, h = 1 << 19
 *   R = clamp((y' + h + 1673527 v') >> 20, 0, 255)
 *   G = clamp((y' + h - 852492 v' - 409993 u') >> 20, 0, 255)
 *   B = clamp((y' + h + 2116026 u') >> 20, 0, 255)
 * So a YUV frame gives bit-identical results to its cv2-converted RGB frame through the RGB entry points. */
enum { VDA_PIX_NV12 = 1, VDA_PIX_I420 = 2 };

/* vda_preprocess_frames for packed YUV 4:2:0 frames in OpenCV's layout: frame i is 3 * H0 * W0 / 2 bytes, the Y plane
 * [H0, W0], then the UV plane [H0/2, W0] (NV12) or the U and V planes [H0/2, W0/2] each (I420), no padding. */
int vda_preprocess_frames_yuv(const uint8_t* frames, const int32_t* idx, int format, float* out, int n, int H0, int W0,
                              int nh, int nw, void* stream);

/* vda_preprocess_frames_ragged for YUV 4:2:0 frames: batch row i reads rows[i] (device memory, read by the kernel).
 * Every plane has its own address and row pitch in bytes, so decoder surfaces are read in place (an NVDEC surface puts
 * its UV plane at Y + pitch * aligned height, not right after row H0 - 1).  NV12: plane = {Y, UV}, pitch[0] >= W0,
 * pitch[1] >= W0, plane[2] / pitch[2] unused; I420: plane = {Y, U, V}, pitch[0] >= W0, pitch[1], pitch[2] >= W0/2.
 * H0 and W0 even, format VDA_PIX_NV12 | VDA_PIX_I420, reserved 0.  The descriptors live in device memory and are not
 * checked by the launcher; the host that writes them checks them (the Python mirror does: windows.group_descriptors).
 * The per-row format leaves room for other pixel formats without an ABI change. */
typedef struct vda_frame_planes {
  const uint8_t* plane[3];
  int64_t pitch[3];
  int32_t H0, W0, format, reserved;
} vda_frame_planes; /* 64 bytes */
int vda_preprocess_frames_planes(const vda_frame_planes* rows, int n, int nh, int nw, float* out, void* stream);

/* Encoder-feature reuse across overlapping windows (video_depth.py:197-201: 10 of a window's 32 slots repeat frames
 * of earlier windows, and the DINOv2 encoder is per-frame): copies n per-frame slabs of frame_bytes bytes, slab
 * src_idx[i] of src -> slab dst_idx[i] of dst (device int32 lists; NULL = identity).  frame_bytes % 16 == 0. */
int vda_copy_frames(const void* src, const int32_t* src_idx, void* dst, const int32_t* dst_idx, int n,
                    int64_t frame_bytes, void* stream);

/* Sequence evaluation (benchmark/eval/eval.py:67-122 eval_depthcrafter + benchmark/eval/metric.py abs_relative_difference,
 * rmse_linear, delta1_acc): pred = predicted disparity fp32 [frames,hw]; gt = depth [frames,hw], fp32 or fp64 (gt_f64),
 * <= 1e-3 or >= max_depth = invalid.  Masked least-squares (scale, shift) of clip(pred,1e-3) to 1/(gt+1e-8) over the whole
 * sequence, then per-frame masked metrics of clip(1/clip(scale pred + shift,1e-3),1e-3,max_depth), averaged over the frames
 * with valid pixels.  All arithmetic in double (as the reference).  out: device double[3] = {AbsRel, RMSE, delta1};
 * scale_shift: device double[2]; scratch: device double[VDA_EVAL_LSQ_PARTIALS*5 + frames*VDA_EVAL_SLABS*4]. */
#define VDA_EVAL_LSQ_PARTIALS 592
#define VDA_EVAL_SLABS 64
int vda_eval_sequence(const float* pred, const void* gt, int gt_f64, int frames, int64_t hw, double max_depth, double* out,
                      double* scale_shift, double* scratch, void* stream);

/* Temporal alignment error (benchmark/eval/eval_tae.py:60-107 tae_torch, :109-213 eval_TAE).
 * vda_eval_aligned_depth: out[i] = clip(1 / clip(scale * clip(pred[i], 1e-3) + shift, 1e-3), 1e-3, max_depth) in double
 * (eval_tae.py:152-160), scale_shift from vda_eval_sequence.
 * vda_eval_tae: `jobs` ordered frame pairs; job j un-projects depth[src_idx[j]] (double [frames, H*W]) with the pinhole
 * intrinsics, applies the rigid motion, projects, rounds (half to even) and scatters the transformed depth into frame
 * dst_idx[j] with the reference's last-writer rule for duplicate targets (largest source index wins: exact integer
 * atomicMax, then a deterministic gather), and returns in out[j] the mean of |depth_dst - proj| / depth_dst over pixels
 * with proj > 0, depth_dst > 0 and masks[dst] != 0 (masks: uint8 [frames, H*W] or NULL), 0 if there is none.
 * params: double [jobs, 16] = R (row-major 3x3), t (3), fx, fy, cx, cy.  winners: int32 scratch [jobs, H*W];
 * partials: double scratch [jobs, VDA_EVAL_SLABS, 2]. */
int vda_eval_aligned_depth(const float* pred, const double* scale_shift, double max_depth, int64_t n, double* out,
                           void* stream);
int vda_eval_tae(const double* depth, const uint8_t* masks, const double* params, const int32_t* src_idx,
                 const int32_t* dst_idx, int jobs, int H, int W, int32_t* winners, double* partials, double* out,
                 void* stream);

/* im2col of the 14x14/14 patch-embed conv (patch_embed.py:66,76): x fp32 [frames,3,H,W] ->
 * A h16 [frames*hp*wp, kpad], column = c*196 + ky*14 + kx, zero padded to kpad. */
int vda_patch_im2col(const float* x, void* A, int frames, int H, int W, int kpad, int dtype, void* stream);

/* tokens[f, 0, :] = cls_token + pos_embed[0]   (dinov2.py:218-219); tokens fp32 [frames, tokens_per_frame, D] */
int vda_write_cls(float* tokens, const float* cls_token, const float* pos, int frames, int tokens_per_frame, int D,
                  void* stream);

/* bicubic pos-embed resampling (dinov2.py:179-210; A=-0.75, src=(dst+0.5)/scale-0.5, clamped taps).
 * pos_in fp32 [1+S*S, D] -> pos_out fp32 [1+hp*wp, D] */
int vda_pos_embed_bicubic(const float* pos_in, float* pos_out, int S, int hp, int wp, int D, void* stream);

/* im2col of a 3x3 / stride 2 / pad 1 conv over NHWC h16 (dpt.py:84-89): out [n*oh*ow, 9*C] */
int vda_im2col3x3_s2(const void* in, void* out, int n, int H, int W, int C, int dtype, void* stream);

/* bilinear, align_corners=True, NHWC h16 [n,ih,iw,C] -> [n,oh,ow,C] (util/blocks.py:156-158, dpt_temporal.py:94-96) */
int vda_bilinear_nhwc(const void* in, void* out, int n, int ih, int iw, int oh, int ow, int C, int dtype,
                      void* stream);

/* Fused depth-head tail (dpt_temporal.py:94-100, dpt.py:118-124): bilinear (align_corners=True) upsample of the
 * output_conv1 map to (OH, OW), 3x3 conv C -> 32 (+bias, ReLU), 1x1 conv 32 -> 1 (+bias, ReLU), one kernel; the
 * upsampled map never exists in memory.  in: h16 NHWC [n, IH, IW, C] (C = 64 or 128), w: h16 [32, 9*C] with
 * K = (ky*3+kx)*C + ci, bias/w2: fp32 [32], out: fp32 [n, OH, OW]. */
int vda_tail_fused(const void* in, const void* w, const float* bias, const float* w2, float b2, float* out, int n,
                   int IH, int IW, int OH, int OW, int C, int dtype, void* stream);

/* bilinear, align_corners=True, single-channel fp32 [n,ih,iw] -> [n,oh,ow] (video_depth.py:162,208) */
int vda_bilinear_f32(const float* in, float* out, int n, int ih, int iw, int oh, int ow, void* stream);

/* The same per row of a ragged batch (video_depth.py:208): row i of in fp32 [n, ih, iw] -> rows[i].dst fp32
 * [rows[i].H0, rows[i].W0] (descriptors in device memory, read by the kernel), bit-identical to vda_bilinear_f32 of that
 * row alone; a row of size (ih, iw) is copied, a row with H0 == 0 writes nothing. */
typedef struct vda_out_desc {
  float* dst;
  int32_t H0, W0;
} vda_out_desc;
int vda_bilinear_f32_ragged(const float* in, const vda_out_desc* rows, int n, int ih, int iw, void* stream);

/* h16 elementwise: out = a + b (either may alias out) */
int vda_add_h16(const void* a, const void* b, void* out, int64_t n, int dtype, void* stream);

/* Key-frame least squares (utils/util.py:40-62 with the all-ones mask of video_depth.py:230-232).
 * pred/target: fp32 [n] (two frames each).  scale_shift: fp32 [2] <- (s, t); identity if det == 0.
 * scratch: double [4 * VDA_LSQ_MAX_PARTIALS] workspace (per-CTA partial sums, reduced in a fixed order so the
 * result is bit-reproducible run to run and across GPU counts). */
#define VDA_LSQ_MAX_PARTIALS 592
int vda_lsq_scale_shift(const float* pred, const float* target, int64_t n, float* scale_shift, double* scratch,
                        void* stream);

/* The whole sequential (scale, shift) recurrence of a video in one cooperative kernel (video_depth.py:216-252): what
 * WindowAligner does window by window with vda_lsq_scale_shift + vda_affine_clamp_blend on the key frame, for the
 * multi-GPU driver, which walks the chain once the anchor frames of every rank's windows are gathered
 * (parallel.py).  anchors: fp32 [n_windows, 3, hw] = raw slots 0, 1, 12 of every window; table: fp32 [n_windows, 2]
 * <- (scale, shift) per window, (1, 0) for window 0; affine == 0 (metric model,
 * metric_depth/video_depth_anything/video_depth.py:132): all (1, 0).  scratch: double [8 * VDA_LSQ_MAX_PARTIALS].
 * Bit-identical to the per-window calls (same thread mapping, accumulation order and solve). */
int vda_align_chain(const float* anchors, int n_windows, int64_t hw, int affine, float* table, double* scratch,
                    void* stream);

/* out = max(0, s*x + t) with (s,t) read from device memory; if blend_w != NULL (fp32 [frames]) then
 * out[f] = prev[f]*(1-w[f]) + max(0, s*x[f]+t)*w[f]  (video_depth.py:234-250, utils/util.py:65-74).
 * x, prev, out: fp32 [frames, hw]. */
int vda_affine_clamp_blend(const float* x, const float* scale_shift, const float* prev, const float* blend_w,
                           float* out, int frames, int64_t hw, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Handle-level API: the whole forward of VideoDepthAnything (video_depth_anything/video_depth.py:36-164) behind five calls,
 * for hosts that do not want to re-implement the engine's launch schedule (csrc/model.cu is that schedule: the same
 * sequence of the operator entry points above as video_depth_anything_b200/engine.py, bit-identical output).
 *
 *   vda_create            encoder "vits" | "vitl" (dinov2.py:339-378), features / out_channels / num_frames as the reference
 *                         constructor (video_depth.py:38-63); dtype = operand type of the encoder (the DPT head uses fp16)
 *   vda_set_weight        one tensor of the reference state dict (same keys as model.state_dict(), SURVEY.md App. C), fp32,
 *                         HOST memory, row-major in the reference's own shape; copies
 *   vda_finalize_weights  packs everything into the kernel layouts on `device` (strict: a missing key is an error)
 *   vda_workspace_bytes   size of the scratch buffer vda_forward needs for a [B,T,3,H,W] input (-1 on error)
 *   vda_forward           x: device fp32 [B,T,3,H,W] (normalised frames, as forward() receives them) -> depth: device fp32
 *                         [B,T,H,W] >= 0.  workspace: device, 1024-byte aligned, >= vda_workspace_bytes.  Enqueues on
 *                         `stream`, does not synchronise or allocate (the first call for a new token grid other than
 *                         37x37 resamples the position embedding into model-owned memory).  H, W multiples of 14
 *                         (patch_embed.py:73-74), T <= num_frames (dpt_temporal.py:38). */
typedef struct vda_model vda_model;
int vda_create(const char* encoder, int features, const int32_t* out_channels, int num_frames, int dtype, int device,
               vda_model** out);
int vda_set_weight(vda_model* m, const char* name, const float* host_data, const int64_t* shape, int ndim);
int vda_finalize_weights(vda_model* m);
int64_t vda_workspace_bytes(vda_model* m, int B, int T, int H, int W);
int vda_forward(vda_model* m, const float* x, int B, int T, int H, int W, float* depth, void* workspace,
                int64_t workspace_bytes, void* stream);
int vda_destroy(vda_model* m);

/* ---------------------------------------------------------------------------------------------------------------
 * Streaming for C hosts: a stream group (several live streams, e.g. cameras, each frame attending to its stream's frame 0
 * and the frames before it) behind a host planner and one device call per push.  The same schedule and the same table
 * encoding as the Python DepthStreamGroup (video_depth_anything_b200/video_depth.py, windows.StreamGroupPlan,
 * engine.py Engine.stream_group_step), bit-identical output.  L = num_frames - 1 (31) context frames per stream.
 *
 * Planner (host only, touches no GPU):
 *   vda_stream_plan_create   max_streams >= 1 streams open at once; max_frames frames per push (<= 0: max(max_streams, 16),
 *                            else >= max_streams); num_frames as given to vda_create (2..32); input_size as for
 *                            infer_video_depth (518).
 *   vda_stream_plan_buckets  the batch sizes the group runs at: powers of two below max_streams, max_streams, then powers
 *                            of two below max_frames, max_frames.  *n = their count; up to `capacity` are written to out.
 *   vda_stream_plan_open     a new stream at t = 0.  Handles are never reused; its pool row is the lowest free one.
 *   vda_stream_plan_close    frees the stream's pool row (a later open starts over on it, with a new frame size).
 *   vda_stream_plan_step     one push of n distinct open streams in batch-row order: handles[i] gives counts[i] (1..L;
 *                            counts NULL: 1 each) consecutive frames of size sizes[2i] x sizes[2i+1] (H0, W0; NULL: not
 *                            checked), at most max_frames frames in all.  A stream's frame size is fixed by its first
 *                            frame, the group's network size (vda_resize_hw) by its first push.  Writes the table of
 *                            the push (bucket bk = the smallest bucket >= the frame count; table_capacity >= bk * (L + 4)
 *                            int32):  rows [bk] | ctx [bk, L + 2] | idx [bk]: batch row i is a frame of stream handles[s]
 *                            at step t with its pool row, ctx = {n_ctx, write slot, context entries...} (a context frame
 *                            of this push is entered as -1 - its batch row, an older one as its cache slot), idx = i; pad
 *                            rows take pool row -1, n_ctx 0.  *nh, *nw = the group's network size (0 if no push gave
 *                            sizes yet).  Advances the streams.  A rejected push changes nothing.
 *   vda_resize_hw            network input size of an (h0, w0) frame (video_depth.py:167-171, util/transform.py:62-107).
 *
 * Device step:
 *   vda_stream_pool_bytes       bytes of the temporal cache of S streams at network size (nh, nw): 8 blocks, block
 *                               2 * m + a (attention block a of motion module m) h16 (fp16) [S, num_frames, hw_m, 2 C_m]
 *                               with hw = (nh / 14) (nw / 14), hw_m = {hw, ceil(nh / 28) ceil(nw / 28), hw, 4 hw}, C_m =
 *                               {out_channels[2], out_channels[3], features, features}, one after the other (each a multiple
 *                               of 256 bytes).  The pool is the caller's, 256-byte aligned; its content needs no
 *                               initialisation (a stream reads only slots it wrote).  -1 on error.
 *   vda_stream_workspace_bytes  scratch of one step of B batch rows (-1 on error).
 *   vda_stream_step             one push: batch row b < B (= the bucket) reads frames[b] (uint8 RGB, any size) and writes
 *                               its depth fp32 [H0, W0] >= 0 to outs[b] (pad rows: any valid frame, H0 = W0 = 0 writes
 *                               nothing); table = the planner's table of the push.  frames, outs, table, pool and
 *                               workspace (1024-byte aligned, >= vda_stream_workspace_bytes) are device memory.  causal != 0
 *                               when the push gives some stream more than one frame (8 more launches: each temporal
 *                               attention then reads the push's own rows and writes the pool afterwards); 0 otherwise.
 *                               Enqueues on `stream`; no allocation and no synchronisation, and every per-push value is in
 *                               the descriptors and the table, so one CUDA graph per (bucket, causal) replays every later
 *                               push.  The first step at a new network size resamples the position embedding into
 *                               model-owned memory: run it outside a capture.  Everything is checked before anything is
 *                               launched; pool rows inside the table are the kernels' business (outside 0..S-1: a pad row).
 */
typedef struct vda_stream_plan vda_stream_plan;
int vda_stream_plan_create(int max_streams, int max_frames, int num_frames, int input_size, vda_stream_plan** out);
int vda_stream_plan_buckets(const vda_stream_plan* p, int32_t* out, int capacity, int* n);
int vda_stream_plan_open(vda_stream_plan* p, int64_t* handle);
int vda_stream_plan_close(vda_stream_plan* p, int64_t handle);
int vda_stream_plan_step(vda_stream_plan* p, const int64_t* handles, const int32_t* sizes, const int32_t* counts, int n,
                         int32_t* table, int64_t table_capacity, int* bucket, int* nh, int* nw);
int vda_stream_plan_destroy(vda_stream_plan* p);
int vda_resize_hw(int h0, int w0, int input_size, int* nh, int* nw);
int64_t vda_stream_pool_bytes(vda_model* m, int S, int nh, int nw);
int64_t vda_stream_workspace_bytes(vda_model* m, int B, int nh, int nw);
int vda_stream_step(vda_model* m, const vda_frame_desc* frames, const vda_out_desc* outs, const int32_t* table, int B,
                    int causal, void* pool, int S, int nh, int nw, void* workspace, int64_t workspace_bytes, void* stream);
/* vda_stream_step for YUV 4:2:0 frames (NV12 / I420 decoder output, see vda_frame_planes): batch row b reads frames[b]
 * through vda_preprocess_frames_planes instead of vda_preprocess_frames_ragged; everything else -- workspace size, pool,
 * table, capture rule, launch count -- is vda_stream_step's, and the depths are bit-identical to vda_stream_step on the
 * cv2-converted RGB frames.  Pad rows: any valid frame (e.g. row 0's descriptor). */
int vda_stream_step_planes(vda_model* m, const vda_frame_planes* frames, const vda_out_desc* outs, const int32_t* table,
                           int B, int causal, void* pool, int S, int nh, int nw, void* workspace, int64_t workspace_bytes,
                           void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Depth frames for displays and encoders: what save_video (utils/dc_utils.py:72-86) does on the host after
 * infer_video_depth -- normalise by a range, look up a colour table, hand uint8 frames to a writer -- on the device,
 * with YUV 4:2:0 output for encoders (NVENC takes NV12).  The codec itself is not part of libvda.
 *
 * Contract, for one depth d (fp32, finite) and a range (lo, hi):
 *   level   q = min(255, max(0, trunc(((d - lo) / (hi - lo)) * 255))), every operation IEEE fp32 round-to-nearest in
 *           this order: the reference's ((depth - d_min) / (d_max - d_min) * 255).astype(np.uint8) on float32 arrays for
 *           every d in [lo, hi]; the clamp matters only for a fixed range.  hi <= lo: q = 0 everywhere (a constant video).
 *   colour  (R, G, B) = table[q], table uint8 [256][3] (OpenCV's inferno, or the caller's own, e.g. matplotlib's).
 *   formats VDA_PIX_RGB   packed [H0][W0][3] at plane[0], rows pitch[0] >= 3 W0 bytes apart;
 *           VDA_PIX_GRAY  q itself, [H0][W0] at plane[0] (save_video(grayscale=True)); no table needed;
 *           VDA_PIX_NV12 / VDA_PIX_I420: cv2.cvtColor(COLOR_RGB2YUV_I420) of the RGB frame (BT.601 limited range), with
 *           the chroma of each 2 x 2 block taken from its top-left pixel, in this integer form (equal to cv2 4.13 on all
 *           2^24 triples):
 *             Y = (269484 R + 528482 G + 102760 B + (16 << 20) + (1 << 19)) >> 20
 *             U = (-155188 R - 305135 G + 460324 B + (128 << 20) + (1 << 19)) >> 20
 *             V = (460324 R - 385875 G - 74448 B + (128 << 20) + (1 << 19)) >> 20
 *           planes as vda_frame_planes (NV12: Y, interleaved UV; I420: Y, U, V); H0, W0 even.  Every plane has its own
 *           pitch, so an encoder surface with its UV plane at Y + pitch * aligned height is written in place.
 */
enum { VDA_PIX_RGB = 0, VDA_PIX_GRAY = 3 };

/* An output frame of vda_colorize_depth: vda_frame_planes with writable planes (64 bytes).  H0 == 0 (a pad row) writes
 * nothing; otherwise H0 x W0 equals the size of the row's depth descriptor, format is a VDA_PIX_*, reserved 0. */
typedef struct vda_color_planes {
  uint8_t* plane[3];
  int64_t pitch[3];
  int32_t H0, W0, format, reserved;
} vda_color_planes;

/* The range of the depths (save_video's frames.min(), frames.max()): rows are depth frames fp32 [H0][W0] (vda_out_desc,
 * the descriptors vda_stream_step writes through; H0 == 0 is an empty row), in device memory.  all_rows == 0: range
 * fp32 [n][2] = (min, max) of each row ("frame" range; an empty row gives (+inf, -inf)); all_rows != 0: range fp32 [2]
 * over every row ("video" range).  min and max are exact, so the result does not depend on the order.  scratch: device,
 * 8-byte aligned, >= vda_depth_range_scratch_bytes(n) = n * VDA_RANGE_PARTIALS * 8 bytes.  Two launches; no allocation
 * and no synchronisation (graph-capturable).  A range over several calls: the all-rows range of a [k][2] array of ranges
 * (one row of H0 = k, W0 = 2) is their combined range, since every lo <= its hi. */
#define VDA_RANGE_PARTIALS 128
int64_t vda_depth_range_scratch_bytes(int n);
int vda_depth_range(const vda_out_desc* rows, int n, int all_rows, float* range, void* scratch, void* stream);

/* Colour-map depth frames (dc_utils.py:72-86, the frame loop of save_video): row i reads the depths of src[i] and writes
 * its frame described by dst[i] (both descriptor arrays in device memory, read by the kernel) with the range
 * range[2i..2i+1] (range_per_row != 0) or range[0..1] (a shared range), fp32 device memory, e.g. from vda_depth_range.
 * table: device uint8 [256][3]; may be NULL only when every row is VDA_PIX_GRAY.  One launch, a thread per 2 x 2 pixel
 * block; reads 4 bytes and writes 1 (grey), 1.5 (YUV) or 3 (RGB) bytes per pixel.  The descriptors are not checked by
 * the launcher (the Python mirror checks what it writes: windows.color_descriptors). */
int vda_colorize_depth(const vda_out_desc* src, const vda_color_planes* dst, int n, const float* range, int range_per_row,
                       const uint8_t* table, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VDA_H_ */
