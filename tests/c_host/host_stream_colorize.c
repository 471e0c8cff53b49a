/* A C host of libvda's streaming API that feeds an encoder (include/vda.h: vda_stream_step_planes, vda_depth_range,
 * vda_colorize_depth): S live streams of NV12 video in, NV12 depth frames out -- each push's depths colour-mapped with
 * OpenCV's inferno table over each frame's own range and written, inside the push's captured graph, into pitched
 * encoder-style input surfaces: Y rows `pitch` bytes apart (W0 rounded up to 256), the UV plane at Y + pitch * aligned
 * height (H0 rounded up to 16), as NVENC takes them.  Input surfaces, planner, graphs and push protocol are
 * host_stream_nv12.c's.  tests/test_colorize_gpu.py builds it with gcc and requires its frames to be bit-identical to the
 * Python DepthStreamGroup's (pixel_format="nv12", output_format="nv12") on the same pushes.
 *
 *   host_stream_colorize <encoder> <features> <oc0> <oc1> <oc2> <oc3> <dtype> <weights.bin> <input.bin> <output.bin>
 *   <table.bin>
 *
 * weights.bin, input.bin: as for host_stream_nv12.c
 * table.bin:   uint8 [256][3], the RGB colour table
 * output.bin:  per push, per item: uint8 frame[count][3 H0 / 2][W0] (NV12 in OpenCV's packed layout)
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "vda.h"

#define DIE(...) do { fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); return 1; } while (0)
#define VDA(call) do { if ((call) != 0) DIE("%s failed: %s", #call, vda_last_error()); } while (0)
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) DIE("%s: %s", #call, cudaGetErrorString(e_)); } while (0)

#define MAX_STREAMS 64
#define MAX_BUCKETS 64

typedef struct { int32_t n, h, w; uint8_t* px; int next; } video;

/* the surface geometry of a decoder: pitch and aligned height of an H0 x W0 frame */
static size_t surf_pitch(int w) { return ((size_t)w + 255) / 256 * 256; }
static size_t surf_rows(int h) { return ((size_t)h + 31) / 32 * 32; }
static size_t surf_bytes(int h, int w) { return surf_pitch(w) * (surf_rows(h) + (size_t)h / 2); }
/* an encoder's input surface: UV at the height aligned to 16 */
static size_t enc_rows(int h) { return ((size_t)h + 15) / 16 * 16; }
static size_t enc_bytes(int h, int w) { return surf_pitch(w) * (enc_rows(h) + (size_t)h / 2); }

static int load_weights(vda_model* m, const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) DIE("cannot open %s", path);
  int32_t count = 0;
  if (fread(&count, 4, 1, f) != 1) DIE("bad weights file");
  for (int i = 0; i < count; ++i) {
    int32_t nl = 0, nd = 0;
    char name[512];
    int64_t shape[8];
    if (fread(&nl, 4, 1, f) != 1 || nl <= 0 || nl >= 512 || fread(name, 1, (size_t)nl, f) != (size_t)nl) DIE("bad tensor name");
    name[nl] = 0;
    if (fread(&nd, 4, 1, f) != 1 || nd < 0 || nd > 8 || fread(shape, 8, (size_t)nd, f) != (size_t)nd) DIE("bad tensor shape");
    size_t n = 1;
    for (int d = 0; d < nd; ++d) n *= (size_t)shape[d];
    float* data = (float*)malloc(n * 4 + 4);
    if (!data || fread(data, 4, n, f) != n) DIE("bad tensor data (%s)", name);
    VDA(vda_set_weight(m, name, data, shape, nd));
    free(data);
  }
  fclose(f);
  return 0;
}

int main(int argc, char** argv) {
  if (argc == 2 && strcmp(argv[1], "--version") == 0) {   /* link check without a GPU */
    printf("%d\n", vda_version());
    return 0;
  }
  if (argc != 12) DIE("usage: %s encoder features oc0 oc1 oc2 oc3 dtype weights.bin input.bin output.bin table.bin", argv[0]);
  const int num_frames = 32, L = num_frames - 1;
  const int32_t oc[4] = {atoi(argv[3]), atoi(argv[4]), atoi(argv[5]), atoi(argv[6])};
  vda_model* m = NULL;
  VDA(vda_create(argv[1], atoi(argv[2]), oc, num_frames, atoi(argv[7]), 0, &m));
  if (load_weights(m, argv[8])) return 1;
  VDA(vda_finalize_weights(m));

  /* the videos and the push sequence */
  FILE* f = fopen(argv[9], "rb");
  if (!f) DIE("cannot open %s", argv[9]);
  int32_t hdr[3];
  if (fread(hdr, 4, 3, f) != 3) DIE("bad input file");
  const int S = hdr[0], input_size = hdr[1], n_pushes = hdr[2];
  if (S < 1 || S > MAX_STREAMS) DIE("bad stream count %d", S);
  video v[MAX_STREAMS];
  size_t max_frame = 0, max_surf = 0;
  for (int s = 0; s < S; ++s) {
    int32_t d[3];
    if (fread(d, 4, 3, f) != 3) DIE("bad video header");
    v[s].n = d[0]; v[s].h = d[1]; v[s].w = d[2]; v[s].next = 0;
    if (d[1] % 2 || d[2] % 2) DIE("an NV12 frame has an even size, got %d x %d", d[1], d[2]);
    const size_t bytes = (size_t)d[0] * d[1] * d[2] * 3 / 2;
    v[s].px = (uint8_t*)malloc(bytes + 1);
    if (!v[s].px || fread(v[s].px, 1, bytes, f) != bytes) DIE("bad video data");
    if ((size_t)d[1] * d[2] > max_frame) max_frame = (size_t)d[1] * d[2];
    if (surf_bytes(d[1], d[2]) > max_surf) max_surf = surf_bytes(d[1], d[2]);
  }
  uint8_t table_h[768];
  FILE* ft = fopen(argv[11], "rb");
  if (!ft || fread(table_h, 1, 768, ft) != 768) DIE("bad colour table %s", argv[11]);
  fclose(ft);
  FILE* fo = fopen(argv[10], "wb");
  if (!fo) DIE("cannot open %s", argv[10]);

  /* planner: S streams, buckets up to max(S, 16) frames per push */
  vda_stream_plan* plan = NULL;
  VDA(vda_stream_plan_create(S, 0, num_frames, input_size, &plan));
  int64_t handle[MAX_STREAMS];
  for (int s = 0; s < S; ++s) VDA(vda_stream_plan_open(plan, &handle[s]));
  int32_t buckets[MAX_BUCKETS];
  int nb = 0;
  VDA(vda_stream_plan_buckets(plan, buckets, MAX_BUCKETS, &nb));
  if (nb > MAX_BUCKETS) DIE("too many buckets");
  const int BK = buckets[nb - 1];

  /* per-push metadata block: frame descriptors [bk] | output descriptors [bk] | int32 table [bk * (L + 4)] | colour
   * descriptors [bk] (64-byte aligned) */
  const size_t meta_bytes = (size_t)BK * (sizeof(vda_frame_planes) + sizeof(vda_out_desc) + 4 * (L + 4)) + 64 +
                            (size_t)BK * sizeof(vda_color_planes);
  uint8_t *meta_h = NULL, *meta_d = NULL, *in_d = NULL, *enc_d = NULL, *lut_d = NULL;
  float *out_d = NULL, *range_d = NULL;
  void* range_scratch = NULL;
  CU(cudaMallocHost((void**)&meta_h, meta_bytes));
  CU(cudaMalloc((void**)&meta_d, meta_bytes));
  CU(cudaMalloc((void**)&in_d, (size_t)BK * max_surf));       /* one decoder surface per batch row */
  CU(cudaMalloc((void**)&out_d, (size_t)BK * max_frame * 4)); /* the depths: an arena, never read by the host */
  CU(cudaMalloc((void**)&enc_d, (size_t)BK * max_surf));      /* one encoder surface per batch row (enc_bytes <= surf_bytes) */
  CU(cudaMalloc((void**)&lut_d, 768));
  CU(cudaMalloc((void**)&range_d, (size_t)BK * 2 * sizeof(float)));
  CU(cudaMalloc(&range_scratch, (size_t)vda_depth_range_scratch_bytes(BK)));
  CU(cudaMemcpy(lut_d, table_h, 768, cudaMemcpyHostToDevice));
  uint8_t* out_h = (uint8_t*)malloc((size_t)BK * max_frame * 3 / 2);
  void *pool = NULL, *ws = NULL;
  int64_t ws_bytes = 0;
  int nh = 0, nw = 0;
  cudaStream_t st;
  CU(cudaStreamCreate(&st));
  cudaGraphExec_t graph[MAX_BUCKETS][2];
  memset(graph, 0, sizeof(graph));

  for (int p = 0; p < n_pushes; ++p) {
    int32_t n = 0;
    if (fread(&n, 4, 1, f) != 1 || n < 1 || n > S) DIE("bad push %d", p);
    int32_t item[2 * MAX_STREAMS], sizes[2 * MAX_STREAMS], counts[MAX_STREAMS];
    int64_t hs[MAX_STREAMS];
    if (fread(item, 4, (size_t)2 * n, f) != (size_t)2 * n) DIE("bad push %d", p);
    int causal = 0;
    for (int i = 0; i < n; ++i) {
      const int s = item[2 * i];
      if (s < 0 || s >= S || v[s].next + item[2 * i + 1] > v[s].n) DIE("push %d: stream %d has no such frames", p, s);
      hs[i] = handle[s];
      sizes[2 * i] = v[s].h;
      sizes[2 * i + 1] = v[s].w;
      counts[i] = item[2 * i + 1];
      causal |= counts[i] > 1;
    }
    int bk = 0;
    int32_t* table = (int32_t*)(meta_h + (size_t)BK * (sizeof(vda_frame_planes) + sizeof(vda_out_desc)));
    VDA(vda_stream_plan_step(plan, hs, sizes, counts, n, table, (int64_t)BK * (L + 4), &bk, &nh, &nw));
    if (!pool) {                                      /* the group's network size is known from its first push */
      const int64_t pool_bytes = vda_stream_pool_bytes(m, S, nh, nw);
      ws_bytes = vda_stream_workspace_bytes(m, BK, nh, nw);
      if (pool_bytes < 0 || ws_bytes < 0) DIE("sizes: %s", vda_last_error());
      CU(cudaMalloc(&pool, (size_t)pool_bytes));
      CU(cudaMalloc(&ws, (size_t)ws_bytes));
    }
    /* this bucket's layout of the block: the descriptors first, then the table (moved behind them) */
    vda_frame_planes* fd = (vda_frame_planes*)meta_h;
    vda_out_desc* od = (vda_out_desc*)(meta_h + (size_t)bk * sizeof(vda_frame_planes));
    const size_t table_off = (size_t)bk * (sizeof(vda_frame_planes) + sizeof(vda_out_desc));
    memmove(meta_h + table_off, table, (size_t)bk * (L + 4) * 4);
    const size_t color_off = (table_off + (size_t)bk * (L + 4) * 4 + 63) / 64 * 64;
    vda_color_planes* cd = (vda_color_planes*)(meta_h + color_off);
    size_t in_off = 0, out_off = 0, enc_off = 0;
    int row = 0;
    for (int i = 0; i < n; ++i) {
      video* vs = &v[item[2 * i]];
      const size_t fb = (size_t)vs->h * vs->w * 3 / 2, pitch = surf_pitch(vs->w);
      for (int j = 0; j < counts[i]; ++j, ++row) {
        /* the frame into a decoder-style surface: Y rows, then the UV rows at the aligned height */
        const uint8_t* y = vs->px + (size_t)(vs->next + j) * fb;
        uint8_t* sy = in_d + in_off;
        uint8_t* suv = sy + pitch * surf_rows(vs->h);
        CU(cudaMemcpy2DAsync(sy, pitch, y, (size_t)vs->w, (size_t)vs->w, (size_t)vs->h, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpy2DAsync(suv, pitch, y + (size_t)vs->h * vs->w, (size_t)vs->w, (size_t)vs->w, (size_t)vs->h / 2,
                             cudaMemcpyHostToDevice, st));
        fd[row].plane[0] = sy;
        fd[row].plane[1] = suv;
        fd[row].plane[2] = NULL;
        fd[row].pitch[0] = fd[row].pitch[1] = (int64_t)pitch;
        fd[row].pitch[2] = 0;
        fd[row].H0 = vs->h;
        fd[row].W0 = vs->w;
        fd[row].format = VDA_PIX_NV12;
        fd[row].reserved = 0;
        od[row].dst = out_d + out_off;
        od[row].H0 = vs->h;
        od[row].W0 = vs->w;
        memset(&cd[row], 0, sizeof(cd[row]));
        cd[row].plane[0] = enc_d + enc_off;
        cd[row].plane[1] = enc_d + enc_off + pitch * enc_rows(vs->h);
        cd[row].pitch[0] = cd[row].pitch[1] = (int64_t)pitch;
        cd[row].H0 = vs->h;
        cd[row].W0 = vs->w;
        cd[row].format = VDA_PIX_NV12;
        enc_off += enc_bytes(vs->h, vs->w);
        in_off += surf_bytes(vs->h, vs->w);
        out_off += (size_t)vs->h * vs->w;
      }
    }
    for (; row < bk; ++row) {                         /* pad rows: read the first frame, write nothing */
      fd[row] = fd[0];
      od[row].dst = NULL;
      od[row].H0 = od[row].W0 = 0;
      memset(&cd[row], 0, sizeof(cd[row]));             /* H0 = 0: nothing written */
    }
    const size_t meta_used = color_off + (size_t)bk * sizeof(vda_color_planes);
    CU(cudaMemcpyAsync(meta_d, meta_h, meta_used, cudaMemcpyHostToDevice, st));
    const vda_frame_planes* fdd = (const vda_frame_planes*)meta_d;
    const vda_out_desc* odd = (const vda_out_desc*)(meta_d + (size_t)bk * sizeof(vda_frame_planes));
    const int32_t* td = (const int32_t*)(meta_d + table_off);
    const vda_color_planes* cdd = (const vda_color_planes*)(meta_d + color_off);
    int bi = 0;
    while (buckets[bi] != bk) ++bi;
    if (!graph[bi][causal]) {
      /* A step writes the pool, so the warm-up and the capture run with every row a pad row (pool row -1), then the push's
       * own table is uploaded again.  The warm-up is outside the capture: the first step at a network size resamples the
       * position embedding into model-owned memory. */
      CU(cudaMemsetAsync(meta_d + table_off, 0xff, (size_t)bk * 4, st));
      VDA(vda_stream_step_planes(m, fdd, odd, td, bk, causal, pool, S, nh, nw, ws, ws_bytes, st));
      VDA(vda_depth_range(odd, bk, 0, range_d, range_scratch, st));
      VDA(vda_colorize_depth(odd, cdd, bk, range_d, 1, lut_d, st));
      CU(cudaStreamSynchronize(st));
      cudaGraph_t g;
      CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      VDA(vda_stream_step_planes(m, fdd, odd, td, bk, causal, pool, S, nh, nw, ws, ws_bytes, st));
      VDA(vda_depth_range(odd, bk, 0, range_d, range_scratch, st));     /* each frame's own (min, max) */
      VDA(vda_colorize_depth(odd, cdd, bk, range_d, 1, lut_d, st));     /* into the encoder surfaces */
      CU(cudaStreamEndCapture(st, &g));
      CU(cudaGraphInstantiate(&graph[bi][causal], g, 0));
      CU(cudaGraphDestroy(g));
      CU(cudaMemcpyAsync(meta_d, meta_h, meta_used, cudaMemcpyHostToDevice, st));
    }
    CU(cudaGraphLaunch(graph[bi][causal], st));
    /* what an encoder would read: here each surface is copied back packed, Y rows then UV rows */
    size_t packed = 0;
    for (int r = 0; r < row && cd[r].H0; ++r) {
      const size_t h = (size_t)cd[r].H0, w = (size_t)cd[r].W0, pitch = (size_t)cd[r].pitch[0];
      CU(cudaMemcpy2DAsync(out_h + packed, w, cd[r].plane[0], pitch, w, h, cudaMemcpyDeviceToHost, st));
      CU(cudaMemcpy2DAsync(out_h + packed + h * w, w, cd[r].plane[1], pitch, w, h / 2, cudaMemcpyDeviceToHost, st));
      packed += h * w * 3 / 2;
    }
    CU(cudaStreamSynchronize(st));
    if (fwrite(out_h, 1, packed, fo) != packed) DIE("cannot write %s", argv[10]);
    for (int i = 0; i < n; ++i) v[item[2 * i]].next += counts[i];
  }
  fclose(f);
  fclose(fo);
  int graphs = 0;
  for (int b = 0; b < nb; ++b)
    for (int c = 0; c < 2; ++c)
      if (graph[b][c]) { ++graphs; cudaGraphExecDestroy(graph[b][c]); }
  printf("ok %d NV12 streams colour-mapped into NV12 surfaces, %d pushes at %d x %d, %d graphs\n", S, n_pushes, nh, nw, graphs);
  for (int s = 0; s < S; ++s) free(v[s].px);
  free(out_h);
  cudaFree(pool); cudaFree(ws); cudaFree(in_d); cudaFree(out_d); cudaFree(meta_d); cudaFreeHost(meta_h);
  cudaFree(enc_d); cudaFree(lut_d); cudaFree(range_d); cudaFree(range_scratch);
  cudaStreamDestroy(st);
  vda_stream_plan_destroy(plan);
  return vda_destroy(m);
}
