// Host planner of a stream group for C hosts: handles, pool rows, per-stream steps, buckets and the per-push context
// table (include/vda.h vda_stream_plan_*).  A line-for-line port of video_depth_anything_b200/windows.py
// (stream_buckets, stream_context, StreamGroupPlan, get_resize_hw); tests/test_c_stream_cpu.py drives both through the
// same random operations and requires the same decisions and the same table bytes.  Pure host code: nothing here
// touches the GPU.
#include <math.h>

#include <map>
#include <set>
#include <utility>
#include <vector>

#include "../../include/vda.h"
#include "common.cuh"

struct vda_stream_plan {
  int max_streams = 0, max_frames = 0, L = 0, input_size = 0;
  std::vector<int> buckets;
  std::map<int64_t, int> row, t;                       // handle -> pool row, handle -> frames pushed so far
  std::map<int64_t, std::pair<int, int>> size;         // handle -> (H0, W0) of its first frame
  bool has_net = false;                                // the group's network size, fixed by the first push with sizes
  int net_h = 0, net_w = 0;
  int64_t next = 0;
};

namespace vda {

// windows._constrain: np.round is round-half-to-even, as rint in the default rounding mode
static int constrain(double x, int min_val) {
  int y = static_cast<int>(rint(x / 14) * 14);
  if (y < min_val) y = static_cast<int>(ceil(x / 14) * 14);
  return y;
}

static void resize_hw(int h0, int w0, int input_size, int* nh, int* nw) {
  const double ratio = static_cast<double>(h0 > w0 ? h0 : w0) / static_cast<double>(h0 > w0 ? w0 : h0);
  if (ratio > 1.78) {
    input_size = static_cast<int>(input_size * 1.777 / ratio);
    input_size = static_cast<int>(rint(input_size / 14.0)) * 14;     // Python round(): half to even
  }
  double scale_h = input_size / static_cast<double>(h0), scale_w = input_size / static_cast<double>(w0);
  if (scale_w > scale_h) scale_h = scale_w;
  else scale_w = scale_h;
  *nh = constrain(scale_h * h0, input_size);
  *nw = constrain(scale_w * w0, input_size);
}

static int slot_of(int j, int L) { return j == 0 ? 0 : 1 + (j - 1) % L; }

}  // namespace vda

using namespace vda;

extern "C" int vda_resize_hw(int h0, int w0, int input_size, int* nh, int* nw) {
  VDA_CHECK(nh && nw, "vda_resize_hw: null pointer");
  VDA_CHECK(h0 >= 1 && w0 >= 1, "vda_resize_hw: empty frame of size (%d, %d)", h0, w0);
  VDA_CHECK(input_size >= 1, "vda_resize_hw: input_size must be >= 1, got %d", input_size);
  resize_hw(h0, w0, input_size, nh, nw);
  return 0;
}

extern "C" int vda_stream_plan_create(int max_streams, int max_frames, int num_frames, int input_size, vda_stream_plan** out) {
  VDA_CHECK(out, "vda_stream_plan_create: null pointer");
  VDA_CHECK(max_streams >= 1, "a stream group needs max_streams >= 1, got %d", max_streams);
  VDA_CHECK(num_frames >= 2 && num_frames <= 32, "streaming needs num_frames in 2..32, got %d", num_frames);
  VDA_CHECK(input_size >= 1, "vda_stream_plan_create: input_size must be >= 1, got %d", input_size);
  if (max_frames <= 0) max_frames = max_streams > 16 ? max_streams : 16;
  VDA_CHECK(max_frames >= max_streams, "max_frames=%d is below max_streams=%d", max_frames, max_streams);
  vda_stream_plan* p = new vda_stream_plan();
  p->max_streams = max_streams;
  p->max_frames = max_frames;
  p->L = num_frames - 1;
  p->input_size = input_size;
  // windows.stream_buckets: powers of two below max_streams, max_streams, then powers of two below max_frames, max_frames
  for (int64_t b = 1; b < max_streams; b <<= 1) p->buckets.push_back(static_cast<int>(b));
  p->buckets.push_back(max_streams);
  if (max_frames != max_streams) {
    for (int64_t b = 1; b < max_frames; b <<= 1)
      if (b > max_streams) p->buckets.push_back(static_cast<int>(b));
    p->buckets.push_back(max_frames);
  }
  *out = p;
  return 0;
}

extern "C" int vda_stream_plan_buckets(const vda_stream_plan* p, int32_t* out, int capacity, int* n) {
  VDA_CHECK(p && n, "vda_stream_plan_buckets: null pointer");
  *n = static_cast<int>(p->buckets.size());
  for (int i = 0; i < *n && i < capacity && out; ++i) out[i] = p->buckets[static_cast<size_t>(i)];
  return 0;
}

extern "C" int vda_stream_plan_open(vda_stream_plan* p, int64_t* handle) {
  VDA_CHECK(p && handle, "vda_stream_plan_open: null pointer");
  VDA_CHECK(static_cast<int>(p->row.size()) < p->max_streams, "the group already holds its max_streams=%d streams",
            p->max_streams);
  std::set<int> used;
  for (const auto& kv : p->row) used.insert(kv.second);
  int r = 0;
  while (used.count(r)) ++r;                           // the lowest free pool row
  const int64_t h = p->next++;
  p->row[h] = r;
  p->t[h] = 0;
  *handle = h;
  return 0;
}

extern "C" int vda_stream_plan_close(vda_stream_plan* p, int64_t handle) {
  VDA_CHECK(p, "vda_stream_plan_close: null pointer");
  VDA_CHECK(p->row.count(handle), "unknown or closed stream handle %lld", static_cast<long long>(handle));
  p->row.erase(handle);
  p->t.erase(handle);
  p->size.erase(handle);
  return 0;
}

extern "C" int vda_stream_plan_step(vda_stream_plan* p, const int64_t* handles, const int32_t* sizes, const int32_t* counts, int n,
                                    int32_t* table, int64_t table_capacity, int* bucket, int* nh, int* nw) {
  VDA_CHECK(p && table && bucket && nh && nw && (handles || n <= 0), "vda_stream_plan_step: null pointer");
  // every check before any state changes: a rejected push leaves the plan as it was (StreamGroupPlan.step)
  for (int i = 0; i < n; ++i)
    VDA_CHECK(p->row.count(handles[i]), "unknown or closed stream handle %lld", static_cast<long long>(handles[i]));
  VDA_CHECK(std::set<int64_t>(handles, handles + (n > 0 ? n : 0)).size() == static_cast<size_t>(n > 0 ? n : 0),
            "a stream is named more than once in one push");
  VDA_CHECK(n > 0, "a push names at least one stream");
  int total = 0;
  for (int i = 0; i < n; ++i) {
    const int c = counts ? counts[i] : 1;
    VDA_CHECK(c >= 1 && c <= p->L, "stream %lld: %d frames in one push; a push gives a stream 1..%d frames",
              static_cast<long long>(handles[i]), c, p->L);
    total += c;
  }
  VDA_CHECK(total <= p->max_frames, "%d frames in one push, more than the group's max_frames=%d", total, p->max_frames);
  bool has_net = p->has_net;
  int net_h = p->net_h, net_w = p->net_w;
  if (sizes) {
    for (int i = 0; i < n; ++i) {
      const int h0 = sizes[2 * i], w0 = sizes[2 * i + 1];
      VDA_CHECK(h0 >= 1 && w0 >= 1, "empty frame of size (%d, %d)", h0, w0);
      auto it = p->size.find(handles[i]);
      VDA_CHECK(it == p->size.end() || it->second == std::make_pair(h0, w0),
                "frame size (%d, %d) of stream %lld differs from its first frame's (%d, %d)", h0, w0,
                static_cast<long long>(handles[i]), it == p->size.end() ? 0 : it->second.first,
                it == p->size.end() ? 0 : it->second.second);
      int a = 0, b = 0;
      resize_hw(h0, w0, p->input_size, &a, &b);
      if (!has_net) {
        has_net = true;
        net_h = a;
        net_w = b;
      } else {
        VDA_CHECK(a == net_h && b == net_w,
                  "frame size (%d, %d) maps to network size (%d, %d), %s (%d, %d); streams of other network sizes need a "
                  "group of their own", h0, w0, a, b, p->has_net ? "the group's" : "that of another frame of this push,",
                  net_h, net_w);
      }
    }
  }
  int bk = 0;
  for (int b : p->buckets)
    if (b >= total) { bk = b; break; }
  const int L = p->L, stride = 2 + L;
  VDA_CHECK(table_capacity >= static_cast<int64_t>(bk) * (L + 4), "vda_stream_plan_step: the table holds %lld int32, a push "
            "at bucket %d needs %lld", static_cast<long long>(table_capacity), bk, static_cast<long long>(bk) * (L + 4));

  if (sizes) {
    p->has_net = has_net;
    p->net_h = net_h;
    p->net_w = net_w;
    for (int i = 0; i < n; ++i) p->size[handles[i]] = std::make_pair(sizes[2 * i], sizes[2 * i + 1]);
  }
  int32_t* rows = table;
  int32_t* ctx = table + bk;
  int32_t* idx = table + bk + static_cast<int64_t>(bk) * stride;
  for (int i = 0; i < bk; ++i) rows[i] = -1, idx[i] = 0;
  for (int64_t i = 0; i < static_cast<int64_t>(bk) * stride; ++i) ctx[i] = 0;
  int i = 0;
  for (int s = 0; s < n; ++s) {
    const int c = counts ? counts[s] : 1, t0 = p->t[handles[s]];
    for (int j = 0; j < c; ++j, ++i) {
      const int t = t0 + j;                            // windows.stream_context(t, L): [0] + [max(1, t - L + 1) .. t - 1]
      int32_t* e = ctx + static_cast<int64_t>(i) * stride;
      rows[i] = p->row[handles[s]];
      idx[i] = i;
      e[1] = slot_of(t, L);
      int k = 0;
      if (t > 0) {
        std::vector<int> ids(1, 0);
        for (int f = (t - L + 1 > 1 ? t - L + 1 : 1); f < t; ++f) ids.push_back(f);
        // frames of this push (ids >= t0) sit f - t0 rows behind the stream's first row i - j
        for (int f : ids) e[2 + k++] = f >= t0 ? -1 - (i - j + f - t0) : slot_of(f, L);
      }
      e[0] = k;
    }
  }
  for (int s = 0; s < n; ++s) p->t[handles[s]] += counts ? counts[s] : 1;
  *bucket = bk;
  *nh = p->net_h;
  *nw = p->net_w;
  return 0;
}

extern "C" int vda_stream_plan_destroy(vda_stream_plan* p) {
  delete p;
  return 0;
}
