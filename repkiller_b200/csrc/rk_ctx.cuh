// The context behind the C ABI (include/rk_b200.h), shared by capi.cu (single GPU) and multi.cu (one comparison over
// several GPUs): device workspace, pinned result buffers, per-kernel event profiler, error plumbing.
#pragma once

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/rk_b200.h"
#include "rk_common.cuh"

namespace rk {

inline u64 align_up(u64 x, u64 a) { return (x + a - 1) / a * a; }
inline int ceil_log2(u64 x) {  // bits needed to represent values 0 .. x-1
  int b = 0;
  while (b < 63 && (1ull << b) < x) ++b;
  return b;
}

// CUDA-event pair around every launch group; folded into per-kernel totals after each synchronisation
struct Profiler {
  bool on = false;
  struct Rec { int kid; cudaEvent_t a, b; u64 units; };
  std::vector<Rec> open_recs;
  std::vector<cudaEvent_t> pool;
  double ms[KID_COUNT] = {0};
  u64 launches[KID_COUNT] = {0};
  u64 units[KID_COUNT] = {0};
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
  }
  void fold() {  // call after the stream was synchronised
    for (auto &r : open_recs) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.kid] += t; launches[r.kid] += 1; units[r.kid] += r.units; }
      else cudaGetLastError();
      pool.push_back(r.a);
      pool.push_back(r.b);
    }
    open_recs.clear();
  }
};
void prof_route(Profiler *p);  // routes the launchers' KScope events of this thread to p (nullptr: off)

struct Counters {  // small device block, mirrored in pinned host memory
  u32 n_dropped;
  u32 err;
  u32 n_groups;
  u32 pad;
  u32 work_x[2];
  u32 work_y[2];
  u32 work_g[8];
};

struct Dist;  // multi.cu: this context's part in a comparison partitioned over several GPUs

// What a load writes and a grouping only reads: the records (staged, or the caller's device pointer), the processing
// order, the bucket sorts of both axes and h (carve_load), plus the side copy of a compact load.  A context owns one; its
// views (rk_create_view) share it, and the last of them to be destroyed frees it.  The context fields that point into it
// (rec4 .. h, aos_dev, pk_*) and the load's sizes are copied into every view.
struct Database {
  std::atomic<int> refs{1};  // the contexts that read it: the one that loaded it and its views
  void *arena = nullptr;
  u64 arena_bytes = 0;
  cudaStream_t copy_stream = nullptr;  // H2D of data only the output formatter reads (rk_load_packed's rest4), beside the kernels
  cudaEvent_t copy_done = nullptr;
  bool side_copy = false;  // the last load queued such a copy; copy_done marks its end
};

}  // namespace rk

struct rk_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool copy_pending = false;  // the database's side copy (Database::copy_done) is not yet waited for on this context's stream
  std::string err;

  // the loaded database (shared with the views) and this context's grouping workspace (one allocation, carve_work())
  rk::Database *db = nullptr;
  bool is_view = false;  // made by rk_create_view: groups on another context's load, never loads
  void *arena = nullptr;
  rk::u64 arena_bytes = 0;

  // pinned host result buffers
  void *h_res = nullptr;
  rk::u64 h_res_cap = 0;
  rk::Counters *h_cnt = nullptr;

  cudaEvent_t ev[RK_NSTAGES + 2];
  rk::Profiler prof;

  // calls on caller data (rk_sort_members): own counters and a grow-only scratch area
  rk::Counters *st_cnt = nullptr;
  void *st_scratch = nullptr;
  rk::u64 st_scratch_bytes = 0;

  // K6 text output: device text + work area (grow-only), pinned host mirror
  const rk::u8 *aos_dev = nullptr;  // the loaded records on the device (own copy, or the caller's device pointer)
  const uint4 *pk_key = nullptr, *pk_rest = nullptr;  // ... or the compact arrays of rk_load_packed (aos_dev == nullptr)
  const rk::u8 *pk_strand = nullptr;
  void *d_text = nullptr;
  rk::u64 d_text_bytes = 0;
  char *h_text[2] = {nullptr, nullptr};  // alternating: a chunk stays valid while the next one is produced
  rk::u64 h_text_bytes[2] = {0, 0};
  int h_text_next = 0;

  // K8 per-group statistics: device array + pinned host mirror (grow-only)
  void *d_stats = nullptr, *h_stats = nullptr;
  rk::u64 stats_cap = 0, h_stats_cap = 0;
  rk::u64 n_groups_last = 0;

  // rk_diagonal_func's table (grow-only)
  rk::u64 *d_diag = nullptr;
  rk::u64 d_diag_bytes = 0;

  bool loaded = false;
  rk::u64 n = 0;
  rk::u32 m = 0;
  rk::Geometry g{};
  int bits_rank = 1, bits_x = 1, bits_y = 1;
  bool have_group = false;

  rk::Dist *dist = nullptr;  // set by rk_dist_init (multi.cu)

  // carved pointers.  Database (carve_load, written by the load only): d_aos .. h below, except the workspace ones marked W.
  // Workspace (carve_work, written by a grouping; the load uses the loading context's scratch and counters too): W.
  rk::u8 *d_aos = nullptr;
  uint4 *rec4 = nullptr;  // file order, two words per record: {xStart, yStart, length, flags} {identity bits, file index, 0, 0}
  float *identity_r = nullptr;  // rank order
  uint4 *hfi_r = nullptr;       // rank order {h, file index, identity bits, 0}
  rk::u32 *key0 = nullptr;
  rk::u32 *link_x = nullptr, *link_y = nullptr;
  rk::u64 link_x_words = 0, link_y_words = 0;
  rk::Counters *d_cnt = nullptr;  // W
  rk::u32 *k0_r = nullptr, *fidx_r = nullptr;
  rk::u32 *tmp_k = nullptr, *tmp_v = nullptr;  // W
  uint2 *xl_r = nullptr, *yl_r = nullptr;  // rank order {center, length} per axis
  rk::u32 *ys_r = nullptr, *kx = nullptr, *ky = nullptr;
  rk::u32 *skx = nullptr, *rx = nullptr, *sky = nullptr, *ry = nullptr;
  rk::u32 *h = nullptr;
  // W from here on
  void *sort_work = nullptr;
  rk::u32 *prehist = nullptr;  // 4 x [4][256]: digit counts of key0, kx, ky, gid gathered by the kernels that produce them
  rk::u32 *xm_bits = nullptr;
  rk::u32 *parent = nullptr, *gid_rank = nullptr, *sgid = nullptr, *srank = nullptr;
  void *forest_work = nullptr;
  void *order_scratch = nullptr;
  rk::u32 *worklist = nullptr;
  rk::u32 work_cap = 0;
  rk::u32 *ent_rank = nullptr, *ent_c = nullptr, *ent_len = nullptr;
  rk::u32 *out_order = nullptr, *out_gid = nullptr;
  rk::u8 *out_repval = nullptr;
  float *out_identity = nullptr;
};

namespace rk {

inline int fail(rk_ctx *c, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  c->err = buf;
  return code;
}

#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return rk::fail(ctx, RK_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

struct ProfGuard {  // routes the launchers' KScope events to this context for the duration of one API call
  rk_ctx *c;
  explicit ProfGuard(rk_ctx *ctx) : c(ctx) { prof_route(ctx->prof.on ? &ctx->prof : nullptr); }
  ~ProfGuard() {
    if (c->prof.on) {
      cudaStreamSynchronize(c->stream);
      c->prof.fold();
    }
    prof_route(nullptr);
  }
};

Geometry make_geometry(u64 seqx_len, u64 seqy_len);
const char *err_bits_text(u32 e);
float ev_ms(cudaEvent_t a, cudaEvent_t b);
void dist_destroy(rk_ctx *c);  // multi.cu: releases c->dist (called by rk_destroy)

// capi.cu: the work behind rk_format_lines / rk_group_statistics, shared with their partitioned forms (multi.cu).
// K6 into the context's device text buffer (records ev[0]); *nbytes = the bytes formatted.  Synchronises.
int format_on_device(rk_ctx *ctx, FormatArgs fa, u64 *nbytes);
// the next of the context's two alternating pinned text buffers, grown to hold nbytes
int format_text_buffer(rk_ctx *ctx, u64 nbytes, char **buf);
// the formatted text to dst (pinned host memory); *ms_device = ev[0] .. the end of the copy.  Synchronises.
int format_to_host(rk_ctx *ctx, u64 nbytes, char *dst, float *ms_device);
// K8 into ctx->d_stats (and ctx->h_stats with RK_F_HOST_RESULT); see launch_group_stats.  Synchronises.
int group_stats_run(rk_ctx *ctx, unsigned flags, const u32 *order, const u32 *gid, const float *identity, const uint4 *rec4,
                    const LineRow *rows, u32 m, u64 ng, u32 gid_base, u32 line_off);

}  // namespace rk
