// The context behind the C ABI (include/rk_b200.h), shared by capi.cu (single GPU) and multi.cu (one comparison over
// several GPUs): the loaded database, device workspace, grow-only buffers, pinned result buffers, per-kernel event
// profiler, error plumbing.
#pragma once

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <utility>
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

// radix bits of a sort key over `range` values: at least 1 (the sort makes at least one pass)
inline int key_bits(u64 range) { return ceil_log2(range) < 1 ? 1 : ceil_log2(range); }

// timing events, recycled: put() returns one for a later get()
struct EventPool {
  std::vector<cudaEvent_t> free;
  cudaEvent_t get() {
    if (!free.empty()) { cudaEvent_t e = free.back(); free.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
  }
  void put(cudaEvent_t e) { free.push_back(e); }
};

// CUDA-event pair around every launch group; folded into per-kernel totals after each synchronisation
struct Profiler {
  bool on = false;
  struct Rec { int kid; cudaEvent_t a, b; u64 units; };
  std::vector<Rec> open_recs;
  EventPool pool;
  double ms[KID_COUNT] = {0};
  u64 launches[KID_COUNT] = {0};
  u64 units[KID_COUNT] = {0};
  void fold() {  // call after the stream was synchronised
    for (auto &r : open_recs) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.kid] += t; launches[r.kid] += 1; units[r.kid] += r.units; }
      else cudaGetLastError();
      pool.put(r.a);
      pool.put(r.b);
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

// A grow-only buffer in device memory (cudaMalloc) or pinned host memory (cudaHostAlloc with the owner's flags).
// reserve(bytes, drain, err) keeps it when it holds `bytes`; otherwise it drains `drain` when one is given (work queued
// there may still use the old buffer), frees it and allocates exactly `bytes`; the contents are not kept.  A caller that
// wants headroom asks for more only when what it needs exceeds cap().  A failed allocation clears the CUDA error, leaves
// the buffer empty and returns RK_ERR_NOMEM; a failed drain returns RK_ERR_CUDA and keeps the buffer.  Either way `err`
// names the call.  The destructor frees the buffer: the owner's device must be current then, with no work queued that
// uses it.
class GrowBuffer {
 public:
  GrowBuffer() = default;                                                          // device memory
  explicit GrowBuffer(unsigned host_flags) : pinned_(true), flags_(host_flags) {}  // pinned host memory
  GrowBuffer(const GrowBuffer &) = delete;
  GrowBuffer &operator=(const GrowBuffer &) = delete;
  GrowBuffer(GrowBuffer &&o) noexcept : p_(o.p_), cap_(o.cap_), pinned_(o.pinned_), flags_(o.flags_) { o.p_ = nullptr, o.cap_ = 0; }
  GrowBuffer &operator=(GrowBuffer &&o) noexcept {
    std::swap(p_, o.p_), std::swap(cap_, o.cap_), std::swap(pinned_, o.pinned_), std::swap(flags_, o.flags_);
    return *this;
  }
  ~GrowBuffer() { release(); }

  int reserve(u64 bytes, cudaStream_t drain, std::string &err) {
    if (bytes <= cap_) return RK_OK;
    cudaError_t e = drain ? cudaStreamSynchronize(drain) : cudaSuccess;
    if (e != cudaSuccess) {
      err = std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e);
      return RK_ERR_CUDA;
    }
    release();
    e = pinned_ ? cudaHostAlloc(&p_, bytes, flags_) : cudaMalloc(&p_, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      p_ = nullptr;
      err = std::string(pinned_ ? "cudaHostAlloc(" : "cudaMalloc(") + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e);
      return RK_ERR_NOMEM;
    }
    cap_ = bytes;
    return RK_OK;
  }
  void *ptr() const { return p_; }
  u64 cap() const { return cap_; }

 private:
  void release() {
    if (p_) pinned_ ? cudaFreeHost(p_) : cudaFree(p_);
    p_ = nullptr, cap_ = 0;
  }
  void *p_ = nullptr;
  u64 cap_ = 0;
  bool pinned_ = false;
  unsigned flags_ = 0;
};

// Two pinned text buffers handed out in turn, so that a chunk of text stays valid while the next one is produced.
// next() grows the other buffer to hold nbytes + 1, with headroom when it has to grow.
class TextBuffers {
 public:
  explicit TextBuffers(unsigned host_flags) : b_{GrowBuffer(host_flags), GrowBuffer(host_flags)} {}
  int next(u64 nbytes, char **buf, std::string &err) {
    GrowBuffer &b = b_[next_];
    next_ ^= 1;
    const int rc = b.reserve(nbytes + 1 > b.cap() ? align_up(nbytes + nbytes / 8 + 4096, 4096) : nbytes + 1, nullptr, err);
    *buf = (char *)b.ptr();
    return rc;
  }

 private:
  GrowBuffer b_[2];
  int next_ = 0;
};

// The pinned host arrays of RK_F_HOST_RESULT for m lines, carved from one buffer of bytes(m) at 256-byte boundaries
struct HostResult {
  static u64 bytes(u64 m) { return 3 * align_up(m * 4, 256) + align_up(m, 256); }
  u32 *order = nullptr, *gid = nullptr;
  float *identity = nullptr;
  u8 *repval = nullptr;
  HostResult() = default;
  HostResult(void *buf, u64 m) {
    u8 *p = (u8 *)buf;
    order = (u32 *)p, gid = (u32 *)(p + align_up(m * 4, 256)), identity = (float *)(p + 2 * align_up(m * 4, 256));
    repval = p + 3 * align_up(m * 4, 256);
  }
  // queues the copies of a result's four device arrays into these
  cudaError_t fetch(const u32 *d_order, const u32 *d_gid, const float *d_identity, const u8 *d_repval, u64 m, cudaStream_t st) const {
    cudaError_t e = cudaMemcpyAsync(order, d_order, m * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(gid, d_gid, m * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(identity, d_identity, m * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(repval, d_repval, m, cudaMemcpyDeviceToHost, st);
    return e;
  }
  void publish(rk_result *out) const { out->order = order, out->gid = gid, out->identity = identity, out->repval = repval; }
};

Geometry make_geometry(u64 seqx_len, u64 seqy_len);
// the word counts of a load's two link maps, and the bit widths of its rank, X and Y sort keys (host side: Geometry is a
// kernel argument, and its parameter block stays as it is)
struct LinkWords { u64 x, y; };
inline LinkWords link_map_words(const Geometry &g) { return {(2ull * g.nbx + 31) / 32 + 1, (2ull * g.nby + 31) / 32 + 1}; }
struct SortBits { int rank, x, y; };
inline SortBits sort_key_bits(const Geometry &g) {
  return {key_bits(g.vsize),
          ceil_log2(2ull * g.nbx),  // >= 2: nbx >= 2
          ceil_log2(2ull * g.nby)};
}

inline bool is_device_pointer(const void *p) {
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, p) == cudaSuccess) return pa.type == cudaMemoryTypeDevice;
  cudaGetLastError();
  return false;
}

struct Dist;  // multi.cu: this context's part in a comparison partitioned over several GPUs

// rk_load_csv's scratch on the loading context: the text on the device with its tile counts, the row arrays, the host
// rows' spans and records, and the pinned ring the text is uploaded through (CSV_RING_SLOTS slots of CSV_CHUNK bytes;
// two per upload thread, each with the event of its last copy).
constexpr int CSV_RING_SLOTS = 8;
constexpr u64 CSV_CHUNK = 4ull << 20;
struct CsvScratch {
  GrowBuffer text, rows, host;
  GrowBuffer ring{cudaHostAllocDefault};
  cudaEvent_t slot_done[CSV_RING_SLOTS] = {};
  CsvScratch() = default;
  CsvScratch(const CsvScratch &) = delete;
  CsvScratch &operator=(const CsvScratch &) = delete;
  ~CsvScratch() {
    for (cudaEvent_t e : slot_done)
      if (e) cudaEventDestroy(e);
  }
};
// the parse's events on ctx->ev, after the ones a load records (0..7)
enum { EV_CSV_UP0 = 8, EV_CSV_UP1, EV_CSV_PARSED };
// rk_dist_load_packed's copies of host arrays: key4 and strand on the context's stream, rest4 on the copy stream
enum { EV_PK_UP0 = EV_CSV_PARSED + 1, EV_PK_UP1, EV_PK_REST };
static_assert(EV_PK_REST < RK_NSTAGES + 2, "the events fit rk_ctx::ev");

// What a load writes and a grouping only reads: the load's sizes, the records (staged, or the caller's device pointer),
// the processing order, the bucket sorts of both axes and h (carve_load), plus the side copy of a compact load.  A
// context owns one; its views (rk_create_view) hold a reference to it instead of a copy, and the last context to be
// destroyed frees it.  It does not change while views are live: loading is refused then.
struct Database {
  std::atomic<int> refs{1};  // the contexts that read it: the one that loaded it and its views
  GrowBuffer arena;
  cudaStream_t copy_stream = nullptr;  // H2D of data only the output formatter reads (rk_load_packed's rest4), beside the kernels
  cudaEvent_t copy_done = nullptr;
  bool side_copy = false;  // the last load queued such a copy; copy_done marks its end

  u64 n = 0;  // records loaded
  u32 m = 0;  // records kept
  Geometry g{};

  GrowBuffer csv_out;  // rk_load_csv: the parsed rows (compact arrays, or 109-byte records when a value is wide)

  const u8 *aos_dev = nullptr;  // the loaded records on the device (own copy, or the caller's device pointer)
  const uint4 *pk_key = nullptr, *pk_rest = nullptr;  // ... or the compact arrays of rk_load_packed (aos_dev == nullptr)
  const u8 *pk_strand = nullptr;

  // carved by carve_load
  u8 *d_aos = nullptr;  // the host records staged on the device
  uint4 *rec4 = nullptr;  // file order, two words per record: {xStart, yStart, length, flags} {identity bits, file index, 0, 0}
  float *identity_r = nullptr;  // rank order
  uint4 *hfi_r = nullptr;       // rank order {h, file index, identity bits, 0}
  u32 *key0 = nullptr;
  u32 *link_x = nullptr, *link_y = nullptr;
  u32 *k0_r = nullptr, *fidx_r = nullptr;
  uint2 *xl_r = nullptr, *yl_r = nullptr;  // rank order {center, length} per axis
  u32 *ys_r = nullptr, *kx = nullptr, *ky = nullptr;
  u32 *skx = nullptr, *rx = nullptr, *sky = nullptr, *ry = nullptr;
  u32 *h = nullptr;

  ~Database() {
    if (copy_stream) cudaStreamSynchronize(copy_stream), cudaStreamDestroy(copy_stream);
    if (copy_done) cudaEventDestroy(copy_done);
  }
};

}  // namespace rk

struct rk_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool copy_pending = false;  // the database's side copy (Database::copy_done) is not yet waited for on this context's stream
  std::string err;

  // the loaded database (shared with the views) and this context's grouping workspace (carve_work)
  rk::Database *db = nullptr;
  bool is_view = false;  // made by rk_create_view: groups on another context's load, never loads
  rk::GrowBuffer arena;

  // pinned host result buffers
  rk::GrowBuffer h_res{cudaHostAllocDefault};
  rk::Counters *h_cnt = nullptr;

  cudaEvent_t ev[RK_NSTAGES + 2];
  rk::Profiler prof;

  // calls on caller data (rk_sort_members): own counters and a grow-only scratch area
  rk::Counters *st_cnt = nullptr;
  rk::GrowBuffer st_scratch;

  // K6 text output: device text + work area, pinned host mirror
  rk::GrowBuffer d_text;
  rk::TextBuffers h_text{cudaHostAllocDefault};

  // K8 per-group statistics: device array + pinned host mirror
  rk::GrowBuffer d_stats, h_stats{cudaHostAllocDefault};
  rk::u64 n_groups_last = 0;

  rk::GrowBuffer d_diag;  // rk_diagonal_func's table

  rk::CsvScratch csv;  // rk_load_csv

  bool loaded = false;
  bool have_group = false;

  rk::Dist *dist = nullptr;  // set by rk_dist_init (multi.cu)

  // the workspace, carved by carve_work: written by a grouping; the load uses the loading context's scratch and counters too
  rk::Counters *d_cnt = nullptr;
  rk::u32 *tmp_k = nullptr, *tmp_v = nullptr;
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

const char *err_bits_text(u32 e);
float ev_ms(cudaEvent_t a, cudaEvent_t b);
void dist_destroy(rk_ctx *c);  // multi.cu: releases c->dist (called by rk_destroy)
void set_create_error(const std::string &s);  // capi.cu: the text rk_create_error() returns

// capi.cu: the work behind rk_format_lines / rk_group_statistics, shared with their partitioned forms (multi.cu).
// K6 into the context's device text buffer (records ev[0]); *nbytes = the bytes formatted.  Synchronises.
int format_on_device(rk_ctx *ctx, FormatArgs fa, u64 *nbytes);
// the formatted text to dst (pinned host memory); *ms_device = ev[0] .. the end of the copy.  Synchronises.
int format_to_host(rk_ctx *ctx, u64 nbytes, char *dst, float *ms_device);
// K8 into ctx->d_stats (and ctx->h_stats with RK_F_HOST_RESULT); see launch_group_stats.  Synchronises.
int group_stats_run(rk_ctx *ctx, unsigned flags, const u32 *order, const u32 *gid, const float *identity, const uint4 *rec4,
                    const LineRow *rows, u32 m, u64 ng, u32 gid_base, u32 line_off);

// capi.cu: rk_load_csv's parse in two halves, shared with rk_dist_load_csv (multi.cu), which exchanges the counts of
// the first half over the ranks before it runs the second.
struct CsvParse {
  bool on_device = false;    // the caller's text is in device memory
  const u8 *text = nullptr;  // the text on the device: the caller's, or the context's copy
  u64 bytes = 0;
  u64 n_rows = 0;            // '\n' + 1: the segment after the last '\n' is a row too
  u64 n_host = 0;            // rows left to the host parser
  u64 n_dev_acc = 0;         // rows accepted on the device
  bool wide = false;         // an accepted row has a value of 33 or more bits
  u64 *start = nullptr;      // the row arrays in CsvScratch::rows
  u32 *slot = nullptr, *row_bsum = nullptr;
  u8 *status = nullptr;
  std::vector<u32> host_rows;  // the host rows readFragment accepted, and their 109-byte records
  std::vector<u8> host_recs;
  u64 n_accepted() const { return n_dev_acc + host_rows.size(); }
};
// copy threads of one text upload
int csv_upload_threads();
// The local half: text scratch, upload with the newline counts (at most `threads` copy threads), tile scan, row starts,
// classify and the host rows.  Records ev[EV_CSV_UP0] and ev[EV_CSV_UP1].  Synchronises.
int csv_parse_local(rk_ctx *ctx, const char *body, u64 bytes, int threads, CsvParse &p);
// bytes of the parsed rows of n accepted rows: three compact arrays, or 109-byte records when wide
u64 csv_out_bytes(u64 n, bool wide);
// The emit: the host-accepted records to the device, `out` grown to csv_out_bytes, and every accepted row at its
// file-order slot in it; *o says where the rows are.  Records ev[EV_CSV_PARSED].
int csv_emit(rk_ctx *ctx, const CsvParse &p, GrowBuffer &out, CsvOut *o);

}  // namespace rk
