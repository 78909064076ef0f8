// C ABI of librk_b200.so (include/rk_b200.h): context, device workspace, and the launch sequences that stand
// in for FragmentsDatabase's constructor (rk_load_aos) and for generate_fragment_groups +
// generate_diagonal_func + sort_groups (rk_group).  Reference call sites: /root/reference/src/repkiller.cpp:52,84-91.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "rk_ctx.cuh"

using namespace rk;

namespace {
std::mutex g_create_mu;        // rk_create may run on several threads (one context per GPU)
std::string g_create_error;   // guarded by g_create_mu; rk_create_error() returns a per-thread copy
thread_local std::string tl_create_error;
}  // namespace

void rk::set_create_error(const std::string &s) {
  std::lock_guard<std::mutex> lk(g_create_mu);
  g_create_error = s;
}

namespace {

const char *const kKernelNames[KID_COUNT] = {"k_decode", "k_radix_hist", "k_scan", "k_radix_scatter", "k_keys", "k_match_small",
                                             "k_match_long", "k_chase", "k_hkey", "k_pack", "k_order_tile",
                                             "k_groupsort_large", "k_finalize", "k_diag_table", "k_groupsort_warp", "k_format", "k_dist_rows",
                                             "k_group_stats", "k_chase_exits", "k_csv_lines", "k_csv_rows"};

thread_local Profiler *tl_prof = nullptr;

}  // namespace

namespace {

auto taker(u8 *base, u64 &off) {
  return [base, &off](u64 bytes) -> u8 * {
    u8 *p = base ? base + off : nullptr;
    off += align_up(bytes ? bytes : 16, 256);
    return p;
  };
}

// The database part for n records (Database::arena): what the load writes and every grouping only reads.  Returns the
// bytes needed; with base == nullptr only sizes are computed.
u64 carve_load(Database &db, u8 *base, u64 n, u64 stage_bytes, LinkWords lw) {
  u64 off = 0;
  auto take = taker(base, off);
  const u64 n1 = n ? n : 1;
  db.d_aos = stage_bytes ? take(stage_bytes) : nullptr;  // host records staged on the device (109 B or 33 B each)
  db.rec4 = (uint4 *)take(n1 * 32);
  db.key0 = (u32 *)take(n1 * 4);
  db.identity_r = (float *)take(n1 * 4);
  db.hfi_r = (uint4 *)take(n1 * 16);
  db.link_x = (u32 *)take(lw.x * 4);
  db.link_y = (u32 *)take(lw.y * 4);
  db.k0_r = (u32 *)take(n1 * 4);
  db.fidx_r = (u32 *)take(n1 * 4);
  db.xl_r = (uint2 *)take(n1 * 8);
  db.yl_r = (uint2 *)take(n1 * 8);
  db.ys_r = (u32 *)take(n1 * 4);
  db.kx = (u32 *)take(n1 * 4);
  db.ky = (u32 *)take(n1 * 4);
  db.skx = (u32 *)take(n1 * 4);
  db.rx = (u32 *)take(n1 * 4);
  db.sky = (u32 *)take(n1 * 4);
  db.ry = (u32 *)take(n1 * 4);
  db.h = (u32 *)take(n1 * 4);
  return off;
}

// The grouping workspace for n loaded records (rk_ctx::arena): everything rk_group and the calls after it write, plus
// the sort scratch and counters the load borrows from the loading context.  Every context has its own.
u64 carve_work(rk_ctx *c, u8 *base, u64 n) {
  u64 off = 0;
  auto take = taker(base, off);
  const u64 n1 = n ? n : 1;
  c->d_cnt = (Counters *)take(sizeof(Counters));
  c->tmp_k = (u32 *)take(n1 * 4);
  c->tmp_v = (u32 *)take(n1 * 4);
  c->sort_work = take(sort_work_bytes(n1));
  c->prehist = (u32 *)take(4 * 4 * 256 * 4);
  c->parent = (u32 *)take(n1 * 4);
  c->xm_bits = (u32 *)take((n1 + 31) / 32 * 4);
  c->gid_rank = (u32 *)take(n1 * 4);
  c->sgid = (u32 *)take(n1 * 4);
  c->srank = (u32 *)take(n1 * 4);
  c->forest_work = take(forest_work_bytes((u32)n1));
  c->order_scratch = take(order_scratch_bytes(n1));
  c->work_cap = (u32)(n1 / 32 + 2);   // segments of more than 32 fragments (K3)
  c->worklist = (u32 *)take((u64)c->work_cap * 4);
  c->ent_rank = (u32 *)take(n1 * 4);
  c->ent_c = (u32 *)take(n1 * 4);
  c->ent_len = (u32 *)take(n1 * 4);
  c->out_order = (u32 *)take(n1 * 4);
  c->out_gid = (u32 *)take(n1 * 4);
  c->out_repval = take(n1);
  c->out_identity = (float *)take(n1 * 4);
  return off;
}

}  // namespace

namespace rk {
Geometry make_geometry(u64 seqx_len, u64 seqy_len) {
  Geometry g{};
  g.lx = seqx_len;
  g.ly = seqy_len;
  g.vsize = (u32)(1 + seqx_len / XBUCKET);  // FragmentsDatabase.cpp:84
  g.mx = (u32)(seqx_len / DIVISOR);         // SequenceOcupationList.cpp:4
  g.my = (u32)(seqy_len / DIVISOR);
  g.nbx = g.mx + 2;
  g.nby = g.my + 2;
  return g;
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) {
    cudaGetLastError();
    return 0.f;
  }
  return ms;
}

const char *err_bits_text(u32 e) {
  if (e & ERR_XBUCKET) return "a fragment has xStart/10 >= vsize (the reference writes out of bounds there)";
  if (e & ERR_CENTER) return "a fragment center lies beyond its sequence's occupation list (xStart+length/2 > sequence length)";
  if (e & ERR_COORD) return "a coordinate, length or center does not fit in 32 bits";
  if (e & ERR_WORKLIST) return "internal: segment worklist overflow";
  if (e & ERR_SPIN) return "internal: bounded wait expired";
  return "unknown device error";
}

void prof_route(Profiler *p) { tl_prof = p; }
void prof_begin(int kid, cudaStream_t st, unsigned long long units) {
  if (!tl_prof) return;
  Profiler::Rec r{kid, tl_prof->pool.get(), tl_prof->pool.get(), (u64)units};
  cudaEventRecord(r.a, st);
  tl_prof->open_recs.push_back(r);
}
void prof_end(cudaStream_t st) {
  if (!tl_prof) return;
  cudaEventRecord(tl_prof->open_recs.back().b, st);
}
}  // namespace rk


namespace {
// K5b tail + K5c on the state the last rk_group left on the device
u64 run_order(rk_ctx *ctx, unsigned flags) {
  OrderArgs oa{};
  oa.sgid = ctx->sgid, oa.srank = ctx->srank, oa.hfi_r = ctx->db->hfi_r;
  oa.m = ctx->db->m, oa.do_sort = (flags & RK_F_NO_SORT) ? 0 : 1;
  order_carve(oa, ctx->order_scratch, ctx->db->n);
  oa.work_count = ctx->d_cnt->work_g;
  oa.out_order = ctx->out_order, oa.out_gid = ctx->out_gid, oa.out_repval = ctx->out_repval, oa.out_identity = ctx->out_identity;
  oa.err = &ctx->d_cnt->err;
  return (u64)launch_order(oa, ctx->stream);
}

// optional D2H of the four output arrays, final synchronisation, error word, result struct (events 0..5 recorded)
int finish_group(rk_ctx *ctx, unsigned flags, rk_result *out, u64 launches) {
  const u32 m = ctx->db->m;
  cudaStream_t st = ctx->stream;
  cudaEvent_t *ev = ctx->ev;
  const bool host = (flags & RK_F_HOST_RESULT) && m;
  if (host) {
    const int rc = ctx->h_res.reserve(HostResult::bytes(m), st, ctx->err);
    if (rc) return rc;
  }
  CK(cudaEventRecord(ev[6], st));
  HostResult hr;
  if (host) {
    hr = HostResult(ctx->h_res.ptr(), m);
    CK(hr.fetch(ctx->out_order, ctx->out_gid, ctx->out_identity, ctx->out_repval, m, st));
  }
  CK(cudaEventRecord(ev[7], st));
  CK(cudaMemcpyAsync(ctx->h_cnt, ctx->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  if (ctx->copy_pending) {  // the formatter-only part of a compact load: done by the time a grouping is handed back
    CK(cudaStreamWaitEvent(st, ctx->db->copy_done, 0));
    ctx->copy_pending = false;
  }
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (ctx->h_cnt->err) return fail(ctx, RK_ERR_INTERNAL, "%s", err_bits_text(ctx->h_cnt->err));
  ctx->have_group = true;
  ctx->n_groups_last = ctx->h_cnt->n_groups;

  out->n_kept = m;
  out->n_groups = ctx->h_cnt->n_groups;
  hr.publish(out);
  out->d_order = ctx->out_order;
  out->d_gid = ctx->out_gid;
  out->d_repval = ctx->out_repval;
  out->d_identity = ctx->out_identity;
  out->n_launches = launches;
  if (flags & RK_F_TIMING) {
    out->ms_stage[RK_ST_XMATCH] = ev_ms(ev[0], ev[1]);
    out->ms_stage[RK_ST_YMATCH] = ev_ms(ev[1], ev[2]);
    out->ms_stage[RK_ST_FOREST] = ev_ms(ev[2], ev[3]);
    out->ms_stage[RK_ST_HKEY] = ev_ms(ev[3], ev[4]);
    out->ms_stage[RK_ST_GSORT] = ev_ms(ev[4], ev[5]);
    out->ms_stage[RK_ST_D2H] = ev_ms(ev[6], ev[7]);
    out->ms_device = ev_ms(ev[0], ev[5]);
  }
  return RK_OK;
}
}  // namespace

extern "C" {

const char *rk_version(void) { return "repkiller-b200 0.1 (sm_100a)"; }
const char *rk_create_error(void) {
  std::lock_guard<std::mutex> lk(g_create_mu);
  tl_create_error = g_create_error;
  return tl_create_error.c_str();
}

rk_ctx *rk_create(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_create_error(std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU path)");
    cudaGetLastError();
    return nullptr;
  }
  if (device < 0 || device >= count) {
    set_create_error("device index out of range");
    return nullptr;
  }
  rk_ctx *c = new rk_ctx;
  c->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaHostAlloc((void **)&c->h_cnt, sizeof(Counters), cudaHostAllocDefault)) != cudaSuccess) {
    set_create_error(cudaGetErrorString(e));
    delete c;
    return nullptr;
  }
  c->own_stream = true;
  if (const char *gr = getenv("RK_L2_GRAN")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(gr));  // tuning switch
  for (auto &ev : c->ev) cudaEventCreate(&ev);
  c->db = new Database;
  cudaStreamCreateWithFlags(&c->db->copy_stream, cudaStreamNonBlocking);
  cudaEventCreateWithFlags(&c->db->copy_done, cudaEventDisableTiming);
  if (cudaMalloc((void **)&c->st_cnt, sizeof(Counters)) != cudaSuccess) c->st_cnt = nullptr;
  // function attributes are per device: every context sets them for its own device (a process-wide flag would leave
  // the second device of a process without the shared-memory opt-in)
  if ((e = decode_init_device()) != cudaSuccess || (e = sort_init_device()) != cudaSuccess || (e = order_init_device()) != cudaSuccess ||
      (e = dist_init_device()) != cudaSuccess) {
    set_create_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    rk_destroy(c);
    return nullptr;
  }
  return c;
}

void rk_destroy(rk_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  dist_destroy(c);
  if (c->st_cnt) cudaFree(c->st_cnt);
  if (c->h_cnt) cudaFreeHost(c->h_cnt);
  for (auto &ev : c->ev) cudaEventDestroy(ev);
  if (c->db && --c->db->refs == 0) delete c->db;  // the load itself stays while views of it are live
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;  // frees the grow-only buffers: the device is current and the stream drained
}

rk_ctx *rk_create_view(rk_ctx *base) {
  if (!base) {
    set_create_error("rk_create_view: null context");
    return nullptr;
  }
  if (base->dist) {
    set_create_error("rk_create_view: the context is part of a comparison partitioned over several GPUs (rk_dist_init / rk_multi), "
                     "which has no views");
    return nullptr;
  }
  if (!base->loaded || !base->db) {
    set_create_error("rk_create_view: the context holds no database (it needs a successful rk_load_aos or rk_load_packed)");
    return nullptr;
  }
  cudaError_t e;
  rk_ctx *c = new rk_ctx;
  c->device = base->device;
  if ((e = cudaSetDevice(c->device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaHostAlloc((void **)&c->h_cnt, sizeof(Counters), cudaHostAllocDefault)) != cudaSuccess) {
    set_create_error(std::string("rk_create_view: ") + cudaGetErrorString(e));
    cudaGetLastError();
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return nullptr;
  }
  c->own_stream = true;
  for (auto &ev : c->ev) cudaEventCreate(&ev);
  if (cudaMalloc((void **)&c->st_cnt, sizeof(Counters)) != cudaSuccess) c->st_cnt = nullptr;
  ++base->db->refs;
  c->db = base->db;
  c->is_view = true;
  c->copy_pending = c->db->side_copy;  // its first grouping waits for the side copy, like the base's
  // all of the grouping workspace now: its size is known from the load, and no later call of a view allocates it
  const int rc = c->arena.reserve(carve_work(c, nullptr, c->db->n), nullptr, c->err);
  if (rc == RK_OK) carve_work(c, (u8 *)c->arena.ptr(), c->db->n);
  if (rc != RK_OK || c->h_res.reserve(HostResult::bytes(c->db->m), c->stream, c->err) != RK_OK ||
      (e = cudaMemsetAsync(c->d_cnt, 0, sizeof(Counters), c->stream)) != cudaSuccess || (e = cudaStreamSynchronize(c->stream)) != cudaSuccess) {
    set_create_error("rk_create_view: " + (c->err.empty() ? std::string(cudaGetErrorString(e)) : c->err));
    cudaGetLastError();
    rk_destroy(c);
    return nullptr;
  }
  c->loaded = true;
  return c;
}

const char *rk_last_error(const rk_ctx *c) { return c ? c->err.c_str() : rk_create_error(); }

int rk_set_stream(rk_ctx *ctx, void *cuda_stream) {
  if (!ctx) return RK_ERR_ARG;
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return RK_OK;
}

}  // extern "C"

namespace {

// The two ingest forms: 109-byte records (rk_load_aos) or the compact arrays of rk_load_packed.
struct LoadSource {
  const void *aos = nullptr;
  const void *key4 = nullptr, *strand = nullptr, *rest4 = nullptr;
  bool packed() const { return aos == nullptr; }
};

// FragmentsDatabase's constructor after parsing (src/FragmentsDatabase.cpp:84-100) on the device: K1, the processing
// order (K2a), the occupation-list buckets of both axes (K2 keys, K2b/c) and generate_diagonal_func per fragment (K5a).
// the refusals of every load, before it touches the context
int load_refusal(rk_ctx *ctx, uint64_t seqx_len, uint64_t seqy_len) {
  if (seqx_len >= (1ull << 32) || seqy_len >= (1ull << 32))
    return fail(ctx, RK_ERR_RANGE, "sequence length does not fit in 32 bits");
  if (ctx->is_view) return fail(ctx, RK_ERR_STATE, "a view groups the database of the context it was made from; load that context instead");
  if (!ctx->db) return fail(ctx, RK_ERR_STATE, "this context has no database");
  if (const int views = ctx->db->refs - 1)
    return fail(ctx, RK_ERR_STATE, "%d view%s of this context %s live: destroy %s before loading another database", views,
                views == 1 ? "" : "s", views == 1 ? "is" : "are", views == 1 ? "it" : "them");
  return RK_OK;
}

int load_common(rk_ctx *ctx, const LoadSource &src, uint64_t n, uint64_t seqx_len, uint64_t seqy_len, unsigned flags, rk_load_stats *stats) {
  if (n >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 records per context; partition the input");
  if (const int rc = load_refusal(ctx, seqx_len, seqy_len)) return rc;
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  ctx->loaded = false;
  ctx->have_group = false;
  Database &db = *ctx->db;
  db.side_copy = false;

  const void *first = src.packed() ? src.key4 : src.aos;
  const bool on_device = n ? is_device_pointer(first) : false;
  if (on_device && (((uintptr_t)first & 15) || (src.rest4 && ((uintptr_t)src.rest4 & 15))))
    return fail(ctx, RK_ERR_ARG, "device record pointers must be 16-byte aligned");
  if (src.packed() && n && (on_device != is_device_pointer(src.strand) || (src.rest4 && on_device != is_device_pointer(src.rest4))))
    return fail(ctx, RK_ERR_ARG, "the arrays of rk_load_packed must all be host or all be device memory");

  const Geometry g = make_geometry(seqx_len, seqy_len);
  const LinkWords lw = link_map_words(g);

  // (re)carve the database and the workspace; the staging area holds the host records on the device: 109 B or 33 B per record
  const u64 stage_bytes = on_device ? 0 : (src.packed() ? align_up(n * 16, 256) + align_up(n, 256) + (src.rest4 ? align_up(n * 16, 256) : 0)
                                                        : align_up(n * RK_FRAG_BYTES, 16) + 16);
  int rc = db.arena.reserve(carve_load(db, nullptr, n, stage_bytes, lw), ctx->stream, ctx->err);
  if (!rc) rc = ctx->arena.reserve(carve_work(ctx, nullptr, n), ctx->stream, ctx->err);
  if (rc) return rc;
  carve_load(db, (u8 *)db.arena.ptr(), n, stage_bytes, lw);
  carve_work(ctx, (u8 *)ctx->arena.ptr(), n);
  db.n = n;
  db.g = g;
  const SortBits bits = sort_key_bits(g);

  cudaStream_t st = ctx->stream;
  cudaEvent_t *ev = ctx->ev;
  CK(cudaEventRecord(ev[0], st));
  const u8 *aos = (const u8 *)src.aos;
  const uint4 *key4 = (const uint4 *)src.key4, *rest4 = (const uint4 *)src.rest4;
  const u8 *strand = (const u8 *)src.strand;
  if (!on_device && n) {
    if (src.packed()) {
      u8 *p = db.d_aos;
      CK(cudaMemcpyAsync(p, src.key4, n * 16, cudaMemcpyHostToDevice, st));
      key4 = (const uint4 *)p, p += align_up(n * 16, 256);
      CK(cudaMemcpyAsync(p, src.strand, n, cudaMemcpyHostToDevice, st));
      strand = p, p += align_up(n, 256);
      if (src.rest4) {  // only rk_format_lines reads these: the copy runs on its own stream while the kernels work
        CK(cudaStreamSynchronize(db.copy_stream));           // (an earlier load's copy into the old arena)
        CK(cudaEventRecord(db.copy_done, st));               // not before the work queued on st is done with the arena
        CK(cudaStreamWaitEvent(db.copy_stream, db.copy_done, 0));
        CK(cudaMemcpyAsync(p, src.rest4, n * 16, cudaMemcpyHostToDevice, db.copy_stream));
        CK(cudaEventRecord(db.copy_done, db.copy_stream));
        db.side_copy = true;
        ctx->copy_pending = true;
        rest4 = (const uint4 *)p;
      }
    } else {
      CK(cudaMemcpyAsync(db.d_aos, src.aos, n * RK_FRAG_BYTES, cudaMemcpyHostToDevice, st));
      aos = db.d_aos;
    }
  }
  db.aos_dev = aos;
  db.pk_key = key4, db.pk_rest = rest4, db.pk_strand = strand;
  CK(cudaEventRecord(ev[1], st));
  CK(cudaMemsetAsync(ctx->d_cnt, 0, sizeof(Counters), st));
  CK(cudaMemsetAsync(db.link_x, 0, lw.x * 4, st));
  CK(cudaMemsetAsync(db.link_y, 0, lw.y * 4, st));
  u64 launches = 0;
  CK(cudaMemsetAsync(ctx->prehist, 0, 3 * 4 * 256 * 4, st));
  auto hist_of = [&](int which, int bits) { return HistOut{ctx->prehist + which * 1024, (bits + 7) / 8, bits}; };
  if (src.packed())
    launches += launch_decode_packed(key4, strand, n, g, db.key0, db.link_x, db.link_y, &ctx->d_cnt->n_dropped, &ctx->d_cnt->err, st,
                                     db.rec4, hist_of(0, bits.rank));
  else
    launches += launch_decode(aos, n, g, nullptr, nullptr, nullptr, nullptr, nullptr, db.key0, db.link_x, db.link_y,
                              &ctx->d_cnt->n_dropped, &ctx->d_cnt->err, st, db.rec4, hist_of(0, bits.rank));
  CK(cudaEventRecord(ev[2], st));
  // the rank sort does not depend on the number of dropped records: they carry the largest key and sort last
  launches += launch_sort_pairs(db.key0, nullptr, db.k0_r, db.fidx_r, ctx->tmp_k, ctx->tmp_v, n, bits.rank, ctx->sort_work, st, &ctx->d_cnt->err,
                                ctx->prehist);
  CK(cudaEventRecord(ev[3], st));
  CK(cudaMemcpyAsync(ctx->h_cnt, ctx->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (ctx->h_cnt->err) return fail(ctx, (ctx->h_cnt->err & (ERR_WORKLIST | ERR_SPIN)) ? RK_ERR_INTERNAL : RK_ERR_RANGE, "%s",
                                   err_bits_text(ctx->h_cnt->err));
  const u32 m = (u32)(n - ctx->h_cnt->n_dropped);
  db.m = m;

  CK(cudaEventRecord(ev[4], st));
  launches += launch_keys(db.fidx_r, m, g, db.rec4, db.link_x, db.link_y, db.xl_r, db.yl_r, db.ys_r, db.kx, db.ky,
                          db.identity_r, st, hist_of(1, bits.x), hist_of(2, bits.y));
  // generate_diagonal_func does not depend on the ratios: h and the per-rank output record are load-time work
  launches += launch_hkey(db.k0_r, db.ys_r, m, db.h, st, db.fidx_r, db.identity_r, db.hfi_r);
  CK(cudaEventRecord(ev[5], st));
  launches += launch_sort_pairs(db.kx, nullptr, db.skx, db.rx, ctx->tmp_k, ctx->tmp_v, m, bits.x, ctx->sort_work, st, &ctx->d_cnt->err,
                                ctx->prehist + 1024);
  CK(cudaEventRecord(ev[6], st));
  launches += launch_sort_pairs(db.ky, nullptr, db.sky, db.ry, ctx->tmp_k, ctx->tmp_v, m, bits.y, ctx->sort_work, st, &ctx->d_cnt->err,
                                ctx->prehist + 2048);
  CK(cudaEventRecord(ev[7], st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  ctx->loaded = true;

  if (stats) {
    memset(stats, 0, sizeof *stats);
    stats->n_loaded = n;
    stats->n_kept = m;
    stats->vsize = g.vsize;
    stats->n_launches = launches;
    if (flags & RK_F_TIMING) {
      stats->ms_stage[RK_ST_H2D] = ev_ms(ev[0], ev[1]);
      stats->ms_stage[RK_ST_DECODE] = ev_ms(ev[1], ev[2]);
      stats->ms_stage[RK_ST_RANKSORT] = ev_ms(ev[2], ev[3]);
      stats->ms_stage[RK_ST_KEYS] = ev_ms(ev[4], ev[5]);
      stats->ms_stage[RK_ST_XSORT] = ev_ms(ev[5], ev[6]);
      stats->ms_stage[RK_ST_YSORT] = ev_ms(ev[6], ev[7]);
      stats->ms_device = ev_ms(ev[1], ev[3]) + ev_ms(ev[4], ev[7]);
    }
  }
  return RK_OK;
}

// The host text to the device through the context's pinned ring, CSV_CHUNK bytes at a time: up to `threads` threads
// (at most CSV_RING_SLOTS / 2) each copy their chunks into their own two slots and queue the upload and the newline count
// of each chunk on the context's stream, so that a chunk's host copy overlaps the uploads and counts queued before it.
int csv_upload(rk_ctx *ctx, const char *body, u64 bytes, u8 *dst, u32 *tile_cnt, int threads) {
  CsvScratch &cs = ctx->csv;
  const u64 chunks = (bytes + CSV_CHUNK - 1) / CSV_CHUNK;
  const int workers = (int)std::min<u64>(std::max(1, std::min(threads, CSV_RING_SLOTS / 2)), chunks);
  const int rc = cs.ring.reserve((u64)2 * workers * CSV_CHUNK, ctx->stream, ctx->err);
  if (rc) return rc;
  for (cudaEvent_t &e : cs.slot_done)
    if (!e) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  u8 *ring = (u8 *)cs.ring.ptr();
  std::mutex mu;
  cudaError_t first = cudaSuccess;
  std::atomic<bool> failed{false};
  auto work = [&](int w) {
    cudaError_t e = cudaSetDevice(ctx->device);
    for (u64 c = w, k = 0; c < chunks && e == cudaSuccess && !failed; c += workers, ++k) {
      const int slot = 2 * w + (int)(k & 1);
      const u64 off = c * CSV_CHUNK, len = std::min(CSV_CHUNK, bytes - off);
      if (k >= 2) e = cudaEventSynchronize(cs.slot_done[slot]);  // the slot's previous upload is done
      if (e != cudaSuccess) break;
      memcpy(ring + slot * CSV_CHUNK, body + off, len);
      e = cudaMemcpyAsync(dst + off, ring + slot * CSV_CHUNK, len, cudaMemcpyHostToDevice, ctx->stream);
      if (e == cudaSuccess) e = cudaEventRecord(cs.slot_done[slot], ctx->stream);
      if (e == cudaSuccess) launch_csv_count(dst, bytes, off / CSV_COUNT_TILE, csv_count_tiles(len), tile_cnt, ctx->stream);
    }
    if (e != cudaSuccess) {
      std::lock_guard<std::mutex> lk(mu);
      if (first == cudaSuccess) first = e;
      failed = true;
    }
  };
  std::vector<std::thread> pool;
  for (int w = 1; w < workers; ++w) pool.emplace_back(work, w);
  work(0);
  for (auto &t : pool) t.join();
  if (first != cudaSuccess) return fail(ctx, RK_ERR_CUDA, "rk_load_csv: text upload: %s", cudaGetErrorString(first));
  return RK_OK;
}

// The rows the device left to the host parser: their bytes (from the caller's host text, or copied back from the device
// text), readFragment on each, and the accepted ones as (row, 109-byte record).  Raises *wide for a wide record.
int csv_host_rows(rk_ctx *ctx, const char *body, bool on_device, const u8 *text, const u32 *d_list, u32 n_host, const u64 *start,
                  std::vector<u32> &rows, std::vector<u8> &recs, bool *wide) {
  CsvScratch &cs = ctx->csv;
  cudaStream_t st = ctx->stream;
  std::vector<u32> list(n_host);
  std::vector<ulonglong2> spans(n_host);
  int rc = cs.host.reserve(align_up((u64)n_host * 16, 256) + align_up((u64)n_host * 8, 256), st, ctx->err);
  if (rc) return rc;
  ulonglong2 *d_spans = (ulonglong2 *)cs.host.ptr();
  launch_csv_host_spans(d_list, n_host, start, d_spans, st);
  CK(cudaMemcpyAsync(list.data(), d_list, (u64)n_host * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(spans.data(), d_spans, (u64)n_host * 16, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::vector<u64> off(n_host + 1, 0);
  for (u32 i = 0; i < n_host; ++i) off[i + 1] = off[i] + (spans[i].y - spans[i].x);
  std::vector<char> copied;
  if (on_device) {  // only these rows' bytes come back
    const u64 a = align_up((u64)n_host * 16, 256), b = align_up((u64)n_host * 8, 256);
    rc = cs.host.reserve(a + b + off[n_host] + 16, st, ctx->err);
    if (rc) return rc;
    u8 *h = (u8 *)cs.host.ptr();
    CK(cudaMemcpyAsync(h, spans.data(), (u64)n_host * 16, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h + a, off.data(), (u64)n_host * 8, cudaMemcpyHostToDevice, st));
    launch_csv_gather(text, (const ulonglong2 *)h, (const u64 *)(h + a), n_host, h + a + b, st);
    copied.resize(off[n_host] + 1);
    CK(cudaMemcpyAsync(copied.data(), h + a + b, off[n_host], cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
  }
  static const int kWideFields[7] = {OFF_XSTART, OFF_YSTART, OFF_LENGTH, OFF_IDENT, OFF_XEND, OFF_YEND, OFF_SCORE};
  u8 rec[RK_FRAG_BYTES];
  for (u32 i = 0; i < n_host; ++i) {
    const char *line = on_device ? copied.data() + off[i] : body + spans[i].x;
    if (!csv_read_row_host(line, spans[i].y - spans[i].x, rec)) continue;
    rows.push_back(list[i]);
    recs.insert(recs.end(), rec, rec + RK_FRAG_BYTES);
    u64 any = 0;
    for (int f : kWideFields) {
      u64 v;
      memcpy(&v, rec + f, 8);
      any |= v;
    }
    if (any >> 32) *wide = true;  // the host route's test for the 109-byte load
  }
  return RK_OK;
}

}  // namespace

namespace rk {

int csv_upload_threads() {
  const u64 cores = std::max(1u, std::thread::hardware_concurrency() / 2);
  return (int)std::min<u64>(CSV_RING_SLOTS / 2, cores);
}

int csv_parse_local(rk_ctx *ctx, const char *body, u64 bytes, int threads, CsvParse &p) {
  CsvScratch &cs = ctx->csv;
  cudaStream_t st = ctx->stream;
  cudaEvent_t *ev = ctx->ev;
  p.bytes = bytes;
  p.on_device = bytes && is_device_pointer(body);
  const bool copy_text = !p.on_device || ((uintptr_t)body & 15);  // the kernels read the text 16 bytes at a time
  // the text scratch: [text][tile counts][their scan words][counters]
  const u64 tiles = csv_count_tiles(bytes);
  const u64 text_b = copy_text ? align_up(bytes + 16, 256) : 0, cnt_b = align_up((tiles + 1) * 4, 256),
            scan_b = align_up(csv_scan_words(tiles) * 4, 256);
  int rc = cs.text.reserve(text_b + cnt_b + scan_b + 256, st, ctx->err);
  if (rc) {
    const std::string e = ctx->err;
    return fail(ctx, rc, "rk_load_csv: %llu bytes of text: %s", (unsigned long long)bytes, e.c_str());
  }
  u8 *tb = (u8 *)cs.text.ptr();
  const u8 *text = copy_text ? tb : (const u8 *)body;
  p.text = text;
  u32 *tile_cnt = (u32 *)(tb + text_b), *tile_bsum = (u32 *)(tb + text_b + cnt_b);
  CsvCounters *cnt = (CsvCounters *)(tb + text_b + cnt_b + scan_b);
  CsvCounters h{};
  CK(cudaMemsetAsync(cnt, 0, sizeof(CsvCounters), st));
  CK(cudaMemsetAsync(tile_cnt, 0, 4, st));
  CK(cudaEventRecord(ev[EV_CSV_UP0], st));
  if (!p.on_device) {
    if (bytes && (rc = csv_upload(ctx, body, bytes, tb, tile_cnt, threads))) return rc;
  } else {
    if (copy_text) CK(cudaMemcpyAsync(tb, body, bytes, cudaMemcpyDeviceToDevice, st));
    launch_csv_count(text, bytes, 0, tiles, tile_cnt, st);
  }
  CK(cudaEventRecord(ev[EV_CSV_UP1], st));
  launch_csv_tile_scan(tile_cnt, tiles, tile_bsum, cnt, st);
  CK(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  const u64 n_rows = (u64)h.n_lines + 1;  // the segment after the last '\n' is a row too (empty after a final '\n')
  p.n_rows = n_rows;
  if (n_rows >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 rows per context; partition the input");

  // the row arrays: [start (n_rows + 1)][slot / host list (n_rows)][scan words][status (n_rows)]
  const u64 start_b = align_up((n_rows + 1) * 8, 256), slot_b = align_up(n_rows * 4, 256), rscan_b = align_up(csv_scan_words(n_rows) * 4, 256);
  rc = cs.rows.reserve(start_b + slot_b + rscan_b + align_up(n_rows, 256), st, ctx->err);
  if (rc) return rc;
  u8 *rb = (u8 *)cs.rows.ptr();
  p.start = (u64 *)rb;
  p.slot = (u32 *)(rb + start_b), p.row_bsum = (u32 *)(rb + start_b + slot_b);
  p.status = rb + start_b + slot_b + rscan_b;
  launch_csv_starts(text, bytes, tile_cnt, p.start, n_rows, st);
  launch_csv_classify(text, bytes, p.start, n_rows, p.status, p.slot, cnt, st);
  CK(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  p.n_host = h.n_host;
  p.n_dev_acc = h.n_accepted;
  p.wide = h.wide != 0;
  p.host_rows.clear();
  p.host_recs.clear();
  if (p.n_host && (rc = csv_host_rows(ctx, body, p.on_device, text, p.slot, (u32)p.n_host, p.start, p.host_rows, p.host_recs, &p.wide)))
    return rc;
  return RK_OK;
}

u64 csv_out_bytes(u64 n, bool wide) {
  return wide ? align_up(n * RK_FRAG_BYTES + 16, 256) : 2 * align_up(n * 16, 256) + align_up(n, 256);
}

int csv_emit(rk_ctx *ctx, const CsvParse &p, GrowBuffer &out, CsvOut *o) {
  CsvScratch &cs = ctx->csv;
  cudaStream_t st = ctx->stream;
  const u64 n_acc = p.n_accepted();
  // the host-accepted records, then the parsed rows at their slots in `out`
  const u64 nh = p.host_rows.size(), hrows_b = align_up(nh * 4, 256);
  if (nh) {
    const int rc = cs.host.reserve(hrows_b + nh * RK_FRAG_BYTES, st, ctx->err);
    if (rc) return rc;
    CK(cudaMemcpyAsync(cs.host.ptr(), p.host_rows.data(), nh * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((u8 *)cs.host.ptr() + hrows_b, p.host_recs.data(), nh * RK_FRAG_BYTES, cudaMemcpyHostToDevice, st));
  }
  const u64 key_b = align_up(n_acc * 16, 256);
  const int rc = out.reserve(csv_out_bytes(n_acc, p.wide), st, ctx->err);
  if (rc) return rc;
  u8 *ob = (u8 *)out.ptr();
  *o = CsvOut{};
  if (p.wide) o->aos = ob;
  else o->key4 = (uint4 *)ob, o->rest4 = (uint4 *)(ob + key_b), o->strand = ob + 2 * key_b;
  launch_csv_emit(p.text, p.bytes, p.start, p.n_rows, p.status, nh ? (const u32 *)cs.host.ptr() : nullptr, (u32)nh,
                  nh ? (const u8 *)cs.host.ptr() + hrows_b : nullptr, p.slot, p.row_bsum, *o, st);
  CK(cudaEventRecord(ctx->ev[EV_CSV_PARSED], st));
  return RK_OK;
}

}  // namespace rk

extern "C" {

int rk_load_csv(rk_ctx *ctx, const char *body, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags, unsigned flags,
                rk_load_stats *stats, rk_csv_stats *csv) {
  if (!ctx) return RK_ERR_ARG;
  if (!body && bytes) return fail(ctx, RK_ERR_ARG, "null text pointer");
  if (const int rc = load_refusal(ctx, seqx_len, seqy_len)) return rc;
  CK(cudaSetDevice(ctx->device));
  ctx->loaded = false;
  ctx->have_group = false;
  cudaEvent_t *ev = ctx->ev;
  CsvParse p;
  LoadSource src;
  {
    ProfGuard pg(ctx);
    int rc = csv_parse_local(ctx, body, bytes, csv_upload_threads(), p);
    if (rc) return rc;
    if (p.n_accepted() > total_frags) return fail(ctx, RK_ERR_RANGE, "Unexpected number of fragments");  // FragmentsDatabase.cpp:99
    CsvOut o;
    if ((rc = csv_emit(ctx, p, ctx->db->csv_out, &o))) return rc;
    if (o.aos) src.aos = o.aos;
    else src.key4 = o.key4, src.rest4 = o.rest4, src.strand = o.strand;
  }
  const u64 n_acc = p.n_accepted();
  const int rc = load_common(ctx, src, n_acc, seqx_len, seqy_len, flags, stats);
  if (rc) return rc;
  const float ms_up = ev_ms(ev[EV_CSV_UP0], ev[EV_CSV_UP1]), ms_parse = ev_ms(ev[EV_CSV_UP1], ev[EV_CSV_PARSED]);
  if (stats && (flags & RK_F_TIMING)) stats->ms_stage[RK_ST_H2D] = p.on_device ? 0.f : ms_up;
  if (csv) {
    memset(csv, 0, sizeof *csv);
    csv->n_rows = p.n_rows, csv->n_accepted = n_acc, csv->n_host_rows = p.n_host, csv->wide = p.wide;
    csv->ms_upload = p.on_device ? 0.f : ms_up;
    csv->ms_parse = ms_parse;
  }
  return RK_OK;
}

}  // extern "C"

extern "C" {

int rk_load_aos(rk_ctx *ctx, const void *frags, uint64_t n, uint64_t seqx_len, uint64_t seqy_len, unsigned flags,
                rk_load_stats *stats) {
  if (!ctx) return RK_ERR_ARG;
  if (!frags && n) return fail(ctx, RK_ERR_ARG, "null record pointer");
  LoadSource src;
  src.aos = frags ? frags : (const void *)"";  // n == 0: any non-null marker of the AoS form
  return load_common(ctx, src, n, seqx_len, seqy_len, flags, stats);
}

int rk_load_packed(rk_ctx *ctx, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n, uint64_t seqx_len,
                   uint64_t seqy_len, unsigned flags, rk_load_stats *stats) {
  if (!ctx) return RK_ERR_ARG;
  if (n && (!key4 || !strand)) return fail(ctx, RK_ERR_ARG, "null array");
  LoadSource src;
  src.key4 = key4, src.strand = strand, src.rest4 = rest4;
  return load_common(ctx, src, n, seqx_len, seqy_len, flags, stats);
}

int rk_group(rk_ctx *ctx, double len_ratio, double pos_ratio, unsigned flags, rk_result *out) {
  if (!ctx || !out) return RK_ERR_ARG;
  if (!ctx->loaded) return fail(ctx, RK_ERR_STATE, "rk_group before a successful rk_load_aos");
  if (!(len_ratio > 0)) return fail(ctx, RK_ERR_ARG, "Ratio between length and position must be greater than zero");
  if (!(pos_ratio > 0)) return fail(ctx, RK_ERR_ARG, "Position proximity must be greater than zero");
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  memset(out, 0, sizeof *out);
  const Database &db = *ctx->db;
  const u32 m = db.m;
  cudaStream_t st = ctx->stream;
  cudaEvent_t *ev = ctx->ev;
  u64 launches = 0;

  CK(cudaEventRecord(ev[0], st));
  MatchArgs mx{};
  mx.skey = db.skx, mx.srank = db.rx, mx.cl_r = db.xl_r, mx.parent = ctx->parent, mx.xm_bits = ctx->xm_bits;
  mx.m = m, mx.max_index = db.g.mx, mx.len_ratio = len_ratio, mx.pos_ratio = pos_ratio, mx.is_y = 0;
  mx.worklist = ctx->worklist, mx.work_count = ctx->d_cnt->work_x, mx.work_cap = ctx->work_cap;
  mx.ent_rank = ctx->ent_rank, mx.ent_c = ctx->ent_c, mx.ent_len = ctx->ent_len, mx.err = &ctx->d_cnt->err;
  launches += launch_match(mx, st);
  CK(cudaEventRecord(ev[1], st));
  MatchArgs my = mx;
  my.skey = db.sky, my.srank = db.ry, my.cl_r = db.yl_r, my.max_index = db.g.my, my.is_y = 1;
  my.work_count = ctx->d_cnt->work_y;
  launches += launch_match(my, st);
  CK(cudaEventRecord(ev[2], st));
  const int bits_g = key_bits(m);
  CK(cudaMemsetAsync(ctx->prehist + 3072, 0, 4 * 256 * 4, st));
  launches += launch_forest(ctx->parent, m, ctx->gid_rank, &ctx->d_cnt->n_groups, ctx->forest_work, st, 0, 0xFFFFFFFFu,
                            HistOut{ctx->prehist + 3072, (bits_g + 7) / 8, bits_g});
  CK(cudaEventRecord(ev[3], st));
  CK(cudaEventRecord(ev[4], st));
  // gids are < number of groups <= m; sorting by ceil_log2(m) bits avoids a host round trip for the count
  launches += launch_sort_pairs(ctx->gid_rank, nullptr, ctx->sgid, ctx->srank, ctx->tmp_k, ctx->tmp_v, m, bits_g,
                                ctx->sort_work, st, &ctx->d_cnt->err, m ? ctx->prehist + 3072 : nullptr);
  launches += run_order(ctx, flags);
  CK(cudaEventRecord(ev[5], st));
  return finish_group(ctx, flags, out, launches);
}

int rk_sort_groups(rk_ctx *ctx, unsigned flags, rk_result *out) {
  if (!ctx || !out) return RK_ERR_ARG;
  if (!ctx->loaded || !ctx->have_group) return fail(ctx, RK_ERR_STATE, "rk_sort_groups before rk_group");
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  memset(out, 0, sizeof *out);
  cudaEvent_t *ev = ctx->ev;
  for (int i = 0; i < 5; ++i) CK(cudaEventRecord(ev[i], ctx->stream));
  const u64 launches = run_order(ctx, flags & ~RK_F_NO_SORT);
  CK(cudaEventRecord(ev[5], ctx->stream));
  return finish_group(ctx, flags, out, launches);
}

}  // extern "C"

// (shared with multi.cu, rk_ctx.cuh)
namespace rk {
int group_stats_run(rk_ctx *ctx, unsigned flags, const u32 *order, const u32 *gid, const float *identity, const uint4 *rec4,
                    const LineRow *rows, u32 m, u64 ng, u32 gid_base, u32 line_off) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const u64 need = ng * sizeof(rk_group_stats), grown = (ng + ng / 8 + 1024) * sizeof(rk_group_stats);
  int rc = ctx->d_stats.reserve(need > ctx->d_stats.cap() ? grown : need, st, ctx->err);
  if (rc) return rc;
  launch_group_stats(order, gid, identity, rec4, rows, m, (u32)ng, gid_base, line_off, (rk_group_stats_dev *)ctx->d_stats.ptr(), st);
  if ((flags & RK_F_HOST_RESULT) && ng) {
    rc = ctx->h_stats.reserve(need > ctx->h_stats.cap() ? grown : need, st, ctx->err);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_stats.ptr(), ctx->d_stats.ptr(), need, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  return RK_OK;
}
}  // namespace rk

extern "C" {

int rk_group_statistics(rk_ctx *ctx, unsigned flags, const rk_group_stats **stats, const rk_group_stats **d_stats, uint64_t *n_groups) {
  static_assert(sizeof(rk_group_stats) == sizeof(rk_group_stats_dev) && sizeof(rk_group_stats) == 40, "stats layout");
  if (!ctx) return RK_ERR_ARG;
  if (!ctx->loaded || !ctx->have_group) return fail(ctx, RK_ERR_STATE, "rk_group_statistics before rk_group");
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  const u64 ng = ctx->n_groups_last;
  const int rc = group_stats_run(ctx, flags, ctx->out_order, ctx->out_gid, ctx->out_identity, ctx->db->rec4, nullptr, ctx->db->m, ng, 0, 0);
  if (rc) return rc;
  if (stats) *stats = ((flags & RK_F_HOST_RESULT) && ng) ? (const rk_group_stats *)ctx->h_stats.ptr() : nullptr;
  if (d_stats) *d_stats = (const rk_group_stats *)ctx->d_stats.ptr();
  if (n_groups) *n_groups = ng;
  return RK_OK;
}

int rk_diagonal_func(rk_ctx *ctx, uint64_t *diag_func) {
  if (!ctx || !diag_func) return RK_ERR_ARG;
  if (!ctx->loaded) return fail(ctx, RK_ERR_STATE, "rk_diagonal_func before rk_load_aos");
  CK(cudaSetDevice(ctx->device));
  const Database &db = *ctx->db;
  const u32 nb = db.g.vsize - 1;
  if (nb == 0) return RK_OK;
  // a grow-only table of the context: a cudaFree per call would synchronise the device, i.e. every other context on it
  const int rc = ctx->d_diag.reserve((u64)nb * 8, ctx->stream, ctx->err);
  if (rc) return rc;
  u64 *d_diag = (u64 *)ctx->d_diag.ptr();
  launch_diag_table(db.k0_r, db.ys_r, db.m, db.g.vsize, d_diag, nullptr, ctx->stream);
  cudaError_t e = cudaMemcpyAsync(diag_func, d_diag, (u64)nb * 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return fail(ctx, RK_ERR_CUDA, "rk_diagonal_func: %s", cudaGetErrorString(e));
  return RK_OK;
}

}  // extern "C"

// (shared with multi.cu, rk_ctx.cuh)
namespace rk {
int format_on_device(rk_ctx *ctx, FormatArgs fa, u64 *nbytes) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const u64 n_lines = fa.n_lines;
  const u64 text_cap = align_up(n_lines * RK_FORMAT_MAX_LINE + 16, 256);
  const u64 need = text_cap + format_work_bytes((u32)n_lines);
  const int rc = ctx->d_text.reserve(need, st, ctx->err);
  if (rc) return rc;
  fa.text = (char *)ctx->d_text.ptr();
  u32 *work = (u32 *)(fa.text + text_cap);
  fa.total_bytes = work;  // first word of the work area; launch_format carves the rest after it
  CK(cudaEventRecord(ctx->ev[0], st));
  launch_format(fa, work + 8, st);
  CK(cudaMemcpyAsync(&ctx->h_cnt->pad, fa.total_bytes, sizeof(u32), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  *nbytes = ctx->h_cnt->pad;
  return RK_OK;
}

int format_to_host(rk_ctx *ctx, u64 nbytes, char *dst, float *ms_device) {
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if (nbytes) CK(cudaMemcpyAsync(dst, ctx->d_text.ptr(), nbytes, cudaMemcpyDeviceToHost, st));
  CK(cudaEventRecord(ctx->ev[1], st));
  CK(cudaStreamSynchronize(st));
  *ms_device = ev_ms(ctx->ev[0], ctx->ev[1]);
  return RK_OK;
}
}  // namespace rk

extern "C" {

int rk_format_lines(rk_ctx *ctx, uint64_t first_line, uint64_t n_lines, rk_text *out) {
  if (!ctx || !out) return RK_ERR_ARG;
  if (!ctx->loaded || !ctx->have_group) return fail(ctx, RK_ERR_STATE, "rk_format_lines before rk_group");
  const Database &db = *ctx->db;
  if (!db.aos_dev && !db.pk_rest)
    return fail(ctx, RK_ERR_STATE, "the database was loaded with rk_load_packed without the xEnd/yEnd/score/similarity array");
  if (first_line > db.m || n_lines > db.m - first_line) return fail(ctx, RK_ERR_ARG, "line range beyond the %u output lines", db.m);
  if (n_lines > RK_FORMAT_MAX_LINES) return fail(ctx, RK_ERR_ARG, "at most %llu lines per call", (unsigned long long)RK_FORMAT_MAX_LINES);
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  memset(out, 0, sizeof *out);
  FormatArgs fa{};
  fa.aos = db.aos_dev, fa.pk_key = db.pk_key, fa.pk_rest = db.pk_rest, fa.pk_strand = db.pk_strand;
  fa.order = ctx->out_order, fa.gid = ctx->out_gid, fa.repval = ctx->out_repval, fa.identity = ctx->out_identity;
  fa.first_line = (u32)first_line, fa.n_lines = (u32)n_lines;
  u64 nbytes = 0;
  char *buf = nullptr;
  int rc = format_on_device(ctx, fa, &nbytes);
  if (!rc) rc = ctx->h_text.next(nbytes, &buf, ctx->err);
  if (!rc) rc = format_to_host(ctx, nbytes, buf, &out->ms_device);
  if (rc) return rc;
  out->text = buf;
  out->n_bytes = nbytes;
  return RK_OK;
}

int64_t rk_debug_fetch(rk_ctx *ctx, const char *name, void *host, uint64_t bytes) {
  if (!ctx || !name) return RK_ERR_ARG;
  if (!ctx->loaded) return fail(ctx, RK_ERR_STATE, "nothing loaded");
  const Database &db = *ctx->db;
  const void *src = nullptr;
  u64 sz = (u64)db.m * 4;
  if (!strcmp(name, "key4") || !strcmp(name, "strand") || !strcmp(name, "rest4")) {  // the loaded compact arrays, file order
    src = name[0] == 'k' ? (const void *)db.pk_key : name[0] == 'r' ? (const void *)db.pk_rest : (const void *)db.pk_strand;
    if (!src) return fail(ctx, RK_ERR_STATE, "the load has no %s array (109-byte records, or rk_load_packed without rest4)", name);
    sz = db.n * (name[0] == 's' ? 1 : 16);
    if (name[0] == 'r' && db.side_copy) CK(cudaStreamWaitEvent(ctx->stream, db.copy_done, 0));
  } else if (!strcmp(name, "rank_fidx")) src = db.fidx_r;
  else if (!strcmp(name, "k0_r")) src = db.k0_r;
  else if (!strcmp(name, "skx")) src = db.skx;
  else if (!strcmp(name, "rx")) src = db.rx;
  else if (!strcmp(name, "sky")) src = db.sky;
  else if (!strcmp(name, "ry")) src = db.ry;
  else if (!strcmp(name, "parent")) src = ctx->parent;
  else if (!strcmp(name, "gid_rank")) src = ctx->gid_rank;
  else if (!strcmp(name, "hkey")) src = db.h;
  else return fail(ctx, RK_ERR_ARG, "unknown array %s", name);
  if ((!strcmp(name, "parent") || !strcmp(name, "gid_rank")) && !ctx->have_group)
    return fail(ctx, RK_ERR_STATE, "no rk_group result yet");
  if (host && bytes >= sz && sz) {
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(host, src, sz, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return (int64_t)sz;
}

int rk_profile_enable(rk_ctx *ctx, int on) {
  if (!ctx) return RK_ERR_ARG;
  ctx->prof.on = on != 0;
  return RK_OK;
}

int rk_profile_read(rk_ctx *ctx, rk_kernel_time *out, int cap, int reset) {
  if (!ctx) return RK_ERR_ARG;
  int k = 0;
  for (int i = 0; i < KID_COUNT && out && k < cap; ++i) {
    if (!ctx->prof.launches[i]) continue;
    out[k].name = kKernelNames[i];
    out[k].launches = ctx->prof.launches[i];
    out[k].ms_total = ctx->prof.ms[i];
    out[k].units = ctx->prof.units[i];
    ++k;
  }
  if (reset) {
    for (int i = 0; i < KID_COUNT; ++i) ctx->prof.ms[i] = 0, ctx->prof.launches[i] = 0, ctx->prof.units[i] = 0;
  }
  return k;
}

void *rk_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void rk_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

uint64_t rk_sort_pairs_work_bytes(uint64_t n) { return sort_work_bytes(n ? n : 1); }

int rk_sort_pairs(rk_ctx *ctx, const uint32_t *keys_in, const uint32_t *values_in, uint32_t *keys_out, uint32_t *values_out,
                  uint32_t *keys_tmp, uint32_t *values_tmp, uint64_t n, int key_bits, void *work) {
  if (!ctx || !keys_in || !keys_out || !values_out || !keys_tmp || !values_tmp || !work) return RK_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  launch_sort_pairs(keys_in, values_in, keys_out, values_out, keys_tmp, values_tmp, n, key_bits, work, ctx->stream);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return RK_OK;
}

// ---- error word of the calls that work on caller data (rk_sort_members) ----------------------------------------

static int st_check_errors(rk_ctx *ctx, bool range_errors) {
  CK(cudaMemcpyAsync(ctx->h_cnt, ctx->st_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  const u32 e = ctx->h_cnt->err;
  if (e) {
    cudaMemsetAsync(&ctx->st_cnt->err, 0, sizeof(u32), ctx->stream);
    return fail(ctx, (range_errors && !(e & (ERR_WORKLIST | ERR_SPIN))) ? RK_ERR_RANGE : RK_ERR_INTERNAL, "%s", err_bits_text(e));
  }
  return RK_OK;
}

// sort_groups (src/commonFunctions.cpp:148-159) as the pure function the reference has: the order of the members of
// every group under std::sort by h = |yStart - diag_func[xStart/10]|, from the arguments alone — no state of an earlier
// rk_group is used.  The caller gathers y = f.yStart and d = diag_func[f.xStart/10] per member (loads, no arithmetic).
int rk_sort_members(rk_ctx *ctx, uint64_t m, const uint32_t *gid, const uint64_t *y, const uint64_t *d, uint32_t *perm) {
  if (!ctx || !ctx->st_cnt || (m && (!gid || !y || !d || !perm))) return RK_ERR_ARG;
  if (m >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 members");
  if (m == 0) return RK_OK;
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  cudaStream_t st = ctx->stream;
  const u64 a4 = align_up(m * 4, 256), a8 = align_up(m * 8, 256);
  const int rc = ctx->st_scratch.reserve(2 * a8 + 7 * a4 + align_up(m, 256) + align_up(order_scratch_bytes(m), 256) + 256, st, ctx->err);
  if (rc != RK_OK) return rc;
  u8 *p = (u8 *)ctx->st_scratch.ptr();
  u64 *d_y = (u64 *)p; p += a8;
  u64 *d_d = (u64 *)p; p += a8;
  u32 *d_gid = (u32 *)p; p += a4;
  u32 *d_h = (u32 *)p; p += a4;
  u32 *d_idx = (u32 *)p; p += a4;
  float *d_zero = (float *)p; p += a4;
  u32 *d_order = (u32 *)p; p += a4;
  u32 *d_ogid = (u32 *)p; p += a4;
  float *d_oident = (float *)p; p += a4;  // (identity is not part of this call: zeros in, zeros out)
  u8 *d_rep = p; p += align_up(m, 256);
  void *oscr = p;
  CK(cudaMemcpyAsync(d_y, y, m * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_d, d, m * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_gid, gid, m * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(ctx->st_cnt, 0, sizeof(Counters), st));
  launch_member_keys(d_y, d_d, (u32)m, d_h, d_idx, d_zero, &ctx->st_cnt->err, st);
  OrderArgs oa{};
  oa.sgid = d_gid, oa.srank = nullptr, oa.hfi_r = nullptr, oa.h = d_h, oa.fidx_r = d_idx, oa.identity_r = d_zero;
  oa.m = (u32)m, oa.do_sort = 1;
  order_carve(oa, oscr, m);
  oa.work_count = ctx->st_cnt->work_g;
  oa.out_order = d_order, oa.out_gid = d_ogid, oa.out_repval = d_rep, oa.out_identity = d_oident;
  oa.err = &ctx->st_cnt->err;
  launch_order(oa, st);
  CK(cudaMemcpyAsync(perm, d_order, m * 4, cudaMemcpyDeviceToHost, st));
  const int rc2 = st_check_errors(ctx, true);
  return rc2;
}

int rk_gen_workload(rk_ctx *ctx, uint64_t seed, uint64_t lx, uint64_t ly, double p_rep, uint64_t families, uint64_t ax, uint64_t ay,
                    uint64_t tandem_every, uint64_t start, uint64_t count, void *out_device) {
  if (!ctx || (count && !out_device)) return RK_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  launch_gen(seed, lx, ly, p_rep, families, ax, ay, tandem_every, start, count, (u8 *)out_device, ctx->stream);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return RK_OK;
}

}  // extern "C"
