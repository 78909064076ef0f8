// One comparison partitioned over several GPUs: the orchestration behind rk_dist_* (one process per GPU) and
// rk_create_multi / rk_multi_* (one process, one host thread per GPU) of include/rk_b200.h.  SURVEY.md §8e.
//
// The reference has no distributed path (SURVEY.md §5); what is reproduced is generate_fragment_groups +
// generate_diagonal_func + sort_groups (/root/reference/src/commonFunctions.cpp:41-80,161-177,148-159) on ONE fragment
// file whose records start out spread over the GPUs in file order.  The kernels and the argument for exactness are in
// k7_dist.cu; this file owns the buffers, the two transports and the order of the launches:
//
//   load   K1 on the local slice -> [all-gather: xStart/10 histogram + link maps] -> cuts -> exchange 1: the split kernel
//          stores every 32-byte record into its owner's arena (peer memory) -> processing order (K2a) -> keys (K2) -> h (K5a)
//          -> X halo rows to the higher GPUs; Y rows (16 B) to the owners of their Y super-bucket range, by copy engines
//          beside the X bucket sort -> X and Y bucket sorts (K2b/c)                              [2 host syncs: counts]
//   group  X pass (K3) -> halo owners stored at their home rank (4 B) -> "matched in X" bytes stored at the Y owners
//          -> Y pass (K3) -> the Y owners stored at the home ranks -> root scan; local chains; chains that leave the GPU in
//          bulk ask/answer rounds (many) or by walking the peers' res[] (few) (K4) -> output rows (16 B) stored at the
//          owner of their group-id range -> K5b/c                                                [2 host syncs: counts]
//          (RK_F_LINE_RECORDS) -> every line asks the rank that loaded its record; that rank stores the 64-byte line row
//          at the asker's line_rows[line], for K6 / K8 on the rank that holds the line            [1 host sync: counts]
//
// Every rank's partition arena is carved identically and mapped into every peer (cudaIpc handles between processes, raw
// pointers + cudaDeviceEnablePeerAccess inside one), so a local buffer address translates to the same buffer on any rank;
// kernels store rows straight into it (k7_dist.cu: k_push_rows, scatter_store), copy engines push the X halo and Y rows
// (Transport::exchange_rows).  Rows travel this one way under both transports; they differ only in the small tables and
// the barrier.  NCCL (dlopen'ed: the process may already hold torch's libnccl.so.2) carries the small tables
// (ncclAllGather of counts, histograms, link maps) and is the barrier behind every push.  Ranks that are threads of one
// process, possibly on the same device (tests on a one-GPU box), exchange the small tables through host memory between
// host barriers instead, and their barrier is a stream synchronisation followed by a host barrier.
#include <dlfcn.h>
#include <nccl.h>
#include <unistd.h>

#include <algorithm>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>

#include "rk_ctx.cuh"

using namespace rk;

namespace rk {

// ---------------------------------------------------------------------------------------------------------------------
// NCCL through dlopen
// ---------------------------------------------------------------------------------------------------------------------
struct NcclApi {
  void *lib = nullptr;
  std::string err;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommInitAll) CommInitAll = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok() const { return lib != nullptr && err.empty(); }
};
static NcclApi &nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    // an already loaded libnccl.so.2 (torch's) is reused: same soname
    api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!api.lib) api.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!api.lib) {
      api.err = std::string("dlopen(libnccl.so.2): ") + dlerror();
      return;
    }
#define RK_NCCL_SYM(field, name)                                         \
  api.field = (decltype(api.field))dlsym(api.lib, name);                 \
  if (!api.field) api.err = std::string("libnccl lacks ") + name;
    RK_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    RK_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    RK_NCCL_SYM(CommInitAll, "ncclCommInitAll")
    RK_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    RK_NCCL_SYM(AllGather, "ncclAllGather")
    RK_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef RK_NCCL_SYM
  });
  return api;
}

// ---------------------------------------------------------------------------------------------------------------------
// transports
// ---------------------------------------------------------------------------------------------------------------------
constexpr int SMALL_WORDS = 96;  // per-rank row of the count exchanges
constexpr int W_CNT_A = 0;       // [nr+1] destination counts (exchange 1 / X halo / output exchange)
constexpr int W_CNT_B = 17;      // [nr+1] destination counts of the Y exchange
constexpr int W_ERR = 40;        // device error word of the rank
constexpr int W_X0 = 41;         // roots on the rank
constexpr int W_X1 = 42;         // total groups
constexpr int W_X2 = 43;         // forest: fragments of the rank whose chain is still waiting for an answer from another rank
constexpr int W_CUTSX = 64;      // [2][nr] the first X super-bucket key every rank owns, per strand class
constexpr int W_CUTS = 44;       // [nr+1] the cuts of the exchange (identical on every rank; the host sizes the local sort keys from them)
constexpr int W_FOFF = 61;       // exchange 1: the file index of the rank's first record (rk_dist_load_aos's file_offset)

struct Exchange {  // counts of one variable all-to-all, as this rank sees it (elements)
  u64 soff[DIST_MAX_RANKS], scnt[DIST_MAX_RANKS], roff[DIST_MAX_RANKS], rcnt[DIST_MAX_RANKS];
  u64 poff[DIST_MAX_RANKS];   // forward: start of my block in rank p's receive buffer (= p's roff[me])
  u64 rpoff[DIST_MAX_RANKS];  // the way back: start of my block in rank p's send-order buffer (= p's soff[me])
  u64 n_send = 0, n_recv = 0;
  // from the gathered count matrix: row s = what rank s sends to every destination
  void from_matrix(const u32 *h_all, int word0, int nr, int me) {
    n_send = n_recv = 0;
    for (int d = 0; d < nr; ++d) {
      soff[d] = n_send;
      scnt[d] = h_all[(size_t)me * SMALL_WORDS + word0 + d];
      n_send += scnt[d];
    }
    for (int s = 0; s < nr; ++s) {
      roff[s] = n_recv;
      rcnt[s] = h_all[(size_t)s * SMALL_WORDS + word0 + me];
      n_recv += rcnt[s];
    }
    for (int p = 0; p < nr; ++p) {
      u64 f = 0, r = 0;
      for (int s = 0; s < me; ++s) f += h_all[(size_t)s * SMALL_WORDS + word0 + p];
      for (int d = 0; d < me; ++d) r += h_all[(size_t)p * SMALL_WORDS + word0 + d];
      poff[p] = f, rpoff[p] = r;
    }
  }
};

// column `word` of the gathered count matrix summed over the ranks (word = W_CNT_A + d: the rows rank d receives)
static u64 column_sum(const u32 *h_all, int word, int nr) {
  u64 s = 0;
  for (int r = 0; r < nr; ++r) s += h_all[(size_t)r * SMALL_WORDS + word];
  return s;
}

struct Transport {
  int rank = 0, world = 1;
  std::string err;
  u64 bytes_sent = 0;  // payload this rank handed to other ranks
  virtual ~Transport() {
    if (ev_a) cudaEventDestroy(ev_a);
    if (ev_b) cudaEventDestroy(ev_b);
    for (auto &a : aux) if (a) cudaStreamDestroy(a);
    for (auto &e : aux_ev) if (e) cudaEventDestroy(e);
  }
  // every rank contributes SMALL_WORDS u32 from device memory.  begin() leaves all rows in DEVICE memory d_all
  // (stream-ordered: kernels queued behind it may read the other ranks' counts), end() brings them to the host
  // h_all[world][SMALL_WORDS] (pinned) and synchronises the stream.
  virtual int gather_small_begin(const u32 *d_row, u32 *d_all, u32 *h_all, cudaStream_t st) = 0;
  virtual int gather_small_end(const u32 *d_all, u32 *h_all, cudaStream_t st) = 0;
  // all ranks' streams meet: work queued behind it starts after every rank's work queued before it is complete
  virtual int barrier(cudaStream_t st) = 0;
  // recv[world][bytes] <- every rank's send[bytes]; stream-ordered; doubles as a barrier between the ranks' streams
  virtual int all_gather(const void *send, void *recv, size_t bytes, cudaStream_t st) = 0;
  // peer memory: every rank's partition arena has the same layout, so a local pointer translates to any peer's copy
  const u8 *my_base = nullptr;
  u8 *peer_base[DIST_MAX_RANKS] = {nullptr};
  template <class T>
  T *on_peer(int p, T *local) const { return (T *)(peer_base[p] + ((const u8 *)local - my_base)); }
  // out[d] = the buffer `local` on rank d, for every rank (kernels store rows straight into it)
  template <class T, class U>
  void peer_table(T *local, U **out) const {
    for (int d = 0; d < world; ++d) out[d] = d == rank ? local : on_peer(d, local);
  }

  // The rows of a variable all-to-all (counts of `ex` in elements of `elem` bytes).  Every rank PUSHES its blocks into
  // the peers' receive buffers with copy-engine copies (peer copies over NVLink between GPUs), then enters barrier().
  // A rank's stream holds its pushes when it enters the barrier, so after the barrier every block addressed to this rank
  // has landed.  The caller makes sure that no rank still reads its receive buffer when the pushes start.
  int exchange_rows(const void *send, const Exchange &ex, void *recv, size_t elem, cudaStream_t st) {
    const int rc = push_blocks(send, ex, recv, elem, st);
    return rc ? rc : barrier(st);
  }
  // The same in two halves, so that rows can travel while kernels run: begin() enqueues the pushes on `side`, ordered
  // after everything queued on st so far; end() makes st wait for them, then enters the barrier.
  int exchange_rows_begin(const void *send, const Exchange &ex, void *recv, size_t elem, cudaStream_t st, cudaStream_t side) {
    if (!ev_a && (cudaEventCreateWithFlags(&ev_a, cudaEventDisableTiming) != cudaSuccess ||
                  cudaEventCreateWithFlags(&ev_b, cudaEventDisableTiming) != cudaSuccess)) {
      err = "row exchange: cudaEventCreate failed";
      return RK_ERR_CUDA;
    }
    cudaEventRecord(ev_a, st);
    cudaStreamWaitEvent(side, ev_a, 0);
    const int rc = push_blocks(send, ex, recv, elem, side);
    if (rc) return rc;
    cudaEventRecord(ev_b, side);
    split_pending = true;
    return RK_OK;
  }
  int exchange_rows_end(cudaStream_t st) {
    if (!split_pending) return RK_OK;
    split_pending = false;
    cudaStreamWaitEvent(st, ev_b, 0);
    return barrier(st);
  }
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  bool split_pending = false;
  // This rank's blocks into the peers' receive buffers, peers in staggered order so that no receiver is hit by everybody
  // at once.  Large exchanges are spread over a few copy streams (one copy engine each), forked from st and joined into
  // it again: a single peer copy does not fill the links of a GPU (measured 550 GB/s for one copy at a time).
  static constexpr int NAUX = 3;
  cudaStream_t aux[NAUX] = {nullptr, nullptr, nullptr};
  cudaEvent_t aux_ev[NAUX + 1] = {nullptr, nullptr, nullptr, nullptr};
  int push_blocks(const void *send, const Exchange &ex, void *recv, size_t elem, cudaStream_t st) {
    u64 total = 0;
    int peers = 0;
    for (int p = 0; p < world; ++p)
      if (p != rank && ex.scnt[p]) total += ex.scnt[p] * elem, ++peers;
    const bool spread = peers > 1 && total >= (8u << 20);
    if (spread && !aux[0]) {
      for (int a = 0; a < NAUX; ++a) cudaStreamCreateWithFlags(&aux[a], cudaStreamNonBlocking);
      for (int a = 0; a <= NAUX; ++a) cudaEventCreateWithFlags(&aux_ev[a], cudaEventDisableTiming);
    }
    if (spread) {
      cudaEventRecord(aux_ev[NAUX], st);
      for (int a = 0; a < NAUX; ++a) cudaStreamWaitEvent(aux[a], aux_ev[NAUX], 0);
    }
    int turn = 0;
    for (int k = 0; k < world; ++k) {
      const int p = (rank + k) % world;
      if (!ex.scnt[p]) continue;
      u8 *dst = (p == rank ? (u8 *)recv : on_peer(p, (u8 *)recv)) + ex.poff[p] * elem;
      cudaStream_t cs = st;
      if (spread && p != rank) cs = (turn % (NAUX + 1)) == NAUX ? st : aux[turn % (NAUX + 1)], ++turn;
      if (cudaMemcpyAsync(dst, (const u8 *)send + ex.soff[p] * elem, ex.scnt[p] * elem, cudaMemcpyDeviceToDevice, cs) != cudaSuccess) {
        err = std::string("row exchange: peer copy failed: ") + cudaGetErrorString(cudaGetLastError());
        return RK_ERR_CUDA;
      }
      if (p != rank) bytes_sent += ex.scnt[p] * elem;
    }
    if (spread)
      for (int a = 0; a < NAUX; ++a) {
        cudaEventRecord(aux_ev[a], aux[a]);
        cudaStreamWaitEvent(st, aux_ev[a], 0);
      }
    return RK_OK;
  }
};

struct NcclTransport : Transport {
  ncclComm_t comm = nullptr;
  bool own_comm = true;
  u32 *d_flag = nullptr, *d_flag_all = nullptr;  // barrier payload (set by the owner of the transport)
  int check(ncclResult_t r, const char *what) {
    if (r == ncclSuccess) return RK_OK;
    err = std::string(what) + ": " + nccl_api().GetErrorString(r);
    return RK_ERR_CUDA;
  }
  ~NcclTransport() override {
    if (comm && own_comm) nccl_api().CommDestroy(comm);
  }
  int gather_small_begin(const u32 *d_row, u32 *d_all, u32 *, cudaStream_t st) override {
    return check(nccl_api().AllGather(d_row, d_all, SMALL_WORDS * sizeof(u32), ncclUint8, comm, st), "ncclAllGather");
  }
  int gather_small_end(const u32 *d_all, u32 *h_all, cudaStream_t st) override {
    cudaError_t e = cudaMemcpyAsync(h_all, d_all, (size_t)world * SMALL_WORDS * sizeof(u32), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      err = std::string("count exchange: ") + cudaGetErrorString(e);
      return RK_ERR_CUDA;
    }
    return RK_OK;
  }
  // a 4-byte all-gather: it completes on a rank only after every rank's stream has reached it
  int barrier(cudaStream_t st) override { return check(nccl_api().AllGather(d_flag, d_flag_all, 4, ncclUint8, comm, st), "ncclAllGather (barrier)"); }
  int all_gather(const void *send, void *recv, size_t bytes, cudaStream_t st) override {
    bytes_sent += bytes * (u64)(world - 1);
    return check(nccl_api().AllGather(send, recv, bytes, ncclUint8, comm, st), "ncclAllGather");
  }
};

// ranks = threads of one process (any devices, also the same one): the small tables meet in host memory between host
// barriers
struct LocalGroup {
  int n = 0;
  std::mutex mu;
  std::condition_variable cv;
  int waiting = 0;
  u64 generation = 0;
  const void *ptr[DIST_MAX_RANKS] = {nullptr};
  u32 small[DIST_MAX_RANKS][SMALL_WORDS] = {{0}};
  void barrier() {
    std::unique_lock<std::mutex> lk(mu);
    const u64 gen = generation;
    if (++waiting == n) {
      waiting = 0;
      ++generation;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != gen; });
    }
  }
};

struct LocalTransport : Transport {
  LocalGroup *g = nullptr;
  int cuda(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return RK_OK;
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return RK_ERR_CUDA;
  }
  // the host exchange, then the matrix goes back to the device
  int gather_small_begin(const u32 *d_row, u32 *d_all, u32 *h_all, cudaStream_t st) override {
    cudaError_t e = cudaMemcpyAsync(h_all + (size_t)rank * SMALL_WORDS, d_row, SMALL_WORDS * sizeof(u32), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) memcpy(g->small[rank], h_all + (size_t)rank * SMALL_WORDS, SMALL_WORDS * sizeof(u32));
    g->barrier();
    for (int r = 0; r < world; ++r) memcpy(h_all + (size_t)r * SMALL_WORDS, g->small[r], SMALL_WORDS * sizeof(u32));
    g->barrier();
    const int rc = cuda(e, "count exchange");
    if (rc) return rc;
    return cuda(cudaMemcpyAsync(d_all, h_all, (size_t)world * SMALL_WORDS * sizeof(u32), cudaMemcpyHostToDevice, st), "count upload");
  }
  int gather_small_end(const u32 *, u32 *, cudaStream_t st) override { return cuda(cudaStreamSynchronize(st), "count exchange"); }
  int barrier(cudaStream_t st) override {
    const cudaError_t e = cudaStreamSynchronize(st);
    g->barrier();
    return cuda(e, "barrier");
  }
  int all_gather(const void *send, void *recv, size_t bytes, cudaStream_t st) override {
    cudaError_t e = cudaStreamSynchronize(st);
    g->ptr[rank] = send;
    g->barrier();
    for (int r = 0; r < world && e == cudaSuccess; ++r)
      e = cudaMemcpyAsync((u8 *)recv + (size_t)r * bytes, g->ptr[r], bytes, cudaMemcpyDefault, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    g->barrier();
    bytes_sent += bytes * (u64)(world - 1);
    return cuda(e, "all_gather");
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// per-rank state
// ---------------------------------------------------------------------------------------------------------------------
// RK_DIST_TRACE=1: CUDA-event pairs around every transport call and the sections between them, printed per rank after
// the final synchronisation of rk_dist_group (a tuning aid: where a step spends its time)
struct Trace {
  bool on = false;
  struct Rec { const char *what; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  EventPool pool;
  void begin(const char *what, cudaStream_t st) {
    if (!on) return;
    Rec r{what, pool.get(), pool.get()};
    cudaEventRecord(r.a, st);
    recs.push_back(r);
  }
  void end(cudaStream_t st) {
    if (on && !recs.empty()) cudaEventRecord(recs.back().b, st);
  }
  void dump(int rank, const std::string &counts) {
    if (!on) return;
    std::string line = "[rk_dist rank " + std::to_string(rank) + "] " + counts;
    float total = 0.f;
    for (auto &r : recs) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) cudaGetLastError();
      // label: the transport function and its first argument, e.g. exchange_rows(D.halo_send
      std::string w(r.what);
      const size_t p0 = w.find("->"), p1 = w.find(',');
      w = w.substr(p0 == std::string::npos ? 0 : p0 + 2, p1 == std::string::npos ? std::string::npos : p1 - (p0 == std::string::npos ? 0 : p0 + 2));
      char buf[160];
      snprintf(buf, sizeof buf, " %s)=%.3f", w.c_str(), ms);
      line += buf;
      total += ms;
      pool.put(r.a);
      pool.put(r.b);
    }
    recs.clear();
    fprintf(stderr, "%s | comm total %.3f ms\n", line.c_str(), total);
  }
};

struct DistBlob {  // what a rank publishes so that its peers can read its parent / root-scan arrays
  u64 pid, ptr, cap;
  int device, view;  // view: the mapped memory is a view's workspace, not a partition arena
  cudaIpcMemHandle_t handle;
};
static_assert(sizeof(DistBlob) <= RK_DIST_BLOB_BYTES, "blob size");

// The partition database of a rank: what a load writes and a grouping only reads.  The sizes and exchange tables of the
// load, the rank's slice of the records, the rank-order and bucket-sorted arrays of both passes, and the load-time
// regions (rec4_loc, send_rows, rec6_arr, the halo rows) that only the load uses.  The rank's base context and its views
// (rk_multi_create_view, rk_dist_create_view) hold a reference to it; the last context to be destroyed frees it.  It
// does not change while views are live: loading is refused then.
struct DistDb {
  std::atomic<int> refs{1};
  GrowBuffer arena;  // carved by dist_carve: this database, then the workspace of the loading context
  u64 cap = 0, hcap = 0;
  // grow-only side buffers whose size depends on the input, not on cap
  GrowBuffer aos_buf;  // this rank's records: a host slice staged (109 B per row), its parsed CSV rows (compact or 109 B), or
                       // its host compact arrays staged (33 B per row, laid out as csv_emit lays out compact rows)
  GrowBuffer link_buf;  // u32 [hist0][linkx_loc][linky_loc] (one all-gather) [linkx][linky][gather: world * the first three]

  // state of the last load
  bool loaded = false;
  Geometry g{};
  int bits_rank = 1, bits_y = 1;
  u32 m_loc = 0, rank_off = 0, n_halo = 0, n_away = 0, m_y = 0;
  u64 m_total = 0, n_total_loaded = 0;
  Exchange ex1, exh, exy;
  const u8 *aos_src = nullptr;          // this rank's slice of the records on the device (aos_buf or the caller's pointer)
  PackedRows pk_src{};                  // ... or its compact rows (rk_dist_load_csv without a wide value, rk_dist_load_packed;
                                        // aos_src == nullptr)
  int rest_missing = -1;                // rk_dist_load_packed: the first rank that loaded records without rest4, or -1
  u32 file_off[DIST_MAX_RANKS] = {0};  // first file index of every rank's slice
  bool slices_in_order = false;         // every slice ends at or before the next rank's starts: file_off[] routes a file index
  u32 roff[DIST_MAX_RANKS + 1] = {0};   // first rank-order index of every rank, then the total (PeerTable::roff)

  // carved device pointers
  u32 *cuts0 = nullptr, *cuts_y = nullptr, *cuts_x = nullptr;
  uint4 *rec4_loc = nullptr, *send_rows = nullptr;
  uint2 *rec6_arr = nullptr;  // the records this rank owns, in arrival order: 24-byte rows stored by the peers' push kernels
  u32 *key0_loc = nullptr, *perm_x = nullptr, *perm_y = nullptr;
  u32 *key0a = nullptr, *k0_r = nullptr, *aidx_r = nullptr;
  uint2 *xl = nullptr, *yl_r = nullptr, *yl_a = nullptr;
  u32 *ys_r = nullptr, *kx2 = nullptr, *ky = nullptr, *gfidx_r = nullptr;
  float *identity_r = nullptr;
  uint4 *hfi_r = nullptr;
  uint4 *halo_send = nullptr, *halo_recv = nullptr;
  u32 *halo_grank = nullptr;
  u32 *skx = nullptr, *rx = nullptr, *ky_a = nullptr, *grank_a = nullptr, *sky_a = nullptr, *ry_a = nullptr;
  u32 *roff_dev = nullptr;
};

// One context's part in a partitioned comparison: its transport, its peers' mappings and its grouping workspace, i.e.
// everything rk_dist_group, rk_dist_format_lines and rk_dist_group_statistics write.  The load runs on the base context
// and uses its workspace as scratch too (counters, count rows, sort scratch, recv_rows for the Y rows).
struct Dist {
  int rank = 0, world = 1;
  Transport *tr = nullptr;
  DistDb *db = nullptr;
  bool is_view = false;  // groups on another context's database (db is shared), never loads
  GrowBuffer arena;      // a view's workspace (dist_carve_work); the base's lies in db->arena
  void *peer_open[DIST_MAX_RANKS] = {nullptr};
  bool peers_ready = false;
  GrowBuffer small_host{cudaHostAllocDefault};
  u32 *h_small = nullptr;  // [world][SMALL_WORDS] in small_host
  PeerTable pt{};
  Trace trace;
  cudaStream_t side = nullptr;  // rows that travel while kernels run (the Y exchange beside the X sort)
  GrowBuffer h_res{cudaHostAllocDefault};
  // the memory the peers map: the base's whole partition arena, or a view's workspace (every peer carves it identically)
  u8 *map_base() const { return (u8 *)(is_view ? arena.ptr() : db->arena.ptr()); }

  // state of the last group: this rank's output lines and groups; line rows (RK_F_LINE_RECORDS) valid
  bool have_rows = false;
  u32 n_lines = 0, gid_base = 0, n_groups_rank = 0;
  u64 line_off = 0;

  // carved device pointers (the workspace)
  Counters *cnt = nullptr;
  u32 *d_small = nullptr, *d_small_all = nullptr, *nroots_mat = nullptr;
  u32 *prehist = nullptr;  // 4 x [4][256]: digit counts of the rank / X / Y / gid sort keys, gathered by their producers
  u32 *hist = nullptr, *hist_all = nullptr, *cuts_g = nullptr;
  uint4 *recv_rows = nullptr;
  LineRow *line_rows = nullptr;  // RK_F_LINE_RECORDS: one row per output line
  u32 *tile_cnt = nullptr, *tmp_k = nullptr, *tmp_v = nullptr;
  void *sort_work = nullptr;
  u32 *away_res = nullptr;
  u32 *parent_x = nullptr, *xm_bits = nullptr, *parent = nullptr, *gidscan = nullptr, *parent_y = nullptr, *yo_s = nullptr;
  u8 *xm_a = nullptr;
  u32 *ent_rank = nullptr, *ent_c = nullptr, *ent_len = nullptr, *worklist = nullptr;
  u32 work_cap = 0;
  u32 *gid_rank = nullptr, *flag = nullptr, *flag_all = nullptr, *lroot = nullptr, *gid_l = nullptr;
  u32 *pend_idx[2] = {nullptr, nullptr}, *pend_key[2] = {nullptr, nullptr}, *n_pend = nullptr;  // forest: pending lists (double buffered)
  u32 *apos = nullptr;
  uint4 *queries = nullptr;  // forest bulk rounds: the ranks other GPUs ask this one about (stored by their push kernels)
  u64 *answers = nullptr;    // ... and the answers to this rank's questions, in the order it sent them (stored by the owners)
  u64 *res = nullptr;  // per fragment: what a walker from another GPU needs (k_chase_local); the peers read it
  void *scan_work = nullptr;
  u32 *gid_a = nullptr, *sgid = nullptr, *srank_g = nullptr;
  void *order_scratch = nullptr;
  u32 *out_order = nullptr, *out_gid = nullptr;
  u8 *out_repval = nullptr;
  float *out_identity = nullptr;
};

// bump allocation of one arena at 256-byte boundaries; base == nullptr only counts the bytes
struct Carve {
  u8 *base;
  u64 off = 0;
  u8 *take(u64 bytes) {
    u8 *p = base ? base + off : nullptr;
    off += align_up(bytes ? bytes : 16, 256);
    return p;
  }
};

// the partition database for B.cap rows per rank (B.hcap halo rows)
static void dist_carve_db(DistDb &B, Carve &c) {
  const u64 M = B.cap, H = B.hcap, MC = M + H;
  B.cuts0 = (u32 *)c.take((DIST_MAX_RANKS + 1) * 4);
  B.cuts_y = (u32 *)c.take((DIST_MAX_RANKS + 1) * 4);
  B.cuts_x = (u32 *)c.take(2 * DIST_MAX_RANKS * 4);
  B.rec4_loc = (uint4 *)c.take(M * 32);
  B.send_rows = (uint4 *)c.take(M * 16);
  B.rec6_arr = (uint2 *)c.take(M * 24);
  B.key0_loc = (u32 *)c.take(M * 4);
  B.perm_x = (u32 *)c.take(H * 4);
  B.perm_y = (u32 *)c.take(M * 4);
  B.key0a = (u32 *)c.take(M * 4);
  B.k0_r = (u32 *)c.take(M * 4);
  B.aidx_r = (u32 *)c.take(M * 4);
  B.xl = (uint2 *)c.take(MC * 8);
  B.yl_r = (uint2 *)c.take(M * 8);
  B.yl_a = (uint2 *)c.take(M * 8);
  B.ys_r = (u32 *)c.take(M * 4);
  B.kx2 = (u32 *)c.take(MC * 4);
  B.ky = (u32 *)c.take(M * 4);
  B.gfidx_r = (u32 *)c.take(M * 4);
  B.identity_r = (float *)c.take(M * 4);
  B.hfi_r = (uint4 *)c.take(M * 16);
  B.halo_send = (uint4 *)c.take(H * 16);
  B.halo_recv = (uint4 *)c.take(H * 16);
  B.halo_grank = (u32 *)c.take(H * 4);
  B.skx = (u32 *)c.take(MC * 4);
  B.rx = (u32 *)c.take(MC * 4);
  B.ky_a = (u32 *)c.take(M * 4);
  B.grank_a = (u32 *)c.take(M * 4);
  B.sky_a = (u32 *)c.take(M * 4);
  B.ry_a = (u32 *)c.take(M * 4);
  B.roff_dev = (u32 *)c.take((DIST_MAX_RANKS + 1) * 4);
}

// a grouping workspace for cap rows per rank (hcap halo rows) over D.world ranks.  A view carries its own line rows,
// 64 B per row of capacity; the base's overlay the load-time regions of its database (dist_carve).
static void dist_carve_work(Dist &D, u64 cap, u64 hcap, Carve &c) {
  const u64 M = cap, H = hcap, MC = M + H;
  const int nr = D.world;
  D.cnt = (Counters *)c.take(sizeof(Counters));
  D.d_small = (u32 *)c.take(SMALL_WORDS * 4);
  D.d_small_all = (u32 *)c.take((u64)nr * SMALL_WORDS * 4);
  D.nroots_mat = (u32 *)c.take((u64)nr * SMALL_WORDS * 4);
  D.prehist = (u32 *)c.take(4 * 4 * 256 * 4);
  D.hist = (u32 *)c.take(DIST_BINS * 4);
  D.hist_all = (u32 *)c.take((u64)nr * DIST_BINS * 4);
  D.cuts_g = (u32 *)c.take((DIST_MAX_RANKS + 1) * 4);
  D.line_rows = D.is_view ? (LineRow *)c.take(M * sizeof(LineRow)) : (LineRow *)D.db->rec4_loc;
  D.recv_rows = (uint4 *)c.take(M * 16);
  D.tile_cnt = (u32 *)c.take(dist_split_work_bytes(M));
  D.tmp_k = (u32 *)c.take(MC * 4);
  D.tmp_v = (u32 *)c.take(MC * 4);
  D.sort_work = c.take(sort_work_bytes(MC));
  D.away_res = (u32 *)c.take(H * 4);
  D.parent_x = (u32 *)c.take(MC * 4);
  D.xm_bits = (u32 *)c.take((MC + 31) / 32 * 4);
  D.parent = (u32 *)c.take(M * 4);
  D.gidscan = (u32 *)c.take(M * 4);
  D.lroot = (u32 *)c.take(M * 4);
  D.gid_l = (u32 *)c.take(M * 4);
  for (int b = 0; b < 2; ++b) D.pend_idx[b] = (u32 *)c.take(M * 4), D.pend_key[b] = (u32 *)c.take(M * 4);
  D.n_pend = (u32 *)c.take(16);
  D.apos = (u32 *)c.take(M * 4);
  D.queries = (uint4 *)c.take(M * 16);
  D.answers = (u64 *)c.take(M * 8);
  D.res = (u64 *)c.take(M * 8);
  D.flag = (u32 *)c.take(16);
  D.flag_all = (u32 *)c.take(DIST_MAX_RANKS * 4);
  D.parent_y = (u32 *)c.take(M * 4);
  D.yo_s = (u32 *)c.take(M * 4);
  D.xm_a = c.take(M);
  D.ent_rank = (u32 *)c.take(MC * 4);
  D.ent_c = (u32 *)c.take(MC * 4);
  D.ent_len = (u32 *)c.take(MC * 4);
  D.work_cap = (u32)(MC / 32 + 2);
  D.worklist = (u32 *)c.take((u64)D.work_cap * 4);
  D.gid_rank = (u32 *)c.take(M * 4);
  D.scan_work = c.take(dist_scan_work_bytes((u32)M));
  D.gid_a = (u32 *)c.take(M * 4);
  D.sgid = (u32 *)c.take(M * 4);
  D.srank_g = (u32 *)c.take(M * 4);
  D.order_scratch = c.take(order_scratch_bytes(M));
  D.out_order = (u32 *)c.take(M * 4);
  D.out_gid = (u32 *)c.take(M * 4);
  D.out_repval = c.take(M);
  D.out_identity = (float *)c.take(M * 4);
}

// the base's partition arena: the database, then its workspace, whose line rows overlay rec4_loc ++ send_rows ++
// rec6_arr.  Only the load reads or writes those three regions, so after it they hold the line rows of rk_dist_group
// with RK_F_LINE_RECORDS: 72 B per row of capacity, back to back, for 64 B per line (a rank never holds more lines than
// rows).  A view cannot share them (two contexts would write the same rows) and carries its own.
static u64 dist_carve(Dist &D, u8 *base) {
  static_assert(sizeof(LineRow) <= 32 + 16 + 24, "line rows fit in the load-time regions");
  Carve c{base};
  dist_carve_db(*D.db, c);
  dist_carve_work(D, D.db->cap, D.db->hcap, c);
  return c.off;
}

static void dist_release_peers(Dist &D) {
  for (int r = 0; r < DIST_MAX_RANKS; ++r) {
    if (D.peer_open[r]) cudaIpcCloseMemHandle(D.peer_open[r]);
    D.peer_open[r] = nullptr;
  }
  D.peers_ready = false;
}

// grows the partition arena of a base context to cap rows per rank; the peers must import again afterwards
static int dist_allocate(rk_ctx *ctx, u64 cap) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  dist_release_peers(D);
  B.cap = B.hcap = 0;
  B.loaded = false;
  if (cap < 1024) cap = 1024;
  if (cap >= 0xFFFFFF00ull) return fail(ctx, RK_ERR_ARG, "capacity per rank must stay below 2^32");
  B.cap = cap;
  B.hcap = cap / 8 + 65536;
  std::string err;
  const int rc = B.arena.reserve(dist_carve(D, nullptr), nullptr, err);
  if (rc) {
    B.cap = B.hcap = 0;
    return fail(ctx, rc, "%llu rows per rank: %s", (unsigned long long)cap, err.c_str());
  }
  dist_carve(D, (u8 *)B.arena.ptr());
  return RK_OK;
}

static int tr_fail(rk_ctx *ctx, int rc) { return fail(ctx, rc, "%s", ctx->dist->tr->err.c_str()); }
#define TR(call)                                  \
  do {                                            \
    D.trace.begin(#call, ctx->stream);            \
    const int rc_ = (call);                       \
    D.trace.end(ctx->stream);                     \
    if (rc_ != RK_OK) return tr_fail(ctx, rc_);   \
  } while (0)

// views that share ctx's load: of a single-GPU load (rk_create_view) or of its partition database
static int live_views(const rk_ctx *ctx) {
  if (ctx->dist) return ctx->dist->is_view ? 0 : ctx->dist->db->refs - 1;
  return ctx->db ? ctx->db->refs - 1 : 0;
}

// the refusals of a load on a rank context, before it touches anything: a view, or a base with live views
static int dist_load_refusal(rk_ctx *ctx) {
  if (ctx->dist->is_view)
    return fail(ctx, RK_ERR_STATE, "a view groups the partition database of the context it was made from; load that context instead");
  if (const int views = live_views(ctx))
    return fail(ctx, RK_ERR_STATE, "%d view%s of this context %s live: destroy %s before loading another database", views,
                views == 1 ? "" : "s", views == 1 ? "is" : "are", views == 1 ? "it" : "them");
  return RK_OK;
}

// rk_dist_init on a view, or on a context with live views
static int dist_init_refusal(rk_ctx *ctx) {
  if (ctx->is_view) return fail(ctx, RK_ERR_STATE, "a view cannot take part in a partitioned comparison");
  if (live_views(ctx)) return fail(ctx, RK_ERR_STATE, "views of this context are live: destroy them before rk_dist_init");
  return RK_OK;
}

static int dist_init_common(rk_ctx *ctx, int rank, int world, Transport *tr, u64 cap) {
  if (world < 1 || world > DIST_MAX_RANKS || rank < 0 || rank >= world) {
    delete tr;
    return fail(ctx, RK_ERR_ARG, "rank %d of %d: at most %d ranks", rank, world, DIST_MAX_RANKS);
  }
  if (const int rc = dist_init_refusal(ctx)) {
    delete tr;
    return rc;
  }
  dist_destroy(ctx);
  Dist *D = new Dist;
  D->rank = rank, D->world = world, D->tr = tr;
  D->db = new DistDb;
  tr->rank = rank, tr->world = world;
  ctx->dist = D;
  D->trace.on = getenv("RK_DIST_TRACE") != nullptr;
  CK(cudaSetDevice(ctx->device));
  const int rc = D->small_host.reserve((u64)world * SMALL_WORDS * sizeof(u32), nullptr, ctx->err);
  if (rc) return rc;
  D->h_small = (u32 *)D->small_host.ptr();
  CK(cudaStreamCreateWithFlags(&D->side, cudaStreamNonBlocking));
  return dist_allocate(ctx, cap);
}

// the reason no view can be made of `base`, or nullptr
static const char *dist_view_refusal(const rk_ctx *base) {
  if (!base || !base->dist) return "the context is not part of a comparison partitioned over several GPUs (rk_dist_init / rk_multi)";
  if (!base->dist->db->loaded)
    return "the context holds no partition database (it needs a successful rk_dist_load_aos, rk_dist_load_csv, rk_dist_load_packed or "
           "rk_multi_load_*)";
  return nullptr;
}

// A view of the rank context `base` (which holds a load): a new context on its device that shares base's partition
// database and has its own transport `tr` (taken over, deleted on failure) and grouping workspace.  The peers' views
// are mapped by dist_export / dist_import afterwards.  NULL on failure, with err set.
static rk_ctx *dist_view_create(rk_ctx *base, Transport *tr, std::string &err) {
  if (const char *why = dist_view_refusal(base)) {
    delete tr;
    err = why;
    return nullptr;
  }
  const Dist &S = *base->dist;
  DistDb &B = *S.db;
  rk_ctx *c = rk_create(base->device);
  if (!c) {
    delete tr;
    err = rk_create_error();
    return nullptr;
  }
  c->is_view = true;
  Dist *V = new Dist;
  V->rank = S.rank, V->world = S.world, V->tr = tr;
  tr->rank = S.rank, tr->world = S.world;
  V->db = &B;
  ++B.refs;
  V->is_view = true;
  c->dist = V;
  V->trace.on = S.trace.on;
  // all of the workspace now, sized by the database's capacity: no later call of a view allocates it
  Carve count{nullptr};
  dist_carve_work(*V, B.cap, B.hcap, count);
  Carve carve{nullptr};
  int rc = V->small_host.reserve((u64)V->world * SMALL_WORDS * sizeof(u32), nullptr, c->err);
  if (!rc) rc = V->arena.reserve(count.off, nullptr, c->err);
  if (!rc) {
    V->h_small = (u32 *)V->small_host.ptr();
    carve.base = (u8 *)V->arena.ptr();
    dist_carve_work(*V, B.cap, B.hcap, carve);
    cudaError_t e = cudaMemsetAsync(V->cnt, 0, sizeof(Counters), c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = fail(c, RK_ERR_CUDA, "%s", cudaGetErrorString(e));
  }
  if (rc) {
    err = c->err;
    rk_destroy(c);
    return nullptr;
  }
  return c;
}

static int dist_export(rk_ctx *ctx, DistBlob *b) {
  Dist &D = *ctx->dist;
  memset(b, 0, sizeof *b);
  b->pid = (u64)getpid(), b->ptr = (u64)(uintptr_t)D.map_base(), b->cap = D.db->cap, b->device = ctx->device, b->view = D.is_view;
  CK(cudaSetDevice(ctx->device));
  CK(cudaIpcGetMemHandle(&b->handle, D.map_base()));
  return RK_OK;
}

static int dist_import(rk_ctx *ctx, const u8 *blobs, size_t stride) {
  Dist &D = *ctx->dist;
  CK(cudaSetDevice(ctx->device));
  for (int r = 0; r < D.world; ++r) {
    DistBlob b;
    memcpy(&b, blobs + (size_t)r * stride, sizeof b);
    if (b.cap != D.db->cap) return fail(ctx, RK_ERR_ARG, "rank %d was initialised with capacity %llu, this rank with %llu", r,
                                        (unsigned long long)b.cap, (unsigned long long)D.db->cap);
    if (b.view != (int)D.is_view)
      return fail(ctx, RK_ERR_ARG, "rank %d exported a %s, this rank is a %s", r, b.view ? "view" : "base context", D.is_view ? "view" : "base context");
    u8 *base = nullptr;
    if (r == D.rank) {
      base = D.map_base();
    } else if (b.pid == (u64)getpid()) {
      base = (u8 *)(uintptr_t)b.ptr;
      if (b.device != ctx->device) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
          return fail(ctx, RK_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", ctx->device, b.device, cudaGetErrorString(e));
        cudaGetLastError();
      }
    } else {
      if (D.peer_open[r]) cudaIpcCloseMemHandle(D.peer_open[r]);
      D.peer_open[r] = nullptr;
      CK(cudaIpcOpenMemHandle((void **)&base, b.handle, cudaIpcMemLazyEnablePeerAccess));
      D.peer_open[r] = base;
    }
    D.tr->peer_base[r] = base;
    // the arenas are carved identically (same capacity, same number of ranks): local offsets hold on every peer
    D.pt.res[r] = (const u64 *)(base + ((const u8 *)D.res - D.map_base()));
  }
  D.tr->my_base = D.map_base();
  if (NcclTransport *nt = dynamic_cast<NcclTransport *>(D.tr)) nt->d_flag = D.flag, nt->d_flag_all = D.flag_all;
  D.pt.nr = D.world, D.pt.me = D.rank;
  D.peers_ready = true;
  return RK_OK;
}

// The count exchange: every rank publishes its row d_small (its error word W_ERR included; the caller has written the
// rest) and gets everybody's rows, on the device in d_small_all and on the host in h_small.  A routed round passes
// `push`: launched once the rows are on the device, it stores rows straight into their owners' buffers (peer memory),
// and a barrier follows it, so the rows have landed everywhere when this returns.  Synchronises.
static int dist_gather_counts(rk_ctx *ctx, const std::function<void()> &push = {}) {
  Dist &D = *ctx->dist;
  CK(cudaMemcpyAsync(D.d_small + W_ERR, &D.cnt->err, sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
  TR(D.tr->gather_small_begin(D.d_small, D.d_small_all, D.h_small, ctx->stream));
  if (push) {
    push();
    TR(D.tr->barrier(ctx->stream));
  }
  TR(D.tr->gather_small_end(D.d_small_all, D.h_small, ctx->stream));
  return RK_OK;
}

// error words of all ranks after a count exchange: every rank sees the same matrix, so every rank returns together.
// With worklist_nomem, ERR_WORKLIST is a capacity error: RK_ERR_NOMEM with that message (it takes the capacity per rank).
static int dist_check_small(rk_ctx *ctx, bool range_errors, const char *worklist_nomem = nullptr) {
  const Dist &D = *ctx->dist;
  u32 e = 0;
  for (int r = 0; r < D.world; ++r) e |= D.h_small[(size_t)r * SMALL_WORDS + W_ERR];
  if (!e) return RK_OK;
  if (worklist_nomem && (e & ERR_WORKLIST)) return fail(ctx, RK_ERR_NOMEM, worklist_nomem, (unsigned long long)D.db->cap);
  return fail(ctx, (range_errors && !(e & (ERR_WORKLIST | ERR_SPIN))) ? RK_ERR_RANGE : RK_ERR_INTERNAL, "%s", err_bits_text(e));
}

// after a count exchange: the rows every rank d receives (column word0 + d, summed over the senders) against bound.
// fmt takes the rank, the rows and the capacity per rank; every rank sees the same matrix, so every rank returns together.
static int check_inbound(rk_ctx *ctx, int word0, u64 bound, const char *fmt) {
  const Dist &D = *ctx->dist;
  for (int d = 0; d < D.world; ++d) {
    const u64 in = column_sum(D.h_small, word0 + d, D.world);
    if (in > bound) return fail(ctx, RK_ERR_NOMEM, fmt, d, (unsigned long long)in, (unsigned long long)D.db->cap);
  }
  return RK_OK;
}

// this rank's slice of a cut table, [cuts[me], cuts[me + 1]) with the end clamped to limit (the last rank's to limit):
// sort keys taken relative to base need `bits` bits
struct KeyRange { u32 base; u64 end; int bits; };
static KeyRange rank_key_range(const u32 *cuts, int me, int nr, u64 limit) {
  const u64 end = me + 1 < nr ? std::min<u64>(cuts[me + 1], limit) : limit;
  return {cuts[me], end, key_bits(end > cuts[me] ? end - cuts[me] : 1)};
}

// block table of a per-pair exchange whose values the producing kernel stores straight into the peers' buffers:
// forward = in send order (blocks by destination, landing where the rows of the load-time exchange landed),
// back = in arrival order (blocks by source, landing in the order this rank's rows were sent)
template <class T>
static ScatterTable scatter_table(const Dist &D, const Exchange &ex, bool back, T *local_buf) {
  ScatterTable t{};
  t.nr = D.world;
  u64 run = 0;
  for (int d = 0; d < D.world; ++d) {
    t.start[d] = (u32)run;
    run += back ? ex.rcnt[d] : ex.scnt[d];
    t.dst_off[d] = (u32)(back ? ex.rpoff[d] : ex.poff[d]);
  }
  t.start[D.world] = (u32)run;
  D.tr->peer_table(local_buf, t.out);
  return t;
}

// ---------------------------------------------------------------------------------------------------------------------
// load: FragmentsDatabase's constructor over the ranks (src/FragmentsDatabase.cpp:84-100)
// ---------------------------------------------------------------------------------------------------------------------
// pk: the slice as compact rows on the device (rk_dist_load_csv) instead of 109-byte records at frags
static int dist_load(rk_ctx *ctx, const void *frags, u64 n_loc, u64 file_off, u64 seqx_len, u64 seqy_len, unsigned flags,
                     rk_load_stats *stats, const PackedRows *pk = nullptr) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  const int nr = D.world, me = D.rank;
  if (!D.peers_ready) return fail(ctx, RK_ERR_STATE, "rk_dist_load_aos before rk_dist_import");
  if (!frags && !pk && n_loc) return fail(ctx, RK_ERR_ARG, "null record pointer");
  if (seqx_len >= (1ull << 32) || seqy_len >= (1ull << 32)) return fail(ctx, RK_ERR_RANGE, "sequence length does not fit in 32 bits");
  if (file_off + n_loc >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 records in one comparison");
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  cudaStream_t st = ctx->stream;
  B.loaded = false;
  B.rest_missing = -1;  // (rk_dist_load_packed sets it after this returns)
  D.have_rows = false;
  ctx->have_group = false;
  // NOTE: argument errors that only ONE rank can see (n_loc > cap) are turned into an error word all ranks receive with
  // the first count exchange, so that no rank is left waiting in a collective.
  const bool too_many = n_loc > B.cap;
  const u64 n_use = too_many ? 0 : n_loc;

  const Geometry g = make_geometry(seqx_len, seqy_len);
  B.g = g;
  const SortBits bits = sort_key_bits(g);
  B.bits_rank = bits.rank, B.bits_y = bits.y;
  const LinkWords lw = link_map_words(g);
  const u64 lxw = lw.x, lyw = lw.y;
  const u64 pub_words = DIST_BINS + lxw + lyw;  // what a rank publishes after K1: its xStart/10 histogram and its link maps
  const u64 link_need = pub_words + lxw + lyw + (u64)nr * pub_words + 64;
  const int rc = B.link_buf.reserve(link_need * 4, st, ctx->err);
  if (rc) return rc;
  u32 *hist0 = (u32 *)B.link_buf.ptr(), *linkx_loc = hist0 + DIST_BINS, *linky_loc = linkx_loc + lxw, *linkx = linky_loc + lyw, *linky = linkx + lxw,
      *pub_all = linky + lyw;

  const bool on_device = n_use && !pk && is_device_pointer(frags);
  if (on_device && ((uintptr_t)frags & 15)) return fail(ctx, RK_ERR_ARG, "device record pointer must be 16-byte aligned");
  const u8 *aos = (const u8 *)frags;
  cudaEvent_t *ev = ctx->ev;
  CK(cudaEventRecord(ev[0], st));
  if (!on_device && !pk && n_use) {
    const int rc2 = B.aos_buf.reserve(align_up(n_use * RK_FRAG_BYTES, 16) + 16, st, ctx->err);
    if (rc2) return rc2;
    CK(cudaMemcpyAsync(B.aos_buf.ptr(), frags, n_use * RK_FRAG_BYTES, cudaMemcpyHostToDevice, st));
    aos = (const u8 *)B.aos_buf.ptr();
  }
  B.aos_src = pk ? nullptr : aos;
  B.pk_src = pk ? *pk : PackedRows{};
  CK(cudaEventRecord(ev[1], st));
  u64 launches = 0;

  // K1 on the local slice of the file
  CK(cudaMemsetAsync(D.cnt, 0, sizeof(Counters), st));
  CK(cudaMemsetAsync(D.d_small, 0, SMALL_WORDS * 4, st));
  CK(cudaMemsetAsync(D.prehist, 0, 3 * 4 * 256 * 4, st));
  CK(cudaMemsetAsync(linkx_loc, 0, (lxw + lyw) * 4, st));
  auto hist_of = [&](int which, int bits) { return HistOut{D.prehist + which * 1024, (bits + 7) / 8, bits}; };
  if (too_many) {
    const u32 e = ERR_WORKLIST;  // reported below as a capacity error
    CK(cudaMemcpyAsync(&D.cnt->err, &e, 4, cudaMemcpyHostToDevice, st));
  }
  if (pk)
    launches += launch_decode_packed(pk->key, pk->strand, n_use, g, B.key0_loc, linkx_loc, linky_loc, &D.cnt->n_dropped, &D.cnt->err, st,
                                     B.rec4_loc, HistOut{nullptr, 0, 0}, (u32)file_off);
  else
    launches += launch_decode(aos, n_use, g, nullptr, nullptr, nullptr, nullptr, nullptr, B.key0_loc, linkx_loc, linky_loc,
                              &D.cnt->n_dropped, &D.cnt->err, st, B.rec4_loc, HistOut{nullptr, 0, 0}, (u32)file_off);
  // exchange 1: to the owner of the xStart/10 range
  const int shift0 = B.bits_rank > 12 ? B.bits_rank - 12 : 0;
  launches += dist_coarse_hist(B.key0_loc, (u32)n_use, shift0, 0, g.vsize - 1, hist0, st);
  // one all-gather for everything K1 produced that the other ranks need: the histogram the cuts are made from and the link
  // maps (OR-ed over the ranks below, so that a run of linked buckets has one key everywhere)
  TR(D.tr->all_gather(hist0, pub_all, pub_words * 4, st));
  launches += dist_cuts_from_hist(pub_all, pub_words, nr, shift0, B.cuts0, st);
  launches += dist_or_rows(pub_all + DIST_BINS, pub_words, nr, lxw, linkx, st);
  launches += dist_or_rows(pub_all + DIST_BINS + lxw, pub_words, nr, lyw, linky, st);
  // count per destination -> all ranks' counts on the device -> every tile stores its records straight into the owners'
  // receive buffers (peer memory over NVLink) -> barrier; the host reads the count matrix while the rows travel
  uint2 *outs[DIST_MAX_RANKS];
  D.tr->peer_table(B.rec6_arr, outs);
  launches += dist_count_plain(B.key0_loc, (u32)n_use, B.cuts0, nr, g.vsize - 1, D.tile_cnt, D.d_small + W_CNT_A, st);
  CK(cudaMemcpyAsync(D.d_small + W_CUTS, B.cuts0, (nr + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  const u32 foff32 = (u32)file_off;
  CK(cudaMemcpyAsync(D.d_small + W_FOFF, &foff32, sizeof(u32), cudaMemcpyHostToDevice, st));  // (pageable source: staged at once)
  if (const int rc = dist_gather_counts(ctx, [&] {  // host sync 1
        launches += dist_push_records(B.key0_loc, (u32)n_use, B.cuts0, nr, g.vsize - 1, B.rec4_loc, outs, (u32)B.cap, D.tile_cnt,
                                      D.d_small_all, SMALL_WORDS, me, st);
      }))
    return rc;
  // (a rank whose slice exceeds the capacity loaded nothing and published ERR_WORKLIST)
  if (const int rc = dist_check_small(ctx, true, "a rank holds more records than the capacity of %llu rows per rank given to rk_dist_init"))
    return rc;
  if (const int rc = check_inbound(ctx, W_CNT_A, B.cap, "rank %d would own %llu fragments, capacity is %llu rows per rank")) return rc;
  B.ex1.from_matrix(D.h_small, W_CNT_A, nr, me);
  // where every rank's slice starts (as its caller said) and, from the row sums of the count matrix (the dropped column
  // included), how long it is: the line records of RK_F_LINE_RECORDS find the rank that loaded a record by these starts,
  // which needs the slices in rank order without overlap.  Every rank sees the same matrix, so all agree on the verdict.
  B.slices_in_order = true;
  for (int s = 0; s < nr; ++s) {
    u64 n_s = 0;
    for (int d = 0; d <= nr; ++d) n_s += D.h_small[(size_t)s * SMALL_WORDS + W_CNT_A + d];
    B.file_off[s] = D.h_small[(size_t)s * SMALL_WORDS + W_FOFF];
    if (s + 1 < nr && B.file_off[s] + n_s > D.h_small[(size_t)(s + 1) * SMALL_WORDS + W_FOFF]) B.slices_in_order = false;
  }
  D.tr->bytes_sent += (B.ex1.n_send - B.ex1.scnt[me]) * 24;  // (the rows this rank's kernels stored into peer memory)
  u64 loaded_total = 0, off = 0;
  for (int d = 0; d <= nr; ++d) loaded_total += column_sum(D.h_small, W_CNT_A + d, nr);
  for (int d = 0; d < nr; ++d) {
    B.roff[d] = (u32)off;
    off += column_sum(D.h_small, W_CNT_A + d, nr);
  }
  B.rank_off = B.roff[me];
  const u64 m_total = off;
  B.roff[nr] = (u32)m_total;
  for (int d = nr + 1; d <= DIST_MAX_RANKS; ++d) B.roff[d] = 0xFFFFFFFFu;
  CK(cudaMemcpyAsync(B.roff_dev, B.roff, (nr + 1) * sizeof(u32), cudaMemcpyHostToDevice, st));  // (pageable source: staged at once)
  B.m_total = m_total, B.n_total_loaded = loaded_total;
  const u32 m = (u32)B.ex1.n_recv;
  B.m_loc = m;

  CK(cudaEventRecord(ev[2], st));
  // processing order: sources arrive in file order, so a stable sort by xStart/10 is the global order
  // the sort keys are taken relative to the rank's first xStart/10 bucket: log2(range of the rank) bits instead of log2(vsize)
  const KeyRange k0 = rank_key_range(D.h_small + (size_t)me * SMALL_WORDS + W_CUTS, me, nr, g.vsize);
  launches += dist_key0_of_rec(B.rec6_arr, m, k0.base, B.key0a, hist_of(0, k0.bits), st);
  launches += launch_sort_pairs(B.key0a, nullptr, B.k0_r, B.aidx_r, D.tmp_k, D.tmp_v, m, k0.bits, D.sort_work, st, &D.cnt->err,
                                m ? D.prehist : nullptr);
  CK(cudaEventRecord(ev[3], st));
  launches += launch_keys(B.aidx_r, m, g, nullptr, linkx, linky, B.xl, B.yl_r, B.ys_r, B.kx2, B.ky, B.identity_r, st,
                          HistOut{nullptr, 0, 0}, HistOut{nullptr, 0, 0}, B.gfidx_r, 1u, B.rec6_arr);
  launches += launch_hkey(B.k0_r, B.ys_r, m, nullptr, st, B.gfidx_r, B.identity_r, B.hfi_r);
  CK(cudaEventRecord(ev[4], st));
  // X halo: fragments whose X super-bucket belongs to a higher rank
  launches += dist_cuts_x(B.cuts0, nr, g, linkx, B.cuts_x, st);
  launches += dist_split_halo(B.kx2, B.xl, m, B.cuts_x, nr, g.nbx, me, B.rank_off, B.halo_send, (u32)B.hcap, B.perm_x, D.tile_cnt,
                              D.d_small + W_CNT_A, st);
  // Y: to the owner of the Y super-bucket range
  const int shift_y = B.bits_y > 12 ? B.bits_y - 12 : 0;
  launches += dist_coarse_hist(B.ky, m, shift_y, 0, 0xFFFFFFFFu, D.hist, st);
  TR(D.tr->all_gather(D.hist, D.hist_all, DIST_BINS * 4, st));
  launches += dist_cuts_from_hist(D.hist_all, DIST_BINS, nr, shift_y, B.cuts_y, st);
  launches += dist_split_axis(B.ky, B.yl_r, m, B.cuts_y, nr, B.rank_off, B.send_rows, B.perm_y, D.tile_cnt, D.d_small + W_CNT_B, st);
  CK(cudaMemcpyAsync(D.d_small + W_CUTS, B.cuts_y, (nr + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(D.d_small + W_CUTSX, B.cuts_x, 2 * nr * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  if (const int rc = dist_gather_counts(ctx)) return rc;  // host sync 2
  if (const int rc = dist_check_small(ctx, true)) return rc;
  B.exh.from_matrix(D.h_small, W_CNT_A, nr, me);
  B.exy.from_matrix(D.h_small, W_CNT_B, nr, me);
  for (int d = 0; d < nr; ++d) {
    const u64 halo_in = column_sum(D.h_small, W_CNT_A + d, nr), y_in = column_sum(D.h_small, W_CNT_B + d, nr);
    u64 halo_out = 0;
    for (int t = 0; t < nr; ++t) halo_out += D.h_small[(size_t)d * SMALL_WORDS + W_CNT_A + t];
    if (halo_in > B.hcap || halo_out > B.hcap)
      return fail(ctx, RK_ERR_NOMEM, "rank %d: %llu halo fragments in / %llu out, the halo capacity is %llu", d,
                  (unsigned long long)halo_in, (unsigned long long)halo_out, (unsigned long long)B.hcap);
    if (y_in > B.cap) return fail(ctx, RK_ERR_NOMEM, "rank %d would own %llu fragments in the Y pass, capacity is %llu rows per rank", d,
                                  (unsigned long long)y_in, (unsigned long long)B.cap);
  }
  B.n_away = (u32)B.exh.n_send, B.n_halo = (u32)B.exh.n_recv, B.m_y = (u32)B.exy.n_recv;
  // Y sort keys relative to the first key of the rank's Y range
  const KeyRange yr = rank_key_range(D.h_small + (size_t)me * SMALL_WORDS + W_CUTS, me, nr, 2ull * g.nby);

  // Both row exchanges come right after host sync 2: every rank's work queued before it is complete, so no rank still
  // reads its halo_recv / recv_rows (last read by the previous load and group) when the peers' pushes start.
  TR(D.tr->exchange_rows(B.halo_send, B.exh, B.halo_recv, 16, st));
  // the Y rows travel (copy engines, NVLink) while this GPU unpacks its halo and sorts its X buckets
  TR(D.tr->exchange_rows_begin(B.send_rows, B.exy, D.recv_rows, 16, st, D.side));
  // X sort keys relative to the first super-bucket of the rank's range (per strand class)
  const u32 *cutsx_h = D.h_small + (size_t)me * SMALL_WORDS + W_CUTSX;
  u32 x_base[2], x_range[2];
  for (int sc = 0; sc < 2; ++sc) {
    x_base[sc] = cutsx_h[sc * nr + me];
    const u32 end = me + 1 < nr ? cutsx_h[sc * nr + me + 1] : (u32)(sc + 1) * g.nbx;
    x_range[sc] = end > x_base[sc] ? end - x_base[sc] : 1u;
  }
  const u32 x_R = std::max(x_range[0], x_range[1]);
  const int bits_x_l = ceil_log2(4ull * ((u64)x_R + 1));
  launches += dist_x_local_keys(B.kx2, m, g.nbx, x_base, x_range, hist_of(1, bits_x_l), st);
  launches += dist_unpack_halo_rows(B.halo_recv, B.n_halo, g.nbx, x_base, x_range, B.kx2 + m, B.xl + m, B.halo_grank, hist_of(1, bits_x_l), st);
  CK(cudaEventRecord(ev[5], st));
  launches += launch_sort_pairs(B.kx2, nullptr, B.skx, B.rx, D.tmp_k, D.tmp_v, (u64)m + B.n_halo, bits_x_l, D.sort_work, st, &D.cnt->err,
                                (m + B.n_halo) ? D.prehist + 1024 : nullptr);
  CK(cudaEventRecord(ev[6], st));
  TR(D.tr->exchange_rows_end(st));
  launches += dist_unpack_axis_rows(D.recv_rows, B.m_y, yr.base, B.ky_a, B.yl_a, B.grank_a, hist_of(2, yr.bits), st);
  launches += launch_sort_pairs(B.ky_a, nullptr, B.sky_a, B.ry_a, D.tmp_k, D.tmp_v, B.m_y, yr.bits, D.sort_work, st, &D.cnt->err,
                                B.m_y ? D.prehist + 2048 : nullptr);
  CK(cudaEventRecord(ev[7], st));
  B.loaded = true;

  if (stats) {
    memset(stats, 0, sizeof *stats);
    stats->n_loaded = loaded_total;
    stats->n_kept = m_total;
    stats->vsize = g.vsize;
    stats->n_launches = launches;
    if (flags & RK_F_TIMING) {
      CK(cudaStreamSynchronize(st));
      stats->ms_stage[RK_ST_H2D] = ev_ms(ev[0], ev[1]);
      stats->ms_stage[RK_ST_DECODE] = ev_ms(ev[1], ev[2]);  // K1 + exchange 1
      stats->ms_stage[RK_ST_RANKSORT] = ev_ms(ev[2], ev[3]);
      stats->ms_stage[RK_ST_KEYS] = ev_ms(ev[3], ev[4]);
      stats->ms_stage[RK_ST_XSORT] = ev_ms(ev[4], ev[6]);   // routing of both axes, halo exchange, X sort
      stats->ms_stage[RK_ST_YSORT] = ev_ms(ev[6], ev[7]);   // Y exchange + Y sort
      stats->ms_device = ev_ms(ev[1], ev[7]);
    }
  }
  return RK_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// load from text: FragmentsDatabase's row loop (src/FragmentsDatabase.cpp:91-100) over the ranks, each rank parsing its slice
// ---------------------------------------------------------------------------------------------------------------------
// The local half of rk_dist_load_csv: rk_load_csv's parse of this rank's slice, up to the host rows.  Needs no other
// rank and no partition buffers (rk_multi_load_csv sizes them from its result).  A failure is kept in the state, not
// returned: it travels to every rank in the count exchange of the collective half.
struct DistCsv {
  CsvParse p;
  int rc = RK_OK;
  std::string err;
  bool nl_end = false;  // the slice ends with '\n'
};
static void dist_csv_local(rk_ctx *ctx, const char *slice, u64 bytes, int threads, DistCsv &L) {
  L = DistCsv{};
  ctx->loaded = ctx->have_group = false;
  if (ctx->dist) ctx->dist->db->loaded = ctx->dist->have_rows = false;
  auto run = [&]() -> int {
    if (!slice && bytes) return fail(ctx, RK_ERR_ARG, "null text pointer");
    CK(cudaSetDevice(ctx->device));
    ProfGuard pg(ctx);
    if (const int rc = csv_parse_local(ctx, slice, bytes, threads, L.p)) return rc;
    if (bytes) {
      char last = 0;
      if (L.p.on_device) CK(cudaMemcpy(&last, slice + bytes - 1, 1, cudaMemcpyDeviceToHost));
      else last = slice[bytes - 1];
      L.nl_end = last == '\n';
    }
    return RK_OK;
  };
  L.rc = run();
  if (L.rc) L.err = ctx->err;
}

// the count exchange of rk_dist_load_csv: one row of CW_WORDS per rank; a rank whose local half failed sends the start of
// its error message in the CW_MSG words, so that every rank returns the same text
enum { CW_ACC, CW_NL, CW_FLAGS, CW_RC, CW_MSG, CW_WORDS = CW_MSG + 28 };
static_assert(CW_WORDS <= SMALL_WORDS, "the count row fits the rows of d_small");
constexpr u32 CWF_WIDE = 1, CWF_BYTES = 2, CWF_NL_END = 4, CWF_ROWS = 8;  // CWF_ROWS: more than 2^32-16 rows in the slice

// The collective half: the counts of every rank, the verdicts every rank reaches from them, this rank's file offset,
// the emit into Dist::aos_buf and dist_load on it.
static int dist_csv_finish(rk_ctx *ctx, DistCsv &L, u64 seqx_len, u64 seqy_len, u64 total_frags, unsigned flags, rk_load_stats *stats,
                           rk_csv_stats *csv) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  const int nr = D.world, me = D.rank;
  if (!D.peers_ready) return fail(ctx, RK_ERR_STATE, "rk_dist_load_csv before rk_dist_import");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const CsvParse &p = L.p;
  u32 row[CW_WORDS] = {0, 0, 0, (u32)L.rc};
  if (L.rc) {
    if (L.rc == RK_ERR_ARG && p.n_rows >= 0xFFFFFFF0ull) row[CW_FLAGS] |= CWF_ROWS;
    memcpy(&row[CW_MSG], L.err.c_str(), std::min<size_t>(L.err.size(), (CW_WORDS - CW_MSG) * 4 - 1));  // (row is zeroed: terminated)
  } else {
    row[CW_ACC] = (u32)p.n_accepted();
    row[CW_NL] = (u32)(p.n_rows - 1);
    row[CW_FLAGS] = (p.wide ? CWF_WIDE : 0) | (p.bytes ? CWF_BYTES : 0) | (L.nl_end ? CWF_NL_END : 0);
  }
  CK(cudaMemcpyAsync(D.d_small, row, sizeof row, cudaMemcpyHostToDevice, st));  // (pageable source: staged at once)
  TR(D.tr->all_gather(D.d_small, D.d_small_all, sizeof row, st));
  std::vector<u32> all((size_t)nr * CW_WORDS);
  CK(cudaMemcpyAsync(all.data(), D.d_small_all, all.size() * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  auto W = [&](int r, int w) { return all[(size_t)r * CW_WORDS + w]; };
  // every rank sees the same words, so every rank reaches the same verdict
  int last = -1;  // the last rank with a non-empty slice
  for (int r = 0; r < nr; ++r)
    if (W(r, CW_FLAGS) & CWF_BYTES) last = r;
  for (int r = 0; r < nr; ++r) {
    if (!W(r, CW_RC)) continue;
    if (W(r, CW_FLAGS) & CWF_ROWS) return fail(ctx, RK_ERR_ARG, "rank %d: more than 2^32-16 rows in its slice of the text", r);
    return fail(ctx, (int)W(r, CW_RC), "rank %d could not parse its slice of the text: %s", r,
                (const char *)&all[(size_t)r * CW_WORDS + CW_MSG]);
  }
  for (int r = 0; r < last; ++r)
    if ((W(r, CW_FLAGS) & CWF_BYTES) && !(W(r, CW_FLAGS) & CWF_NL_END))
      return fail(ctx, RK_ERR_ARG, "rank %d: its slice of the text does not end with '\\n' (every slice before the last must end a row)", r);
  u64 total = 0, file_off = 0;
  for (int r = 0; r < nr; ++r) {
    if (r == me) file_off = total;
    total += W(r, CW_ACC);
  }
  if (total > total_frags) return fail(ctx, RK_ERR_RANGE, "Unexpected number of fragments");  // FragmentsDatabase.cpp:99
  if (total >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 records in one comparison");
  for (int r = 0; r < nr; ++r)
    if (W(r, CW_ACC) > B.cap)
      return fail(ctx, RK_ERR_NOMEM, "a rank holds more records than the capacity of %llu rows per rank given to rk_dist_init",
                  (unsigned long long)B.cap);
  // the final row of the text (the empty one after a final '\n') is the last slice's; every other slice ends with '\n',
  // and the empty segment after it is no row
  const int holder = (last >= 0 && !(W(last, CW_FLAGS) & CWF_NL_END)) ? last : nr - 1;
  const u64 n_rows = (u64)W(me, CW_NL) + (holder == me ? 1 : 0);

  CsvOut o;
  {
    ProfGuard pg(ctx);
    if (const int rc = csv_emit(ctx, p, B.aos_buf, &o)) return rc;
  }
  const PackedRows pk{o.key4, o.rest4, o.strand};
  const u64 n_acc = p.n_accepted();
  if (const int rc = dist_load(ctx, o.aos, n_acc, file_off, seqx_len, seqy_len, flags, stats, o.aos ? nullptr : &pk)) return rc;
  CK(cudaStreamSynchronize(st));
  cudaEvent_t *ev = ctx->ev;
  const float ms_up = p.on_device ? 0.f : ev_ms(ev[EV_CSV_UP0], ev[EV_CSV_UP1]), ms_parse = ev_ms(ev[EV_CSV_UP1], ev[EV_CSV_PARSED]);
  if (stats && (flags & RK_F_TIMING)) stats->ms_stage[RK_ST_H2D] = ms_up;
  if (csv) {
    memset(csv, 0, sizeof *csv);
    csv->n_rows = n_rows, csv->n_accepted = n_acc, csv->n_host_rows = p.n_host, csv->wide = p.wide;
    csv->ms_upload = ms_up;
    csv->ms_parse = ms_parse;
  }
  return RK_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// load from compact arrays: rk_load_packed over the ranks
// ---------------------------------------------------------------------------------------------------------------------
// the device of a device pointer; -1 for host memory of any kind
static int device_of(const void *p) {
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, p) == cudaSuccess && pa.type == cudaMemoryTypeDevice) return pa.device;
  cudaGetLastError();
  return -1;
}

// the status row of rk_dist_load_packed, gathered before anything is copied or loaded: a rank whose own checks failed
// sends its code and the start of its message, so that every rank returns the same code and text
enum { PW_RC, PW_NO_REST, PW_MSG, PW_WORDS = PW_MSG + 28 };
static_assert(PW_WORDS <= SMALL_WORDS, "the status row fits the rows of d_small");

// The rank-local checks of rk_dist_load_packed and, for host arrays, the staging area in aos_buf (key4, rest4, strand as
// csv_emit places them).  Touches no peer; the verdict travels in the status row.
static int dist_packed_local(rk_ctx *ctx, const u32 *key4, const u8 *strand, const u32 *rest4, u64 n, u64 file_off, u64 seqx_len,
                             u64 seqy_len, PackedRows *pk) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  if (!D.peers_ready) return fail(ctx, RK_ERR_STATE, "rk_dist_load_packed before rk_dist_import");
  if (seqx_len >= (1ull << 32) || seqy_len >= (1ull << 32)) return fail(ctx, RK_ERR_RANGE, "sequence length does not fit in 32 bits");
  if (file_off + n >= 0xFFFFFFF0ull) return fail(ctx, RK_ERR_ARG, "more than 2^32-16 records in one comparison");
  if (n > B.cap)
    return fail(ctx, RK_ERR_NOMEM, "a rank holds more records than the capacity of %llu rows per rank given to rk_dist_init",
                (unsigned long long)B.cap);
  *pk = PackedRows{};
  if (!n) return RK_OK;
  if (!key4 || !strand) return fail(ctx, RK_ERR_ARG, "null array");
  const int dev = device_of(key4);
  if (device_of(strand) != dev || (rest4 && device_of(rest4) != dev))
    return fail(ctx, RK_ERR_ARG, "the arrays of rk_dist_load_packed must all be host or all be device memory");
  if (dev >= 0) {
    if (dev != ctx->device) return fail(ctx, RK_ERR_ARG, "the arrays are on device %d, this rank's context on device %d", dev, ctx->device);
    if (((uintptr_t)key4 & 15) || ((uintptr_t)rest4 & 15)) return fail(ctx, RK_ERR_ARG, "device arrays key4 and rest4 must be 16-byte aligned");
    *pk = PackedRows{(const uint4 *)key4, (const uint4 *)rest4, strand};
    return RK_OK;
  }
  CK(cudaSetDevice(ctx->device));
  if (const int rc = B.aos_buf.reserve(csv_out_bytes(n, false), ctx->stream, ctx->err)) {
    const std::string e = ctx->err;
    return fail(ctx, rc, "rk_dist_load_packed: %llu rows: %s", (unsigned long long)n, e.c_str());
  }
  const u64 key_b = align_up(n * 16, 256);
  u8 *ob = (u8 *)B.aos_buf.ptr();
  *pk = PackedRows{(const uint4 *)ob, rest4 ? (const uint4 *)(ob + key_b) : nullptr, ob + 2 * key_b};
  return RK_OK;
}

// rk_dist_load_packed: the local checks, one status all-gather (every rank reaches the same verdict), then the copies of
// host arrays — key4 and strand on the context's stream before K1, rest4 on the database's copy stream beside the load's
// kernels — and dist_load on the compact rows.  Every copy has finished when this returns, whatever the outcome.
static int dist_load_packed(rk_ctx *ctx, const u32 *key4, const u8 *strand, const u32 *rest4, u64 n, u64 file_off, u64 seqx_len,
                            u64 seqy_len, unsigned flags, rk_load_stats *stats) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  B.loaded = false;
  B.aos_src = nullptr, B.pk_src = PackedRows{};
  D.have_rows = false;
  ctx->loaded = ctx->have_group = false;
  PackedRows pk;
  const int lrc = dist_packed_local(ctx, key4, strand, rest4, n, file_off, seqx_len, seqy_len, &pk);
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  u32 row[PW_WORDS] = {(u32)lrc, (u32)(n && !rest4)};
  if (lrc) memcpy(&row[PW_MSG], ctx->err.c_str(), std::min<size_t>(ctx->err.size(), (PW_WORDS - PW_MSG) * 4 - 1));
  CK(cudaMemcpyAsync(D.d_small, row, sizeof row, cudaMemcpyHostToDevice, st));  // (pageable source: staged at once)
  TR(D.tr->all_gather(D.d_small, D.d_small_all, sizeof row, st));
  std::vector<u32> all((size_t)D.world * PW_WORDS);
  CK(cudaMemcpyAsync(all.data(), D.d_small_all, all.size() * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  int no_rest = -1;
  for (int r = 0; r < D.world; ++r) {
    const u32 *w = &all[(size_t)r * PW_WORDS];
    if (w[PW_RC]) return fail(ctx, (int)w[PW_RC], "rank %d: %s", r, (const char *)&w[PW_MSG]);
    if (w[PW_NO_REST] && no_rest < 0) no_rest = r;
  }
  const bool staged = n && pk.key != (const uint4 *)key4;
  cudaEvent_t *ev = ctx->ev;
  Database &db = *ctx->db;
  if (staged) {
    CK(cudaEventRecord(ev[EV_PK_UP0], st));
    CK(cudaMemcpyAsync((void *)pk.key, key4, n * 16, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync((void *)pk.strand, strand, n, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ev[EV_PK_UP1], st));
    if (rest4) {  // only the line records read it: it travels while K1 and the exchanges run
      CK(cudaStreamWaitEvent(db.copy_stream, ev[EV_PK_UP0], 0));  // (after the work queued on st is done with aos_buf)
      CK(cudaMemcpyAsync((void *)pk.rest, rest4, n * 16, cudaMemcpyHostToDevice, db.copy_stream));
      CK(cudaEventRecord(ev[EV_PK_REST], db.copy_stream));
    }
  }
  const int rc = dist_load(ctx, nullptr, n, file_off, seqx_len, seqy_len, flags, stats, &pk);
  // the caller may overwrite or free its arrays once this returns: wait for every copy, on success and failure alike
  const cudaError_t e1 = staged ? cudaEventSynchronize(ev[EV_PK_UP1]) : cudaSuccess;
  const cudaError_t e2 = staged && rest4 ? cudaEventSynchronize(ev[EV_PK_REST]) : cudaSuccess;
  if (rc) return rc;
  CK(e1);
  CK(e2);
  B.rest_missing = no_rest;
  if (stats && (flags & RK_F_TIMING))
    stats->ms_stage[RK_ST_H2D] = !staged ? 0.f : std::max(ev_ms(ev[EV_PK_UP0], ev[EV_PK_UP1]), rest4 ? ev_ms(ev[EV_PK_UP0], ev[EV_PK_REST]) : 0.f);
  return RK_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// group: generate_fragment_groups + generate_diagonal_func + sort_groups over the ranks
// ---------------------------------------------------------------------------------------------------------------------
static int dist_group(rk_ctx *ctx, double len_ratio, double pos_ratio, unsigned flags, rk_result *out, rk_dist_info *info) {
  Dist &D = *ctx->dist;
  DistDb &B = *D.db;
  const int nr = D.world, me = D.rank;
  if (!B.loaded) return fail(ctx, RK_ERR_STATE, "rk_dist_group before a successful rk_dist_load_aos");
  if (!D.peers_ready) return fail(ctx, RK_ERR_STATE, "rk_dist_group before rk_dist_import");
  if (!(len_ratio > 0)) return fail(ctx, RK_ERR_ARG, "Ratio between length and position must be greater than zero");
  if (!(pos_ratio > 0)) return fail(ctx, RK_ERR_ARG, "Position proximity must be greater than zero");
  if ((flags & RK_F_LINE_RECORDS) && !B.slices_in_order)
    return fail(ctx, RK_ERR_ARG, "RK_F_LINE_RECORDS needs the ranks' slices of the file in rank order (file_offset of rk_dist_load_aos)");
  if ((flags & RK_F_LINE_RECORDS) && B.rest_missing >= 0)
    return fail(ctx, RK_ERR_ARG, "RK_F_LINE_RECORDS needs the xEnd/yEnd/score/similarity array: rank %d loaded its compact rows without rest4",
                B.rest_missing);
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  memset(out, 0, sizeof *out);
  cudaStream_t st = ctx->stream;
  cudaEvent_t *ev = ctx->ev;
  const u32 m = B.m_loc, nh = B.n_halo, mc = m + nh;
  memcpy(D.pt.roff, B.roff, sizeof B.roff);
  u64 launches = 0;
  const u64 sent0 = D.tr->bytes_sent;
  const bool line_records = (flags & RK_F_LINE_RECORDS) != 0;
  D.have_rows = false;
  CK(cudaMemsetAsync(D.d_small, 0, SMALL_WORDS * 4, st));

  CK(cudaEventRecord(ev[0], st));
  // X pass at home over [own fragments ++ halo]
  MatchArgs mx{};
  mx.skey = B.skx, mx.srank = B.rx, mx.cl_r = B.xl, mx.parent = D.parent_x, mx.xm_bits = D.xm_bits;
  mx.m = mc, mx.max_index = B.g.mx, mx.len_ratio = len_ratio, mx.pos_ratio = pos_ratio, mx.is_y = 0;
  mx.worklist = D.worklist, mx.work_count = D.cnt->work_x, mx.work_cap = D.work_cap;
  mx.ent_rank = D.ent_rank, mx.ent_c = D.ent_c, mx.ent_len = D.ent_len, mx.err = &D.cnt->err;
  mx.key_shift = 1;
  launches += launch_match(mx, st);
  launches += dist_x_owners(D.parent_x, m, nh, B.rank_off, B.halo_grank, D.parent, scatter_table(D, B.exh, true, D.away_res), st);
  TR(D.tr->barrier(st));  // the halo owners are stored by the kernel above straight into their home ranks' away_res
  launches += dist_apply_away(D.away_res, B.perm_x, B.n_away, D.parent, st);
  CK(cudaEventRecord(ev[1], st));
  // Y pass on the owners of the Y ranges: X-matched fragments insert without a query (commonFunctions.cpp:59)
  launches += dist_pack_xm(D.parent, B.perm_y, m, scatter_table(D, B.exy, false, D.xm_a), st);
  if (m) CK(cudaMemsetAsync(D.yo_s, 0xFF, (size_t)m * 4, st));  // "no Y owner" until a peer stores one (after the barrier)
  TR(D.tr->barrier(st));
  if (B.m_y) CK(cudaMemsetAsync(D.parent_y, 0xFF, (size_t)B.m_y * 4, st));
  MatchArgs my = mx;
  my.skey = B.sky_a, my.srank = B.ry_a, my.cl_r = B.yl_a, my.parent = D.parent_y, my.m = B.m_y, my.max_index = B.g.my, my.is_y = 1;
  my.work_count = D.cnt->work_y, my.key_shift = 0, my.xm_bytes = D.xm_a;
  launches += launch_match(my, st);
  launches += dist_y_owners(D.parent_y, B.grank_a, B.m_y, scatter_table(D, B.exy, true, D.yo_s), st);
  TR(D.tr->barrier(st));
  launches += dist_merge_y(D.yo_s, B.perm_y, m, D.parent, st);
  CK(cudaEventRecord(ev[2], st));
  // forest: roots per rank; local chains; the chains that leave the GPU are resolved in bulk rounds while there are many
  // of them anywhere, the rest by walking through the peers' memory (k7_dist.cu)
  launches += dist_root_scan(D.parent, m, D.gidscan, D.d_small + W_X0, D.scan_work, st);
  launches += dist_chase_local(D.parent, D.gidscan, m, B.rank_off, D.lroot, D.res, D.pend_idx[0], D.pend_key[0], D.n_pend, st);
  CK(cudaMemcpyAsync(D.d_small + W_X2, D.n_pend, sizeof(u32), cudaMemcpyDeviceToDevice, st));
  // host sync: roots and pending chains of every rank (also: every rank's res[] is final)
  if (const int rc = dist_gather_counts(ctx)) return rc;
  // the root counts stay on the device as a column of the gathered matrix, in a copy that later gathers do not overwrite
  CK(cudaMemcpyAsync(D.nroots_mat, D.d_small_all, (size_t)nr * SMALL_WORDS * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  const u32 *nroots = D.nroots_mat + W_X0;
  // (RK_DIST_BULK_MIN: tuning and tests — 1 resolves every chain in bulk rounds, a huge value only by walking)
  const u64 bulk_min = getenv("RK_DIST_BULK_MIN") ? strtoull(getenv("RK_DIST_BULK_MIN"), nullptr, 10) : (1ull << 20);
  int cur = 0;
  for (int round = 0; round < nr; ++round) {
    u64 most = 0;
    for (int r = 0; r < nr; ++r) most = std::max<u64>(most, D.h_small[(size_t)r * SMALL_WORDS + W_X2]);
    if (most == 0 || most < bulk_min) break;
    const u32 bound = (u32)std::min<u64>(D.h_small[(size_t)me * SMALL_WORDS + W_X2], m);  // this rank's pending chains
    // ask: the ranks in question go to their owners
    uint4 *qouts[DIST_MAX_RANKS];
    D.tr->peer_table(D.queries, qouts);
    launches += dist_chase_ask_count(D.pend_key[cur], bound, D.n_pend, B.roff_dev, nr, D.tile_cnt, D.d_small + W_CNT_A, st);
    if (const int rc = dist_gather_counts(ctx, [&] {
          launches += dist_chase_ask_push(D.pend_key[cur], bound, D.n_pend, B.roff_dev, nr, qouts, (u32)B.cap, D.apos, D.tile_cnt,
                                          D.d_small_all, SMALL_WORDS, me, st);
        }))
      return rc;
    if (const int rc = check_inbound(ctx, W_CNT_A, B.cap, "rank %d is asked about %llu chain ends, capacity is %llu rows per rank")) return rc;
    Exchange exq;
    exq.from_matrix(D.h_small, W_CNT_A, nr, me);
    D.tr->bytes_sent += (exq.n_send - exq.scnt[me]) * 16 + (exq.n_recv - exq.rcnt[me]) * 8;
    // answer: every owner returns its res[] words, block by block, into the asking ranks' answer buffers
    launches += dist_chase_answer(D.queries, (u32)exq.n_recv, D.res, B.rank_off, scatter_table(D, exq, true, D.answers), st);
    TR(D.tr->barrier(st));
    // apply: roots end a chain, anything else is asked about in the next round
    launches += dist_chase_apply(D.pt, nroots, SMALL_WORDS, bound, D.pend_idx[cur], D.pend_key[cur], D.apos, D.answers, D.n_pend, D.gid_l,
                                 D.pend_idx[cur ^ 1], D.pend_key[cur ^ 1], D.n_pend + 1, st);
    CK(cudaMemcpyAsync(D.n_pend, D.n_pend + 1, sizeof(u32), cudaMemcpyDeviceToDevice, st));
    cur ^= 1;
    CK(cudaMemcpyAsync(D.d_small + W_X2, D.n_pend, sizeof(u32), cudaMemcpyDeviceToDevice, st));
    if (const int rc = dist_gather_counts(ctx)) return rc;  // how many chains are still open, everywhere
  }
  launches += dist_chase_finish(D.pt, nroots, SMALL_WORDS, m, D.res, D.lroot, D.pend_idx[cur], D.pend_key[cur], D.n_pend, D.gid_l, D.gid_rank, st);
  // (no second barrier: the count exchange of the output stage below completes on a rank only after every rank has
  // entered it, i.e. finished chasing, and parent[] is not written again before the next rk_dist_group)
  CK(cudaEventRecord(ev[3], st));
  // output exchange: to the owner of the group-id range.  The ranges are cut for about equal sort_groups WORK: lines, with
  // the lines of groups with several members weighted up (groups founded early are the large ones: equal numbers of
  // groups gave rank 0 far more lines, equal numbers of lines still far more work — see k_cuts_from_hist).
  const int bits_gid = key_bits(B.m_total);  // group ids are < number of fragments
  const int shift_g = bits_gid > 12 ? bits_gid - 12 : 0;
  launches += dist_cuts_gid(nroots, SMALL_WORDS, nr, D.cuts_g, D.d_small + W_X1, st);  // (the total; the cuts are replaced below)
  launches += dist_coarse_hist(D.gid_rank, m, shift_g, 0, 0xFFFFFFFFu, D.hist, st);
  TR(D.tr->all_gather(D.hist, D.hist_all, DIST_BINS * 4, st));
  // no range may hold more lines than a rank has rows (RK_DIST_LINE_CAP: tests — a tighter bound than the capacity)
  const u64 line_cap = getenv("RK_DIST_LINE_CAP") ? std::min<u64>(B.cap, strtoull(getenv("RK_DIST_LINE_CAP"), nullptr, 10)) : B.cap;
  launches += dist_cuts_from_hist(D.hist_all, DIST_BINS, nr, shift_g, D.cuts_g, st, D.d_small + W_X1, line_cap);
  CK(cudaMemcpyAsync(D.d_small + W_CNT_B, D.cuts_g, (nr + 1) * sizeof(u32), cudaMemcpyDeviceToDevice, st));
  uint4 *outs[DIST_MAX_RANKS];
  D.tr->peer_table(D.recv_rows, outs);
  launches += dist_count_plain(D.gid_rank, m, D.cuts_g, nr, 0xFFFFFFFFu, D.tile_cnt, D.d_small + W_CNT_A, st);
  if (const int rc = dist_gather_counts(ctx, [&] {  // host sync 3
        launches += dist_push_gid(D.gid_rank, B.hfi_r, m, D.cuts_g, nr, outs, (u32)B.cap, D.tile_cnt, D.d_small_all, SMALL_WORDS, me, st);
      }))
    return rc;
  if (const int rc = dist_check_small(ctx, false)) return rc;
  if (const int rc = check_inbound(ctx, W_CNT_A, B.cap, "rank %d would own %llu output lines, capacity is %llu rows per rank")) return rc;
  Exchange exg;
  exg.from_matrix(D.h_small, W_CNT_A, nr, me);
  D.tr->bytes_sent += (exg.n_send - exg.scnt[me]) * 16;
  const u64 total_groups = D.h_small[(size_t)me * SMALL_WORDS + W_X1];
  u64 line_off = 0;
  for (int d = 0; d < me; ++d) line_off += column_sum(D.h_small, W_CNT_A + d, nr);
  const u32 mg = (u32)exg.n_recv;
  const KeyRange gr = rank_key_range(D.h_small + (size_t)me * SMALL_WORDS + W_CNT_B, me, nr, total_groups);
  CK(cudaMemsetAsync(D.prehist + 3072, 0, 4 * 256 * 4, st));
  launches += dist_gid_keys(D.recv_rows, mg, gr.base, D.gid_a, HistOut{D.prehist + 3072, (gr.bits + 7) / 8, gr.bits}, st);
  CK(cudaEventRecord(ev[4], st));
  // members arrive in processing order (sources in rank order): a stable sort by group id is push_back order
  launches += launch_sort_pairs(D.gid_a, nullptr, D.sgid, D.srank_g, D.tmp_k, D.tmp_v, mg, gr.bits, D.sort_work, st, &D.cnt->err,
                                mg ? D.prehist + 3072 : nullptr);
  OrderArgs oa{};
  oa.sgid = D.sgid, oa.srank = D.srank_g, oa.hfi_r = D.recv_rows;
  oa.m = mg, oa.do_sort = (flags & RK_F_NO_SORT) ? 0 : 1, oa.gid_base = gr.base;
  order_carve(oa, D.order_scratch, B.cap);
  oa.work_count = D.cnt->work_g;
  oa.out_order = D.out_order, oa.out_gid = D.out_gid, oa.out_repval = D.out_repval, oa.out_identity = D.out_identity;
  oa.err = &D.cnt->err;
  launches += launch_order(oa, st);
  CK(cudaEventRecord(ev[5], st));
  // line records: every line asks the rank that loaded its record for what the line prints, and that rank stores the
  // 64-byte row straight into line_rows[line] here.  A bulk round of the forest in form: a count exchange, the requests
  // pushed into the owners' `queries` (free again: the forest is done), the answers stored back by the owners' kernel,
  // a barrier.  The gid cuts are spent, so cuts_g carries the slice starts.
  if (line_records) {
    CK(cudaMemcpyAsync(D.cuts_g, B.file_off, nr * sizeof(u32), cudaMemcpyHostToDevice, st));  // (pageable source: staged at once)
    uint4 *qouts[DIST_MAX_RANKS];
    D.tr->peer_table(D.queries, qouts);
    launches += dist_count_plain(D.out_order, mg, D.cuts_g, nr, 0xFFFFFFFFu, D.tile_cnt, D.d_small + W_CNT_A, st);
    if (const int rc = dist_gather_counts(ctx, [&] {  // host sync 4
          launches += dist_line_ask_push(D.out_order, mg, D.cuts_g, nr, qouts, (u32)B.cap, D.tile_cnt, D.d_small_all, SMALL_WORDS, me, st);
        }))
      return rc;
    if (const int rc = dist_check_small(ctx, false)) return rc;
    // (a rank is asked only about the records of its slice, which fits its rows)
    if (const int rc = check_inbound(ctx, W_CNT_A, B.cap, "rank %d is asked for %llu line records, capacity is %llu rows per rank")) return rc;
    Exchange exl;
    exl.from_matrix(D.h_small, W_CNT_A, nr, me);
    D.tr->bytes_sent += (exl.n_send - exl.scnt[me]) * 16 + (exl.n_recv - exl.rcnt[me]) * sizeof(LineRow);
    launches += dist_line_answer(D.queries, (u32)exl.n_recv, B.aos_src, B.pk_src, B.file_off[me], scatter_table(D, exl, true, D.line_rows), st);
    TR(D.tr->barrier(st));
    CK(cudaEventRecord(ev[8], st));
  }

  HostResult hr;
  if ((flags & RK_F_HOST_RESULT) && mg) {
    const u64 need = HostResult::bytes(mg);
    const int rc2 = D.h_res.reserve(need > D.h_res.cap() ? need + need / 4 : need, st, ctx->err);
    if (rc2) return rc2;
    hr = HostResult(D.h_res.ptr(), mg);
    CK(cudaEventRecord(ev[6], st));
    CK(hr.fetch(D.out_order, D.out_gid, D.out_identity, D.out_repval, mg, st));
    CK(cudaEventRecord(ev[7], st));
  }
  CK(cudaMemcpyAsync(ctx->h_cnt, D.cnt, sizeof(Counters), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (ctx->h_cnt->err) return fail(ctx, RK_ERR_INTERNAL, "%s", err_bits_text(ctx->h_cnt->err));
  if (D.trace.on) {
    char cb[240];
    snprintf(cb, sizeof cb, "ranked=%u halo_in=%u halo_out=%u y=%u lines=%u groups=%llu stages x=%.3f y=%.3f forest=%.3f exch=%.3f order=%.3f |", m, nh,
             B.n_away, B.m_y, mg, (unsigned long long)total_groups, ev_ms(ev[0], ev[1]), ev_ms(ev[1], ev[2]), ev_ms(ev[2], ev[3]),
             ev_ms(ev[3], ev[4]), ev_ms(ev[4], ev[5]));
    if (line_records) {
      const size_t k = strlen(cb) - 2;  // before the closing " |"
      snprintf(cb + k, sizeof cb - k, " rows=%.3f |", ev_ms(ev[5], ev[8]));
    }
    D.trace.dump(me, cb);
  }
  D.n_lines = mg, D.line_off = line_off;
  D.gid_base = (u32)std::min<u64>(gr.base, total_groups);
  D.n_groups_rank = (u32)(gr.end > D.gid_base ? gr.end - D.gid_base : 0);
  D.have_rows = line_records;

  out->n_kept = mg;
  out->n_groups = total_groups;
  hr.publish(out);
  out->d_order = D.out_order, out->d_gid = D.out_gid, out->d_repval = D.out_repval, out->d_identity = D.out_identity;
  out->n_launches = launches;
  if (flags & RK_F_TIMING) {
    out->ms_stage[RK_ST_XMATCH] = ev_ms(ev[0], ev[1]);
    out->ms_stage[RK_ST_YMATCH] = ev_ms(ev[1], ev[2]);
    out->ms_stage[RK_ST_FOREST] = ev_ms(ev[2], ev[3]);
    out->ms_stage[RK_ST_HKEY] = ev_ms(ev[3], ev[4]);   // output exchange
    out->ms_stage[RK_ST_GSORT] = ev_ms(ev[4], ev[5]);
    if (hr.order) out->ms_stage[RK_ST_D2H] = ev_ms(ev[6], ev[7]);
    out->ms_device = ev_ms(ev[0], line_records ? ev[8] : ev[5]);
  }
  if (info) {
    memset(info, 0, sizeof *info);
    info->rank = me, info->world = nr;
    info->total_loaded = B.n_total_loaded;
    info->total_kept = B.m_total;
    info->total_groups = total_groups;
    info->line_offset = line_off;
    info->n_lines = mg;
    info->rank_offset = B.rank_off;
    info->n_ranked = m;
    info->n_halo_in = nh;
    info->n_halo_out = B.n_away;
    info->n_y = B.m_y;
    info->bytes_sent = D.tr->bytes_sent - sent0;
  }
  return RK_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// output of a rank from its line rows: K6 and K8 as on one GPU (no collective step)
// ---------------------------------------------------------------------------------------------------------------------
static int dist_rows_ready(rk_ctx *ctx, const char *what) {
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "%s before rk_dist_init", what);
  if (!ctx->dist->have_rows) return fail(ctx, RK_ERR_STATE, "%s needs the last rk_dist_group to have RK_F_LINE_RECORDS", what);
  return RK_OK;
}

// K6 over local lines first_line .. first_line+n_lines of the last grouping, into the context's device text buffer
static int dist_format_device(rk_ctx *ctx, u64 first_line, u64 n_lines, u64 *nbytes) {
  const int rc = dist_rows_ready(ctx, "rk_dist_format_lines");
  if (rc) return rc;
  const Dist &D = *ctx->dist;
  if (first_line > D.n_lines || n_lines > D.n_lines - first_line)
    return fail(ctx, RK_ERR_ARG, "line range beyond the %u output lines of rank %d", D.n_lines, D.rank);
  if (n_lines > RK_FORMAT_MAX_LINES) return fail(ctx, RK_ERR_ARG, "at most %llu lines per call", (unsigned long long)RK_FORMAT_MAX_LINES);
  FormatArgs fa{};
  fa.rows = D.line_rows;
  fa.order = D.out_order, fa.gid = D.out_gid, fa.repval = D.out_repval, fa.identity = D.out_identity;
  fa.first_line = (u32)first_line, fa.n_lines = (u32)n_lines;
  return format_on_device(ctx, fa, nbytes);
}

static int dist_group_stats(rk_ctx *ctx, unsigned flags) {
  const int rc = dist_rows_ready(ctx, "rk_dist_group_statistics");
  if (rc) return rc;
  const Dist &D = *ctx->dist;
  return group_stats_run(ctx, flags, D.out_order, D.out_gid, D.out_identity, nullptr, D.line_rows, D.n_lines, D.n_groups_rank, D.gid_base,
                         (u32)D.line_off);
}

void dist_destroy(rk_ctx *c) {
  if (!c || !c->dist) return;
  Dist *D = c->dist;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  dist_release_peers(*D);
  if (D->side) cudaStreamSynchronize(D->side), cudaStreamDestroy(D->side);
  delete D->tr;
  if (--D->db->refs == 0) delete D->db;  // the partition database stays while other contexts of it are live
  delete D;
  c->dist = nullptr;
}

}  // namespace rk

// ---------------------------------------------------------------------------------------------------------------------
// C ABI: one process per GPU
// ---------------------------------------------------------------------------------------------------------------------
extern "C" {

int rk_dist_unique_id(void *id128) {
  if (!id128) return RK_ERR_ARG;
  NcclApi &N = nccl_api();
  if (!N.ok()) return RK_ERR_CUDA;
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == RK_DIST_ID_BYTES, "unique id size");
  if (N.GetUniqueId(&id) != ncclSuccess) return RK_ERR_CUDA;
  memcpy(id128, &id, sizeof id);
  return RK_OK;
}

int rk_dist_init(rk_ctx *ctx, int rank, int nranks, const void *id128, uint64_t cap_per_rank) {
  if (!ctx || !id128) return RK_ERR_ARG;
  if (const int rc = dist_init_refusal(ctx)) return rc;  // (before the communicator: every rank refuses alike)
  NcclApi &N = nccl_api();
  if (!N.ok()) return fail(ctx, RK_ERR_CUDA, "NCCL is not available: %s", N.err.c_str());
  CK(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  NcclTransport *tr = new NcclTransport;
  const ncclResult_t r = N.CommInitRank(&tr->comm, nranks, id, rank);
  if (r != ncclSuccess) {
    const int rc = fail(ctx, RK_ERR_CUDA, "ncclCommInitRank: %s", N.GetErrorString(r));
    tr->comm = nullptr;
    delete tr;
    return rc;
  }
  return dist_init_common(ctx, rank, nranks, tr, cap_per_rank);
}

rk_ctx *rk_dist_create_view(rk_ctx *base, const void *id128) {
  if (!id128) {
    set_create_error("rk_dist_create_view: null unique id");
    return nullptr;
  }
  // the refusals before the communicator starts: every rank's base is in the same state, so every rank refuses alike
  if (const char *why = dist_view_refusal(base)) {
    set_create_error(std::string("rk_dist_create_view: ") + why);
    return nullptr;
  }
  NcclApi &N = nccl_api();
  if (!N.ok()) {
    set_create_error("rk_dist_create_view: NCCL is not available: " + N.err);
    return nullptr;
  }
  const Dist &S = *base->dist;
  if (cudaSetDevice(base->device) != cudaSuccess) {
    cudaGetLastError();
    set_create_error("rk_dist_create_view: cudaSetDevice failed");
    return nullptr;
  }
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  NcclTransport *tr = new NcclTransport;
  const ncclResult_t r = N.CommInitRank(&tr->comm, S.world, id, S.rank);
  if (r != ncclSuccess) {
    tr->comm = nullptr;
    delete tr;
    set_create_error(std::string("rk_dist_create_view: ncclCommInitRank: ") + N.GetErrorString(r));
    return nullptr;
  }
  std::string err;
  rk_ctx *v = dist_view_create(base, tr, err);
  if (!v) {
    set_create_error("rk_dist_create_view: " + err);
    return nullptr;
  }
  return v;
}

int rk_dist_export(rk_ctx *ctx, void *blob) {
  if (!ctx || !blob) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_export before rk_dist_init");
  memset(blob, 0, RK_DIST_BLOB_BYTES);
  return dist_export(ctx, (DistBlob *)blob);
}

int rk_dist_import(rk_ctx *ctx, const void *blobs) {
  if (!ctx || !blobs) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_import before rk_dist_init");
  return dist_import(ctx, (const u8 *)blobs, RK_DIST_BLOB_BYTES);
}

int rk_dist_load_aos(rk_ctx *ctx, const void *frags, uint64_t n_local, uint64_t file_offset, uint64_t seqx_len, uint64_t seqy_len,
                     unsigned flags, rk_load_stats *stats) {
  if (!ctx) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_load_aos before rk_dist_init");
  if (const int rc = dist_load_refusal(ctx)) return rc;
  return dist_load(ctx, frags, n_local, file_offset, seqx_len, seqy_len, flags, stats);
}

int rk_dist_load_csv(rk_ctx *ctx, const char *slice, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags,
                     unsigned flags, rk_load_stats *stats, rk_csv_stats *csv) {
  if (!ctx) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_load_csv before rk_dist_init");
  if (const int rc = dist_load_refusal(ctx)) return rc;
  DistCsv L;
  dist_csv_local(ctx, slice, bytes, csv_upload_threads(), L);
  return dist_csv_finish(ctx, L, seqx_len, seqy_len, total_frags, flags, stats, csv);
}

int rk_dist_load_packed(rk_ctx *ctx, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n_local,
                        uint64_t file_offset, uint64_t seqx_len, uint64_t seqy_len, unsigned flags, rk_load_stats *stats) {
  if (!ctx) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_load_packed before rk_dist_init");
  if (const int rc = dist_load_refusal(ctx)) return rc;
  return dist_load_packed(ctx, key4, strand, rest4, n_local, file_offset, seqx_len, seqy_len, flags, stats);
}

int rk_dist_group(rk_ctx *ctx, double len_ratio, double pos_ratio, unsigned flags, rk_result *out, rk_dist_info *info) {
  if (!ctx || !out) return RK_ERR_ARG;
  if (!ctx->dist) return fail(ctx, RK_ERR_STATE, "rk_dist_group before rk_dist_init");
  return dist_group(ctx, len_ratio, pos_ratio, flags, out, info);
}

int rk_dist_format_lines(rk_ctx *ctx, uint64_t first_line, uint64_t n_lines, rk_text *out) {
  if (!ctx || !out) return RK_ERR_ARG;
  memset(out, 0, sizeof *out);
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  u64 nbytes = 0;
  char *buf = nullptr;
  int rc = dist_format_device(ctx, first_line, n_lines, &nbytes);
  if (!rc) rc = ctx->h_text.next(nbytes, &buf, ctx->err);
  if (!rc) rc = format_to_host(ctx, nbytes, buf, &out->ms_device);
  if (rc) return rc;
  out->text = buf;
  out->n_bytes = nbytes;
  return RK_OK;
}

int rk_dist_group_statistics(rk_ctx *ctx, unsigned flags, const rk_group_stats **stats, const rk_group_stats **d_stats,
                             uint64_t *first_gid, uint64_t *n_groups) {
  if (!ctx) return RK_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ProfGuard pg(ctx);
  const int rc = dist_group_stats(ctx, flags);
  if (rc) return rc;
  const Dist &D = *ctx->dist;
  const u64 ng = D.n_groups_rank;
  if (stats) *stats = ((flags & RK_F_HOST_RESULT) && ng) ? (const rk_group_stats *)ctx->h_stats.ptr() : nullptr;
  if (d_stats) *d_stats = (const rk_group_stats *)ctx->d_stats.ptr();
  if (first_gid) *first_gid = D.gid_base;
  if (n_groups) *n_groups = ng;
  return RK_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------------
// C ABI: one process, one host thread per GPU
// ---------------------------------------------------------------------------------------------------------------------
struct rk_multi {
  int n = 0;
  std::vector<rk_ctx *> ctx;
  std::vector<int> devices;
  LocalGroup local;
  bool use_nccl = false;
  std::vector<ncclComm_t> comms;
  std::string err;
  u64 cap = 0;
  bool have_load = false;
  // merged host result of the last rk_multi_group
  GrowBuffer h_res{cudaHostAllocDefault};
  std::vector<rk_dist_info> infos;
  // rk_multi_format_lines' text and rk_multi_group_statistics' groups (pinned, portable: copied into by every GPU)
  TextBuffers h_text{cudaHostAllocPortable};
  GrowBuffer h_stats{cudaHostAllocPortable};
};

namespace {

// the transport of rank r: over mg's communicators, or through its LocalGroup
Transport *multi_transport(rk_multi *mg, int r) {
  if (mg->use_nccl) {
    NcclTransport *t = new NcclTransport;
    t->comm = mg->comms[r];
    t->own_comm = false;
    return t;
  }
  LocalTransport *t = new LocalTransport;
  t->g = &mg->local;
  return t;
}

// one communicator per device when the devices are distinct (NCCL); else, or when NCCL fails to start, the ranks are
// threads of this process and the local transport always works
void multi_init_comms(rk_multi *mg) {
  if (!mg->use_nccl) return;
  NcclApi &N = nccl_api();
  mg->comms.resize(mg->n);
  if (!N.ok() || N.CommInitAll(mg->comms.data(), mg->n, mg->devices.data()) != ncclSuccess) {
    mg->comms.clear();
    mg->use_nccl = false;
  }
}

template <class F>
int run_ranks(rk_multi *mg, F fn) {  // fn(rank) on one thread per rank; first failing rank's code and message
  std::vector<int> rc(mg->n, RK_OK);
  std::vector<std::thread> th;
  for (int r = 0; r < mg->n; ++r) th.emplace_back([&, r] { rc[r] = fn(r); });
  for (auto &t : th) t.join();
  for (int r = 0; r < mg->n; ++r)
    if (rc[r] != RK_OK) {
      mg->err = "rank " + std::to_string(r) + ": " + rk_last_error(mg->ctx[r]);
      return rc[r];
    }
  return RK_OK;
}

// every rank's partition arena (a view: its workspace) mapped into every other rank
int multi_map_peers(rk_multi *mg) {
  std::vector<u8> blobs((size_t)mg->n * RK_DIST_BLOB_BYTES, 0);
  const int rc = run_ranks(mg, [&](int r) { return dist_export(mg->ctx[r], (DistBlob *)(blobs.data() + (size_t)r * RK_DIST_BLOB_BYTES)); });
  return rc ? rc : run_ranks(mg, [&](int r) { return dist_import(mg->ctx[r], blobs.data(), RK_DIST_BLOB_BYTES); });
}

int multi_set_capacity(rk_multi *mg, u64 cap) {
  int rc = run_ranks(mg, [&](int r) {
    rk_ctx *c = mg->ctx[r];
    if (!c->dist) return dist_init_common(c, r, mg->n, multi_transport(mg, r), cap);
    return dist_allocate(c, cap);
  });
  if (rc) return rc;
  if ((rc = multi_map_peers(mg))) return rc;
  mg->cap = cap;
  return RK_OK;
}

// the slices of an n-record file, lo[r] .. lo[r + 1] for rank r (rk_multi_load_aos, rk_multi_load_packed): every rank starts
// with a contiguous slice of the file (slices start on a 16-record boundary: 16-byte aligned records); the capacity grows
// to 1.5 x the largest slice + 65536
int multi_record_slices(rk_multi *mg, u64 n, std::vector<u64> &lo) {
  lo.assign(mg->n + 1, 0);
  for (int r = 0; r <= mg->n; ++r) {
    u64 b = n * (u64)r / (u64)mg->n;
    if (r < mg->n) b -= b % 16;
    lo[r] = r == mg->n ? n : b;
  }
  u64 biggest = 0;
  for (int r = 0; r < mg->n; ++r) biggest = std::max(biggest, lo[r + 1] - lo[r]);
  const u64 want = biggest + biggest / 2 + (1u << 16);
  return want > mg->cap ? multi_set_capacity(mg, want) : RK_OK;
}

// the load refusals of rk_multi_load_*: a view, or a base with live views (rank 0 speaks for all: they are made together)
int multi_load_refusal(rk_multi *mg) {
  rk_ctx *c = mg->ctx[0];
  if (!c->dist) return RK_OK;
  const int rc = dist_load_refusal(c);
  if (rc) mg->err = c->err;
  return rc;
}

}  // namespace

extern "C" {

rk_multi *rk_create_multi(const int *devices, int ndev) {
  if (!devices || ndev < 1 || ndev > DIST_MAX_RANKS) return nullptr;
  rk_multi *mg = new rk_multi;
  mg->n = ndev;
  mg->local.n = ndev;
  mg->devices.assign(devices, devices + ndev);
  bool distinct = true;
  for (int i = 0; i < ndev; ++i)
    for (int j = 0; j < i; ++j) distinct = distinct && devices[i] != devices[j];
  mg->use_nccl = distinct && ndev > 1;
  for (int r = 0; r < ndev; ++r) {
    rk_ctx *c = rk_create(devices[r]);
    if (!c) {
      for (rk_ctx *p : mg->ctx) rk_destroy(p);
      delete mg;
      return nullptr;
    }
    mg->ctx.push_back(c);
  }
  multi_init_comms(mg);
  return mg;
}

rk_multi *rk_multi_create_view(rk_multi *base) {
  if (!base) {
    set_create_error("rk_multi_create_view: null rk_multi");
    return nullptr;
  }
  if (!base->have_load) {
    set_create_error("rk_multi_create_view: no partition database (it needs a successful rk_multi_load_aos, rk_multi_load_csv or "
                     "rk_multi_load_packed)");
    return nullptr;
  }
  rk_multi *v = new rk_multi;
  v->n = base->n;
  v->local.n = base->n;
  v->devices = base->devices;
  v->use_nccl = base->use_nccl;
  multi_init_comms(v);
  for (int r = 0; r < v->n; ++r) {
    std::string err;
    rk_ctx *c = dist_view_create(base->ctx[r], multi_transport(v, r), err);
    if (!c) {
      set_create_error("rk_multi_create_view: rank " + std::to_string(r) + ": " + err);
      rk_destroy_multi(v);
      return nullptr;
    }
    v->ctx.push_back(c);
  }
  if (multi_map_peers(v)) {
    set_create_error("rk_multi_create_view: " + v->err);
    rk_destroy_multi(v);
    return nullptr;
  }
  v->cap = base->cap;
  v->have_load = true;
  return v;
}

void rk_destroy_multi(rk_multi *mg) {
  if (!mg) return;
  for (rk_ctx *c : mg->ctx) rk_destroy(c);
  for (ncclComm_t c : mg->comms) nccl_api().CommDestroy(c);
  delete mg;
}

const char *rk_multi_last_error(const rk_multi *mg) { return mg ? mg->err.c_str() : "null rk_multi"; }
int rk_multi_ranks(const rk_multi *mg) { return mg ? mg->n : 0; }
rk_ctx *rk_multi_ctx(rk_multi *mg, int rank) { return (mg && rank >= 0 && rank < mg->n) ? mg->ctx[rank] : nullptr; }
const char *rk_multi_transport(const rk_multi *mg) { return !mg ? "" : (mg->use_nccl ? "nccl" : "local"); }

int rk_multi_load_aos(rk_multi *mg, const void *frags, uint64_t n, uint64_t seqx_len, uint64_t seqy_len, unsigned flags,
                      rk_load_stats *stats) {
  if (!mg || (!frags && n)) return RK_ERR_ARG;
  if (const int rc = multi_load_refusal(mg)) return rc;
  mg->have_load = false;
  std::vector<u64> lo;
  if (const int rc = multi_record_slices(mg, n, lo)) return rc;
  std::vector<rk_load_stats> st(mg->n);
  const int rc = run_ranks(mg, [&](int r) {
    return dist_load(mg->ctx[r], (const u8 *)frags + lo[r] * RK_FRAG_BYTES, lo[r + 1] - lo[r], lo[r], seqx_len, seqy_len, flags, &st[r]);
  });
  if (rc) return rc;
  if (stats) {
    *stats = st[0];
    for (int r = 1; r < mg->n; ++r) stats->n_launches += st[r].n_launches;
  }
  mg->have_load = true;
  return RK_OK;
}

int rk_multi_load_csv(rk_multi *mg, const char *body, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags,
                      unsigned flags, rk_load_stats *stats, rk_csv_stats *csv) {
  if (!mg || (!body && bytes)) return RK_ERR_ARG;
  if (const int rc = multi_load_refusal(mg)) return rc;
  mg->have_load = false;
  if (bytes && is_device_pointer(body)) {
    mg->err = "rk_multi_load_csv takes the text in host memory";
    return RK_ERR_ARG;
  }
  // cut r: one byte past the first '\n' at or after bytes * r / N (the end of the text when there is none)
  const int n = mg->n;
  std::vector<u64> lo(n + 1, bytes);
  lo[0] = 0;
  for (int r = 1; r < n; ++r) {
    const u64 a = bytes * (u64)r / (u64)n;
    const void *nl = a < bytes ? memchr(body + a, '\n', bytes - a) : nullptr;
    lo[r] = nl ? (u64)((const char *)nl - body) + 1 : bytes;
  }
  // step 1, the local half on every rank; the capacity follows from the rows each rank may load: the device's accepted
  // rows plus the rows left to the host (the rule of rk_multi_load_aos: the largest slice x 1.5 + 65536)
  // the copy threads of all ranks together: those of one rk_load_csv, or one per rank (its own thread) when there are more ranks
  const int threads = std::max(1, csv_upload_threads() / n);
  std::vector<DistCsv> loc(n);
  int rc = run_ranks(mg, [&](int r) {
    dist_csv_local(mg->ctx[r], body + lo[r], lo[r + 1] - lo[r], threads, loc[r]);
    return RK_OK;
  });
  if (rc) return rc;
  u64 biggest = 0;
  for (int r = 0; r < n; ++r)
    if (!loc[r].rc) biggest = std::max(biggest, loc[r].p.n_dev_acc + loc[r].p.n_host);
  const u64 want = biggest + biggest / 2 + (1u << 16);
  if (want > mg->cap && (rc = multi_set_capacity(mg, want))) return rc;
  // step 2, the collective half
  std::vector<rk_load_stats> st(n);
  std::vector<rk_csv_stats> cs(n);
  rc = run_ranks(mg, [&](int r) { return dist_csv_finish(mg->ctx[r], loc[r], seqx_len, seqy_len, total_frags, flags, &st[r], &cs[r]); });
  if (rc) return rc;
  if (stats) {
    *stats = st[0];
    for (int r = 1; r < n; ++r) {
      stats->n_launches += st[r].n_launches;
      stats->ms_stage[RK_ST_H2D] = std::max(stats->ms_stage[RK_ST_H2D], st[r].ms_stage[RK_ST_H2D]);
    }
  }
  if (csv) {
    memset(csv, 0, sizeof *csv);
    for (int r = 0; r < n; ++r) {
      csv->n_rows += cs[r].n_rows, csv->n_accepted += cs[r].n_accepted, csv->n_host_rows += cs[r].n_host_rows;
      csv->wide |= cs[r].wide;
      csv->ms_upload = std::max(csv->ms_upload, cs[r].ms_upload);
      csv->ms_parse = std::max(csv->ms_parse, cs[r].ms_parse);
    }
  }
  mg->have_load = true;
  return RK_OK;
}

int rk_multi_load_packed(rk_multi *mg, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n, uint64_t seqx_len,
                         uint64_t seqy_len, unsigned flags, rk_load_stats *stats) {
  if (!mg || (n && (!key4 || !strand))) return RK_ERR_ARG;
  if (const int rc = multi_load_refusal(mg)) return rc;
  mg->have_load = false;
  if (n && (is_device_pointer(key4) || is_device_pointer(strand) || (rest4 && is_device_pointer(rest4)))) {
    mg->err = "rk_multi_load_packed takes the arrays in host memory";
    return RK_ERR_ARG;
  }
  std::vector<u64> lo;  // the slices and the capacity of rk_multi_load_aos: both loads partition a file alike
  if (const int rc = multi_record_slices(mg, n, lo)) return rc;
  std::vector<rk_load_stats> st(mg->n);
  const int rc = run_ranks(mg, [&](int r) {
    return dist_load_packed(mg->ctx[r], key4 ? key4 + lo[r] * 4 : nullptr, strand ? strand + lo[r] : nullptr,
                            rest4 ? rest4 + lo[r] * 4 : nullptr, lo[r + 1] - lo[r], lo[r], seqx_len, seqy_len, flags, &st[r]);
  });
  if (rc) return rc;
  if (stats) {
    *stats = st[0];
    for (int r = 1; r < mg->n; ++r) {
      stats->n_launches += st[r].n_launches;
      stats->ms_stage[RK_ST_H2D] = std::max(stats->ms_stage[RK_ST_H2D], st[r].ms_stage[RK_ST_H2D]);
    }
  }
  mg->have_load = true;
  return RK_OK;
}

int rk_multi_group(rk_multi *mg, double len_ratio, double pos_ratio, unsigned flags, rk_result *out) {
  if (!mg || !out) return RK_ERR_ARG;
  if (!mg->have_load) {
    mg->err = "rk_multi_group before a successful rk_multi_load_aos";
    return RK_ERR_STATE;
  }
  std::vector<rk_result> res(mg->n);
  mg->infos.assign(mg->n, rk_dist_info{});
  const int rc = run_ranks(mg, [&](int r) { return dist_group(mg->ctx[r], len_ratio, pos_ratio, flags | RK_F_HOST_RESULT, &res[r], &mg->infos[r]); });
  if (rc) return rc;
  // the ranks hold consecutive ranges of output lines: concatenate them
  u64 total = 0;
  for (int r = 0; r < mg->n; ++r) total += res[r].n_kept;
  const int rc2 = mg->h_res.reserve(HostResult::bytes(total), nullptr, mg->err);
  if (rc2) return rc2;
  const HostResult hr(mg->h_res.ptr(), total);
  std::vector<std::thread> th;
  for (int r = 0; r < mg->n; ++r)
    th.emplace_back([&, r] {
      const u64 off = mg->infos[r].line_offset, k = res[r].n_kept;
      if (!k) return;
      memcpy(hr.order + off, res[r].order, k * 4);
      memcpy(hr.gid + off, res[r].gid, k * 4);
      memcpy(hr.identity + off, res[r].identity, k * 4);
      memcpy(hr.repval + off, res[r].repval, k);
    });
  for (auto &t : th) t.join();
  memset(out, 0, sizeof *out);
  out->n_kept = total;
  out->n_groups = res[0].n_groups;
  hr.publish(out);
  for (int r = 0; r < mg->n; ++r) {
    out->n_launches += res[r].n_launches;
    out->ms_device = std::max(out->ms_device, res[r].ms_device);
    for (int s = 0; s < RK_NSTAGES; ++s) out->ms_stage[s] = std::max(out->ms_stage[s], res[r].ms_stage[s]);
  }
  return RK_OK;
}

int rk_multi_info(const rk_multi *mg, int rank, rk_dist_info *info) {
  if (!mg || !info || rank < 0 || rank >= (int)mg->infos.size()) return RK_ERR_ARG;
  *info = mg->infos[rank];
  return RK_OK;
}

int rk_multi_format_lines(rk_multi *mg, uint64_t first_line, uint64_t n_lines, rk_text *out) {
  if (!mg || !out) return RK_ERR_ARG;
  memset(out, 0, sizeof *out);
  if ((int)mg->infos.size() != mg->n) {
    mg->err = "rk_multi_format_lines before a successful rk_multi_group";
    return RK_ERR_STATE;
  }
  u64 total = 0;
  for (const rk_dist_info &i : mg->infos) total += i.n_lines;
  if (first_line > total || n_lines > total - first_line) {
    mg->err = "line range beyond the " + std::to_string(total) + " output lines";
    return RK_ERR_ARG;
  }
  if (n_lines > RK_FORMAT_MAX_LINES) {
    mg->err = "at most " + std::to_string(RK_FORMAT_MAX_LINES) + " lines per call";
    return RK_ERR_ARG;
  }
  // every rank formats its part of the range on its GPU (an empty part too: every rank checks its state) ...
  std::vector<u64> nb(mg->n, 0), pos(mg->n + 1, 0);
  std::vector<float> ms(mg->n, 0.f);
  int rc = run_ranks(mg, [&](int r) -> int {
    rk_ctx *ctx = mg->ctx[r];
    const u64 lo = mg->infos[r].line_offset, hi = lo + mg->infos[r].n_lines;
    const u64 a = std::max<u64>(first_line, lo), b = std::min<u64>(first_line + n_lines, hi);
    CK(cudaSetDevice(ctx->device));
    ProfGuard pg(ctx);
    return dist_format_device(ctx, b > a ? a - lo : 0, b > a ? b - a : 0, &nb[r]);
  });
  if (rc) return rc;
  // ... and copies it to its place in one buffer: the parts in rank order are the lines in order
  for (int r = 0; r < mg->n; ++r) pos[r + 1] = pos[r] + nb[r];
  const u64 nbytes = pos[mg->n];
  char *buf = nullptr;
  rc = mg->h_text.next(nbytes, &buf, mg->err);
  if (rc) return rc;
  rc = run_ranks(mg, [&](int r) { return format_to_host(mg->ctx[r], nb[r], buf + pos[r], &ms[r]); });
  if (rc) return rc;
  out->text = buf;
  out->n_bytes = nbytes;
  out->ms_device = *std::max_element(ms.begin(), ms.end());
  return RK_OK;
}

int rk_multi_group_statistics(rk_multi *mg, const rk_group_stats **stats, uint64_t *n_groups) {
  if (!mg) return RK_ERR_ARG;
  if ((int)mg->infos.size() != mg->n) {
    mg->err = "rk_multi_group_statistics before a successful rk_multi_group";
    return RK_ERR_STATE;
  }
  const u64 total = mg->infos[0].total_groups;
  const u64 need = total * sizeof(rk_group_stats);
  const int rc2 = mg->h_stats.reserve(need > mg->h_stats.cap() ? need + need / 8 + 4096 : need, nullptr, mg->err);
  if (rc2) return rc2;
  rk_group_stats *h = (rk_group_stats *)mg->h_stats.ptr();
  // every rank reduces its own groups (a group is never split) and copies them to their place in gid order
  const int rc = run_ranks(mg, [&](int r) -> int {
    rk_ctx *ctx = mg->ctx[r];
    CK(cudaSetDevice(ctx->device));
    ProfGuard pg(ctx);
    const int rc2 = dist_group_stats(ctx, 0);
    if (rc2) return rc2;
    const Dist &D = *ctx->dist;
    if ((u64)D.gid_base + D.n_groups_rank > total)
      return fail(ctx, RK_ERR_INTERNAL, "groups %u .. %u of rank %d beyond the %llu groups", D.gid_base, D.gid_base + D.n_groups_rank, r,
                  (unsigned long long)total);
    if (D.n_groups_rank) {
      CK(cudaMemcpyAsync(h + D.gid_base, ctx->d_stats.ptr(), (u64)D.n_groups_rank * sizeof(rk_group_stats), cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
    }
    return RK_OK;
  });
  if (rc) return rc;
  if (stats) *stats = total ? h : nullptr;
  if (n_groups) *n_groups = total;
  return RK_OK;
}

}  // extern "C"
