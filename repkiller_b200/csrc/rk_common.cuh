// Shared device helpers and the launcher declarations of the grouping kernels (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define RK_NONE32 0xFFFFFFFFu

namespace rk {

typedef uint32_t u32;
typedef uint64_t u64;
typedef uint8_t u8;

// record layout: /root/reference/src/structs.h:12-51 under #pragma pack(1)
constexpr int FRAG_BYTES = 109;
constexpr int OFF_XSTART = 8;
constexpr int OFF_YSTART = 16;
constexpr int OFF_LENGTH = 40;
constexpr int OFF_IDENT = 48;
constexpr int OFF_STRAND = 92;
constexpr int OFF_XEND = 24, OFF_YEND = 32, OFF_SCORE = 56, OFF_SIMILARITY = 64;  // printed only (K6)

// constants of the reference
constexpr u32 XBUCKET = 10;   // FragmentsDatabase.cpp:84,96 ; commonFunctions.cpp:152,154
constexpr u32 DIVISOR = 100;  // SequenceOcupationList.h:11

// per-fragment flag bits
constexpr u8 FL_REVERSE = 1;  // strand != 'f' (commonFunctions.cpp:52-53)
constexpr u8 FL_DROPPED = 2;  // xStart/10 == vsize-1 (FragmentsDatabase.h:29-31)

// error bits raised by kernels (device word, OR-ed)
constexpr u32 ERR_COORD = 1;     // coordinate >= 2^31
constexpr u32 ERR_XBUCKET = 2;   // xStart/10 >= vsize
constexpr u32 ERR_CENTER = 4;    // center/100 beyond the occupation list
constexpr u32 ERR_WORKLIST = 8;  // long-segment worklist overflow
constexpr u32 ERR_SPIN = 16;     // bounded spin expired

struct Geometry {
  u64 lx, ly;      // loaded sequence lengths (header + 1)
  u32 vsize;       // 1 + lx/10
  u32 mx, my;      // max_index = len / 100 (SequenceOcupationList.cpp:4)
  u32 nbx, nby;    // buckets per strand class on each axis (max_index + 2: one slack bucket for "next" links)
};

__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lanemask_lt() {
  u32 m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// Random gathers of one sector: ask L2 for a 64-byte fill instead of the default promotion to the whole 128-byte line
// (ncu showed ~108 B of DRAM traffic per 32-byte gather).  Measured: k_keys 0.270 -> 0.258 ms; no gain for the 8- and
// 16-byte gathers of K3 and K5, which keep plain loads.
__device__ __forceinline__ uint4 ldg_gather_u4(const uint4 *p) {
  uint4 v;
  asm volatile("ld.global.nc.L2::64B.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

// streaming loads/stores: data touched once should not displace the gather targets in L1
__device__ __forceinline__ u32 ld_stream(const u32 *p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(u32 *p, u32 v) { __stcs(p, v); }

// "next"-bucket probes of get_associated_group (SequenceOcupationList.cpp:58,80): center+1 is probed iff
// center < max_index, center+2 iff center < max_index-1 in unsigned arithmetic (wraps when max_index == 0).
__device__ __forceinline__ bool probes_next(u32 c, u32 max_index) {
  const u32 r = c % DIVISOR;
  if (r == 99) return c < max_index || max_index == 0;
  if (r == 98) return max_index == 0 || c < max_index - 1;
  return false;
}
// "previous"-bucket probes (:47,69): center-1 iff center > 0, center-2 iff center > 1.
__device__ __forceinline__ bool probes_prev(u32 c) { return (c % DIVISOR) <= 1 && c >= DIVISOR; }

__device__ __forceinline__ u32 absdiff(u32 a, u32 b) { return a > b ? a - b : b - a; }

// first bucket of the run of linked buckets that bucket k belongs to (link bit k: k is processed together with k-1)
__device__ __forceinline__ u32 run_start(const u32 *__restrict__ bm, u32 k) {
  // largest k' <= k whose link bit is clear (bit 0 of every strand class is never set)
  u32 w = k >> 5;
  u32 m = 0xFFFFFFFFu >> (31 - (k & 31));
  for (;;) {
    const u32 z = ~bm[w] & m;
    if (z) return (w << 5) + (31 - __clz(z));
    if (w == 0) return 0;
    --w;
    m = 0xFFFFFFFFu;
  }
}


// ---- digit histograms of a sort key, accumulated by the kernel that PRODUCES the key (saves the sort's own histogram
// pass: one more read of the keys and a launch).  ghist: [4][256] global counters (zeroed by the caller), or nullptr.
struct HistOut {
  u32 *ghist;
  int passes;    // ceil(key_bits / 8)
  int key_bits;
};
constexpr int HIST_PASSES = 4, HIST_RADIX = 256;

// One key per lane into a CTA's shared-memory histograms.  Every lane of the warp must call it (valid = false for
// lanes without a key): a digit shared by the whole warp — the top digits of nearly sorted keys — is counted once by
// lane 0 instead of serialising 32 atomics on one address.
__device__ __forceinline__ void hist_add(u32 (*h)[HIST_RADIX], u32 key, bool valid, const HistOut &ho) {
  const u32 last_mask = (1u << (ho.key_bits - 8 * (ho.passes - 1))) - 1;
  const u32 lane = threadIdx.x & 31;
#pragma unroll
  for (int p = 0; p < HIST_PASSES; ++p) {
    if (p < ho.passes) {
      const u32 d = (key >> (8 * p)) & (p == ho.passes - 1 ? last_mask : 0xFFu);
      const u32 d0 = __shfl_sync(0xFFFFFFFFu, d, 0);
      if (__all_sync(0xFFFFFFFFu, valid && d == d0)) {
        if (lane == 0) atomicAdd(&h[p][d], 32u);
      } else if (valid) {
        atomicAdd(&h[p][d], 1u);
      }
    }
  }
}
// all threads of the CTA: zero / flush (blockDim.x >= 256 or any multiple of 32; strided)
__device__ __forceinline__ void hist_zero(u32 (*h)[HIST_RADIX]) {
  for (u32 i = threadIdx.x; i < (u32)(HIST_PASSES * HIST_RADIX); i += blockDim.x) (&h[0][0])[i] = 0;
}
__device__ __forceinline__ void hist_flush(u32 (*h)[HIST_RADIX], const HistOut &ho) {
  for (u32 i = threadIdx.x; i < (u32)(ho.passes * HIST_RADIX); i += blockDim.x) {
    const u32 c = (&h[0][0])[i];
    if (c) atomicAdd(&ho.ghist[i], c);
  }
}

// ---- per-kernel timing (CUDA events around every launch; off unless rk_profile_enable) ---------------
enum KernelId {
  KID_DECODE = 0, KID_RADIX_HIST, KID_SCAN, KID_RADIX_SCATTER, KID_KEYS, KID_MATCH_SMALL, KID_MATCH_LONG, KID_CHASE,
  KID_HKEY, KID_PACK, KID_GSORT_SMALL, KID_GSORT_LARGE, KID_FINALIZE, KID_DIAG, KID_GSORT_WARP, KID_FORMAT, KID_DIST_ROWS, KID_STATS, KID_CHASE_EXITS,
  KID_CSV_LINES, KID_CSV_ROWS, KID_COUNT
};
void prof_begin(int kid, cudaStream_t st, unsigned long long units);
void prof_end(cudaStream_t st);
struct KScope {
  cudaStream_t st;
  KScope(int kid, cudaStream_t s, unsigned long long units) : st(s) { prof_begin(kid, s, units); }
  ~KScope() { prof_end(st); }
};

// per-device kernel attributes (dynamic shared memory opt-ins); rk_create calls these for the context's device
cudaError_t decode_init_device();
cudaError_t sort_init_device();
cudaError_t order_init_device();
cudaError_t dist_init_device();

// ---- launchers (each returns the number of kernels it launched) -------------------------------------

// tooling: synthetic workload on the device, identical to repkiller_b200/gen.py
int launch_gen(u64 seed, u64 lx, u64 ly, double p_rep, u64 families, u64 ax, u64 ay, u64 tandem_every, u64 start, u64 count,
               u8 *out, cudaStream_t st);

// K1: decode n packed records (device, 16-byte aligned) into file-order SoA, raise link bits.
int launch_decode(const u8 *aos, u64 n, Geometry g, u32 *xs, u32 *ys, u32 *len, u8 *flags, float *identity,
                  u32 *key0, u32 *link_x, u32 *link_y, u32 *n_dropped, u32 *err, cudaStream_t st, uint4 *rec4 = nullptr,
                  HistOut hist = HistOut{nullptr, 0, 0}, u32 fidx_base = 0);

// K1 for the compact ingest: {xStart, yStart, length, ident} words + strand bytes instead of 109-byte records
int launch_decode_packed(const uint4 *key4, const u8 *strand, u64 n, Geometry g, u32 *key0, u32 *link_x, u32 *link_y, u32 *n_dropped,
                         u32 *err, cudaStream_t st, uint4 *rec4, HistOut hist, u32 fidx_base = 0);

// K2: stable LSD radix sort of (key,value) pairs; result in keys_out/vals_out.
u64 sort_work_bytes(u64 n);
// prehist: [4][256] digit counts of keys_in already accumulated by the producer of the keys (HistOut), or nullptr
int launch_sort_pairs(const u32 *keys_in, const u32 *vals_in, u32 *keys_out, u32 *vals_out, u32 *keys_tmp,
                      u32 *vals_tmp, u64 n, int key_bits, void *work, cudaStream_t st, u32 *err_word = nullptr,
                      u32 *prehist = nullptr);

// K2 keys: rank-order SoA + super-bucket sort keys.
// rec4: file order, two 16-byte words per record {xStart, yStart, length, flags} {identity bits, 0, 0, 0} (one 32-byte
// sector per gather); xl_r/yl_r: rank-order {center, length} per axis (one 8-byte gather per fragment in the match
// kernels); identity_r: rank order.  Multi-GPU: gfidx_r = the record's global file index (second word of rec4), and with
// own_bit the X key is written as 2*key+1 so that halo entries (2*key) of the same super-bucket sort before the rank's own;
// rec6 (instead of rec4): the 24-byte rows of exchange 1, {xStart, yStart} {length, flags} {identity, file index}
int launch_keys(const u32 *fidx_r, u32 m, Geometry g, const uint4 *rec4, const u32 *link_x, const u32 *link_y, uint2 *xl_r,
                uint2 *yl_r, u32 *ys_r, u32 *kx, u32 *ky, float *identity_r, cudaStream_t st, HistOut hist_x = HistOut{nullptr, 0, 0},
                HistOut hist_y = HistOut{nullptr, 0, 0}, u32 *gfidx_r = nullptr, u32 own_bit = 0, const uint2 *rec6 = nullptr);

// K3: one axis pass of generate_fragment_groups.  is_y: fragments with parent != NONE insert unconditionally.
struct MatchArgs {
  const u32 *skey;   // sorted super-bucket keys
  const u32 *srank;  // index (in the pass's working list) of the fragment at each sorted position
  const uint2 *cl_r; // {center on this axis, length}, list order
  u32 *parent;       // list-indexed; X pass writes every entry, Y pass fills unmatched ones
  u32 *xm_bits;      // one bit per rank: matched in the X pass (written by the X pass, read by the Y pass)
  u32 m;
  u32 max_index;     // axis max_index
  double len_ratio, pos_ratio;
  int is_y;
  u32 *worklist;     // long segments (start positions)
  u32 *work_count;   // [0] number of long segments
  u32 work_cap;
  u32 *ent_rank, *ent_c, *ent_len;  // scratch of m entries each for long segments
  u32 *err;
  int key_shift;       // segments are runs of equal (skey >> key_shift); multi-GPU X pass: bit 0 = "own fragment, not halo"
  const u8 *xm_bytes;  // Y pass, when set: one byte per rank instead of the xm_bits map (multi-GPU: the flags travel as bytes)
};
int launch_match(const MatchArgs &a, cudaStream_t st);

// K4: roots, group ids.
u64 forest_work_bytes(u32 m);
// lo/cnt: resolve only ranks [lo, lo+cnt) of a parent array of m entries
int launch_forest(const u32 *parent, u32 m, u32 *gid_rank, u32 *n_groups, void *work, cudaStream_t st, u32 lo = 0,
                  u32 cnt = 0xFFFFFFFFu, HistOut hist = HistOut{nullptr, 0, 0});

// K5a: h = |yStart - yStart(last fragment of the same xStart/10 bucket)| per rank.
// With hfi_r: also the packed per-rank record {h, file index, identity bits, 0} K5b/c gathers (h may then be null).
int launch_hkey(const u32 *k0_r, const u32 *ys_r, u32 m, u32 *h, cudaStream_t st, const u32 *fidx_r = nullptr,
                const float *identity_r = nullptr, uint4 *hfi_r = nullptr);

// K5a': the full diag_func table with carry-forward (only for rk_diagonal_func).
int launch_diag_table(const u32 *k0_r, const u32 *ys_r, u32 m, u32 vsize, u64 *diag, void *work, cudaStream_t st);

// K5b/c: after the stable sort by gid: pack (h, rank), per-group libstdc++ std::sort order, outputs.
struct OrderArgs {
  const u32 *sgid;    // sorted gids
  const u32 *srank;   // rank at each sorted position
  const uint4 *hfi_r; // single GPU: {h, file index, identity bits, 0} by rank (gathered through srank)
  // direct layout (srank == nullptr, rk_sort_members): the three arrays are already in gid-sorted order
  const u32 *h;
  const u32 *fidx_r;
  const float *identity_r;
  // scratch of the giant groups (order_carve): (h, index) words, position lists, chunk words, ranges handed to warps
  u64 *packed, *packed2;
  u32 *chunk_words;
  u64 chunk_stride;
  uint4 *ranges;
  u32 range_cap;
  u32 m;
  int do_sort;
  u32 gid_base;  // added to sgid for out_gid (multi-GPU: a rank sorts its range of groups by gid - first gid of the range)
  // start positions of the groups of more than 16 / 128 / 1024 members; work_count[2*i] = entries of list i,
  // work_count[2*i+1] = its pop cursor; work_count[6], [7]: the same for `ranges`
  u32 *worklist[3];
  u32 *work_count;
  u32 work_cap[3];
  u32 *out_order, *out_gid;
  u8 *out_repval;
  float *out_identity;
  u32 *err;
};
// What one output line prints of its record, in line order: a partitioned comparison brings it to the rank that holds the
// line (RK_F_LINE_RECORDS), since the record itself sits on the rank that loaded it.  The integers stay 64-bit as in the file.
struct __align__(16) LineRow {
  u64 xs, ys, len, xe, ye, score, ident;
  u32 sim_bits, strand;
};
static_assert(sizeof(LineRow) == 64, "line row size");
__device__ __forceinline__ u64 ldg_u64_unaligned(const u8 *p) {  // records are 109 bytes apart: no alignment to rely on
  u64 v = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) v |= (u64)p[i] << (8 * i);
  return v;
}
__device__ __forceinline__ LineRow line_row_of_record(const u8 *rec) {
  LineRow f;
  f.xs = ldg_u64_unaligned(rec + OFF_XSTART), f.ys = ldg_u64_unaligned(rec + OFF_YSTART);
  f.xe = ldg_u64_unaligned(rec + OFF_XEND), f.ye = ldg_u64_unaligned(rec + OFF_YEND);
  f.len = ldg_u64_unaligned(rec + OFF_LENGTH), f.score = ldg_u64_unaligned(rec + OFF_SCORE), f.ident = ldg_u64_unaligned(rec + OFF_IDENT);
  f.sim_bits = (u32)rec[OFF_SIMILARITY] | ((u32)rec[OFF_SIMILARITY + 1] << 8) | ((u32)rec[OFF_SIMILARITY + 2] << 16) |
               ((u32)rec[OFF_SIMILARITY + 3] << 24);
  f.strand = rec[OFF_STRAND];
  return f;
}
// the compact rows of rk_load_packed / rk_load_csv: {xStart, yStart, length, ident} {xEnd, yEnd, score, similarity bits}, strand
struct PackedRows {
  const uint4 *key, *rest;
  const u8 *strand;
};
// the same fields from the compact rows: two 16-byte words and a byte per row
__device__ __forceinline__ LineRow line_row_of_packed(const uint4 *pk_key, const uint4 *pk_rest, const u8 *pk_strand, u32 fidx) {
  LineRow f;
  const uint4 k = pk_key[fidx], r = pk_rest[fidx];
  f.xs = k.x, f.ys = k.y, f.len = k.z, f.ident = k.w;
  f.xe = r.x, f.ye = r.y, f.score = r.z, f.sim_bits = r.w;
  f.strand = pk_strand[fidx];
  return f;
}
// K6: the text of output lines first_line .. first_line+n_lines (commonFunctions.cpp:101-115) from the loaded records and
// the result arrays of the last grouping.
struct FormatArgs {
  const LineRow *rows;     // the line rows, indexed by line (partitioned comparisons) — or, indexed by order[line]:
  const u8 *aos;           // the loaded records, file order, 109 bytes each — or, after rk_load_packed (aos == nullptr):
  const uint4 *pk_key;     //   {xStart, yStart, length, ident}
  const uint4 *pk_rest;    //   {xEnd, yEnd, score, similarity bits}
  const u8 *pk_strand;
  const u32 *order, *gid;  // result arrays (output order)
  const u8 *repval;
  const float *identity;
  u32 first_line, n_lines;
  char *text;              // out: n_lines lines, back to back
  u32 *total_bytes;        // out (device): bytes written
  u32 *line_len, *line_off;  // set by launch_format (carved from its work area)
};
u64 format_work_bytes(u32 n_lines);
constexpr u32 RK_FORMAT_MAX_LINE = 208;  // upper bound of one line in bytes
int launch_format(FormatArgs a, void *work, cudaStream_t st);

// K7 (k7_dist.cu): one comparison partitioned over several GPUs — cuts, routing, row movers, forest over peer memory
constexpr int DIST_BINS = 4096;       // coarse histogram bins a range partition is cut on
constexpr int DIST_MAX_RANKS = 16;
struct PeerTable {                    // what a rank needs to follow a parent chain across GPUs
  const u64 *res[DIST_MAX_RANKS];     // every rank's per-fragment word (k_chase_local), mapped peer memory
  u32 roff[DIST_MAX_RANKS + 1];       // first global rank of every rank
  int nr, me;
};
struct ScatterTable {                 // positions 0..n of a kernel's output in nr consecutive blocks, block d stored on rank d
  u32 start[DIST_MAX_RANKS + 1];      // first position of every block
  u32 dst_off[DIST_MAX_RANKS];        // where block d starts in rank d's buffer
  void *out[DIST_MAX_RANKS];          // that buffer on every rank (mapped peer memory; this rank's own for d == me)
  int nr;
};
int dist_coarse_hist(const u32 *keys, u32 n, int shift, int pre_shift, u32 drop_key, u32 *hist, cudaStream_t st);
int dist_cuts_from_hist(const u32 *hist_all, u64 row_stride, int nr, int shift, u32 *cuts, cudaStream_t st,
                        const u32 *gid_total = nullptr, u64 line_cap = 0);
int dist_cuts_gid(const u32 *nroots, u32 stride, int nr, u32 *cuts, u32 *total, cudaStream_t st);
int dist_cuts_x(const u32 *cuts0, int nr, Geometry g, const u32 *link_x, u32 *cuts_x, cudaStream_t st);
u64 dist_split_work_bytes(u64 n);
int dist_count_plain(const u32 *keys, u32 n, const u32 *cuts, int nr, u32 drop_key, u32 *tile_cnt, u32 *counts, cudaStream_t st,
                     const u32 *n_ptr = nullptr);
int dist_push_records(const u32 *key0, u32 n, const u32 *cuts, int nr, u32 drop_key, const uint4 *rec, uint2 *const *outs, u32 out_cap,
                      u32 *tile_cnt, const u32 *counts_all, u32 row_stride, int me, cudaStream_t st);
int dist_push_gid(const u32 *gid_rank, const uint4 *hfi_r, u32 n, const u32 *cuts, int nr, uint4 *const *outs, u32 out_cap, u32 *tile_cnt,
                  const u32 *counts_all, u32 row_stride, int me, cudaStream_t st);
int dist_split_halo(const u32 *keys2, const uint2 *cl, u32 n, const u32 *cuts_x, int nr, u32 nbx, int me, u32 rank_off, uint4 *out,
                    u32 out_cap, u32 *perm, u32 *tile_cnt, u32 *counts, cudaStream_t st);
int dist_split_axis(const u32 *keys, const uint2 *cl, u32 n, const u32 *cuts, int nr, u32 rank_off, uint4 *out, u32 *perm,
                    u32 *tile_cnt, u32 *counts, cudaStream_t st);
int dist_key0_of_rec(const uint2 *rec6, u32 n, u32 key_base, u32 *key0, HistOut ho, cudaStream_t st);
int dist_unpack_axis_rows(const uint4 *rows, u32 n, u32 key_base, u32 *keys, uint2 *cl, u32 *grank, HistOut ho, cudaStream_t st);
int dist_x_local_keys(u32 *keys2, u32 n, u32 nbx, const u32 *base, const u32 *range, HistOut ho, cudaStream_t st);
int dist_unpack_halo_rows(const uint4 *rows, u32 n, u32 nbx, const u32 *base, const u32 *range, u32 *keys, uint2 *cl, u32 *grank, HistOut ho,
                          cudaStream_t st);
int dist_gid_keys(const uint4 *rows, u32 n, u32 gid_base, u32 *keys, HistOut ho, cudaStream_t st);
int dist_x_owners(const u32 *parent_x, u32 m, u32 nh, u32 rank_off, const u32 *halo_grank, u32 *parent, const ScatterTable &home,
                  cudaStream_t st);
int dist_apply_away(const u32 *away_res, const u32 *away_perm, u32 n, u32 *parent, cudaStream_t st);
int dist_pack_xm(const u32 *parent, const u32 *perm, u32 n, const ScatterTable &owners, cudaStream_t st);
int dist_y_owners(const u32 *parent_y, const u32 *grank, u32 n, const ScatterTable &home, cudaStream_t st);
int dist_merge_y(const u32 *yo_back, const u32 *perm, u32 n, u32 *parent, cudaStream_t st);
u64 dist_scan_work_bytes(u32 m);
int dist_root_scan(const u32 *parent, u32 m, u32 *gidscan, u32 *nroots, void *work, cudaStream_t st);
int dist_chase_local(const u32 *parent, const u32 *gidscan, u32 m, u32 lo, u32 *lroot, u64 *res, u32 *pend_idx, u32 *pend_key, u32 *n_pend,
                     cudaStream_t st);
int dist_chase_ask_count(const u32 *pend_key, u32 bound, const u32 *n_pend, const u32 *roff_dev, int nr, u32 *tile_cnt, u32 *counts,
                         cudaStream_t st);
int dist_chase_ask_push(const u32 *pend_key, u32 bound, const u32 *n_pend, const u32 *roff_dev, int nr, uint4 *const *outs, u32 out_cap,
                        u32 *apos, u32 *tile_cnt, const u32 *counts_all, u32 row_stride, int me, cudaStream_t st);
int dist_chase_answer(const uint4 *queries, u32 n, const u64 *res, u32 lo, const ScatterTable &back, cudaStream_t st);
int dist_chase_apply(const PeerTable &pt, const u32 *nroots, u32 stride, u32 bound, const u32 *pend_idx, const u32 *pend_key, const u32 *apos,
                     const u64 *ans, const u32 *n_pend, u32 *gid_l, u32 *next_idx, u32 *next_key, u32 *n_next, cudaStream_t st);
int dist_chase_finish(const PeerTable &pt, const u32 *nroots, u32 stride, u32 m, const u64 *res, const u32 *lroot, const u32 *pend_idx,
                      const u32 *pend_key, const u32 *n_pend, u32 *gid_l, u32 *gid_rank, cudaStream_t st);
int dist_or_rows(const u32 *all, u64 row_stride, int nr, u64 words, u32 *out, cudaStream_t st);
// line records: every line asks the rank that loaded its record ({file index, line} to the owner of the file range,
// cuts = the ranks' first file indices); the owner answers with the line row, stored at the asking rank's rows[line]
int dist_line_ask_push(const u32 *order, u32 n, const u32 *file_cuts, int nr, uint4 *const *outs, u32 out_cap, u32 *tile_cnt,
                       const u32 *counts_all, u32 row_stride, int me, cudaStream_t st);
// (the owner's rows: its 109-byte records aos, or its compact rows pk when aos is null)
int dist_line_answer(const uint4 *requests, u32 n, const u8 *aos, const PackedRows &pk, u32 file_lo, const ScatterTable &back,
                     cudaStream_t st);

// sort_groups as a function of (groups, diag_func): h = |y - d| per member, member index, zero identity (sol.cu)
int launch_member_keys(const u64 *y, const u64 *d, u32 m, u32 *h, u32 *idx, float *zero, u32 *err, cudaStream_t st);

// K8: per-group statistics over the output arrays (same layout as rk_group_stats of include/rk_b200.h)
struct rk_group_stats_dev {
  u32 count, x_lo, y_lo, first_line;
  u64 x_hi, y_hi;
  double mean_identity, multiplicity;
};
// K8's per-group accumulators: integers only, so their final values do not depend on the order of the atomics
struct StatsAcc {
  u32 count, x_lo, y_lo, first_line;
  u64 x_hi, y_hi, len_sum;
  u64 digit[4];    // identity * 2^49 in 32-bit digits, each column summed over the members
  u64 n_nan_inf;   // NaN members in the low word, +inf members in the high word
};
// The span fields come from rec4[2 * order[j]] (one GPU) or from rows[j] (rows != nullptr: a rank of a partitioned
// comparison, whose groups gid_base .. gid_base+n_groups-1 are all on the rank and whose line j is line line_off + j).
// acc: n_groups accumulators of scratch; *err ends nonzero when an identity lies outside K1's bound (see k8_stats.cu).
int launch_group_stats(const u32 *out_order, const u32 *out_gid, const float *out_identity, const uint4 *rec4, const LineRow *rows,
                       u32 m, u32 n_groups, u32 gid_base, u32 line_off, rk_group_stats_dev *st, StatsAcc *acc, u32 *err,
                       cudaStream_t stream);

// K9 (k9_csv.cu): CSV rows parsed on the device (rk_load_csv).  Row status bytes:
constexpr u8 CSV_REJECT = 0, CSV_ACCEPT = 1, CSV_HOST = 2, CSV_HOST_ACCEPT = 3;  // host: readFragment decides
constexpr u8 CSV_WIDE = 4;  // an accepted row with a value of 33 or more bits
constexpr u32 CSV_COUNT_TILE = 4096;  // bytes per CTA of the newline count (256 threads x 16 bytes)
inline u64 csv_count_tiles(u64 bytes) { return (bytes + CSV_COUNT_TILE - 1) / CSV_COUNT_TILE; }
struct CsvCounters {
  u32 n_lines;     // '\n' in the text (the scan total of the tile counts)
  u32 n_host;      // rows appended to the host list
  u32 n_accepted;  // rows accepted on the device
  u32 wide;        // an accepted row is wide
};
struct CsvOut {  // where the accepted rows go: the compact arrays, or the 109-byte records when aos is set
  uint4 *key4, *rest4;
  u8 *strand;
  u8 *aos;
};
// '\n' counts of count tiles tile0 .. tile0 + n_tiles (the text up to the end of them must be on the device)
int launch_csv_count(const u8 *text, u64 bytes, u64 tile0, u64 n_tiles, u32 *tile_cnt, cudaStream_t st);
u64 csv_scan_words(u64 n);  // the scan's work words for n elements (rk_scan.cuh: scan_work_words)
// exclusive scan of the tile counts in place (bsum: csv_scan_words(tiles) words); the total to cnt->n_lines
int launch_csv_tile_scan(u32 *tile_cnt, u64 n_tiles, u32 *bsum, CsvCounters *cnt, cudaStream_t st);
// the start offset of every row from the scanned tile counts, start[n_rows] = bytes + 1
int launch_csv_starts(const u8 *text, u64 bytes, const u32 *tile_base, u64 *start, u64 n_rows, cudaStream_t st);
// status of every row; host rows appended to host_list (cnt->n_host), rows accepted here counted (cnt->n_accepted),
// cnt->wide raised by a wide accepted row
int launch_csv_classify(const u8 *text, u64 bytes, const u64 *start, u64 n_rows, u8 *status, u32 *host_list, CsvCounters *cnt,
                        cudaStream_t st);
// {start, end} of the listed rows; their bytes back to back from dst + off[i]
int launch_csv_host_spans(const u32 *rows, u32 n, const u64 *start, ulonglong2 *spans, cudaStream_t st);
int launch_csv_gather(const u8 *text, const ulonglong2 *spans, const u64 *off, u32 n, u8 *dst, cudaStream_t st);
// the accepted rows at their file-order slots: host_rows / host_recs are the rows readFragment accepted on the host
// (row index, 109-byte record); slot: n_rows words, bsum: csv_scan_words(n_rows)
int launch_csv_emit(const u8 *text, u64 bytes, const u64 *start, u64 n_rows, u8 *status, const u32 *host_rows, u32 n_host_acc,
                    const u8 *host_recs, u32 *slot, u32 *bsum, CsvOut o, cudaStream_t st);
// host side: readFragment (the host parser's rule for one row) into a 109-byte record; false = the row is rejected
bool csv_read_row_host(const char *line, u64 len, void *record);

u64 order_scratch_bytes(u64 m);
void order_carve(OrderArgs &a, void *scratch, u64 m);  // sets packed .. worklist, work_cap
int launch_order(const OrderArgs &a, cudaStream_t st);

}  // namespace rk
