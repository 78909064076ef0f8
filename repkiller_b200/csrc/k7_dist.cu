// K7 — the kernels of ONE comparison partitioned over several GPUs (multi.cu drives them; SURVEY.md §8e).
//
// The reference is single-process (no distributed backend, SURVEY.md §5); what has to be preserved is the order its
// greedy loop visits fragments in (/root/reference/src/commonFunctions.cpp:51-77) and the reach of one
// get_associated_group query (/root/reference/src/SequenceOcupationList.cpp:47-89: the own center/100 bucket and at
// most one neighbour).  Every routing decision below is a function of key VALUES (cuts), never of a GPU id, and ties are
// always broken by the global processing rank, so the result is bit-identical for any number of GPUs:
//   * exchange 1: fragments go to the GPU that owns their xStart/10 range (processing order, generate_diagonal_func buckets);
//   * X pass at home: the X super-bucket of a fragment starts at or after its xStart/100 bucket, so only fragments whose
//     center reaches past the next cut travel ("halo", to higher GPUs only), and their owners travel back;
//   * Y pass: fragments are regrouped by Y super-bucket ranges; only the 1-byte "matched in X" flags and the 4-byte
//     owners move per (len_ratio, pos_ratio) pair;
//   * forest: parents always have a smaller global rank; a chain that leaves the GPU is followed through the peers'
//     parent arrays over NVLink (peer loads), group ids = per-GPU root scan + the root counts of the lower GPUs;
//   * output: fragments go to the GPU that owns their group-id range for sort_groups.
#include "rk_common.cuh"
#include "rk_scan.cuh"

namespace rk {

// ---- cuts: contiguous key ranges of about equal population ---------------------------------------------------------

// bin = key >> shift (at most DIST_BINS bins); keys equal to drop_key are not counted (the never-visited last X bucket)
__global__ void __launch_bounds__(256) k_coarse_hist(const u32 *__restrict__ keys, u32 n, int shift, int pre_shift, u32 drop_key,
                                                     u32 *__restrict__ hist) {
  __shared__ u32 s_h[DIST_BINS];
  for (u32 i = threadIdx.x; i < (u32)DIST_BINS; i += blockDim.x) s_h[i] = 0;
  __syncthreads();
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u32 k = keys[i] >> pre_shift;
    if (k != drop_key) atomicAdd(&s_h[min(k >> shift, (u32)DIST_BINS - 1)], 1u);
  }
  __syncthreads();
  for (u32 i = threadIdx.x; i < (u32)DIST_BINS; i += blockDim.x)
    if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
}

// one CTA of 1024 threads: the ranks' histograms (row r at hist_all + r * row_stride words) summed, cuts[r] = first bin boundary (as a key value)
// at which the cumulative count reaches total*r/nr; cuts[0] = 0, cuts[nr] = 0xFFFFFFFF.  Identical on every rank.
// gid_total (output exchange only): the bins are blocks of 2^shift group ids and *gid_total is the number of groups; a bin
// then weighs 3 per line + 8 per line beyond one per group — sort_groups costs per member of a group with several members,
// and the groups founded early (low ids) are the large ones: with equal LINE counts rank 0 needed 0.63 ms for its range
// where the last rank needed 0.37 ms (8 GPUs, 10M lines each).
struct CutsSmem {
  unsigned long long cum[DIST_BINS + 1];  // exclusive prefix of the (weighted) bin counts
  u32 lin[DIST_BINS + 1];                 // exclusive prefix of the plain bin counts (lines)
  unsigned long long wtot[32];
  u32 ltot[32], lmax[32];
};
// first c in [0, n] with a[c] >= x (a ascending; n + 1 entries)
template <class T>
__device__ __forceinline__ u32 first_ge(const T *a, u32 n, T x) {
  u32 lo = 0, hi = n;
  while (lo < hi) {
    const u32 mid = (lo + hi) >> 1;
    if (a[mid] >= x) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}
// line_cap (weighted cuts only): no rank's range may hold more than line_cap lines — the weighted cut is moved to the nearest
// bin boundary that leaves every rank, this one and the ones after it, within its rows (possible whenever the lines fit at all)
__global__ void __launch_bounds__(1024) k_cuts_from_hist(const u32 *__restrict__ hist_all, u64 row_stride, int nr, int shift,
                                                         u32 *__restrict__ cuts, const u32 *__restrict__ gid_total, u64 line_cap) {
  extern __shared__ __align__(16) unsigned char cuts_smem_raw[];
  CutsSmem &sm = *reinterpret_cast<CutsSmem *>(cuts_smem_raw);
  constexpr int PER = DIST_BINS / 1024;
  const u32 lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  unsigned long long v[PER], sum = 0;
  u32 l[PER], lsum = 0, lbig = 0;
  for (int j = 0; j < PER; ++j) {
    const u32 b = threadIdx.x * PER + j;
    unsigned long long c = 0;
    for (int r = 0; r < nr; ++r) c += hist_all[(u64)r * row_stride + b];
    l[j] = (u32)c;
    lsum += (u32)c;
    lbig = max(lbig, (u32)c);
    if (gid_total) {
      const unsigned long long first = (unsigned long long)b << shift, total_g = *gid_total;
      const unsigned long long groups = first >= total_g ? 0 : (total_g - first < (1ull << shift) ? total_g - first : (1ull << shift));
      c = 3 * c + 8 * (c > groups ? c - groups : 0);
    }
    v[j] = c;
    sum += c;
  }
  // block-wide exclusive scan of (sum, lsum): warp scan, then the 32 warp totals by warp 0
  unsigned long long inc = sum;
  u32 linc = lsum;
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
    const u32 lt = __shfl_up_sync(0xFFFFFFFFu, linc, d);
    if (lane >= (u32)d) inc += t, linc += lt;
  }
  lbig = __reduce_max_sync(0xFFFFFFFFu, lbig);
  if (lane == 31) sm.wtot[w] = inc, sm.ltot[w] = linc, sm.lmax[w] = lbig;
  __syncthreads();
  if (w == 0) {
    unsigned long long t = sm.wtot[lane];
    u32 lt = sm.ltot[lane];
    const unsigned long long own = t;
    const u32 lown = lt;
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long u = __shfl_up_sync(0xFFFFFFFFu, t, d);
      const u32 lu = __shfl_up_sync(0xFFFFFFFFu, lt, d);
      if (lane >= (u32)d) t += u, lt += lu;
    }
    const u32 big = __reduce_max_sync(0xFFFFFFFFu, sm.lmax[lane]);
    sm.wtot[lane] = t - own, sm.ltot[lane] = lt - lown;
    if (lane == 31) sm.cum[DIST_BINS] = t, sm.lin[DIST_BINS] = lt, sm.lmax[0] = big;
  }
  __syncthreads();
  unsigned long long run = sm.wtot[w] + inc - sum;
  u32 lrun = sm.ltot[w] + linc - lsum;
  for (int j = 0; j < PER; ++j) {
    sm.cum[threadIdx.x * PER + j] = run, sm.lin[threadIdx.x * PER + j] = lrun;  // exclusive
    run += v[j], lrun += l[j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long total = sm.cum[DIST_BINS];
    const unsigned long long lines = sm.lin[DIST_BINS];
    u32 prev = 0;
    cuts[0] = 0;
    for (int r = 1; r < nr; ++r) {
      u32 c = first_ge(sm.cum, (u32)DIST_BINS, total * (unsigned long long)r / (unsigned long long)nr);
      if (line_cap) {
        // what the ranks r.. can hold — each counted one bin short, so that a boundary between this bound and the bound of
        // rank r-1's own rows below always exists (cuts fall on bin boundaries)
        const unsigned long long big = sm.lmax[0];
        const unsigned long long rest = (unsigned long long)(nr - r) * (line_cap > big ? line_cap - big : 0);
        if (lines > rest) {
          const u32 lo = first_ge(sm.lin, (u32)DIST_BINS, (u32)(lines - rest));
          c = c < lo ? lo : c;
        }
        const unsigned long long room = (unsigned long long)sm.lin[prev] + line_cap;  // what rank r-1 can hold
        if (room < lines) {
          const u32 over = first_ge(sm.lin, (u32)DIST_BINS, (u32)(room + 1));  // first boundary that is too far
          c = c >= over ? (over > 0 ? over - 1 : 0) : c;
        }
      }
      c = c < prev ? prev : c;
      prev = c;
      const unsigned long long key = (unsigned long long)c << shift;
      cuts[r] = key > 0xFFFFFFFEull ? 0xFFFFFFFEu : (u32)key;
    }
    cuts[nr] = 0xFFFFFFFFu;
  }
}

// group-id cuts: cuts[r] = floor(total_groups * r / nr) from the all-gathered root counts; also the total
__global__ void k_cuts_gid(const u32 *__restrict__ nroots, u32 stride, int nr, u32 *__restrict__ cuts, u32 *__restrict__ total_out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    unsigned long long total = 0;
    for (int r = 0; r < nr; ++r) total += nroots[(u64)r * stride];
    for (int r = 0; r < nr; ++r) cuts[r] = (u32)(total * (unsigned long long)r / (unsigned long long)nr);
    cuts[nr] = 0xFFFFFFFFu;
    *total_out = (u32)total;
  }
}

// X cuts: the first super-bucket (per strand class) a rank owns = run start of the bucket its xStart/10 range begins in
__global__ void k_cuts_x(const u32 *__restrict__ cuts0, int nr, Geometry g, const u32 *__restrict__ link_x, u32 *__restrict__ cuts_x) {
  const int t = threadIdx.x;
  if (t >= 2 * nr) return;
  const int s = t / nr, r = t % nr;
  u32 b = 0;
  if (r > 0) {
    const u32 c = cuts0[r];
    b = min(c / (DIVISOR / XBUCKET), g.nbx - 1);
  }
  // bit 0 of every strand class is never set (nothing links bucket 0 to a predecessor), so run_start stays in class s
  cuts_x[t] = r == 0 ? (u32)s * g.nbx : run_start(link_x, (u32)s * g.nbx + b);
}

// ---- routing: a stable split of the local elements by destination rank, fused with the packing of the rows ----------
// dest(key) = largest r with cuts[r] <= key; key == drop_key -> nr ("nowhere": the never-visited last X bucket).
// MODE 0: plain keys against cuts[nr+1].  MODE 1 (X halo): key = keys[i] >> 1 against the per-strand table cuts[2][nr],
// strand class = key >= nbx; elements that stay on this rank get dest nr as well (only the travellers are packed).
// Three launches: per-tile counts -> exclusive offsets (per destination over the tiles) -> every tile writes its rows at
// their final place in the send buffer, reading its inputs coalesced.  Stable: inside a destination the elements keep
// their order (file order / processing order), which is what carries the reference's visiting order across GPUs.
struct RouteArgs {
  const u32 *keys;
  u32 n;
  const u32 *cuts;
  int nr, me;
  u32 drop_key, nbx;
  u32 out_cap;  // rows the send buffer holds: nothing is written past it (the host checks the counts afterwards)
  const u32 *n_ptr;  // when set: the number of elements lives on the device (n is then the launch bound)
};
__device__ __forceinline__ u32 route_n(const RouteArgs &a) { return a.n_ptr ? min(*a.n_ptr, a.n) : a.n; }
constexpr int SPLIT_ROUNDS = 8;
constexpr int SPLIT_TILE = 256 * SPLIT_ROUNDS;
constexpr int NRP = DIST_MAX_RANKS + 1;

template <int MODE>
__device__ __forceinline__ int route_of(u32 k, const u32 *s_cuts, const RouteArgs &a) {
  int d = 0;
  if (MODE == 1) {
    k >>= 1;
    const u32 *c = s_cuts + (k >= a.nbx ? a.nr : 0);
    for (int r = 1; r < a.nr; ++r) d = c[r] <= k ? r : d;
    if (d == a.me) d = a.nr;
  } else if (k == a.drop_key) {
    d = a.nr;
  } else {
    for (int r = 1; r < a.nr; ++r) d = s_cuts[r] <= k ? r : d;
  }
  return d;
}

template <int MODE>
__global__ void __launch_bounds__(256) k_route_count(RouteArgs a, u32 *__restrict__ tile_cnt, u32 *__restrict__ counts) {
  __shared__ u32 s_cuts[2 * DIST_MAX_RANKS + 2];
  __shared__ u32 s_cnt[NRP];
  const int ncut = MODE == 1 ? 2 * a.nr : a.nr + 1;
  if (threadIdx.x < (u32)ncut) s_cuts[threadIdx.x] = a.cuts[threadIdx.x];
  if (threadIdx.x < (u32)NRP) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const u32 lane = threadIdx.x & 31;
  u32 acc = 0;  // lane r accumulates destination r
  const u64 base = (u64)blockIdx.x * SPLIT_TILE;
#pragma unroll
  for (int j = 0; j < SPLIT_ROUNDS; ++j) {
    const u64 i = base + (u64)j * 256 + threadIdx.x;
    const int d = i < route_n(a) ? route_of<MODE>(a.keys[i], s_cuts, a) : -1;
    for (int r = 0; r <= a.nr; ++r) {
      const u32 b = __ballot_sync(0xFFFFFFFFu, d == r);
      if (lane == (u32)r) acc += __popc(b);
    }
  }
  if (lane <= (u32)a.nr && acc) atomicAdd(&s_cnt[lane], acc);
  __syncthreads();
  if (threadIdx.x <= (u32)a.nr) {
    const u32 c = s_cnt[threadIdx.x];
    tile_cnt[(u64)blockIdx.x * NRP + threadIdx.x] = c;
    if (c) atomicAdd(&counts[threadIdx.x], c);
  }
}

// block d: tile_cnt[.][d] -> exclusive prefix over the tiles + where this rank's block for destination d starts:
//   in the local send buffer (counts_all == nullptr): after the blocks for the lower destinations;
//   in rank d's receive buffer (pushing straight into peer memory): after the blocks of the lower SOURCE ranks, from the
//   all-gathered count matrix counts_all[s * row_stride + d] = what rank s sends to d.
__global__ void __launch_bounds__(1024) k_tile_offsets(u32 *__restrict__ tile_cnt, u32 tiles, const u32 *__restrict__ counts,
                                                       const u32 *__restrict__ counts_all, u32 row_stride, int me) {
  const int d = blockIdx.x;
  __shared__ u32 s_carry;
  if (threadIdx.x == 0) {
    u32 base = 0;
    if (counts_all) {
      for (int r = 0; r < me; ++r) base += counts_all[(u64)r * row_stride + d];
    } else {
      for (int r = 0; r < d; ++r) base += counts[r];
    }
    s_carry = base;
  }
  __syncthreads();
  for (u32 t0 = 0; t0 < tiles; t0 += 1024) {
    const u32 t = t0 + threadIdx.x;
    const u32 v = t < tiles ? tile_cnt[(u64)t * NRP + d] : 0;
    u32 total;
    const u32 ex = block_excl_scan<1024>(v, &total);
    const u32 c = s_carry;
    if (t < tiles) tile_cnt[(u64)t * NRP + d] = c + ex;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = c + total;
    __syncthreads();
  }
}

// `out` of a payload: one pointer per destination — the local send buffer for all of them, or every rank's receive buffer
// (mapped peer memory: the rows then cross NVLink as the stores of this kernel, no send buffer and no copy in between)
template <class W>
struct RowOutsT {
  W *p[DIST_MAX_RANKS];
};
typedef RowOutsT<uint4> RowOuts;
// exchange 1: the six words of a record that the owner needs — {xStart, yStart} {length, flags} {identity, file index} —
// 24 bytes on the wire instead of the 32-byte rec4 form K1 writes (25 % of the largest exchange)
struct PayRec24 {
  typedef uint2 Word;
  static constexpr int WPR = 3;
  const uint4 *rec;
  RowOutsT<uint2> out;
  __device__ __forceinline__ void load(u32 i, uint2 *v) const {
    const uint4 a = rec[2 * (u64)i], b = rec[2 * (u64)i + 1];
    v[0] = make_uint2(a.x, a.y), v[1] = make_uint2(a.z, a.w), v[2] = make_uint2(b.x, b.y);
  }
};
struct PayAxisRow {  // one axis pass: {key, center, length, global rank}
  const u32 *keys;
  const uint2 *cl;
  u32 rank_off, key_and;
  uint4 *out;
  __device__ __forceinline__ void operator()(u32 i, int, u32 pos) const {
    const uint2 c = cl[i];
    out[pos] = make_uint4(keys[i] & key_and, c.x, c.y, rank_off + i);
  }
};
struct PayGidRow {  // output exchange: {h, file index, identity bits, gid}
  typedef uint4 Word;
  static constexpr int WPR = 1;
  const uint4 *hfi_r;
  const u32 *gid_rank;
  RowOuts out;
  __device__ __forceinline__ void load(u32 i, uint4 *v) const {
    v[0] = hfi_r[i];
    v[0].w = gid_rank[i];
  }
};

struct PayQuery {  // forest: "what is behind global rank keys[i]?" asked of the rank that owns it
  typedef uint4 Word;
  static constexpr int WPR = 1;
  const u32 *keys;
  RowOuts out;
  __device__ __forceinline__ void load(u32 i, uint4 *v) const { v[0] = make_uint4(keys[i], 0u, 0u, 0u); }
};

struct PayLineReq {  // line records: "send me the record of file index keys[i] for my line i", asked of the rank that loaded it
  typedef uint4 Word;
  static constexpr int WPR = 1;
  const u32 *keys;
  RowOuts out;
  __device__ __forceinline__ void load(u32 i, uint4 *v) const { v[0] = make_uint4(keys[i], i, 0u, 0u); }
};

template <int MODE, class Pay>
__global__ void __launch_bounds__(256) k_split_pack(RouteArgs a, const u32 *__restrict__ tile_off, Pay pay, u32 *__restrict__ perm) {
  __shared__ u32 s_cuts[2 * DIST_MAX_RANKS + 2];
  __shared__ u32 s_run[NRP];
  __shared__ u32 s_w[8][NRP];
  const int ncut = MODE == 1 ? 2 * a.nr : a.nr + 1;
  const u32 tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid < (u32)ncut) s_cuts[tid] = a.cuts[tid];
  if (tid < (u32)NRP) s_run[tid] = tid < (u32)a.nr ? tile_off[(u64)blockIdx.x * NRP + tid] : 0;
  __syncthreads();
  const u32 lt = lanemask_lt();
  const u64 base = (u64)blockIdx.x * SPLIT_TILE;
  for (int j = 0; j < SPLIT_ROUNDS; ++j) {
    const u64 i = base + (u64)j * 256 + tid;
    const int d = i < a.n ? route_of<MODE>(a.keys[i], s_cuts, a) : -1;
    u32 before = 0, cnt = 0;
    for (int r = 0; r < a.nr; ++r) {
      const u32 b = __ballot_sync(0xFFFFFFFFu, d == r);
      if (d == r) before = __popc(b & lt);
      if (lane == (u32)r) cnt = __popc(b);
    }
    if (lane < (u32)a.nr) s_w[w][lane] = cnt;
    __syncthreads();
    if (d >= 0 && d < a.nr) {
      u32 pos = s_run[d] + before;
      for (u32 q = 0; q < w; ++q) pos += s_w[q][d];
      if (pos < a.out_cap) {
        pay((u32)i, d, pos);
        if (perm) perm[pos] = (u32)i;
      }
    }
    __syncthreads();
    if (tid < (u32)a.nr) {
      u32 t = 0;
      for (int q = 0; q < 8; ++q) t += s_w[q][tid];
      s_run[tid] += t;
    }
    __syncthreads();
  }
}

// The push form of the split: rows of a tile are first gathered in shared memory, destination by destination, and then
// stored to the destination ranks' receive buffers as contiguous runs (consecutive threads -> consecutive 16-byte words).
// Row-by-row stores from the routing loop reach a peer as scattered 32-byte writes, which NVLink moves at a fraction of
// its rate (measured at 8 GPUs: 1.7 ms per step in these kernels against 1.05 ms for the same rows through the copy engines).
template <class W, int WPR>
struct PushSmem {
  W rows[SPLIT_TILE * WPR];
  unsigned char dest[SPLIT_TILE];
};
// apos (optional): for every element, the position of its row in this rank's SEND order (blocks by destination) — where
// a value that the destination returns block by block will land; needs the count matrix to undo the receiver offsets.
template <class Pay>
__global__ void __launch_bounds__(256) k_push_rows(RouteArgs a, const u32 *__restrict__ tile_off, Pay pay, u32 *__restrict__ apos,
                                                   const u32 *__restrict__ counts_all, u32 row_stride) {
  typedef typename Pay::Word W;
  constexpr int WPR = Pay::WPR;
  extern __shared__ __align__(16) unsigned char push_smem_raw[];
  PushSmem<W, WPR> &sm = *reinterpret_cast<PushSmem<W, WPR> *>(push_smem_raw);
  __shared__ u32 s_cuts[DIST_MAX_RANKS + 2];
  __shared__ u32 s_run[NRP], s_start[NRP], s_goff[NRP];
  __shared__ u32 s_w[8][NRP];
  const u32 tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid < (u32)(a.nr + 1)) s_cuts[tid] = a.cuts[tid];
  __shared__ u32 s_back[NRP];  // send-order position minus receiver position of this rank's block for destination d
  if (tid < (u32)NRP) {
    s_run[tid] = 0;
    s_goff[tid] = tid < (u32)a.nr ? tile_off[(u64)blockIdx.x * NRP + tid] : 0;
    u32 soff = 0, poff = 0;
    if (apos && tid < (u32)a.nr) {
      for (int r = 0; r < a.me; ++r) poff += counts_all[(u64)r * row_stride + tid];
      for (u32 r = 0; r < tid; ++r) soff += counts_all[(u64)a.me * row_stride + r];
    }
    s_back[tid] = soff - poff;
  }
  __syncthreads();
  const u32 lt = lanemask_lt();
  const u64 base = (u64)blockIdx.x * SPLIT_TILE;
  int dsts[SPLIT_ROUNDS];
  u32 ranks[SPLIT_ROUNDS];
  // pass 1: destination and stable rank inside the destination (within the tile) of every element
#pragma unroll
  for (int j = 0; j < SPLIT_ROUNDS; ++j) {
    const u64 i = base + (u64)j * 256 + tid;
    const int d = i < route_n(a) ? route_of<0>(a.keys[i], s_cuts, a) : -1;
    u32 before = 0, cnt = 0;
    for (int r = 0; r < a.nr; ++r) {
      const u32 b = __ballot_sync(0xFFFFFFFFu, d == r);
      if (d == r) before = __popc(b & lt);
      if (lane == (u32)r) cnt = __popc(b);
    }
    if (lane < (u32)a.nr) s_w[w][lane] = cnt;
    __syncthreads();
    u32 pos = 0;
    if (d >= 0 && d < a.nr) {
      pos = s_run[d] + before;
      for (u32 q = 0; q < w; ++q) pos += s_w[q][d];
    }
    dsts[j] = d;
    ranks[j] = pos;
    __syncthreads();
    if (tid < (u32)a.nr) {
      u32 t = 0;
      for (int q = 0; q < 8; ++q) t += s_w[q][tid];
      s_run[tid] += t;
    }
    __syncthreads();
  }
  if (tid == 0) {
    u32 run = 0;
    for (int r = 0; r < a.nr; ++r) {
      s_start[r] = run;
      run += s_run[r];
    }
    s_start[a.nr] = run;
  }
  __syncthreads();
  // pass 2: the rows into shared memory, grouped by destination
#pragma unroll
  for (int j = 0; j < SPLIT_ROUNDS; ++j) {
    const int d = dsts[j];
    if (d >= 0 && d < a.nr) {
      const u32 slot = s_start[d] + ranks[j];
      W v[WPR];
      pay.load((u32)(base + (u64)j * 256 + tid), v);
      if (apos) apos[base + (u64)j * 256 + tid] = s_goff[d] + ranks[j] + s_back[d];
#pragma unroll
      for (int q = 0; q < WPR; ++q) sm.rows[slot * WPR + q] = v[q];
      sm.dest[slot] = (unsigned char)d;
    }
  }
  __syncthreads();
  // copy-out: consecutive threads store consecutive words of a destination's run
  const u32 total = s_start[a.nr];
  for (u32 x = tid; x < total * WPR; x += 256) {
    const u32 slot = x / WPR, q = x % WPR;
    const int d = sm.dest[slot];
    const u32 pos = s_goff[d] + (slot - s_start[d]);
    if (pos < a.out_cap) pay.out.p[d][(u64)pos * WPR + q] = sm.rows[x];
  }
}

// ---- row movers ----------------------------------------------------------------------------------------------------

// The three kernels below produce the keys of a sort; like K1/K2 on one GPU they count the digits of those keys on the way
// (HistOut), so that the sort needs no histogram pass of its own.  Warp-uniform loops: every lane votes in hist_add.

// key0 = xStart / 10 of the arrived records (24-byte rows; the sort key of the processing order)
__global__ void __launch_bounds__(256) k_key0_of_rec(const uint2 *__restrict__ rec6, u32 n, u32 key_base, u32 *__restrict__ key0, HistOut ho) {
  __shared__ u32 s_h[HIST_PASSES][HIST_RADIX];
  hist_zero(s_h);
  __syncthreads();
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 i = base + threadIdx.x;
    u32 k = 0;
    if (i < n) key0[i] = k = rec6[3 * i].x / XBUCKET - key_base;  // relative to the rank's first key: fewer sort passes
    hist_add(s_h, k, i < n, ho);
  }
  __syncthreads();
  hist_flush(s_h, ho);
}

// X bucket keys of a rank, made local before the X sort: key2 = 2 * (global super-bucket key) + own bit becomes
// 2 * (strand * (R + 1) + min(key - first key of the rank's range in that strand, R)) + own bit — log2(4 (R + 1)) bits
// instead of log2(4 nbx): one radix pass fewer from 4 GPUs on.  Keys past the range (fragments that were sent away as halo:
// their local result is overwritten anyway) share the one extra slot R.
struct XRemap {
  u32 nbx, base[2], range[2], R;
};
__device__ __forceinline__ u32 x_local_key(u32 key2, const XRemap &x) {
  const u32 k = key2 >> 1, s = k >= x.nbx ? 1u : 0u;
  const u32 loc = k - x.base[s];
  return 2u * (s * (x.R + 1u) + (loc < x.range[s] ? loc : x.R)) + (key2 & 1u);
}
__global__ void __launch_bounds__(256) k_x_remap(u32 *__restrict__ keys2, u32 n, XRemap x, HistOut ho) {
  __shared__ u32 s_h[HIST_PASSES][HIST_RADIX];
  hist_zero(s_h);
  __syncthreads();
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 i = base + threadIdx.x;
    u32 k = 0;
    if (i < n) keys2[i] = k = x_local_key(keys2[i], x);
    hist_add(s_h, k, i < n, ho);
  }
  __syncthreads();
  hist_flush(s_h, ho);
}

// arrival of the rows of one axis pass: keys[j], cl[j], grank[j] of row j
template <bool XLOCAL>
__global__ void __launch_bounds__(256) k_unpack_axis_rows(const uint4 *__restrict__ rows, u32 n, u32 key_base, XRemap x, u32 *__restrict__ keys,
                                                          uint2 *__restrict__ cl, u32 *__restrict__ grank, HistOut ho) {
  __shared__ u32 s_h[HIST_PASSES][HIST_RADIX];
  hist_zero(s_h);
  __syncthreads();
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 j = base + threadIdx.x;
    u32 k = 0;
    if (j < n) {
      const uint4 r = rows[j];
      keys[j] = k = XLOCAL ? x_local_key(r.x, x) : r.x - key_base;
      cl[j] = make_uint2(r.y, r.z);
      grank[j] = r.w;
    }
    hist_add(s_h, k, j < n, ho);
  }
  __syncthreads();
  hist_flush(s_h, ho);
}

__global__ void __launch_bounds__(256) k_gid_keys(const uint4 *__restrict__ rows, u32 n, u32 gid_base, u32 *__restrict__ keys, HistOut ho) {
  __shared__ u32 s_h[HIST_PASSES][HIST_RADIX];
  hist_zero(s_h);
  __syncthreads();
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 j = base + threadIdx.x;
    u32 k = 0;
    if (j < n) keys[j] = k = rows[j].w - gid_base;
    hist_add(s_h, k, j < n, ho);
  }
  __syncthreads();
  hist_flush(s_h, ho);
}

// ---- owners: from indices of a rank's working list to global ranks ---------------------------------------------------

// X pass: the working list is [own fragments 0..m) ++ [halo m..m+nh).  parent_x[i] = list index of the owner or NONE.
//   own i  -> parent[i] (global rank) ; halo j -> halo_res[j] (travels back to the fragment's home rank)
// The three small per-pair exchanges (halo owners home, "matched in X" flags to the Y owners, Y owners home) have no
// send buffer either: their values are already grouped by the rank they go to (arrival order = blocks by source, send
// order = blocks by destination), so the kernel that produces them stores each block straight into its rank's buffer.
template <class T>
__device__ __forceinline__ void scatter_store(const ScatterTable &t, u32 j, T v) {
  int d = 0;
  for (int r = 1; r < t.nr; ++r) d = t.start[r] <= j ? r : d;  // block of position j
  reinterpret_cast<T *>(t.out[d])[t.dst_off[d] + (j - t.start[d])] = v;
}

__global__ void __launch_bounds__(256) k_x_owners(const u32 *__restrict__ parent_x, u32 m, u32 nh, u32 rank_off,
                                                  const u32 *__restrict__ halo_grank, u32 *__restrict__ parent, ScatterTable home) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m + nh) return;
  u32 o = parent_x[i];
  if (o != RK_NONE32) o = o < m ? rank_off + o : halo_grank[o - m];
  if (i < m) parent[i] = o;
  else scatter_store<u32>(home, i - m, o);  // a halo fragment: its owner goes to the rank it came from
}
// the owners of the fragments this rank sent away come back in send order: away_perm[t] = local rank of the t-th
__global__ void __launch_bounds__(256) k_apply_away(const u32 *__restrict__ away_res, const u32 *__restrict__ away_perm, u32 n,
                                                    u32 *__restrict__ parent) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) parent[away_perm[t]] = away_res[t];
}
// "matched in the X pass" flags in the order the Y rows were sent, stored at the Y owners
__global__ void __launch_bounds__(256) k_pack_xm(const u32 *__restrict__ parent, const u32 *__restrict__ perm, u32 n, ScatterTable owners) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) scatter_store<u8>(owners, t, parent[perm[t]] != RK_NONE32 ? 1 : 0);
}
// Y pass: parent_y[j] = arrival index of the owner or NONE -> its global rank, stored at the fragment's home rank
__global__ void __launch_bounds__(256) k_y_owners(const u32 *__restrict__ parent_y, const u32 *__restrict__ grank, u32 n, ScatterTable home) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const u32 o = parent_y[j];
  // only the matches travel: every rank fills its yo buffer with NONE before the ranks meet (a few per cent of the
  // fragments have a Y owner)
  if (o != RK_NONE32) scatter_store<u32>(home, j, grank[o]);
}
// the Y owners come back in send order; a fragment matched in X keeps its X owner (commonFunctions.cpp:56-61)
__global__ void __launch_bounds__(256) k_merge_y(const u32 *__restrict__ yo_back, const u32 *__restrict__ perm, u32 n, u32 *__restrict__ parent) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const u32 i = perm[t];
  if (parent[i] == RK_NONE32) parent[i] = yo_back[t];
}

// ---- forest over peer memory ---------------------------------------------------------------------------------------
struct LoadIsRootD {
  const u32 *parent;
  __device__ __forceinline__ u32 operator()(u64 i) const { return parent[i] == RK_NONE32 ? 1u : 0u; }
};
__global__ void k_store_total(const u32 *total, u32 *out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) *out = *total;
}

// Group ids, so that NVLink is only crossed where a chain really leaves the GPU:
//   A  every fragment follows its parents while they are LOCAL to the last local node of its chain (lroot) — a root of the
//      forest, or an "exit" whose parent lives on a lower GPU (parents always have a smaller global rank) — and publishes
//      what a walker arriving at this fragment needs as ONE 64-bit word: res[i] = ROOT | (roots before lroot on this GPU),
//      or the global rank of the exit's parent.  The exits are collected in a pending list (fragment, rank to ask about).
//   B  the pending list is resolved.  In bulk rounds while it is long: the ranks asked about are pushed to their owners
//      (the split/push kernels of the row exchanges), the owners answer with their res[] word, block by block, and an
//      answer is either a root (done) or the next rank to ask about.  A short list is walked by its own threads through
//      the peers' res[] — one 8-byte NVLink read per GPU visited; fine-grained remote reads run at about 1 M per ms, which
//      is fine for a few hundred thousand exits and hopeless for the tens of millions of a dense 1e9-fragment comparison
//      (measured: 412 ms there).
//   C  everybody takes the id of its lroot (a local root: from res; an exit: from B).
constexpr u64 RES_ROOT = 1ull << 63;

// appends (idx, key) pairs of a CTA to a global list through a shared-memory stage (a global atomic per warp on the one list
// counter costs more than the whole chase: measured +0.3 ms on the GPU with the most exits)
struct PendStage {
  static constexpr u32 CAP = 2048;
  u32 idx[CAP], key[CAP];
  u32 n, base;
};
__device__ __forceinline__ void pend_flush(PendStage &sg, u32 *__restrict__ out_idx, u32 *__restrict__ out_key, u32 *__restrict__ n_out) {
  if (threadIdx.x == 0) sg.base = sg.n ? atomicAdd(n_out, sg.n) : 0;
  __syncthreads();
  for (u32 k = threadIdx.x; k < sg.n; k += blockDim.x) out_idx[sg.base + k] = sg.idx[k], out_key[sg.base + k] = sg.key[k];
  __syncthreads();
  if (threadIdx.x == 0) sg.n = 0;
  __syncthreads();
}
// every thread of the CTA calls this once per loop iteration (uniform control flow); 256 threads add at most 256 pairs
__device__ __forceinline__ void pend_push(PendStage &sg, bool add, u32 idx, u32 key, u32 *__restrict__ out_idx, u32 *__restrict__ out_key,
                                          u32 *__restrict__ n_out) {
  const u32 lane = threadIdx.x & 31;
  const u32 bal = __ballot_sync(0xFFFFFFFFu, add);
  if (bal) {
    u32 off = 0;
    const int leader = __ffs(bal) - 1;
    if ((int)lane == leader) off = atomicAdd(&sg.n, (u32)__popc(bal));
    off = __shfl_sync(0xFFFFFFFFu, off, leader);
    if (add) {
      const u32 slot = off + __popc(bal & lanemask_lt());
      sg.idx[slot] = idx, sg.key[slot] = key;
    }
  }
  __syncthreads();
  if (sg.n > PendStage::CAP - 256) pend_flush(sg, out_idx, out_key, n_out);
}

__global__ void __launch_bounds__(256) k_chase_local(const u32 *__restrict__ parent, const u32 *__restrict__ gidscan, u32 m, u32 lo,
                                                     u32 *__restrict__ lroot, u64 *__restrict__ res, u32 *__restrict__ pend_idx,
                                                     u32 *__restrict__ pend_key, u32 *__restrict__ n_pend) {
  __shared__ PendStage sg;
  if (threadIdx.x == 0) sg.n = 0;
  __syncthreads();
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < m; base += (u64)gridDim.x * blockDim.x) {
    const u64 i = base + threadIdx.x;
    bool is_exit = false;
    u32 p = RK_NONE32;
    if (i < m) {
      u32 r = (u32)i;
      for (;;) {
        p = parent[r];
        if (p == RK_NONE32 || p < lo) break;  // a root, or the parent is on a lower GPU
        r = p - lo;                           // p < own global rank: stays inside this GPU's range
      }
      lroot[i] = r;
      res[i] = p == RK_NONE32 ? (RES_ROOT | gidscan[r]) : (u64)p;
      is_exit = r == (u32)i && p != RK_NONE32;
    }
    pend_push(sg, is_exit, (u32)i, p, pend_idx, pend_key, n_pend);
  }
  pend_flush(sg, pend_idx, pend_key, n_pend);
}

// roots on every rank: nroots[r * stride] (a column of the all-gathered count matrix)
__device__ __forceinline__ void load_groot(u32 *s_groot, const u32 *__restrict__ nroots, u32 stride, int nr) {
  if (threadIdx.x == 0) {
    u32 run = 0;
    for (int r = 0; r < nr; ++r) {
      s_groot[r] = run;
      run += nroots[(u64)r * stride];
    }
  }
  __syncthreads();
}

// B, short list: every pending fragment walks through the peers' res[]
__global__ void __launch_bounds__(256) k_chase_walk(PeerTable pt, const u32 *__restrict__ nroots, u32 stride, const u32 *__restrict__ pend_idx,
                                                    const u32 *__restrict__ pend_key, const u32 *__restrict__ n_pend, u32 *__restrict__ gid_l) {
  __shared__ u32 s_groot[DIST_MAX_RANKS];
  load_groot(s_groot, nroots, stride, pt.nr);
  const u32 n = *n_pend;
  for (u32 t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
    int s = pt.me;
    u64 w = pend_key[t];  // the global rank to ask about, on a lower GPU
    do {
      const u32 p = (u32)w;
      while (p < pt.roff[s]) --s;  // global rank p lives on the last rank whose offset is <= p
      w = pt.res[s][p - pt.roff[s]];
    } while (!(w & RES_ROOT));
    gid_l[pend_idx[t]] = s_groot[s] + (u32)w;
  }
}

// B, bulk round, owner side: the res[] word of every rank asked about, back to the asking rank block by block
__global__ void __launch_bounds__(256) k_chase_answer(const uint4 *__restrict__ queries, u32 n, const u64 *__restrict__ res, u32 lo,
                                                      ScatterTable back) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) scatter_store<unsigned long long>(back, j, (unsigned long long)res[queries[j].x - lo]);
}

// B, bulk round, asking side: a root ends the walk, anything else is the next rank to ask about
__global__ void __launch_bounds__(256) k_chase_apply(PeerTable pt, const u32 *__restrict__ nroots, u32 stride, const u32 *__restrict__ pend_idx,
                                                     const u32 *__restrict__ pend_key, const u32 *__restrict__ apos, const u64 *__restrict__ ans,
                                                     const u32 *__restrict__ n_pend, u32 *__restrict__ gid_l, u32 *__restrict__ next_idx,
                                                     u32 *__restrict__ next_key, u32 *__restrict__ n_next) {
  __shared__ u32 s_groot[DIST_MAX_RANKS];
  __shared__ PendStage sg;
  if (threadIdx.x == 0) sg.n = 0;
  load_groot(s_groot, nroots, stride, pt.nr);
  const u32 n = *n_pend;
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 t = base + threadIdx.x;
    bool again = false;
    u32 idx = 0, key = 0;
    if (t < n) {
      idx = pend_idx[t];
      const u32 p = pend_key[t];
      const u64 w = ans[apos[t]];
      if (w & RES_ROOT) {
        int s = pt.me;
        while (p < pt.roff[s]) --s;  // the rank that answered: the owner of p
        gid_l[idx] = s_groot[s] + (u32)w;
      } else {
        again = true;
        key = (u32)w;
      }
    }
    pend_push(sg, again, idx, key, next_idx, next_key, n_next);
  }
  pend_flush(sg, next_idx, next_key, n_next);
}

__global__ void __launch_bounds__(256) k_chase_map(const u64 *__restrict__ res, const u32 *__restrict__ lroot, const u32 *__restrict__ gid_l,
                                                   const u32 *__restrict__ nroots, u32 stride, int me, u32 m, u32 *__restrict__ gid_rank) {
  __shared__ u32 s_base;
  if (threadIdx.x == 0) {
    u32 run = 0;
    for (int r = 0; r < me; ++r) run += nroots[(u64)r * stride];
    s_base = run;
  }
  __syncthreads();
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const u64 w = res[i];
  gid_rank[i] = (w & RES_ROOT) ? s_base + (u32)w : gid_l[lroot[i]];
}

// ---- line records ----------------------------------------------------------------------------------------------------
// The rank that loaded a record answers every request for it with the line row, stored straight into the asking rank's
// rows[line] (requests arrive in blocks by source rank: the block gives the asking rank, the request its line).
// PACKED: the rank holds compact rows (pk) instead of 109-byte records (aos).
template <bool PACKED>
__global__ void __launch_bounds__(256) k_line_answer(const uint4 *__restrict__ requests, u32 n, const u8 *__restrict__ aos, u32 file_lo,
                                                     ScatterTable back, PackedRows pk) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint4 q = requests[t];
  int s = 0;
  for (int r = 1; r < back.nr; ++r) s = back.start[r] <= t ? r : s;
  const LineRow row = PACKED ? line_row_of_packed(pk.key, pk.rest, pk.strand, q.x - file_lo)
                             : line_row_of_record(aos + (u64)(q.x - file_lo) * FRAG_BYTES);
  uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<LineRow *>(back.out[s]) + q.y);
  const uint4 *src = reinterpret_cast<const uint4 *>(&row);
#pragma unroll
  for (int k = 0; k < 4; ++k) dst[k] = src[k];
}

// ---- small helpers ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_or_rows(const u32 *__restrict__ all, u64 row_stride, int nr, u64 words, u32 *__restrict__ out) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= words) return;
  u32 v = 0;
  for (int r = 0; r < nr; ++r) v |= all[(u64)r * row_stride + i];
  out[i] = v;
}

static inline unsigned blocks_for(u64 n, int per = 256) { return (unsigned)((n + per - 1) / per); }
static inline int sm_count() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

int dist_coarse_hist(const u32 *keys, u32 n, int shift, int pre_shift, u32 drop_key, u32 *hist, cudaStream_t st) {
  cudaMemsetAsync(hist, 0, DIST_BINS * sizeof(u32), st);
  if (n == 0) return 0;
  unsigned b = blocks_for(n, 256 * 8);
  const unsigned cap = (unsigned)sm_count() * 4;
  k_coarse_hist<<<b > cap ? cap : b, 256, 0, st>>>(keys, n, shift, pre_shift, drop_key, hist);
  return 1;
}
int dist_cuts_from_hist(const u32 *hist_all, u64 row_stride, int nr, int shift, u32 *cuts, cudaStream_t st, const u32 *gid_total,
                        u64 line_cap) {
  k_cuts_from_hist<<<1, 1024, sizeof(CutsSmem), st>>>(hist_all, row_stride, nr, shift, cuts, gid_total, gid_total ? line_cap : 0);
  return 1;
}
int dist_cuts_gid(const u32 *nroots, u32 stride, int nr, u32 *cuts, u32 *total, cudaStream_t st) {
  k_cuts_gid<<<1, 32, 0, st>>>(nroots, stride, nr, cuts, total);
  return 1;
}
int dist_cuts_x(const u32 *cuts0, int nr, Geometry g, const u32 *link_x, u32 *cuts_x, cudaStream_t st) {
  k_cuts_x<<<1, 64, 0, st>>>(cuts0, nr, g, link_x, cuts_x);
  return 1;
}
u64 dist_split_work_bytes(u64 n) { return ((n + SPLIT_TILE - 1) / SPLIT_TILE + 1) * NRP * 4; }

template <int MODE, class Pay>
static int split_pack(const RouteArgs &a, u32 *tile_cnt, u32 *counts, const Pay &pay, u32 *perm, cudaStream_t st) {
  cudaMemsetAsync(counts, 0, (a.nr + 1) * sizeof(u32), st);
  if (a.n == 0) return 0;
  const u32 tiles = (a.n + SPLIT_TILE - 1) / SPLIT_TILE;
  KScope ks(KID_DIST_ROWS, st, a.n);
  k_route_count<MODE><<<tiles, 256, 0, st>>>(a, tile_cnt, counts);
  k_tile_offsets<<<a.nr, 1024, 0, st>>>(tile_cnt, tiles, counts, nullptr, 0, 0);
  k_split_pack<MODE, Pay><<<tiles, 256, 0, st>>>(a, tile_cnt, pay, perm);
  return 3;
}

// The two big exchanges (records to the owner of their xStart/10 range; rows to the owner of their group-id range) in two
// halves: count (per tile and per destination) — the counts of all ranks are then all-gathered on the device — and push:
// every tile stores its rows straight into the destination ranks' receive buffers at the place the count matrix gives it.
int dist_count_plain(const u32 *keys, u32 n, const u32 *cuts, int nr, u32 drop_key, u32 *tile_cnt, u32 *counts, cudaStream_t st,
                     const u32 *n_ptr) {
  cudaMemsetAsync(counts, 0, (nr + 1) * sizeof(u32), st);
  if (n == 0) return 0;
  const u32 tiles = (n + SPLIT_TILE - 1) / SPLIT_TILE;
  KScope ks(KID_DIST_ROWS, st, n);
  k_route_count<0><<<tiles, 256, 0, st>>>(RouteArgs{keys, n, cuts, nr, 0, drop_key, 0, 0xFFFFFFFFu, n_ptr}, tile_cnt, counts);
  return 1;
}
template <class Pay>
static int push_rows(const RouteArgs &a, u32 *tile_cnt, const u32 *counts_all, u32 row_stride, int me, const Pay &pay, cudaStream_t st,
                     u32 *apos = nullptr) {
  if (a.n == 0) return 0;
  const u32 tiles = (a.n + SPLIT_TILE - 1) / SPLIT_TILE;
  KScope ks(KID_DIST_ROWS, st, a.n);
  k_tile_offsets<<<a.nr, 1024, 0, st>>>(tile_cnt, tiles, nullptr, counts_all, row_stride, me);
  k_push_rows<Pay><<<tiles, 256, sizeof(PushSmem<typename Pay::Word, Pay::WPR>), st>>>(a, tile_cnt, pay, apos, counts_all, row_stride);
  return 2;
}
cudaError_t dist_init_device() {  // dynamic shared memory opt-in of the push kernels (per device)
  cudaError_t e = cudaFuncSetAttribute(k_cuts_from_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CutsSmem));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_push_rows<PayRec24>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PushSmem<uint2, 3>));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_push_rows<PayQuery>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PushSmem<uint4, 1>));
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_push_rows<PayLineReq>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PushSmem<uint4, 1>));
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(k_push_rows<PayGidRow>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PushSmem<uint4, 1>));
}
template <class W>
static RowOutsT<W> row_outs(W *const *outs, int nr) {
  RowOutsT<W> o{};
  for (int d = 0; d < nr; ++d) o.p[d] = outs[d];
  return o;
}
int dist_push_records(const u32 *key0, u32 n, const u32 *cuts, int nr, u32 drop_key, const uint4 *rec, uint2 *const *outs, u32 out_cap,
                      u32 *tile_cnt, const u32 *counts_all, u32 row_stride, int me, cudaStream_t st) {
  return push_rows(RouteArgs{key0, n, cuts, nr, 0, drop_key, 0, out_cap, nullptr}, tile_cnt, counts_all, row_stride, me,
                   PayRec24{rec, row_outs<uint2>(outs, nr)}, st);
}
int dist_push_gid(const u32 *gid_rank, const uint4 *hfi_r, u32 n, const u32 *cuts, int nr, uint4 *const *outs, u32 out_cap, u32 *tile_cnt,
                  const u32 *counts_all, u32 row_stride, int me, cudaStream_t st) {
  return push_rows(RouteArgs{gid_rank, n, cuts, nr, 0, 0xFFFFFFFFu, 0, out_cap, nullptr}, tile_cnt, counts_all, row_stride, me,
                   PayGidRow{hfi_r, gid_rank, row_outs<uint4>(outs, nr)}, st);
}
// X halo: the fragments whose X super-bucket belongs to another rank; perm[t] = local rank of the t-th row sent
int dist_split_halo(const u32 *keys2, const uint2 *cl, u32 n, const u32 *cuts_x, int nr, u32 nbx, int me, u32 rank_off, uint4 *out,
                    u32 out_cap, u32 *perm, u32 *tile_cnt, u32 *counts, cudaStream_t st) {
  return split_pack<1>(RouteArgs{keys2, n, cuts_x, nr, me, 0xFFFFFFFFu, nbx, out_cap, nullptr}, tile_cnt, counts,
                       PayAxisRow{keys2, cl, rank_off, 0xFFFFFFFEu, out}, perm, st);
}
// Y pass: every fragment to the owner of its Y super-bucket range
int dist_split_axis(const u32 *keys, const uint2 *cl, u32 n, const u32 *cuts, int nr, u32 rank_off, uint4 *out, u32 *perm,
                    u32 *tile_cnt, u32 *counts, cudaStream_t st) {
  return split_pack<0>(RouteArgs{keys, n, cuts, nr, 0, 0xFFFFFFFFu, 0, 0xFFFFFFFFu, nullptr}, tile_cnt, counts,
                       PayAxisRow{keys, cl, rank_off, 0xFFFFFFFFu, out}, perm, st);
}
static unsigned hist_grid(u64 n) {  // few CTAs: few histogram flushes
  const unsigned b = blocks_for(n), cap = (unsigned)sm_count() * 8;
  return b > cap ? cap : b;
}
int dist_key0_of_rec(const uint2 *rec6, u32 n, u32 key_base, u32 *key0, HistOut ho, cudaStream_t st) {
  if (n == 0) return 0;
  k_key0_of_rec<<<hist_grid(n), 256, 0, st>>>(rec6, n, key_base, key0, ho);
  return 1;
}
int dist_unpack_axis_rows(const uint4 *rows, u32 n, u32 key_base, u32 *keys, uint2 *cl, u32 *grank, HistOut ho, cudaStream_t st) {
  if (n == 0) return 0;
  KScope ks(KID_DIST_ROWS, st, n);
  k_unpack_axis_rows<false><<<hist_grid(n), 256, 0, st>>>(rows, n, key_base, XRemap{}, keys, cl, grank, ho);
  return 1;
}
// the X side: the rank's own keys in place, the arrived halo rows while they are unpacked
static XRemap make_xremap(u32 nbx, const u32 *base, const u32 *range) {
  XRemap x{};
  x.nbx = nbx;
  x.base[0] = base[0], x.base[1] = base[1], x.range[0] = range[0], x.range[1] = range[1];
  x.R = range[0] > range[1] ? range[0] : range[1];
  return x;
}
int dist_x_local_keys(u32 *keys2, u32 n, u32 nbx, const u32 *base, const u32 *range, HistOut ho, cudaStream_t st) {
  if (n == 0) return 0;
  KScope ks(KID_DIST_ROWS, st, n);
  k_x_remap<<<hist_grid(n), 256, 0, st>>>(keys2, n, make_xremap(nbx, base, range), ho);
  return 1;
}
int dist_unpack_halo_rows(const uint4 *rows, u32 n, u32 nbx, const u32 *base, const u32 *range, u32 *keys, uint2 *cl, u32 *grank, HistOut ho,
                          cudaStream_t st) {
  if (n == 0) return 0;
  KScope ks(KID_DIST_ROWS, st, n);
  k_unpack_axis_rows<true><<<hist_grid(n), 256, 0, st>>>(rows, n, 0, make_xremap(nbx, base, range), keys, cl, grank, ho);
  return 1;
}
int dist_gid_keys(const uint4 *rows, u32 n, u32 gid_base, u32 *keys, HistOut ho, cudaStream_t st) {
  if (n == 0) return 0;
  k_gid_keys<<<hist_grid(n), 256, 0, st>>>(rows, n, gid_base, keys, ho);
  return 1;
}
int dist_x_owners(const u32 *parent_x, u32 m, u32 nh, u32 rank_off, const u32 *halo_grank, u32 *parent, const ScatterTable &home,
                  cudaStream_t st) {
  if (m + nh == 0) return 0;
  k_x_owners<<<blocks_for((u64)m + nh), 256, 0, st>>>(parent_x, m, nh, rank_off, halo_grank, parent, home);
  return 1;
}
int dist_apply_away(const u32 *away_res, const u32 *away_perm, u32 n, u32 *parent, cudaStream_t st) {
  if (n == 0) return 0;
  k_apply_away<<<blocks_for(n), 256, 0, st>>>(away_res, away_perm, n, parent);
  return 1;
}
int dist_pack_xm(const u32 *parent, const u32 *perm, u32 n, const ScatterTable &owners, cudaStream_t st) {
  if (n == 0) return 0;
  k_pack_xm<<<blocks_for(n), 256, 0, st>>>(parent, perm, n, owners);
  return 1;
}
int dist_y_owners(const u32 *parent_y, const u32 *grank, u32 n, const ScatterTable &home, cudaStream_t st) {
  if (n == 0) return 0;
  k_y_owners<<<blocks_for(n), 256, 0, st>>>(parent_y, grank, n, home);
  return 1;
}
int dist_merge_y(const u32 *yo_back, const u32 *perm, u32 n, u32 *parent, cudaStream_t st) {
  if (n == 0) return 0;
  k_merge_y<<<blocks_for(n), 256, 0, st>>>(yo_back, perm, n, parent);
  return 1;
}
u64 dist_scan_work_bytes(u32 m) { return scan_work_words(m ? m : 1) * 4 + 256; }
// gidscan[i] = roots among local ranks < i; *nroots = roots on this rank
int dist_root_scan(const u32 *parent, u32 m, u32 *gidscan, u32 *nroots, void *work, cudaStream_t st) {
  if (m == 0) {
    cudaMemsetAsync(nroots, 0, sizeof(u32), st);
    return 0;
  }
  u32 *bsum = (u32 *)work;
  const int l = exclusive_scan_u32(LoadIsRootD{parent}, gidscan, m, bsum, st);
  const u32 nb = (u32)(((u64)m + SCAN_CHUNK - 1) / SCAN_CHUNK);
  k_store_total<<<1, 32, 0, st>>>(bsum + nb, nroots);
  return l + 1;
}
int dist_chase_local(const u32 *parent, const u32 *gidscan, u32 m, u32 lo, u32 *lroot, u64 *res, u32 *pend_idx, u32 *pend_key, u32 *n_pend,
                     cudaStream_t st) {
  cudaMemsetAsync(n_pend, 0, sizeof(u32), st);
  if (m == 0) return 0;
  KScope ks(KID_CHASE, st, m);
  unsigned grid = blocks_for(m);
  const unsigned cap = (unsigned)sm_count() * 8;
  k_chase_local<<<grid > cap ? cap : grid, 256, 0, st>>>(parent, gidscan, m, lo, lroot, res, pend_idx, pend_key, n_pend);
  return 1;
}
// one bulk round, asking side, first half: the ranks asked about go to their owners (cuts = the ranks' first global ranks)
int dist_chase_ask_count(const u32 *pend_key, u32 bound, const u32 *n_pend, const u32 *roff_dev, int nr, u32 *tile_cnt, u32 *counts,
                         cudaStream_t st) {
  return dist_count_plain(pend_key, bound, roff_dev, nr, 0xFFFFFFFFu, tile_cnt, counts, st, n_pend);
}
int dist_chase_ask_push(const u32 *pend_key, u32 bound, const u32 *n_pend, const u32 *roff_dev, int nr, uint4 *const *outs, u32 out_cap,
                        u32 *apos, u32 *tile_cnt, const u32 *counts_all, u32 row_stride, int me, cudaStream_t st) {
  return push_rows(RouteArgs{pend_key, bound, roff_dev, nr, me, 0xFFFFFFFFu, 0, out_cap, n_pend}, tile_cnt, counts_all, row_stride, me,
                   PayQuery{pend_key, row_outs<uint4>(outs, nr)}, st, apos);
}
int dist_chase_answer(const uint4 *queries, u32 n, const u64 *res, u32 lo, const ScatterTable &back, cudaStream_t st) {
  if (n == 0) return 0;
  KScope ks(KID_CHASE_EXITS, st, n);
  k_chase_answer<<<blocks_for(n), 256, 0, st>>>(queries, n, res, lo, back);
  return 1;
}
int dist_chase_apply(const PeerTable &pt, const u32 *nroots, u32 stride, u32 bound, const u32 *pend_idx, const u32 *pend_key, const u32 *apos,
                     const u64 *ans, const u32 *n_pend, u32 *gid_l, u32 *next_idx, u32 *next_key, u32 *n_next, cudaStream_t st) {
  cudaMemsetAsync(n_next, 0, sizeof(u32), st);
  if (bound == 0) return 0;
  KScope ks(KID_CHASE_EXITS, st, bound);
  unsigned grid = blocks_for(bound);
  const unsigned cap = (unsigned)sm_count() * 8;
  k_chase_apply<<<grid > cap ? cap : grid, 256, 0, st>>>(pt, nroots, stride, pend_idx, pend_key, apos, ans, n_pend, gid_l, next_idx, next_key,
                                                         n_next);
  return 1;
}
// a short pending list walks through the peers' memory; then every fragment takes the id of its lroot
int dist_chase_finish(const PeerTable &pt, const u32 *nroots, u32 stride, u32 m, const u64 *res, const u32 *lroot, const u32 *pend_idx,
                      const u32 *pend_key, const u32 *n_pend, u32 *gid_l, u32 *gid_rank, cudaStream_t st) {
  if (m == 0) return 0;
  unsigned grid = blocks_for(m);
  const unsigned cap = (unsigned)sm_count() * 8;  // every walk of a typical pending list is in flight at once
  {
    KScope ks(KID_CHASE_EXITS, st, m);
    k_chase_walk<<<grid > cap ? cap : grid, 256, 0, st>>>(pt, nroots, stride, pend_idx, pend_key, n_pend, gid_l);
  }
  KScope ks(KID_CHASE, st, m);
  k_chase_map<<<blocks_for(m), 256, 0, st>>>(res, lroot, gid_l, nroots, stride, pt.me, m, gid_rank);
  return 2;
}
int dist_line_ask_push(const u32 *order, u32 n, const u32 *file_cuts, int nr, uint4 *const *outs, u32 out_cap, u32 *tile_cnt,
                       const u32 *counts_all, u32 row_stride, int me, cudaStream_t st) {
  return push_rows(RouteArgs{order, n, file_cuts, nr, me, 0xFFFFFFFFu, 0, out_cap, nullptr}, tile_cnt, counts_all, row_stride, me,
                   PayLineReq{order, row_outs<uint4>(outs, nr)}, st);
}
int dist_line_answer(const uint4 *requests, u32 n, const u8 *aos, const PackedRows &pk, u32 file_lo, const ScatterTable &back,
                     cudaStream_t st) {
  if (n == 0) return 0;
  KScope ks(KID_DIST_ROWS, st, n);
  if (aos) k_line_answer<false><<<blocks_for(n), 256, 0, st>>>(requests, n, aos, file_lo, back, pk);
  else k_line_answer<true><<<blocks_for(n), 256, 0, st>>>(requests, n, aos, file_lo, back, pk);
  return 1;
}
int dist_or_rows(const u32 *all, u64 row_stride, int nr, u64 words, u32 *out, cudaStream_t st) {
  if (words == 0) return 0;
  k_or_rows<<<blocks_for(words), 256, 0, st>>>(all, row_stride, nr, words, out);
  return 1;
}

}  // namespace rk
