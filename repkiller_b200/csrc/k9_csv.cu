// K9 — GECKO CSV rows parsed on the device (rk_load_csv): FragmentsDatabase's row loop (/root/reference/src/
// FragmentsDatabase.cpp:91-100) with readFragment's rules (:17-50) applied to every row at once.
//
//   count   '\n' per 4 KB tile of the text (runs per uploaded chunk, beside the upload of the next one)
//   scan    tile counts -> the index of every tile's first row (rk_scan.cuh)
//   starts  the 64-bit start offset of every row, plus a sentinel: row k spans [start[k], start[k+1] - 1)
//   rows    per 16 KB tile staged in shared memory (with a 1 KB halo), the rows that START in the tile are parsed
//           by one thread each; a row that runs past the halo is read from global memory.  Classify mode writes a
//           status byte per row (reject / accept / host, plus a wide bit) and appends host rows to a list; emit mode
//           parses the accepted rows again and writes them at their file-order slot (the scan of the accept flags)
//   put     the host-decided records (readFragment's result) at their slots
//
// A row is decided here only when each of its tokens is in the grammar the host parser's fast path accepts
// (rk_csv_row.cuh: the same plain_u64 / plain_float code); every other row goes to readFragment on the host.  Empty
// tokens and a first token other than "Frag" reject a row whatever else it holds, on both sides.
//
// HBM-bound: the text is read three times (count, classify, emit) and every accepted row writes 33 B (key4, strand,
// rest4) or a 109-byte record; per row also 8 B of start offset (written once, read by both row passes), one status
// byte and one slot word.
#include "rk_csv_row.cuh"
#include "rk_common.cuh"
#include "rk_scan.cuh"

namespace rk {

constexpr u32 CSV_ROW_TILE = 16384;  // bytes of text per CTA of the row passes
constexpr u32 CSV_HALO = 1024;       // staged past the tile: rows that start near its end usually end inside
constexpr int CSV_ROW_THREADS = 256;
static_assert(CSV_ROW_TILE % CSV_COUNT_TILE == 0, "a row tile is a whole number of count tiles");

struct CsvRow {
  u64 xs, ys, xe, ye, len, score, ident;
  long long blk;
  float sim;
  u8 strand;
};

// readFragment's token walk over one row (row[0 .. n), no '\n' inside): 14 tokens split on ',', the last one
// repeated once the row is exhausted; values through the fast-path helpers.  Returns CSV_REJECT, CSV_ACCEPT or CSV_HOST.
__device__ __forceinline__ u8 csv_parse_row(const char *row, u64 n, CsvRow &r) {
  u64 pos = 0, cur = 0, curlen = 0;
  bool exhausted = false, host = false;
  r.sim = 0.f;
  r.xs = r.ys = r.xe = r.ye = r.len = r.score = 0;
  r.blk = 0;
  r.strand = 0;
  for (int i = 0; i < 14; ++i) {
    if (!exhausted) {
      const u64 s = pos;
      while (pos < n && row[pos] != ',') ++pos;
      cur = s;
      curlen = pos - s;
      if (pos < n) ++pos;
      else exhausted = true;
    }
    if (curlen == 0) return CSV_REJECT;
    const char *t = row + cur;
    if (i == 0) {
      if (!(curlen == 4 && t[0] == 'F' && t[1] == 'r' && t[2] == 'a' && t[3] == 'g')) return CSV_REJECT;
    } else if (i == 5) {
      r.strand = (u8)t[0];
    } else if (i == 10) {
      host |= !rk_csv::plain_float(t, curlen, r.sim);
    } else if (i <= 8) {
      u64 v = 0;
      host |= !rk_csv::plain_u64(t, curlen, v);
      if (i == 1) r.xs = v;
      else if (i == 2) r.ys = v;
      else if (i == 3) r.xe = v;
      else if (i == 4) r.ye = v;
      else if (i == 6) r.blk = (long long)v;
      else if (i == 7) r.len = v;
      else r.score = v;
    }
  }
  if (host) return CSV_HOST;
  r.ident = (u64)r.sim;
  return CSV_ACCEPT;
}

__device__ __forceinline__ bool csv_wide(const CsvRow &r) {  // the host route's test for the 109-byte load
  return ((r.xs | r.ys | r.len | r.ident | r.xe | r.ye | r.score) >> 32) != 0;
}

__device__ __forceinline__ void st_u64_bytes(u8 *p, u64 v) {
#pragma unroll
  for (int i = 0; i < 8; ++i) p[i] = (u8)(v >> (8 * i));
}

// one record as readFragment writes it (struct FragFile, 109 bytes, little endian)
__device__ void csv_write_record(u8 *rec, const CsvRow &r) {
  st_u64_bytes(rec + 0, (u64)((long long)r.xs - (long long)r.ys));
  st_u64_bytes(rec + OFF_XSTART, r.xs);
  st_u64_bytes(rec + OFF_YSTART, r.ys);
  st_u64_bytes(rec + OFF_XEND, r.xe);
  st_u64_bytes(rec + OFF_YEND, r.ye);
  st_u64_bytes(rec + OFF_LENGTH, r.len);
  st_u64_bytes(rec + OFF_IDENT, r.ident);
  st_u64_bytes(rec + OFF_SCORE, r.score);
  const u32 sb = __float_as_uint(r.sim);
#pragma unroll
  for (int i = 0; i < 4; ++i) rec[OFF_SIMILARITY + i] = (u8)(sb >> (8 * i));
  st_u64_bytes(rec + 68, 0);  // seqX
  st_u64_bytes(rec + 76, 1);  // seqY
  st_u64_bytes(rec + 84, (u64)r.blk);
  rec[OFF_STRAND] = r.strand;
#pragma unroll
  for (int i = 0; i < 16; ++i) rec[93 + i] = 0;  // evalue
}

__device__ __forceinline__ void csv_write_compact(const CsvOut &o, u32 slot, const CsvRow &r) {
  o.key4[slot] = make_uint4((u32)r.xs, (u32)r.ys, (u32)r.len, (u32)r.ident);
  o.rest4[slot] = make_uint4((u32)r.xe, (u32)r.ye, (u32)r.score, __float_as_uint(r.sim));
  o.strand[slot] = r.strand;
}

// newlines of 16 bytes at text[p, p+16) (fewer at the end of the text)
__device__ __forceinline__ u32 csv_newlines16(const u8 *text, u64 bytes, u64 p, u32 &mask) {
  mask = 0;
  if (p + 16 <= bytes) {
    const uint4 v = *reinterpret_cast<const uint4 *>(text + p);
    const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const u32 eq = __vcmpeq4(w[j], 0x0A0A0A0Au);  // 0xFF per matching byte
#pragma unroll
      for (int b = 0; b < 4; ++b)
        if ((eq >> (8 * b)) & 1) mask |= 1u << (4 * j + b);
    }
  } else {
    for (u64 i = p; i < bytes; ++i)
      if (text[i] == '\n') mask |= 1u << (u32)(i - p);
  }
  return __popc(mask);
}

__global__ void __launch_bounds__(256) k_csv_count(const u8 *__restrict__ text, u64 bytes, u64 tile0, u32 *__restrict__ tile_cnt) {
  const u64 tile = tile0 + blockIdx.x;
  u32 mask;
  const u32 c = csv_newlines16(text, bytes, tile * CSV_COUNT_TILE + threadIdx.x * 16, mask);
  u32 total;
  block_excl_scan<256>(c, &total);
  if (threadIdx.x == 0) tile_cnt[tile] = total;
}

// start[0] = 0, start[k + 1] = (position of the k-th '\n') + 1, start[n_rows] = bytes + 1
__global__ void __launch_bounds__(256) k_csv_starts(const u8 *__restrict__ text, u64 bytes, const u32 *__restrict__ tile_base,
                                                    u64 *__restrict__ start, u64 n_rows) {
  const u64 tile = blockIdx.x;
  const u64 p = tile * CSV_COUNT_TILE + threadIdx.x * 16;
  u32 mask;
  const u32 c = csv_newlines16(text, bytes, p, mask);
  u64 k = (u64)tile_base[tile] + block_excl_scan<256>(c, nullptr);
  while (mask) {
    const u32 b = __ffs(mask) - 1;
    mask &= mask - 1;
    start[++k] = p + b + 1;
  }
  if (tile == 0 && threadIdx.x == 0) start[0] = 0, start[n_rows] = bytes + 1;
}

// Classify (EMIT = false) or emit (EMIT = true) the rows that start in this CTA's tile.
template <bool EMIT>
__global__ void __launch_bounds__(CSV_ROW_THREADS) k_csv_rows(const u8 *__restrict__ text, u64 bytes, const u64 *__restrict__ start, u64 n_rows,
                                                              u8 *__restrict__ status, u32 *__restrict__ host_list, CsvCounters *cnt,
                                                              const u32 *__restrict__ slot, CsvOut o) {
  __shared__ __align__(16) u8 win[CSV_ROW_TILE + CSV_HALO];
  __shared__ u64 s_rows[2];
  const u64 w0 = (u64)blockIdx.x * CSV_ROW_TILE;
  const u64 w1 = min(bytes, w0 + CSV_ROW_TILE + CSV_HALO);
  if (threadIdx.x < 2) {  // rows [r0, r1) start in [w0, w0 + CSV_ROW_TILE): lower bounds in the sorted start array
    const u64 key = w0 + threadIdx.x * CSV_ROW_TILE;
    u64 lo = 0, hi = n_rows;
    while (lo < hi) {
      const u64 mid = (lo + hi) / 2;
      if (start[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    s_rows[threadIdx.x] = lo;
  }
  for (u64 p = w0 + threadIdx.x * 16; p < w1; p += CSV_ROW_THREADS * 16) {
    if (p + 16 <= w1) *reinterpret_cast<uint4 *>(win + (p - w0)) = *reinterpret_cast<const uint4 *>(text + p);
    else
      for (u64 i = p; i < w1; ++i) win[i - w0] = text[i];
  }
  __syncthreads();
  const u64 r0 = s_rows[0], r1 = s_rows[1];
  u32 wide = 0, accepted = 0;
  for (u64 k = r0 + threadIdx.x; k < r1; k += CSV_ROW_THREADS) {
    if (EMIT && (status[k] & 3) != CSV_ACCEPT) continue;
    const u64 s = start[k], e = start[k + 1] - 1;
    const char *row = (const char *)(e <= w1 ? win + (s - w0) : text + s);
    CsvRow r;
    const u8 st = csv_parse_row(row, e - s, r);
    if (EMIT) {
      if (o.aos) csv_write_record(o.aos + (u64)slot[k] * FRAG_BYTES, r);
      else csv_write_compact(o, slot[k], r);
    } else {
      const bool w = st == CSV_ACCEPT && csv_wide(r);
      status[k] = st | (w ? CSV_WIDE : 0);
      wide |= w;
      accepted += st == CSV_ACCEPT;
      if (st == CSV_HOST) host_list[atomicAdd(&cnt->n_host, 1u)] = (u32)k;
    }
  }
  if (!EMIT) {
    u32 total;
    block_excl_scan<CSV_ROW_THREADS>(accepted, &total);
    if (__syncthreads_or(wide) && threadIdx.x == 0) atomicOr(&cnt->wide, 1u);
    if (threadIdx.x == 0 && total) atomicAdd(&cnt->n_accepted, total);
  }
}

// host-decided rows: the accepted ones get their slot in the accept scan
__global__ void k_csv_mark(const u32 *__restrict__ rows, u32 n, u8 *__restrict__ status) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) status[rows[i]] = CSV_HOST_ACCEPT;
}

// spans {start, end} of the listed rows
__global__ void k_csv_spans(const u32 *__restrict__ rows, u32 n, const u64 *__restrict__ start, ulonglong2 *__restrict__ spans) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) spans[i] = make_ulonglong2(start[rows[i]], start[rows[i] + 1] - 1);
}

// bytes of the listed spans, back to back from dst + off[i] (one warp per row)
__global__ void k_csv_gather(const u8 *__restrict__ text, const ulonglong2 *__restrict__ spans, const u64 *__restrict__ off, u32 n,
                             u8 *__restrict__ dst) {
  const u32 i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  const ulonglong2 sp = spans[i];
  for (u64 j = sp.x + lane_id(); j < sp.y; j += 32) dst[off[i] + (j - sp.x)] = text[j];
}

// the host parser's records (109 bytes each) at the slots of their rows
__global__ void k_csv_put(const u8 *__restrict__ recs, const u32 *__restrict__ rows, u32 n, const u32 *__restrict__ slot, CsvOut o) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u8 *f = recs + (u64)i * FRAG_BYTES;
  const u32 s = slot[rows[i]];
  if (o.aos) {
    for (int b = 0; b < FRAG_BYTES; ++b) o.aos[(u64)s * FRAG_BYTES + b] = f[b];
    return;
  }
  const LineRow r = line_row_of_record(f);
  o.key4[s] = make_uint4((u32)r.xs, (u32)r.ys, (u32)r.len, (u32)r.ident);
  o.rest4[s] = make_uint4((u32)r.xe, (u32)r.ye, (u32)r.score, r.sim_bits);
  o.strand[s] = (u8)r.strand;
}

struct CsvAccepted {  // scan input: 1 for a row that loads
  const u8 *status;
  __device__ __forceinline__ u32 operator()(u64 i) const {
    const u8 s = status[i] & 3;
    return s == CSV_ACCEPT || s == CSV_HOST_ACCEPT;
  }
};

static unsigned blocks_of(u64 n, u32 per) { return (unsigned)((n + per - 1) / per); }

u64 csv_scan_words(u64 n) { return scan_work_words(n); }

int launch_csv_count(const u8 *text, u64 bytes, u64 tile0, u64 n_tiles, u32 *tile_cnt, cudaStream_t st) {
  if (!n_tiles) return 0;
  KScope ks(KID_CSV_LINES, st, n_tiles * CSV_COUNT_TILE);
  k_csv_count<<<(unsigned)n_tiles, 256, 0, st>>>(text, bytes, tile0, tile_cnt);
  return 1;
}

int launch_csv_tile_scan(u32 *tile_cnt, u64 n_tiles, u32 *bsum, CsvCounters *cnt, cudaStream_t st) {
  if (!n_tiles) return 0;
  const int launches = exclusive_scan_u32(LoadU32{tile_cnt}, tile_cnt, n_tiles, bsum, st);
  cudaMemcpyAsync(&cnt->n_lines, bsum + (n_tiles + SCAN_CHUNK - 1) / SCAN_CHUNK, sizeof(u32), cudaMemcpyDeviceToDevice, st);
  return launches;
}

int launch_csv_starts(const u8 *text, u64 bytes, const u32 *tile_base, u64 *start, u64 n_rows, cudaStream_t st) {
  const u64 n_tiles = csv_count_tiles(bytes);
  KScope ks(KID_CSV_LINES, st, bytes);
  // (an empty text still has its one row: one CTA writes start[0] and the sentinel; tile_base[0] is 0 then)
  k_csv_starts<<<(unsigned)(n_tiles ? n_tiles : 1), 256, 0, st>>>(text, bytes, tile_base, start, n_rows);
  return 1;
}

int launch_csv_classify(const u8 *text, u64 bytes, const u64 *start, u64 n_rows, u8 *status, u32 *host_list, CsvCounters *cnt,
                        cudaStream_t st) {
  KScope ks(KID_CSV_ROWS, st, n_rows);
  k_csv_rows<false><<<blocks_of(bytes + 1, CSV_ROW_TILE), CSV_ROW_THREADS, 0, st>>>(text, bytes, start, n_rows, status, host_list, cnt,
                                                                                   nullptr, CsvOut{});
  return 1;
}

int launch_csv_host_spans(const u32 *rows, u32 n, const u64 *start, ulonglong2 *spans, cudaStream_t st) {
  if (!n) return 0;
  k_csv_spans<<<blocks_of(n, 256), 256, 0, st>>>(rows, n, start, spans);
  return 1;
}

int launch_csv_gather(const u8 *text, const ulonglong2 *spans, const u64 *off, u32 n, u8 *dst, cudaStream_t st) {
  if (!n) return 0;
  k_csv_gather<<<blocks_of((u64)n * 32, 256), 256, 0, st>>>(text, spans, off, n, dst);
  return 1;
}

int launch_csv_emit(const u8 *text, u64 bytes, const u64 *start, u64 n_rows, u8 *status, const u32 *host_rows, u32 n_host_acc,
                    const u8 *host_recs, u32 *slot, u32 *bsum, CsvOut o, cudaStream_t st) {
  int launches = 0;
  if (n_host_acc) {
    k_csv_mark<<<blocks_of(n_host_acc, 256), 256, 0, st>>>(host_rows, n_host_acc, status);
    ++launches;
  }
  launches += exclusive_scan_u32(CsvAccepted{status}, slot, n_rows, bsum, st);
  {
    KScope ks(KID_CSV_ROWS, st, n_rows);
    k_csv_rows<true><<<blocks_of(bytes + 1, CSV_ROW_TILE), CSV_ROW_THREADS, 0, st>>>(text, bytes, start, n_rows, status, nullptr, nullptr,
                                                                                    slot, o);
    ++launches;
  }
  if (n_host_acc) {
    k_csv_put<<<blocks_of(n_host_acc, 256), 256, 0, st>>>(host_recs, host_rows, n_host_acc, slot, o);
    ++launches;
  }
  return launches;
}

#if !defined(__CUDA_ARCH__)  // readFragment is host code
bool csv_read_row_host(const char *line, u64 len, void *record) {
  FragFile f;
  memset(&f, 0, sizeof f);
  if (!readFragment(&f, line, (size_t)len)) return false;
  memcpy(record, &f, sizeof f);
  return true;
}
#endif

}  // namespace rk
