// K6 — the output lines of save_frags_from_group / store_frag as text, on the device.
//
// Reference: /root/reference/src/commonFunctions.cpp:101-104 (store_frag: one line per fragment,
//   Frag,xStart,yStart,xEnd,yEnd,strand,gid,length,score,ident,similarity,identity,0,repval\n
// integers through ostream << uint64_t, the two floats through ostream << float == printf("%g")), :106-115 (repval),
// :117-129 (groups in creation order).  In the reference this formatting is 28 s of the 88 s of a 10M-fragment run.
//
// Two passes over a range of output lines: (1) the length of every line (the same formatter with a counting sink),
// an exclusive scan gives the byte offset of every line; (2) a CTA formats its 128 lines into shared memory and copies
// the block out with coalesced stores.  The "%g" digits are exact (rk_fmt.cuh: integer arithmetic on the binary value).
// A line's fields come from its record (order[j] into the loaded records) or, on a rank of a partitioned comparison, from
// the line row that rk_dist_group brought to the rank (RK_F_LINE_RECORDS): the same fields, so the same bytes.
#include "rk_common.cuh"
#include "rk_fmt.cuh"
#include "rk_scan.cuh"

namespace rk {

constexpr int FMT_THREADS = 128;
constexpr int FMT_MAX_LINE = RK_FORMAT_MAX_LINE;  // 5 + 8 x 20 digits + 10 (gid) + 1 + 2 x 13 ("%g") + 2 + 13 commas + newline, rounded up

// what output line j prints of its record: its line row, or the record order[j] (109-byte records or the compact arrays)
__device__ __forceinline__ LineRow load_fields(const FormatArgs &a, u32 j) {
  if (a.rows) return a.rows[j];
  const u32 fidx = a.order[j];
  if (a.aos) return line_row_of_record(a.aos + (u64)fidx * FRAG_BYTES);
  return line_row_of_packed(a.pk_key, a.pk_rest, a.pk_strand, fidx);  // compact ingest
}

template <class Sink>
__device__ __forceinline__ void format_line(Sink &s, const LineRow &f, u32 gid, u32 identity_bits, u32 repval) {
  s.put('F'), s.put('r'), s.put('a'), s.put('g'), s.put(',');
  rkfmt::put_u64(s, f.xs), s.put(',');
  rkfmt::put_u64(s, f.ys), s.put(',');
  rkfmt::put_u64(s, f.xe), s.put(',');
  rkfmt::put_u64(s, f.ye), s.put(',');
  s.put((char)f.strand), s.put(',');
  rkfmt::put_u64(s, gid), s.put(',');
  rkfmt::put_u64(s, f.len), s.put(',');
  rkfmt::put_u64(s, f.score), s.put(',');
  rkfmt::put_u64(s, f.ident), s.put(',');
  rkfmt::put_g6(s, f.sim_bits), s.put(',');
  rkfmt::put_g6(s, identity_bits);
  s.put(','), s.put('0'), s.put(',');
  s.put((char)('0' + repval)), s.put('\n');
}

__global__ void __launch_bounds__(FMT_THREADS) k_format_len(FormatArgs a) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n_lines) return;
  const u32 j = a.first_line + i;
  rkfmt::CountSink s;
  format_line(s, load_fields(a, j), a.gid[j], __float_as_uint(a.identity[j]), a.repval[j]);
  a.line_len[i] = s.n;
}

__global__ void __launch_bounds__(FMT_THREADS) k_format_write(FormatArgs a) {
  __shared__ char s_text[FMT_THREADS * FMT_MAX_LINE];
  const u32 i0 = blockIdx.x * FMT_THREADS, i = i0 + threadIdx.x;
  const u32 last = min(i0 + (u32)FMT_THREADS, a.n_lines);  // one past the CTA's last line
  const u32 base = a.line_off[i0];
  const u32 end = last < a.n_lines ? a.line_off[last] : *a.total_bytes;
  if (i < a.n_lines) {
    const u32 j = a.first_line + i;
    rkfmt::BufSink s(s_text + (a.line_off[i] - base));
    format_line(s, load_fields(a, j), a.gid[j], __float_as_uint(a.identity[j]), a.repval[j]);
  }
  __syncthreads();
  char *out = a.text + base;
  for (u32 k = threadIdx.x; k < end - base; k += FMT_THREADS) out[k] = s_text[k];
}

struct LoadLen {
  const u32 *len;
  __device__ __forceinline__ u32 operator()(u64 i) const { return len[i]; }
};

u64 format_work_bytes(u32 n_lines) { return ((u64)2 * n_lines + scan_work_words(n_lines) + 16) * 4 + 256; }

// line_len / line_off / scan scratch are carved from `work`; text must hold n_lines * FMT_MAX_LINE bytes at most (the
// caller sizes it from an upper bound); *total_bytes (device) receives the number of bytes written.
int launch_format(FormatArgs a, void *work, cudaStream_t st) {
  if (a.n_lines == 0) {
    cudaMemsetAsync(a.total_bytes, 0, sizeof(u32), st);
    return 0;
  }
  u32 *w = reinterpret_cast<u32 *>(work);
  a.line_len = w;
  a.line_off = w + a.n_lines;
  u32 *bsum = a.line_off + a.n_lines;
  const u32 blocks = (a.n_lines + FMT_THREADS - 1) / FMT_THREADS;
  {
    KScope ks(KID_FORMAT, st, a.n_lines);
    k_format_len<<<blocks, FMT_THREADS, 0, st>>>(a);
  }
  const int launches = 2 + exclusive_scan_u32(LoadLen{a.line_len}, a.line_off, a.n_lines, bsum, st);
  const u32 nb = (u32)(((u64)a.n_lines + SCAN_CHUNK - 1) / SCAN_CHUNK);
  cudaMemcpyAsync(a.total_bytes, bsum + nb, sizeof(u32), cudaMemcpyDeviceToDevice, st);
  KScope ks(KID_FORMAT, st, a.n_lines);
  k_format_write<<<blocks, FMT_THREADS, 0, st>>>(a);
  return launches;
}

}  // namespace rk
