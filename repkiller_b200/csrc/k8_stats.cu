// K8 — per-group statistics over the output of sort_groups (BASELINE north_star kernel 5; SURVEY.md §8 row a10:
// "optional extra per-group stats (span, count, multiplicity, mean identity) — not in the reference output").
//
// The groups they reduce over are the reference's: the FragsGroups of generate_fragment_groups in creation order
// (/root/reference/src/commonFunctions.cpp:56-76), written group by group by save_frag_pair (:117-129), so in the
// output arrays of rk_group every group is one contiguous run of lines with the same gid.  Per group:
//   count                              members (save_frags_from_group's fg.size(), :106)
//   x_lo, x_hi, y_lo, y_hi             min xStart / max (xStart + length) and the same on Y: the span the group covers
//   first_line                         index of its first output line
//   mean_identity                      mean of the per-fragment identity column, (float)ident*100/(float)length (:103)
//   multiplicity                       sum of the lengths / (x_hi - x_lo): how many times the X span is covered (repeat copies)
// One thread per output line; a warp reduces its runs of equal gid with shuffles (segmented), the last lane of every run
// adds the run's partial to the group's accumulators — integer atomics, and double atomics on integer-valued sums of
// lengths (exact in any order) and on the identity sum (double accumulation of floats: ~1e-16 relative per add).
#include "rk_common.cuh"

namespace rk {

__global__ void __launch_bounds__(256) k_stats_init(rk_group_stats_dev *__restrict__ st, u32 n_groups) {
  const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  rk_group_stats_dev s;
  s.count = 0, s.x_lo = 0xFFFFFFFFu, s.x_hi = 0, s.y_lo = 0xFFFFFFFFu, s.y_hi = 0, s.first_line = 0xFFFFFFFFu;
  s.mean_identity = 0.0, s.multiplicity = 0.0;
  st[g] = s;
}

__global__ void __launch_bounds__(256) k_group_stats(const u32 *__restrict__ out_order, const u32 *__restrict__ out_gid,
                                                     const float *__restrict__ out_identity, const uint4 *__restrict__ rec4,
                                                     const LineRow *__restrict__ rows, u32 m, u32 gid_base, u32 line_off,
                                                     rk_group_stats_dev *__restrict__ st) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 lane = threadIdx.x & 31;
  const bool valid = j < m;
  u32 gid = 0xFFFFFFFFu, cnt = 0, xlo = 0xFFFFFFFFu, xhi = 0, ylo = 0xFFFFFFFFu, yhi = 0, first = 0xFFFFFFFFu;
  double slen = 0.0, sid = 0.0;
  if (valid) {
    gid = out_gid[j];
    u32 xs, ys, len;
    if (rows) {
      xs = (u32)rows[j].xs, ys = (u32)rows[j].ys, len = (u32)rows[j].len;  // K1 refused anything wider
    } else {
      const uint4 r = rec4[2 * (u64)out_order[j]];  // {xStart, yStart, length, flags}
      xs = r.x, ys = r.y, len = r.z;
    }
    cnt = 1, xlo = xs, xhi = xs + len, ylo = ys, yhi = ys + len, first = line_off + j;
    slen = (double)len;
    sid = (double)out_identity[j];
  }
  // segmented inclusive scan inside the warp: lane l accumulates the lanes of its run at or before it
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const u32 g2 = __shfl_up_sync(0xFFFFFFFFu, gid, d);
    const u32 c2 = __shfl_up_sync(0xFFFFFFFFu, cnt, d);
    const u32 a2 = __shfl_up_sync(0xFFFFFFFFu, xlo, d), b2 = __shfl_up_sync(0xFFFFFFFFu, xhi, d);
    const u32 e2 = __shfl_up_sync(0xFFFFFFFFu, ylo, d), f2 = __shfl_up_sync(0xFFFFFFFFu, yhi, d);
    const u32 h2 = __shfl_up_sync(0xFFFFFFFFu, first, d);
    const double l2 = __shfl_up_sync(0xFFFFFFFFu, slen, d), i2 = __shfl_up_sync(0xFFFFFFFFu, sid, d);
    // gids are sorted: if the lane d below has my gid, every lane between has it too
    if ((int)lane >= d && g2 == gid) {
      cnt += c2;
      xlo = min(xlo, a2), xhi = max(xhi, b2), ylo = min(ylo, e2), yhi = max(yhi, f2), first = min(first, h2);
      slen += l2, sid += i2;
    }
  }
  const u32 gnext = __shfl_down_sync(0xFFFFFFFFu, gid, 1);
  const bool run_end = valid && (lane == 31 || gnext != gid);
  if (run_end) {
    rk_group_stats_dev *s = st + (gid - gid_base);
    atomicAdd(&s->count, cnt);
    atomicMin(&s->x_lo, xlo);
    atomicMax(&s->x_hi, xhi);
    atomicMin(&s->y_lo, ylo);
    atomicMax(&s->y_hi, yhi);
    atomicMin(&s->first_line, first);
    atomicAdd(&s->multiplicity, slen);    // integer-valued partial sums < 2^53: exact in any order
    atomicAdd(&s->mean_identity, sid);
  }
}

__global__ void __launch_bounds__(256) k_stats_final(rk_group_stats_dev *__restrict__ st, u32 n_groups) {
  const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  rk_group_stats_dev s = st[g];
  const u32 span = s.x_hi - s.x_lo;
  s.mean_identity = s.count ? s.mean_identity / (double)s.count : 0.0;
  s.multiplicity = span ? s.multiplicity / (double)span : 0.0;  // length-0 groups cover nothing
  st[g] = s;
}

int launch_group_stats(const u32 *out_order, const u32 *out_gid, const float *out_identity, const uint4 *rec4, const LineRow *rows,
                       u32 m, u32 n_groups, u32 gid_base, u32 line_off, rk_group_stats_dev *st, cudaStream_t stream) {
  if (n_groups == 0) return 0;
  KScope ks(KID_STATS, stream, m);
  k_stats_init<<<(n_groups + 255) / 256, 256, 0, stream>>>(st, n_groups);
  k_group_stats<<<(m + 255) / 256, 256, 0, stream>>>(out_order, out_gid, out_identity, rec4, rows, m, gid_base, line_off, st);
  k_stats_final<<<(n_groups + 255) / 256, 256, 0, stream>>>(st, n_groups);
  return 3;
}

}  // namespace rk
