// K8 — per-group statistics over the output of sort_groups (BASELINE north_star kernel 5; SURVEY.md §8 row a10:
// "optional extra per-group stats (span, count, multiplicity, mean identity) — not in the reference output").
//
// The groups they reduce over are the reference's: the FragsGroups of generate_fragment_groups in creation order
// (/root/reference/src/commonFunctions.cpp:56-76), written group by group by save_frag_pair (:117-129), so in the
// output arrays of rk_group every group is one contiguous run of lines with the same gid.  Per group:
//   count                              members (save_frags_from_group's fg.size(), :106)
//   x_lo, x_hi, y_lo, y_hi             min xStart / max (xStart + length) and the same on Y: the span the group covers
//                                      (the ends as uint64: xStart and length are each below 2^32, their sum is not)
//   first_line                         index of its first output line
//   mean_identity                      RN(S) / count, S the exact sum of the per-fragment identity column
//                                      (float)ident*100/(float)length (:103); NaN if a member is NaN, else +inf if one is
//   multiplicity                       (double)(exact uint64 sum of the lengths) / (x_hi - x_lo), 0 for an empty span
// Every result is a function of the group's members alone: the same bits in any launch order, on any number of ranks.
//
// The identity sum is exact because K1 bounds the column: a finite identity is 0 or lies in [100/2^32, 100*2^64], and a
// float32 there is a multiple of 2^-49 (its ulp at >= 2^-26) below 2^71.  So identity * 2^49 is an integer below 2^120,
// kept as four 32-bit digits; every digit column sums in uint64 without overflow for fewer than 2^32 members.  A value
// outside the bound (negative, subnormal, too small or too large) sets the error word: RK_ERR_INTERNAL, never a wrong sum.
//
// One thread per output line; a warp reduces its runs of equal gid with shuffles (segmented), the last lane of every run
// adds the run's partial to the group's accumulators with integer atomics (StatsAcc); k_stats_final carries the digits,
// rounds once to binary64 and writes the public rk_group_stats.
#include "rk_common.cuh"

namespace rk {

__global__ void __launch_bounds__(256) k_stats_init(StatsAcc *__restrict__ acc, u32 n_groups, u32 *__restrict__ err) {
  const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0) *err = 0;
  if (g >= n_groups) return;
  StatsAcc a;
  a.count = 0, a.x_lo = 0xFFFFFFFFu, a.y_lo = 0xFFFFFFFFu, a.first_line = 0xFFFFFFFFu;
  a.x_hi = 0, a.y_hi = 0, a.len_sum = 0;
  a.digit[0] = a.digit[1] = a.digit[2] = a.digit[3] = 0;
  a.n_nan_inf = 0;
  acc[g] = a;
}

// identity * 2^49 as an integer {lo, hi} (< 2^120); false when the value lies outside K1's bound
__device__ __forceinline__ bool identity_fixed(u32 b, u64 &lo, u64 &hi) {
  lo = hi = 0;
  if (b == 0) return true;
  const u32 e = b >> 23;  // sign bit included: any negative value is out of bound
  if (e == 0 || e >= 0xFF) return false;
  u64 mant = (b & 0x7FFFFFu) | 0x800000u;
  const int s = (int)e - 101;  // value = mant * 2^(e-150), times 2^49
  if (s < 0) {
    if (s < -23 || (mant & ((1ull << -s) - 1))) return false;
    lo = mant >> -s;
  } else if (s > 96) {
    return false;
  } else if (s < 64) {
    lo = mant << s;
    hi = s ? mant >> (64 - s) : 0;
  } else {
    hi = mant << (s - 64);
  }
  return true;
}

__global__ void __launch_bounds__(256) k_group_stats(const u32 *__restrict__ out_order, const u32 *__restrict__ out_gid,
                                                     const float *__restrict__ out_identity, const uint4 *__restrict__ rec4,
                                                     const LineRow *__restrict__ rows, u32 m, u32 gid_base, u32 line_off,
                                                     StatsAcc *__restrict__ acc, u32 *__restrict__ err) {
  const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
  const u32 lane = threadIdx.x & 31;
  const bool valid = j < m;
  u32 gid = 0xFFFFFFFFu, cnt = 0, xlo = 0xFFFFFFFFu, ylo = 0xFFFFFFFFu, first = 0xFFFFFFFFu;
  u32 nan_inf = 0;  // NaN members in the low half, +inf members in the high half (a warp run has at most 32)
  u64 xhi = 0, yhi = 0, slen = 0, d[4] = {0, 0, 0, 0};
  if (valid) {
    gid = out_gid[j];
    u32 xs, ys, len;
    if (rows) {
      xs = (u32)rows[j].xs, ys = (u32)rows[j].ys, len = (u32)rows[j].len;  // K1 refused anything wider
    } else {
      const uint4 r = rec4[2 * (u64)out_order[j]];  // {xStart, yStart, length, flags}
      xs = r.x, ys = r.y, len = r.z;
    }
    cnt = 1, xlo = xs, xhi = (u64)xs + len, ylo = ys, yhi = (u64)ys + len, first = line_off + j;
    slen = len;
    const float f = out_identity[j];
    const u32 b = __float_as_uint(f);
    if (f != f) {
      nan_inf = 1;
    } else if (b == 0x7F800000u) {
      nan_inf = 1u << 16;
    } else {
      u64 lo, hi;
      if (!identity_fixed(b, lo, hi)) atomicOr(err, 1u);
      d[0] = (u32)lo, d[1] = lo >> 32, d[2] = (u32)hi, d[3] = hi >> 32;
    }
  }
  // segmented inclusive scan inside the warp: lane l accumulates the lanes of its run at or before it
#pragma unroll
  for (int k = 1; k < 32; k <<= 1) {
    const u32 g2 = __shfl_up_sync(0xFFFFFFFFu, gid, k);
    const u32 c2 = __shfl_up_sync(0xFFFFFFFFu, cnt, k), n2 = __shfl_up_sync(0xFFFFFFFFu, nan_inf, k);
    const u32 a2 = __shfl_up_sync(0xFFFFFFFFu, xlo, k), e2 = __shfl_up_sync(0xFFFFFFFFu, ylo, k);
    const u32 h2 = __shfl_up_sync(0xFFFFFFFFu, first, k);
    const u64 b2 = __shfl_up_sync(0xFFFFFFFFu, xhi, k), f2 = __shfl_up_sync(0xFFFFFFFFu, yhi, k);
    const u64 l2 = __shfl_up_sync(0xFFFFFFFFu, slen, k);
    u64 dd[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) dd[q] = __shfl_up_sync(0xFFFFFFFFu, d[q], k);
    // gids are sorted: if the lane k below has my gid, every lane between has it too
    if ((int)lane >= k && g2 == gid) {
      cnt += c2, nan_inf += n2;
      xlo = min(xlo, a2), xhi = max(xhi, b2), ylo = min(ylo, e2), yhi = max(yhi, f2), first = min(first, h2);
      slen += l2;
#pragma unroll
      for (int q = 0; q < 4; ++q) d[q] += dd[q];
    }
  }
  const u32 gnext = __shfl_down_sync(0xFFFFFFFFu, gid, 1);
  const bool run_end = valid && (lane == 31 || gnext != gid);
  if (run_end) {
    StatsAcc *a = acc + (gid - gid_base);
    atomicAdd(&a->count, cnt);
    atomicMin(&a->x_lo, xlo);
    atomicMax((unsigned long long *)&a->x_hi, (unsigned long long)xhi);
    atomicMin(&a->y_lo, ylo);
    atomicMax((unsigned long long *)&a->y_hi, (unsigned long long)yhi);
    atomicMin(&a->first_line, first);
    atomicAdd((unsigned long long *)&a->len_sum, (unsigned long long)slen);  // < 2^32 lengths of < 2^32: below 2^64
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (d[q]) atomicAdd((unsigned long long *)&a->digit[q], (unsigned long long)d[q]);
    if (nan_inf) atomicAdd((unsigned long long *)&a->n_nan_inf, (unsigned long long)(nan_inf & 0xFFFFu) | ((u64)(nan_inf >> 16) << 32));
  }
}

// sum_q digit[q] * 2^(32q - 49), rounded to nearest even once
__device__ __forceinline__ double fixed_to_double(const u64 *digit) {
  // carry the digit columns into a 192-bit integer v[0..2] (digit[q] < 2^64, so every partial stays below 2^64)
  u64 w[5];
  u64 carry = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const u64 t = (digit[q] & 0xFFFFFFFFull) + carry;
    w[q] = t & 0xFFFFFFFFull;
    carry = (digit[q] >> 32) + (t >> 32);
  }
  w[4] = carry;  // < 2^33
  const u64 v0 = w[0] | (w[1] << 32), v1 = w[2] | (w[3] << 32), v2 = w[4];
  // the top 64 bits from the highest set bit down, with every bit below them folded into bit 0 (sticky): bit 0 lies
  // below the rounding bit of a 53-bit mantissa, so __ull2double_rn rounds the folded word as it rounds the whole value
  int shift;
  u64 top, below;
  if (v2) {
    const int p = 128 + 63 - __clzll((long long)v2);
    shift = p - 63;                                        // 65 .. 96
    const int r = shift - 64;                              // bits of v1 below the window
    top = (v2 << (64 - r)) | (v1 >> r);
    below = (v1 << (64 - r)) | v0;
  } else if (v1) {
    const int p = 64 + 63 - __clzll((long long)v1);
    shift = p - 63;                                        // 1 .. 64
    top = shift == 64 ? v1 : (v1 << (64 - shift)) | (v0 >> shift);
    below = shift == 64 ? v0 : v0 << (64 - shift);
  } else {
    shift = 0, top = v0, below = 0;
  }
  return ldexp(__ull2double_rn(top | (below != 0)), shift - 49);
}

__global__ void __launch_bounds__(256) k_stats_final(const StatsAcc *__restrict__ acc, rk_group_stats_dev *__restrict__ st,
                                                     u32 n_groups) {
  const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_groups) return;
  const StatsAcc a = acc[g];
  rk_group_stats_dev s;
  s.count = a.count, s.x_lo = a.x_lo, s.y_lo = a.y_lo, s.first_line = a.first_line;
  s.x_hi = a.x_hi, s.y_hi = a.y_hi;
  const u64 span = a.x_hi - a.x_lo;
  s.multiplicity = span ? __ull2double_rn(a.len_sum) / __ull2double_rn(span) : 0.0;  // length-0 groups cover nothing
  if (a.n_nan_inf & 0xFFFFFFFFull)
    s.mean_identity = __longlong_as_double((long long)0xFFF8000000000000ull);  // the column's 0xFFC00000, widened
  else if (a.n_nan_inf)
    s.mean_identity = __longlong_as_double(0x7FF0000000000000ll);
  else
    s.mean_identity = a.count ? fixed_to_double(a.digit) / (double)a.count : 0.0;
  st[g] = s;
}

int launch_group_stats(const u32 *out_order, const u32 *out_gid, const float *out_identity, const uint4 *rec4, const LineRow *rows,
                       u32 m, u32 n_groups, u32 gid_base, u32 line_off, rk_group_stats_dev *st, StatsAcc *acc, u32 *err,
                       cudaStream_t stream) {
  if (n_groups == 0) return 0;
  KScope ks(KID_STATS, stream, m);
  k_stats_init<<<(n_groups + 255) / 256, 256, 0, stream>>>(acc, n_groups, err);
  k_group_stats<<<(m + 255) / 256, 256, 0, stream>>>(out_order, out_gid, out_identity, rec4, rows, m, gid_base, line_off, acc, err);
  k_stats_final<<<(n_groups + 255) / 256, 256, 0, stream>>>(acc, st, n_groups);
  return 3;
}

}  // namespace rk
