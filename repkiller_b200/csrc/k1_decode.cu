// K1 — AoS -> SoA decode of the packed 109-byte fragment records, validity mask and link bits.
//
// Replaces the record hand-off of FragmentsDatabase's loading loop (/root/reference/src/FragmentsDatabase.cpp:
// 91-100: bucket index xStart/10, :96) and precomputes what generate_fragment_groups derives per fragment
// (/root/reference/src/commonFunctions.cpp:52-55: strand class, centers xStart+length/2, yStart+length/2).
//
// Data movement: records are 109 bytes with no alignment, so a tile of 256 records (27,904 B, a multiple of
// 16) is staged into shared memory with one cp.async.bulk (TMA 1-D bulk copy, SASS UBLKCP) per tile, three
// tiles in flight per CTA behind mbarriers; each thread then pulls its record's fields out of shared memory
// with aligned 32-bit reads + funnel shifts (record stride 27.25 words: near conflict-free) and the SoA is
// written fully coalesced.  HBM-bound: 109 B read + 36 B written per fragment (a 32-byte record + the sort key); the
// digit counts of the key are gathered on the way for the rank sort (HistOut).
#include "rk_common.cuh"

namespace rk {

constexpr int DEC_TILE = 256;
constexpr int DEC_THREADS = 256;
constexpr int DEC_TILE_BYTES = DEC_TILE * FRAG_BYTES;  // 27904
constexpr int DEC_STAGES = 3;
static_assert(DEC_TILE_BYTES % 16 == 0, "bulk copies move multiples of 16 bytes");

__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(u64 *bar, u32 phase) {
  u32 ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(phase)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, u32 bytes, u64 *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// unaligned little-endian 64-bit read from shared memory through aligned words
__device__ __forceinline__ u64 lds_u64_unaligned(const u8 *base, u32 byte_off) {
  const u32 *w = reinterpret_cast<const u32 *>(base) + (byte_off >> 2);
  const u32 sh = (byte_off & 3) * 8;
  const u32 w0 = w[0], w1 = w[1], w2 = w[2];
  const u32 lo = __funnelshift_r(w0, w1, sh);
  const u32 hi = __funnelshift_r(w1, w2, sh);
  return ((u64)hi << 32) | lo;
}

__device__ __forceinline__ u64 ldg_u64_bytes(const u8 *p) {
  u64 v = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) v |= (u64)p[i] << (8 * i);
  return v;
}

struct DecodeOut {
  u32 *xs, *ys, *len;
  uint4 *rec4;  // when set: two 16-byte words per record {xStart, yStart, length, flags} {identity bits, file index, 0, 0}
                // instead of the five arrays (one 32-byte sector per gather in k_keys)
  u8 *flags;
  float *identity;
  u32 *key0;
  u32 *link_x, *link_y;
  u32 *n_dropped;
  u32 *err;
  HistOut hist;  // digit counts of key0 for the rank sort (ghist == nullptr: off)
  u32 fidx_base; // file index of record 0 of this slice (multi-GPU: a rank decodes a slice of the file)
};

__device__ __forceinline__ u32 emit_fragment(u64 idx, u64 xs, u64 ys, u64 len, u64 ident, u8 strand, const Geometry &g,
                                             const DecodeOut &o, u32 &dropped, u32 &err) {
  u8 fl = (strand != 'f') ? FL_REVERSE : 0;
  const u64 cx = xs + len / 2, cy = ys + len / 2;
  if ((xs | ys | len | cx | cy) >> 32) {
    err |= ERR_COORD;
    xs &= 0xFFFFFFFFu, ys &= 0xFFFFFFFFu, len &= 0xFFFFFFFFu;
  }
  const u64 b0 = xs / XBUCKET;
  u32 key0;
  if (b0 >= g.vsize) {
    err |= ERR_XBUCKET;
    key0 = g.vsize - 1;
    fl |= FL_DROPPED;
  } else {
    key0 = (u32)b0;
    if (key0 == g.vsize - 1) fl |= FL_DROPPED;
  }
  if (fl & FL_DROPPED) {
    ++dropped;
  } else if (!(err & ERR_COORD)) {
    const u32 c32x = (u32)cx, c32y = (u32)cy;
    const u32 bx = c32x / DIVISOR, by = c32y / DIVISOR;
    if (bx > g.mx || by > g.my) {
      err |= ERR_CENTER;
    } else {
      const u32 sc = fl & FL_REVERSE;
      // bit k of the link map: bucket k is processed together with bucket k-1
      const u32 kx = sc * g.nbx + bx, ky = sc * g.nby + by;
      if (probes_prev(c32x)) atomicOr(&o.link_x[kx >> 5], 1u << (kx & 31));
      if (probes_next(c32x, g.mx)) atomicOr(&o.link_x[(kx + 1) >> 5], 1u << ((kx + 1) & 31));
      if (probes_prev(c32y)) atomicOr(&o.link_y[ky >> 5], 1u << (ky & 31));
      if (probes_next(c32y, g.my)) atomicOr(&o.link_y[(ky + 1) >> 5], 1u << ((ky + 1) & 31));
    }
  }
  // (float)ident * 100 / (float)length — commonFunctions.cpp:103, float32 arithmetic without contraction
  // 0/0 (ident == 0, length == 0) is the only NaN this can produce; x86 SSE returns the default NaN with the
  // sign bit set (0xFFC00000, printed "-nan" by the reference's writer), so mirror that bit pattern.
  float idv = __fdiv_rn(__fmul_rn(__ull2float_rn(ident), 100.0f), __ull2float_rn(len));
  if (idv != idv) idv = __int_as_float(0xFFC00000);
  o.key0[idx] = key0;
  if (o.rec4) {
    o.rec4[2 * idx] = make_uint4((u32)xs, (u32)ys, (u32)len, fl);
    o.rec4[2 * idx + 1] = make_uint4(__float_as_uint(idv), o.fidx_base + (u32)idx, 0u, 0u);
  } else {
    o.xs[idx] = (u32)xs;
    o.ys[idx] = (u32)ys;
    o.len[idx] = (u32)len;
    o.flags[idx] = fl;
    o.identity[idx] = idv;
  }
  return key0;
}

__global__ void __launch_bounds__(DEC_THREADS) k_decode(const u8 *__restrict__ aos, u64 n, Geometry g, DecodeOut o) {
  extern __shared__ __align__(128) u8 stage_mem[];
  __shared__ __align__(8) u64 full_bar[DEC_STAGES];
  __shared__ u32 s_dropped, s_err;
  __shared__ u32 s_hist[HIST_PASSES][HIST_RADIX];

  const u32 tid = threadIdx.x;
  const u64 full_tiles = n / DEC_TILE;
  if (o.hist.ghist) hist_zero(s_hist);
  if (tid == 0) {
    for (int s = 0; s < DEC_STAGES; ++s) mbar_init(&full_bar[s], 1);
    s_dropped = 0;
    s_err = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (tid == 0) {
    for (int s = 0; s < DEC_STAGES; ++s) {
      const u64 t = blockIdx.x + (u64)s * gridDim.x;
      if (t < full_tiles) {
        mbar_expect_tx(&full_bar[s], DEC_TILE_BYTES);
        bulk_g2s(stage_mem + s * DEC_TILE_BYTES, aos + t * DEC_TILE_BYTES, DEC_TILE_BYTES, &full_bar[s]);
      }
    }
  }

  u32 dropped = 0, err = 0;
  for (u64 k = 0;; ++k) {
    const u64 tile = blockIdx.x + k * gridDim.x;
    if (tile >= full_tiles) break;
    const int s = (int)(k % DEC_STAGES);
    const u32 phase = (u32)(k / DEC_STAGES) & 1;
    u32 spins = 0;
    while (!mbar_try_wait(&full_bar[s], phase)) {
      if (++spins > (1u << 24)) {  // a bulk copy never takes this long; fail loudly instead of hanging
        err |= ERR_SPIN;
        break;
      }
    }
    const u8 *rec_base = stage_mem + s * DEC_TILE_BYTES;
    const u32 off = tid * FRAG_BYTES;
    const u64 xs = lds_u64_unaligned(rec_base, off + OFF_XSTART);
    const u64 ys = lds_u64_unaligned(rec_base, off + OFF_YSTART);
    const u64 len = lds_u64_unaligned(rec_base, off + OFF_LENGTH);
    const u64 ident = lds_u64_unaligned(rec_base, off + OFF_IDENT);
    const u8 strand = rec_base[off + OFF_STRAND];
    const u32 k0 = emit_fragment(tile * DEC_TILE + tid, xs, ys, len, ident, strand, g, o, dropped, err);
    if (o.hist.ghist) hist_add(s_hist, k0, true, o.hist);
    __syncthreads();  // every thread is done reading stage s
    if (tid == 0) {
      const u64 nt = tile + (u64)DEC_STAGES * gridDim.x;
      if (nt < full_tiles) {
        mbar_expect_tx(&full_bar[s], DEC_TILE_BYTES);
        bulk_g2s(stage_mem + s * DEC_TILE_BYTES, aos + nt * DEC_TILE_BYTES, DEC_TILE_BYTES, &full_bar[s]);
      }
    }
  }

  // ragged tail (n % 256 records): plain byte loads, one CTA
  if (blockIdx.x == 0) {
    const u64 idx = full_tiles * DEC_TILE + tid;
    u32 k0 = 0;
    if (idx < n) {
      const u8 *p = aos + idx * FRAG_BYTES;
      k0 = emit_fragment(idx, ldg_u64_bytes(p + OFF_XSTART), ldg_u64_bytes(p + OFF_YSTART), ldg_u64_bytes(p + OFF_LENGTH),
                         ldg_u64_bytes(p + OFF_IDENT), p[OFF_STRAND], g, o, dropped, err);
    }
    if (o.hist.ghist) hist_add(s_hist, k0, idx < n, o.hist);
  }

  // one atomic per CTA for the dropped count and the error word
  for (int d = 16; d > 0; d >>= 1) {
    dropped += __shfl_xor_sync(0xFFFFFFFFu, dropped, d);
    err |= __shfl_xor_sync(0xFFFFFFFFu, err, d);
  }
  if ((tid & 31) == 0) {
    if (dropped) atomicAdd(&s_dropped, dropped);
    if (err) atomicOr(&s_err, err);
  }
  __syncthreads();
  if (o.hist.ghist) hist_flush(s_hist, o.hist);
  if (tid == 0) {
    if (s_dropped) atomicAdd(o.n_dropped, s_dropped);
    if (s_err) atomicOr(o.err, s_err);
  }
}

// Compact ingest (rk_load_packed): the host parser hands over {xStart, yStart, length, ident} as four 32-bit words per
// fragment plus one strand byte, 17 B instead of the 109-byte record (the 16 B of xEnd/yEnd/score/similarity that only
// the output lines need travel beside them and are not touched here).  Same outputs as k_decode.
__global__ void __launch_bounds__(256) k_decode_packed(const uint4 *__restrict__ key4, const u8 *__restrict__ strand, u64 n, Geometry g,
                                                       DecodeOut o) {
  __shared__ u32 s_dropped, s_err;
  __shared__ u32 s_hist[HIST_PASSES][HIST_RADIX];
  if (o.hist.ghist) hist_zero(s_hist);
  if (threadIdx.x == 0) s_dropped = 0, s_err = 0;
  __syncthreads();
  u32 dropped = 0, err = 0;
  for (u64 base = (u64)blockIdx.x * blockDim.x; base < n; base += (u64)gridDim.x * blockDim.x) {
    const u64 i = base + threadIdx.x;
    u32 k0 = 0;
    if (i < n) {
      const uint4 k = key4[i];
      k0 = emit_fragment(i, k.x, k.y, k.z, k.w, strand[i], g, o, dropped, err);
    }
    if (o.hist.ghist) hist_add(s_hist, k0, i < n, o.hist);
  }
  for (int d = 16; d > 0; d >>= 1) {
    dropped += __shfl_xor_sync(0xFFFFFFFFu, dropped, d);
    err |= __shfl_xor_sync(0xFFFFFFFFu, err, d);
  }
  if ((threadIdx.x & 31) == 0) {
    if (dropped) atomicAdd(&s_dropped, dropped);
    if (err) atomicOr(&s_err, err);
  }
  __syncthreads();
  if (o.hist.ghist) hist_flush(s_hist, o.hist);
  if (threadIdx.x == 0) {
    if (s_dropped) atomicAdd(o.n_dropped, s_dropped);
    if (s_err) atomicOr(o.err, s_err);
  }
}

int launch_decode_packed(const uint4 *key4, const u8 *strand, u64 n, Geometry g, u32 *key0, u32 *link_x, u32 *link_y, u32 *n_dropped,
                         u32 *err, cudaStream_t st, uint4 *rec4, HistOut hist, u32 fidx_base) {
  if (n == 0) return 0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  u64 grid = (n + 255) / 256;
  if (grid > (u64)sms * 8) grid = (u64)sms * 8;
  DecodeOut o{nullptr, nullptr, nullptr, rec4, nullptr, nullptr, key0, link_x, link_y, n_dropped, err, hist, fidx_base};
  KScope ks(KID_DECODE, st, n);
  k_decode_packed<<<(unsigned)grid, 256, 0, st>>>(key4, strand, n, g, o);
  return 1;
}

// per-device opt-in to the 84 KB of dynamic shared memory (called by rk_create for the context's device)
cudaError_t decode_init_device() {
  return cudaFuncSetAttribute(k_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, DEC_STAGES * DEC_TILE_BYTES);
}

int launch_decode(const u8 *aos, u64 n, Geometry g, u32 *xs, u32 *ys, u32 *len, u8 *flags, float *identity, u32 *key0,
                  u32 *link_x, u32 *link_y, u32 *n_dropped, u32 *err, cudaStream_t st, uint4 *rec4, HistOut hist, u32 fidx_base) {
  if (n == 0) return 0;
  const int smem = DEC_STAGES * DEC_TILE_BYTES;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const u64 full_tiles = n / DEC_TILE;
  u64 grid = (u64)sms * 2;  // two CTAs (2 x 84 KB of staging) per SM, persistent over the tiles
  if (grid > full_tiles) grid = full_tiles ? full_tiles : 1;
  DecodeOut o{xs, ys, len, rec4, flags, identity, key0, link_x, link_y, n_dropped, err, hist, fidx_base};
  KScope ks(KID_DECODE, st, n);
  k_decode<<<(unsigned)grid, DEC_THREADS, smem, st>>>(aos, n, g, o);
  return 1;
}

}  // namespace rk
