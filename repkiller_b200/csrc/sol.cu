// The reference's SequenceOcupationList as a device-resident object behind the C ABI (rk_sol_*), and sort_groups as a
// pure function of (groups, diag_func) (rk_sort_members).
//
// Reference: /root/reference/src/SequenceOcupationList.h:13-33 and SequenceOcupationList.cpp:3-96 — per center/100 bucket
// a forward_list of {center, length, group*} with push_front (newest first); get_associated_group scans the buckets of
// center, center-1, center+1, center-2, center+2 (the +1/+2 probes under the reference's `center < max_index` /
// `center < max_index - 1` conditions, unsigned) and keeps the entry with the STRICTLY greatest deviation().
// Here: bucket heads + an entry pool in device memory (head[b] -> newest entry, next[] -> older), inserts are queued on
// the host and applied in order by one thread before the next query, a query is one kernel whose single warp leader walks
// the lists exactly like the reference loop.  This is the single-call interface for code that drives the lists itself
// (the reference's own generate_fragment_groups body compiles against it unchanged); whole databases go through rk_group,
// whose K3 kernels evaluate all queries of an axis in parallel.
#include <cstring>
#include <string>
#include <vector>

#include "rk_ctx.cuh"

using namespace rk;

namespace {

struct SolEntry {
  u64 center, length, tag;
  u32 next, pad;
};
struct SolInsert {
  u64 center, length, tag;
};

// deviation() of the reference (SequenceOcupationList.cpp:20-31) for 64-bit operands: binary64, no contraction
__device__ __forceinline__ double deviation64(u64 oc_center, u64 oc_length, u64 center, u64 length, double len_ratio, double pos_ratio) {
  const u64 dif_len = length > oc_length ? length - oc_length : oc_length - length;
  const double sim_len = __dadd_rn(-fabs(__ddiv_rn(__ull2double_rn(dif_len), __dmul_rn(__ull2double_rn(length), len_ratio))), 1.0);
  if (sim_len < 0) return 0.0;
  const u64 dif_cen = center > oc_center ? center - oc_center : oc_center - center;
  const double sim_pos = __dadd_rn(-fabs(__ddiv_rn(__ull2double_rn(dif_cen), __dmul_rn(__ull2double_rn(length), pos_ratio))), 1.0);
  if (sim_pos < 0) return 0.0;
  return __dadd_rn(__dmul_rn(sim_len, 0.4), __dmul_rn(sim_pos, 0.6));
}

// insert(): push_front into bucket center/100, in call order (SequenceOcupationList.cpp:93-96)
__global__ void k_sol_apply(const SolInsert *__restrict__ ins, u32 n, SolEntry *__restrict__ pool, u32 first, u32 *__restrict__ head) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  for (u32 i = 0; i < n; ++i) {
    const SolInsert v = ins[i];
    const u64 b = v.center / DIVISOR;
    SolEntry e;
    e.center = v.center, e.length = v.length, e.tag = v.tag, e.next = head[b], e.pad = 0;
    pool[first + i] = e;
    head[b] = first + i;
  }
}

// get_associated_group() (SequenceOcupationList.cpp:33-91); result[0] = tag of the winner (0: none)
__global__ void k_sol_query(const SolEntry *__restrict__ pool, const u32 *__restrict__ head, u64 center, u64 length, u64 max_index,
                            double len_ratio, double pos_ratio, u64 *__restrict__ result) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  double d = 0.0;
  u64 fg = 0;
  auto scan = [&](u64 p) {
    for (u32 e = head[p / DIVISOR]; e != RK_NONE32; e = pool[e].next) {
      const SolEntry oc = pool[e];
      const double cur = deviation64(oc.center, oc.length, center, length, len_ratio, pos_ratio);
      if (cur > d) {
        d = cur;
        fg = oc.tag;
      }
    }
  };
  scan(center);
  if (center > 0) scan(center - 1);
  if (center < max_index) scan(center + 1);
  if (center > 1) scan(center - 2);
  if (center < max_index - 1) scan(center + 2);  // unsigned: wraps when max_index == 0, like the reference
  *result = fg;
}

// h = |y - d| per member (commonFunctions.cpp:152-155); values that do not fit K5b's 32-bit keys raise the error word
__global__ void __launch_bounds__(256) k_member_keys(const u64 *__restrict__ y, const u64 *__restrict__ d, u32 m, u32 *__restrict__ h,
                                                     u32 *__restrict__ idx, float *__restrict__ zero, u32 *__restrict__ err) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const u64 a = y[i], b = d[i];
  const u64 hv = a > b ? a - b : b - a;
  if (hv >> 32) atomicOr(err, ERR_COORD);
  h[i] = (u32)hv;
  idx[i] = i;
  zero[i] = 0.f;
}

}  // namespace

namespace rk {
int launch_member_keys(const u64 *y, const u64 *d, u32 m, u32 *h, u32 *idx, float *zero, u32 *err, cudaStream_t st) {
  if (m == 0) return 0;
  k_member_keys<<<(m + 255) / 256, 256, 0, st>>>(y, d, m, h, idx, zero, err);
  return 1;
}
}  // namespace rk

struct rk_sol {
  int device = 0;
  double len_ratio = 0, pos_ratio = 0;
  u64 max_index = 0, n_buckets = 0;
  cudaStream_t stream = nullptr;
  u32 *head = nullptr;
  SolEntry *pool = nullptr;
  u64 pool_cap = 0, n_entries = 0;
  GrowBuffer d_ins, h_ins{cudaHostAllocDefault};  // staging of the queued inserts (device, pinned host)
  std::vector<SolInsert> pending;
  u64 *h_result = nullptr, *d_result = nullptr;
  std::string err;
};

namespace {

int sol_fail(rk_sol *s, int code, const std::string &msg) {
  s->err = msg;
  return code;
}
#define SK(call)                                                                                               \
  do {                                                                                                         \
    cudaError_t e_ = (call);                                                                                   \
    if (e_ != cudaSuccess) return sol_fail(s, RK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

int sol_flush(rk_sol *s) {
  const u64 n = s->pending.size();
  if (!n) return RK_OK;
  SK(cudaSetDevice(s->device));
  if (s->n_entries + n > s->pool_cap) {
    u64 cap = s->pool_cap ? s->pool_cap : 4096;
    while (cap < s->n_entries + n) cap *= 2;
    SolEntry *np = nullptr;
    SK(cudaMalloc((void **)&np, cap * sizeof(SolEntry)));
    if (s->n_entries) SK(cudaMemcpyAsync(np, s->pool, s->n_entries * sizeof(SolEntry), cudaMemcpyDeviceToDevice, s->stream));
    SK(cudaStreamSynchronize(s->stream));
    if (s->pool) cudaFree(s->pool);
    s->pool = np, s->pool_cap = cap;
  }
  u64 cap = s->h_ins.cap() ? s->h_ins.cap() / sizeof(SolInsert) : 256;
  while (cap < n) cap *= 2;
  int rc = s->d_ins.reserve(cap * sizeof(SolInsert), s->stream, s->err);
  if (!rc) rc = s->h_ins.reserve(cap * sizeof(SolInsert), s->stream, s->err);
  if (rc) return rc;
  SolInsert *d_ins = (SolInsert *)s->d_ins.ptr(), *h_ins = (SolInsert *)s->h_ins.ptr();
  memcpy(h_ins, s->pending.data(), n * sizeof(SolInsert));
  SK(cudaMemcpyAsync(d_ins, h_ins, n * sizeof(SolInsert), cudaMemcpyHostToDevice, s->stream));
  k_sol_apply<<<1, 32, 0, s->stream>>>(d_ins, (u32)n, s->pool, (u32)s->n_entries, s->head);
  SK(cudaStreamSynchronize(s->stream));  // the pinned staging buffer is reused by the next flush
  s->n_entries += n;
  s->pending.clear();
  return RK_OK;
}

}  // namespace

extern "C" {

rk_sol *rk_sol_create(int device, double len_ratio, double pos_ratio, uint64_t seq_size) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
    cudaGetLastError();
    return nullptr;
  }
  rk_sol *s = new rk_sol;
  s->device = device, s->len_ratio = len_ratio, s->pos_ratio = pos_ratio;
  s->max_index = seq_size / DIVISOR;     // SequenceOcupationList.cpp:4
  s->n_buckets = s->max_index + 1;       // :5 — the reference allocates max_index + 1 lists
  bool ok = cudaSetDevice(device) == cudaSuccess && cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaMalloc((void **)&s->head, (s->n_buckets + 4) * sizeof(u32)) == cudaSuccess &&
            cudaMemsetAsync(s->head, 0xFF, (s->n_buckets + 4) * sizeof(u32), s->stream) == cudaSuccess &&
            cudaMalloc((void **)&s->d_result, 8) == cudaSuccess &&
            cudaHostAlloc((void **)&s->h_result, 8, cudaHostAllocDefault) == cudaSuccess;
  if (!ok) {
    cudaGetLastError();
    rk_sol_destroy(s);
    return nullptr;
  }
  return s;
}

void rk_sol_destroy(rk_sol *s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  if (s->head) cudaFree(s->head);
  if (s->pool) cudaFree(s->pool);
  if (s->d_result) cudaFree(s->d_result);
  if (s->h_result) cudaFreeHost(s->h_result);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;  // frees the insert staging: the device is current and the stream drained
}

const char *rk_sol_last_error(const rk_sol *s) { return s ? s->err.c_str() : "null rk_sol"; }

int rk_sol_insert(rk_sol *s, uint64_t center, uint64_t length, uint64_t tag) {
  if (!s) return RK_ERR_ARG;
  // the reference indexes ocupations[center / 100] without a bound check (undefined behaviour beyond max_index)
  if (center / DIVISOR >= s->n_buckets) return sol_fail(s, RK_ERR_RANGE, "center lies beyond the occupation list (the reference writes out of bounds here)");
  if (tag == 0) return sol_fail(s, RK_ERR_ARG, "tag 0 means `no group`");
  s->pending.push_back(SolInsert{center, length, tag});
  if (s->pending.size() >= (1u << 16)) return sol_flush(s);
  return RK_OK;
}

int rk_sol_get_associated(rk_sol *s, uint64_t center, uint64_t length, uint64_t *tag) {
  if (!s || !tag) return RK_ERR_ARG;
  // every bucket a probe can touch must exist: center/100, and (center+2)/100 when the +1/+2 probes fire
  const bool probes_up = center < s->max_index || center < s->max_index - 1;  // second term: unsigned wrap at max_index == 0
  if (center / DIVISOR >= s->n_buckets || (probes_up && (center + 2) / DIVISOR >= s->n_buckets + 4))
    return sol_fail(s, RK_ERR_RANGE, "center lies beyond the occupation list (the reference reads out of bounds here)");
  const int rc = sol_flush(s);
  if (rc != RK_OK) return rc;
  SK(cudaSetDevice(s->device));
  k_sol_query<<<1, 32, 0, s->stream>>>(s->pool, s->head, center, length, s->max_index, s->len_ratio, s->pos_ratio, s->d_result);
  SK(cudaMemcpyAsync(s->h_result, s->d_result, 8, cudaMemcpyDeviceToHost, s->stream));
  SK(cudaStreamSynchronize(s->stream));
  SK(cudaGetLastError());
  *tag = *s->h_result;
  return RK_OK;
}

}  // extern "C"
