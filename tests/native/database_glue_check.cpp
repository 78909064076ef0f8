// The FragmentsDatabase constructors against a RECORDING stand-in for librk_b200 (test only: nothing is computed; the
// stand-in notes what the constructor hands to the library).  Checks the host glue without a GPU: the arguments of the load
// call (count, sequence lengths, the compact arrays or records, the CSV body) and what the database then answers.  The CSV
// loads accept the rows readFragment accepts, so that n_loaded and the over-count refusal are the library's.
// Build: g++ this file + host/FragmentsDatabase.cpp + host/GeckoFrags.cpp (no librk_b200).
//   database_glue_check <input> [ranks] [host|device]     builds one database, prints one line per fact
//   host (default): the host parser (detect_frags_input); device: the CSV rows parsed by the device (CsvOnDevice)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <string>
#include <vector>

#include "../../repkiller_b200/csrc/host/FragmentsDatabase.h"

namespace {
uint64_t fnv(const void *p, size_t n, uint64_t h = 1469598103934665603ull) {
  const unsigned char *b = (const unsigned char *)p;
  for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}
int g_live_ctx = 0, g_live_multi = 0, g_live_host = 0;
std::string g_error;
uint64_t g_loaded = 0;
void fill(rk_load_stats *st, uint64_t n) {
  memset(st, 0, sizeof *st);
  st->n_loaded = n, st->n_kept = n;
  g_loaded = n;
}
// rk_load_csv's row rules: rows split on '\n' (the segment after the last one is a row too), accepted by readFragment
int load_csv(const char *body, uint64_t bytes, uint64_t total, const char *refusal, rk_load_stats *st, rk_csv_stats *csv) {
  uint64_t rows = 0, acc = 0;
  for (uint64_t pos = 0;; ++rows) {
    const uint64_t s = pos;
    while (pos < bytes && body[pos] != '\n') ++pos;
    FragFile f;
    acc += readFragment(&f, body + s, pos - s);
    if (pos++ >= bytes) break;
  }
  if (acc > total) {
    g_error = refusal;
    return RK_ERR_RANGE;
  }
  fill(st, acc);
  memset(csv, 0, sizeof *csv);
  csv->n_rows = rows + 1, csv->n_accepted = acc;
  return 0;
}
}  // namespace

struct rk_ctx { int device; };
struct rk_multi { int n; };

extern "C" {
rk_ctx *rk_create(int device) { ++g_live_ctx; return new rk_ctx{device}; }
void rk_destroy(rk_ctx *c) { --g_live_ctx; delete c; }
rk_multi *rk_create_multi(const int *, int n) { ++g_live_multi; return new rk_multi{n}; }
void rk_destroy_multi(rk_multi *m) { --g_live_multi; delete m; }
const char *rk_create_error(void) { return ""; }
const char *rk_last_error(const rk_ctx *) { return g_error.c_str(); }
const char *rk_multi_last_error(const rk_multi *) { return g_error.c_str(); }
void *rk_host_alloc(size_t bytes) { ++g_live_host; return malloc(bytes); }
void rk_host_free(void *p) { --g_live_host; free(p); }
int64_t rk_debug_fetch(rk_ctx *, const char *name, void *host, uint64_t bytes) {  // rank_fidx: every record kept, file order
  if (strcmp(name, "rank_fidx") != 0) return -1;
  for (uint64_t i = 0; host && i < g_loaded && (i + 1) * 4 <= bytes; ++i) ((uint32_t *)host)[i] = (uint32_t)i;
  return (int64_t)(g_loaded * 4);
}
int rk_load_packed(rk_ctx *, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n, uint64_t lx, uint64_t ly,
                   unsigned, rk_load_stats *st) {
  printf("call rk_load_packed n=%llu seqx_len=%llu seqy_len=%llu key4=%016llx strand=%016llx rest4=%016llx\n", (unsigned long long)n,
         (unsigned long long)lx, (unsigned long long)ly, (unsigned long long)fnv(key4, n * 16), (unsigned long long)fnv(strand, n),
         (unsigned long long)fnv(rest4, n * 16));
  fill(st, n);
  return 0;
}
int rk_load_aos(rk_ctx *, const void *frags, uint64_t n, uint64_t lx, uint64_t ly, unsigned, rk_load_stats *st) {
  printf("call rk_load_aos n=%llu seqx_len=%llu seqy_len=%llu records=%016llx\n", (unsigned long long)n, (unsigned long long)lx,
         (unsigned long long)ly, (unsigned long long)fnv(frags, n * 109));
  fill(st, n);
  return 0;
}
int rk_multi_load_aos(rk_multi *m, const void *frags, uint64_t n, uint64_t lx, uint64_t ly, unsigned, rk_load_stats *st) {
  printf("call rk_multi_load_aos ranks=%d n=%llu seqx_len=%llu seqy_len=%llu records=%016llx\n", m->n, (unsigned long long)n,
         (unsigned long long)lx, (unsigned long long)ly, (unsigned long long)fnv(frags, n * 109));
  fill(st, n);
  return 0;
}
int rk_load_csv(rk_ctx *, const char *body, uint64_t bytes, uint64_t lx, uint64_t ly, uint64_t total, unsigned, rk_load_stats *st,
                rk_csv_stats *csv) {
  printf("call rk_load_csv bytes=%llu body=%016llx seqx_len=%llu seqy_len=%llu total_frags=%llu\n", (unsigned long long)bytes,
         (unsigned long long)fnv(body, bytes), (unsigned long long)lx, (unsigned long long)ly, (unsigned long long)total);
  return load_csv(body, bytes, total, "Unexpected number of fragments", st, csv);
}
int rk_multi_load_csv(rk_multi *m, const char *body, uint64_t bytes, uint64_t lx, uint64_t ly, uint64_t total, unsigned,
                      rk_load_stats *st, rk_csv_stats *csv) {
  printf("call rk_multi_load_csv ranks=%d bytes=%llu body=%016llx seqx_len=%llu seqy_len=%llu total_frags=%llu\n", m->n,
         (unsigned long long)bytes, (unsigned long long)fnv(body, bytes), (unsigned long long)lx, (unsigned long long)ly,
         (unsigned long long)total);
  return load_csv(body, bytes, total, "rank 0: Unexpected number of fragments", st, csv);  // every rank refuses alike
}
}

int main(int argc, char **argv) {
  if (argc < 2) return 2;
  std::vector<int> devices(argc >= 3 ? atoi(argv[2]) : 1);
  for (size_t i = 0; i < devices.size(); ++i) devices[i] = (int)i;
  const bool device_parser = argc >= 4 && !strcmp(argv[3], "device");
  int rc = 0;
  try {
    std::ifstream in(argv[1], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    std::unique_ptr<FragmentsDatabase> db(device_parser ? new FragmentsDatabase(in, sm, devices, CsvOnDevice{})
                                                        : new FragmentsDatabase(in, sm, devices, detect_frags_input(argv[1], in)));
    const uint64_t n = db->getTotalFrags();
    printf("getA=%zu total=%llu seqs=%llu len0=%llu len1=%llu max=%llu parser=%d multi=%d\n", db->getA(), (unsigned long long)n,
           (unsigned long long)sm.get_number_of_sequences(), (unsigned long long)sm.get_sequence_by_label(0).len,
           (unsigned long long)sm.get_sequence_by_label(1).len, (unsigned long long)sm.get_maximum_length(), (int)db->device_parser(),
           (int)(db->multi() != nullptr && db->ctx() == nullptr));
    printf("records=%016llx\n", (unsigned long long)fnv(db->records(), n * sizeof(FragFile)));
    if (devices.size() == 1) {  // the visiting order comes from the device's rank_fidx, which a partitioned load does not keep
      uint64_t h = fnv(nullptr, 0);
      for (const std::vector<FragFile> *b = db->begin(); b != db->end(); ++b) {
        const uint64_t size = b->size();
        h = fnv(b->data(), size * sizeof(FragFile), fnv(&size, sizeof size, h));
      }
      printf("buckets=%016llx\n", (unsigned long long)h);
    }
    printf("header_lines=%zu header=%016llx\n", (size_t)std::count(sm.raw_header().begin(), sm.raw_header().end(), '\n'),
           (unsigned long long)fnv(sm.raw_header().data(), sm.raw_header().size()));
  } catch (const std::exception &e) {
    printf("exception: %s\n", e.what());
    rc = 1;
  }
  printf("live ctx=%d multi=%d host=%d\n", g_live_ctx, g_live_multi, g_live_host);
  return rc;
}
