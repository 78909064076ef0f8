// The FragmentsDatabase constructor that parses the CSV rows on several devices (CsvOnDevice with a device list,
// host/FragmentsDatabaseMultiCsv.cpp) against a RECORDING stand-in for librk_b200 (test only: the stand-in notes what the
// constructor hands to rk_multi_load_csv and loads what readFragment accepts, so that n_loaded is what the library would
// report).  Checks the host glue without a GPU: the body handed over, the lengths and the stated count; and that
// records(), getA() and getTotalFrags() equal those of the host parser's constructor for several devices on the same file.
// Build: g++ this file + host/FragmentsDatabase.cpp + host/FragmentsDatabaseMultiCsv.cpp + host/GeckoFrags.cpp.
//   multi_csv_glue_check <in.csv> [device]     prints one line per fact ("device": only the CsvOnDevice constructor)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <string>
#include <vector>

#include "../../repkiller_b200/csrc/host/FragmentsDatabase.h"

namespace {
uint64_t fnv(const void *p, size_t n, uint64_t h = 1469598103934665603ull) {
  const unsigned char *b = (const unsigned char *)p;
  for (size_t i = 0; i < n; ++i) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}
std::string g_error;
}  // namespace

struct rk_ctx { int device; };
struct rk_multi { int n; };

extern "C" {
rk_ctx *rk_create(int device) { return new rk_ctx{device}; }
void rk_destroy(rk_ctx *c) { delete c; }
rk_multi *rk_create_multi(const int *, int n) { return new rk_multi{n}; }
void rk_destroy_multi(rk_multi *m) { delete m; }
const char *rk_create_error(void) { return ""; }
const char *rk_last_error(const rk_ctx *) { return ""; }
const char *rk_multi_last_error(const rk_multi *) { return g_error.c_str(); }
void *rk_host_alloc(size_t bytes) { return malloc(bytes); }
void rk_host_free(void *p) { free(p); }
int64_t rk_debug_fetch(rk_ctx *, const char *, void *, uint64_t) { return -1; }
static void fill(rk_load_stats *st, uint64_t n) {
  memset(st, 0, sizeof *st);
  st->n_loaded = n, st->n_kept = n;
}
int rk_load_packed(rk_ctx *, const uint32_t *, const uint8_t *, const uint32_t *, uint64_t n, uint64_t, uint64_t, unsigned, rk_load_stats *st) {
  fill(st, n);
  return 0;
}
int rk_load_aos(rk_ctx *, const void *, uint64_t n, uint64_t, uint64_t, unsigned, rk_load_stats *st) {
  fill(st, n);
  return 0;
}
int rk_multi_load_aos(rk_multi *m, const void *, uint64_t n, uint64_t, uint64_t, unsigned, rk_load_stats *st) {
  printf("call rk_multi_load_aos ranks=%d n=%llu\n", m->n, (unsigned long long)n);
  fill(st, n);
  return 0;
}
int rk_multi_load_csv(rk_multi *m, const char *body, uint64_t bytes, uint64_t lx, uint64_t ly, uint64_t total, unsigned,
                      rk_load_stats *st, rk_csv_stats *csv) {
  printf("call rk_multi_load_csv ranks=%d bytes=%llu body=%016llx seqx_len=%llu seqy_len=%llu total_frags=%llu\n", m->n,
         (unsigned long long)bytes, (unsigned long long)fnv(body, bytes), (unsigned long long)lx, (unsigned long long)ly,
         (unsigned long long)total);
  uint64_t rows = 0, acc = 0;
  for (uint64_t pos = 0;; ++rows) {  // rows split on '\n'; the segment after the last one is a row too
    const uint64_t s = pos;
    while (pos < bytes && body[pos] != '\n') ++pos;
    FragFile f;
    acc += readFragment(&f, body + s, pos - s);
    if (pos++ >= bytes) break;
  }
  if (acc > total) {
    g_error = "rank 0: Unexpected number of fragments";
    return RK_ERR_RANGE;
  }
  fill(st, acc);
  memset(csv, 0, sizeof *csv);
  csv->n_rows = rows + 1, csv->n_accepted = acc;
  return 0;
}
}

int main(int argc, char **argv) {
  if (argc < 2) return 2;
  const std::vector<int> devices{0, 0, 0};
  try {
    if (argc >= 3 && !strcmp(argv[2], "device")) {
      std::ifstream in(argv[1], std::ifstream::in | std::ifstream::binary);
      sequence_manager sm;
      FragmentsDatabase dev(in, sm, devices, CsvOnDevice{});
      printf("device total=%llu\n", (unsigned long long)dev.getTotalFrags());
      return 0;
    }
    std::ifstream ih(argv[1], std::ifstream::in | std::ifstream::binary), id(argv[1], std::ifstream::in | std::ifstream::binary);
    sequence_manager sh, sd;
    FragmentsDatabase dev(id, sd, devices, CsvOnDevice{});
    FragmentsDatabase host(ih, sh, devices, FragsInput::csv);
    const uint64_t n = dev.getTotalFrags();
    printf("device getA=%zu total=%llu len0=%llu len1=%llu parser=%d multi=%d\n", dev.getA(), (unsigned long long)n,
           (unsigned long long)sd.get_sequence_by_label(0).len, (unsigned long long)sd.get_sequence_by_label(1).len, (int)dev.device_parser(),
           (int)(dev.multi() != nullptr && dev.ctx() == nullptr));
    printf("host getA=%zu total=%llu len0=%llu len1=%llu parser=%d multi=%d\n", host.getA(), (unsigned long long)host.getTotalFrags(),
           (unsigned long long)sh.get_sequence_by_label(0).len, (unsigned long long)sh.get_sequence_by_label(1).len, (int)host.device_parser(),
           (int)(host.multi() != nullptr && host.ctx() == nullptr));
    const bool same_records = n == host.getTotalFrags() && (n == 0 || memcmp(dev.records(), host.records(), n * sizeof(FragFile)) == 0);
    printf("records=%016llx same_records=%d same_header=%d\n", (unsigned long long)fnv(dev.records(), n * sizeof(FragFile)),
           (int)same_records, (int)(sd.raw_header() == sh.raw_header()));
  } catch (const std::exception &e) {
    printf("exception: %s\n", e.what());
    return 1;
  }
  return 0;
}
