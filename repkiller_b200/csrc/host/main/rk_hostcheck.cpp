// Test helper for the host side of the drop-in.
//   rk_hostcheck parse <in.csv> <out.bin> [threads]
//                                             readFragment over every data row: accepted records, 109 B each (no GPU);
//                                             with a thread count: through parse_rows_parallel, the database's parser
//   rk_hostcheck floatcheck <n> <seed>        the float fast path of the parser against strtof on n generated tokens (no GPU)
//   rk_hostcheck write <in.csv> <out.csv>     writer format: parses, then writes every accepted record as its own
//                                             singleton group in file order (no GPU)
//   rk_hostcheck steps <in.csv> <out.csv> <len_ratio> <pos_ratio>
//                                             the reference's call sequence (repkiller.cpp:83-96):
//                                             generate_fragment_groups -> generate_diagonal_func -> sort_groups ->
//                                             save_all_frag_pairs, each through its own facade (GPU)
//   rk_hostcheck steps_device <in.csv> <out.csv> <len_ratio> <pos_ratio>
//                                             the same on a database whose CSV rows were parsed on the device (the
//                                             CsvOnDevice constructor, rk_load_csv) (GPU)
//   rk_hostcheck pool <in.csv> <out_prefix> <threads> <len_ratio> <pos_ratio> [<len_ratio> <pos_ratio>]...
//                                             the body of the reference's execWithParams (the four calls of steps) for
//                                             every pair, run by <threads> threads that share one FragmentsDatabase, as
//                                             the reference's thread pool does (repkiller.cpp:60-72); pair k writes
//                                             <out_prefix>-<k>.csv.  Prints how many grouping contexts the facades used (GPU)
//   rk_hostcheck group_pool <in.csv> <devices> <threads> <len_ratio> <pos_ratio> [<len_ratio> <pos_ratio>]...
//                                             group_and_sort of every pair on one database over <devices> (a comma list,
//                                             as RK_DEVICES; "0,0,0" is three ranks on device 0), run by <threads> threads
//                                             that share it.  Prints "pair <k> groups=<n> lines=<m> hash=<h>" per pair in
//                                             pair order (h: FNV-1a over the file indices of the members, group by group),
//                                             then how many grouping contexts the pool used (GPU)
//   rk_hostcheck steps_pure <in.csv> <out.csv> <len_ratio> <pos_ratio> <len_ratio2> <pos_ratio2>
//                                             sort_groups is a pure function: a second grouping with other ratios is
//                                             made BEFORE the first list is sorted; the output is the first one's (GPU)
//   rk_hostcheck sort_any <in.csv> <len_ratio> <pos_ratio>
//                                             sort_groups with an arbitrary diag_func table against std::sort with the
//                                             reference's comparator (commonFunctions.cpp:148-159) on the same lists (GPU)
//   rk_hostcheck buckets <in.csv> <out.bin>   the records visited by begin()..end(), in visiting order (GPU)
//   rk_hostcheck tofrags <in.csv> <out.frags> the accepted records of a CSV as a GECKO binary file (GeckoFrags.h; no GPU)
//   rk_hostcheck fragsbin <in.frags> <out.bin>
//                                             the records a binary file loads as, 109 B each; prints "<seqX length>
//                                             <seqY length> <records>" (no GPU)
//   rk_hostcheck ingest <in> <out.bin> <out.header> [threads]
//                                             the input stage of the FragmentsDatabase constructor (detect_frags_input,
//                                             read_frags_head, read_frags_records) on a CSV or a .frags file: records,
//                                             header text; prints "<seqX len> <seqY len> <stated records> <binary>" (no GPU)
// Every mode that builds a FragmentsDatabase takes a CSV or a .frags file (detect_frags_input).
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../FragmentsDatabase.h"
#include "../GeckoFrags.h"
#include "../SaverQueue.h"
#include "../commonFunctions.h"

static std::vector<FragFile> parse_rows(const char *path, std::string *header) {
  std::ifstream in(path, std::ifstream::in | std::ifstream::binary);
  std::string data((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  size_t pos = 0;
  for (int ln = 0; ln < 16; ++ln) {
    const size_t s = pos;
    while (pos < data.size() && data[pos] != '\n') ++pos;
    if (header) header->append(data, s, pos - s).append("\n");
    if (pos < data.size()) ++pos;
  }
  std::vector<FragFile> out;
  bool eof = data.empty();
  while (!eof) {
    const size_t s = pos;
    while (pos < data.size() && data[pos] != '\n') ++pos;
    const size_t l = pos - s;
    if (pos < data.size()) ++pos; else eof = true;
    FragFile f;
    memset(&f, 0, sizeof f);
    if (readFragment(&f, data.data() + s, l)) out.push_back(f);
  }
  return out;
}

int main(int argc, char **argv) {
  if (argc < 4) return 2;
  const std::string mode = argv[1];
  if (mode == "parse") {
    std::vector<FragFile> recs;
    if (argc >= 5) {  // the multi-threaded parser of FragmentsDatabase
      std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
      std::string data((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
      size_t pos = 0;
      for (int ln = 0; ln < 16; ++ln) {
        while (pos < data.size() && data[pos] != '\n') ++pos;
        if (pos < data.size()) ++pos;
      }
      for (auto &c : parse_rows_parallel(data.data(), data.size(), pos, (unsigned)atoi(argv[4]))) recs.insert(recs.end(), c.begin(), c.end());
    } else {
      recs = parse_rows(argv[2], nullptr);
    }
    FILE *f = fopen(argv[3], "wb");
    if (!f) return 3;
    if (!recs.empty()) fwrite(recs.data(), sizeof(FragFile), recs.size(), f);
    fclose(f);
    return 0;
  }
  if (mode == "tofrags") {
    std::string header;
    std::vector<FragFile> recs = parse_rows(argv[2], &header);
    uint64_t len[2] = {0, 0};
    size_t pos = 0;
    for (int ln = 1; ln <= 8; ++ln) {  // lines 7 and 8: "SeqX length : N", "SeqY length : N"
      const size_t e = header.find('\n', pos);
      const std::string line = header.substr(pos, e - pos);
      if (ln >= 7) len[ln - 7] = (uint64_t)atoll(line.c_str() + line.find(':') + 1);
      pos = e + 1;
    }
    std::vector<unsigned char> file(GECKO_FRAGS_HEADER_BYTES + recs.size() * sizeof(FragFile));
    gecko_frags_encode(len[0], len[1], recs.data(), recs.size(), file.data());
    FILE *f = fopen(argv[3], "wb");
    if (!f) return 3;
    fwrite(file.data(), 1, file.size(), f);
    fclose(f);
    return 0;
  }
  if (mode == "fragsbin") {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    std::vector<unsigned char> file((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    if (!gecko_frags_layout_ok(file.size())) return 4;
    uint64_t nx, ny;
    gecko_frags_lengths(file.data(), &nx, &ny);
    const uint64_t n = gecko_frags_count(file.size());
    std::vector<FragFile> recs(n);
    gecko_frags_decode(file.data(), 0, n, recs.data());
    FILE *f = fopen(argv[3], "wb");
    if (!f) return 3;
    if (n) fwrite(recs.data(), sizeof(FragFile), n, f);
    fclose(f);
    printf("%llu %llu %llu\n", (unsigned long long)nx, (unsigned long long)ny, (unsigned long long)n);
    return 0;
  }
  if (mode == "ingest" && argc >= 5) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    if (!in) return 3;
    const FragsInput input = detect_frags_input(argv[2], in);
    in.seekg(0, std::ios::end);
    std::string data((size_t)in.tellg(), '\0');
    in.seekg(0);
    in.read(&data[0], (std::streamsize)data.size());
    try {
      const auto t0 = std::chrono::steady_clock::now();
      const FragsHead head = read_frags_head(data.data(), data.size(), input);
      const auto chunks = read_frags_records(data.data(), data.size(), head, argc >= 6 ? (unsigned)atoi(argv[5]) : 0);
      if (getenv("RK_TIMING"))
        fprintf(stderr, "[rk] records_ms=%.1f\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
      FILE *f = fopen(argv[3], "wb");
      if (!f) return 3;
      for (const auto &c : chunks)
        if (!c.empty()) fwrite(c.data(), sizeof(FragFile), c.size(), f);
      fclose(f);
      std::ofstream(argv[4], std::ofstream::binary) << head.header;
      printf("%llu %llu %llu %d\n", (unsigned long long)head.seqx_len, (unsigned long long)head.seqy_len,
             (unsigned long long)head.total_frags, (int)head.binary);
    } catch (const std::exception &e) {
      fprintf(stderr, "%s\n", e.what());
      return 4;
    }
    return 0;
  }
  if (mode == "floatcheck") {
    uint64_t rng = 88172645463325252ull ^ (uint64_t)atoll(argv[3]);
    auto nx = [&]() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; };
    long bad = 0, fast = 0, total = 0;
    char t[64];
    for (long i = 0, n = atol(argv[2]); i < n; ++i) {
      const int kind = (int)(nx() % 4);
      if (kind == 0) snprintf(t, sizeof t, "%.9g", (double)(float)((nx() % 1000000) / 10000.0));   // what gen.py writes
      else if (kind == 1) snprintf(t, sizeof t, "%llu.%0*llu", (unsigned long long)(nx() % 1000), (int)(1 + nx() % 15), (unsigned long long)(nx() % 100000000));
      else if (kind == 2) snprintf(t, sizeof t, "%.17g", (double)(nx() % (1ull << 40)) / (double)(1 + nx() % 100000));
      else snprintf(t, sizeof t, "%llu", (unsigned long long)(nx() % (1ull << 54)));
      if (strchr(t, 'e')) continue;
      float f;
      ++total;
      if (parse_plain_float(t, strlen(t), &f)) {
        ++fast;
        const float w = strtof(t, nullptr);
        if (memcmp(&f, &w, 4) != 0) {
          if (bad < 10) printf("MISMATCH %s fast=%.9g strtof=%.9g\n", t, f, w);
          ++bad;
        }
      }
    }
    printf("%ld tokens, %ld fast, %ld mismatches\n", total, fast, bad);
    return bad != 0;
  }
  if (mode == "write") {
    std::string header;
    auto recs = parse_rows(argv[2], &header);
    sequence_manager sm;
    sm.sequences.emplace_back(0, 0);
    sm.sequences.emplace_back(1, 0);
    sm.read_header(header);
    FGList *fgl = new FGList;
    for (auto &r : recs) fgl->push_back(new FragsGroup{&r});
    SaverQueue sq(sm);  // the writer thread of the drop-in: start, one request, drain
    sq.start();
    sq.addRequest(argv[3], fgl);
    sq.stop();
    return 0;
  }
  if ((mode == "steps" || mode == "steps_device") && argc >= 6) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    std::unique_ptr<FragmentsDatabase> owner(mode == "steps" ? new FragmentsDatabase(in, sm, 0, detect_frags_input(argv[2], in))
                                                             : new FragmentsDatabase(in, sm, 0, CsvOnDevice{}));
    const FragmentsDatabase &db = *owner;
    FGList groups;
    generate_fragment_groups(db, groups, sm, std::stod(argv[4]), std::stod(argv[5]));
    std::vector<size_t> diag(db.getA());
    generate_diagonal_func(db, diag.data());
    sort_groups(groups, diag.data());
    save_all_frag_pairs(argv[3], sm, groups);
    return 0;
  }
  if (mode == "pool" && argc >= 7) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    FragmentsDatabase db(in, sm, 0, detect_frags_input(argv[2], in));
    const std::string prefix = argv[3];
    const int nthreads = std::max(1, atoi(argv[4]));
    std::vector<std::pair<double, double>> pairs;
    for (int i = 5; i + 1 < argc; i += 2) pairs.emplace_back(std::stod(argv[i]), std::stod(argv[i + 1]));
    std::atomic<size_t> next{0};
    std::mutex err_mu;
    std::string err;
    auto worker = [&] {
      for (size_t k; (k = next++) < pairs.size();) {
        try {
          FGList groups;
          generate_fragment_groups(db, groups, sm, pairs[k].first, pairs[k].second);
          std::vector<size_t> diag(db.getA());
          generate_diagonal_func(db, diag.data());
          sort_groups(groups, diag.data());
          save_all_frag_pairs(prefix + "-" + std::to_string(k) + ".csv", sm, groups);
          for (FragsGroup *g : groups) delete g;
        } catch (const std::exception &e) {
          std::lock_guard<std::mutex> lk(err_mu);
          err = e.what();
        }
      }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; ++t) pool.emplace_back(worker);
    for (auto &th : pool) th.join();
    if (!err.empty()) {
      fprintf(stderr, "%s\n", err.c_str());
      return 4;
    }
    printf("%zu pairs on %d threads, %zu grouping contexts\n", pairs.size(), nthreads, 1 + db.pool().views.size());
    return 0;
  }
  if (mode == "group_pool" && argc >= 7) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    std::vector<int> devices;
    for (const char *p = argv[3]; *p;) {
      devices.push_back(atoi(p));
      while (*p && *p != ',') ++p;
      if (*p == ',') ++p;
    }
    FragmentsDatabase db(in, sm, devices, detect_frags_input(argv[2], in));
    const int nthreads = std::max(1, atoi(argv[4]));
    std::vector<std::pair<double, double>> pairs;
    for (int i = 5; i + 1 < argc; i += 2) pairs.emplace_back(std::stod(argv[i]), std::stod(argv[i + 1]));
    std::vector<std::string> lines(pairs.size());
    std::atomic<size_t> next{0};
    std::mutex err_mu;
    std::string err;
    auto worker = [&] {
      for (size_t k; (k = next++) < pairs.size();) {
        try {
          FGList *fgl = group_and_sort(db, pairs[k].first, pairs[k].second);
          uint64_t h = 1469598103934665603ull, m = 0;
          auto mix = [&](uint64_t v) { h = (h ^ v) * 1099511628211ull; };
          for (const FragsGroup *g : *fgl) {
            for (const FragFile *f : *g) mix((uint64_t)(f - db.records())), ++m;
            mix(~0ull);
          }
          lines[k] = "pair " + std::to_string(k) + " groups=" + std::to_string(fgl->size()) + " lines=" + std::to_string(m) +
                     " hash=" + std::to_string(h);
          free_groups(fgl);
        } catch (const std::exception &e) {
          std::lock_guard<std::mutex> lk(err_mu);
          err = e.what();
        }
      }
    };
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; ++t) pool.emplace_back(worker);
    for (auto &th : pool) th.join();
    if (!err.empty()) {
      fprintf(stderr, "%s\n", err.c_str());
      return 4;
    }
    for (const std::string &l : lines) printf("%s\n", l.c_str());
    printf("%zu grouping contexts\n", 1 + (db.multi() ? db.pool().multi_views.size() : db.pool().views.size()));
    return 0;
  }
  if (mode == "steps_pure" && argc >= 8) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    FragmentsDatabase db(in, sm, 0, detect_frags_input(argv[2], in));
    FGList groups, other;
    generate_fragment_groups(db, groups, sm, std::stod(argv[4]), std::stod(argv[5]));
    generate_fragment_groups(db, other, sm, std::stod(argv[6]), std::stod(argv[7]));  // leaves ITS state on the device
    std::vector<size_t> diag(db.getA());
    generate_diagonal_func(db, diag.data());
    sort_groups(other, diag.data());
    sort_groups(groups, diag.data());
    save_all_frag_pairs(argv[3], sm, groups);
    return 0;
  }
  if (mode == "sort_any" && argc >= 5) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    FragmentsDatabase db(in, sm, 0, detect_frags_input(argv[2], in));
    FGList groups;
    generate_fragment_groups(db, groups, sm, std::stod(argv[3]), std::stod(argv[4]));
    std::vector<size_t> diag(db.getA());
    for (size_t b = 0; b < diag.size(); ++b) diag[b] = (b * 2654435761ull) % 977;  // any table: many ties, no relation to the data
    FGList want;
    for (FragsGroup *g : groups) want.push_back(new FragsGroup(*g));
    for (FragsGroup *g : want) {
      if (g->size() <= 1) continue;
      const size_t *df = diag.data();
      std::sort(g->begin(), g->end(), [df](const FragFile *f1, const FragFile *f2) {
        const uint64_t d1 = df[f1->xStart / 10], d2 = df[f2->xStart / 10];
        const uint64_t h1 = f1->yStart > d1 ? f1->yStart - d1 : d1 - f1->yStart;
        const uint64_t h2 = f2->yStart > d2 ? f2->yStart - d2 : d2 - f2->yStart;
        return h1 < h2;
      });
    }
    sort_groups(groups, diag.data());
    size_t bad = 0, big = 0;
    for (size_t i = 0; i < groups.size(); ++i) {
      if (groups[i]->size() > 16) ++big;
      if (*groups[i] != *want[i]) ++bad;
    }
    printf("%zu groups, %zu with more than 16 members, %zu differ from std::sort\n", groups.size(), big, bad);
    return bad != 0;
  }
  if (mode == "buckets" && argc >= 4) {
    std::ifstream in(argv[2], std::ifstream::in | std::ifstream::binary);
    sequence_manager sm;
    FragmentsDatabase db(in, sm, 0, detect_frags_input(argv[2], in));
    FILE *f = fopen(argv[3], "wb");
    if (!f) return 3;
    for (const auto &fl : db)
      for (const auto &fr : fl) fwrite(&fr, sizeof(FragFile), 1, f);
    fclose(f);
    return 0;
  }
  return 2;
}
