#include "FragmentsDatabase.h"

#include "GeckoFrags.h"

#include <algorithm>
#include <atomic>

#include <chrono>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <memory>
#include <stdexcept>
#include <thread>
#include <vector>

bool parse_plain_float(const char *p, size_t n, float *out) { return rk_csv::plain_float(p, n, *out); }

namespace {
long long value_after_colon(const std::string &line) {  // atoll(line.substr(line.find(':') + 1)), :62,65,72
  const size_t p = line.find(':');
  return atoll(line.c_str() + (p == std::string::npos ? 0 : p + 1));
}
}  // namespace

namespace {
// rows of data[begin, end) in file order, parsed by one thread ("\n"-separated like std::getline; the caller makes
// sure a range starts at the beginning of a row)
struct ParsedChunk {
  std::vector<FragFile> rows;
};
void parse_range(const char *data, size_t begin, size_t end, bool last_range, ParsedChunk *out) {
  size_t pos = begin;
  bool eof = begin >= end && !last_range;
  while (!eof) {  // reference: FragmentsDatabase.cpp:92-100; the final getline on an exhausted stream yields one empty line
    const size_t s = pos;
    while (pos < end && data[pos] != '\n') ++pos;
    const size_t l = pos - s;
    if (pos < end) {
      ++pos;
      if (pos >= end && !last_range) eof = true;  // the row after this '\n' belongs to the next range
    } else {
      eof = true;
    }
    FragFile tmp;
    memset(&tmp, 0, sizeof tmp);
    if (readFragment(&tmp, data + s, l)) out->rows.push_back(tmp);
  }
}
}  // namespace

// The data rows of text[pos, size) parsed by nthreads threads: the text is cut at row boundaries into one range per
// thread, every thread keeps its accepted rows in file order, and the ranges are returned in order — the same
// records, in the same order, as the reference's row-by-row loop (FragmentsDatabase.cpp:92-100).
std::vector<std::vector<FragFile>> parse_rows_parallel(const char *data, size_t size, size_t pos, unsigned nthreads) {
  if (nthreads < 1) nthreads = 1;
  if (nthreads > 64) nthreads = 64;
  const size_t body = size - pos;
  std::vector<size_t> cut(nthreads + 1, size);
  cut[0] = pos;
  for (unsigned t = 1; t < nthreads; ++t) {
    size_t c = pos + body / nthreads * t;
    if (c < cut[t - 1]) c = cut[t - 1];
    while (c > 0 && c < size && data[c - 1] != '\n') ++c;  // move to the start of the next row
    cut[t] = c;
  }
  std::vector<ParsedChunk> chunks(nthreads);
  if (size != 0) {  // reference: an empty stream never enters the row loop
    std::vector<std::thread> pool;
    for (unsigned t = 0; t < nthreads; ++t) {
      const bool last = t + 1 == nthreads;
      if (!last && cut[t] >= cut[t + 1]) continue;  // empty range
      chunks[t].rows.reserve((cut[t + 1] - cut[t]) / 48 + 16);  // GECKO rows are 60..90 bytes
      pool.emplace_back(parse_range, data, cut[t], cut[t + 1], last, &chunks[t]);
    }
    for (auto &th : pool) th.join();
  }
  std::vector<std::vector<FragFile>> out(nthreads);
  for (unsigned t = 0; t < nthreads; ++t) out[t].swap(chunks[t].rows);
  return out;
}

FragsHead read_frags_head(const char *data, size_t size, FragsInput input) {
  FragsHead h;
  h.binary = input == FragsInput::gecko_binary;
  if (h.binary) {  // GeckoFrags.h: 16-byte header, 109-byte big-endian records
    if (!gecko_frags_layout_ok(size))
      throw std::runtime_error("repkiller-b200: not a GECKO binary fragments file (16-byte header + 109-byte records)");
    uint64_t nx = 0, ny = 0;
    gecko_frags_lengths((const unsigned char *)data, &nx, &ny);
    h.total_frags = gecko_frags_count(size);
    // the header the output file starts with: the 16 lines GECKO's CSV rendering of this file would carry
    h.header = "All by-Identity Ungapped Fragments (Hits based approach)\n"
               "[Abr.2015 -- < bitlab - Departamento de Arquitectura de Computadores >\n"
               "SeqX filename : (binary fragments file)\nSeqY filename : (binary fragments file)\n"
               "SeqX name : X\nSeqY name : Y\n"
               "SeqX length : " + std::to_string(nx) + "\nSeqY length : " + std::to_string(ny) + "\n"
               "Min.fragment.length : 0\nMin.Identity : 0.00\nTot Hits (seeds) : 0\nTot Hits (seeds) used: 0\n"
               "Total fragments : " + std::to_string(h.total_frags) + "\n"
               "========================================================\n"
               "Type,xStart,yStart,xEnd,yEnd,strand(f/r),block,length,score,ident,similarity,%ident,SeqX,SeqY\n"
               "========================================================\n";
    h.seqx_len = nx + 1, h.seqy_len = ny + 1;  // like the CSV route: header value + 1 (:62,65)
    h.body_pos = GECKO_FRAGS_HEADER_BYTES;
    return h;
  }
  size_t pos = 0;
  auto next_line = [&](std::string &out) {
    const size_t s = pos;
    while (pos < size && data[pos] != '\n') ++pos;
    out.assign(data + s, pos - s);
    if (pos < size) ++pos;
  };
  std::string line;
  for (int ln = 1; ln <= 16; ++ln) {  // reference: :57-77
    next_line(line);
    h.header.append(line).append("\n");
    if (ln == 7) h.seqx_len = (uint64_t)(value_after_colon(line) + 1);
    if (ln == 8) h.seqy_len = (uint64_t)(value_after_colon(line) + 1);
    if (ln == 13) h.total_frags = (uint64_t)value_after_colon(line);
  }
  h.body_pos = pos;
  return h;
}

std::vector<std::vector<FragFile>> read_frags_records(const char *data, size_t size, const FragsHead &head, unsigned nthreads) {
  // by all host cores (RK_PARSE_THREADS overrides the count)
  if (nthreads == 0) {
    nthreads = std::thread::hardware_concurrency();
    if (nthreads < 1 || size - head.body_pos < (1u << 20)) nthreads = 1;
    if (const char *e = getenv("RK_PARSE_THREADS")) nthreads = (unsigned)atoi(e);
  }
  if (nthreads < 1) nthreads = 1;
  if (nthreads > 64) nthreads = 64;
  if (!head.binary) return parse_rows_parallel(data, size, head.body_pos, nthreads);
  // consecutive record ranges, byte-swapped
  std::vector<std::vector<FragFile>> chunks(nthreads);
  std::vector<std::thread> pool;
  const uint64_t n = head.total_frags;
  for (unsigned t = 0; t < nthreads; ++t) {
    const uint64_t lo = n / nthreads * t + std::min<uint64_t>(t, n % nthreads), hi = n / nthreads * (t + 1) + std::min<uint64_t>(t + 1, n % nthreads);
    if (hi > lo)
      pool.emplace_back([&chunks, t, lo, hi, data] {
        chunks[t].resize(hi - lo);
        gecko_frags_decode((const unsigned char *)data, lo, hi - lo, chunks[t].data());
      });
  }
  for (auto &th : pool) th.join();
  return chunks;
}

FragsInput detect_frags_input(const std::string &path, std::ifstream &stream) {
  if (const char *e = getenv("RK_INPUT_FORMAT")) {
    if (!strcmp(e, "frags")) return FragsInput::gecko_binary;
    if (!strcmp(e, "csv")) return FragsInput::csv;
  }
  static const char suffix[] = ".frags";
  const size_t sl = sizeof suffix - 1;
  if (path.size() < sl || path.compare(path.size() - sl, sl, suffix) != 0) return FragsInput::csv;
  const std::streampos here = stream.tellg();
  stream.seekg(0, std::ios::end);
  const std::streampos fin = stream.tellg();
  if (here == std::streampos(-1) || fin == std::streampos(-1) || fin < here) {
    stream.clear();
    return FragsInput::csv;
  }
  stream.seekg(here);
  const int first = stream.peek();
  stream.clear();
  stream.seekg(here);
  return (gecko_frags_layout_ok((size_t)(fin - here)) && first == 0) ? FragsInput::gecko_binary : FragsInput::csv;
}

void read_stream_rest(std::ifstream &in, FragsText &out) {
  const std::streampos here = in.tellg();
  in.seekg(0, std::ios::end);
  const std::streampos fin = in.tellg();
  if (here != std::streampos(-1) && fin != std::streampos(-1) && fin >= here) {
    in.seekg(here);
    const size_t want = (size_t)(fin - here);
    out.raw.reset(new char[want + 1]);
    in.read(out.raw.get(), (std::streamsize)want);
    out.size = (size_t)in.gcount();
    out.data = out.raw.get();
  } else {  // not seekable
    in.clear();
    out.fallback.assign((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    out.data = out.fallback.data();
    out.size = out.fallback.size();
  }
}

// Both public constructors delegate to the empty one first, so that the destructor releases the contexts and buffers when
// ingest() throws.
FragmentsDatabase::FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices,
                                     FragsInput input)
    : FragmentsDatabase() {
  ingest(frags_file, seq_manager, devices, input, false);
}

FragmentsDatabase::FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices,
                                     CsvOnDevice)
    : FragmentsDatabase() {
  ingest(frags_file, seq_manager, devices, FragsInput::csv, true);
}

void FragmentsDatabase::ingest(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices,
                               FragsInput input, bool csv_on_device) {
  using clk = std::chrono::steady_clock;
  const auto t0 = clk::now();
  // CUDA start-up (a few hundred ms, every device's) runs beside the file read and the host parse
  std::thread create_thread([this, &devices] {
    if (devices.size() > 1) multi_ = rk_create_multi(devices.data(), (int)devices.size());
    else ctx_ = rk_create(devices.empty() ? 0 : devices[0]);
  });
  struct Joiner {
    std::thread &t;
    ~Joiner() { if (t.joinable()) t.join(); }
  } create_joiner{create_thread};
  // slurp the rest of the stream in one read; lines are split on '\n' like std::getline
  std::unique_ptr<FragsText> text(new FragsText);
  read_stream_rest(frags_file, *text);
  const char *data = text->data;
  const size_t size = text->size;
  const auto t1 = clk::now();
  const FragsHead head = read_frags_head(data, size, input);
  header = head.header;
  seq_manager.sequences.emplace_back(0, head.seqx_len);
  seq_manager.sequences.emplace_back(1, head.seqy_len);
  const uint64_t total_frags = head.total_frags;
  seq_manager.read_header(header);
  vsize = 1 + seq_manager.get_sequence_by_label(0).len / 10;  // :84
  create_thread.join();
  if (!ctx_ && !multi_) throw std::runtime_error(std::string("repkiller-b200: ") + rk_create_error());

  int rc;
  uint64_t accepted = 0;
  auto t2 = clk::now();
  if (csv_on_device) {  // the device splits and parses the rows; over several devices every one parses its slice
    const char *body = data + head.body_pos;
    const uint64_t bytes = size - head.body_pos;
    rc = multi_ ? rk_multi_load_csv(multi_, body, bytes, head.seqx_len, head.seqy_len, total_frags, RK_F_TIMING, &load_stats_, &csv_stats_)
                : rk_load_csv(ctx_, body, bytes, head.seqx_len, head.seqy_len, total_frags, RK_F_TIMING, &load_stats_, &csv_stats_);
  } else {
    // The device gets the compact form (rk_load_packed: 33 B per fragment over PCIe instead of the 109-byte record):
    // pinned memory for it is allocated beside the parse, for min(T, bytes / 28) records — a full GECKO row has 14
    // non-empty fields and 13 commas, i.e. at least 30 bytes with its line end.  This is only a guess: readFragment's
    // short-row padding also accepts rows like "Frag,5" (7 bytes), so the count is checked after the parse and the buffers
    // are re-allocated for exactly `accepted` records when the guess was too small.  (A binary file states its count.)
    const uint64_t rows_upper = head.binary ? total_frags : (size - head.body_pos) / 28 + 1;
    uint64_t cap = (rows_upper < total_frags ? rows_upper : total_frags) + 2;
    auto packed_bytes = [](uint64_t records) { return records * 33 + 64; };
    std::thread alloc_thread([this, cap, &packed_bytes] { packed_ = (unsigned char *)rk_host_alloc(packed_bytes(cap)); });
    Joiner alloc_joiner{alloc_thread};
    std::vector<std::vector<FragFile>> chunks = read_frags_records(data, size, head, 0);
    for (const auto &c : chunks) accepted += c.size();
    alloc_thread.join();
    if (accepted > total_frags) throw std::runtime_error("Unexpected number of fragments");  // :99
    if (accepted > cap) {  // short rows: more records than bytes / 28
      if (packed_) rk_host_free(packed_);
      cap = accepted;
      packed_ = (unsigned char *)rk_host_alloc(packed_bytes(cap));
    }
    records_ = (FragFile *)malloc((accepted ? accepted : 1) * sizeof(FragFile));
    if (!records_ || !packed_) throw std::runtime_error("Could not allocate memory for fragments!");  // :86
    // records in file order (the facades hand out pointers into them) and, beside them, the compact arrays for the device:
    // key4 = {xStart, yStart, length, ident}, rest4 = {xEnd, yEnd, score, similarity bits}, one strand byte
    uint32_t *key4 = (uint32_t *)packed_, *rest4 = key4 + 4 * cap;
    unsigned char *strand = (unsigned char *)(rest4 + 4 * cap);
    std::atomic<bool> wide{false};  // a value beyond 32 bits: the device then takes the 109-byte records (rk_load_aos)
    {
      std::vector<std::thread> pool;
      uint64_t off = 0;
      for (auto &c : chunks) {
        if (!c.empty())
          pool.emplace_back([this, off, &c, key4, rest4, strand, &wide] {
            memcpy(records_ + off, c.data(), c.size() * sizeof(FragFile));
            bool w = false;
            for (size_t k = 0; k < c.size(); ++k) {
              const FragFile &f = c[k];
              const uint64_t i = off + k;
              w = w || ((f.xStart | f.yStart | f.length | f.ident | f.xEnd | f.yEnd | f.score) >> 32) != 0;
              key4[4 * i] = (uint32_t)f.xStart, key4[4 * i + 1] = (uint32_t)f.yStart, key4[4 * i + 2] = (uint32_t)f.length, key4[4 * i + 3] = (uint32_t)f.ident;
              rest4[4 * i] = (uint32_t)f.xEnd, rest4[4 * i + 1] = (uint32_t)f.yEnd, rest4[4 * i + 2] = (uint32_t)f.score;
              memcpy(&rest4[4 * i + 3], &f.similarity, 4);
              strand[i] = (unsigned char)f.strand;
            }
            if (w) wide = true;
          });
        off += c.size();
      }
      for (auto &th : pool) th.join();
    }
    t2 = clk::now();
    const uint64_t lx1 = seq_manager.get_sequence_by_label(0).len, ly1 = seq_manager.get_sequence_by_label(1).len;
    rc = multi_  ? rk_multi_load_aos(multi_, records_, accepted, lx1, ly1, RK_F_TIMING, &load_stats_)  // consecutive slices per rank
         : wide  ? rk_load_aos(ctx_, records_, accepted, lx1, ly1, RK_F_TIMING, &load_stats_)
                 : rk_load_packed(ctx_, key4, strand, rest4, accepted, lx1, ly1, RK_F_TIMING, &load_stats_);
  }
  if (rc != RK_OK) {
    const std::string err = multi_ ? rk_multi_last_error(multi_) : rk_last_error(ctx_);
    // the device parser's count refusal, as the host route throws it (:99); over several devices it carries a "rank r: " prefix
    if (rc == RK_ERR_RANGE && err.find("Unexpected number of fragments") != std::string::npos)
      throw std::runtime_error("Unexpected number of fragments");
    throw std::runtime_error("repkiller-b200: " + err);
  }
  const auto t3 = clk::now();
  count_ = csv_on_device ? load_stats_.n_loaded : accepted;
  device_parser_ = csv_on_device;
  if (csv_on_device) {  // the text is kept for records(), which parses it with the host parser on first use
    body_pos_ = head.body_pos;
    text_ = std::move(text);
  }
  ms_read_ = std::chrono::duration<double, std::milli>(t1 - t0).count();
  // host route: the host parse; device route: the device's text upload and row parse (over several devices the largest rank's)
  ms_parse_ = csv_on_device ? csv_stats_.ms_upload + csv_stats_.ms_parse : std::chrono::duration<double, std::milli>(t2 - t1).count();
  ms_device_load_ = std::chrono::duration<double, std::milli>(t3 - t2).count();
}

// FragmentsDatabase.cpp:84-97 of the reference fills loaded_frags[xStart/10] by push_back in file order.  Here the
// visiting order comes from the device (rank_fidx = the stable radix sort of K2a: bucket by bucket, file order inside),
// so iterating begin()..end() visits exactly the fragments, in exactly the order, that rk_group processes.
void FragmentsDatabase::build_buckets() const {
  std::unique_ptr<std::vector<FragFile>[]> b(new std::vector<FragFile>[vsize]);
  const FragFile *recs = records();
  const uint64_t kept = load_stats_.n_kept;
  std::vector<uint32_t> rank_fidx(kept ? kept : 1);
  if (kept) {
    const int64_t got = rk_debug_fetch(ctx_, "rank_fidx", rank_fidx.data(), kept * sizeof(uint32_t));
    if (got < 0) throw std::runtime_error(std::string("repkiller-b200: ") + rk_last_error(ctx_));
  }
  for (uint64_t i = 0; i < kept; ++i) {
    const FragFile &f = recs[rank_fidx[i]];
    b[f.xStart / 10].push_back(f);
  }
  if (kept < count_)  // fragments of bucket getA()-1: loaded by the reference, never visited (FragmentsDatabase.h:29-31)
    for (uint64_t i = 0; i < count_; ++i)
      if (recs[i].xStart / 10 == vsize - 1) b[vsize - 1].push_back(recs[i]);
  buckets_ = std::move(b);
}

// After a device parse the host records come from the kept text, parsed by the host parser: the same records the device
// loaded (both apply readFragment's rules), and the same bytes the host route's constructor holds.
const FragFile *FragmentsDatabase::records() const {
  std::call_once(records_once_, [this] {
    if (!text_) return;
    FragsHead head;
    head.body_pos = body_pos_;
    std::vector<std::vector<FragFile>> chunks = read_frags_records(text_->data, text_->size, head, 0);  // all cores
    uint64_t accepted = 0;
    for (const auto &c : chunks) accepted += c.size();
    if (accepted != count_) throw std::runtime_error("repkiller-b200: the host parser accepted a different number of rows than the device");
    records_ = (FragFile *)malloc((accepted ? accepted : 1) * sizeof(FragFile));
    if (!records_) throw std::runtime_error("Could not allocate memory for fragments!");
    uint64_t off = 0;
    for (const auto &c : chunks) {
      if (!c.empty()) memcpy(records_ + off, c.data(), c.size() * sizeof(FragFile));
      off += c.size();
    }
    text_.reset();
  });
  return records_;
}

const std::vector<FragFile> *FragmentsDatabase::begin() const {
  std::call_once(buckets_once_, [this] { build_buckets(); });
  return buckets_.get();
}

FragmentsDatabase::~FragmentsDatabase() {
  for (rk_ctx *v : pool_.views) rk_destroy(v);
  for (rk_multi *v : pool_.multi_views) rk_destroy_multi(v);
  if (ctx_) rk_destroy(ctx_);
  if (multi_) rk_destroy_multi(multi_);
  free(records_);
  if (packed_) rk_host_free(packed_);
}
