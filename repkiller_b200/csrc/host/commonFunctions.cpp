#include "commonFunctions.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <map>
#include <mutex>
#include <stdexcept>
#include <thread>

void print_help() {
  std::cout << "Repkiller v0.9.b\n";
  std::cout << "Usage: ./repkiller <input_file_path> <output_file_path> <length_ratio> <position_ratio>\n";
  std::cout << std::flush;
}

void init_args(const std::vector<std::string> &args, std::ifstream &multifrags, std::string &out_file_base_path,
               std::string &path_frags, std::queue<std::pair<double, double>> &params) {
  out_file_base_path.clear();
  path_frags.clear();
  if (args.size() < 4) throw std::invalid_argument("Invalid number of arguments.");
  path_frags = args.at(1);
  multifrags.open(path_frags, std::ifstream::in | std::ifstream::binary);
  if (!multifrags) throw std::runtime_error("Could not open input file " + path_frags + ".");
  out_file_base_path = args.at(2);
  if (out_file_base_path.empty()) throw std::runtime_error("Output file name is missing");
  for (size_t i = 3; i < args.size(); i += 2) {
    const double len_ratio = std::stod(args.at(i), nullptr);
    const double pos_ratio = std::stod(args.at(i + 1), nullptr);  // odd count: at() throws out_of_range, as the reference
    if (len_ratio <= 0) throw std::invalid_argument("Ratio between length and position must be greater than zero");
    if (pos_ratio <= 0) throw std::invalid_argument("Position proximity must be greater than zero");
    params.push(std::make_pair(len_ratio, pos_ratio));
  }
}

namespace {

void build_groups(const FragmentsDatabase &db, const rk_result &r, FGList &out) {
  const FragFile *recs = db.records();
  out.clear();
  out.reserve(r.n_groups);
  uint64_t j = 0;
  while (j < r.n_kept) {
    const uint32_t g = r.gid[j];
    uint64_t e = j;
    while (e < r.n_kept && r.gid[e] == g) ++e;
    FragsGroup *fg = new FragsGroup();
    fg->reserve(e - j);
    for (uint64_t k = j; k < e; ++k) fg->push_back(recs + r.order[k]);
    out.push_back(fg);
    j = e;
  }
}

[[noreturn]] void device_error(const FragmentsDatabase &db) {
  throw std::runtime_error(std::string("repkiller-b200: ") + (db.multi() ? rk_multi_last_error(db.multi()) : rk_last_error(db.ctx())));
}
[[noreturn]] void device_error(rk_ctx *ctx) { throw std::runtime_error(std::string("repkiller-b200: ") + rk_last_error(ctx)); }

// One grouping context of the database's pool (FragmentsDatabase::ContextPool) for the duration of one facade call:
// the base (ctx(), or multi() over several GPUs) when it is free, so that one thread makes exactly the calls it always
// made; else an idle view, or a new one.  H is rk_ctx or rk_multi.
template <class H>
class Pooled {
  const FragmentsDatabase &db_;
  H *h_ = nullptr;
  static H *base(const FragmentsDatabase &db);
  static std::vector<H *> &views(FragmentsDatabase::ContextPool &p);
  static std::vector<H *> &idle(FragmentsDatabase::ContextPool &p);
  static H *create_view(H *base);

 public:
  explicit Pooled(const FragmentsDatabase &db) : db_(db) {
    if (!base(db)) return;  // the other device count: no such context (the calls below then report the error)
    FragmentsDatabase::ContextPool &p = db.pool();
    std::lock_guard<std::mutex> lk(p.mu);
    if (!p.base_busy) {
      p.base_busy = true;
      h_ = base(db);
    } else if (!idle(p).empty()) {
      h_ = idle(p).back();
      idle(p).pop_back();
    } else {  // reads only the load of the base, which may be grouping on another thread meanwhile
      h_ = create_view(base(db));
      if (!h_) throw std::runtime_error(std::string("repkiller-b200: ") + rk_create_error());
      views(p).push_back(h_);
    }
  }
  ~Pooled() {
    if (!h_) return;
    FragmentsDatabase::ContextPool &p = db_.pool();
    std::lock_guard<std::mutex> lk(p.mu);
    if (h_ == base(db_)) p.base_busy = false;
    else idle(p).push_back(h_);
  }
  Pooled(const Pooled &) = delete;
  Pooled &operator=(const Pooled &) = delete;
  H *get() const { return h_; }
};
template <> rk_ctx *Pooled<rk_ctx>::base(const FragmentsDatabase &db) { return db.ctx(); }
template <> std::vector<rk_ctx *> &Pooled<rk_ctx>::views(FragmentsDatabase::ContextPool &p) { return p.views; }
template <> std::vector<rk_ctx *> &Pooled<rk_ctx>::idle(FragmentsDatabase::ContextPool &p) { return p.idle_views; }
template <> rk_ctx *Pooled<rk_ctx>::create_view(rk_ctx *b) { return rk_create_view(b); }
template <> rk_multi *Pooled<rk_multi>::base(const FragmentsDatabase &db) { return db.multi(); }
template <> std::vector<rk_multi *> &Pooled<rk_multi>::views(FragmentsDatabase::ContextPool &p) { return p.multi_views; }
template <> std::vector<rk_multi *> &Pooled<rk_multi>::idle(FragmentsDatabase::ContextPool &p) { return p.idle_multi_views; }
template <> rk_multi *Pooled<rk_multi>::create_view(rk_multi *b) { return rk_multi_create_view(b); }
using PooledContext = Pooled<rk_ctx>;

}  // namespace

size_t generate_fragment_groups(const FragmentsDatabase &frags_db, FGList &efrags_groups, const sequence_manager &,
                                double lensim, double possim) {
  rk_result r;
  PooledContext pc(frags_db);
  if (rk_group(pc.get(), lensim, possim, RK_F_HOST_RESULT | RK_F_NO_SORT, &r) != RK_OK) device_error(pc.get());
  build_groups(frags_db, r, efrags_groups);  // (before the context goes back: r's host arrays are the context's)
  std::cout << std::flush;  // reference: commonFunctions.cpp:78
  return efrags_groups.size();
}

void generate_diagonal_func(const FragmentsDatabase &fdb, size_t *diag_func) {
  static_assert(sizeof(size_t) == sizeof(uint64_t), "64-bit host");
  PooledContext pc(fdb);
  if (rk_diagonal_func(pc.get(), reinterpret_cast<uint64_t *>(diag_func)) != RK_OK) device_error(pc.get());
}

namespace {
// sort_groups has no database argument: it owns a small context (created on first use, calls serialised)
struct SortContext {
  std::mutex mtx;
  rk_ctx *ctx = nullptr;
  ~SortContext() { if (ctx) rk_destroy(ctx); }
};
SortContext g_sort;
}  // namespace

void sort_groups(FGList &fgl, const size_t *diag_func) {
  uint64_t m = 0;
  for (const FragsGroup *fg : fgl) m += fg->size();
  if (m == 0) return;
  std::vector<uint32_t> gid(m), perm(m);
  std::vector<uint64_t> y(m), d(m);
  uint64_t j = 0;
  uint32_t g = 0;
  for (const FragsGroup *fg : fgl) {
    for (const FragFile *f : *fg) {
      gid[j] = g;
      y[j] = f->yStart;
      d[j] = diag_func[f->xStart / 10];  // reference: commonFunctions.cpp:152,154
      ++j;
    }
    ++g;
  }
  std::lock_guard<std::mutex> lk(g_sort.mtx);
  if (!g_sort.ctx) {
    const char *e = getenv("RK_DEVICE");
    g_sort.ctx = rk_create(e ? atoi(e) : 0);
    if (!g_sort.ctx) throw std::runtime_error(std::string("repkiller-b200: ") + rk_create_error());
  }
  if (rk_sort_members(g_sort.ctx, m, gid.data(), y.data(), d.data(), perm.data()) != RK_OK)
    throw std::runtime_error(std::string("repkiller-b200: ") + rk_last_error(g_sort.ctx));
  j = 0;
  std::vector<const FragFile *> tmp;
  for (FragsGroup *fg : fgl) {
    const size_t n = fg->size();
    if (n > 1) {
      tmp.assign(fg->begin(), fg->end());
      for (size_t k = 0; k < n; ++k) (*fg)[k] = tmp[perm[j + k] - j];  // perm holds member indices of the whole list
    }
    j += n;
  }
}

FGList *group_and_sort(const FragmentsDatabase &frags_db, double len_ratio, double pos_ratio, rk_result *stats) {
  rk_result r;
  FGList *fgl = new FGList;
  if (frags_db.multi()) {  // one comparison over several GPUs: the ranks' ranges of lines come back concatenated
    Pooled<rk_multi> pm(frags_db);
    if (rk_multi_group(pm.get(), len_ratio, pos_ratio, RK_F_TIMING, &r) != RK_OK) {
      delete fgl;
      throw std::runtime_error(std::string("repkiller-b200: ") + rk_multi_last_error(pm.get()));
    }
    build_groups(frags_db, r, *fgl);
  } else {
    PooledContext pc(frags_db);
    if (rk_group(pc.get(), len_ratio, pos_ratio, RK_F_HOST_RESULT | RK_F_TIMING, &r) != RK_OK) {
      delete fgl;
      device_error(pc.get());
    }
    build_groups(frags_db, r, *fgl);
  }
  if (stats) *stats = r;  // (its host arrays are the context's, valid until its next grouping)
  return fgl;
}

void free_groups(FGList *fgl) {
  if (!fgl) return;
  for (FragsGroup *g : *fgl) delete g;
  delete fgl;
}

// ---- writer: byte-identical to commonFunctions.cpp:101-146 ---------------------------------------------
namespace {
inline char *put_u64(char *p, uint64_t v) {
  char tmp[24];
  int n = 0;
  do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
  while (n) *p++ = tmp[--n];
  return p;
}
inline char *put_float(char *p, float f) {  // ostream << float, default format: %g with precision 6
  return p + snprintf(p, 32, "%g", (double)f);
}
void store_frag(std::ostream &out, const FragFile *f, uint64_t gid, unsigned repval) {
  char line[320];
  char *p = line;
  memcpy(p, "Frag,", 5), p += 5;
  p = put_u64(p, f->xStart), *p++ = ',';
  p = put_u64(p, f->yStart), *p++ = ',';
  p = put_u64(p, f->xEnd), *p++ = ',';
  p = put_u64(p, f->yEnd), *p++ = ',';
  *p++ = f->strand, *p++ = ',';
  p = put_u64(p, gid), *p++ = ',';
  p = put_u64(p, f->length), *p++ = ',';
  p = put_u64(p, f->score), *p++ = ',';
  p = put_u64(p, f->ident), *p++ = ',';
  p = put_float(p, f->similarity), *p++ = ',';
  p = put_float(p, (float)f->ident * 100 / (float)f->length);  // reference: :103
  memcpy(p, ",0,", 3), p += 3;
  p = put_u64(p, repval), *p++ = '\n';
  out.write(line, p - line);
}
}  // namespace

void save_frags_from_group(std::ostream &out_file, FragsGroup &fg, uint64_t gid) {
  if (fg.size() == 1) {
    store_frag(out_file, fg.front(), gid, 0);
  } else {
    store_frag(out_file, fg.front(), gid, 1);
    for (auto it = fg.begin() + 1; it != fg.end(); ++it) store_frag(out_file, *it, gid, 2);
  }
}

void save_frag_pair(std::ostream &out_file, uint64_t, uint64_t, const sequence_manager &seq_mngr, const FGList &fgl) {
  uint64_t gid = 0;
  seq_mngr.write_header(out_file);
  for (auto fg : fgl) save_frags_from_group(out_file, *fg, gid++);
}

// The same file as save_all_frag_pairs, without the detour over an FGList: the lines of the last rk_group on this
// database are formatted on the device (rk_format_lines, K6; over several GPUs rk_multi_format_lines, every GPU its own
// lines) and written chunk by chunk.
void save_device_text(const std::string &out_file_base_path, const sequence_manager &seq_manager, const FragmentsDatabase &db,
                      float *ms_format) {
  std::ofstream out_file(out_file_base_path, std::ofstream::out | std::ofstream::binary);
  if (!out_file) throw std::runtime_error("Could not open output directory " + out_file_base_path);
  seq_manager.write_header(out_file);
  // chunks of 1M lines: the device formats chunk k+1 (rk_format_lines alternates between two pinned buffers) while
  // this thread's helper writes chunk k
  const uint64_t kChunk = 1000000;
  const uint64_t kept = db.load_stats().n_kept;
  uint64_t done = 0;
  float ms = 0.f;
  std::thread writer;
  while (done < kept) {
    const uint64_t cnt = kept - done < kChunk ? kept - done : kChunk;
    rk_text t;
    const int rc = db.multi() ? rk_multi_format_lines(db.multi(), done, cnt, &t) : rk_format_lines(db.ctx(), done, cnt, &t);
    if (writer.joinable()) writer.join();  // chunk k-1 is on its way to the file before chunk k+1 may reuse its buffer
    if (rc != RK_OK) device_error(db);
    writer = std::thread([&out_file, t] { out_file.write(t.text, (std::streamsize)t.n_bytes); });
    ms += t.ms_device;
    done += cnt;
  }
  if (writer.joinable()) writer.join();
  out_file.close();
  if (ms_format) *ms_format = ms;
}

void save_all_frag_pairs(const std::string &out_file_base_path, const sequence_manager &seq_manager, const FGList &fgl) {
  const uint64_t n_seq = seq_manager.get_number_of_sequences();
  std::ofstream out_file;
  for (uint64_t i = 0; i < n_seq; i++)
    for (uint64_t j = i + 1; j < n_seq; j++) {
      out_file.open(out_file_base_path, std::ofstream::out);
      if (!out_file) throw std::runtime_error("Could not open output directory " + out_file_base_path);
      save_frag_pair(out_file, i, j, seq_manager, fgl);
      out_file.close();
    }
}
