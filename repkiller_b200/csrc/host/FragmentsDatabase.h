// Drop-in for the reference's FragmentsDatabase (/root/reference/src/FragmentsDatabase.h:15-35): same
// constructor and accessors, but the per-bucket vector<FragFile>[] is replaced by the records in file order
// plus the device-side processing order built by the load.  Every constructor runs one routine (ingest): the file read
// beside the CUDA start-up, the 16 header lines, then one load call — the host parser's records to rk_load_packed /
// rk_load_aos / rk_multi_load_aos, or the CSV body to rk_load_csv / rk_multi_load_csv, which parse the rows on the devices.
#pragma once

#include <cstdint>
#include <fstream>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../rk_csv_row.cuh"  // readFragment (reference: FragmentsDatabase.cpp:17-50) and the number rules the device shares
#include "rk_b200.h"
#include "structs.h"

// the strtof fast path of readFragment (digits[.digits]): true and the correctly rounded float, or false = ask strtof
bool parse_plain_float(const char *p, size_t n, float *out);
// data rows of text[pos, size) parsed by nthreads threads; the accepted records of consecutive ranges, in file order
std::vector<std::vector<FragFile>> parse_rows_parallel(const char *text, size_t size, size_t pos, unsigned nthreads);

// what the stream holds: the GECKO CSV the reference reads, or GECKO's binary container (GeckoFrags.h; SURVEY §8f N4)
enum class FragsInput { csv, gecko_binary };
// What the CLI uses to choose: RK_INPUT_FORMAT=csv|frags decides; otherwise a file is taken as binary only when its name
// ends in ".frags", its size is a header plus whole records and it starts with a zero byte (a sequence length below 2^56;
// the CSV starts with text).  Everything else is read as the reference reads it.
FragsInput detect_frags_input(const std::string &path, std::ifstream &stream);
// The input stage of the constructor (no device involved).  Head: the header text the output file will start with, the
// sequence lengths as the reference holds them (file value + 1, FragmentsDatabase.cpp:62,65), the record count the file
// states, where the records start.  Records: the accepted records of consecutive ranges of the file, in file order,
// read by nthreads threads (0: all cores / RK_PARSE_THREADS).
struct FragsHead {
  std::string header;
  uint64_t seqx_len = 0, seqy_len = 0, total_frags = 0;
  size_t body_pos = 0;
  bool binary = false;
};
FragsHead read_frags_head(const char *data, size_t size, FragsInput input);
std::vector<std::vector<FragFile>> read_frags_records(const char *data, size_t size, const FragsHead &head, unsigned nthreads);
// The rest of a stream in one buffer (not a std::string when the stream can seek: resize() would zero-fill ~1 GB first).
struct FragsText {
  std::unique_ptr<char[]> raw;
  std::string fallback;  // a stream that cannot seek
  const char *data = nullptr;
  size_t size = 0;
};
void read_stream_rest(std::ifstream &in, FragsText &out);

// Tag of the constructors that parse the CSV rows on the device (rk_load_csv; over several devices rk_multi_load_csv).
struct CsvOnDevice {};

class FragmentsDatabase {
  mutable FragFile *records_ = nullptr;  // file order (built by records() on first use after a device parse)
  unsigned char *packed_ = nullptr;  // pinned: the compact arrays handed to rk_load_packed
  uint64_t count_ = 0;
  size_t vsize = 0;
  rk_ctx *ctx_ = nullptr;
  rk_multi *multi_ = nullptr;  // several GPUs: one comparison partitioned over them (rk_create_multi)
  std::string header;
  rk_load_stats load_stats_{};
  double ms_read_ = 0, ms_parse_ = 0, ms_device_load_ = 0;  // host wall clock of the three ingest phases
  // device parse: the file, kept so that records() can parse it on the host when a caller asks for host records
  mutable std::unique_ptr<FragsText> text_;
  size_t body_pos_ = 0;
  mutable std::once_flag records_once_;
  bool device_parser_ = false;
  rk_csv_stats csv_stats_{};
  // the reference's bucket array, built on first use from the processing order the device computed (K2a)
  mutable std::unique_ptr<std::vector<FragFile>[]> buckets_;
  mutable std::once_flag buckets_once_;
  void build_buckets() const;
  FragmentsDatabase() = default;
  // the body of every constructor; devices.size() > 1 partitions the comparison over them
  void ingest(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices, FragsInput input,
              bool csv_on_device);

 public:
  // The grouping contexts of the facades (generate_fragment_groups, generate_diagonal_func, group_and_sort), so that they
  // may run on several threads at once like the reference's: a call checks out ctx() when it is free, else an idle view
  // of it (rk_create_view, made by commonFunctions.cpp when every pooled context is busy), and checks it back in.  Over
  // several GPUs the same holds for multi() and its views (rk_multi_create_view).
  struct ContextPool {
    std::mutex mu;
    bool base_busy = false;              // ctx() (several GPUs: multi()) is checked out
    std::vector<rk_ctx *> views;         // every view made for the pool; destroyed with the database
    std::vector<rk_ctx *> idle_views;    // the ones not checked out
    std::vector<rk_multi *> multi_views, idle_multi_views;  // the same over several GPUs
  };
  ContextPool &pool() const { return pool_; }

 private:
  mutable ContextPool pool_;

 public:
  // Parses the GECKO CSV exactly like the reference (16 header lines, Frag rows, readFragment's accept/pad
  // rules), fills seq_manager, then hands the records to the GPU.  Throws std::runtime_error like the
  // reference on "Unexpected number of fragments"; also on device errors (message from rk_last_error).  Every
  // constructor that throws has released the contexts and buffers it made.
  FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, int device = 0, FragsInput input = FragsInput::csv)
      : FragmentsDatabase(frags_file, seq_manager, std::vector<int>{device}, input) {}
  // several devices: the comparison is partitioned over them (rk_multi_*); ctx() is then null and multi() is set
  // input = gecko_binary: the stream is a .frags file; every record loads as readFragment would load its CSV row
  FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices,
                    FragsInput input = FragsInput::csv);
  // CSV input with the rows parsed on the device (rk_load_csv; over several devices every one parses its slice,
  // rk_multi_load_csv) into the same database the host parser's constructor builds.  The file text is kept; records(),
  // begin() and the facades that read host records parse it on first use with the host parser (parse_rows_parallel), so
  // they hand out the same records.
  FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, int device, CsvOnDevice)
      : FragmentsDatabase(frags_file, seq_manager, std::vector<int>{device}, CsvOnDevice{}) {}
  FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices, CsvOnDevice);
  ~FragmentsDatabase();
  FragmentsDatabase(const FragmentsDatabase &) = delete;
  FragmentsDatabase &operator=(const FragmentsDatabase &) = delete;

  size_t getA() const { return vsize; }                 // reference: FragmentsDatabase.h:23-25
  uint64_t getTotalFrags() const { return count_; }      // reference: FragmentsDatabase.h:32-34
  // reference: FragmentsDatabase.h:26-31 — the xStart/10 bucket array; end() is begin() + getA() - 1, i.e. the last
  // bucket is never visited.  Built lazily (a host copy of every record, like the reference holds) from the device's
  // processing order; the grouping functions of this repo do not need it.
  const std::vector<FragFile> *begin() const;
  const std::vector<FragFile> *end() const { return begin() + vsize - 1; }
  const FragFile *records() const;                      // the records in file order
  rk_ctx *ctx() const { return ctx_; }
  rk_multi *multi() const { return multi_; }
  const rk_load_stats &load_stats() const { return load_stats_; }
  double ms_read() const { return ms_read_; }
  double ms_parse() const { return ms_parse_; }
  double ms_device_load() const { return ms_device_load_; }
  bool device_parser() const { return device_parser_; }  // built by a CsvOnDevice constructor
  const rk_csv_stats &csv_stats() const { return csv_stats_; }
};
