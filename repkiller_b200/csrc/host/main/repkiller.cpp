// repkiller — same command line, stdout and output file as the reference CLI (/root/reference/src/repkiller.cpp),
// with the grouping path on the GPU.
//   repkiller <input_file_path> <output_file_path> <length_ratio> <position_ratio> [<length_ratio> <position_ratio>]...
// Parameter pairs are processed in argv order on one device context while the writer thread saves the previous
// result; every pair writes the same path (as in the reference, repkiller.cpp:95-96), so the last pair's file
// remains ([survey choice]: the reference's 3-thread pool makes the survivor timing dependent).
// RK_TIMING=1 prints per-stage device times on stderr (parser=device|host: which parser read the CSV rows, with the parse
// milliseconds, over several GPUs the largest rank's, and the rows left to the host parser summed over the ranks;
// writer=device|host: which writer made the file); RK_DEVICE selects
// the GPU; RK_LEGACY_WRITER=1 formats the output on the host through FGList + SaverQueue instead of on the device (K6).
// RK_DEVICES=0,1,... partitions the comparison over several GPUs (rk_create_multi; NCCL between distinct devices); every
// GPU formats its own range of output lines (RK_F_LINE_RECORDS, rk_multi_format_lines), or the host writer does it
// under RK_LEGACY_WRITER=1.
#include <chrono>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <memory>
#include <queue>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../FragmentsDatabase.h"
#include "../SaverQueue.h"
#include "../commonFunctions.h"
#include "../structs.h"

static size_t fallback_count = 0;

static void execWithParams(const FragmentsDatabase &frag_db, const sequence_manager &seq_manager, std::pair<double, double> param,
                           const std::string &out_path, SaverQueue &sq, bool timing, bool legacy_writer) {
  rk_result st;
  if (legacy_writer) {  // RK_LEGACY_WRITER=1: host lists + the host formatter behind the reference's SaverQueue interface
    FGList *groups = group_and_sort(frag_db, param.first, param.second, &st);  // repkiller.cpp:83-91 in one device pass
    if (timing)
      std::cerr << "[rk] len_ratio=" << param.first << " pos_ratio=" << param.second << " groups=" << st.n_groups
                << " device_ms=" << st.ms_device << " launches=" << st.n_launches << " writer=host\n";
    sq.addRequest(out_path, groups);  // repkiller.cpp:95-96
    return;
  }
  // grouping (K3-K5) and the text of the output file (K6) on the device; the host only writes bytes.  Over several GPUs
  // every line's record is first brought to the GPU that holds the line.
  if (frag_db.multi()) {
    if (rk_multi_group(frag_db.multi(), param.first, param.second, RK_F_LINE_RECORDS | RK_F_TIMING, &st) != RK_OK)
      throw std::runtime_error(std::string("repkiller-b200: ") + rk_multi_last_error(frag_db.multi()));
  } else if (rk_group(frag_db.ctx(), param.first, param.second, RK_F_TIMING, &st) != RK_OK) {
    throw std::runtime_error(std::string("repkiller-b200: ") + rk_last_error(frag_db.ctx()));
  }
  float ms_format = 0.f;
  const auto tw0 = std::chrono::steady_clock::now();
  try {
    save_device_text(out_path, seq_manager, frag_db, &ms_format);
  } catch (const std::runtime_error &) {  // reference: SaverQueue.cpp:16-20
    const std::string default_path = "represults-" + std::to_string(++fallback_count) + ".csv";
    std::cerr << "Couldn't access " << out_path << ", saving into " << default_path << "\n" << std::flush;
    save_device_text(default_path, seq_manager, frag_db, &ms_format);
  }
  if (timing)
    std::cerr << "[rk] len_ratio=" << param.first << " pos_ratio=" << param.second << " groups=" << st.n_groups
              << " device_ms=" << st.ms_device << " launches=" << st.n_launches << " format_ms=" << ms_format << " write_call_ms="
              << std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tw0).count() << " writer=device\n";
}

int main(int argc, char *argv[]) {
  std::string out_file_base_path, multifrags_path;
  std::queue<std::pair<double, double>> params;
  std::ifstream frags_file;
  try {
    std::vector<std::string> args(argv, argv + argc);
    init_args(args, frags_file, out_file_base_path, multifrags_path, params);
  } catch (const std::invalid_argument &e) {
    std::cerr << e.what() << std::endl;
    print_help();
    exit(1);
  }
  std::cout << "--- Running REPKILLER v0.9.b ---\n"
               "     Bitlab - Arquitectura de Computadores\n"
               "           Universidad de M\xc3\xa1laga 2018\n"
               "\n"
            << std::flush;
  const bool timing = getenv("RK_TIMING") != nullptr;
  std::vector<int> devices;
  if (const char *list = getenv("RK_DEVICES")) {
    for (const char *p = list; *p;) {
      devices.push_back(atoi(p));
      while (*p && *p != ',') ++p;
      if (*p == ',') ++p;
    }
  }
  if (devices.empty()) devices.push_back(getenv("RK_DEVICE") ? atoi(getenv("RK_DEVICE")) : 0);
  const bool legacy_writer = getenv("RK_LEGACY_WRITER") != nullptr;

  sequence_manager seq_manager;
  // (beside the reference's CSV: GECKO's binary .frags container, see FragmentsDatabase.h).  CSV input: the rows are parsed
  // on the device, over several devices each parsing its slice; .frags input takes the host parser.
  const FragsInput input = detect_frags_input(multifrags_path, frags_file);
  std::unique_ptr<FragmentsDatabase> db_owner(input == FragsInput::csv ? new FragmentsDatabase(frags_file, seq_manager, devices, CsvOnDevice{})
                                                                       : new FragmentsDatabase(frags_file, seq_manager, devices, input));
  const FragmentsDatabase &frag_db = *db_owner;
  frags_file.close();
  if (timing) {
    const rk_load_stats &ls = frag_db.load_stats();
    std::cerr << "[rk] loaded=" << ls.n_loaded << " kept=" << ls.n_kept << " device_ms=" << ls.ms_device << " host: read_ms=" << frag_db.ms_read()
              << " parse_ms=" << frag_db.ms_parse() << " load_call_ms=" << frag_db.ms_device_load();
    if (frag_db.device_parser())
      std::cerr << " parser=device upload_ms=" << frag_db.csv_stats().ms_upload << " device_parse_ms=" << frag_db.csv_stats().ms_parse
                << " host_rows=" << frag_db.csv_stats().n_host_rows << "\n";
    else
      std::cerr << " parser=host\n";
  }

  SaverQueue sq(seq_manager);
  sq.start();
  while (!params.empty()) {
    auto param = params.front();
    params.pop();
    execWithParams(frag_db, seq_manager, param, out_file_base_path, sq, timing, legacy_writer);
  }
  sq.stop();
  std::cout << "Repkiller finished with no errors\n";
  return 0;
}
