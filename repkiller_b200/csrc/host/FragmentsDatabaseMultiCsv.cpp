// FragmentsDatabase for a comparison partitioned over several devices and CSV input, every device parsing its slice of
// the rows (rk_multi_load_csv).  Its own translation unit: FragmentsDatabase.cpp and FragmentsDatabaseDeviceCsv.cpp do not
// reference rk_multi_load_csv.
#include <chrono>
#include <stdexcept>
#include <thread>

#include "FragmentsDatabase.h"

FragmentsDatabase::FragmentsDatabase(std::ifstream &frags_file, sequence_manager &seq_manager, const std::vector<int> &devices,
                                     CsvOnDevice) {
  using clk = std::chrono::steady_clock;
  const auto t0 = clk::now();
  // CUDA start-up of every device runs beside the file read
  std::thread create_thread([this, &devices] { multi_ = rk_create_multi(devices.data(), (int)devices.size()); });
  struct Joiner {
    std::thread &t;
    ~Joiner() { if (t.joinable()) t.join(); }
  } create_joiner{create_thread};
  text_.reset(new FragsText);
  read_stream_rest(frags_file, *text_);
  const auto t1 = clk::now();
  const FragsHead head = read_frags_head(text_->data, text_->size, FragsInput::csv);
  header = head.header;
  body_pos_ = head.body_pos;
  seq_manager.sequences.emplace_back(0, head.seqx_len);
  seq_manager.sequences.emplace_back(1, head.seqy_len);
  seq_manager.read_header(header);
  vsize = 1 + seq_manager.get_sequence_by_label(0).len / 10;  // :84
  create_thread.join();
  if (!multi_) throw std::runtime_error(std::string("repkiller-b200: ") + rk_create_error());
  const auto t2 = clk::now();
  const int rc = rk_multi_load_csv(multi_, text_->data + head.body_pos, text_->size - head.body_pos, head.seqx_len, head.seqy_len,
                                   head.total_frags, RK_F_TIMING, &load_stats_, &csv_stats_);
  // (every rank refuses alike; the message carries the first rank's number)
  if (rc == RK_ERR_RANGE && std::string(rk_multi_last_error(multi_)).find("Unexpected number of fragments") != std::string::npos)
    throw std::runtime_error("Unexpected number of fragments");  // :99, as the host route throws it
  if (rc != RK_OK) throw std::runtime_error(std::string("repkiller-b200: ") + rk_multi_last_error(multi_));
  count_ = load_stats_.n_loaded;
  device_parser_ = true;
  const auto t3 = clk::now();
  ms_read_ = std::chrono::duration<double, std::milli>(t1 - t0).count();
  ms_parse_ = csv_stats_.ms_upload + csv_stats_.ms_parse;  // the largest rank's device time of the upload and the parse
  ms_device_load_ = std::chrono::duration<double, std::milli>(t3 - t2).count();
}
