// Drop-in for the free functions of /root/reference/src/commonFunctions.h used on the grouping path.  Same
// names, argument meaning and error behaviour; the work is done by librk_b200.so.
#pragma once

#include <queue>
#include <string>
#include <utility>
#include <vector>

#include "FragmentsDatabase.h"
#include "SequenceOcupationList.h"
#include "structs.h"

void print_help();  // reference: commonFunctions.cpp:3-7
void init_args(const std::vector<std::string> &args, std::ifstream &multifrags, std::string &out_file_base_path,
               std::string &path_frags, std::queue<std::pair<double, double>> &params);  // :9-30

// The three grouping facades below may be called from several threads on one FragmentsDatabase, as the reference's
// thread pool calls its functions (repkiller.cpp:60-72): each call groups on a context of the database's pool
// (FragmentsDatabase::ContextPool) — frags_db.ctx() when it is free, else a view sharing its load (rk_create_view).
// reference: commonFunctions.cpp:41-80.  Fills efrags_groups (groups in creation order, members in processing
// order, pointers into frags_db.records()) and returns the number of groups.  Runs K3+K4 on the device.
size_t generate_fragment_groups(const FragmentsDatabase &frags_db, FGList &efrags_groups, const sequence_manager &seq_manager,
                                double len_pos_ratio, double pos_ratio);
// reference: commonFunctions.cpp:161-177; diag_func has frags_db.getA() entries, [0, getA()-2] are written.
void generate_diagonal_func(const FragmentsDatabase &fdb, size_t *diag_func);
// reference: commonFunctions.cpp:148-159.  A pure function of its arguments, like the reference's: any list of groups,
// any diag_func.  Per member the host gathers yStart and diag_func[xStart/10]; h and libstdc++'s std::sort order of
// every group are computed on the device (rk_sort_members, K5b) on a context of its own (GPU RK_DEVICE, default 0).
void sort_groups(FGList &fgl, const size_t *diag_func);
// One call for the three above (what the CLI uses: no intermediate host lists).  stats' host arrays belong to the
// context that grouped (over several GPUs: its rk_multi), valid until that context's next grouping.
FGList *group_and_sort(const FragmentsDatabase &frags_db, double len_ratio, double pos_ratio, rk_result *stats = nullptr);

// reference: commonFunctions.cpp:101-146 (the writer; byte-identical output)
void save_frags_from_group(std::ostream &out_file, FragsGroup &fg, uint64_t gid);
void save_frag_pair(std::ostream &out_file, uint64_t seq1_label, uint64_t seq2_label, const sequence_manager &seq_mngr,
                    const FGList &fgl);
void save_all_frag_pairs(const std::string &out_file_base_path, const sequence_manager &seq_manager, const FGList &fgl);
// The same file for the result of the last rk_group on frags_db.ctx() (single-threaded use), its lines formatted on the device (K6, rk_format_lines):
// no FGList, no per-line host formatting.  Over several GPUs (frags_db.multi()) the last rk_multi_group must have had
// RK_F_LINE_RECORDS; every GPU formats its own lines (rk_multi_format_lines).  Throws std::runtime_error when the path cannot be opened (like the above).
void save_device_text(const std::string &out_file_base_path, const sequence_manager &seq_manager, const FragmentsDatabase &frags_db,
                      float *ms_format = nullptr);
void free_groups(FGList *fgl);
