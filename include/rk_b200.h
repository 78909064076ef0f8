/* rk_b200.h — C ABI of the B200-native repkiller grouping path (librk_b200.so).
 *
 * The reference has no FFI layer: its boundary for this path is the C++ surface called from
 * execWithParams/main (/root/reference/src/repkiller.cpp:52,83-96).  Each entry point below names the
 * reference interface it replaces.  Plain pointers and sizes only; no exceptions cross this boundary; every
 * function returns an rk_status (0 = ok, negative = error, message via rk_last_error).  There is no CPU
 * fallback: without a CUDA device rk_create fails.
 */
#ifndef RK_B200_H
#define RK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RK_FRAG_BYTES 109u /* sizeof(struct FragFile) under #pragma pack(1), src/structs.h:2,12-51 */
#define RK_NONE 0xFFFFFFFFu

typedef enum {
  RK_OK = 0,
  RK_ERR_CUDA = -1,     /* a CUDA call failed (rk_last_error has the CUDA message) */
  RK_ERR_ARG = -2,      /* bad argument (null, misaligned device pointer, non-positive ratio, ...) */
  RK_ERR_RANGE = -3,    /* input the reference itself cannot process: xStart/10 >= vsize (out-of-bounds write at
                           src/FragmentsDatabase.cpp:96-97), a center outside the occupation lists
                           (src/SequenceOcupationList.cpp:16-18), or a coordinate >= 2^31 */
  RK_ERR_STATE = -4,    /* call order: rk_group before rk_load_aos, ... */
  RK_ERR_NOMEM = -5,    /* a device or pinned host allocation failed: the last-error text names the call and the byte
                           count, and the CUDA error is cleared, so the object stays usable; or a rank of a partitioned
                           comparison is asked for more records than its capacity */
  RK_ERR_INTERNAL = -6  /* an internal invariant failed (bounded spin expired, worklist overflow) */
} rk_status;

/* rk_group / rk_load_aos flags */
#define RK_F_HOST_RESULT 1u /* copy order/gid/repval/identity to library-owned pinned host arrays */
#define RK_F_NO_SORT 2u     /* stop after generate_fragment_groups: members stay in push_back (rank) order */
#define RK_F_TIMING 4u      /* record per-stage CUDA-event times into rk_result / rk_load_stats */
#define RK_F_LINE_RECORDS 8u /* rk_dist_group / rk_multi_group: also bring every output line's record to the rank that holds
                                the line, for rk_dist_format_lines / rk_dist_group_statistics (rk_group ignores it) */

enum { /* stage indices of ms_stage[] */
  RK_ST_H2D = 0,     /* host -> device copy of the records or of rk_load_csv's text (0 for a device pointer) */
  RK_ST_DECODE,      /* K1  AoS -> SoA decode + validity + link bits                                  */
  RK_ST_RANKSORT,    /* K2a stable LSD radix sort by xStart/10                                        */
  RK_ST_KEYS,        /* K2  rank-order SoA gather + super-bucket keys                                  */
  RK_ST_XSORT,       /* K2b stable sort by (strand class, X super-bucket)                              */
  RK_ST_YSORT,       /* K2c stable sort by (strand class, Y super-bucket)                              */
  RK_ST_XMATCH,      /* K3  X pass of generate_fragment_groups                                         */
  RK_ST_YMATCH,      /* K3  Y pass                                                                     */
  RK_ST_FOREST,      /* K4  roots + group ids                                                          */
  RK_ST_HKEY,        /* K5a generate_diagonal_func evaluated per fragment + sort key                   */
  RK_ST_GSORT,       /* K5b stable sort by gid + per-group std::sort order                             */
  RK_ST_FINAL,       /* K5c output order, repval, identity                                             */
  RK_ST_D2H,         /* device -> host copy of the result (RK_F_HOST_RESULT)                           */
  RK_NSTAGES
};

typedef struct rk_ctx rk_ctx;

typedef struct {
  uint64_t n_loaded;  /* records handed to rk_load_aos */
  uint64_t n_kept;    /* records the reference iterates: xStart/10 < vsize-1 (FragmentsDatabase.h:29-31) */
  uint64_t vsize;     /* FragmentsDatabase::getA(), src/FragmentsDatabase.cpp:84 */
  float ms_stage[RK_NSTAGES];
  float ms_device;    /* first kernel to last kernel on the context's stream */
  uint64_t n_launches; /* kernels launched by this call */
} rk_load_stats;

typedef struct {
  uint64_t n_kept;
  uint64_t n_groups;  /* return value of generate_fragment_groups, src/commonFunctions.cpp:79 */
  /* n_kept entries each, in output order: groups by id (creation order), members as sort_groups leaves them.
   * Host pointers (pinned, owned by the context, valid until the next rk_group/rk_destroy) when
   * RK_F_HOST_RESULT was given, else NULL. */
  const uint32_t *order;    /* index of the record in the loaded array (file order) */
  const uint32_t *gid;      /* the `block` column the writer prints, src/commonFunctions.cpp:102,127 */
  const uint8_t *repval;    /* 0 singleton, 1 first of a group, 2 rest: src/commonFunctions.cpp:106-115 */
  const float *identity;    /* (float)ident*100/(float)length, src/commonFunctions.cpp:103 */
  /* the same four arrays on the device (always valid until the next rk_group/rk_destroy) */
  const uint32_t *d_order;
  const uint32_t *d_gid;
  const uint8_t *d_repval;
  const float *d_identity;
  float ms_stage[RK_NSTAGES];
  float ms_device;
  uint64_t n_launches; /* kernels launched by this call */
} rk_result;

/* One context per GPU and per concurrent grouping (mirrors one FragmentsDatabase + the per-call
 * SequenceOcupationLists, src/repkiller.cpp:52, src/commonFunctions.cpp:45-48); concurrent groupings of one loaded
 * database share the load through views (rk_create_view).  Returns NULL on failure; rk_create_error() then has the
 * reason. */
rk_ctx *rk_create(int device);
const char *rk_create_error(void);
/* Releases the context's own stream, workspace and buffers.  Its database goes with the last context that uses it: a
 * base destroyed while views of it are live leaves the load to them. */
void rk_destroy(rk_ctx *ctx);
const char *rk_last_error(const rk_ctx *ctx);

/* A second grouping context over the database loaded into `base`: same device, its own stream, events, counters, grouping
 * workspace and result/text/statistics buffers; the loaded records, processing order, bucket sorts and h are shared
 * read-only.  rk_group / rk_sort_groups / rk_format_lines / rk_group_statistics / rk_diagonal_func / rk_debug_fetch /
 * rk_set_stream / rk_profile_* work on it as on base, and give bit-identical results for the same ratio pair.  Calls on
 * different contexts that share a database may run concurrently from different host threads (calls on ONE context are
 * still serialised by the caller).  NULL on failure (rk_create_error).
 *  - base must hold a successful single-GPU load (rk_load_aos / rk_load_packed); a view of a view shares the same
 *    database.  Contexts of a partitioned comparison (rk_dist_init, rk_multi_ctx) are refused.
 *  - rk_create_view only reads the load of base, so it may run while another thread groups on base; not while base
 *    loads or is destroyed.
 *  - The database is reference-counted: it is freed with the last of base and its views.
 *  - rk_load_* on a view, rk_load_* on a context with live views (the message names how many; nothing changes) and
 *    rk_dist_init on either return RK_ERR_STATE.
 *  - The grouping workspace and the pinned result arrays of a view are allocated here, sized from the load; later calls
 *    allocate only the grow-only text, statistics and diagonal-table buffers on first use.
 *  - After rk_load_packed with rest4, every context's first grouping waits for the side copy of that array. */
rk_ctx *rk_create_view(rk_ctx *base);

/* Use `cuda_stream` (a cudaStream_t) for all work of this context instead of its own stream. */
int rk_set_stream(rk_ctx *ctx, void *cuda_stream);

/* Replaces FragmentsDatabase::FragmentsDatabase after text parsing (src/FragmentsDatabase.cpp:84-100):
 * takes n records in the struct FragFile layout, file order, from host or device memory (a device pointer
 * must be 16-byte aligned), and builds the processing order (the xStart/10 bucket array) and the
 * occupation-list buckets on the device.  seqx_len/seqy_len are the LOADED lengths (header value + 1,
 * src/FragmentsDatabase.cpp:62,65).  Synchronous. */
int rk_load_aos(rk_ctx *ctx, const void *frags, uint64_t n, uint64_t seqx_len, uint64_t seqy_len, unsigned flags,
                rk_load_stats *stats);

/* The same as rk_load_aos from the compact form a CSV parser can fill directly (33 B per fragment instead of 109 B over
 * PCIe): key4 = {xStart, yStart, length, ident} as four uint32 per fragment, strand = one byte per fragment, rest4 =
 * {xEnd, yEnd, score, similarity bits} as four uint32 per fragment (only rk_format_lines reads it; NULL when the caller
 * writes the output itself).  All host or all device memory; every value must fit in 32 bits (the reference's uint64
 * fields: use rk_load_aos otherwise).  Synchronous. */
int rk_load_packed(rk_ctx *ctx, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n, uint64_t seqx_len,
                   uint64_t seqy_len, unsigned flags, rk_load_stats *stats);

/* Replaces FragmentsDatabase::FragmentsDatabase from the text on (src/FragmentsDatabase.cpp:91-100): takes the body of a
 * GECKO CSV (the bytes after its 16 header lines) in host memory of any kind or in device memory, splits it into rows on
 * '\n' as std::getline does, applies readFragment's rules (src/FragmentsDatabase.cpp:17-50) to every row on the device, and
 * loads the accepted rows in file order: the database rk_load_packed (or rk_load_aos, when a value needs 33 or more bits)
 * builds from the host parser's records.  A row whose tokens leave the plain grammar (digits; digits[.digits] for the
 * similarity: signs, blanks, exponents, 19+ digits, a float on a rounding midpoint, ...) is parsed by the host parser
 * inside this call; only such rows' bytes come back from a device body.  seqx_len/seqy_len are the LOADED lengths
 * (header value + 1); total_frags is the header's "Total fragments": more accepted rows than that return RK_ERR_RANGE
 * ("Unexpected number of fragments", src/FragmentsDatabase.cpp:99) and leave nothing loaded.  The parsed arrays belong
 * to the context's database, so body may be freed when the call returns.  A body larger than the device's free memory
 * returns RK_ERR_NOMEM.  ms_stage[RK_ST_H2D] of stats is the text upload.  csv may be NULL.  Synchronous. */
typedef struct {
  uint64_t n_rows;       /* rows of the body, the empty one after a final '\n' included */
  uint64_t n_accepted;   /* records loaded (= rk_load_stats.n_loaded) */
  uint64_t n_host_rows;  /* rows outside the plain grammar, decided by the host parser */
  int wide;              /* 1: a value needs 33 or more bits; the records were loaded as 109-byte records */
  float ms_upload;       /* host -> device copy of the text (0 for a device body) */
  float ms_parse;        /* row split, parse, host rows and compaction on the device */
} rk_csv_stats;
int rk_load_csv(rk_ctx *ctx, const char *body, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags,
                unsigned flags, rk_load_stats *stats, rk_csv_stats *csv);

/* Replaces generate_fragment_groups + generate_diagonal_func + sort_groups
 * (src/commonFunctions.cpp:41-80,161-177,148-159; call sites src/repkiller.cpp:84-91) for one
 * (len_ratio, pos_ratio) pair.  Both ratios must be > 0 (src/commonFunctions.cpp:26-27).  Synchronous. */
int rk_group(rk_ctx *ctx, double len_ratio, double pos_ratio, unsigned flags, rk_result *out);

/* Replaces sort_groups (src/commonFunctions.cpp:148-159) when it is called as a separate step: after an
 * rk_group with RK_F_NO_SORT, orders the members of every group on the device and returns the result again. */
int rk_sort_groups(rk_ctx *ctx, unsigned flags, rk_result *out);

/* Per-group statistics of the last rk_group / rk_sort_groups (not part of the reference's output file; its groups are the
 * FragsGroups of src/commonFunctions.cpp:56-76 in creation order): one entry per group id.  x/y span = [min start,
 * max(start + length)); mean_identity = mean of the identity column; multiplicity = sum of lengths / X span (how many
 * copies cover the span).  Integers are exact; the two doubles agree with a sequential evaluation to ~1e-15 relative.
 * stats: pinned host array owned by the context (valid until the next call), d_stats: the same on the device. */
typedef struct {
  uint32_t count, x_lo, x_hi, y_lo, y_hi, first_line;
  double mean_identity, multiplicity;
} rk_group_stats;
int rk_group_statistics(rk_ctx *ctx, unsigned flags, const rk_group_stats **stats, const rk_group_stats **d_stats, uint64_t *n_groups);

/* Replaces sort_groups (src/commonFunctions.cpp:148-159) as the PURE function the reference has: perm[j] = index (into
 * the member arrays handed in) of the member that std::sort leaves at position j, for m members given group by group
 * (gid nondecreasing), y[j] = yStart and d[j] = diag_func[xStart/10] of member j (host arrays).  Nothing of an earlier
 * rk_group is used: any list, any diag_func.  Synchronous. */
int rk_sort_members(rk_ctx *ctx, uint64_t m, const uint32_t *gid, const uint64_t *y, const uint64_t *d, uint32_t *perm);

/* Replaces SequenceOcupationList (src/SequenceOcupationList.h:13-33) for code that drives the occupation lists call by call
 * (the reference's generate_fragment_groups body, src/commonFunctions.cpp:41-80, runs unchanged on top of it): the lists
 * live in device memory, insert() is queued and applied in order before the next query, get_associated_group() is one
 * kernel that scans the probed buckets newest-first with the reference's strict `>` on the binary64 deviation.  A tag is
 * the caller's group handle (the facade passes the FragsGroup pointer); 0 = no group.  Whole databases should use
 * rk_group, which evaluates all queries of an axis in parallel. */
typedef struct rk_sol rk_sol;
rk_sol *rk_sol_create(int device, double len_ratio, double pos_ratio, uint64_t seq_size);
void rk_sol_destroy(rk_sol *s);
int rk_sol_insert(rk_sol *s, uint64_t center, uint64_t length, uint64_t tag);
int rk_sol_get_associated(rk_sol *s, uint64_t center, uint64_t length, uint64_t *tag);
const char *rk_sol_last_error(const rk_sol *s);

/* Replaces the formatting half of save_frags_from_group / store_frag (src/commonFunctions.cpp:101-115) for the
 * result of the last rk_group / rk_sort_groups: the text of output lines first_line .. first_line+n_lines-1
 *   Frag,xStart,yStart,xEnd,yEnd,strand,gid,length,score,ident,similarity,identity,0,repval\n
 * byte for byte what the reference writes (integers as ostream << uint64_t, the two floats as printf("%g")),
 * formatted on the device from the loaded records.  At most RK_FORMAT_MAX_LINES lines per call; the caller writes
 * the 16 header lines itself (sequence_manager::write_header) and appends the chunks.  text: pinned host memory owned
 * by the context, valid until the next-but-one rk_format_lines call (two buffers alternate, so that a chunk can be
 * written to disk while the next one is formatted) or rk_destroy.  The records must still be where rk_load_aos
 * found them when they were given as a DEVICE pointer (host records are kept in the context).  Synchronous. */
#define RK_FORMAT_MAX_LINES 8000000ull
typedef struct {
  const char *text;
  uint64_t n_bytes;
  float ms_device; /* formatting kernels + device -> host copy */
} rk_text;
int rk_format_lines(rk_ctx *ctx, uint64_t first_line, uint64_t n_lines, rk_text *out);

/* Pinned host memory for record arrays handed to rk_load_aos (full-speed H2D); NULL on failure. */
void *rk_host_alloc(size_t bytes);
void rk_host_free(void *p);

/* Replaces generate_diagonal_func (src/commonFunctions.cpp:161-177): fills diag_func[0 .. vsize-2] (host
 * memory, vsize = FragmentsDatabase::getA()) including the carry-forward over empty buckets. */
int rk_diagonal_func(rk_ctx *ctx, uint64_t *diag_func);

/* Test/diagnostic access to intermediate device arrays of the last load/group, copied to `host` (capacity
 * `bytes`).  Names: "rank_fidx", "parent", "gid_rank", "hkey", and the loaded compact arrays of a load that has them
 * (rk_load_packed, rk_load_csv without wide values): "key4" (n_loaded x 4 uint32), "strand" (n_loaded bytes), "rest4"
 * (n_loaded x 4 uint32).  Returns the number of bytes the array has, or a negative rk_status. */
int64_t rk_debug_fetch(rk_ctx *ctx, const char *name, void *host, uint64_t bytes);

/* Per-kernel device time: when enabled, every kernel launch of later calls on this context is bracketed by a
 * CUDA-event pair on the context's stream.  rk_profile_read fills up to `cap` entries (one per kernel that
 * ran; consecutive launches of the 3-kernel scan are one entry) and returns how many; reset != 0 clears. */
typedef struct {
  const char *name;
  uint64_t launches;
  double ms_total;
  uint64_t units; /* fragments (or sort elements, buckets) the launches processed in total */
} rk_kernel_time;
int rk_profile_enable(rk_ctx *ctx, int on);
int rk_profile_read(rk_ctx *ctx, rk_kernel_time *out, int cap, int reset);

/* Stand-alone stable LSD radix sort of (u32 key, u32 value) pairs on the device (kernel K2), exported for
 * tests.  All pointers are device pointers; values_in may be NULL (values = 0..n-1).
 * `work` needs rk_sort_pairs_work_bytes(n) bytes.  The result is in keys_out/values_out. */
uint64_t rk_sort_pairs_work_bytes(uint64_t n);
int rk_sort_pairs(rk_ctx *ctx, const uint32_t *keys_in, const uint32_t *values_in, uint32_t *keys_out,
                  uint32_t *values_out, uint32_t *keys_tmp, uint32_t *values_tmp, uint64_t n, int key_bits, void *work);

/* ---- one comparison partitioned over several GPUs (SURVEY.md section 8e) ---------------------------------------------
 * The reference is one process on one host (src/repkiller.cpp); these entry points run the same
 * FragmentsDatabase -> generate_fragment_groups -> generate_diagonal_func -> sort_groups sequence on ONE fragment file
 * whose records are spread over the GPUs of a box, with output bit-identical to rk_load_aos + rk_group on one GPU.
 * Fragments are range-partitioned by xStart/10 (processing order), the X pass runs at home with a halo of the fragments
 * whose center crosses a cut, the Y pass on the owners of the Y ranges, group ids come from per-GPU root counts plus parent
 * chains followed through peer memory (NVLink), and rank r ends up with the r-th range of output lines.
 *
 * (a) one process per GPU (torchrun, MPI): rank 0 calls rk_dist_unique_id and broadcasts the RK_DIST_ID_BYTES bytes; every rank
 *     calls rk_dist_init, rk_dist_export, all-gathers the RK_DIST_BLOB_BYTES blobs (any transport the application has),
 *     rk_dist_import, then rk_dist_load_aos / rk_dist_group.  These calls are collective: every rank must make them.
 * (b) one process, several GPUs: rk_create_multi and rk_multi_*; the library runs one host thread per GPU. */
#define RK_DIST_ID_BYTES 128u
#define RK_DIST_BLOB_BYTES 128u
typedef struct {
  int rank, world;
  uint64_t total_loaded;  /* records of the whole file */
  uint64_t total_kept;    /* fragments the reference iterates, all ranks */
  uint64_t total_groups;
  uint64_t line_offset;   /* index of this rank's first output line in the whole output */
  uint64_t n_lines;       /* output lines this rank holds (== rk_result.n_kept of rk_dist_group) */
  uint64_t rank_offset;   /* first processing rank this GPU owns */
  uint64_t n_ranked;      /* fragments this GPU owns in processing order */
  uint64_t n_halo_in, n_halo_out; /* X-pass halo fragments received from lower / sent to higher GPUs */
  uint64_t n_y;           /* fragments this GPU owns in the Y pass */
  uint64_t bytes_sent;    /* payload this rank sent to other ranks during the call */
} rk_dist_info;
int rk_dist_unique_id(void *id128);
/* cap_per_rank: rows of workspace per GPU, the same on every rank; 1.5 x the fragments per GPU + 65536 is what
 * rk_create_multi and bench.py use.  It bounds what ONE rank may own at any stage: the records of its xStart/10 range, the
 * rows of its Y range, and the output lines of its group-id range (a group is never split: a comparison whose largest
 * group alone exceeds the capacity needs a larger one).  A stage that would exceed it fails on every rank with
 * RK_ERR_NOMEM and a message naming the rank and the count; nothing is truncated. */
int rk_dist_init(rk_ctx *ctx, int rank, int nranks, const void *id128, uint64_t cap_per_rank);
int rk_dist_export(rk_ctx *ctx, void *blob);
int rk_dist_import(rk_ctx *ctx, const void *blobs /* nranks x RK_DIST_BLOB_BYTES, in rank order */);
/* frags: this rank's contiguous slice of the file (host or 16-byte aligned device memory), file_offset = index of its first
 * record; slices in rank order make up the file.  Replaces FragmentsDatabase::FragmentsDatabase like rk_load_aos. */
int rk_dist_load_aos(rk_ctx *ctx, const void *frags, uint64_t n_local, uint64_t file_offset, uint64_t seqx_len, uint64_t seqy_len,
                     unsigned flags, rk_load_stats *stats);
/* rk_load_csv over the ranks.  slice: this rank's part of a GECKO CSV body (the bytes after the 16 header lines), in host
 * memory of any kind or in device memory; the slices in rank order make up the body.  Every non-empty slice before the
 * last non-empty one must end with '\n', so that every cut falls at the start of a row; a slice may be empty.  A row
 * belongs to the rank whose slice holds its first byte; the empty row after a final '\n' to the last rank.  The library
 * counts the rows of every rank and gives each record its index among the accepted rows of the whole body (no file
 * offset to pass).  Groups, text and statistics are bit-identical to rk_load_csv + rk_group on one GPU and to
 * rk_dist_load_aos on the same records.  The parsed rows belong to the rank (compact rows, or 109-byte records when a
 * value of its slice needs 33 or more bits), so the slice may be freed when the call returns.  csv: this rank's counts
 * (n_rows: the rows that start in its slice; their sum over the ranks is rk_load_csv's n_rows).  stats as
 * rk_dist_load_aos reports them, ms_stage[RK_ST_H2D] = the text upload.  Refusals reach every rank with the same code
 * and message, and leave nothing loaded: a slice that does not end a row (RK_ERR_ARG), more accepted rows over the ranks
 * than total_frags (RK_ERR_RANGE, "Unexpected number of fragments"), 2^32-16 or more of them (RK_ERR_ARG), a rank with
 * more than its capacity (RK_ERR_NOMEM), and a rank whose own parse failed (its text allocation, more than 2^32-16 rows
 * in its slice).  Collective. */
int rk_dist_load_csv(rk_ctx *ctx, const char *slice, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags,
                     unsigned flags, rk_load_stats *stats, rk_csv_stats *csv);
/* rk_load_packed over the ranks: this rank's contiguous slice of the file in the compact form of rk_load_packed (key4,
 * strand, rest4 or NULL; 33 B per fragment instead of 109 B), n_local fragments, file_offset = index of its first one, as
 * rk_dist_load_aos takes them.  Groups, text and statistics are bit-identical to rk_dist_load_aos on the same records.
 *  - Host arrays, pinned or pageable, are copied into the rank's buffers (rest4 beside the load's kernels), and every copy
 *    has finished when the call returns: the caller may overwrite or free all three arrays then.
 *  - Device arrays must be on the rank's device, key4 and rest4 16-byte aligned; they are used in place and must stay where
 *    they are for rk_dist_group with RK_F_LINE_RECORDS, as device records of rk_dist_load_aos must.
 *  - rest4 == NULL: grouping works; a later rk_dist_group with RK_F_LINE_RECORDS returns RK_ERR_ARG on every rank when any
 *    rank loaded fragments without rest4.
 *  - Refusals reach every rank with the same code and message (prefixed by the rank that refused) and leave nothing
 *    loaded: a null key4 or strand with n_local > 0, arrays partly in host and partly in device memory, a misaligned device
 *    array or one on another device (RK_ERR_ARG), n_local over the capacity or a failed staging allocation
 *    (RK_ERR_NOMEM), a sequence length of 2^32 or more (RK_ERR_RANGE), 2^32-16 or more records (RK_ERR_ARG); then the
 *    refusals of rk_dist_load_aos (a coordinate beyond the sequence: RK_ERR_RANGE).  Collective. */
int rk_dist_load_packed(rk_ctx *ctx, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n_local,
                        uint64_t file_offset, uint64_t seqx_len, uint64_t seqy_len, unsigned flags, rk_load_stats *stats);
/* out: THIS RANK's range of output lines (order = file indices of the whole file, gid = global group ids); n_groups is
 * the global count.  info may be NULL. */
int rk_dist_group(rk_ctx *ctx, double len_ratio, double pos_ratio, unsigned flags, rk_result *out, rk_dist_info *info);
/* After an rk_dist_group with RK_F_LINE_RECORDS: the output of THIS rank, with no collective step (the group call brought
 * the record of every line to the rank that holds the line).  Both return RK_ERR_STATE after a group without the flag.
 * The records must still be where rk_dist_load_aos found them when they were given as a DEVICE pointer.  rk_dist_group refuses
 * RK_F_LINE_RECORDS with RK_ERR_ARG (on every rank) when the ranks' slices, by their file_offset, overlap or are out of rank order.
 * rk_dist_format_lines: the text of local lines first_line .. first_line+n_lines-1 (0 .. rk_dist_info.n_lines), byte for byte
 *   what rk_format_lines writes for the same lines on one GPU; the same limits and the same two alternating buffers.
 * rk_dist_group_statistics: rk_group_statistics of the groups of this rank, first_gid .. first_gid+n_groups-1 (a group is
 *   never split over ranks; first_line is the global line index). */
int rk_dist_format_lines(rk_ctx *ctx, uint64_t first_line, uint64_t n_lines, rk_text *out);
int rk_dist_group_statistics(rk_ctx *ctx, unsigned flags, const rk_group_stats **stats, const rk_group_stats **d_stats,
                             uint64_t *first_gid, uint64_t *n_groups);
/* Views of a partitioned comparison: a second grouping context per rank over the partition database the ranks loaded,
 * so that several ratio pairs group one load at the same time.  A rank's view shares its load read-only (the records,
 * the processing order and the bucket sorts of both passes) and has its own stream, transport, grouping workspace
 * (mapped into the peers' views) and result, text and statistics buffers.
 *  - rk_dist_group / rk_dist_format_lines / rk_dist_group_statistics / rk_set_stream work on a view as on its base and
 *    give bit-identical results for the same pair.  Calls on different contexts of one partitioned load may run at the
 *    same time from different host threads (on one context they are still serialised by the caller).
 *  - The partition database is reference-counted per rank: it is freed with the last of the base and its views.
 *  - rk_dist_load_* (rk_multi_load_*) on a view, or on a base with live views (the message names how many; nothing
 *    changes), and rk_dist_init on either return RK_ERR_STATE.  rk_create_view refuses rank contexts and views alike.
 *  - A view of a view shares the same database.
 * rk_dist_create_view: the process-per-GPU form, collective like rk_dist_init.  Rank 0 calls rk_dist_unique_id and
 * broadcasts the id; every rank calls rk_dist_create_view on its base, then rk_dist_export and rk_dist_import on the
 * view.  The view has its own NCCL communicator.  NULL (rk_create_error) when base holds no partitioned load, which
 * every rank sees alike, or when this rank's workspace cannot be allocated: the other ranks must then destroy theirs. */
rk_ctx *rk_dist_create_view(rk_ctx *base, const void *id128);

typedef struct rk_multi rk_multi;
/* One context per listed device.  The ranks push their rows into each other's device memory.  Distinct devices exchange
 * the small tables and meet at barriers over NCCL; a device listed twice (tests on a one-GPU box), or NCCL failing to
 * start, makes the ranks do that through host memory.  NULL on failure (rk_create_error). */
rk_multi *rk_create_multi(const int *devices, int ndev);
void rk_destroy_multi(rk_multi *m);
const char *rk_multi_last_error(const rk_multi *m);
int rk_multi_ranks(const rk_multi *m);
rk_ctx *rk_multi_ctx(rk_multi *m, int rank);
const char *rk_multi_transport(const rk_multi *m); /* "nccl" or "local" */
/* frags: the whole file in HOST memory; the ranks take consecutive slices. */
int rk_multi_load_aos(rk_multi *m, const void *frags, uint64_t n, uint64_t seqx_len, uint64_t seqy_len, unsigned flags,
                      rk_load_stats *stats);
/* body: a whole GECKO CSV body in HOST memory (a device pointer returns RK_ERR_ARG).  Cut r of N is one byte past the first
 * '\n' at or after byte bytes*r/N (the end of the body when there is none), and each rank parses its slice as
 * rk_dist_load_csv does.  The capacity per rank is sized after the rows are counted: 1.5 x the most rows one rank may
 * load + 65536.  csv: sums over the ranks; wide = 1 when any rank is wide; ms_upload / ms_parse = the largest of the
 * ranks'.  The text is copied by at most max(N, T) host threads in all, T = the copy threads of one rk_load_csv
 * (at most 4): each rank copies on its own thread, and helpers only while the ranks are fewer than T. */
int rk_multi_load_csv(rk_multi *m, const char *body, uint64_t bytes, uint64_t seqx_len, uint64_t seqy_len, uint64_t total_frags,
                      unsigned flags, rk_load_stats *stats, rk_csv_stats *csv);
/* key4, strand, rest4 (or NULL): the whole file in the compact form of rk_load_packed, in HOST memory (a device array
 * returns RK_ERR_ARG); the ranks take the slices of rk_multi_load_aos, and the capacity per rank is sized as there, so
 * rk_multi_info reports the same partition for both loads.  Every rank loads its slice as rk_dist_load_packed does; the
 * arrays may be freed when the call returns.  ms_stage[RK_ST_H2D] of stats = the largest of the ranks' copies. */
int rk_multi_load_packed(rk_multi *m, const uint32_t *key4, const uint8_t *strand, const uint32_t *rest4, uint64_t n, uint64_t seqx_len,
                         uint64_t seqy_len, unsigned flags, rk_load_stats *stats);
/* out: the whole result in pinned host memory owned by m (device pointers are NULL), valid until the next call. */
int rk_multi_group(rk_multi *m, double len_ratio, double pos_ratio, unsigned flags, rk_result *out);
int rk_multi_info(const rk_multi *m, int rank, rk_dist_info *info);
/* After an rk_multi_group with RK_F_LINE_RECORDS, as rk_format_lines / rk_group_statistics on one GPU:
 * rk_multi_format_lines: GLOBAL lines first_line .. first_line+n_lines-1; every rank formats its part on its GPU, the parts
 *   land in one pinned buffer owned by m in rank order (two buffers alternate, as in rk_format_lines).
 * rk_multi_group_statistics: all groups in gid order, in host memory owned by m (valid until the next call). */
int rk_multi_format_lines(rk_multi *m, uint64_t first_line, uint64_t n_lines, rk_text *out);
int rk_multi_group_statistics(rk_multi *m, const rk_group_stats **stats, uint64_t *n_groups);
/* A view of base's partitioned load (see rk_dist_create_view for what a view shares and the rules): the same devices,
 * one view context per rank, mapped into each other, with a new NCCL communicator over the devices when base uses NCCL
 * and its own host-memory group otherwise.  rk_multi_group, rk_multi_format_lines, rk_multi_group_statistics and
 * rk_multi_info work on it as on base, with its own result buffers; rk_multi_ctx gives its rank contexts.  Destroy it
 * with rk_destroy_multi, before or after base.  NULL (rk_create_error) before a successful load of base, or when an
 * allocation fails. */
rk_multi *rk_multi_create_view(rk_multi *base);

/* Tooling: records start .. start+count of the synthetic workload of repkiller_b200/gen.py, generated on the device
 * (lx, ly are the header values, i.e. loaded length - 1). */
int rk_gen_workload(rk_ctx *ctx, uint64_t seed, uint64_t lx, uint64_t ly, double p_rep, uint64_t families, uint64_t ax, uint64_t ay,
                    uint64_t tandem_every, uint64_t start, uint64_t count, void *out_device);

const char *rk_version(void);

#ifdef __cplusplus
}
#endif
#endif
