/* TEST INFRASTRUCTURE — NOT part of the product path.
 *
 * CPU restatement ("oracle") of the reference's fragment-grouping path, in plain C.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may use it, and only as the
 * checker.  Nothing under repkiller_b200/ links, imports or executes this.
 *
 * Pinning: the reference ships no golden vectors (SURVEY.md §4).  This restatement is pinned against the
 * reference itself: oracle/_ref/repkiller_ref (the unmodified reference sources + oracle/ref_driver.cpp)
 * on the fuzz classes and workloads of tests/golden/make_golden.py; see tests/test_oracle_golden.py.
 */
#ifndef RK_ORACLE_H
#define RK_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* struct FragFile under #pragma pack(1): /root/reference/src/structs.h:2,12-51 (109 bytes). */
#pragma pack(push, 1)
typedef struct {
  int64_t diag;
  uint64_t xStart, yStart, xEnd, yEnd, length, ident, score;
  float similarity;
  uint64_t seqX, seqY;
  int64_t block;
  char strand;
  unsigned char evalue[16];
} rko_frag;
#pragma pack(pop)

#define RKO_NONE 0xFFFFFFFFu

typedef struct {
  uint64_t n_kept;     /* fragments that are iterated (last X bucket dropped, FragmentsDatabase.h:29-31) */
  uint64_t n_groups;
  uint64_t vsize;      /* FragmentsDatabase.cpp:84 */
  /* arrays of n_kept entries, indexed by processing rank (A.2) */
  uint32_t *rank_fidx; /* file index of the fragment at this rank */
  uint32_t *xowner;    /* rank of the X-list entry that matched, or RKO_NONE */
  uint32_t *yowner;    /* rank of the Y-list entry that matched, or RKO_NONE (only queried when no X match) */
  uint32_t *parent;    /* xowner if any else yowner if any else RKO_NONE */
  uint32_t *gid;       /* group id = creation order (commonFunctions.cpp:72-74) */
  uint64_t *h;         /* sort_groups key |yStart - diag_func[xStart/10]| (commonFunctions.cpp:149-156) */
  /* arrays of n_kept entries in output order (groups by gid, members after sort_groups) */
  uint32_t *order;     /* file index */
  uint32_t *out_gid;
  uint8_t *repval;     /* commonFunctions.cpp:106-115 */
  float *identity;     /* (float)ident*100/(float)length, commonFunctions.cpp:103 */
  /* diag_func[vsize-1] (commonFunctions.cpp:161-177), only when requested */
  uint64_t *diag_func;
} rko_result;

/* readFragment (FragmentsDatabase.cpp:17-50): 1 = accepted. */
int rko_parse_row(const char *line, size_t len, rko_frag *out);

/* FragmentsDatabase ctor (FragmentsDatabase.cpp:54-101), without the bucket array: records in file order.
 * Returns 0, or -1 cannot open, -2 more accepted rows than "Total fragments" (the reference throws). */
int rko_load_csv(const char *path, rko_frag **recs, uint64_t *n, uint64_t *lx1, uint64_t *ly1, char **header);

/* generate_fragment_groups + generate_diagonal_func + sort_groups (commonFunctions.cpp:41-80,148-177).
 * lx1/ly1 are the loaded lengths (header value + 1).  want_diag: also fill diag_func.
 * Returns 0, or -3 when a fragment has xStart/10 >= vsize (out-of-bounds write in the reference). */
int rko_group(const rko_frag *recs, uint64_t n, uint64_t lx1, uint64_t ly1, double len_ratio, double pos_ratio,
              int want_diag, rko_result *out);
void rko_result_free(rko_result *r);

/* save_all_frag_pairs (commonFunctions.cpp:101-146). Returns 0 or -1. */
int rko_write_output(const char *path, const char *header, const rko_frag *recs, const rko_result *r);

/* Input-CSV writer for generated workloads (tooling, no reference counterpart). */
int rko_write_input_csv(const char *path, const rko_frag *recs, uint64_t n, uint64_t lx_header, uint64_t ly_header);

/* libstdc++ std::sort order of idx[0..n) under comp(a,b) = h[a] < h[b] (sort_groups, commonFunctions.cpp:158) */
void rko_std_sort_by_key(uint32_t *idx, uint64_t n, const uint64_t *h);

/* One SequenceOcupationList (SequenceOcupationList.cpp:3-96) with a 64-bit tag per entry in place of the FragsGroup
 * pointer: the checker of rk_sol_*.  insert returns -1 when center/100 lies beyond the lists, -2 when memory runs out
 * (nothing inserted); get stores the tag of the winner (0: none) and returns -2 when a probe would read beyond the
 * lists (the reference reads out of bounds). */
typedef struct rko_sol rko_sol;
rko_sol *rko_sol_create(double len_ratio, double pos_ratio, uint64_t seq_size);
int rko_sol_insert(rko_sol *s, uint64_t center, uint64_t length, uint64_t tag);
int rko_sol_get(const rko_sol *s, uint64_t center, uint64_t length, uint64_t *tag);
void rko_sol_destroy(rko_sol *s);

void rko_free(void *p);

#ifdef __cplusplus
}
#endif
#endif
