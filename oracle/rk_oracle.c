/* TEST INFRASTRUCTURE — NOT part of the product path.  See rk_oracle.h.
 *
 * A sequential, line-for-line restatement of the reference's grouping path in plain C.  Every function
 * cites the reference lines it follows (paths relative to /root/reference).  Data structures are index
 * based (no STL), the arithmetic and the visiting orders are the reference's.
 */
#define _GNU_SOURCE
#include "rk_oracle.h"

#include <errno.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

void rko_free(void *p) { free(p); }

/* ------------------------------------------------------------------------------------------------
 * readFragment — src/FragmentsDatabase.cpp:17-50
 * 14 x getline(s, buf, ','): a token ends at ',' or at end of line.  When the stream is already at EOF the
 * extraction fails and `buf` keeps the previous token (short rows are padded with their last field);
 * an empty token rejects the row (:25).  A trailing ',' yields one empty token (rejected).
 * ---------------------------------------------------------------------------------------------- */
int rko_parse_row(const char *line, size_t len, rko_frag *out) {
  char tok[14][64];
  size_t pos = 0;
  int at_eof = 0;       /* eofbit of the istringstream */
  char buf[64] = "";
  size_t buflen = 0;
  for (int i = 0; i < 14; ++i) {
    if (!at_eof) {
      /* sentry ok: buf is erased, characters are extracted up to ',' or end of input */
      size_t s = pos;
      while (pos < len && line[pos] != ',') ++pos;
      buflen = pos - s;
      if (buflen > 63) {
        /* longer than any numeric field the reference can parse; keep the head, atoll/stof semantics are
         * unaffected for the fuzz classes (never generated) */
        buflen = 63;
      }
      memcpy(buf, line + s, buflen);
      buf[buflen] = 0;
      if (pos < len) ++pos; /* consume the delimiter */
      else at_eof = 1;      /* hit end of input while extracting */
    }
    if (buflen == 0) return 0; /* :25 */
    memcpy(tok[i], buf, buflen + 1);
  }
  if (strcmp(tok[0], "Frag") != 0) return 0; /* :29 */
  out->xStart = (uint64_t)atoll(tok[1]);
  out->yStart = (uint64_t)atoll(tok[2]);
  out->diag = (int64_t)out->xStart - (int64_t)out->yStart;
  out->xEnd = (uint64_t)atoll(tok[3]);
  out->yEnd = (uint64_t)atoll(tok[4]);
  out->strand = tok[5][0];
  out->block = atoll(tok[6]);
  out->length = (uint64_t)atoll(tok[7]);
  out->score = (uint64_t)atoll(tok[8]);
  /* std::stof (:39-40): throws (row rejected, :46-48) when nothing converts or on ERANGE */
  char *endp = NULL;
  errno = 0;
  float sim = strtof(tok[10], &endp);
  if (endp == tok[10] || errno == ERANGE) return 0;
  out->ident = (uint64_t)sim;
  out->similarity = sim;
  out->seqX = 0;
  out->seqY = 1;
  memset(out->evalue, 0, sizeof out->evalue);
  return 1;
}

/* value after the first ':' of a header line, atoll — src/FragmentsDatabase.cpp:62,65,72 */
static long long header_value(const char *line, size_t len) {
  size_t i = 0;
  while (i < len && line[i] != ':') ++i;
  size_t s = (i < len) ? i + 1 : 0; /* find()==npos -> npos+1 == 0 -> whole line */
  char tmp[128];
  size_t l = len - s;
  if (l > 127) l = 127;
  memcpy(tmp, line + s, l);
  tmp[l] = 0;
  return atoll(tmp);
}

/* FragmentsDatabase::FragmentsDatabase — src/FragmentsDatabase.cpp:54-101 */
int rko_load_csv(const char *path, rko_frag **recs, uint64_t *n, uint64_t *lx1, uint64_t *ly1, char **header) {
  FILE *f = fopen(path, "rb");
  if (!f) return -1;
  fseek(f, 0, SEEK_END);
  long sz = ftell(f);
  fseek(f, 0, SEEK_SET);
  char *data = (char *)malloc((size_t)sz + 1);
  if (fread(data, 1, (size_t)sz, f) != (size_t)sz) { fclose(f); free(data); return -1; }
  fclose(f);
  data[sz] = 0;

  size_t pos = 0;
  uint64_t total_frags = 0;
  size_t hdr_cap = 4096, hdr_len = 0;
  char *hdr = (char *)malloc(hdr_cap);
  for (int ln = 1; ln <= 16; ++ln) { /* :57-77, each line is re-emitted with '\n' appended */
    size_t s = pos;
    while (pos < (size_t)sz && data[pos] != '\n') ++pos;
    size_t l = pos - s;
    if (pos < (size_t)sz) ++pos;
    if (hdr_len + l + 2 > hdr_cap) { hdr_cap = (hdr_len + l + 2) * 2; hdr = (char *)realloc(hdr, hdr_cap); }
    memcpy(hdr + hdr_len, data + s, l);
    hdr_len += l;
    hdr[hdr_len++] = '\n';
    if (ln == 7) *lx1 = (uint64_t)(header_value(data + s, l) + 1);
    if (ln == 8) *ly1 = (uint64_t)(header_value(data + s, l) + 1);
    if (ln == 13) total_frags = (uint64_t)header_value(data + s, l);
  }
  hdr[hdr_len] = 0;

  size_t cap = 1024, cnt = 0;
  rko_frag *out = (rko_frag *)malloc(cap * sizeof(rko_frag));
  int rc = 0;
  /* :92-100 — while(!eof) getline; the final getline on an exhausted stream yields an empty line */
  int eof = (pos >= (size_t)sz) && sz == 0;
  while (!eof) {
    size_t s = pos;
    while (pos < (size_t)sz && data[pos] != '\n') ++pos;
    size_t l = pos - s;
    if (pos < (size_t)sz) ++pos; else eof = 1;
    rko_frag tmp;
    memset(&tmp, 0, sizeof tmp);
    if (!rko_parse_row(data + s, l, &tmp)) continue;
    if (cnt == cap) { cap *= 2; out = (rko_frag *)realloc(out, cap * sizeof(rko_frag)); }
    out[cnt++] = tmp;
    if (cnt > total_frags) { rc = -2; break; } /* :99 */
  }
  free(data);
  *recs = out;
  *n = cnt;
  if (header) *header = hdr; else free(hdr);
  return rc;
}

/* ------------------------------------------------------------------------------------------------
 * SequenceOcupationList — src/SequenceOcupationList.{h,cpp}
 * One singly linked list per center/100 bucket, newest entry first (push_front, :93-96).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  uint64_t center, length;
  uint32_t group; /* FragsGroup* in the reference */
  uint32_t rank;  /* the inserting fragment (not in the reference; lets tests see x/y owners) */
  int64_t next;
} ocupation;

typedef struct {
  double len_ratio, pos_ratio;
  uint64_t max_index; /* seq_size / DIVISOR (:4) */
  int64_t *head;      /* max_index + 1 lists (:5-7) */
} sol_t;

typedef struct {
  ocupation *e;
  size_t n, cap;
} pool_t;

static int sol_init(sol_t *s, double lr, double pr, uint64_t seq_size) {
  s->len_ratio = lr;
  s->pos_ratio = pr;
  s->max_index = seq_size / 100;
  s->head = (int64_t *)malloc((s->max_index + 1) * sizeof(int64_t));
  if (!s->head) return -1;
  for (uint64_t i = 0; i < s->max_index + 1; ++i) s->head[i] = -1;
  return 0;
}

/* deviation — src/SequenceOcupationList.cpp:20-31 (binary64, same operation order, no contraction) */
static double deviation(const sol_t *s, const ocupation *oc, uint64_t center, uint64_t length) {
  uint64_t dif_len = length > oc->length ? length - oc->length : oc->length - length;
  volatile double t1 = (double)length * s->len_ratio;
  volatile double q1 = (double)dif_len / t1;
  double sim_len = -fabs(q1) + 1.0;
  if (sim_len < 0) return 0.0;
  uint64_t dif_cen = center > oc->center ? center - oc->center : oc->center - center;
  volatile double t2 = (double)length * s->pos_ratio;
  volatile double q2 = (double)dif_cen / t2;
  double sim_pos = -fabs(q2) + 1.0;
  if (sim_pos < 0) return 0.0;
  volatile double a = sim_len * 0.4;
  volatile double b = sim_pos * 0.6;
  return a + b;
}

typedef struct { double d; int64_t ent; } best_t;

/* one `for (auto oc : *sind)` loop of get_associated_group (:38-44 and the four repeats) */
static int scan_list(const sol_t *s, const pool_t *p, uint64_t probe, uint64_t center, uint64_t length, best_t *b) {
  uint64_t idx = probe / 100; /* get_suitable_indices, :16-18 */
  if (idx > s->max_index) return -1; /* out of bounds in the reference */
  for (int64_t k = s->head[idx]; k >= 0; k = p->e[k].next) {
    double cur = deviation(s, &p->e[k], center, length);
    if (cur > b->d) { b->d = cur; b->ent = k; }
  }
  return 0;
}

/* get_associated_group — src/SequenceOcupationList.cpp:33-91; returns entry index or -1, -2 on OOB */
static int64_t sol_get(const sol_t *s, const pool_t *p, uint64_t center, uint64_t length) {
  best_t b = {0.0, -1};
  if (scan_list(s, p, center, center, length, &b)) return -2;
  if (center > 0 && scan_list(s, p, center - 1, center, length, &b)) return -2;                 /* :47 */
  if (center < s->max_index && scan_list(s, p, center + 1, center, length, &b)) return -2;      /* :58 */
  if (center > 1 && scan_list(s, p, center - 2, center, length, &b)) return -2;                 /* :69 */
  if (center < s->max_index - 1 /* unsigned */ && scan_list(s, p, center + 2, center, length, &b)) return -2; /* :80 */
  return b.ent;
}

/* insert — src/SequenceOcupationList.cpp:93-96 */
static int sol_insert(sol_t *s, pool_t *p, uint64_t center, uint64_t length, uint32_t group, uint32_t rank) {
  uint64_t idx = center / 100;
  if (idx > s->max_index) return -1;
  if (p->n == p->cap) {
    p->cap = p->cap ? p->cap * 2 : 1024;
    p->e = (ocupation *)realloc(p->e, p->cap * sizeof(ocupation));
  }
  ocupation *o = &p->e[p->n];
  o->center = center; o->length = length; o->group = group; o->rank = rank;
  o->next = s->head[idx];
  s->head[idx] = (int64_t)p->n++;
  return 0;
}

/* the lists above behind an exported handle (rk_oracle.h); the entry's `rank` field is unused, its tag is tag[entry] */
struct rko_sol {
  sol_t s;
  pool_t p;
  uint64_t *tag;
  size_t tag_cap;
};

rko_sol *rko_sol_create(double len_ratio, double pos_ratio, uint64_t seq_size) {
  rko_sol *h = (rko_sol *)calloc(1, sizeof *h);
  if (!h) return NULL;
  if (sol_init(&h->s, len_ratio, pos_ratio, seq_size)) { free(h); return NULL; }
  return h;
}

int rko_sol_insert(rko_sol *h, uint64_t center, uint64_t length, uint64_t tag) {
  if (sol_insert(&h->s, &h->p, center, length, 0, 0)) return -1;
  if (h->p.n > h->tag_cap) {
    uint64_t *t = (uint64_t *)realloc(h->tag, h->p.cap * sizeof(uint64_t));
    if (!t) { /* take the entry just pushed back: the list stays as it was */
      const ocupation *o = &h->p.e[--h->p.n];
      h->s.head[o->center / 100] = o->next;
      return -2;
    }
    h->tag = t;
    h->tag_cap = h->p.cap;
  }
  h->tag[h->p.n - 1] = tag;
  return 0;
}

int rko_sol_get(const rko_sol *h, uint64_t center, uint64_t length, uint64_t *tag) {
  const int64_t e = sol_get(&h->s, &h->p, center, length);
  if (e == -2) return -2;
  *tag = e >= 0 ? h->tag[e] : 0;
  return 0;
}

void rko_sol_destroy(rko_sol *h) {
  if (!h) return;
  free(h->s.head);
  free(h->p.e);
  free(h->tag);
  free(h);
}

/* ------------------------------------------------------------------------------------------------
 * std::sort as libstdc++ implements it (bits/stl_algo.h: __sort, __introsort_loop,
 * __unguarded_partition_pivot, __move_median_to_first, __final_insertion_sort; bits/stl_heap.h) —
 * the reference's sort_groups (src/commonFunctions.cpp:148-159) calls it with comp(a,b) = h(a) < h(b), and
 * std::sort is not stable, so tie order is the algorithm's.  Elements are ranks; keys are looked up in h[].
 * ---------------------------------------------------------------------------------------------- */
typedef struct { const uint64_t *h; } cmp_t;
#define LESS(c, a, b) ((c)->h[(a)] < (c)->h[(b)])

static void sw(uint32_t *a, uint32_t *b) { uint32_t t = *a; *a = *b; *b = t; }

static void move_median_to_first(uint32_t *result, uint32_t *a, uint32_t *b, uint32_t *c, const cmp_t *cm) {
  if (LESS(cm, *a, *b)) {
    if (LESS(cm, *b, *c)) sw(result, b);
    else if (LESS(cm, *a, *c)) sw(result, c);
    else sw(result, a);
  } else if (LESS(cm, *a, *c)) sw(result, a);
  else if (LESS(cm, *b, *c)) sw(result, c);
  else sw(result, b);
}

static uint32_t *unguarded_partition(uint32_t *first, uint32_t *last, uint32_t *pivot, const cmp_t *cm) {
  for (;;) {
    while (LESS(cm, *first, *pivot)) ++first;
    --last;
    while (LESS(cm, *pivot, *last)) --last;
    if (!(first < last)) return first;
    sw(first, last);
    ++first;
  }
}

static void push_heap_(uint32_t *first, long hole, long top, uint32_t value, const cmp_t *cm) {
  long parent = (hole - 1) / 2;
  while (hole > top && LESS(cm, first[parent], value)) {
    first[hole] = first[parent];
    hole = parent;
    parent = (hole - 1) / 2;
  }
  first[hole] = value;
}

static void adjust_heap(uint32_t *first, long hole, long len, uint32_t value, const cmp_t *cm) {
  const long top = hole;
  long child = hole;
  while (child < (len - 1) / 2) {
    child = 2 * (child + 1);
    if (LESS(cm, first[child], first[child - 1])) child--;
    first[hole] = first[child];
    hole = child;
  }
  if ((len & 1) == 0 && child == (len - 2) / 2) {
    child = 2 * (child + 1);
    first[hole] = first[child - 1];
    hole = child - 1;
  }
  push_heap_(first, hole, top, value, cm);
}

static void heap_sort(uint32_t *first, uint32_t *last, const cmp_t *cm) {
  /* __partial_sort(first, last, last): __heap_select == make_heap, then __sort_heap */
  long len = last - first;
  if (len >= 2) {
    long parent = (len - 2) / 2;
    for (;;) {
      uint32_t v = first[parent];
      adjust_heap(first, parent, len, v, cm);
      if (parent == 0) break;
      parent--;
    }
  }
  while (last - first > 1) {
    --last;
    uint32_t v = *last;
    *last = *first;
    adjust_heap(first, 0, last - first, v, cm);
  }
}

static void introsort_loop(uint32_t *first, uint32_t *last, long depth_limit, const cmp_t *cm) {
  while (last - first > 16) {
    if (depth_limit == 0) { heap_sort(first, last, cm); return; }
    --depth_limit;
    uint32_t *mid = first + (last - first) / 2;
    move_median_to_first(first, first + 1, mid, last - 1, cm);
    uint32_t *cut = unguarded_partition(first + 1, last, first, cm);
    introsort_loop(cut, last, depth_limit, cm);
    last = cut;
  }
}

static void unguarded_linear_insert(uint32_t *last, const cmp_t *cm) {
  uint32_t val = *last;
  uint32_t *next = last - 1;
  while (LESS(cm, val, *next)) { *last = *next; last = next; --next; }
  *last = val;
}

static void insertion_sort(uint32_t *first, uint32_t *last, const cmp_t *cm) {
  if (first == last) return;
  for (uint32_t *i = first + 1; i != last; ++i) {
    if (LESS(cm, *i, *first)) {
      uint32_t val = *i;
      memmove(first + 1, first, (size_t)(i - first) * sizeof(uint32_t));
      *first = val;
    } else unguarded_linear_insert(i, cm);
  }
}

static void std_sort(uint32_t *first, uint32_t *last, const cmp_t *cm) {
  if (first == last) return;
  long n = last - first, lg = 0;
  for (long t = n; t > 1; t >>= 1) ++lg; /* std::__lg */
  introsort_loop(first, last, lg * 2, cm);
  if (last - first > 16) {
    insertion_sort(first, first + 16, cm);
    for (uint32_t *i = first + 16; i != last; ++i) unguarded_linear_insert(i, cm);
  } else insertion_sort(first, last, cm);
}

/* std::sort of ranks by h[rank] (exported for tests that re-state single stages) */
void rko_std_sort_by_key(uint32_t *idx, uint64_t n, const uint64_t *h) {
  cmp_t cm = {h};
  std_sort(idx, idx + n, &cm);
}

/* ------------------------------------------------------------------------------------------------ */
void rko_result_free(rko_result *r) {
  free(r->rank_fidx); free(r->xowner); free(r->yowner); free(r->parent); free(r->gid); free(r->h);
  free(r->order); free(r->out_gid); free(r->repval); free(r->identity); free(r->diag_func);
  memset(r, 0, sizeof *r);
}

int rko_group(const rko_frag *recs, uint64_t n, uint64_t lx1, uint64_t ly1, double len_ratio, double pos_ratio,
              int want_diag, rko_result *out) {
  memset(out, 0, sizeof *out);
  const uint64_t vsize = 1 + lx1 / 10; /* FragmentsDatabase.cpp:84 */
  out->vsize = vsize;

  /* loaded_frags[xStart/10].push_back (FragmentsDatabase.cpp:96-97): stable bucketing in file order.
   * Iteration is begin()..end() with end = begin + vsize - 1 (FragmentsDatabase.h:29-31): the last bucket
   * is never visited. */
  uint64_t *bstart = (uint64_t *)calloc(vsize + 1, sizeof(uint64_t));
  for (uint64_t i = 0; i < n; ++i) {
    uint64_t b = recs[i].xStart / 10;
    if (b >= vsize) { free(bstart); return -3; }
    bstart[b + 1]++;
  }
  for (uint64_t b = 0; b < vsize; ++b) bstart[b + 1] += bstart[b];
  const uint64_t m = bstart[vsize - 1]; /* fragments in buckets 0 .. vsize-2 */
  uint32_t *rank_fidx = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  {
    uint64_t *cur = (uint64_t *)malloc(vsize * sizeof(uint64_t));
    memcpy(cur, bstart, vsize * sizeof(uint64_t));
    for (uint64_t i = 0; i < n; ++i) {
      uint64_t b = recs[i].xStart / 10;
      if (b == vsize - 1) continue;
      rank_fidx[cur[b]++] = (uint32_t)i;
    }
    free(cur);
  }
  out->n_kept = m;
  out->rank_fidx = rank_fidx;
  out->xowner = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->yowner = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->parent = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->gid = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->h = (uint64_t *)malloc((m ? m : 1) * sizeof(uint64_t));

  /* generate_fragment_groups — src/commonFunctions.cpp:41-80 */
  sol_t solxf, solyf, solxr, solyr;
  pool_t pool = {0, 0, 0};
  int rc = 0;
  if (sol_init(&solxf, len_ratio, pos_ratio, lx1) || sol_init(&solyf, len_ratio, pos_ratio, ly1) ||
      sol_init(&solxr, len_ratio, pos_ratio, lx1) || sol_init(&solyr, len_ratio, pos_ratio, ly1)) return -5;
  uint32_t n_groups = 0;
  for (uint64_t r = 0; r < m && rc == 0; ++r) { /* :51 — buckets in order, file order inside */
    const rko_frag *f = &recs[rank_fidx[r]];
    sol_t *solx = f->strand == 'f' ? &solxf : &solxr; /* :52-53 */
    sol_t *soly = f->strand == 'f' ? &solyf : &solyr;
    const uint64_t cx = f->xStart + f->length / 2, cy = f->yStart + f->length / 2;
    out->xowner[r] = out->yowner[r] = out->parent[r] = RKO_NONE;
    int64_t agx = sol_get(solx, &pool, cx, f->length); /* :55 */
    if (agx == -2) { rc = -4; break; }
    if (agx >= 0) {
      out->xowner[r] = out->parent[r] = pool.e[agx].rank;
      out->gid[r] = pool.e[agx].group;                                         /* :58 */
      if (sol_insert(soly, &pool, cy, f->length, out->gid[r], (uint32_t)r)) rc = -4; /* :59 */
      continue;
    }
    int64_t agy = sol_get(soly, &pool, cy, f->length); /* :63 */
    if (agy == -2) { rc = -4; break; }
    if (agy >= 0) {
      out->yowner[r] = out->parent[r] = pool.e[agy].rank;
      out->gid[r] = pool.e[agy].group;                                         /* :66 */
      if (sol_insert(solx, &pool, cx, f->length, out->gid[r], (uint32_t)r)) rc = -4; /* :67 */
      continue;
    }
    out->gid[r] = n_groups++;                                                  /* :72-74 */
    if (sol_insert(solx, &pool, cx, f->length, out->gid[r], (uint32_t)r)) rc = -4;   /* :75 */
    if (sol_insert(soly, &pool, cy, f->length, out->gid[r], (uint32_t)r)) rc = -4;   /* :76 */
  }
  free(solxf.head); free(solyf.head); free(solxr.head); free(solyr.head);
  free(pool.e);
  if (rc) { free(bstart); rko_result_free(out); return rc; }
  out->n_groups = n_groups;

  /* generate_diagonal_func — src/commonFunctions.cpp:161-177: yStart of the LAST fragment of the bucket
   * (`nh < oh` with oh = +inf never updated is always true), carried forward over empty buckets. */
  uint64_t *diag = (uint64_t *)malloc((vsize ? vsize : 1) * sizeof(uint64_t));
  for (uint64_t b = 0; b + 1 < vsize; ++b) {
    if (bstart[b + 1] == bstart[b]) diag[b] = b == 0 ? 0 : diag[b - 1];
    else diag[b] = recs[rank_fidx[bstart[b + 1] - 1]].yStart;
  }
  /* sort key of sort_groups' comparator — src/commonFunctions.cpp:149-156 */
  for (uint64_t r = 0; r < m; ++r) {
    const rko_frag *f = &recs[rank_fidx[r]];
    uint64_t dx = diag[f->xStart / 10];
    out->h[r] = f->yStart > dx ? f->yStart - dx : dx - f->yStart;
  }
  free(bstart);
  if (want_diag) out->diag_func = diag; else free(diag);

  /* members in push_back order == rank order (:58,66,73); groups in creation order */
  uint64_t *gstart = (uint64_t *)calloc((size_t)n_groups + 1, sizeof(uint64_t));
  for (uint64_t r = 0; r < m; ++r) gstart[out->gid[r] + 1]++;
  for (uint32_t g = 0; g < n_groups; ++g) gstart[g + 1] += gstart[g];
  uint32_t *members = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  {
    uint64_t *cur = (uint64_t *)malloc(((size_t)n_groups + 1) * sizeof(uint64_t));
    memcpy(cur, gstart, ((size_t)n_groups + 1) * sizeof(uint64_t));
    for (uint64_t r = 0; r < m; ++r) members[cur[out->gid[r]]++] = (uint32_t)r;
    free(cur);
  }
  /* sort_groups — src/commonFunctions.cpp:158 */
  cmp_t cm = {out->h};
  for (uint32_t g = 0; g < n_groups; ++g)
    if (gstart[g + 1] - gstart[g] > 1) std_sort(members + gstart[g], members + gstart[g + 1], &cm);

  /* save_frag_pair / save_frags_from_group / store_frag — src/commonFunctions.cpp:101-129 */
  out->order = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->out_gid = (uint32_t *)malloc((m ? m : 1) * sizeof(uint32_t));
  out->repval = (uint8_t *)malloc(m ? m : 1);
  out->identity = (float *)malloc((m ? m : 1) * sizeof(float));
  for (uint32_t g = 0; g < n_groups; ++g) {
    const uint64_t s = gstart[g], e = gstart[g + 1];
    for (uint64_t j = s; j < e; ++j) {
      const uint32_t fi = rank_fidx[members[j]];
      out->order[j] = fi;
      out->out_gid[j] = g;
      out->repval[j] = (e - s == 1) ? 0 : (j == s ? 1 : 2);
      out->identity[j] = (float)recs[fi].ident * 100 / (float)recs[fi].length;
    }
  }
  free(gstart);
  free(members);
  return 0;
}

/* ostream << float with the default format == printf("%g") with precision 6 */
int rko_write_output(const char *path, const char *header, const rko_frag *recs, const rko_result *r) {
  FILE *f = fopen(path, "wb");
  if (!f) return -1;
  setvbuf(f, NULL, _IOFBF, 1 << 22);
  fputs(header, f); /* sequence_manager::write_header, src/class_structs.cpp:8-11 */
  for (uint64_t j = 0; j < r->n_kept; ++j) {
    const rko_frag *q = &recs[r->order[j]];
    fprintf(f, "Frag,%llu,%llu,%llu,%llu,", (unsigned long long)q->xStart, (unsigned long long)q->yStart,
            (unsigned long long)q->xEnd, (unsigned long long)q->yEnd);
    fputc(q->strand, f);
    fprintf(f, ",%llu,%llu,%llu,%llu,%g,%g,0,%u\n", (unsigned long long)r->out_gid[j],
            (unsigned long long)q->length, (unsigned long long)q->score, (unsigned long long)q->ident,
            (double)q->similarity, (double)r->identity[j], (unsigned)r->repval[j]);
  }
  return fclose(f) ? -1 : 0;
}

int rko_write_input_csv(const char *path, const rko_frag *recs, uint64_t n, uint64_t lx_header, uint64_t ly_header) {
  FILE *f = fopen(path, "wb");
  if (!f) return -1;
  setvbuf(f, NULL, _IOFBF, 1 << 22);
  fprintf(f,
          "All by-Identity Ungapped Fragments (Hits based approach)\n"
          "[Abr.2015 -- < bitlab - Departamento de Arquitectura de Computadores >\n"
          "SeqX filename : synthX.fasta\nSeqY filename : synthY.fasta\nSeqX name : synthX\nSeqY name : synthY\n"
          "SeqX length : %llu\nSeqY length : %llu\nMin.fragment.length : 0\nMin.Identity : 0.00\n"
          "Tot Hits (seeds) : 0\nTot Hits (seeds) used: 0\nTotal fragments : %llu\n"
          "========================================================\n"
          "Type,xStart,yStart,xEnd,yEnd,strand(f/r),block,length,score,ident,similarity,%%ident,SeqX,SeqY\n"
          "========================================================\n",
          (unsigned long long)lx_header, (unsigned long long)ly_header, (unsigned long long)n);
  for (uint64_t i = 0; i < n; ++i) {
    const rko_frag *q = &recs[i];
    fprintf(f, "Frag,%llu,%llu,%llu,%llu,%c,%lld,%llu,%llu,%llu,%.9g,%.9g,0,0\n", (unsigned long long)q->xStart,
            (unsigned long long)q->yStart, (unsigned long long)q->xEnd, (unsigned long long)q->yEnd, q->strand,
            (long long)q->block, (unsigned long long)q->length, (unsigned long long)q->score,
            (unsigned long long)q->ident, (double)q->similarity, (double)q->similarity);
  }
  return fclose(f) ? -1 : 0;
}
