/*
 * pcsr_oracle.c -- TEST INFRASTRUCTURE ONLY (the parity oracle).
 *
 * A plain-C, single-threaded restatement of the edge-update path of the reference
 * (domargan/parallel-packed-csr): the packed-memory-array CSR with one sentinel slot per
 * vertex, gap-tolerant binary search, slide_right/slide_left, in-place redistribute, the
 * density-bound walk, double_list/half_list, plus the read side (edge_exists,
 * get_neighbourhood, one PageRank push step) and the PPPCSR vertex-range partition table.
 * Every function cites the reference file:line it follows.  With one thread the
 * reference's locking protocol reduces to: search -> (window pre-computation done while
 * "acquiring locks") -> insert/remove; that sequential behaviour is what is restated here.
 *
 * Parity pinning: tests/test_oracle.py checks this file against (a) committed golden
 * fixtures produced by the UNMODIFIED reference compiled into oracle/_ref/ (generator:
 * tests/golden/make_golden.py) and (b) live runs of oracle/_ref/ref_driver when present.
 * Beyond the logical graph it also reproduces the reference's physical geometry (N, logN,
 * H after every resize) for sequential streams, which the fixtures record.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may load this
 * library; the product (parallel-packed-csr_b200/) never does.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define SENT UINT32_MAX

typedef struct {
  uint32_t src, dest, value; /* reference src/pcsr/PCSR.h:30-35 */
} oslot_t;

typedef struct {
  uint32_t beginning, end, num_neighbors; /* reference src/pcsr/PCSR.h:18-23 */
} overt_t;

typedef struct {
  uint64_t N; /* slots */
  int logN;   /* leaf size */
  int H;      /* tree height */
  oslot_t *items;
  overt_t *nodes;
  uint64_t n, ncap;
  uint64_t not_found; /* count of "not found" removes (reference prints a line, PCSR.cpp:751) */
  uint64_t resizes;
} opcsr_t;

/* ---------- geometry: reference src/pcsr/PCSR.cpp:22-33 (bsr), :68-73 (resizeEdgeArray) ---------- */
static int bsr64(uint64_t w) { /* index of the most significant set bit; undefined for 0 like the asm */
  int r = 0;
  while (w >>= 1) r++;
  return r;
}

static void set_geometry(opcsr_t *g, uint64_t new_n) {
  g->N = new_n;
  g->logN = 1 << bsr64((uint64_t)bsr64(g->N) * 2 + 1);
  g->H = bsr64(g->N / (uint64_t)g->logN);
  g->resizes++;
}

static int slot_null(const oslot_t *s) { return s->value == 0; }                         /* PCSR.h:57-60 */
static int slot_sentinel(const oslot_t *s) { return s->dest == SENT || s->value == SENT; } /* PCSR.cpp:64 */

/* reference src/pcsr/PCSR.cpp:168-183 (fix_sentinel) */
static void repoint(opcsr_t *g, const oslot_t *s, uint64_t where) {
  if (!slot_sentinel(s)) return;
  uint32_t v = s->value;
  if (v == SENT) {
    v = 0;
  } else {
    g->nodes[v - 1].end = (uint32_t)where;
  }
  g->nodes[v].beginning = (uint32_t)where;
  if (v == g->n - 1) g->nodes[v].end = (uint32_t)(g->N - 1);
}

/* reference src/pcsr/PCSR.cpp:126-133 (get_density): live slots / len as a double */
static double window_density(const opcsr_t *g, int64_t start, int64_t len) {
  int64_t live = 0;
  for (int64_t i = start; i < start + len; i++) live += !slot_null(&g->items[i]);
  return (double)live / (double)len;
}

/* reference src/pcsr/PCSR.cpp:156-165 (density_bound) */
static double bound_upper(const opcsr_t *g, int depth) { return 3.0 / 4.0 + ((.25 * depth) / g->H); }
static double bound_lower(const opcsr_t *g, int depth) { return 1.0 / 4.0 - ((0.125 * depth) / g->H); }

/* reference src/pcsr/PCSR.cpp:222-249 (in-place redistribute) */
static void spread(opcsr_t *g, int64_t start, int64_t len) {
  oslot_t *it = g->items;
  int64_t live = 0;
  const int64_t stop = start + len;
  for (int64_t i = start; i < stop; i++) { /* pack to the left */
    it[start + live] = it[i];
    live += !slot_null(&it[start + live]);
  }
  for (int64_t i = start + live; i < stop; i++) {
    it[i].src = (uint32_t)-1;
    it[i].value = 0;
    it[i].dest = 0;
  }
  const double step = (double)len / (double)live;
  double pos = (double)start + (double)(live - 1) * step;
  for (int64_t i = start + live - 1; i > start; i--) { /* spread right-to-left */
    const int64_t to = (int64_t)pos;
    oslot_t tmp = it[to];
    it[to] = it[i];
    it[i] = tmp;
    repoint(g, &it[to], (uint64_t)to);
    pos -= step;
  }
  repoint(g, &it[start], (uint64_t)start);
}

/* reference src/pcsr/PCSR.cpp:251-282 (double_list) */
static void grow(opcsr_t *g) {
  const uint64_t old = g->N;
  set_geometry(g, old * 2);
  g->items = (oslot_t *)realloc(g->items, g->N * sizeof(oslot_t));
  for (uint64_t i = old; i < g->N; i++) {
    g->items[i].value = 0;
    g->items[i].dest = 0;
  }
  spread(g, 0, (int64_t)g->N);
}

/* reference src/pcsr/PCSR.cpp:284-320 (half_list) */
static void shrink(opcsr_t *g) {
  const uint64_t old = g->N;
  set_geometry(g, old / 2);
  uint64_t j = 0;
  for (uint64_t i = 0; i < old; i++) {
    if (!slot_null(&g->items[i])) g->items[j++] = g->items[i];
  }
  for (; j < g->N; j++) {
    g->items[j].value = 0;
    g->items[j].dest = 0;
  }
  g->items = (oslot_t *)realloc(g->items, g->N * sizeof(oslot_t));
  spread(g, 0, (int64_t)g->N);
}

static void push_left(opcsr_t *g, int64_t index);

/* reference src/pcsr/PCSR.cpp:326-355 (slide_right): returns -1 if it ran off the right end */
static int push_right(opcsr_t *g, int64_t index) {
  int rval = 0;
  oslot_t carry = g->items[index];
  g->items[index].src = (uint32_t)-1;
  g->items[index].dest = 0;
  g->items[index].value = 0;
  index++;
  while (index < (int64_t)g->N && !slot_null(&g->items[index])) {
    oslot_t t = g->items[index];
    g->items[index] = carry;
    if (!slot_null(&carry)) repoint(g, &carry, (uint64_t)index);
    carry = t;
    index++;
  }
  if (!slot_null(&carry)) repoint(g, &carry, (uint64_t)index);
  if (index == (int64_t)g->N) {
    index--;
    push_left(g, index);
    rval = -1;
  }
  g->items[index] = carry;
  return rval;
}

/* reference src/pcsr/PCSR.cpp:360-390 (slide_left) */
static void push_left(opcsr_t *g, int64_t index) {
  oslot_t carry = g->items[index];
  g->items[index].src = (uint32_t)-1;
  g->items[index].dest = 0;
  g->items[index].value = 0;
  index--;
  while (index >= 0 && !slot_null(&g->items[index])) {
    oslot_t t = g->items[index];
    g->items[index] = carry;
    if (!slot_null(&carry)) repoint(g, &carry, (uint64_t)index);
    carry = t;
    index--;
  }
  if (index == -1) {
    grow(g);
    push_right(g, 0);
    index = 0;
  }
  if (!slot_null(&carry)) repoint(g, &carry, (uint64_t)index);
  g->items[index] = carry;
}

/* reference src/pcsr/PCSR.cpp:427-502 (binary_search, minus the version counters):
 * smallest live slot in [start,end) whose dest >= key, else `end`; empty probes walk outwards. */
static uint32_t gap_search(const opcsr_t *g, uint32_t key, uint32_t start, uint32_t end) {
  const oslot_t *it = g->items;
  while (start + 1 < end) {
    const uint32_t mid = (start + end) / 2;
    oslot_t item = it[mid];
    uint32_t change = 1, check = mid;
    int more = 1;
    while (slot_null(&item) && more) {
      more = 0;
      check = mid + change;
      if (check < end) {
        more = 1;
        item = it[check];
        if (!slot_null(&item)) break;
      }
      check = mid - change;
      if (check >= start) {
        more = 1;
        item = it[check];
      }
      change++;
    }
    if (slot_null(&item) || start == check || end == check) {
      if (!slot_null(&item) && start == check && key <= item.dest) return check;
      return mid;
    }
    if (key == item.dest) return check;
    if (key < item.dest) {
      end = check;
    } else {
      start = check;
    }
  }
  if (end < start) start = end;
  if (key <= it[start].dest && !slot_null(&it[start])) return start;
  return end;
}

typedef struct {
  int have;       /* 0: walk inside place() like info==nullptr */
  int must_grow;  /* info->double_list */
  int64_t len;    /* info->max_len */
  int64_t start;  /* info->node_index_final */
} owindow_t;

/* reference src/pcsr/PCSR.cpp:1012-1084: the redistribute window the insert will use, computed
 * before the insert with density + 1/len ("as if the element were already there"). */
static owindow_t predict_window(const opcsr_t *g, uint32_t index) {
  owindow_t w = {1, 0, 0, 0};
  int64_t len = g->logN;
  int64_t start = ((int64_t)index / len) * len;
  int level = g->H;
  if (window_density(g, start, len) + (1.0 / (double)len) == 1) start = (start / (2 * len)) * (2 * len);
  double ub = bound_upper(g, level);
  double dens = window_density(g, start, len) + (1.0 / (double)len);
  while (dens >= ub) {
    len *= 2;
    if (len <= (int64_t)g->N) {
      level--;
      start = (start / len) * len;
      ub = bound_upper(g, level);
      dens = window_density(g, start, len) + (1.0 / (double)len);
    } else {
      w.must_grow = 1;
      return w;
    }
  }
  w.len = len;
  w.start = (start / len) * len;
  return w;
}

/* reference src/pcsr/PCSR.cpp:519-595 (insert) */
static void place(opcsr_t *g, uint32_t index, oslot_t elem, uint32_t src, const owindow_t *info) {
  int64_t len = g->logN;
  int64_t start = ((int64_t)index / len) * len;
  int level = g->H;
  if (!slot_null(&g->items[index])) {
    if (!slot_sentinel(&elem) && g->items[index].dest == elem.dest) {
      g->items[index].value = elem.value; /* duplicate insert overwrites (:529-532) */
      return;
    }
    if (index == g->N - 1) { /* :533-540 */
      grow(g);
      uint32_t again = gap_search(g, elem.dest, g->nodes[src].beginning + 1, g->nodes[src].end);
      place(g, again, elem, src, NULL);
      return;
    }
    if (push_right(g, index) == -1) {
      index -= 1;
      push_left(g, index);
    }
  }
  g->items[index] = elem;

  double dens = window_density(g, start, len);
  if (dens == 1) { /* leaf completely full: rewrite the parent (:555-560) */
    start = (start / (2 * len)) * (2 * len);
    spread(g, start, 2 * len);
  } else {
    spread(g, start, len);
  }
  double ub = bound_upper(g, level);
  dens = window_density(g, start, len);
  if (info != NULL && info->have) {
    if (info->must_grow) {
      grow(g);
      return;
    }
    len = info->len;
    start = info->start;
  } else {
    while (dens >= ub) { /* :578-591 */
      len *= 2;
      if (len <= (int64_t)g->N) {
        level--;
        start = (start / len) * len;
        ub = bound_upper(g, level);
        dens = window_density(g, start, len);
      } else {
        grow(g);
        return;
      }
    }
  }
  if (len > g->logN) spread(g, start, len);
}

/* reference src/pcsr/PCSR.cpp:597-630 (remove) */
static void erase(opcsr_t *g, uint32_t index, uint32_t dest) {
  int64_t len = g->logN;
  int64_t start = ((int64_t)index / len) * len;
  int level = g->H;
  if (slot_null(&g->items[index]) || g->items[index].dest != dest) return;
  g->items[index].value = 0;
  g->items[index].dest = 0;
  spread(g, start, len);
  double lb = bound_lower(g, level);
  double dens = window_density(g, start, len);
  while (dens < lb) {
    len *= 2;
    if (len <= (int64_t)g->N) {
      level--;
      start = (start / len) * len;
      lb = bound_lower(g, level);
      dens = window_density(g, start, len);
    } else {
      shrink(g);
      return;
    }
  }
  spread(g, start, len);
}

/* ------------------------------------------------------------------------------------------- */
/* public surface (loaded through ctypes by tests/oracle_py.py)                                 */
/* ------------------------------------------------------------------------------------------- */

/* reference src/pcsr/PCSR.cpp:775-838 (constructor: N, sentinels at floor(i*N/src_n)) */
opcsr_t *opcsr_create(uint32_t init_n, uint32_t src_n) {
  opcsr_t *g = (opcsr_t *)calloc(1, sizeof(opcsr_t));
  uint32_t m = init_n + src_n;
  if (m < 1024u) m = 1024u;
  set_geometry(g, (uint64_t)2 << bsr64(m));
  g->resizes = 0;
  g->items = (oslot_t *)malloc(g->N * sizeof(oslot_t));
  g->n = src_n;
  g->ncap = src_n ? src_n : 1;
  g->nodes = (overt_t *)calloc(g->ncap, sizeof(overt_t));
  double pos = 0.0;
  const double step = (double)g->N / (double)src_n;
  for (uint32_t i = 0; i < src_n; i++) {
    g->nodes[i].beginning = (i == 0) ? 0 : g->nodes[i - 1].end;
    pos += step;
    g->nodes[i].end = (uint32_t)(int)pos;
    g->nodes[i].num_neighbors = 0;
  }
  if (src_n != 0) g->nodes[src_n - 1].end = (uint32_t)(g->N - 1);
  pos = 0.0;
  int64_t next = 0;
  uint32_t cur = 0;
  for (int64_t i = 0; i < (int64_t)g->N; i++) {
    if (i == next && cur < src_n) {
      g->items[i].src = cur;
      g->items[i].dest = SENT;
      g->items[i].value = (i == 0) ? SENT : cur;
      cur++;
      pos += step;
      next = (int64_t)(int)pos;
    } else {
      g->items[i].src = (uint32_t)-1;
      g->items[i].dest = 0;
      g->items[i].value = 0;
    }
  }
  return g;
}

void opcsr_destroy(opcsr_t *g) {
  if (!g) return;
  free(g->items);
  free(g->nodes);
  free(g);
}

/* reference src/pcsr/PCSR.cpp:1374-1445 with retries == 0 and one thread */
void opcsr_add_edge(opcsr_t *g, uint32_t src, uint32_t dest, uint32_t value) {
  if (value == 0 || src >= g->n) return; /* :1375 */
  oslot_t e = {src, dest, value};
  g->nodes[src].num_neighbors++; /* :1392 -- counts calls, not distinct edges */
  uint32_t where = gap_search(g, dest, g->nodes[src].beginning + 1, g->nodes[src].end);
  if (where == g->N - 1 && !slot_null(&g->items[where])) { /* :992-997 -> :1433-1437 with info == nullptr */
    where = gap_search(g, dest, g->nodes[src].beginning + 1, g->nodes[src].end);
    place(g, where, e, src, NULL);
    return;
  }
  owindow_t w = predict_window(g, where);
  if (w.must_grow) where = gap_search(g, dest, g->nodes[src].beginning + 1, g->nodes[src].end);
  place(g, where, e, src, &w);
}

/* reference src/pcsr/PCSR.cpp:709-773 + :1179-1188 (not-found detection) */
void opcsr_remove_edge(opcsr_t *g, uint32_t src, uint32_t dest) {
  if (src >= g->n) return; /* the reference has no check here (out-of-bounds read); refuse instead */
  uint32_t where = gap_search(g, dest, g->nodes[src].beginning + 1, g->nodes[src].end);
  g->nodes[src].num_neighbors--; /* :747 -- before knowing whether the edge exists */
  if (slot_null(&g->items[where]) || g->items[where].dest != dest || dest == SENT) {
    g->not_found++;
    return;
  }
  erase(g, where, dest);
}

/* reference src/pcsr/PCSR.cpp:681-703 (add_node) */
void opcsr_add_node(opcsr_t *g) {
  if (g->n == g->ncap) {
    g->ncap *= 2;
    g->nodes = (overt_t *)realloc(g->nodes, g->ncap * sizeof(overt_t));
  }
  const uint64_t id = g->n;
  overt_t v;
  oslot_t s = {(uint32_t)id, SENT, (uint32_t)id};
  if (id > 0) {
    v.beginning = g->nodes[id - 1].end;
    v.end = v.beginning + 1;
  } else {
    v.beginning = 0;
    v.end = 1;
    s.value = SENT;
  }
  v.num_neighbors = 0;
  g->nodes[g->n++] = v;
  place(g, v.beginning, s, (uint32_t)id, NULL);
}

/* reference src/pcsr/PCSR.cpp:860-869 */
int opcsr_edge_exists(const opcsr_t *g, uint32_t src, uint32_t dest) {
  if (src >= g->n) return 0;
  uint32_t where = gap_search(g, dest, g->nodes[src].beginning + 1, g->nodes[src].end);
  const oslot_t *s = &g->items[where];
  return !slot_null(s) && !slot_sentinel(s) && s->dest == dest;
}

uint64_t opcsr_n(const opcsr_t *g) { return g->n; }
uint64_t opcsr_slots(const opcsr_t *g) { return g->N; }
int opcsr_leaf(const opcsr_t *g) { return g->logN; }
int opcsr_height(const opcsr_t *g) { return g->H; }
uint64_t opcsr_not_found(const opcsr_t *g) { return g->not_found; }
uint64_t opcsr_resizes(const opcsr_t *g) { return g->resizes; }
uint32_t opcsr_num_neighbors(const opcsr_t *g, uint32_t v) { return g->nodes[v].num_neighbors; }

/* reference src/pcsr/PCSR.cpp:901-912 (get_neighbourhood): returns the degree, fills out[0..cap) */
uint64_t opcsr_neighbourhood(const opcsr_t *g, uint32_t v, uint32_t *out, uint64_t cap) {
  uint64_t k = 0;
  if (v >= g->n) return 0;
  for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++) {
    if (g->items[i].value != 0) {
      if (out && k < cap) out[k] = g->items[i].dest;
      k++;
    }
  }
  return k;
}

/* whole-graph export: rowptr[n+1], col[E] (col may be NULL to size), num_neighbors[n] */
uint64_t opcsr_export(const opcsr_t *g, uint64_t *rowptr, uint32_t *col, uint32_t *nn) {
  uint64_t k = 0;
  for (uint64_t v = 0; v < g->n; v++) {
    if (rowptr) rowptr[v] = k;
    for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++) {
      if (g->items[i].value != 0) {
        if (col) col[k] = g->items[i].dest;
        k++;
      }
    }
    if (nn) nn[v] = g->nodes[v].num_neighbors;
  }
  if (rowptr) rowptr[g->n] = k;
  return k;
}

/* the stored values in the order of opcsr_export's col (val may be NULL to size) */
uint64_t opcsr_export_values(const opcsr_t *g, uint32_t *val) {
  uint64_t k = 0;
  for (uint64_t v = 0; v < g->n; v++)
    for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++)
      if (g->items[i].value != 0) {
        if (val) val[k] = g->items[i].value;
        k++;
      }
  return k;
}

/* batch front end used by tests and the cpu_baseline leg: value 0 = delete */
void opcsr_apply(opcsr_t *g, const uint32_t *src, const uint32_t *dst, const uint32_t *val, uint64_t count) {
  for (uint64_t i = 0; i < count; i++) {
    if (val == NULL || val[i] != 0) {
      opcsr_add_edge(g, src[i], dst[i], val ? val[i] : 1u);
    } else {
      opcsr_remove_edge(g, src[i], dst[i]);
    }
  }
}

/* reference src/utility/pagerank.h:16-29 with weight_t = double: one push step */
void opcsr_pagerank_f64(const opcsr_t *g, const double *in, double *out) {
  for (uint64_t v = 0; v < g->n; v++) out[v] = 0.0;
  for (uint64_t v = 0; v < g->n; v++) {
    const double contrib = in[v] / (double)g->nodes[v].num_neighbors;
    for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++) {
      if (g->items[i].value != 0) out[g->items[i].dest] += contrib;
    }
  }
}

/* same with weight_t = float (what reference test/DataStructureTest.cpp:205 instantiates) */
void opcsr_pagerank_f32(const opcsr_t *g, const float *in, float *out) {
  for (uint64_t v = 0; v < g->n; v++) out[v] = 0.0f;
  for (uint64_t v = 0; v < g->n; v++) {
    const float contrib = in[v] / (float)g->nodes[v].num_neighbors;
    for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++) {
      if (g->items[i].value != 0) out[g->items[i].dest] += contrib;
    }
  }
}

/* reference src/utility/bfs.h:15-36: sequential queue BFS, UINT32_MAX = unreached */
void opcsr_bfs(const opcsr_t *g, uint32_t start, uint32_t *dist) {
  uint32_t *queue = (uint32_t *)malloc((g->n ? g->n : 1) * sizeof(uint32_t));
  uint64_t head = 0, tail = 0;
  for (uint64_t v = 0; v < g->n; v++) dist[v] = UINT32_MAX;
  if (start >= g->n) {
    free(queue);
    return;
  }
  queue[tail++] = start;
  dist[start] = 0;
  while (head < tail) {
    const uint32_t a = queue[head++];
    for (uint32_t i = g->nodes[a].beginning + 1; i < g->nodes[a].end; i++) {
      if (g->items[i].value != 0) {
        const uint32_t d = g->items[i].dest;
        if (d < g->n && dist[d] == UINT32_MAX) {
          dist[d] = dist[a] + 1;
          queue[tail++] = d;
        }
      }
    }
  }
  free(queue);
}

/* PMA invariants I2/I3/I6 of SURVEY.md §8a checked on the oracle's own state (self-test) */
int opcsr_check(const opcsr_t *g) {
  uint64_t live = 0;
  for (uint64_t i = 0; i < g->N; i++) live += !slot_null(&g->items[i]);
  uint64_t edges = 0;
  for (uint64_t v = 0; v < g->n; v++) {
    const oslot_t *s = &g->items[g->nodes[v].beginning];
    if (!slot_sentinel(s) || s->src != v) return 2;
    if (v + 1 < g->n && g->nodes[v].end != g->nodes[v + 1].beginning) return 3;
    if (v + 1 == g->n && g->nodes[v].end != g->N - 1) return 4;
    int64_t prev = -1;
    for (uint32_t i = g->nodes[v].beginning + 1; i < g->nodes[v].end; i++) {
      if (g->items[i].value != 0) {
        if (g->items[i].src != v) return 5;
        if ((int64_t)g->items[i].dest <= prev) return 6;
        prev = g->items[i].dest;
        edges++;
      }
    }
  }
  if (live != edges + g->n) return 7;
  return 0;
}

/* ---------- PPPCSR partition table: reference src/pppcsr/PPPCSR.cpp:13-34, :58-66 ---------- */
/* Fills starts[0..parts) with the first vertex of each partition and sizes[0..parts). */
void opppcsr_table(uint32_t init_n, uint32_t parts, uint64_t *starts, uint64_t *sizes) {
  uint64_t psize = init_n / parts; /* std::ceil of an integer quotient is a no-op (:20) */
  uint64_t cur = 0;
  for (uint32_t p = 0; p < parts; p++) {
    if (p > 0) cur += psize;
    starts[p] = cur;
    if (p == parts - 1) psize = init_n - (uint64_t)p * psize; /* last takes the remainder (:27-29) */
    sizes[p] = psize;
  }
}

uint32_t opppcsr_owner(const uint64_t *starts, uint32_t parts, uint64_t vertex) {
  for (uint32_t i = 1; i < parts; i++) {
    if (starts[i] > vertex) return i - 1;
  }
  return parts - 1;
}

/* reference src/thread_pool_pppcsr/thread_pool_pppcsr.cpp:32-47: thread -> domain table */
void opool_domain_table(int threads, int domains, int *thread_to_domain, int *first_thread, int *num_threads) {
  const int min_threads = threads / domains;
  const int threshold = threads % domains;
  int counter = 0, cur = 0;
  for (int d = 0; d < domains; d++) {
    first_thread[d] = 0;
    num_threads[d] = 0;
  }
  for (int i = 0; i < threads; i++) {
    thread_to_domain[i] = cur;
    counter++;
    if (counter == min_threads + (cur < threshold)) {
      num_threads[cur] = counter;
      first_thread[cur] = i - counter + 1;
      counter = 0;
      cur++;
    }
  }
}
