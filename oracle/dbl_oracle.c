/*
 * dbl_oracle.c -- CPU ORACLE (test infrastructure only; see dbl_oracle.h for the parity status).
 *
 * Reference paths are relative to /root/reference/src/main/scala/com/github/cleanzr/dblink/ ;
 * GU = GibbsUpdates.scala.  Nothing here is copied from the reference (which is Scala/Spark);
 * each function restates the arithmetic of the cited lines in plain C.
 *
 * Compile with -ffp-contract=off: the draw protocol is defined in terms of individually rounded
 * IEEE-754 double operations.
 */
#define _POSIX_C_SOURCE 200809L
#include "dbl_oracle.h"
#include "dbl_oracle_priv.h"

#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

/* ------------------------------------------------------------------------------------------ */
/* RNG protocol: Philox4x32-10 (Salmon et al., SC'11), counter = (id, sub, iteration, phase),   */
/* key = 64-bit seed.  Replaces the reference's per-partition MersenneTwister (GU:139-140).     */
/* ------------------------------------------------------------------------------------------ */

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  uint32_t k0 = key[0], k1 = key[1];
  for (int round = 0; round < 10; ++round) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* two uniforms in the OPEN interval (0,1): u = ((bits >> 12) + 0.5) * 2^-52 */
static double bits_to_unit(uint32_t lo, uint32_t hi) {
  uint64_t x = ((uint64_t)hi << 32) | lo;
  return ((double)(x >> 12) + 0.5) * (1.0 / 4503599627370496.0);
}

void orc_uniform2(uint64_t seed, uint32_t phase, uint32_t iter, uint32_t id, uint32_t sub, double u[2]) {
  uint32_t ctr[4] = {id, sub, iter, phase};
  uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  uint32_t o[4];
  orc_philox4x32_10(ctr, key, o);
  u[0] = bits_to_unit(o[0], o[1]);
  u[1] = bits_to_unit(o[2], o[3]);
}

/* ------------------------------------------------------------------------------------------ */
/* Similarity function -- SimilarityFn.scala:61-98                                              */
/* ------------------------------------------------------------------------------------------ */

/* unit-cost Levenshtein distance (commons-lang3 StringUtils.getLevenshteinDistance, SimilarityFn.scala:22,95) */
int orc_levenshtein(const char *a, const char *b) {
  int la = (int)strlen(a), lb = (int)strlen(b);
  if (la == 0) return lb;
  if (lb == 0) return la;
  int *row = (int *)malloc(sizeof(int) * (size_t)(lb + 1));
  for (int j = 0; j <= lb; ++j) row[j] = j;
  for (int i = 1; i <= la; ++i) {
    int diag = row[0];
    row[0] = i;
    for (int j = 1; j <= lb; ++j) {
      int up = row[j];
      int sub = diag + (a[i - 1] != b[j - 1]);
      int best = sub;
      if (up + 1 < best) best = up + 1;
      if (row[j - 1] + 1 < best) best = row[j - 1] + 1;
      row[j] = best;
      diag = up;
    }
  }
  int d = row[lb];
  free(row);
  return d;
}

static double sim_from_distance(int dist, int la, int lb, double threshold, double max_sim) {
  /* SimilarityFn.scala:84-89: unit = 1 - 2 d / (|a|+|b|+d), 1 when both empty */
  int total = la + lb;
  double unit;
  if (total > 0) {
    double d = (double)dist;
    unit = 1.0 - 2.0 * d / ((double)total + d);
  } else {
    unit = 1.0;
  }
  /* SimilarityFn.scala:65-70 */
  double trans_factor = max_sim / (max_sim - threshold);
  double trans = trans_factor * (max_sim * unit - threshold);
  return trans > 0.0 ? trans : 0.0;
}

double orc_lev_similarity(const char *a, const char *b, double threshold, double max_sim) {
  return sim_from_distance(orc_levenshtein(a, b), (int)strlen(a), (int)strlen(b), threshold, max_sim);
}

/* ------------------------------------------------------------------------------------------ */
/* Attribute index -- AttributeIndex.scala:107-245                                              */
/* ------------------------------------------------------------------------------------------ */


typedef struct { const char *s; double w; } sw_pair;
static int cmp_sw(const void *a, const void *b) { return strcmp(((const sw_pair *)a)->s, ((const sw_pair *)b)->s); }

static void index_finish(orc_index *ix) {
  int V = ix->V;
  /* norms: AttributeIndex.scala:234-245 (uses `probs`, not the renormalised distribution) */
  ix->norm = (double *)malloc(sizeof(double) * (size_t)V);
  ix->invnorm = (double *)malloc(sizeof(double) * (size_t)V);
  for (int v = 0; v < V; ++v) {
    if (ix->is_const) { ix->norm[v] = 1.0; ix->invnorm[v] = 1.0; continue; }
    double acc = 0.0;
    int p = ix->rowptr[v], pe = ix->rowptr[v + 1];
    for (int w = 0; w < V; ++w) {
      double e = 1.0;
      if (p < pe && ix->col[p] == w) { e = ix->expsim[p]; ++p; }
      acc += ix->probs[w] * e;
    }
    ix->invnorm[v] = acc;
    ix->norm[v] = 1.0 / acc;
  }
  /* base pmfs B_k(v) ~ probs(v) * norm(v)^k (AttributeIndex.scala:209-216; DiscreteDist normalises,
     random/IndexNonUniformDiscreteDist.scala:66-88).  Protocol: the power is k repeated multiplications. */
  int K = ix->kmax;
  ix->pk = (double *)malloc(sizeof(double) * (size_t)(K + 1) * (size_t)V);
  ix->cdf = (double *)malloc(sizeof(double) * (size_t)(K + 1) * (size_t)V);
  for (int k = 0; k <= K; ++k) {
    double *pk = ix->pk + (size_t)k * V, *cdf = ix->cdf + (size_t)k * V;
    double z = 0.0;
    for (int v = 0; v < V; ++v) {
      double w = ix->probs[v];
      if (!ix->is_const)
        for (int i = 0; i < k; ++i) w = w * ix->norm[v];
      pk[v] = w;
      z += w;
    }
    double c = 0.0;
    for (int v = 0; v < V; ++v) {
      pk[v] = pk[v] / z;
      c += pk[v];
      cdf[v] = c;
    }
  }
  ix->phi = (double *)malloc(sizeof(double) * (size_t)V);
  memcpy(ix->phi, ix->pk, sizeof(double) * (size_t)V);
}

orc_index *orc_index_build(const char *const *values, const double *weights, int V, int is_const,
                           double threshold, double max_sim, int kmax) {
  if (V <= 0) return NULL;
  orc_index *ix = (orc_index *)calloc(1, sizeof(orc_index));
  ix->V = V; ix->is_const = is_const; ix->kmax = kmax;
  sw_pair *sw = (sw_pair *)malloc(sizeof(sw_pair) * (size_t)V);
  for (int i = 0; i < V; ++i) { sw[i].s = values[i]; sw[i].w = weights[i]; }
  qsort(sw, (size_t)V, sizeof(sw_pair), cmp_sw); /* AttributeIndex.scala:113: ids in sorted-string order */
  ix->values = (char **)malloc(sizeof(char *) * (size_t)V);
  ix->probs = (double *)malloc(sizeof(double) * (size_t)V);
  double total = 0.0;
  for (int i = 0; i < V; ++i) total += sw[i].w; /* :114 foldLeft */
  for (int i = 0; i < V; ++i) {
    ix->values[i] = strdup(sw[i].s);
    ix->probs[i] = sw[i].w / total; /* :115 */
  }
  free(sw);
  ix->rowptr = (int32_t *)calloc((size_t)V + 1, sizeof(int32_t));
  if (!is_const) {
    /* AttributeIndex.scala:219-231: all pairs, keep exp(sim) > 1.0 */
    int *len = (int *)malloc(sizeof(int) * (size_t)V);
    for (int i = 0; i < V; ++i) len[i] = (int)strlen(ix->values[i]);
    size_t cap = (size_t)V * 8, nnz = 0;
    int32_t *ri = (int32_t *)malloc(sizeof(int32_t) * cap), *ci = (int32_t *)malloc(sizeof(int32_t) * cap);
    double *ev = (double *)malloc(sizeof(double) * cap);
    for (int i = 0; i < V; ++i)
      for (int j = i; j < V; ++j) {
        int d = orc_levenshtein(ix->values[i], ix->values[j]);
        double e = exp(sim_from_distance(d, len[i], len[j], threshold, max_sim));
        if (e > 1.0) {
          if (nnz + 2 > cap) {
            cap *= 2;
            ri = (int32_t *)realloc(ri, sizeof(int32_t) * cap);
            ci = (int32_t *)realloc(ci, sizeof(int32_t) * cap);
            ev = (double *)realloc(ev, sizeof(double) * cap);
          }
          ri[nnz] = i; ci[nnz] = j; ev[nnz] = e; ++nnz;
          if (i != j) { ri[nnz] = j; ci[nnz] = i; ev[nnz] = e; ++nnz; }
        }
      }
    free(len);
    for (size_t k = 0; k < nnz; ++k) ix->rowptr[ri[k] + 1]++;
    for (int i = 0; i < V; ++i) ix->rowptr[i + 1] += ix->rowptr[i];
    ix->col = (int32_t *)malloc(sizeof(int32_t) * (nnz ? nnz : 1));
    ix->expsim = (double *)malloc(sizeof(double) * (nnz ? nnz : 1));
    int32_t *fill = (int32_t *)malloc(sizeof(int32_t) * (size_t)V);
    memcpy(fill, ix->rowptr, sizeof(int32_t) * (size_t)V);
    /* entries were generated with (i, j>=i) ascending and mirrored; a stable two-key placement keeps
       each row sorted by column: insert in increasing column order */
    /* simple approach: counting by row then insertion sort inside each row */
    for (size_t k = 0; k < nnz; ++k) {
      int r = ri[k];
      int pos = fill[r]++;
      ix->col[pos] = ci[k];
      ix->expsim[pos] = ev[k];
    }
    for (int r = 0; r < V; ++r) {
      int lo = ix->rowptr[r], hi = ix->rowptr[r + 1];
      for (int p = lo + 1; p < hi; ++p) {
        int32_t c = ix->col[p]; double e = ix->expsim[p];
        int q = p - 1;
        while (q >= lo && ix->col[q] > c) { ix->col[q + 1] = ix->col[q]; ix->expsim[q + 1] = ix->expsim[q]; --q; }
        ix->col[q + 1] = c; ix->expsim[q + 1] = e;
      }
    }
    free(fill); free(ri); free(ci); free(ev);
  } else {
    ix->col = (int32_t *)malloc(sizeof(int32_t));
    ix->expsim = (double *)malloc(sizeof(double));
  }
  index_finish(ix);
  return ix;
}

orc_index *orc_index_from_tables(int V, int is_const, const double *phi, const int32_t *rowptr,
                                 const int32_t *col, const double *expsim, int kmax) {
  orc_index *ix = (orc_index *)calloc(1, sizeof(orc_index));
  ix->V = V; ix->is_const = is_const; ix->kmax = kmax;
  ix->values = NULL;
  ix->probs = (double *)malloc(sizeof(double) * (size_t)V);
  memcpy(ix->probs, phi, sizeof(double) * (size_t)V);
  ix->rowptr = (int32_t *)calloc((size_t)V + 1, sizeof(int32_t));
  int nnz = 0;
  if (!is_const) {
    memcpy(ix->rowptr, rowptr, sizeof(int32_t) * ((size_t)V + 1));
    nnz = rowptr[V];
  }
  ix->col = (int32_t *)malloc(sizeof(int32_t) * (size_t)(nnz ? nnz : 1));
  ix->expsim = (double *)malloc(sizeof(double) * (size_t)(nnz ? nnz : 1));
  if (nnz) {
    memcpy(ix->col, col, sizeof(int32_t) * (size_t)nnz);
    memcpy(ix->expsim, expsim, sizeof(double) * (size_t)nnz);
  }
  index_finish(ix);
  return ix;
}

void orc_index_free(orc_index *ix) {
  if (!ix) return;
  if (ix->values) { for (int i = 0; i < ix->V; ++i) free(ix->values[i]); free(ix->values); }
  free(ix->probs); free(ix->phi); free(ix->norm); free(ix->invnorm);
  free(ix->rowptr); free(ix->col); free(ix->expsim); free(ix->pk); free(ix->cdf);
  free(ix);
}
int orc_index_num_values(const orc_index *ix) { return ix->V; }
int orc_index_is_const(const orc_index *ix) { return ix->is_const; }
int orc_index_value_id(const orc_index *ix, const char *value) {
  int lo = 0, hi = ix->V - 1;
  while (lo <= hi) {
    int mid = (lo + hi) / 2;
    int c = strcmp(ix->values[mid], value);
    if (c == 0) return mid;
    if (c < 0) lo = mid + 1; else hi = mid - 1;
  }
  return -1;
}
const char *orc_index_value(const orc_index *ix, int v) { return (ix->values && v >= 0 && v < ix->V) ? ix->values[v] : NULL; }
const double *orc_index_phi(const orc_index *ix) { return ix->phi; }
const double *orc_index_norm(const orc_index *ix) { return ix->norm; }
const double *orc_index_invnorm(const orc_index *ix) { return ix->invnorm; }
const int32_t *orc_index_rowptr(const orc_index *ix) { return ix->rowptr; }
const int32_t *orc_index_col(const orc_index *ix) { return ix->col; }
const double *orc_index_expsim(const orc_index *ix) { return ix->expsim; }
int orc_index_nnz(const orc_index *ix) { return ix->rowptr[ix->V]; }
int orc_index_kmax(const orc_index *ix) { return ix->kmax; }
const double *orc_index_pk(const orc_index *ix) { return ix->pk; }
const double *orc_index_cdf(const orc_index *ix) { return ix->cdf; }

/* sparse row look-up; returns 1 and *e when (v1, v2) is stored */
static int row_find(const orc_index *ix, int v1, int v2, double *e) {
  int lo = ix->rowptr[v1], hi = ix->rowptr[v1 + 1] - 1;
  while (lo <= hi) {
    int mid = (lo + hi) >> 1;
    int c = ix->col[mid];
    if (c == v2) { *e = ix->expsim[mid]; return 1; }
    if (c < v2) lo = mid + 1; else hi = mid - 1;
  }
  return 0;
}
/* expSimOf: AttributeIndex.scala:183-186 (default 1.0) */
double orc_index_exp_sim_of(const orc_index *ix, int v1, int v2) {
  double e;
  if (ix->is_const) return 1.0;
  return row_find(ix, v1, v2, &e) ? e : 1.0;
}

/* ------------------------------------------------------------------------------------------ */
/* k-d tree partition function -- partitioning/KDTreePartitioner.scala:37-62,80-105,            */
/* MutableBST.scala:51-111, DomainSplitter.scala:43-110                                         */
/* ------------------------------------------------------------------------------------------ */


static orc_kdtree *tree_alloc(int n_nodes) {
  orc_kdtree *t = (orc_kdtree *)calloc(1, sizeof(orc_kdtree));
  t->n_nodes = n_nodes;
  t->attr = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_nodes);
  t->kind = (int32_t *)calloc((size_t)n_nodes, sizeof(int32_t));
  t->split = (int32_t *)calloc((size_t)n_nodes, sizeof(int32_t));
  t->set_ptr = (int32_t *)calloc((size_t)n_nodes + 1, sizeof(int32_t));
  t->leaf_no = (int32_t *)malloc(sizeof(int32_t) * (size_t)n_nodes);
  for (int i = 0; i < n_nodes; ++i) { t->attr[i] = -1; t->leaf_no[i] = -1; }
  t->set_cap = 64; t->set_len = 0;
  t->set_val = (int32_t *)malloc(sizeof(int32_t) * (size_t)t->set_cap);
  return t;
}

void orc_kdtree_free(orc_kdtree *t) {
  if (!t) return;
  free(t->attr); free(t->kind); free(t->split); free(t->set_ptr); free(t->set_val); free(t->leaf_no); free(t);
}

static int node_in_set(const orc_kdtree *t, int node, int32_t v) {
  int lo = t->set_ptr[node], hi = t->set_ptr[node + 1] - 1;
  while (lo <= hi) {
    int mid = (lo + hi) >> 1;
    if (t->set_val[mid] == v) return 1;
    if (t->set_val[mid] < v) lo = mid + 1; else hi = mid - 1;
  }
  return 0;
}

/* MutableBST.getLeafNodeId (MutableBST.scala:61-79) */
static int tree_leaf_node(const orc_kdtree *t, const int32_t *yrow) {
  int node = 0;
  while (node < t->n_nodes && t->attr[node] >= 0) {
    int32_t v = yrow[t->attr[node]];
    int right = t->kind[node] ? node_in_set(t, node, v) : (v > t->split[node]);
    node = right ? 2 * node + 2 : 2 * node + 1;
  }
  return node;
}
int orc_kdtree_leaf(const orc_kdtree *t, const int32_t *yrow) { return t->leaf_no[tree_leaf_node(t, yrow)]; }
int orc_kdtree_num_nodes(const orc_kdtree *t) { return t->n_nodes; }
int orc_kdtree_num_leaves(const orc_kdtree *t) { return t->n_leaves; }
int orc_kdtree_set_len(const orc_kdtree *t) { return t->set_len; }

typedef struct { int32_t value; double weight; } vw_pair;
static int cmp_vw_value(const void *a, const void *b) {
  int32_t x = ((const vw_pair *)a)->value, y = ((const vw_pair *)b)->value;
  return (x > y) - (x < y);
}
static int cmp_vw_weight_desc(const void *a, const void *b) {
  const vw_pair *p = (const vw_pair *)a, *q = (const vw_pair *)b;
  if (p->weight > q->weight) return -1;
  if (p->weight < q->weight) return 1;
  return (p->value > q->value) - (p->value < q->value); /* protocol tie-break: ascending value */
}
static int cmp_i32(const void *a, const void *b) {
  int32_t x = *(const int32_t *)a, y = *(const int32_t *)b;
  return (x > y) - (x < y);
}

/* Fit level by level.  Unpinned orders in the reference (Map iteration in KDTreePartitioner.scala:54 and
   the stable-sort tie order in DomainSplitter.scala:92) are fixed here as: nodes in ascending id,
   equal weights in ascending value. */
orc_kdtree *orc_kdtree_fit(const int32_t *y, int64_t E, int A, int num_levels, const int32_t *attr_ids,
                           int n_attr_ids) {
  int n_nodes = (1 << (num_levels + 1)) - 1;
  orc_kdtree *t = tree_alloc(n_nodes);
  t->leaf_no[0] = 0;
  t->n_leaves = 1;
  /* set_ptr is built at the end: collect sets per node first */
  int32_t **sets = (int32_t **)calloc((size_t)n_nodes, sizeof(int32_t *));
  int *set_n = (int *)calloc((size_t)n_nodes, sizeof(int));
  int32_t *node_of = (int32_t *)malloc(sizeof(int32_t) * (size_t)(E ? E : 1));
  for (int level = 0; level < num_levels; ++level) {
    int attr = attr_ids[level % n_attr_ids]; /* KDTreePartitioner.scala:45-49: cycle through attributeIds */
    for (int64_t e = 0; e < E; ++e) {
      /* MutableBST.getLeafNodeId on the tree built so far (set_ptr/set_val are assembled after the last level) */
      int node = 0;
      while (node < n_nodes && t->attr[node] >= 0) {
        int32_t v = y[e * A + t->attr[node]];
        int right;
        if (t->kind[node]) {
          right = 0;
          for (int q = 0; q < set_n[node] && !right; ++q) right = (sets[node][q] == v);
        } else {
          right = v > t->split[node];
        }
        node = right ? 2 * node + 2 : 2 * node + 1;
      }
      node_of[e] = node;
    }
    int first = (1 << level) - 1, last = (1 << (level + 1)) - 2;
    for (int node = first; node <= last; ++node) {
      if (t->leaf_no[node] < 0) continue;
      /* domain of (value, count) among entities in this node (KDTreePartitioner.scala:85-104) */
      int64_t cnt = 0;
      for (int64_t e = 0; e < E; ++e) cnt += (node_of[e] == node);
      if (cnt == 0) continue; /* node never appears in the accumulator -> stays a leaf */
      int32_t *vals = (int32_t *)malloc(sizeof(int32_t) * (size_t)cnt);
      int64_t k = 0;
      for (int64_t e = 0; e < E; ++e) if (node_of[e] == node) vals[k++] = y[e * A + attr];
      qsort(vals, (size_t)cnt, sizeof(int32_t), cmp_i32);
      vw_pair *dom = (vw_pair *)malloc(sizeof(vw_pair) * (size_t)cnt);
      int nd = 0;
      for (int64_t i = 0; i < cnt; ++i) {
        if (nd && dom[nd - 1].value == vals[i]) dom[nd - 1].weight += 1.0;
        else { dom[nd].value = vals[i]; dom[nd].weight = 1.0; ++nd; }
      }
      free(vals);
      double half = 0.0;
      for (int i = 0; i < nd; ++i) half += dom[i].weight;
      half = half / 2.0;
      if (nd <= 30) {
        /* LPTDomainSplitter (DomainSplitter.scala:86-110) */
        qsort(dom, (size_t)nd, sizeof(vw_pair), cmp_vw_weight_desc);
        double left = 0.0, right = 0.0;
        int32_t *rs = (int32_t *)malloc(sizeof(int32_t) * (size_t)nd);
        int nr = 0;
        for (int i = 0; i < nd; ++i) {
          if (left >= right) { rs[nr++] = dom[i].value; right += dom[i].weight; }
          else left += dom[i].weight;
        }
        qsort(rs, (size_t)nr, sizeof(int32_t), cmp_i32);
        t->kind[node] = 1;
        sets[node] = rs; set_n[node] = nr;
      } else {
        /* RanDomainSplitter (DomainSplitter.scala:57-75) */
        qsort(dom, (size_t)nd, sizeof(vw_pair), cmp_vw_value);
        double cum = 0.0;
        int i = 0;
        while (cum <= half && i < nd - 1) { cum += dom[i].weight; ++i; }
        t->kind[node] = 0;
        t->split[node] = dom[i].value;
      }
      free(dom);
      /* MutableBST.splitNode (MutableBST.scala:87-111) */
      t->attr[node] = attr;
      t->leaf_no[2 * node + 1] = t->leaf_no[node];
      t->leaf_no[2 * node + 2] = t->n_leaves;
      t->n_leaves += 1;
    }
  }
  free(node_of);
  int total = 0;
  for (int n = 0; n < n_nodes; ++n) { t->set_ptr[n] = total; total += set_n[n]; }
  t->set_ptr[n_nodes] = total;
  free(t->set_val);
  t->set_val = (int32_t *)malloc(sizeof(int32_t) * (size_t)(total ? total : 1));
  t->set_len = total; t->set_cap = total ? total : 1;
  for (int n = 0; n < n_nodes; ++n) {
    if (set_n[n]) memcpy(t->set_val + t->set_ptr[n], sets[n], sizeof(int32_t) * (size_t)set_n[n]);
    free(sets[n]);
  }
  free(sets); free(set_n);
  return t;
}

orc_kdtree *orc_kdtree_from_arrays(int n_nodes, const int32_t *attr, const int32_t *kind, const int32_t *split,
                                   const int32_t *set_ptr, const int32_t *set_val, const int32_t *leaf_no) {
  orc_kdtree *t = tree_alloc(n_nodes);
  memcpy(t->attr, attr, sizeof(int32_t) * (size_t)n_nodes);
  memcpy(t->kind, kind, sizeof(int32_t) * (size_t)n_nodes);
  memcpy(t->split, split, sizeof(int32_t) * (size_t)n_nodes);
  memcpy(t->set_ptr, set_ptr, sizeof(int32_t) * ((size_t)n_nodes + 1));
  memcpy(t->leaf_no, leaf_no, sizeof(int32_t) * (size_t)n_nodes);
  int total = set_ptr[n_nodes];
  free(t->set_val);
  t->set_val = (int32_t *)malloc(sizeof(int32_t) * (size_t)(total ? total : 1));
  if (total) memcpy(t->set_val, set_val, sizeof(int32_t) * (size_t)total);
  t->set_len = total;
  int nl = 0;
  for (int n = 0; n < n_nodes; ++n) if (leaf_no[n] + 1 > nl && attr[n] < 0) nl = leaf_no[n] + 1;
  t->n_leaves = nl;
  return t;
}

void orc_kdtree_export(const orc_kdtree *t, int32_t *attr, int32_t *kind, int32_t *split, int32_t *set_ptr,
                       int32_t *set_val, int32_t *leaf_no) {
  memcpy(attr, t->attr, sizeof(int32_t) * (size_t)t->n_nodes);
  memcpy(kind, t->kind, sizeof(int32_t) * (size_t)t->n_nodes);
  memcpy(split, t->split, sizeof(int32_t) * (size_t)t->n_nodes);
  memcpy(set_ptr, t->set_ptr, sizeof(int32_t) * ((size_t)t->n_nodes + 1));
  if (t->set_len) memcpy(set_val, t->set_val, sizeof(int32_t) * (size_t)t->set_len);
  memcpy(leaf_no, t->leaf_no, sizeof(int32_t) * (size_t)t->n_nodes);
}

/* ------------------------------------------------------------------------------------------ */
/* Model / state                                                                                */
/* ------------------------------------------------------------------------------------------ */



orc_model *orc_model_create(int A, int F, orc_index *const *idx, const double *alpha, const double *beta,
                            const orc_kdtree *tree, uint64_t seed) {
  orc_model *m = (orc_model *)calloc(1, sizeof(orc_model));
  m->A = A; m->F = F; m->seed = seed; m->tree = tree;
  m->idx = (orc_index **)malloc(sizeof(orc_index *) * (size_t)A);
  m->alpha = (double *)malloc(sizeof(double) * (size_t)A);
  m->beta = (double *)malloc(sizeof(double) * (size_t)A);
  for (int a = 0; a < A; ++a) { m->idx[a] = idx[a]; m->alpha[a] = alpha[a]; m->beta[a] = beta[a]; }
  return m;
}
void orc_model_free(orc_model *m) { if (!m) return; free(m->idx); free(m->alpha); free(m->beta); free(m); }

int orc_invcdf(const double *cdf, int V, double u) {
  /* first v with cdf[v] > u; V-1 when rounding leaves none */
  int lo = 0, hi = V; /* answer in [lo, hi] */
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (cdf[mid] > u) hi = mid; else lo = mid + 1;
  }
  return lo < V ? lo : V - 1;
}

static orc_state *state_alloc(const orc_model *m, int64_t R, int64_t E) {
  orc_state *s = (orc_state *)calloc(1, sizeof(orc_state));
  int A = m->A;
  s->m = m; s->R = R; s->E = E;
  s->x = (int32_t *)malloc(sizeof(int32_t) * (size_t)(R * A + 1));
  s->file = (int32_t *)malloc(sizeof(int32_t) * (size_t)(R + 1));
  s->link = (int32_t *)malloc(sizeof(int32_t) * (size_t)(R + 1));
  s->z = (uint8_t *)malloc((size_t)(R * A + 1));
  s->y = (int32_t *)malloc(sizeof(int32_t) * (size_t)(E * A + 1));
  s->blk = (int32_t *)malloc(sizeof(int32_t) * (size_t)(E + 1));
  s->theta = (double *)malloc(sizeof(double) * (size_t)(A * m->F));
  s->file_sizes = (int64_t *)calloc((size_t)m->F, sizeof(int64_t));
  return s;
}

static void state_finish(orc_state *s) {
  int A = s->m->A;
  memset(s->file_sizes, 0, sizeof(int64_t) * (size_t)s->m->F);
  for (int64_t r = 0; r < s->R; ++r) s->file_sizes[s->file[r]]++;
  for (int64_t e = 0; e < s->E; ++e) s->blk[e] = s->m->tree ? orc_kdtree_leaf(s->m->tree, s->y + e * A) : 0;
}

/* State.deterministic (State.scala:205-334) with a single input split: record i -> entity i mod E,
   entity values copied from the first record, missing values drawn from phi (State.scala:269-281),
   z = (x >= 0 && x != y) (:284-286), extra isolated entities drawn from phi (:296-301),
   theta = prior mean (DistortionProbs.scala:38-40). */
orc_state *orc_state_init(const orc_model *m, int64_t R, const int32_t *x, const int32_t *file, int64_t pop_size) {
  int A = m->A;
  int64_t E = pop_size > 0 ? pop_size : R;
  orc_state *s = state_alloc(m, R, E);
  memcpy(s->x, x, sizeof(int32_t) * (size_t)(R * A));
  memcpy(s->file, file, sizeof(int32_t) * (size_t)R);
  for (int64_t e = 0; e < E; ++e) {
    for (int a = 0; a < A; ++a) {
      int32_t v = (e < R) ? x[e * A + a] : -1;
      if (v < 0) {
        double u[2];
        orc_uniform2(m->seed, ORC_PHASE_INIT, 0, (uint32_t)e, (uint32_t)a, u);
        v = orc_invcdf(m->idx[a]->cdf, m->idx[a]->V, u[1]);
      }
      s->y[e * A + a] = v;
    }
  }
  for (int64_t r = 0; r < R; ++r) {
    int64_t e = r % E;
    s->link[r] = (int32_t)e;
    for (int a = 0; a < A; ++a) {
      int32_t xv = x[r * A + a];
      s->z[r * A + a] = (uint8_t)((xv >= 0) && (xv != s->y[e * A + a]));
    }
  }
  for (int a = 0; a < A; ++a)
    for (int f = 0; f < m->F; ++f) s->theta[a * m->F + f] = m->alpha[a] / (m->alpha[a] + m->beta[a]);
  s->iteration = 0;
  state_finish(s);
  return s;
}

orc_state *orc_state_from_arrays(const orc_model *m, int64_t R, int64_t E, const int32_t *x, const int32_t *file,
                                 const uint8_t *z, const int32_t *link, const int32_t *y, const double *theta,
                                 int64_t iteration) {
  int A = m->A;
  orc_state *s = state_alloc(m, R, E);
  memcpy(s->x, x, sizeof(int32_t) * (size_t)(R * A));
  memcpy(s->file, file, sizeof(int32_t) * (size_t)R);
  memcpy(s->z, z, (size_t)(R * A));
  memcpy(s->link, link, sizeof(int32_t) * (size_t)R);
  memcpy(s->y, y, sizeof(int32_t) * (size_t)(E * A));
  memcpy(s->theta, theta, sizeof(double) * (size_t)(A * m->F));
  s->iteration = iteration;
  state_finish(s);
  return s;
}

void orc_state_free(orc_state *s) {
  if (!s) return;
  free(s->x); free(s->file); free(s->link); free(s->z); free(s->y); free(s->blk); free(s->theta);
  free(s->file_sizes); free(s);
}
int64_t orc_state_R(const orc_state *s) { return s->R; }
int64_t orc_state_E(const orc_state *s) { return s->E; }
int64_t orc_state_iteration(const orc_state *s) { return s->iteration; }
const int32_t *orc_state_y(const orc_state *s) { return s->y; }
const int32_t *orc_state_link(const orc_state *s) { return s->link; }
const uint8_t *orc_state_z(const orc_state *s) { return s->z; }
const int32_t *orc_state_block(const orc_state *s) { return s->blk; }
const double *orc_state_theta(const orc_state *s) { return s->theta; }

/* CSR entity -> linked records (ascending record id); LinksIndex, GU:84-119 */
static void build_links_csr(const orc_state *s, int64_t **ptr_out, int64_t **rec_out) {
  int64_t *ptr = (int64_t *)calloc((size_t)s->E + 2, sizeof(int64_t));
  int64_t *rec = (int64_t *)malloc(sizeof(int64_t) * (size_t)(s->R + 1));
  for (int64_t r = 0; r < s->R; ++r) ptr[s->link[r] + 1]++;
  for (int64_t e = 0; e < s->E; ++e) ptr[e + 1] += ptr[e];
  int64_t *fill = (int64_t *)malloc(sizeof(int64_t) * (size_t)(s->E + 1));
  memcpy(fill, ptr, sizeof(int64_t) * (size_t)(s->E + 1));
  for (int64_t r = 0; r < s->R; ++r) rec[fill[s->link[r]]++] = r;
  free(fill);
  *ptr_out = ptr; *rec_out = rec;
}

/* updateSummaryVariables, GU:219-301 (literal: log() of each probability, sequential accumulation) */
void orc_state_summary(const orc_state *s, orc_summary_head *head, int64_t *agg_dist, int64_t *rec_dist) {
  const orc_model *m = s->m;
  int A = m->A, F = m->F;
  int64_t *ptr, *rec;
  build_links_csr(s, &ptr, &rec);
  memset(agg_dist, 0, sizeof(int64_t) * (size_t)(A * F));
  memset(rec_dist, 0, sizeof(int64_t) * (size_t)(A + 1));
  double ll = 0.0;
  int64_t isolates = 0;
  for (int64_t e = 0; e < s->E; ++e) {
    const int32_t *ye = s->y + e * A;
    for (int a = 0; a < A; ++a) ll += log(m->idx[a]->phi[ye[a]]); /* GU:234-237, 271-274 */
    if (ptr[e] == ptr[e + 1]) { ++isolates; continue; }            /* GU:267-269 */
    for (int64_t p = ptr[e]; p < ptr[e + 1]; ++p) {
      int64_t r = rec[p];
      int nd = 0;
      for (int a = 0; a < A; ++a) {
        if (!s->z[r * A + a]) continue;
        ++nd;
        agg_dist[a * F + s->file[r]]++; /* GU:244-246: counts missing attributes too */
        int32_t xv = s->x[r * A + a];
        double prob = 1.0;
        if (xv >= 0) {
          const orc_index *ix = m->idx[a];
          if (ix->is_const) prob = ix->phi[xv];
          else prob = ix->phi[xv] * ix->norm[ye[a]] * orc_index_exp_sim_of(ix, xv, ye[a]); /* GU:253-255 */
        }
        ll += log(prob);
      }
      rec_dist[nd]++; /* GU:265 */
    }
  }
  for (int a = 0; a < A; ++a)
    for (int f = 0; f < F; ++f) { /* GU:286-293 */
      double th = s->theta[a * F + f];
      double nd = (double)agg_dist[a * F + f];
      ll += (m->alpha[a] + nd - 1.0) * log(th) + (m->beta[a] + (double)s->file_sizes[f] - nd - 1.0) * log(1.0 - th);
    }
  head->iteration = s->iteration;
  head->num_isolates = isolates;
  head->log_likelihood = ll;
  free(ptr); free(rec);
}

/* ------------------------------------------------------------------------------------------ */
/* theta draw -- updateDistProbs, GU:305-320.  The reference draws Beta variates from           */
/* commons-math3 on the driver MersenneTwister; the protocol keeps the distribution and fixes    */
/* the algorithm: Beta = X/(X+Y), X,Y Gamma by Marsaglia-Tsang, normals by the polar method,     */
/* all uniforms from the Philox stream (phase THETA, id = a*F+f, sub = call counter).            */
/* log and exp are PROTOCOL functions (DESIGN.md 4.5), not libm: the product draws theta on the  */
/* device, and only individually rounded + - * / (and sqrt) are bit-reproducible across CPU and  */
/* GPU.  Recipe: log x = k ln2 + 2s + s R(s^2) with x = 2^k m, m in (sqrt(1/2), sqrt(2)],        */
/* s = (m-1)/(m+1), R(z) = sum_{i=1..11} 2/(2i+1) z^i (Horner from i = 11);                      */
/* exp x = 2^k sum_{n=0..14} r^n/n! with k = floor(x/ln2 + 1/2), r = (x - k ln2_hi) - k ln2_lo.  */
/* ------------------------------------------------------------------------------------------ */

static const double LN2_HI = 0x1.62e42p-1;            /* ln 2 rounded to 21 significant bits */
static const double LN2_LO = 0x1.fdf473de6af28p-22;   /* ln 2 - LN2_HI */

static double u64_as_double(uint64_t b) { double d; memcpy(&d, &b, sizeof d); return d; }
static uint64_t double_as_u64(double d) { uint64_t b; memcpy(&b, &d, sizeof b); return b; }

double orc_det_log(double x) {
  static const double c[11] = { /* 2/3, 2/5, ..., 2/23 */
    2.0 / 3.0, 2.0 / 5.0, 2.0 / 7.0, 2.0 / 9.0, 2.0 / 11.0, 2.0 / 13.0,
    2.0 / 15.0, 2.0 / 17.0, 2.0 / 19.0, 2.0 / 21.0, 2.0 / 23.0 };
  int k = 0;
  uint64_t b = double_as_u64(x);
  if (((b >> 52) & 0x7ff) == 0) { x = x * 0x1p54; k = -54; b = double_as_u64(x); }
  k += (int)((b >> 52) & 0x7ff) - 1023;
  double m = u64_as_double((b & 0xfffffffffffffULL) | 0x3ff0000000000000ULL);
  if (m > 0x1.6a09e667f3bcdp+0) { m = m * 0.5; k += 1; }
  double f = m - 1.0;
  double s = f / (2.0 + f);
  double z = s * s;
  double R = c[10];
  for (int i = 9; i >= 0; --i) { R = R * z; R = R + c[i]; }
  R = R * z;
  double dk = (double)k;
  double t = s * R;
  t = 2.0 * s + t;
  t = t + dk * LN2_LO;
  return dk * LN2_HI + t;
}

double orc_det_exp(double x) {
  if (x > 709.0) return INFINITY;
  if (x < -745.0) return 0.0;
  double t = x * 0x1.71547652b82fep+0 + 0.5;   /* 1/ln 2 */
  long long ki = (long long)t;
  if ((double)ki > t) ki -= 1;
  double kf = (double)ki;
  double r = x - kf * LN2_HI;
  r = r - kf * LN2_LO;
  double fact = 87178291200.0;                 /* 14! */
  double p = 1.0 / fact;
  for (int n = 13; n >= 0; --n) {              /* p = p r + 1/n! */
    fact = fact / (double)(n + 1);
    p = p * r;
    p = p + 1.0 / fact;
  }
  if (ki < -1000) { p = p * u64_as_double((uint64_t)(1023 - 1000) << 52); ki += 1000; }
  return p * u64_as_double((uint64_t)(1023 + ki) << 52);
}

typedef struct { uint64_t seed; uint32_t iter, id, calls; } theta_stream;
static void ts_next(theta_stream *t, double u[2]) { orc_uniform2(t->seed, ORC_PHASE_THETA, t->iter, t->id, t->calls++, u); }
static double ts_normal(theta_stream *t) {
  for (;;) {
    double u[2];
    ts_next(t, u);
    double v1 = 2.0 * u[0] - 1.0, v2 = 2.0 * u[1] - 1.0;
    double s = v1 * v1;
    s = s + v2 * v2;
    if (s >= 1.0 || s == 0.0) continue;
    double q = -2.0 * orc_det_log(s);
    q = q / s;
    return v1 * sqrt(q);
  }
}
static double ts_uniform(theta_stream *t) { double u[2]; ts_next(t, u); return u[0]; }
static double ts_gamma(theta_stream *t, double shape) {
  if (shape < 1.0) {
    double g = ts_gamma(t, shape + 1.0);
    double u = ts_uniform(t);
    return g * orc_det_exp(orc_det_log(u) / shape);
  }
  double d = shape - 1.0 / 3.0;
  double c = 1.0 / sqrt(9.0 * d);
  for (;;) {
    double xn = ts_normal(t);
    double v = 1.0 + c * xn;
    if (v <= 0.0) continue;
    v = v * v * v;
    double u = ts_uniform(t);
    double lhs = orc_det_log(u);
    double t1 = 0.5 * xn;
    t1 = t1 * xn;
    double rhs = t1 + d;
    rhs = rhs - d * v;
    rhs = rhs + d * orc_det_log(v);
    if (lhs < rhs) return d * v;
  }
}

void orc_draw_theta(const orc_model *m, const int64_t *agg_dist, const int64_t *file_sizes, uint32_t iter,
                    double *theta_out) {
  int A = m->A, F = m->F;
  for (int a = 0; a < A; ++a)
    for (int f = 0; f < F; ++f) {
      double nd = (double)agg_dist[a * F + f];
      double s1 = nd + m->alpha[a];                            /* GU:312 */
      double s2 = (double)file_sizes[f] - nd + m->beta[a];     /* GU:313 */
      theta_stream t = {m->seed, iter, (uint32_t)(a * F + f), 0};
      double gx = ts_gamma(&t, s1);
      double gy = ts_gamma(&t, s2);
      theta_out[a * F + f] = gx / (gx + gy);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Categorical draw protocol (replaces DiscreteDist(weights).sample(), GU:394,427,465, which    */
/* builds an alias table per draw).  Candidates in canonical order, padded to a multiple of 32; */
/* a "step" is 32 consecutive candidates (lane l owns candidate step*32+l); steps are grouped    */
/* into at most 32 "chunks" of whole 128-candidate tiles; inside a chunk every lane sums its    */
/* own candidates in step order,                                                                 */
/* the chunk total is a 5-level xor-butterfly sum of the 32 lane sums, chunk totals accumulate   */
/* sequentially and are check-pointed; u*total is located chunk -> lane (Kogge-Stone inclusive   */
/* scan of the lane sums) -> step (sequential walk of that lane).                                */
/* ------------------------------------------------------------------------------------------ */

static double butterfly32(const double *w) {
  double v[32], nv[32];
  memcpy(v, w, sizeof(v));
  for (int d = 16; d >= 1; d >>= 1) {
    for (int l = 0; l < 32; ++l) nv[l] = v[l] + v[l ^ d];
    memcpy(v, nv, sizeof(v));
  }
  return v[0];
}

static void load_step(const double *w, int64_t n, int64_t step, double out[32]) {
  for (int l = 0; l < 32; ++l) {
    int64_t j = step * 32 + l;
    out[l] = j < n ? w[j] : 0.0;
  }
}

/* status: 0 ok, 1 zero/non-finite total mass (reference throws, IndexNonUniformDiscreteDist.scala:71-79) */
int orc_draw_index(const double *w, int64_t n, double u, int *status) {
  if (status) *status = 0;
  /* candidates are laid out in tiles of 128 (= 4 steps); a chunk is a whole number of tiles */
  int64_t ntiles = (n + 127) / 128;
  if (ntiles == 0) { if (status) *status = 1; return -1; }
  int64_t nsteps = 4 * ntiles;          /* steps beyond the last candidate only add zeros */
  int64_t tpc = (ntiles + 31) / 32;     /* tiles per chunk */
  if (tpc < 1) tpc = 1;
  int64_t spc = 4 * tpc;                /* steps per chunk */
  int64_t nchunks = (nsteps + spc - 1) / spc;
  double Q[32];
  double run = 0.0;
  double sw[32], ls[32];
  /* pass 1: per chunk, lane sums (each lane adds its own candidates in step order), chunk total =
     butterfly of the lane sums, running total over chunks check-pointed in Q */
  for (int64_t c = 0; c < nchunks; ++c) {
    int64_t s0 = c * spc, s1 = s0 + spc < nsteps ? s0 + spc : nsteps;
    for (int l = 0; l < 32; ++l) ls[l] = 0.0;
    for (int64_t s = s0; s < s1; ++s) {
      load_step(w, n, s, sw);
      for (int l = 0; l < 32; ++l) ls[l] = ls[l] + sw[l];
    }
    run = run + butterfly32(ls);
    Q[c] = run;
  }
  double total = run;
  if (!(total > 0.0) || isinf(total)) { if (status) *status = 1; return -1; }
  double t = u * total;
  int64_t chunk = nchunks - 1; /* u*total < total always holds for u < 1, so the scan below always hits */
  for (int64_t c = 0; c < nchunks; ++c) if (Q[c] > t) { chunk = c; break; }
  double r = chunk ? Q[chunk - 1] : 0.0;
  /* pass 2a: lane sums of that chunk again, Kogge-Stone inclusive scan over lanes -> lane */
  int64_t s0 = chunk * spc, s1 = s0 + spc < nsteps ? s0 + spc : nsteps;
  for (int l = 0; l < 32; ++l) ls[l] = 0.0;
  for (int64_t s = s0; s < s1; ++s) {
    load_step(w, n, s, sw);
    for (int l = 0; l < 32; ++l) ls[l] = ls[l] + sw[l];
  }
  double P[32], nP[32];
  memcpy(P, ls, sizeof(P));
  for (int d = 1; d < 32; d <<= 1) {
    for (int l = 0; l < 32; ++l) nP[l] = l >= d ? P[l] + P[l - d] : P[l];
    memcpy(P, nP, sizeof(P));
  }
  int lane = -1;
  for (int l = 0; l < 32; ++l) if (r + P[l] > t) { lane = l; break; }
  if (lane < 0) for (int l = 31; l >= 0; --l) if (ls[l] > 0.0) { lane = l; break; } /* scan vs butterfly rounding */
  if (lane < 0) lane = 0;
  double base = lane ? r + P[lane - 1] : r;
  /* pass 2b: walk that lane's candidates of the chunk in step order */
  double cum = 0.0;
  int64_t step = -1, last_pos = -1;
  for (int64_t s = s0; s < s1; ++s) {
    int64_t j = s * 32 + lane;
    double wj = j < n ? w[j] : 0.0;
    cum = cum + wj;
    if (wj > 0.0) last_pos = s;
    if (base + cum > t) { step = s; break; }
  }
  if (step < 0) step = last_pos >= 0 ? last_pos : s0;
  int64_t j = step * 32 + lane;
  if (j >= n) j = n - 1;
  return (int)j;
}

/* ------------------------------------------------------------------------------------------ */
/* Link update                                                                                  */
/* ------------------------------------------------------------------------------------------ */

/* literal restatement: updateEntityIdCollapsed GU:363-395 (PCG-II) and updateEntityIdSeq GU:434-466
   (dense form of the PCG-I / Gibbs conditional, GU:399-430) */
void orc_ref_link_weights(const orc_state *s, int64_t r, int sampler, const int32_t *cand, int64_t n_cand,
                          double *w_out) {
  const orc_model *m = s->m;
  int A = m->A, F = m->F;
  int f = s->file[r];
  for (int64_t j = 0; j < n_cand; ++j) {
    const int32_t *ye = s->y + (int64_t)cand[j] * A;
    double weight = 1.0;
    if (sampler == ORC_PCG_II) {
      for (int a = 0; a < A; ++a) {
        int32_t xv = s->x[r * A + a];
        if (xv < 0) continue; /* GU:373-375 */
        const orc_index *ix = m->idx[a];
        double px = ix->phi[xv];
        double th = s->theta[a * F + f];
        if (ix->is_const) weight = weight * (((xv == ye[a]) ? 1.0 - th : 0.0) + th * px); /* GU:384-385 */
        else weight = weight * (((xv == ye[a]) ? 1.0 - th : 0.0) +
                                th * px * ix->norm[ye[a]] * orc_index_exp_sim_of(ix, xv, ye[a])); /* GU:387-389 */
      }
    } else {
      for (int a = 0; a < A && weight > 0; ++a) { /* GU:444 */
        int32_t xv = s->x[r * A + a];
        if (xv < 0) continue;
        const orc_index *ix = m->idx[a];
        if (!s->z[r * A + a]) { if (xv != ye[a]) weight = 0.0; } /* GU:449-450 */
        else if (ix->is_const) weight *= ix->phi[xv];              /* GU:455 */
        else weight *= ix->norm[ye[a]] * orc_index_exp_sim_of(ix, xv, ye[a]) * ix->phi[xv]; /* GU:457 */
      }
    }
    w_out[j] = weight;
  }
}

/* per-record constants of the protocol weights */
typedef struct {
  int32_t x;
  int kind;       /* 0 skip, 1 const compare, 2 non-const sparse row, 3 missing non-const, 4 must-match */
  double rmatch;  /* multiplier when y == x (kinds 1, 2)                                              */
} rec_attr_t;

static void prep_record(const orc_state *s, int64_t r, int sampler, rec_attr_t *ra) {
  const orc_model *m = s->m;
  int A = m->A, F = m->F, f = s->file[r];
  for (int a = 0; a < A; ++a) {
    const orc_index *ix = m->idx[a];
    int32_t xv = s->x[r * A + a];
    ra[a].x = xv; ra[a].kind = 0; ra[a].rmatch = 1.0;
    if (sampler == ORC_PCG_II) {
      if (xv < 0) { ra[a].kind = ix->is_const ? 0 : 3; continue; }
      double th = s->theta[a * F + f];
      double d = th * ix->phi[xv];
      if (ix->is_const) { ra[a].kind = 1; ra[a].rmatch = 1.0 + (1.0 - th) / d; ra[a].rmatch = (ra[a].rmatch - 1.0) + 1.0; }
      else {
        d = d * ix->norm[xv];
        double ediag = 1.0;
        row_find(ix, xv, xv, &ediag);
        ra[a].kind = 2; ra[a].rmatch = ediag + (1.0 - th) / d;
        /* the kernels keep (rmatch - 1) and rebuild rmatch as fl(that + 1): the identity below ~2^53 */
        ra[a].rmatch = (ra[a].rmatch - 1.0) + 1.0;
      }
    } else {
      if (xv < 0) continue;
      if (!s->z[r * A + a]) ra[a].kind = 4;
      else if (!ix->is_const) ra[a].kind = 2; /* rmatch unused: the stored diagonal is used */
    }
  }
}

static double entity_norm_product(const orc_state *s, const int32_t *ye) {
  const orc_model *m = s->m;
  double nprod = 1.0;
  for (int a = 0; a < m->A; ++a)
    if (!m->idx[a]->is_const) nprod = nprod * m->idx[a]->norm[ye[a]];
  return nprod;
}

/* Protocol weights.  PCG-II: w = N(e) * prod_a rho_a(x_a, y_a) where N(e) = prod_{non-const a} n_a(y_a)
   and rho_a = [GU:384-389 factor] / (theta*phi(x_a)*n_a(y_a)); the record-constant prod_a theta*phi(x_a)
   cancels in the categorical.  PCG-I/Gibbs: GU:444-459 with the record-constant phi(x_a) dropped. */
static double protocol_weight(const orc_state *s, int sampler, const rec_attr_t *ra, const int32_t *ye, double nprod) {
  const orc_model *m = s->m;
  int A = m->A;
  double w;
  /* multiplication order of the protocol (DESIGN.md 4.1): passes over the attributes, each in attribute order */
  if (sampler == ORC_PCG_II) {
    double c = 1.0; /* (i) exact matches: the constant attributes form their own product, applied to N(e) once */
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 1 && ye[a] == ra[a].x) c = c * ra[a].rmatch;
    w = nprod * c;
    for (int a = 0; a < A; ++a) { /* (ii) non-constant attributes, one factor each: equal, or similar but different */
      double e;
      if (ra[a].kind != 2) continue;
      if (ye[a] == ra[a].x) w = w * ra[a].rmatch;
      else if (row_find(m->idx[a], ra[a].x, ye[a], &e)) w = w * e;
    }
    for (int a = 0; a < A; ++a) /* (iii) missing record attributes */
      if (ra[a].kind == 3) w = w * m->idx[a]->invnorm[ye[a]];
  } else {
    w = 1.0;
    for (int a = 0; a < A; ++a)
      if (ra[a].kind == 4 && ye[a] != ra[a].x) return 0.0;
    for (int a = 0; a < A; ++a) /* (i) normalisations */
      if (ra[a].kind == 2) w = w * m->idx[a]->norm[ye[a]];
    for (int a = 0; a < A; ++a) { /* (ii) similarities (diagonal included) */
      double e;
      if (ra[a].kind == 2 && row_find(m->idx[a], ra[a].x, ye[a], &e)) w = w * e;
    }
  }
  return w;
}

void orc_link_weights(const orc_state *s, int64_t r, int sampler, const int32_t *cand, int64_t n_cand, double *w_out) {
  int A = s->m->A;
  rec_attr_t *ra = (rec_attr_t *)malloc(sizeof(rec_attr_t) * (size_t)A);
  prep_record(s, r, sampler, ra);
  for (int64_t j = 0; j < n_cand; ++j) {
    const int32_t *ye = s->y + (int64_t)cand[j] * A;
    w_out[j] = protocol_weight(s, sampler, ra, ye, entity_norm_product(s, ye));
  }
  free(ra);
}

/* ------------------------------------------------------------------------------------------ */
/* Entity-value update                                                                          */
/* ------------------------------------------------------------------------------------------ */

/* base pmf entry and cdf for power k (getSimNormDist, AttributeIndex.scala:197-206); beyond kmax the
   table is evaluated on the fly with the same arithmetic as index_finish */
typedef struct { const orc_index *ix; int k; double zk; const double *pk, *cdf; } base_dist;

static double base_weight(const orc_index *ix, int k, int v) {
  double w = ix->probs[v];
  if (!ix->is_const) for (int i = 0; i < k; ++i) w = w * ix->norm[v];
  return w;
}
static void base_init(base_dist *b, const orc_index *ix, int k) {
  b->ix = ix;
  if (ix->is_const) k = 0;
  b->k = k;
  if (k <= ix->kmax) { b->pk = ix->pk + (size_t)k * ix->V; b->cdf = ix->cdf + (size_t)k * ix->V; b->zk = 0.0; }
  else {
    b->pk = NULL; b->cdf = NULL;
    double z = 0.0;
    for (int v = 0; v < ix->V; ++v) z += base_weight(ix, k, v);
    b->zk = z;
  }
}
static double base_prob(const base_dist *b, int v) { return b->pk ? b->pk[v] : base_weight(b->ix, b->k, v) / b->zk; }
static int base_draw(const base_dist *b, double u) {
  if (b->cdf) return orc_invcdf(b->cdf, b->ix->V, u);
  double c = 0.0;
  for (int v = 0; v < b->ix->V; ++v) { c += base_weight(b->ix, b->k, v) / b->zk; if (c > u) return v; }
  return b->ix->V - 1;
}

/* g_r(v): factor contributed by record r to value v (GU:552-563 collapsed, GU:717-720 non-collapsed).
   Returns 0 when v is not in the record's support (factor 1). */
static int g_factor(const orc_state *s, int64_t r, int a, int collapsed, int v, double *g) {
  const orc_model *m = s->m;
  const orc_index *ix = m->idx[a];
  int32_t xr = s->x[r * m->A + a];
  if (ix->is_const) {
    if (v != xr || !collapsed) return 0;
    double th = s->theta[a * m->F + s->file[r]];
    *g = 1.0 + (1.0 / th - 1.0) / ix->phi[xr]; /* GU:553 */
    return 1;
  }
  double e;
  if (!row_find(ix, xr, v, &e)) return 0;
  if (collapsed && v == xr) {
    double th = s->theta[a * m->F + s->file[r]];
    *g = e + (1.0 / th - 1.0) / (ix->phi[xr] * ix->norm[xr]); /* GU:557,560 */
  } else {
    *g = e;
  }
  return 1;
}

/* support of record r for attribute a as (values, count): the sparse row of x_r, or {x_r} for constant attrs */
static int support_of(const orc_state *s, int64_t r, int a, const int32_t **vals, int32_t *single) {
  const orc_index *ix = s->m->idx[a];
  int32_t xr = s->x[r * s->m->A + a];
  if (ix->is_const) { *single = xr; *vals = single; return 1; }
  *vals = ix->col + ix->rowptr[xr];
  return ix->rowptr[xr + 1] - ix->rowptr[xr];
}
static int in_support(const orc_state *s, int64_t r, int a, int v) {
  const orc_index *ix = s->m->idx[a];
  int32_t xr = s->x[r * s->m->A + a];
  double e;
  if (ix->is_const) return v == xr;
  return row_find(ix, xr, v, &e);
}

/* The mixture of GU:593-597 in the log domain (DESIGN.md 4.3), for the draws whose sum of perturbation weights is not
   finite (a large cluster of agreeing records overflows prod_r g_r(v); beyond the cached powers n(v)^k can underflow):
   log b_k(v) = log probs(v) + k log n(v), log W(v) = log b_k(v) + log(G(v) - 1), or + sum_r log g_r(v) where G
   overflows.  Same candidates, same order and the same det_log / det_exp operations as value_update_log of the
   engine (dblink_b200/csrc/dbl_engine.cu). */
static double lbase_of(const orc_index *ix, double kk, int v) { return orc_det_log(ix->probs[v]) + kk * orc_det_log(ix->norm[v]); }
static int value_draw_log(const orc_state *s, const int64_t *obs, int64_t k, int a, int collapsed, double u0, double u1) {
  const orc_index *ix = s->m->idx[a];
  const double kk = ix->is_const ? 0.0 : (double)k;
  double bmax = lbase_of(ix, kk, 0), Z = 0.0;
  for (int v = 1; v < ix->V; ++v) { double l = lbase_of(ix, kk, v); if (l > bmax) bmax = l; }
  for (int v = 0; v < ix->V; ++v) Z += orc_det_exp(lbase_of(ix, kk, v) - bmax);
  double lmax = 0.0, S = 0.0, target = 0.0, cum = 0.0;
  int any = 0, base = 0, picked = -1, last_pos = -1;
  for (int pass = 0; pass < 3 && !base && picked < 0; ++pass) {
    for (int64_t i = 0; i < k && picked < 0; ++i) {
      const int32_t *vals; int32_t single;
      int nv = support_of(s, obs[i], a, &vals, &single);
      for (int q = 0; q < nv && picked < 0; ++q) {
        int v = vals[q];
        int seen = 0;
        for (int64_t j = 0; j < i && !seen; ++j) seen = in_support(s, obs[j], a, v);
        if (seen) continue;
        double G = 1.0, L = 0.0;
        for (int64_t j = i; j < k; ++j) { double g; if (g_factor(s, obs[j], a, collapsed, v, &g)) { G = G * g; L = L + orc_det_log(g); } }
        if (!(G > 1.0)) continue; /* W(v) = 0 */
        const double lw = lbase_of(ix, kk, v) + (G <= DBL_MAX ? orc_det_log(G - 1.0) : L);
        if (pass == 0) { if (!any || lw > lmax) lmax = lw; any = 1; }
        else if (pass == 1) S += orc_det_exp(lw - lmax);
        else {
          const double W = orc_det_exp(lw - lmax);
          cum += W;
          if (W > 0.0) last_pos = v;
          if (cum > target) picked = v;
        }
      }
    }
    if (pass == 0 && !any) base = 1;
    if (pass == 1) { /* P(base) = Z / (Z + sum W) (GU:593-594) */
      const double d = (lmax + orc_det_log(S)) - (bmax + orc_det_log(Z));
      base = u0 < 1.0 / (1.0 + orc_det_exp(d));
      target = u1 * S;
    }
  }
  if (!base) return picked >= 0 ? picked : last_pos;
  const double bt = u1 * Z;
  double c = 0.0;
  for (int v = 0; v < ix->V; ++v) { c += orc_det_exp(lbase_of(ix, kk, v) - bmax); if (c > bt) return v; }
  return ix->V - 1;
}

/* Protocol draw of y_{e,a}: updateEntityValueCollapsed GU:576-599 / updateEntityValue GU:605-646.
   lrec = linked records (ascending id), nl = their count. */
static int value_draw(const orc_state *s, const int64_t *lrec, int64_t nl, int a, int sampler, double u0, double u1) {
  const orc_model *m = s->m;
  const orc_index *ix = m->idx[a];
  int A = m->A;
  int collapsed = (sampler == ORC_PCG_I || sampler == ORC_PCG_II);
  /* observed linked records (GU:582 / 610) */
  int64_t k = 0;
  int64_t *obs = (int64_t *)malloc(sizeof(int64_t) * (size_t)(nl + 1));
  for (int64_t i = 0; i < nl; ++i) if (s->x[lrec[i] * A + a] >= 0) obs[k++] = lrec[i];
  base_dist b;
  int result;
  if (k == 0) { base_init(&b, ix, 0); result = base_draw(&b, u1); free(obs); return result; } /* GU:588-589 */
  if (!collapsed) {
    for (int64_t i = 0; i < k; ++i) /* GU:619-630 */
      if (!s->z[obs[i] * A + a]) { result = s->x[obs[i] * A + a]; free(obs); return result; }
    if (ix->is_const) { base_init(&b, ix, 0); result = base_draw(&b, u1); free(obs); return result; } /* GU:633-634 */
  }
  base_init(&b, ix, (int)k); /* GU:584-586 */
  double total = 0.0;
  int picked = -1, last_pos = -1;
  double target = 0.0, cum = 0.0;
  for (int pass = 0; pass < 2; ++pass) {
    for (int64_t i = 0; i < k; ++i) {
      const int32_t *vals; int32_t single;
      int nv = support_of(s, obs[i], a, &vals, &single);
      if (!collapsed && ix->is_const) nv = 0;
      for (int q = 0; q < nv; ++q) {
        int v = vals[q];
        int seen = 0;
        for (int64_t j = 0; j < i && !seen; ++j) seen = in_support(s, obs[j], a, v);
        if (seen) continue;
        double G = 1.0;
        for (int64_t j = i; j < k; ++j) { double g; if (g_factor(s, obs[j], a, collapsed, v, &g)) G = G * g; }
        double W = base_prob(&b, v) * (G - 1.0); /* GU:567 / 724 */
        if (pass == 0) total += W;
        else {
          cum += W;
          if (W > 0.0) last_pos = v;
          if (picked < 0 && cum > target) picked = v;
        }
      }
    }
    if (pass == 0) {
      if (!isfinite(total)) { result = value_draw_log(s, obs, k, a, collapsed, u0, u1); free(obs); return result; }
      if (u0 < 1.0 / (1.0 + total)) { result = base_draw(&b, u1); free(obs); return result; } /* GU:593-594 */
      target = u1 * total;
    }
  }
  if (picked < 0) picked = last_pos;
  if (picked < 0) picked = base_draw(&b, u1);
  free(obs);
  return picked;
}

int orc_value_draw(const orc_state *s, int64_t e, int a, int sampler, double u0, double u1) {
  int64_t *ptr, *rec;
  build_links_csr(s, &ptr, &rec);
  int v = value_draw(s, rec + ptr[e], ptr[e + 1] - ptr[e], a, sampler, u0, u1);
  free(ptr); free(rec);
  return v;
}

/* literal full-domain conditional for distribution tests.  PCG-*: p(v) ~ B_k(v) prod_r g_r(v), i.e. the
   mixture of GU:593-597 written out; Gibbs: GU:619-643; Gibbs-Sequential: GU:661-695. */
void orc_ref_value_pmf(const orc_state *s, int64_t e, int a, int sampler, double *pmf) {
  const orc_model *m = s->m;
  const orc_index *ix = m->idx[a];
  int A = m->A, V = ix->V;
  int collapsed = (sampler == ORC_PCG_I || sampler == ORC_PCG_II);
  int64_t *ptr, *rec;
  build_links_csr(s, &ptr, &rec);
  int64_t k = 0, nl = ptr[e + 1] - ptr[e];
  int64_t *obs = (int64_t *)malloc(sizeof(int64_t) * (size_t)(nl + 1));
  for (int64_t i = 0; i < nl; ++i) if (s->x[rec[ptr[e] + i] * A + a] >= 0) obs[k++] = rec[ptr[e] + i];
  int forced = -1;
  if (!collapsed) for (int64_t i = 0; i < k && forced < 0; ++i) if (!s->z[obs[i] * A + a]) forced = s->x[obs[i] * A + a];
  /* log p(v), then exp(log p - max): a large cluster overflows the product of its factors */
  double lmax = -HUGE_VAL, z = 0.0;
  for (int v = 0; v < V; ++v) {
    double lp;
    if (forced >= 0) lp = (v == forced) ? 0.0 : -HUGE_VAL;
    else if (k == 0 || (!collapsed && ix->is_const)) lp = log(ix->phi[v]);
    else if (sampler == ORC_GIBBS_SEQ) {
      lp = log(ix->phi[v]);
      for (int64_t i = 0; i < k; ++i) { /* GU:689 */
        int32_t xr = s->x[obs[i] * A + a];
        lp += log(orc_index_exp_sim_of(ix, xr, v) * ix->norm[v] * ix->phi[xr]);
      }
    } else {
      lp = log(ix->probs[v]) + (ix->is_const ? 0.0 : (double)k * log(ix->norm[v]));
      for (int64_t i = 0; i < k; ++i) { double g; if (g_factor(s, obs[i], a, collapsed, v, &g)) lp += log(g); }
    }
    pmf[v] = lp;
    if (lp > lmax) lmax = lp;
  }
  for (int v = 0; v < V; ++v) { pmf[v] = exp(pmf[v] - lmax); z += pmf[v]; }
  for (int v = 0; v < V; ++v) pmf[v] /= z;
  free(obs); free(ptr); free(rec);
}

/* updateDistortions GU:324-359: P(z = 1) */
double orc_ref_dist_prob(const orc_state *s, int64_t r, int a) {
  const orc_model *m = s->m;
  const orc_index *ix = m->idx[a];
  int A = m->A;
  int32_t xv = s->x[r * A + a];
  double th = s->theta[a * m->F + s->file[r]];
  if (xv < 0) return th;                                  /* GU:331-334 */
  int32_t yv = s->y[(int64_t)s->link[r] * A + a];
  if (xv != yv) return 1.0;                               /* GU:352-354 */
  double pr1;
  if (ix->is_const) pr1 = th * ix->phi[xv];               /* GU:343 */
  else pr1 = th * ix->phi[xv] * ix->norm[xv] * orc_index_exp_sim_of(ix, xv, xv); /* GU:345-347 */
  double pr0 = 1.0 - th;
  return (pr1 + pr0 != 0.0) ? pr1 / (pr1 + pr0) : 0.0;    /* GU:349-350 */
}

/* ------------------------------------------------------------------------------------------ */
/* One sweep: State.nextState (State.scala:78-99) -> updatePartition (GU:156-211)               */
/* ------------------------------------------------------------------------------------------ */

typedef struct {
  orc_state *s;
  int sampler, tid, nthreads, status;
  uint32_t it;
  int64_t maxn;
  const int64_t *bptr;
  const int32_t *bent;
  const double *entN;     /* N(e) of bent[i] (block order) */
  const int32_t *ysorted; /* entity rows in block order: row i = entity bent[i] */
  const int64_t *rorder;  /* records grouped by block: consecutive records score the same (cache-resident) table */
  int32_t *newlink;
} link_job;

/* PCG-II weight with the record's sparse similarity rows scattered into dense per-attribute tables (0.0 = not
   similar): the same multiplications in the same order as protocol_weight, one load instead of a binary search per
   (candidate, attribute).  Only the link phase of whole sweeps uses it (full-size parity tests need the speed);
   orc_link_weights keeps the plain form and tests/test_oracle_distribution.py compares the two. */
typedef struct { int n1, n2, n3; int a1[64], a2[64], a3[64]; } kind_lists; /* attributes of kind 1 / 2 / 3, ascending */

static double protocol_weight_pcg2_dense(const orc_model *m, const rec_attr_t *ra, const kind_lists *kl,
                                         double *const *dense, const int32_t *ye, double nprod) {
  double c = 1.0;
  for (int i = 0; i < kl->n1; ++i) { const int a = kl->a1[i]; if (ye[a] == ra[a].x) c = c * ra[a].rmatch; }
  double w = nprod * c;
  for (int i = 0; i < kl->n2; ++i) {
    const int a = kl->a2[i];
    if (ye[a] == ra[a].x) w = w * ra[a].rmatch;
    else {
      const double e = dense[a][ye[a]];
      if (e != 0.0) w = w * e;
    }
  }
  for (int i = 0; i < kl->n3; ++i) { const int a = kl->a3[i]; w = w * m->idx[a]->invnorm[ye[a]]; }
  return w;
}

/* link update of the records tid, tid + nthreads, ...: every record against every entity of its block */
static void *link_worker(void *arg) {
  link_job *jb = (link_job *)arg;
  orc_state *s = jb->s;
  const orc_model *m = s->m;
  const int A = m->A;
  rec_attr_t *ra = (rec_attr_t *)malloc(sizeof(rec_attr_t) * (size_t)A);
  double *w = (double *)malloc(sizeof(double) * (size_t)(jb->maxn + 1));
  double **dense = (double **)calloc((size_t)A, sizeof(double *));
  const int use_dense = (jb->sampler == ORC_PCG_II) && !getenv("ORC_NO_DENSE");
  if (use_dense)
    for (int a = 0; a < A; ++a)
      if (!m->idx[a]->is_const) dense[a] = (double *)calloc((size_t)m->idx[a]->V + 1, sizeof(double));
  const int64_t i0 = s->R * jb->tid / jb->nthreads, i1 = s->R * (jb->tid + 1) / jb->nthreads;
  for (int64_t i = i0; i < i1; ++i) {
    const int64_t r = jb->rorder[i];
    int b = s->blk[s->link[r]];
    const int32_t *cand = jb->bent + jb->bptr[b];
    const int32_t *yrows = jb->ysorted + jb->bptr[b] * A;
    const double *nrows = jb->entN + jb->bptr[b];
    int64_t n = jb->bptr[b + 1] - jb->bptr[b];
    prep_record(s, r, jb->sampler, ra);
    if (use_dense) {
      kind_lists kl;
      kl.n1 = kl.n2 = kl.n3 = 0;
      for (int a = 0; a < A; ++a) {
        if (ra[a].kind == 1) kl.a1[kl.n1++] = a;
        else if (ra[a].kind == 2) kl.a2[kl.n2++] = a;
        else if (ra[a].kind == 3) kl.a3[kl.n3++] = a;
      }
      for (int a = 0; a < A; ++a)
        if (ra[a].kind == 2) {
          const orc_index *ix = m->idx[a];
          for (int q = ix->rowptr[ra[a].x]; q < ix->rowptr[ra[a].x + 1]; ++q) dense[a][ix->col[q]] = ix->expsim[q];
        }
      for (int64_t j = 0; j < n; ++j)
        w[j] = protocol_weight_pcg2_dense(m, ra, &kl, dense, yrows + j * A, nrows[j]);
      for (int a = 0; a < A; ++a)
        if (ra[a].kind == 2) {
          const orc_index *ix = m->idx[a];
          for (int q = ix->rowptr[ra[a].x]; q < ix->rowptr[ra[a].x + 1]; ++q) dense[a][ix->col[q]] = 0.0;
        }
    } else {
      for (int64_t j = 0; j < n; ++j)
        w[j] = protocol_weight(s, jb->sampler, ra, yrows + j * A, nrows[j]);
    }
    double u[2];
    orc_uniform2(m->seed, ORC_PHASE_LINK, jb->it, (uint32_t)r, 0, u);
    int st;
    int j = orc_draw_index(w, n, u[0], &st);
    if (st) { jb->status = 1; jb->newlink[r] = s->link[r]; } else jb->newlink[r] = cand[j];
  }
  for (int a = 0; a < A; ++a) free(dense[a]);
  free(dense); free(w); free(ra);
  return NULL;
}

/* phases (3)-(5) of a sweep over the entities [e0,e1) / records [r0,r1): independent rows, so any split over
   threads gives the same state (every draw has its own counter) */
typedef struct {
  orc_state *s;
  int sampler, phase, tid, nthreads;
  uint32_t it;
  const int64_t *ptr, *rec;
  int32_t *ynew;
} rest_job;

static void rest_values(rest_job *jb, int64_t e0, int64_t e1) {
  orc_state *s = jb->s;
  const orc_model *m = s->m;
  const int A = m->A;
  for (int64_t e = e0; e < e1; ++e)
    for (int a = 0; a < A; ++a) {
      double u[2];
      orc_uniform2(m->seed, ORC_PHASE_VALUE, jb->it, (uint32_t)e, (uint32_t)a, u);
      jb->ynew[e * A + a] = value_draw(s, jb->rec + jb->ptr[e], jb->ptr[e + 1] - jb->ptr[e], a, jb->sampler, u[0], u[1]);
    }
}

static void rest_dist(rest_job *jb, int64_t r0, int64_t r1) {
  orc_state *s = jb->s;
  const orc_model *m = s->m;
  const int A = m->A, F = m->F;
  for (int64_t r = r0; r < r1; ++r)
    for (int a = 0; a < A; ++a) {
      const orc_index *ix = m->idx[a];
      int32_t xv = s->x[r * A + a];
      double th = s->theta[a * F + s->file[r]];
      double u[2];
      orc_uniform2(m->seed, ORC_PHASE_DIST, jb->it, (uint32_t)r, (uint32_t)a, u);
      uint8_t znew;
      if (xv < 0) znew = (uint8_t)(u[0] < th);
      else {
        int32_t yv = s->y[(int64_t)s->link[r] * A + a];
        if (xv != yv) znew = 1;
        else {
          double pr1 = th * ix->phi[xv];
          if (!ix->is_const) {
            double ediag = 1.0;
            row_find(ix, xv, xv, &ediag);
            pr1 = pr1 * ix->norm[xv];
            pr1 = pr1 * ediag;
          }
          double pr0 = 1.0 - th;
          double den = pr1 + pr0;
          double p = (den != 0.0) ? pr1 / den : 0.0;
          znew = (uint8_t)(u[0] < p);
        }
      }
      s->z[r * A + a] = znew;
    }
}

static void rest_blocks(rest_job *jb, int64_t e0, int64_t e1) {
  orc_state *s = jb->s;
  const orc_model *m = s->m;
  for (int64_t e = e0; e < e1; ++e) s->blk[e] = m->tree ? orc_kdtree_leaf(m->tree, s->y + e * m->A) : 0;
}

static void *rest_worker(void *arg) {
  rest_job *jb = (rest_job *)arg;
  const int64_t n = (jb->phase == 1) ? jb->s->R : jb->s->E;
  const int64_t lo = n * jb->tid / jb->nthreads, hi = n * (jb->tid + 1) / jb->nthreads;
  if (jb->phase == 0) rest_values(jb, lo, hi);
  else if (jb->phase == 1) rest_dist(jb, lo, hi);
  else rest_blocks(jb, lo, hi);
  return NULL;
}

static void rest_run(rest_job *proto, int phase, int nthreads) {
  rest_job jobs[256];
  pthread_t th[256];
  if (nthreads < 1) nthreads = 1;
  if (nthreads > 256) nthreads = 256;
  for (int t = 0; t < nthreads; ++t) {
    jobs[t] = *proto;
    jobs[t].phase = phase; jobs[t].tid = t; jobs[t].nthreads = nthreads;
    if (nthreads == 1) rest_worker(&jobs[t]);
    else pthread_create(&th[t], NULL, rest_worker, &jobs[t]);
  }
  if (nthreads > 1) for (int t = 0; t < nthreads; ++t) pthread_join(th[t], NULL);
}

static double wall_s(void) {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* (3) entity values GU:731-755, (4) distortions with the new y GU:205-210,324-359, (5) re-route GU:206;
   sec[0..2] = wall seconds of the three phases (may be NULL) */
static void sweep_rest(orc_state *s, int sampler, uint32_t it, int nthreads, double *sec) {
  const int A = s->m->A;
  int64_t *ptr, *rec;
  double t0 = wall_s();
  build_links_csr(s, &ptr, &rec);
  int32_t *ynew = (int32_t *)malloc(sizeof(int32_t) * (size_t)(s->E * A + 1));
  rest_job jb = {s, sampler, 0, 0, 1, it, ptr, rec, ynew};
  rest_run(&jb, 0, nthreads);
  memcpy(s->y, ynew, sizeof(int32_t) * (size_t)(s->E * A));
  free(ynew); free(ptr); free(rec);
  double t1 = wall_s();
  rest_run(&jb, 1, nthreads);
  double t2 = wall_s();
  rest_run(&jb, 2, nthreads);
  double t3 = wall_s();
  if (sec) { sec[0] = t1 - t0; sec[1] = t2 - t1; sec[2] = t3 - t2; }
}

/* bench only: phases (3)-(5) + the summary pass (GU:219-301) of one sweep on `nthreads` threads, from the current
   links; sec[0..3] = values, distortions, re-route, summary.  Mutates the state like a sweep would. */
void orc_rest_of_sweep_timed(orc_state *s, int sampler, int nthreads, double *sec) {
  const int A = s->m->A, F = s->m->F;
  sweep_rest(s, sampler, (uint32_t)(s->iteration + 1), nthreads, sec);
  double t0 = wall_s();
  orc_summary_head h;
  int64_t *agg = (int64_t *)malloc(sizeof(int64_t) * (size_t)(A * F));
  int64_t *rd = (int64_t *)malloc(sizeof(int64_t) * (size_t)(A + 1));
  orc_state_summary(s, &h, agg, rd);
  free(agg); free(rd);
  if (sec) sec[3] = wall_s() - t0;
  s->iteration += 1;
}

int orc_state_sweep(orc_state *s, int sampler) {
  const orc_model *m = s->m;
  int A = m->A, F = m->F;
  int status = 0;
  uint32_t it = (uint32_t)(s->iteration + 1);
  int nthreads = 1;
  {
    const char *ev = getenv("ORC_THREADS");
    if (ev && atoi(ev) > 1) nthreads = atoi(ev);
    if (nthreads > 256) nthreads = 256;
  }
  /* (1) theta from the previous state's summary (State.scala:83, GU:305-320) */
  double *theta_old = (double *)malloc(sizeof(double) * (size_t)(A * F));
  memcpy(theta_old, s->theta, sizeof(double) * (size_t)(A * F));
  {
    orc_summary_head h;
    int64_t *agg = (int64_t *)malloc(sizeof(int64_t) * (size_t)(A * F));
    int64_t *rd = (int64_t *)malloc(sizeof(int64_t) * (size_t)(A + 1));
    orc_state_summary(s, &h, agg, rd);
    orc_draw_theta(m, agg, s->file_sizes, it, s->theta);
    free(agg); free(rd);
  }
  /* (2) links: every record against every entity of its block, old y / old z (GU:192-198) */
  int nblk = m->tree ? orc_kdtree_num_leaves(m->tree) : 1;
  int64_t *bptr = (int64_t *)calloc((size_t)nblk + 1, sizeof(int64_t));
  for (int64_t e = 0; e < s->E; ++e) bptr[s->blk[e] + 1]++;
  for (int b = 0; b < nblk; ++b) bptr[b + 1] += bptr[b];
  int32_t *bent = (int32_t *)malloc(sizeof(int32_t) * (size_t)(s->E + 1));
  {
    int64_t *fill = (int64_t *)malloc(sizeof(int64_t) * (size_t)(nblk + 1));
    memcpy(fill, bptr, sizeof(int64_t) * (size_t)(nblk + 1));
    for (int64_t e = 0; e < s->E; ++e) bent[fill[s->blk[e]]++] = (int32_t)e; /* ascending id inside a block */
    free(fill);
  }
  /* block-ordered copies of what a record scans (same values, contiguous) and the records grouped by block */
  double *entN = (double *)malloc(sizeof(double) * (size_t)(s->E + 1));
  int32_t *ysorted = (int32_t *)malloc(sizeof(int32_t) * (size_t)(s->E * A + 1));
  for (int64_t i = 0; i < s->E; ++i) {
    memcpy(ysorted + i * A, s->y + (int64_t)bent[i] * A, sizeof(int32_t) * (size_t)A);
    entN[i] = entity_norm_product(s, s->y + (int64_t)bent[i] * A);
  }
  int64_t *rorder = (int64_t *)malloc(sizeof(int64_t) * (size_t)(s->R + 1));
  {
    int64_t *rfill = (int64_t *)calloc((size_t)nblk + 1, sizeof(int64_t));
    for (int64_t r = 0; r < s->R; ++r) rfill[s->blk[s->link[r]] + 1]++;
    for (int b = 0; b < nblk; ++b) rfill[b + 1] += rfill[b];
    for (int64_t r = 0; r < s->R; ++r) rorder[rfill[s->blk[s->link[r]]]++] = r;
    free(rfill);
  }
  int32_t *newlink = (int32_t *)malloc(sizeof(int32_t) * (size_t)(s->R + 1));
  int64_t maxn = 0;
  for (int b = 0; b < nblk; ++b) if (bptr[b + 1] - bptr[b] > maxn) maxn = bptr[b + 1] - bptr[b];
  {
    /* the draws of different records are independent (own counter each): ORC_THREADS > 1 splits the records over
       threads so that full-size states can be checked in seconds; the result does not depend on the split */
    link_job jobs[256];
    pthread_t th[256];
    for (int t = 0; t < nthreads; ++t) {
      link_job *jb = &jobs[t];
      jb->s = s; jb->sampler = sampler; jb->it = it; jb->tid = t; jb->nthreads = nthreads; jb->maxn = maxn;
      jb->bptr = bptr; jb->bent = bent; jb->entN = entN; jb->ysorted = ysorted; jb->rorder = rorder;
      jb->newlink = newlink; jb->status = 0;
      if (nthreads == 1) link_worker(jb);
      else pthread_create(&th[t], NULL, link_worker, jb);
    }
    for (int t = 0; t < nthreads; ++t) {
      if (nthreads > 1) pthread_join(th[t], NULL);
      status |= jobs[t].status;
    }
  }
  free(entN); free(ysorted); free(rorder); free(bent); free(bptr);
  if (status) {
    /* a categorical without mass fails the reference's task (IndexNonUniformDiscreteDist.scala:78-79): no new
       state exists afterwards -- the sweep is abandoned and the state is the one before the call */
    memcpy(s->theta, theta_old, sizeof(double) * (size_t)(A * F));
    free(theta_old); free(newlink);
    return status;
  }
  free(theta_old);
  memcpy(s->link, newlink, sizeof(int32_t) * (size_t)s->R);
  free(newlink);
  /* (3)-(5): entity values, distortions, re-route */
  sweep_rest(s, sampler, it, nthreads, NULL);
  s->iteration += 1;
  return 0;
}

/* ------------------------------------------------------------------------------------------ */
/* Alias sampler -- random/AliasSampler.scala:49-118 (kept for the reference-style CPU baseline */
/* and for the error conventions pinned by AliasSamplerTest.scala:46-62)                        */
/* ------------------------------------------------------------------------------------------ */

int orc_alias_build(const double *w, int n, double *prob, int32_t *alias) {
  double total = 0.0;
  for (int i = 0; i < n; ++i) {
    if (w[i] < 0 || isinf(w[i]) || isnan(w[i])) return -1; /* AliasSampler.scala:58-61 */
    total += w[i];
  }
  if (!(total > 0.0)) return -2; /* :76 */
  int32_t *work = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n ? n : 1));
  int small = 0, large = n;
  for (int i = 0; i < n; ++i) {
    prob[i] = w[i] * n / total; /* :78 */
    alias[i] = 0;
    if (prob[i] < 1.0) work[small++] = i; else work[--large] = i; /* :89-98 */
  }
  if (small > 0) {
    small = 0;
    while (small < n && large < n) { /* :101-110 */
      int l = work[small++];
      int g = work[large];
      alias[l] = g;
      prob[g] = (prob[g] + prob[l]) - 1.0;
      if (prob[g] < 1.0) large += 1;
    }
  }
  for (int i = 0; i < n; ++i) prob[i] += i; /* :113-117 */
  free(work);
  return 0;
}

int orc_alias_sample(const double *prob, const int32_t *alias, int n, double u) {
  double U = u * n; /* AliasSampler.scala:33-37 */
  int i = (int)U;
  if (i >= n) i = n - 1;
  return (U < prob[i]) ? i : alias[i];
}
