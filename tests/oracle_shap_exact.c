/* oracle_shap_exact.c — exact TreeSHAP contributions and SHAP interaction values in extended precision (test
 * infrastructure only; nothing in the product may include, link or call it).  It works on the model and DMatrix the
 * C oracle (oracle/qc_oracle.c) loads and builds, and shares no code with the library or with
 * tests/oracle_contribs.c: the paths come straight from the trees, and each path's Shapley values come from the
 * coefficients of its product game, not from ExtendPath / UnwoundPathSum.  Built by tests/oracle_shap_exact.py.
 *
 * A root-to-leaf path P with leaf value v is a product game over its distinct features: repeated splits on one
 * feature merge into one element j with
 *   o_j  one fraction: a present value x follows every split of j (`x < thr` on a left side, `!(x < thr)` on a right
 *        side); a missing value (also a column >= ncol) follows iff every split of j sends missing values its way;
 *   z_j  zero fraction: the product, root to leaf, of cover(child) / cover(parent) over the splits of j.
 * The library's path tables hold z~ = (float) of the float64 product (forest.cpp build_shap); `exact_z` = 0 uses z~,
 * 1 the product in long double.  With D elements, f(S) = v prod_{j in S} o_j prod_{j not in S} z_j and
 *   phi_e = v (o_e - z_e) W_e,   W_e = sum_k k! (D-1-k)! / D! c_k >= 0,   c = coefficients of prod_{j != e}(z_j + o_j t),
 * c from prefix and suffix products (no division).  Interaction values (libxgboost 1.6.0's conditioned definition):
 *   M[c][k] = 1/2 sum over paths holding c and k of (o_c - z_c) phi_k(P minus c),   M[c][c] = phi_c - sum_{k != c} M[c][k],
 * the bias row and column 0 but M[F][F] = the bias.  The bias is libxgboost's, float32 in its order:
 * ((0 + mean_0(root)) + mean_1(root) + ...) + base_score with FillNodeMeanValue's float32 node means.
 * Each value comes with a magnitude: A_f = sum over paths of |v| W_f (|o_f - z_f| + z_f) for contributions, and
 * 1/2 sum |v| (|o_c - z_c| + z_c) W_k(P minus c) (|o_k - z_k| + z_k) for M[c][k] (A[c][c] = A_c + sum_{k != c} A[c][k]),
 * a bound on what a relative perturbation of every o - z, z and W can move the value by. */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "qc_oracle.h"

typedef long double real;

#define SE_MAXD 64 /* distinct features on one path */

static _Thread_local char g_err[512];
const char *se_last_error(void) { return g_err; }
#define FAIL(ret, ...)                          \
  do {                                          \
    snprintf(g_err, sizeof g_err, __VA_ARGS__); \
    return ret;                                 \
  } while (0)

typedef struct {
  uint32_t feat;
  int miss;           /* AND over the element's splits of (default direction == this side) */
  int split0, nsplit; /* its splits: sp[split0, split0 + nsplit) */
  real zt, z;         /* (float) of the float64 product; the long double product */
} se_elem;

typedef struct {
  real v;
  int D, e0;
} se_path;

typedef struct {
  float thr;
  int right; /* the path takes the right child */
} se_split;

typedef struct {
  se_path *p;
  se_elem *e;
  se_split *sp;
  size_t np, ne, ns, cp, ce, cs;
} se_paths;

static void *grow(void *p, size_t *cap, size_t need, size_t size) {
  if (need <= *cap) return p;
  size_t c = *cap ? *cap : 64;
  while (c < need) c *= 2;
  void *q = realloc(p, c * size);
  if (!q) abort();
  *cap = c;
  return q;
}

/* route[i] = node at depth i, side[i] = 0 left / 1 right of it */
static int leaf_path(const orc_tree *t, const int *route, const unsigned char *side, int depth, int leaf, se_paths *s) {
  int nf = 0;
  uint32_t feats[SE_MAXD];
  for (int i = 0; i < depth; ++i) {
    const uint32_t f = t->nodes[route[i]].sindex & 0x7FFFFFFFu;
    int j = 0;
    while (j < nf && feats[j] != f) ++j;
    if (j == nf) {
      if (nf == SE_MAXD) FAIL(-1, "a path has more than %d distinct features", SE_MAXD);
      feats[nf++] = f;
    }
  }
  s->p = grow(s->p, &s->cp, s->np + 1, sizeof(se_path));
  s->e = grow(s->e, &s->ce, s->ne + (size_t)nf, sizeof(se_elem));
  s->sp = grow(s->sp, &s->cs, s->ns + (size_t)depth, sizeof(se_split));
  se_path *p = &s->p[s->np++];
  p->v = (real)t->nodes[leaf].info;
  p->D = nf;
  p->e0 = (int)s->ne;
  for (int j = 0; j < nf; ++j) {
    se_elem *e = &s->e[s->ne++];
    double zd = 1.0;
    e->feat = feats[j];
    e->miss = 1;
    e->z = 1.0L;
    e->split0 = (int)s->ns;
    e->nsplit = 0;
    for (int i = 0; i < depth; ++i) {
      const orc_node *nd = &t->nodes[route[i]];
      if ((nd->sindex & 0x7FFFFFFFu) != feats[j]) continue;
      const int child = side[i] ? nd->cright : nd->cleft;
      const int dl = (int)(nd->sindex >> 31);
      e->miss &= dl == (side[i] == 0);
      zd *= (double)t->stats[child].sum_hess / (double)t->stats[route[i]].sum_hess;
      e->z *= (real)t->stats[child].sum_hess / (real)t->stats[route[i]].sum_hess;
      s->sp[s->ns].thr = nd->info;
      s->sp[s->ns].right = side[i];
      s->ns++, e->nsplit++;
    }
    e->zt = (real)(float)zd;
  }
  return 0;
}

static int walk(const orc_tree *t, int nid, int *route, unsigned char *side, int depth, int cap, se_paths *s) {
  const orc_node *nd = &t->nodes[nid];
  if (nd->cleft == -1) return leaf_path(t, route, side, depth, nid, s);
  if (depth == cap) FAIL(-1, "a tree is deeper than %d", cap);
  route[depth] = nid;
  for (int sd = 0; sd < 2; ++sd) {
    side[depth] = (unsigned char)sd;
    if (walk(t, sd ? nd->cright : nd->cleft, route, side, depth + 1, cap, s)) return -1;
  }
  return 0;
}

static float fill_node_mean(const orc_tree *t, int nid, float *mean) {
  const orc_node *nd = &t->nodes[nid];
  float r;
  if (nd->cleft == -1) {
    r = nd->info;
  } else {
    r = fill_node_mean(t, nd->cleft, mean) * t->stats[nd->cleft].sum_hess;
    r += fill_node_mean(t, nd->cright, mean) * t->stats[nd->cright].sum_hess;
    r /= t->stats[nid].sum_hess;
  }
  mean[nid] = r;
  return r;
}

/* g_w[D][k] = k! (D-1-k)! / D! = 1 / (D binom(D-1, k)) */
static real g_w[SE_MAXD + 1][SE_MAXD];

static void init_weights(void) {
  for (int D = 1; D <= SE_MAXD; ++D) {
    uint64_t b = 1; /* binom(D-1, k), exact: binom(63, 31) < 2^60 */
    for (int k = 0; k < D; ++k) {
      g_w[D][k] = 1.0L / ((real)D * (real)b);
      b = (uint64_t)((unsigned __int128)b * (unsigned)(D - 1 - k) / (unsigned)(k + 1));
    }
  }
}

/* W[e] for the D elements (o, z): pre[i] = prod_{j < i}(z_j + o_j t), suf[i] = prod_{j >= i}(z_j + o_j t), and
 * W_e = sum_a pre[e]_a sum_b w_{a+b} suf[e+1]_b.  scratch: 2 (SE_MAXD + 1)^2 reals. */
static void path_weights(int D, const real *o, const real *z, real *W, real *scratch) {
  real(*pre)[SE_MAXD + 1] = (real(*)[SE_MAXD + 1])scratch;
  real(*suf)[SE_MAXD + 1] = pre + SE_MAXD + 1;
  pre[0][0] = 1.0L;
  for (int i = 0; i < D; ++i) {
    pre[i + 1][0] = z[i] * pre[i][0];
    for (int a = 1; a <= i; ++a) pre[i + 1][a] = z[i] * pre[i][a] + o[i] * pre[i][a - 1];
    pre[i + 1][i + 1] = o[i] * pre[i][i];
  }
  suf[D][0] = 1.0L;
  for (int i = D - 1; i >= 0; --i) {
    const int n = D - 1 - i; /* degree of suf[i + 1] */
    suf[i][0] = z[i] * suf[i + 1][0];
    for (int a = 1; a <= n; ++a) suf[i][a] = z[i] * suf[i + 1][a] + o[i] * suf[i + 1][a - 1];
    suf[i][n + 1] = o[i] * suf[i + 1][n];
  }
  const real *w = g_w[D];
  for (int e = 0; e < D; ++e) {
    real acc = 0.0L;
    for (int a = 0; a <= e; ++a) {
      real inner = 0.0L;
      for (int b = 0; b <= D - 1 - e; ++b) inner += w[a + b] * suf[e + 1][b];
      acc += pre[e][a] * inner;
    }
    W[e] = acc;
  }
}

static int one_fraction(const se_paths *s, const se_elem *e, const float *x, const unsigned char *present) {
  if (!present[e->feat]) return e->miss;
  const float xv = x[e->feat];
  for (int i = 0; i < e->nsplit; ++i) {
    const int lt = xv < s->sp[e->split0 + i].thr;
    if (s->sp[e->split0 + i].right ? lt : !lt) return 0;
  }
  return 1;
}

/* Contributions (interactions = 0: val / mag [nrow][nf + 1]) or interaction values (interactions = 1: val / mag
 * [nrow][nf + 1][nf + 1]) of the first ntree_limit trees (0: all).  *max_d: the most elements on one path.
 * Returns 0, or -1 with se_last_error(). */
int se_shap(const orc_model *m, const orc_dmatrix *d, unsigned ntree_limit, int exact_z, int interactions, real *val,
            real *mag, int *max_d) {
  if (!m || !d) FAIL(-1, "null handle");
  static int ready = 0;
  if (!ready) init_weights(), ready = 1; /* first call from one thread (the wrapper holds the GIL) */
  int ntree = m->num_trees;
  if (ntree_limit != 0 && (int)ntree_limit < ntree) ntree = (int)ntree_limit;
  const uint32_t nf = m->num_feature;
  const uint64_t nc = (uint64_t)nf + 1, nrow = d->nrow;
  const uint64_t per_row = interactions ? nc * nc : nc;
  for (int t = 0; t < ntree; ++t)
    for (int n = 0; n < m->trees[t].num_nodes; ++n) {
      const float c = m->trees[t].stats[n].sum_hess;
      if (!isfinite(c) || !(c > 0.f)) FAIL(-1, "tree %d node %d has cover %g: contributions need positive node covers", t, n, c);
    }
  /* the bias, float32 in libxgboost's order */
  float bias = 0.f;
  for (int t = 0; t < ntree; ++t) {
    float *mean = malloc(sizeof(float) * (size_t)m->trees[t].num_nodes);
    fill_node_mean(&m->trees[t], 0, mean);
    float tc = 0.f;
    tc += mean[0];
    bias += tc;
    free(mean);
  }
  bias += m->base_score;
  /* the rows, dense */
  float *xs = calloc(nrow * (nf ? nf : 1), sizeof(float));
  unsigned char *pres = calloc(nrow * (nf ? nf : 1), 1);
  for (uint64_t r = 0; r < nrow; ++r)
    for (uint64_t o = d->offset[r]; o < d->offset[r + 1]; ++o)
      if (d->index[o] < nf) xs[r * nf + d->index[o]] = d->value[o], pres[r * nf + d->index[o]] = 1;
  memset(val, 0, sizeof(real) * nrow * per_row);
  memset(mag, 0, sizeof(real) * nrow * per_row);
  *max_d = 0;
  int rc = 0;
  for (int t = 0; t < ntree && rc == 0; ++t) {
    const orc_tree *tr = &m->trees[t];
    se_paths s;
    memset(&s, 0, sizeof s);
    const int cap = tr->num_nodes;
    int *route = malloc(sizeof(int) * (size_t)cap);
    unsigned char *side = malloc((size_t)cap);
    rc = walk(tr, 0, route, side, 0, cap, &s);
    free(route), free(side);
    for (size_t p = 0; p < s.np; ++p)
      if (s.p[p].D > *max_d) *max_d = s.p[p].D;
    for (size_t e = 0; e < s.ne && rc == 0; ++e)
      if (s.e[e].feat >= nf) rc = -1, snprintf(g_err, sizeof g_err, "tree %d splits on feature %u of %u", t, s.e[e].feat, nf);
    if (rc == 0) {
#pragma omp parallel
      {
        real *scratch = malloc(sizeof(real) * 2 * (SE_MAXD + 1) * (SE_MAXD + 1));
        real o[SE_MAXD], z[SE_MAXD], W[SE_MAXD], o2[SE_MAXD], z2[SE_MAXD], W2[SE_MAXD];
#pragma omp for schedule(dynamic, 4)
        for (int64_t r = 0; r < (int64_t)nrow; ++r) {
          real *vr = val + (uint64_t)r * per_row, *ar = mag + (uint64_t)r * per_row;
          const float *x = xs + (uint64_t)r * nf;
          const unsigned char *pr = pres + (uint64_t)r * nf;
          for (size_t p = 0; p < s.np; ++p) {
            const se_path *P = &s.p[p];
            const se_elem *E = s.e + P->e0;
            const int D = P->D;
            const real v = P->v, av = fabsl(v);
            for (int j = 0; j < D; ++j) {
              o[j] = (real)one_fraction(&s, &E[j], x, pr);
              z[j] = exact_z ? E[j].z : E[j].zt;
            }
            if (!interactions) {
              path_weights(D, o, z, W, scratch);
              for (int j = 0; j < D; ++j) {
                vr[E[j].feat] += v * (o[j] - z[j]) * W[j];
                ar[E[j].feat] += av * W[j] * (fabsl(o[j] - z[j]) + z[j]);
              }
              continue;
            }
            path_weights(D, o, z, W, scratch);
            for (int c = 0; c < D; ++c) {
              const uint32_t fc = E[c].feat;
              vr[fc * nc + fc] += v * (o[c] - z[c]) * W[c]; /* phi_c, for the diagonal */
              ar[fc * nc + fc] += av * W[c] * (fabsl(o[c] - z[c]) + z[c]);
              if (D < 2) continue;
              for (int j = 0, k = 0; j < D; ++j)
                if (j != c) o2[k] = o[j], z2[k] = z[j], ++k;
              path_weights(D - 1, o2, z2, W2, scratch);
              const real hc = 0.5L * v * (o[c] - z[c]), ahc = 0.5L * av * (fabsl(o[c] - z[c]) + z[c]);
              for (int j = 0, k = 0; j < D; ++j) {
                if (j == c) continue;
                const uint32_t fk = E[j].feat;
                vr[fc * nc + fk] += hc * W2[k] * (o[j] - z[j]);
                ar[fc * nc + fk] += ahc * W2[k] * (fabsl(o[j] - z[j]) + z[j]);
                ++k;
              }
            }
          }
        }
        free(scratch);
      }
    }
    free(s.p), free(s.e), free(s.sp);
  }
  free(xs), free(pres);
  if (rc) return rc;
  for (uint64_t r = 0; r < nrow; ++r) {
    real *vr = val + r * per_row, *ar = mag + r * per_row;
    if (!interactions) {
      vr[nf] = (real)bias;
      continue;
    }
    /* the diagonal holds phi_c so far: M[c][c] = phi_c - sum_{k != c} M[c][k] */
    for (uint32_t c = 0; c < nf; ++c) {
      real off = 0.0L, aoff = 0.0L;
      for (uint32_t k = 0; k < nf; ++k)
        if (k != c) off += vr[c * nc + k], aoff += ar[c * nc + k];
      vr[c * nc + c] -= off;
      ar[c * nc + c] += aoff;
    }
    vr[nf * nc + nf] = (real)bias;
  }
  return 0;
}
