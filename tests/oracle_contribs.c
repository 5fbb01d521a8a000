/* oracle_contribs.c — CPU restatement of libxgboost 1.6.0's per-feature contributions (test infrastructure only;
 * nothing in the product may include, link or call it).  It works on the model and DMatrix the C oracle
 * (oracle/qc_oracle.c) loads and builds: the caller passes its orc_model / orc_dmatrix pointers.  Parity unpinned,
 * like the rest of the oracle.  Built by tests/oracle_contribs.py with the oracle's flags (-ffp-contract=off: every
 * float32 operation a separate IEEE operation). */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "qc_oracle.h"

static _Thread_local char g_err[512];
const char *oc_last_error(void) { return g_err; }
#define FAIL(ret, ...)                          \
  do {                                          \
    snprintf(g_err, sizeof g_err, __VA_ARGS__); \
    return ret;                                 \
  } while (0)

/* one dense feature slot, as oracle/qc_oracle.c fills it: flag -1 = missing */
typedef union {
  float fvalue;
  int32_t flag;
} fvec_entry;
/* ======================================================================================
 * Per-feature contributions — libxgboost 1.6.0 CPUPredictor::PredictContribution
 * (src/predictor/cpu_predictor.cc) with RegTree::CalculateContributions (recursive path-dependent TreeShap:
 * ExtendPath / UnwindPath / UnwoundPathSum, src/tree/tree_model.cc), CalculateContributionsApprox and
 * FillNodeMeanValue, all in float32 and in libxgboost's order.  Per row and tree a zeroed per-tree vector is filled
 * and added column by column; base_score goes to the bias column last.
 * ==================================================================================== */
typedef struct {
  int feature_index;
  float zero_fraction, one_fraction, pweight;
} orc_path_elem;

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

static void extend_path(orc_path_elem *up, unsigned d, float zf, float of, int fi) {
  up[d].feature_index = fi;
  up[d].zero_fraction = zf;
  up[d].one_fraction = of;
  up[d].pweight = d == 0 ? 1.0f : 0.0f;
  for (int i = (int)d - 1; i >= 0; i--) {
    up[i + 1].pweight += of * up[i].pweight * (i + 1) / (float)(d + 1);
    up[i].pweight = zf * up[i].pweight * (d - i) / (float)(d + 1);
  }
}

static void unwind_path(orc_path_elem *up, unsigned d, unsigned pi) {
  const float of = up[pi].one_fraction, zf = up[pi].zero_fraction;
  float next = up[d].pweight;
  for (int i = (int)d - 1; i >= 0; --i) {
    if (of != 0) {
      const float tmp = up[i].pweight;
      up[i].pweight = next * (d + 1) / (float)((i + 1) * of);
      next = tmp - up[i].pweight * zf * (d - i) / (float)(d + 1);
    } else {
      up[i].pweight = (up[i].pweight * (d + 1)) / (float)((d - i) * zf);
    }
  }
  for (unsigned i = pi; i < d; ++i) {
    up[i].feature_index = up[i + 1].feature_index;
    up[i].zero_fraction = up[i + 1].zero_fraction;
    up[i].one_fraction = up[i + 1].one_fraction;
  }
}

static float unwound_path_sum(const orc_path_elem *up, unsigned d, unsigned pi) {
  const float of = up[pi].one_fraction, zf = up[pi].zero_fraction;
  float next = up[d].pweight, total = 0;
  for (int i = (int)d - 1; i >= 0; --i) {
    if (of != 0) {
      const float tmp = next * (d + 1) / (float)((i + 1) * of);
      total += tmp;
      next = up[i].pweight - tmp * zf * ((d - i) / (float)(d + 1));
    } else {
      total += (up[i].pweight / zf) / ((d - i) / (float)(d + 1));
    }
  }
  return total;
}

static void tree_shap(const orc_tree *t, const fvec_entry *fv, float *phi, int nid, unsigned depth, orc_path_elem *parent_path,
                      float parent_zero, float parent_one, int parent_feature) {
  const orc_node *nd = &t->nodes[nid];
  orc_path_elem *up = parent_path + depth + 1;
  memcpy(up, parent_path, sizeof(orc_path_elem) * (depth + 1));
  extend_path(up, depth, parent_zero, parent_one, parent_feature);
  if (nd->cleft == -1) {
    for (unsigned i = 1; i <= depth; ++i) {
      const float w = unwound_path_sum(up, depth, i);
      const orc_path_elem *el = &up[i];
      phi[el->feature_index] += w * (el->one_fraction - el->zero_fraction) * nd->info;
    }
    return;
  }
  const int split = (int)(nd->sindex & 0x7FFFFFFFu);
  int hot;
  if (fv[split].flag == -1) hot = (nd->sindex >> 31) ? nd->cleft : nd->cright;
  else if (fv[split].fvalue < nd->info) hot = nd->cleft;
  else hot = nd->cright;
  const int cold = hot == nd->cleft ? nd->cright : nd->cleft;
  const float w = t->stats[nid].sum_hess;
  const float hot_zero = t->stats[hot].sum_hess / w, cold_zero = t->stats[cold].sum_hess / w;
  float in_zero = 1, in_one = 1;
  unsigned pi = 0;
  for (; pi <= depth; ++pi)
    if (up[pi].feature_index == split) break;
  if (pi != depth + 1) {
    in_zero = up[pi].zero_fraction;
    in_one = up[pi].one_fraction;
    unwind_path(up, depth, pi);
    depth -= 1;
  }
  tree_shap(t, fv, phi, hot, depth + 1, up, hot_zero * in_zero, in_one, split);
  tree_shap(t, fv, phi, cold, depth + 1, up, cold_zero * in_zero, 0, split);
}

static void tree_approx(const orc_tree *t, const fvec_entry *fv, const float *mean, float *phi, uint32_t nf) {
  unsigned split = 0;
  float node_value = mean[0];
  phi[nf] += node_value;
  if (t->nodes[0].cleft == -1) return;
  int nid = 0;
  while (t->nodes[nid].cleft != -1) {
    const orc_node *nd = &t->nodes[nid];
    split = nd->sindex & 0x7FFFFFFFu;
    if (fv[split].flag == -1) nid = (nd->sindex >> 31) ? nd->cleft : nd->cright;
    else nid = nd->cleft + !(fv[split].fvalue < nd->info);
    const float new_value = mean[nid];
    phi[split] += new_value - node_value;
    node_value = new_value;
  }
  phi[split] += t->nodes[nid].info - node_value;
}

static int tree_max_depth(const orc_tree *t, int nid) {
  if (t->nodes[nid].cleft == -1) return 0;
  const int l = tree_max_depth(t, t->nodes[nid].cleft), r = tree_max_depth(t, t->nodes[nid].cright);
  return 1 + (l > r ? l : r);
}

uint64_t oc_predict_contribs(const orc_model *m, const orc_dmatrix *d, int approximate, unsigned ntree_limit, float *out) {
  if (!m || !d) FAIL(0, "null handle");
  if (d->ncol > m->num_feature && m->num_feature != 0)
    FAIL(0, "Number of columns does not match number of features in booster.");
  int ntree = m->num_trees;
  if (ntree_limit != 0 && (int)ntree_limit < ntree) ntree = (int)ntree_limit;
  const uint32_t nf = m->num_feature;
  const uint64_t ncolumns = (uint64_t)nf + 1;
  for (int t = 0; t < ntree; ++t)
    for (int n = 0; n < m->trees[t].num_nodes; ++n) {
      const float c = m->trees[t].stats[n].sum_hess;
      if (!isfinite(c) || !(c > 0.f)) FAIL(0, "tree %d node %d has cover %g: contributions need positive node covers", t, n, c);
    }
  float **mean = (float **)calloc((size_t)ntree + 1, sizeof(float *));
  int maxd = 0;
  for (int t = 0; t < ntree; ++t) {
    mean[t] = (float *)malloc(sizeof(float) * (size_t)m->trees[t].num_nodes);
    fill_node_mean(&m->trees[t], 0, mean[t]);
    const int dd = tree_max_depth(&m->trees[t], 0);
    if (dd > maxd) maxd = dd;
  }
  const size_t path_cap = (size_t)(maxd + 2) * (size_t)(maxd + 3) / 2 + 1;
#pragma omp parallel
  {
    fvec_entry *fv = (fvec_entry *)malloc(sizeof(fvec_entry) * (nf ? nf : 1));
    float *tc = (float *)malloc(sizeof(float) * ncolumns);
    orc_path_elem *path = (orc_path_elem *)malloc(sizeof(orc_path_elem) * path_cap);
#pragma omp for schedule(dynamic, 1)
    for (int64_t r = 0; r < (int64_t)d->nrow; ++r) {
      memset(fv, 0xFF, sizeof(fvec_entry) * nf);
      for (uint64_t o = d->offset[r]; o < d->offset[r + 1]; ++o)
        if (d->index[o] < nf) fv[d->index[o]].fvalue = d->value[o];
      float *p = out + (uint64_t)r * ncolumns;
      for (uint64_t c = 0; c < ncolumns; ++c) p[c] = 0.f;
      for (int t = 0; t < ntree; ++t) {
        for (uint64_t c = 0; c < ncolumns; ++c) tc[c] = 0.f;
        if (approximate) {
          tree_approx(&m->trees[t], fv, mean[t], tc, nf);
        } else {
          tc[nf] += mean[t][0];
          tree_shap(&m->trees[t], fv, tc, 0, 0, path, 1, 1, -1);
        }
        for (uint64_t c = 0; c < ncolumns; ++c) p[c] += tc[c];
      }
      p[nf] += m->base_score;
    }
    free(fv);
    free(tc);
    free(path);
  }
  for (int t = 0; t < ntree; ++t) free(mean[t]);
  free(mean);
  return d->nrow * ncolumns;
}
