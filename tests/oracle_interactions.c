/* oracle_interactions.c — CPU restatement of libxgboost 1.6.0's SHAP interaction values (test infrastructure only;
 * nothing in the product may include, link or call it).  It builds on the contributions restatement, which it
 * includes whole (ExtendPath / UnwindPath / UnwoundPathSum, FillNodeMeanValue, CalculateContributionsApprox and the
 * model / DMatrix types of the C oracle), and adds the conditioned TreeShap and the PredictInteractionContributions
 * loop.  Parity unpinned, like the rest of the oracle.  Built by tests/oracle_interactions.py with the flags of
 * tests/oracle_contribs.py (-ffp-contract=off: every float32 operation a separate IEEE operation). */
#include "oracle_contribs.c"

/* RegTree::TreeShap with its condition arguments: condition 0 is plain TreeShap; +1 / -1 fix feature
 * condition_feature present / absent — it is never extended into the path, at its splits the cold branch gets
 * condition fraction 0 (+1) or each branch its cover ratio (-1), and the leaf terms are scaled by the fraction. */
static void tree_shap_cond(const orc_tree *t, const fvec_entry *fv, float *phi, int nid, unsigned depth, orc_path_elem *parent_path,
                           float parent_zero, float parent_one, int parent_feature, int condition, unsigned condition_feature,
                           float condition_fraction) {
  const orc_node *nd = &t->nodes[nid];
  if (condition_fraction == 0) return;
  orc_path_elem *up = parent_path + depth + 1;
  memcpy(up, parent_path, sizeof(orc_path_elem) * (depth + 1));
  if (condition == 0 || condition_feature != (unsigned)parent_feature) extend_path(up, depth, parent_zero, parent_one, parent_feature);
  if (nd->cleft == -1) {
    for (unsigned i = 1; i <= depth; ++i) {
      const float w = unwound_path_sum(up, depth, i);
      const orc_path_elem *el = &up[i];
      phi[el->feature_index] += w * (el->one_fraction - el->zero_fraction) * nd->info * condition_fraction;
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
  float hot_cond = condition_fraction, cold_cond = condition_fraction;
  if (condition > 0 && (unsigned)split == condition_feature) {
    cold_cond = 0;
    depth -= 1;
  } else if (condition < 0 && (unsigned)split == condition_feature) {
    hot_cond *= hot_zero;
    cold_cond *= cold_zero;
    depth -= 1;
  }
  tree_shap_cond(t, fv, phi, hot, depth + 1, up, hot_zero * in_zero, in_one, split, condition, condition_feature, hot_cond);
  tree_shap_cond(t, fv, phi, cold, depth + 1, up, cold_zero * in_zero, 0, split, condition, condition_feature, cold_cond);
}

/* PredictContribution(condition, condition_feature), as oc_predict_contribs does it for condition 0: approximate
 * ignores the condition, and the bias mean is added only without one.  Returns nrow * (num_feature + 1), 0 on error. */
static uint64_t contributions(const orc_model *m, const orc_dmatrix *d, int approximate, unsigned ntree_limit, int condition,
                              unsigned condition_feature, float *out) {
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
          if (condition == 0) tc[nf] += mean[t][0];
          tree_shap_cond(&m->trees[t], fv, tc, 0, 0, path, 1, 1, -1, condition, condition_feature, 1);
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

/* libxgboost 1.6.0 CPUPredictor::PredictInteractionContributions: contributions with no condition (diag), then per
 * feature i (bias included) with i off and on; out[row][i][k] = on[k] / 2.0 - off[k] / 2.0 (in double, stored as
 * float) for k != i, and out[row][i][i] = 0 + diag[i] minus those, in float32 in k order. */
uint64_t oc_predict_interactions(const orc_model *m, const orc_dmatrix *d, int approximate, unsigned ntree_limit, float *out) {
  if (!m || !d) FAIL(0, "null handle");
  const uint64_t nc = (uint64_t)m->num_feature + 1, n = d->nrow * nc;
  float *diag = (float *)malloc(sizeof(float) * (n ? n : 1)), *off = (float *)malloc(sizeof(float) * (n ? n : 1)),
        *on = (float *)malloc(sizeof(float) * (n ? n : 1));
  int ok = contributions(m, d, approximate, ntree_limit, 0, 0, diag) == n;
  for (uint64_t i = 0; ok && i < nc; ++i) {
    ok = contributions(m, d, approximate, ntree_limit, -1, (unsigned)i, off) == n &&
         contributions(m, d, approximate, ntree_limit, 1, (unsigned)i, on) == n;
    for (uint64_t j = 0; ok && j < d->nrow; ++j) {
      float *o = out + j * nc * nc + i * nc;
      const float *cd = diag + j * nc, *cn = on + j * nc, *cf = off + j * nc;
      o[i] = 0;
      for (uint64_t k = 0; k < nc; ++k) {
        if (k == i) {
          o[i] += cd[k];
        } else {
          o[k] = (float)((double)cn[k] / 2.0 - (double)cf[k] / 2.0);
          o[i] -= o[k];
        }
      }
    }
  }
  free(diag);
  free(off);
  free(on);
  return ok ? n * nc : 0;
}
