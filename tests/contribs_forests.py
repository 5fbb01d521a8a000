"""Boosters with node covers and checks shared by the contribution tests (test_contribs_cpu.py, test_gpu_contribs.py)."""
import numpy as np

from quickchem_b200 import synth, xgbmodel

NF = synth.NFEAT


def key(v):
    """The order-preserving integer key of a float32 (kernels.cu), -0.0 folded into +0.0."""
    b = (np.asarray(v, np.float32) + np.float32(0)).view(np.uint32)
    return b ^ np.where(b >> 31, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))


def stump(feature, thr, default_left, v_left, v_right, c_left, c_right, base_score=0.5) -> xgbmodel.Forest:
    t = xgbmodel.tree_from_nested((feature, thr, default_left, v_left, v_right))
    t.sum_hess = np.asarray([c_left + c_right, c_left, c_right], np.float32)
    return xgbmodel.Forest(trees=[t], base_score=base_score, num_feature=NF)


def few_feature_forest(cols, n_trees, max_depth, seed, n_sample=6000) -> xgbmodel.Forest:
    """A booster grown (synth.grow_forest, covers = sample counts) on a C12 sample with only the columns `cols` offered,
    its split indices mapped back to those columns of the 27-feature matrix."""
    rng = np.random.default_rng(seed)
    x = synth.quick_features(synth.raw_fields(12, seed=seed))
    x = x[rng.choice(x.shape[0], n_sample, replace=False)]
    y = synth.synthetic_log10_oh(x, rng)
    f = synth.grow_forest(x[:, cols], y, n_trees=n_trees, max_depth=max_depth, min_leaf=8, seed=seed)
    cols = np.asarray(cols, np.uint32)
    for t in f.trees:
        t.split_index = np.where(t.left != -1, cols[t.split_index], 0).astype(np.uint32)
    f.num_feature = NF
    return f


def sklearn_tree(model) -> xgbmodel.Tree:
    """sklearn DecisionTreeRegressor -> xgbmodel.Tree (breadth-first, children adjacent; `x <= thr64` as `x < t32`
    for float32 x) with covers = weighted_n_node_samples."""
    t = model.tree_
    left, right, parent, sidx, cond, dl, cov, skid = [-1], [-1], [-1], [0], [0.0], [0], [0.0], [0]
    queue = [0]
    while queue:
        nid = queue.pop(0)
        s = skid[nid]
        cov[nid] = float(t.weighted_n_node_samples[s])
        if t.children_left[s] == -1:
            cond[nid] = float(np.float32(t.value[s, 0, 0]))
            continue
        t32 = np.float32(t.threshold[s])
        if float(t32) > t.threshold[s]:
            t32 = np.nextafter(t32, np.float32(-np.inf), dtype=np.float32)
        l = len(left)
        for child in (t.children_left[s], t.children_right[s]):
            left.append(-1), right.append(-1), parent.append(nid), sidx.append(0), cond.append(0.0), dl.append(0)
            cov.append(0.0), skid.append(int(child))
        left[nid], right[nid], sidx[nid] = l, l + 1, int(t.feature[s])
        cond[nid] = float(np.nextafter(t32, np.float32(np.inf), dtype=np.float32))
        dl[nid] = (nid * 7 + s) % 2  # both default directions occur
        queue += [l, l + 1]
    return xgbmodel.Tree(left=np.asarray(left, np.int32), right=np.asarray(right, np.int32),
                         parent=np.asarray(parent, np.int32), split_index=np.asarray(sidx, np.uint32),
                         split_cond=np.asarray(cond, np.float32), default_left=np.asarray(dl, np.uint8),
                         sum_hess=np.asarray(cov, np.float32))  # fmt: skip


def sklearn_forest(cols, n_trees=4, max_depth=6, seed=3):
    """(forest, query rows): sklearn-grown regression trees on the columns `cols`, and C8 rows with some values
    exactly on the trees' thresholds."""
    from sklearn.tree import DecisionTreeRegressor

    rng = np.random.default_rng(seed)
    x = synth.quick_features(synth.raw_fields(6, seed=seed))
    y = synth.synthetic_log10_oh(x, rng)
    trees = []
    for i in range(n_trees):
        m = DecisionTreeRegressor(max_depth=max_depth, min_samples_leaf=5, random_state=i, splitter="random" if i % 2 else "best")
        m.fit(x[i::n_trees][:, cols], y[i::n_trees] - 0.1 * i)
        t = sklearn_tree(m)
        t.split_index = np.where(t.left != -1, np.asarray(cols, np.uint32)[t.split_index], 0).astype(np.uint32)
        trees.append(t)
    forest = xgbmodel.Forest(trees=trees, base_score=0.25, num_feature=NF)
    return forest, synth.quick_features(synth.raw_fields(8, seed=seed + 1))


def on_thresholds(x, forest, rng, k=200):
    """Put k entries exactly on split thresholds of the forest."""
    x = x.copy()
    for _ in range(k):
        t = forest.trees[rng.integers(len(forest.trees))]
        internal = np.nonzero(t.left != -1)[0]
        if len(internal):
            n = rng.choice(internal)
            x[rng.integers(len(x)), int(t.split_index[n])] = t.split_cond[n]
    return x


def with_missing(x, rng, frac=0.05):
    x = x.copy()
    m = rng.random(x.shape)
    x[m < frac] = np.float32(-999.0)
    x[(m >= frac) & (m < 1.5 * frac)] = np.nan
    return x


def assert_shap_close(got, ref, what=""):
    """The bar for exact contributions: per row, max_f |dphi_f| <= 1e-5 * (sum_f |phi_f| + |bias|).  Returns the
    largest ratio seen (of |dphi| to that scale)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    scale = np.abs(ref).sum(axis=1)
    ratio = np.abs(got - ref).max(axis=1) / np.maximum(scale, 1e-30)
    worst = float(ratio.max()) if ratio.size else 0.0
    assert worst <= 1e-5, f"{what}: max |dphi| / (sum |phi| + |bias|) = {worst:.3e} at row {int(ratio.argmax())}"
    return worst


def replay_paths(bins, tree_bin, x, nfeat, missing=-999.0, ntree=None):
    """The path-form TreeSHAP of the exact kernel restated in numpy (float64, vectorised over rows) on the tables of
    qcoh_booster_get_shap_paths: per path, one fractions from the key bounds / missing flags, ExtendPath over its
    elements, UnwoundPathSum per element.  [nrow, nfeat] without the bias."""
    x = np.asarray(x, np.float32)
    nrow, ncol = x.shape
    miss = np.isnan(x) | (x == np.float32(missing))
    k = key(np.where(miss, np.float32(0), x)).astype(np.int64)
    out = np.zeros((nrow, nfeat))
    nb = int(tree_bin[-1] if ntree is None else tree_bin[ntree])
    for b in range(nb):
        lanes = bins[b]
        l = 0
        while l < 32:
            ln = int(lanes[l, 2]) >> 24
            if ln == 0:
                l += 1
                continue
            assert (int(lanes[l, 2]) >> 16) & 31 == l and int(lanes[l, 2]) & 0xFF == 0xFF
            g = lanes[l : l + ln]
            v = float(g[0, 3:4].view(np.float32)[0])
            D = ln - 1
            o = np.ones((nrow, ln))
            z = np.ones(ln)
            feats = []
            for e in range(1, ln):
                f = int(g[e, 2]) & 0xFF
                feats.append(f)
                z[e] = float(g[e, 3:4].view(np.float32)[0])
                mf = (int(g[e, 2]) >> 8) & 1
                if f < ncol:
                    o[:, e] = np.where(miss[:, f], mf, (int(g[e, 0]) <= k[:, f]) & (k[:, f] < int(g[e, 1])))
                else:
                    o[:, e] = mf
            assert len(set(feats)) == len(feats)  # repeated splits are merged into one element
            pw = np.zeros((nrow, ln))
            pw[:, 0] = 1.0
            for i in range(1, D + 1):
                new = np.zeros_like(pw)
                for j in range(0, i + 1):
                    new[:, j] = z[i] * pw[:, j] * (i - j) / (i + 1)
                    if j > 0:
                        new[:, j] += o[:, i] * pw[:, j - 1] * j / (i + 1)
                pw = new
            for e in range(1, ln):
                nxt, total = pw[:, D].copy(), np.zeros(nrow)
                one = o[:, e] != 0
                for i in range(D - 1, -1, -1):
                    tmp = nxt * (D + 1) / (i + 1)
                    t_one, n_one = total + tmp, pw[:, i] - tmp * z[e] * (D - i) / (D + 1)
                    t_zero = total + pw[:, i] / z[e] * (D + 1) / (D - i)
                    total, nxt = np.where(one, t_one, t_zero), np.where(one, n_one, nxt)
                out[:, feats[e - 1]] += total * (o[:, e] - z[e]) * v
            l += ln
    return out
