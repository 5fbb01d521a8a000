"""Checks shared by the interaction tests (test_interactions_cpu.py, test_gpu_interactions.py): the conditioned path
form of the interactions kernel replayed in numpy on the library's path tables, and the bar for exact values."""
import numpy as np

from contribs_forests import key, replay_paths


def _unwound_sums(o, z):
    """W[:, e] for the elements e = 1 .. D of one path (bias at 0): ExtendPath over all of them, then UnwoundPathSum of
    each, float64, as replay_paths does.  o: [nrow, D + 1] one fractions, z: [D + 1] zero fractions."""
    nrow, ln = o.shape
    D = ln - 1
    pw = np.zeros((nrow, ln))
    pw[:, 0] = 1.0
    for i in range(1, D + 1):
        new = np.zeros_like(pw)
        for j in range(0, i + 1):
            new[:, j] = z[i] * pw[:, j] * (i - j) / (i + 1)
            if j > 0:
                new[:, j] += o[:, i] * pw[:, j - 1] * j / (i + 1)
        pw = new
    w = np.zeros((nrow, ln))
    for e in range(1, ln):
        nxt, total = pw[:, D].copy(), np.zeros(nrow)
        one = o[:, e] != 0
        for i in range(D - 1, -1, -1):
            tmp = nxt * (D + 1) / (i + 1)
            t_one, n_one = total + tmp, pw[:, i] - tmp * z[e] * (D - i) / (D + 1)
            t_zero = total + pw[:, i] / z[e] * (D + 1) / (D - i)
            total, nxt = np.where(one, t_one, t_zero), np.where(one, n_one, nxt)
        w[:, e] = total
    return w


def replay_interactions(bins, tree_bin, x, nfeat, missing=-999.0, ntree=None):
    """The conditioned path form of the interactions kernel restated in numpy (float64) on the tables of
    qcoh_booster_get_shap_paths: for every path P with leaf v and every element c of P, each other element i adds
    1/2 (o_c - z_c) W_i(P without c) (o_i - z_i) v to M[c][f_i], W the UnwoundPathSum in P extended without c; the
    diagonal is replay_paths' phi_c minus the row's off-diagonal sum.  [nrow, nfeat, nfeat] without the bias."""
    x = np.asarray(x, np.float32)
    nrow, ncol = x.shape
    miss = np.isnan(x) | (x == np.float32(missing))
    k = key(np.where(miss, np.float32(0), x)).astype(np.int64)
    out = np.zeros((nrow, nfeat, nfeat))
    nb = int(tree_bin[-1] if ntree is None else tree_bin[ntree])
    for b in range(nb):
        lanes = bins[b]
        l = 0
        while l < 32:
            ln = int(lanes[l, 2]) >> 24
            if ln == 0:
                l += 1
                continue
            g = lanes[l : l + ln]
            v = float(g[0, 3:4].view(np.float32)[0])
            o, z, feats = np.ones((nrow, ln)), np.ones(ln), [0xFF]
            for e in range(1, ln):
                f = int(g[e, 2]) & 0xFF
                feats.append(f)
                z[e] = float(g[e, 3:4].view(np.float32)[0])
                mf = (int(g[e, 2]) >> 8) & 1
                if f < ncol:
                    o[:, e] = np.where(miss[:, f], mf, (int(g[e, 0]) <= k[:, f]) & (k[:, f] < int(g[e, 1])))
                else:
                    o[:, e] = mf
            for c in range(1, ln):
                keep = [e for e in range(ln) if e != c]
                w = _unwound_sums(o[:, keep], z[keep])
                for r, e in enumerate(keep[1:], start=1):
                    out[:, feats[c], feats[e]] += 0.5 * (o[:, c] - z[c]) * w[:, r] * (o[:, e] - z[e]) * v
            l += ln
    phi = replay_paths(bins, tree_bin, x, nfeat, missing, ntree)
    for c in range(nfeat):
        out[:, c, c] = phi[:, c] - (out[:, c, :].sum(axis=1) - out[:, c, c])
    return out


def assert_interactions_close(got, ref, what=""):
    """The bar for exact interaction values: per row, max |dM| <= 1e-5 * sum |M_ref|.  Returns the largest ratio."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    n = got.shape[0]
    scale = np.abs(ref).reshape(n, -1).sum(axis=1)
    ratio = np.abs(got - ref).reshape(n, -1).max(axis=1) / np.maximum(scale, 1e-30)
    worst = float(ratio.max()) if ratio.size else 0.0
    assert worst <= 1e-5, f"{what}: max |dM| / sum |M| = {worst:.3e} at row {int(ratio.argmax())}"
    return worst
