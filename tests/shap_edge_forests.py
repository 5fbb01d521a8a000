"""Boosters (with covers) at the edges of the exact SHAP kernels' path tables, and rows for them, shared by
test_shap_reference_cpu.py and test_gpu_shap_precision.py.

* `caterpillar`: 31 features, depth 31, a new feature per level and one leaf per level: paths of every length 2..32
  lanes (bias included), the longest a full 32-lane bin, M of shape [32][32].
* `repeats`: one feature split several times on a path — nested intervals in one direction, bounded and contradictory
  intervals, alternating default directions — at thresholds -0.0 / +0.0, denormals and +-FLT_MAX.
* `stumps`: nb trees = nb bins (a tree's paths share its bins), so the 16 bin slices hold 0, 1 or 2 bins; single-leaf
  trees mixed in and feature 26 never split on.
* `covers`: zero fractions above 1 (a child with more cover than its parent), within 2^-20 of 1, and near 1e-6.
* `underflow` / `overflow`: a product of cover ratios that float32 cannot hold (+0 / +inf).
"""
import numpy as np

from quickchem_b200 import xgbmodel

FLT_MAX = float(np.finfo(np.float32).max)
DENORM = float(np.float32(1e-40))
TINY = float(np.float32(1.4e-45))  # the smallest denormal


def build_tree(spec) -> xgbmodel.Tree:
    """spec := (leaf value, cover) | (feature, threshold, default_left, cover, left spec, right spec).  Nodes are
    numbered breadth-first with adjacent children, as xgbmodel.tree_from_nested numbers them."""
    from collections import deque

    left, right, parent, sidx, cond, dl, cov = [], [], [], [], [], [], []

    def new(p):
        for a, v in ((left, -1), (right, -1), (parent, p), (sidx, 0), (cond, 0.0), (dl, 0), (cov, 0.0)):
            a.append(v)
        return len(left) - 1

    q = deque([(new(-1), spec)])
    while q:
        n, sp = q.popleft()
        if len(sp) == 2:
            cond[n], cov[n] = float(sp[0]), float(sp[1])
            continue
        f, thr, d, c, ls, rs = sp
        l, r = new(n), new(n)
        left[n], right[n], sidx[n], cond[n], dl[n], cov[n] = l, r, int(f), float(thr), int(bool(d)), float(c)
        q.append((l, ls)), q.append((r, rs))
    return xgbmodel.Tree(left=np.asarray(left, np.int32), right=np.asarray(right, np.int32),
                         parent=np.asarray(parent, np.int32), split_index=np.asarray(sidx, np.uint32),
                         split_cond=np.asarray(cond, np.float32), default_left=np.asarray(dl, np.uint8),
                         sum_hess=np.asarray(cov, np.float32))  # fmt: skip


def forest(specs, num_feature, base_score=0.5) -> xgbmodel.Forest:
    return xgbmodel.Forest(trees=[build_tree(s) for s in specs], base_score=base_score, num_feature=num_feature)


# ---- caterpillar ----------------------------------------------------------------------------------------------
def caterpillar(mirror=False, seed=1):
    """(forest, thresholds, continuing side per level).  Level d splits on feature d; one child is a leaf, the other
    goes on (the right child, or alternating sides in the mirrored copy, which also alternates default directions).
    Level 30 ends in two leaves."""
    rng = np.random.default_rng(seed)
    thr = rng.uniform(-1, 1, 31).astype(np.float32)
    cont = [(d % 2 if mirror else 1) for d in range(31)]
    cover = np.float32(1e9)

    def level(d, c):
        dflt = d % 2 if mirror else int(d % 3 == 0)
        r = np.float32(rng.uniform(0.1, 0.9))
        c_leaf = np.float32(c * r)
        c_on = np.float32(c - c_leaf)
        leaf = (float(rng.normal(0, 0.1)), c_leaf)
        on = (float(rng.normal(0, 0.1)), c_on) if d == 30 else level(d + 1, c_on)
        kids = (leaf, on) if cont[d] else (on, leaf)
        return (d, thr[d], dflt, c, *kids)

    return forest([level(0, cover)], 31, base_score=0.25), thr, np.asarray(cont)


def caterpillar_rows(thr, cont, n, seed, frac_missing=0.05):
    """Rows that stop at every level: x follows the continuing side above a random level L and leaves at L; some
    values exactly on the thresholds (a value on a threshold goes right), some missing (-999 or NaN)."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, 31), np.float32)
    stop = rng.integers(0, 32, n)
    for d in range(31):
        gap = np.abs(rng.normal(0, 0.3, n)).astype(np.float32) + np.float32(1e-3)
        go_right = np.where(d < stop, cont[d] == 1, cont[d] == 0)
        x[:, d] = np.where(go_right, thr[d] + gap, thr[d] - gap)
        on = go_right & (rng.random(n) < 0.1)
        x[on, d] = thr[d]
    m = rng.random(x.shape)
    x[m < frac_missing] = np.float32(-999.0)
    x[(m >= frac_missing) & (m < 1.5 * frac_missing)] = np.nan
    return x


# ---- repeated splits on one feature ---------------------------------------------------------------------------
def repeats():
    """Four features, feature 0 split up to five times on one path."""
    lf = lambda v, c: (v, c)  # noqa: E731
    nested_right = (0, -0.0, 1, 1000.0,
                    (1, 0.5, 0, 400.0, lf(0.3, 150.0), lf(-0.2, 250.0)),
                    (0, DENORM, 0, 600.0,
                     lf(0.7, 100.0),
                     (2, 0.25, 1, 500.0,
                      (0, 1.0, 1, 200.0, lf(-0.4, 120.0), (0, FLT_MAX, 0, 80.0, lf(0.15, 60.0), lf(1.5, 20.0))),
                      (0, 2.5, 0, 300.0, lf(0.05, 100.0), (0, 3.0, 1, 200.0, lf(-0.6, 90.0), lf(0.9, 110.0))))))  # fmt: skip
    nested_left = (0, 2.0, 0, 900.0,
                   (0, 0.0, 1, 700.0,
                    (1, -0.25, 0, 300.0, (0, -DENORM, 1, 120.0, (0, -FLT_MAX, 0, 50.0, lf(2.0, 20.0), lf(-1.0, 30.0)), lf(0.4, 70.0)),
                     lf(-0.3, 180.0)),
                    lf(0.25, 400.0)),
                   (3, 0.1, 1, 200.0, lf(-0.8, 90.0), lf(0.6, 110.0)))  # fmt: skip
    bounded = (0, 0.0, 0, 1000.0,
               (0, -1.0, 1, 300.0, (1, 0.5, 1, 100.0, lf(0.2, 40.0), lf(-0.1, 60.0)), (0, -0.5, 0, 200.0, lf(0.35, 90.0), lf(-0.45, 110.0))),
               (0, 2.5, 1, 700.0,
                (3, 0.1, 0, 400.0, (0, -0.5, 1, 100.0, lf(1.25, 40.0), lf(-0.75, 60.0)), lf(0.5, 300.0)),
                (0, TINY, 0, 300.0, lf(-2.0, 100.0), (2, -0.0, 1, 200.0, lf(0.1, 80.0), lf(-0.2, 120.0)))))  # fmt: skip
    alternating = (0, 1.0, 1, 800.0,
                   (0, 0.5, 0, 500.0, (0, 0.25, 1, 300.0, (2, 0.0, 0, 200.0, lf(0.45, 90.0), lf(-0.15, 110.0)), lf(0.3, 100.0)),
                    (0, 0.75, 1, 200.0, lf(-0.9, 50.0), lf(0.2, 150.0))),
                   (1, -0.0, 0, 300.0, (0, 3.0, 1, 100.0, lf(1.1, 40.0), lf(-0.3, 60.0)), (0, 2.0, 0, 200.0, lf(0.8, 120.0), lf(-0.05, 80.0))))  # fmt: skip
    return forest([nested_right, nested_left, bounded, alternating], 4, base_score=0.5)


REPEAT_VALUES = np.asarray([-0.0, 0.0, DENORM, -DENORM, TINY, -TINY, FLT_MAX, -FLT_MAX, 0.25, 0.5, 0.75, 1.0, 2.0, 2.5,
                            3.0, -1.0, -0.5, -0.25, 0.1], np.float32)  # fmt: skip


def special_rows(forest, n, seed, frac_missing=0.08):
    """Rows of values on every threshold of the forest, their float32 neighbours, +-0.0, denormals and +-FLT_MAX,
    with -999 / NaN entries."""
    rng = np.random.default_rng(seed)
    thr = {float(c) for t in forest.trees for c, l in zip(t.split_cond, t.left) if l != -1}
    vals = set(map(float, REPEAT_VALUES)) | thr
    with np.errstate(over="ignore"):
        for c in thr:
            vals |= {float(np.nextafter(np.float32(c), np.float32(s))) for s in (np.inf, -np.inf)}
    vals = np.asarray(sorted(v for v in vals if np.isfinite(v)), np.float32)
    x = rng.choice(vals, (n, forest.num_feature)).astype(np.float32)
    x[rng.random(x.shape) < 0.05] = np.float32(-0.0)  # the set above holds one zero
    m = rng.random(x.shape)
    x[m < frac_missing] = np.float32(-999.0)
    x[(m >= frac_missing) & (m < 1.5 * frac_missing)] = np.nan
    return x


# ---- bin counts ------------------------------------------------------------------------------------------------
def stumps(nb, seed=0):
    """nb trees, so nb bins: stumps on features (7 i) % 26 (feature 26 is never split on) and every fifth tree a
    single leaf."""
    rng = np.random.default_rng(seed)
    specs = []
    for i in range(nb):
        c_l, c_r = (float(np.float32(c)) for c in rng.uniform(10, 1000, 2))
        if i % 5 == 4:
            specs.append((float(rng.normal(0, 0.5)), c_l + c_r))
        else:
            specs.append(((7 * i) % 26, float(np.float32(rng.uniform(-1, 1))), int(rng.integers(2)), c_l + c_r,
                          (float(rng.normal(0, 0.5)), c_l), (float(rng.normal(0, 0.5)), c_r)))  # fmt: skip
    return forest(specs, 27, base_score=0.5)


def single_leaves(n=5):
    return forest([(0.1 * (i + 1), 10.0 + i) for i in range(n)], 27, base_score=0.5)


# ---- covers ----------------------------------------------------------------------------------------------------
def covers():
    """Zero fractions above 1, within 2^-20 of 1 and near 1e-6."""
    big = float(2**22)
    above_one = (0, 0.5, 1, 100.0, (2.0, 300.0),  # z = 3
                 (1, 0.0, 0, 50.0, (-1.0, 80.0), (1, 0.25, 1, 10.0, (0.5, 40.0), (-0.5, 2.0))))  # fmt: skip
    near_one = (2, 0.3, 0, big, (0, 1.0, 1, big - 2, (0.75, big - 3), (-0.25, 1.0)), (1.5, 2.0))  # z = 1 - 2^-21, 1 - 3 2^-22
    small = (1, -0.5, 1, 1e6, (5.0, 1.0), (3, 0.7, 0, 1e6 - 1, (0, 0.2, 0, 2.0, (-3.0, 1.5), (2.5, 0.5)), (0.01, 1e6 - 3)))  # fmt: skip
    return forest([above_one, near_one, small], 4, base_score=-0.5)


def underflow():
    """cover 1e-30 under a parent of 1e30: the zero fraction 1e-60 is +0 in float32."""
    return forest([(1, 0.0, 0, 1.0, (0.5, 1.0), (0, 0.5, 0, 1e30, (1.0, 1e-30), (-1.0, 1e30)))], 4)


def overflow():
    """cover 1e30 under a parent of 1e-30: the zero fraction 1e60 is +inf in float32."""
    return forest([(1, 0.0, 0, 1.0, (0.5, 1.0), (0, 0.5, 0, 1e-30, (1.0, 1e30), (-1.0, 1e-30)))], 4)
