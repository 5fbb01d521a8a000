"""Randomised parity of the CUDA predictor against BOTH CPU restatements on adversarial values.

The device compares order-preserving integer keys (kernels.cu) instead of floats; this test aims at
every place where that could differ from float32 `<`: +-0.0, denormals, FLT_MAX, +-inf thresholds,
values exactly on thresholds, NaN / -999.0 (missing) at default-left and default-right nodes, matrices
narrower than the booster.  Leaf ids and float32 sums must be bit-exact against oracle/qc_oracle.c
and against the pure-numpy traverser."""
import numpy as np
import pytest

from oracle import naive
from quickchem_b200 import xgbmodel

pytestmark = pytest.mark.gpu

F32 = np.float32
POOL = np.array(
    [0.0, -0.0, 1e-45, -1e-45, 1.17549435e-38, -1.17549435e-38, 5e-39, 3.4028235e38, -3.4028235e38, 1.0, -1.0,
     np.nextafter(F32(1), F32(2)), np.nextafter(F32(1), F32(0)), 0.5, -0.5, 2.0, 123.456, -123.456, 1e-10, 1e10,
     -1e10, 287.15, 1013.25, 4.0e-8],
    dtype=np.float32,
)  # fmt: skip


def random_tree(rng, nfeat, max_depth, thr_pool):
    def spec(d):
        if d == max_depth or (d > 0 and rng.random() < 0.25):
            return float(F32(rng.normal(0, 1)))
        return (int(rng.integers(nfeat)), float(rng.choice(thr_pool)), bool(rng.random() < 0.5), spec(d + 1), spec(d + 1))

    return xgbmodel.tree_from_nested(spec(0))


@pytest.mark.parametrize("seed", range(12))
def test_adversarial_values(capi, oracle, tmp_path, seed):
    rng = np.random.default_rng(1000 + seed)
    nfeat = int(rng.choice([1, 2, 5, 27, 31]))
    ntree = int(rng.choice([1, 3, 4, 5, 9, 17]))
    thr_pool = np.concatenate([POOL, [np.inf, -np.inf]]).astype(np.float32) if seed % 3 == 0 else POOL
    forest = xgbmodel.Forest(trees=[random_tree(rng, nfeat, int(rng.integers(1, 9)), thr_pool) for _ in range(ntree)],
                             base_score=float(F32(rng.normal())), num_feature=nfeat)  # fmt: skip
    p = str(tmp_path / "fuzz.model")
    xgbmodel.write_legacy_binary(forest, p)
    nrow = int(rng.choice([1, 33, 300, 777, 2049]))
    ncol = nfeat if seed % 4 else max(1, nfeat - int(rng.integers(0, 3)))  # sometimes narrower than the booster
    x = rng.choice(POOL, size=(nrow, ncol)).astype(np.float32)
    m = rng.random(x.shape)
    x[m < 0.06] = np.nan
    x[(m >= 0.06) & (m < 0.12)] = F32(-999.0)
    if seed % 2:  # a clean matrix: exercises the no-missing specialisation
        x = np.where(np.isnan(x) | (x == F32(-999.0)), F32(0.25), x).astype(np.float32)
        if ncol < nfeat:
            ncol, x = nfeat, np.concatenate([x, np.zeros((nrow, nfeat - ncol), np.float32)], axis=1)
    b = capi.Booster(p)
    om, nm = oracle.Model(p), naive.read_legacy(p)
    got_leaf = b.predict(capi.DMatrix(x), option_mask=2)
    assert np.array_equal(got_leaf.astype(np.int64), naive.leaf_ids(nm, x))
    assert np.array_equal(got_leaf, om.predict(x, option_mask=2))
    got = b.predict(capi.DMatrix(x))
    assert np.array_equal(got.view(np.uint32), om.predict(x).view(np.uint32))
    assert np.array_equal(got.view(np.uint32), naive.predict(nm, x).view(np.uint32))
    # device-resident entry point (no pipelined create) agrees too
    d = capi.DMatrix.device(nrow, ncol)
    d.upload(x)
    d.seal()
    out = capi.DeviceArray(nrow)
    b.predict_device(d, out)
    capi.synchronize()
    assert np.array_equal(out.get().view(np.uint32), got.view(np.uint32))


def test_every_float_neighbourhood_of_a_threshold(capi, oracle, tmp_path):
    """For a set of thresholds, the 5 floats around each (and their negatives) must fall on the same side as
    float32 `<` says."""
    thr = np.array([0.0, -0.0, 1e-45, 1.17549435e-38, 1.0, 287.15, 3.4028235e38, -1.0, -1e-45, -3.4028235e38], np.float32)
    trees = [xgbmodel.tree_from_nested((0, float(t), False, -1.0, 1.0)) for t in thr]
    forest = xgbmodel.Forest(trees=trees, base_score=0.0, num_feature=1)
    p = str(tmp_path / "thr.model")
    xgbmodel.write_legacy_binary(forest, p)
    vals = []
    with np.errstate(over="ignore"):
        vals = _neighbours(thr)
    x = np.array([v for v in vals if np.isfinite(v)], np.float32).reshape(-1, 1)
    leaf = capi.Booster(p).predict(capi.DMatrix(x), option_mask=2)
    expect = np.where(x < thr[None, :], 1, 2).astype(np.float32)  # left child id 1, right child id 2
    assert np.array_equal(leaf, expect)
    assert np.array_equal(leaf, oracle.Model(p).predict(x, option_mask=2))


def _neighbours(thr):
    vals = []
    for t in thr:
        v = F32(t)
        lo = v
        for _ in range(2):
            lo = np.nextafter(lo, F32(-np.inf), dtype=np.float32)
        cur = lo
        for _ in range(5):
            vals.append(cur)
            cur = np.nextafter(cur, F32(np.inf), dtype=np.float32)
    return vals


@pytest.mark.parametrize("duo", [1, 0], ids=["duo", "nodes8"])
def test_any_number_of_rows_with_missing_entries(capi, oracle, tmp_path, duo):
    """The seal kernel orders each tile's rows (clean first) so that only warps holding rows with missing entries
    take the default-direction walk: any number of such rows per tile — none, one, a warp's worth +-1, all — in the
    first, a middle and the ragged last tile must give the oracle's leaf ids and sums, on both layouts."""
    from quickchem_b200 import synth

    rng = np.random.default_rng(77)
    forest = synth.random_forest_structure(9, 11, seed=6, p_leaf=0.12)
    p = str(tmp_path / "m.model")
    xgbmodel.write_legacy_binary(forest, p)
    om = oracle.Model(p)
    b = capi.Booster(p)
    nrow = 3 * 256 + 77
    capi.set_param("duo", duo)
    try:
        for nmiss in (0, 1, 31, 32, 33, 255, 256, 300, nrow):
            x = rng.normal(0, 1, (nrow, 27)).astype(np.float32)
            rows = rng.choice(nrow, nmiss, replace=False)
            for r in rows:  # one to three missing entries per chosen row, NaN or -999.0
                cols = rng.choice(27, int(rng.integers(1, 4)), replace=False)
                x[r, cols] = np.where(rng.random(len(cols)) < 0.5, np.nan, F32(-999.0))
            if nmiss == 300:
                x[512:768] = rng.normal(0, 1, (256, 27)).astype(np.float32)  # one tile stays clean inside a missing matrix
            d = capi.DMatrix(x)
            assert np.array_equal(b.predict(d).view(np.uint32), om.predict(x).view(np.uint32)), nmiss
            fam = ("duo" if duo else "nodes8") + ("_missing" if nmiss else "")
            assert capi.last_predict_kernel() == fam
            assert np.array_equal(b.predict(d, option_mask=2), om.predict(x, option_mask=2)), nmiss
            assert np.array_equal(b.predict(d, ntree_limit=7).view(np.uint32), om.predict(x, ntree_limit=7).view(np.uint32)), nmiss
    finally:
        capi.set_param("duo", -1)
