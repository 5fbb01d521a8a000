"""GPU parity on the BASELINE.json configurations with the production-shape booster
("Depth18_eta1_100Trees", OH_GridCompMod.F90:224: 100 trees, depth <= 18, 27 features; seeded synthetic,
build/oh_booster_100x18.model), through the xgb_fortran_api C ABI, against the CPU oracle.

configs[1] "C90 x 72L single timestep on 1 B200 (correctness vs CPU leaf indices)": the matrix is what the
reference packs (OH_GridCompMod.F90:303-345) from synthetic fields — assembled by the oracle's Run1 restatement —
and every per-tree leaf index [N][100] and every float32 margin bit must equal the oracle's, on BOTH node layouts,
with the kernel family that served each launch asserted (a fallback to another kernel fails the test).
The same with -999.0 / NaN entries and values exactly on split thresholds injected (missing-value default
direction, float32 threshold compare semantics: BASELINE.json north_star).
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, inject_specials
from quickchem_b200 import synth, xgbmodel

pytestmark = [pytest.mark.gpu]


@pytest.fixture(scope="module")
def prod_model_path():
    sys.path.insert(0, ROOT)
    import bench

    return bench.booster_path()  # grown once (seeded) and cached under build/


@pytest.fixture(scope="module")
def c90(oracle, prod_model_path):
    """X[3 499 200 x 27] packed by the oracle's Run1 from C90 synthetic fields (all 72 levels), the oracle's leaf
    ids and margins for it, and the same with special values injected."""
    fields = synth.raw_fields(90)
    om = oracle.Model(prod_model_path)
    oracle.use_all_cores()
    r = oracle.run1(om, fields, synth.MAPL, tropp_min=0.0, want_features=True)
    assert r["k1"] == 1
    x = np.ascontiguousarray(r["X"])
    assert x.shape == (90 * 90 * 6 * 72, 27)
    return dict(fields=fields, x=x, run1=r, om=om)


def _leaf_and_margin(capi, booster, x, missing=-999.0):
    """Leaf ids, margins and values of one matrix, with the kernel family that served the first two.  The
    prediction pipelined into XGDMatrixCreateFromMat is switched off so that every predict is its own launch."""
    capi.set_param("speculate", 0)
    try:
        d = capi.DMatrix(x, missing)
        leaf = booster.predict(d, option_mask=2)
        k_leaf = capi.last_predict_kernel()
        margin = booster.predict(d, option_mask=1)
        k_margin = capi.last_predict_kernel()
        d.free()
    finally:
        capi.set_param("speculate", 1)
    d = capi.DMatrix(x, missing)  # pipelined create + speculative predict: what the reference's call sequence gets
    value = booster.predict(d, option_mask=0)
    d.free()
    return leaf, margin, value, k_leaf, k_margin


@pytest.mark.parametrize("duo", [1, 0], ids=["duo", "nodes8"])
def test_c90_leaf_indices_and_margins_production_booster(capi, c90, prod_model_path, duo):
    """configs[1].  Clean matrix (what the reference's physical fields give)."""
    x, om = c90["x"], c90["om"]
    ref_leaf = om.predict(x, option_mask=2)
    ref_margin = om.predict(x, option_mask=1)
    capi.set_param("duo", duo)
    try:
        b = capi.Booster(prod_model_path)
        assert b.info().num_trees == 100 and b.info().max_depth == 18
        leaf, margin, value, k_leaf, k_margin = _leaf_and_margin(capi, b, x)
    finally:
        capi.set_param("duo", -1)
    fam = "duo" if duo else "nodes8"
    assert (k_leaf, k_margin) == (fam + "_leaf", fam)  # the kernel under test is the kernel that ran
    assert leaf.shape == ref_leaf.shape == (x.shape[0], 100)
    assert np.array_equal(leaf, ref_leaf)  # per-tree leaf indices, bit-exact
    assert np.array_equal(margin.view(np.uint32), ref_margin.view(np.uint32))  # float32 sum in tree order, bit-exact
    assert np.array_equal(value.view(np.uint32), margin.view(np.uint32))  # reg:squarederror: identity transform


@pytest.mark.parametrize("duo", [1, 0], ids=["duo", "nodes8"])
def test_c90_missing_and_on_threshold_production_booster(capi, oracle, c90, prod_model_path, duo):
    """configs[1] with 1 % -999.0, 0.5 % NaN and values exactly on split thresholds: default direction and
    `fvalue < split_cond` semantics, on the kernels that serve matrices with missing entries."""
    from oracle import naive

    forest = naive.read_legacy(prod_model_path)  # (independent python reader; used only to find the thresholds)
    rng = np.random.default_rng(90)
    x = inject_specials(c90["x"][: 1 << 20], forest, rng, frac_on_threshold=0.002)
    om = c90["om"]
    ref_leaf = om.predict(x, option_mask=2)
    ref_margin = om.predict(x, option_mask=1)
    capi.set_param("duo", duo)
    try:
        b = capi.Booster(prod_model_path)
        leaf, margin, _, k_leaf, k_margin = _leaf_and_margin(capi, b, x)
    finally:
        capi.set_param("duo", -1)
    fam = "duo_missing" if duo else "nodes8_missing"
    assert (k_leaf, k_margin) == (fam + "_leaf", fam)
    assert np.array_equal(leaf, ref_leaf)
    assert np.array_equal(margin.view(np.uint32), ref_margin.view(np.uint32))


def test_c90_fused_run1_production_booster(capi, c90, prod_model_path):
    """The fused device-resident Run1 at C90 x 72 (40 hPa slab, as in production): raw booster output bit-exact,
    OH within 1e-6, served by the two-level records."""
    fields, om = c90["fields"], c90["om"]
    from oracle import cpu as oracle

    ref = oracle.run1(om, fields, synth.MAPL, want_features=True)
    km, ncol = fields["T"].shape
    b = capi.Booster(prod_model_path)
    oh = capi.OhRun1(b, ncol, km, synth.MAPL)
    n0 = capi.kernel_launches("soa_duo")
    got = oh.run(oh.make_in(fields), want=("OH", "OH_boost", "pred"))
    assert capi.kernel_launches("soa_duo") == n0 + 1
    assert got["k1"] == ref["k1"]
    assert np.array_equal(got["pred"].view(np.uint32), ref["pred"].view(np.uint32))
    a, r = got["OH"].astype(np.float64), ref["OH"].astype(np.float64)
    assert np.max(np.abs(a - r) / np.maximum(np.abs(r), 1e-300)) <= 1e-6


def test_seal_builds_key_tiles(capi):
    """XGDMatrixCreateFromMat's device form: Xt[tile][1 + col][256] order-preserving keys, missing = 0xFFFFFFFF; word-row
    0 of a tile is its row order — rows without a missing entry first, both groups in their original order."""
    rng = np.random.default_rng(1)
    for nrow, ncol, pmiss in ((1000, 27, 0.02), (256, 27, 0.0), (1, 5, 0.5), (700, 12, 0.05), (513, 32 - 1, 0.3), (4096, 27, 0.001)):
        x = rng.normal(0, 1, (nrow, ncol)).astype(np.float32)
        x[rng.random(x.shape) < pmiss] = -999.0
        x[rng.random(x.shape) < pmiss] = np.nan
        x[0, 0] = -0.0
        x.flat[1 % x.size] = np.float32(1e-42)
        d = capi.DMatrix(x)
        p, nt = capi.vp(), capi.u64()
        capi.check(capi.lib().qcoh_dmatrix_tiles_ptr(d.handle, C.byref(p), C.byref(nt)))
        assert nt.value == (nrow + 255) // 256
        t = np.empty((nt.value, ncol + 1, 256), np.uint32)
        capi.check(capi.lib().qcoh_memcpy_d2h(t.ctypes.data_as(capi.vp), p, t.nbytes))
        b = (x + np.float32(0)).view(np.uint32)
        key = b ^ np.where(b >> 31, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))
        miss = np.isnan(x) | (x == np.float32(-999.0))
        key = np.where(miss, np.uint32(0xFFFFFFFF), key)
        rowmiss = miss.any(axis=1)
        for ti in range(nt.value):
            order = t[ti, 0]
            orig, flag = (order & 0xFF).astype(np.int64), (order >> 8) & 1
            assert sorted(orig) == list(range(256))  # a permutation of the tile's rows
            nr = min(256, nrow - ti * 256)
            real = orig < nr
            rm = np.zeros(256, bool)
            rm[real] = rowmiss[ti * 256 + orig[real]]
            assert np.array_equal(flag.astype(bool), rm)
            assert np.all(np.diff(flag.astype(np.int64)) >= 0)  # clean rows first ...
            assert np.all(np.diff(orig[flag == 0]) > 0) and np.all(np.diff(orig[flag == 1]) > 0)  # ... both stable
            got = t[ti, 1:, :].T  # [position][col]
            assert np.array_equal(got[real], key[ti * 256 + orig[real]]), (nrow, ncol, ti)
        d.free()


def test_tile_loop_over_sizes_and_ragged_tiles(capi, oracle, tmp_path, small_forest, small_model_path):
    """The tile loop of the two-level kernel gives the oracle's sums and leaf ids over sizes from one tile to 972
    tiles, with a ragged last tile, with and without missing entries."""
    x_all = synth.quick_features(synth.raw_fields(24))  # 248 832 rows = 972 tiles
    om = oracle.Model(small_model_path)
    b = capi.Booster(small_model_path)
    rng = np.random.default_rng(2)
    for nrow in (255, 256 * 148 * 3 + 17, x_all.shape[0]):
        for special in (False, True):
            x = x_all[:nrow]
            if special:
                x = inject_specials(x, small_forest, rng)
            d = capi.DMatrix(x)
            assert np.array_equal(b.predict(d).view(np.uint32), om.predict(x).view(np.uint32)), (nrow, special)
            assert capi.last_predict_kernel() == ("duo_missing" if special else "duo")
            assert np.array_equal(b.predict(d, option_mask=2), om.predict(x, option_mask=2)), (nrow, special)
            d.free()


def test_more_than_480_trees_stay_on_the_fast_path(capi, oracle, tmp_path):
    """A launch walks at most 120 trees (the constant-memory tables hold 480 and are re-filled when a range leaves
    them); the float32 partial sum is carried through the output buffer, so a forest of any size stays on the
    two-level records and keeps the sum order."""
    f = synth.random_forest_structure(1100, 7, seed=77, p_leaf=0.1)
    p = str(tmp_path / "many.model")
    xgbmodel.write_legacy_binary(f, p)
    rng = np.random.default_rng(3)
    x = rng.normal(0, 1, (5000, 27)).astype(np.float32)
    om = oracle.Model(p)
    b = capi.Booster(p)
    n0 = capi.kernel_launches("duo")
    got = b.predict(capi.DMatrix(x))
    assert capi.kernel_launches("duo") == n0 + 10 and capi.last_predict_kernel() == "duo"  # 9 x 120 + 20 trees
    assert np.array_equal(got.view(np.uint32), om.predict(x).view(np.uint32))
    for lim in (1, 120, 121, 480, 481, 960, 1000):
        assert np.array_equal(b.predict(capi.DMatrix(x), ntree_limit=lim).view(np.uint32),
                              om.predict(x, ntree_limit=lim).view(np.uint32)), lim  # fmt: skip
    assert np.array_equal(b.predict(capi.DMatrix(x), option_mask=2), om.predict(x, option_mask=2))
    assert capi.last_predict_kernel() == "duo_leaf"
    x[rng.random(x.shape) < 0.03] = np.nan
    assert np.array_equal(b.predict(capi.DMatrix(x)).view(np.uint32), om.predict(x).view(np.uint32))
    assert capi.last_predict_kernel() == "duo_missing"
    # device-resident predict with the fused export transform only after the last range
    d = capi.DMatrix(x)
    out = capi.DeviceArray(x.shape[0])
    b.predict_device(d, out, exp10=True, scale=0.5)
    capi.synchronize()
    ref = (np.float32(10.0) ** (om.predict(x) * np.float32(0.01))).astype(np.float32)  # (only to bound the magnitude)
    assert np.all(np.isfinite(out.get())) and ref.shape == out.get().shape
    b.predict_device(d, out)
    capi.synchronize()
    assert np.array_equal(out.get().view(np.uint32), om.predict(x).view(np.uint32))


def test_wide_tree_records_without_default_bits(capi, oracle, tmp_path):
    """A tree with more than 2^14 record blocks gets the 17-bit block pointer and no default-direction bits: clean
    matrices still walk the records, matrices with missing entries walk the 8-byte nodes."""
    f = synth.random_forest_structure(2, 17, seed=5, p_leaf=0.0)  # complete trees: 262 143 nodes each
    p = str(tmp_path / "wide.model")
    xgbmodel.write_legacy_binary(f, p)
    b = capi.Booster(p)
    assert b.duo_info() == (15, False)
    om = oracle.Model(p)
    rng = np.random.default_rng(6)
    x = rng.normal(0, 1, (20000, 27)).astype(np.float32)
    assert np.array_equal(b.predict(capi.DMatrix(x)).view(np.uint32), om.predict(x).view(np.uint32))
    assert capi.last_predict_kernel() == "duo"
    assert np.array_equal(b.predict(capi.DMatrix(x), option_mask=2), om.predict(x, option_mask=2))
    x[rng.random(x.shape) < 0.02] = -999.0
    assert np.array_equal(b.predict(capi.DMatrix(x)).view(np.uint32), om.predict(x).view(np.uint32))
    assert capi.last_predict_kernel() == "nodes8_missing"


def test_booster_without_trees_and_handle_lifetimes(capi, oracle, tmp_path, small_model_path):
    f = xgbmodel.Forest(trees=[], base_score=0.25, num_feature=27)
    p = str(tmp_path / "empty_forest.model")
    xgbmodel.write_legacy_binary(f, p)
    b = capi.Booster(p)
    x = np.zeros((300, 27), np.float32)
    assert np.all(b.predict(capi.DMatrix(x)) == np.float32(0.25))
    assert b.predict(capi.DMatrix(x), option_mask=2).size == 0
    # a booster a fused-Run1 handle predicts with cannot be freed under it; a freed handle is refused, not read
    b2 = capi.Booster(small_model_path)
    oh = capi.OhRun1(b2, 24, 72, synth.MAPL)
    with pytest.raises(capi.QcohError, match="fused-Run1"):
        capi.check(capi.lib().XGBoosterFree(b2.handle))
    oh.free()
    h = b2.handle
    capi.check(capi.lib().XGBoosterFree(h))
    b2.handle = capi.vp()
    assert capi.lib().XGBoosterFree(h) == -1 and "Invalid booster handle" in capi.last_error()
