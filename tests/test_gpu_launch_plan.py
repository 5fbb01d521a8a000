"""Which walk serves a predict launch, when the constant-memory table of tree tops moves between boosters and between
windows of one booster's trees, and which path and kernel family serve the fused Run1.  Every result is compared with
the oracle bit for bit, and the family that served it is asserted, on both layouts of the duo_mode fixture."""
import numpy as np
import pytest

from quickchem_b200 import synth, xgbmodel

pytestmark = [pytest.mark.gpu]


def _check(capi, booster, om, x, family, **kw):
    d = capi.DMatrix(x)
    got = booster.predict(d, **kw)
    served = capi.last_predict_kernel()
    d.free()
    ref = om.predict(x, **kw)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), kw
    assert served == family, kw


def _fused_run1(capi, oracle, booster, model_path, fields):
    km, ncol = fields["T"].shape
    oh = capi.OhRun1(booster, ncol, km, synth.MAPL)
    got = oh.run(oh.make_in(fields), want=("OH", "pred"))
    oh.free()
    ref = oracle.run1(oracle.Model(model_path), fields, synth.MAPL, want_features=True)
    assert got["k1"] == ref["k1"]
    assert np.array_equal(got["pred"].view(np.uint32), ref["pred"].view(np.uint32))


def test_two_boosters_share_the_constant_table(capi, oracle, tmp_path, small_model_path, duo_mode):
    """The 1 100-tree forest and the small forest take turns on one thread.  ntree_limit 1 000, 481 and 0 move the
    big forest's window of 480 trees; a predict on the small booster and a fused Run1 in between take the table
    over.  Leaf ids and a matrix with missing entries follow the same moves."""
    big = synth.random_forest_structure(1100, 7, seed=77, p_leaf=0.1)
    big_path = str(tmp_path / "many.model")
    xgbmodel.write_legacy_binary(big, big_path)
    fam = "duo" if duo_mode else "nodes8"
    rng = np.random.default_rng(11)
    xb = rng.normal(0, 1, (3000, 27)).astype(np.float32)
    fields = synth.raw_fields(4)
    xs = synth.quick_features(fields)
    b_big, b_small = capi.Booster(big_path), capi.Booster(small_model_path)
    om_big, om_small = oracle.Model(big_path), oracle.Model(small_model_path)

    _check(capi, b_big, om_big, xb, fam, ntree_limit=1000)
    _check(capi, b_small, om_small, xs, fam)
    _check(capi, b_big, om_big, xb, fam, ntree_limit=481)
    soa = "soa_duo" if duo_mode else "soa_nodes8"
    n0 = capi.kernel_launches(soa)
    _fused_run1(capi, oracle, b_small, small_model_path, fields)
    assert capi.kernel_launches(soa) == n0 + 1
    _check(capi, b_big, om_big, xb, fam, ntree_limit=0)
    _check(capi, b_big, om_big, xb, fam + "_leaf", option_mask=2, ntree_limit=481)
    _check(capi, b_small, om_small, xs, fam + "_leaf", option_mask=2)
    xb[rng.random(xb.shape) < 0.03] = np.nan
    xs = xs.copy()
    xs[rng.random(xs.shape) < 0.03] = np.nan
    _check(capi, b_big, om_big, xb, fam + "_missing", ntree_limit=1000)
    _check(capi, b_small, om_small, xs, fam + "_missing")
    _check(capi, b_big, om_big, xb, fam + "_missing", ntree_limit=0)


def test_fused_run1_over_120_trees_takes_the_matrix_path(capi, oracle, tmp_path, small_forest, duo_mode):
    """A 27-feature booster of more than 120 trees needs ranged launches, which the fused kernel does not make: the
    Run1 packs the matrix and predicts it with the predict kernel (no fused launch)."""
    f = synth.replicate_forest(small_forest, 11)  # 132 trees
    p = str(tmp_path / "132.model")
    xgbmodel.write_legacy_binary(f, p)
    fam = "duo" if duo_mode else "nodes8"
    soa = (capi.kernel_launches("soa_duo"), capi.kernel_launches("soa_nodes8"))
    n0 = capi.kernel_launches(fam)
    _fused_run1(capi, oracle, capi.Booster(p), p, synth.raw_fields(4))
    assert (capi.kernel_launches("soa_duo"), capi.kernel_launches("soa_nodes8")) == soa
    assert capi.kernel_launches(fam) > n0 and capi.last_predict_kernel() == fam
