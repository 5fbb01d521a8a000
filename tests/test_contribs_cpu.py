"""Per-feature contributions on the CPU: the oracle's restatement of libxgboost 1.6.0 PredictContribution against
hand-derived answers, brute-force Shapley values and the naive Saabas walk; the library's path tables (what the
exact kernel walks) replayed in numpy against the oracle; covers and XGBoosterPredictFromDMatrix config errors."""
import os

import numpy as np
import pytest

from contribs_forests import (NF, assert_shap_close, few_feature_forest, on_thresholds, replay_paths, sklearn_forest,
                              stump, with_missing)  # fmt: skip
import oracle_contribs as oc
from quickchem_b200 import synth, xgbmodel

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _model(oracle, forest, tmp_path, name):
    p = str(tmp_path / f"{name}.model")
    xgbmodel.write_legacy_binary(forest, p)
    return oracle.Model(p), p


@pytest.mark.parametrize("default_left", [True, False])
def test_stump_known_answer(oracle, tmp_path, default_left):
    """A stump on feature f with covers (c_l, c_r): phi_f = v_hot - (c_l v_l + c_r v_r) / (c_l + c_r), every other
    feature 0, bias = mean + base_score; a missing entry takes the default child."""
    f, thr, vl, vr, cl, cr, base = 3, 0.5, -1.25, 2.0, 3.0, 5.0, 0.5
    forest = stump(f, thr, default_left, vl, vr, cl, cr, base)
    m, _ = _model(oracle, forest, tmp_path, "stump")
    x = np.zeros((4, NF), np.float32)
    x[:, f] = [0.25, 0.5, 0.75, -999.0]  # left, on the threshold (right), right, missing
    mean = (cl * vl + cr * vr) / (cl + cr)
    hot = np.array([vl, vr, vr, vl if default_left else vr])
    want = np.zeros((4, NF + 1))
    want[:, f] = hot - mean
    want[:, NF] = np.float32(mean) + np.float32(base)
    for approximate in (False, True):
        got = oc.predict_contribs(m, x, approximate=approximate)
        assert np.allclose(got, want, rtol=1e-6, atol=1e-6), (approximate, got, want)
        assert np.array_equal(got[:, NF], np.full(4, np.float32(np.float32(mean) + np.float32(base))))
    assert np.allclose(oc.shapley_brute_force(forest, x), want, rtol=1e-12, atol=1e-12)
    assert np.array_equal(oc.saabas(forest, x), oc.predict_contribs(m, x, approximate=True))


def _cases():
    rng = np.random.default_rng(7)
    for i, (cols, nt, d) in enumerate((([2, 4, 20], 3, 4), ([0, 1, 2, 5, 15, 26], 6, 6), ([3, 7, 11, 19, 23, 24, 25, 26], 4, 9))):
        f = few_feature_forest(cols, nt, d, seed=20 + i)
        yield f"grown{i}", f, synth.quick_features(synth.raw_fields(6, seed=40 + i))[:300], rng
    f, xq = sklearn_forest([1, 2, 4, 18, 20, 22], n_trees=4, max_depth=6)
    yield "sklearn", f, xq[:300], rng


@pytest.mark.parametrize("case", ["grown0", "grown1", "grown2", "sklearn"])
def test_oracle_exact_is_brute_force_shapley(oracle, tmp_path, case):
    name, forest, x, rng = next(c for c in _cases() if c[0] == case)
    x = with_missing(on_thresholds(x, forest, rng), rng)
    m, _ = _model(oracle, forest, tmp_path, name)
    got = oc.predict_contribs(m, x)
    ref = oc.shapley_brute_force(forest, x)
    assert_shap_close(got, ref, name)
    # additivity: the row's contributions and bias sum to the margin
    margin = m.predict(x, option_mask=1).astype(np.float64)
    assert np.allclose(got.astype(np.float64).sum(axis=1), margin, rtol=1e-5, atol=1e-5)
    # a shorter forest: only the first trees count
    assert_shap_close(oc.predict_contribs(m, x, ntree_limit=2), oc.shapley_brute_force(forest, x, ntree_limit=2), name)


@pytest.mark.parametrize("case", ["grown1", "sklearn"])
def test_oracle_approximate_is_naive_saabas_bit_for_bit(oracle, tmp_path, case, small_forest):
    name, forest, x, rng = next(c for c in _cases() if c[0] == case)
    x = with_missing(on_thresholds(x, forest, rng), rng)
    m, _ = _model(oracle, forest, tmp_path, name)
    assert np.array_equal(oc.predict_contribs(m, x, approximate=True), oc.saabas(forest, x))
    assert np.array_equal(oc.predict_contribs(m, x, approximate=True, ntree_limit=3), oc.saabas(forest, x, ntree_limit=3))
    ms, _ = _model(oracle, small_forest, tmp_path, "small")
    xs = with_missing(synth.quick_features(synth.raw_fields(6, seed=3))[:400], rng)
    assert np.array_equal(oc.predict_contribs(ms, xs, approximate=True), oc.saabas(small_forest, xs))


@pytest.mark.parametrize("case", ["grown2", "sklearn", "small"])
def test_path_tables_replay_like_the_recursive_oracle(capi, oracle, tmp_path, case, small_forest):
    """forest.cpp build_shap: the paths with merged repeated features, key bounds, missing flags and zero fractions,
    replayed in the path form the exact kernel runs, give the recursive oracle's contributions — also for a matrix
    with fewer columns than the booster has features."""
    rng = np.random.default_rng(5)
    if case == "small":
        forest, x = small_forest, synth.quick_features(synth.raw_fields(6, seed=8))[:200]
    else:
        _, forest, x, _ = next(c for c in _cases() if c[0] == case)
        x = x[:200]
    x = with_missing(on_thresholds(x, forest, rng), rng)
    m, p = _model(oracle, forest, tmp_path, case)
    b = capi.Booster(p, parse_only=True)
    bins, tree_bin, mean = b.shap_paths()
    assert tree_bin[0] == 0 and tree_bin[-1] == len(bins) and np.all(np.diff(tree_bin) >= 1)
    assert b.info().num_nodes == len(mean)
    ref = oc.predict_contribs(m, x)
    got = replay_paths(bins, tree_bin, x, NF)
    nodes, off, _, _ = b.flat()
    bias = np.float32(0)
    for t in range(len(off) - 1):
        bias = np.float32(bias + np.float32(np.float32(0) + mean[off[t]]))
    bias = np.float32(bias + np.float32(forest.base_score))
    assert np.all(ref[:, NF] == bias)
    assert_shap_close(np.concatenate([got, ref[:, NF:]], axis=1), ref, case)
    # the node means are libxgboost's, bit for bit
    _, _, _, orig = b.flat()
    for t, tree in enumerate(forest.trees):
        assert np.array_equal(mean[off[t] : off[t + 1]], oc.node_means(tree)[orig[off[t] : off[t + 1]]])
    xn = x[:, :20]  # absent columns count as missing
    assert_shap_close(np.concatenate([replay_paths(bins, tree_bin, xn, NF), ref[:, NF:]], axis=1), oc.predict_contribs(m, xn), case)
    assert_shap_close(np.concatenate([replay_paths(bins, tree_bin, x, NF, ntree=2), ref[:, NF:]], axis=1),
                      np.concatenate([oc.predict_contribs(m, x, ntree_limit=2)[:, :NF], ref[:, NF:]], axis=1), case)  # fmt: skip


def test_boosters_without_covers_are_rejected(capi, oracle, tmp_path, small_forest):
    for name in ("tiny.model", "tiny.json", "tiny.ubj"):
        b = capi.Booster(os.path.join(GOLD, name), parse_only=True)
        with pytest.raises(capi.QcohError, match="cover"):
            b.shap_paths()
        with pytest.raises(capi.QcohError, match="cannot be explained"):
            b.predict_contribs(None)
    f = synth.random_forest_structure(3, 5, seed=1)
    p = str(tmp_path / "nocover.model")
    xgbmodel.write_legacy_binary(f, p)
    with pytest.raises(capi.QcohError, match="sum_hess"):
        capi.Booster(p, parse_only=True).shap_paths()
    with pytest.raises(oc.OracleContribsError, match="cover"):
        oc.predict_contribs(oracle.Model(p), np.zeros((2, NF), np.float32))
    # the grown boosters (small_forest, the bench booster) have a positive cover at every internal node
    for t in small_forest.trees:
        assert np.all(t.sum_hess[t.left != -1] > 0)
    p = str(tmp_path / "small.model")
    xgbmodel.write_legacy_binary(small_forest, p)
    bins, _, _ = capi.Booster(p, parse_only=True).shap_paths()
    assert len(bins) > 0


def test_predict_from_dmatrix_config_errors(capi, small_model_path):
    b = capi.Booster(small_model_path, parse_only=True)
    ok = {"type": 2, "training": False, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}
    for k in ok:
        with pytest.raises(capi.QcohError, match=f"missing the key '{k}'"):
            b.predict_from_dmatrix(None, {kk: v for kk, v in ok.items() if kk != k})
    for ty in (4, 5):
        with pytest.raises(capi.QcohError, match="interaction"):
            b.predict_from_dmatrix(None, dict(ok, type=ty))
    with pytest.raises(capi.QcohError, match="unknown prediction type"):
        b.predict_from_dmatrix(None, dict(ok, type=7))
    for ty in (2, 3):
        with pytest.raises(capi.QcohError, match="iteration_begin = 0"):
            b.predict_from_dmatrix(None, dict(ok, type=ty, iteration_begin=1, iteration_end=3))
    with pytest.raises(capi.QcohError, match="iteration_begin = 2 is not supported"):
        b.predict_from_dmatrix(None, dict(ok, type=0, iteration_begin=2))
    with pytest.raises(capi.QcohError, match="not valid JSON"):
        b.predict_from_dmatrix(None, "{type: 2")
    if capi.device_count() == 0:
        for ty in (0, 1, 2, 3, 6):
            with pytest.raises(capi.QcohError, match="no CPU fallback"):
                b.predict_from_dmatrix(None, dict(ok, type=ty))
