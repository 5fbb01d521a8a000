"""SHAP interaction values on the CPU: the oracle's restatement of libxgboost 1.6.0 PredictInteractionContributions
against the Shapley interaction index from its definition and hand-derived answers; the conditioned path form the
interactions kernel runs, replayed in numpy on the library's path tables, against the oracle; refusals."""
import os

import numpy as np
import pytest

from contribs_forests import NF, on_thresholds, stump, with_missing
import oracle_contribs as oc
import oracle_interactions as oi
from interactions_forests import assert_interactions_close, replay_interactions
from quickchem_b200 import synth, xgbmodel
from test_contribs_cpu import _cases, _model

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("case", ["grown0", "grown1", "grown2", "sklearn"])
def test_oracle_is_the_brute_force_interaction_index(oracle, tmp_path, case):
    name, forest, x, rng = next(c for c in _cases() if c[0] == case)
    x = with_missing(on_thresholds(x, forest, rng), rng)[:120]
    m, _ = _model(oracle, forest, tmp_path, name)
    got = oi.predict_interactions(m, x)
    assert_interactions_close(got, oi.shapley_interactions_brute_force(forest, x), name)
    # rows sum to the contributions, the matrix to the margin; the bias entry is the contributions' bias, bit for bit
    phi = oc.predict_contribs(m, x)
    assert np.array_equal(got[:, NF, NF], phi[:, NF])
    assert np.all(got[:, NF, :NF] == 0) and np.all(got[:, :NF, NF] == 0)
    scale = np.abs(got).astype(np.float64).sum(axis=(1, 2))
    assert np.all(np.abs(got.astype(np.float64).sum(axis=2) - phi).max(axis=1) <= 1e-5 * scale)
    margin = m.predict(x, option_mask=1).astype(np.float64)
    assert np.all(np.abs(got.astype(np.float64).sum(axis=(1, 2)) - margin) <= 1e-5 * scale)
    unused = np.setdiff1d(np.arange(NF), np.unique(np.concatenate([t.split_index[t.left != -1] for t in forest.trees])))
    assert np.all(got[:, unused, :] == 0) and np.all(got[:, :, unused] == 0)
    assert_interactions_close(oi.predict_interactions(m, x, ntree_limit=2),
                              oi.shapley_interactions_brute_force(forest, x, ntree_limit=2), name)  # fmt: skip


@pytest.mark.parametrize("default_left", [True, False])
def test_stump_has_no_interactions(oracle, tmp_path, default_left):
    """One split feature: the off-diagonal is 0 and the diagonal is phi."""
    f = 5
    forest = stump(f, 0.5, default_left, -1.25, 2.0, 3.0, 5.0)
    m, _ = _model(oracle, forest, tmp_path, "stump")
    x = np.zeros((4, NF), np.float32)
    x[:, f] = [0.25, 0.5, 0.75, -999.0]
    got = oi.predict_interactions(m, x)
    phi = oc.predict_contribs(m, x)
    off = got.copy()
    off[:, np.arange(NF + 1), np.arange(NF + 1)] = 0
    assert np.all(off == 0)
    assert np.array_equal(np.diagonal(got, axis1=1, axis2=2), phi)


def test_two_feature_tree_pair_value(oracle, tmp_path):
    """Root on feature a, both children on feature b, covers n = 4 + 4 + 4 + 4, leaves (v_ll, v_lr, v_rl, v_rr).  With
    x left of both thresholds, the Shapley interaction index of the pair is
        Phi_ab = 1/2 [v(ab) - v(a) - v(b) + v({})],
    v(ab) = v_ll, v(a) = (v_ll + v_lr) / 2, v(b) = (v_ll + v_rl) / 2, v({}) = mean of the four leaves."""
    a, b = 2, 9
    vll, vlr, vrl, vrr = 1.0, -2.0, 0.5, 4.0
    t = xgbmodel.tree_from_nested((a, 0.0, True, (b, 0.0, True, vll, vlr), (b, 1.0, False, vrl, vrr)))
    t.sum_hess = np.full(len(t.left), 4.0, np.float32)
    t.sum_hess[t.left != -1] = [16.0, 8.0, 8.0]
    forest = xgbmodel.Forest(trees=[t], base_score=0.0, num_feature=NF)
    m, _ = _model(oracle, forest, tmp_path, "pair")
    x = np.zeros((1, NF), np.float32)
    x[0, a], x[0, b] = -1.0, -1.0
    want = 0.5 * (vll - (vll + vlr) / 2 - (vll + vrl) / 2 + (vll + vlr + vrl + vrr) / 4)
    got = oi.predict_interactions(m, x)
    assert got[0, a, b] == pytest.approx(want, abs=1e-6) and got[0, b, a] == pytest.approx(want, abs=1e-6)
    assert np.allclose(oi.shapley_interactions_brute_force(forest, x)[0, a, b], want, atol=1e-12)


@pytest.mark.parametrize("case", ["grown2", "sklearn", "small"])
def test_path_tables_replay_the_interactions(capi, oracle, tmp_path, case, small_forest):
    """The conditioned path form on forest.cpp's bins gives the recursive oracle's interaction values, with fewer
    columns than features and a tree limit too."""
    rng = np.random.default_rng(9)
    if case == "small":
        forest, x = small_forest, synth.quick_features(synth.raw_fields(6, seed=8))[:40]
    else:
        _, forest, x, _ = next(c for c in _cases() if c[0] == case)
        x = x[:40]
    x = with_missing(on_thresholds(x, forest, rng, k=40), rng)
    m, p = _model(oracle, forest, tmp_path, case)
    bins, tree_bin, _ = capi.Booster(p, parse_only=True).shap_paths()

    def full(feat_block, ref):
        out = ref.astype(np.float64).copy()
        out[:, :NF, :NF] = feat_block
        return out

    ref = oi.predict_interactions(m, x)
    assert_interactions_close(full(replay_interactions(bins, tree_bin, x, NF), ref), ref, case)
    xn = x[:, :20]
    ref = oi.predict_interactions(m, xn)
    assert_interactions_close(full(replay_interactions(bins, tree_bin, xn, NF), ref), ref, case)
    ref = oi.predict_interactions(m, x, ntree_limit=2)
    assert_interactions_close(full(replay_interactions(bins, tree_bin, x, NF, ntree=2), ref), ref, case)


@pytest.mark.parametrize("case", ["grown1", "sklearn"])
def test_oracle_approximate_is_the_saabas_diagonal(oracle, tmp_path, case):
    name, forest, x, rng = next(c for c in _cases() if c[0] == case)
    x = with_missing(on_thresholds(x, forest, rng), rng)[:100]
    m, _ = _model(oracle, forest, tmp_path, name)
    for ntree in (0, 3):
        got = oi.predict_interactions(m, x, approximate=True, ntree_limit=ntree)
        want = np.zeros_like(got)
        want[:, np.arange(NF + 1), np.arange(NF + 1)] = np.float32(0) + oc.predict_contribs(m, x, approximate=True, ntree_limit=ntree)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_refusals(capi, oracle, tmp_path, small_model_path):
    for name in ("tiny.model", "tiny.json", "tiny.ubj"):
        b = capi.Booster(os.path.join(GOLD, name), parse_only=True)
        with pytest.raises(capi.QcohError, match="cannot be explained"):
            b.predict_interactions_device(None, None)
    with pytest.raises(capi.QcohError, match="Invalid booster handle"):
        capi.check(capi.lib().qcoh_booster_predict_interactions_device(None, None, 0, 0, None))
    p = str(tmp_path / "nocover.model")
    xgbmodel.write_legacy_binary(synth.random_forest_structure(3, 5, seed=1), p)
    with pytest.raises(capi.QcohError, match="cannot be explained"):
        capi.Booster(p, parse_only=True).predict_interactions_device(None, None)
    with pytest.raises(oc.OracleContribsError, match="cover"):
        oi.predict_interactions(oracle.Model(p), np.zeros((2, NF), np.float32))
    if capi.device_count() == 0:
        b = capi.Booster(small_model_path, parse_only=True)
        for approximate in (False, True):
            with pytest.raises(capi.QcohError, match="no CPU fallback"):
                b.predict_interactions_device(None, None, approximate=approximate)
