"""Per-feature contributions on the GPU (XGBoosterPredictFromDMatrix types 2 / 3, qcoh_booster_predict_contribs_device)
against the C oracle's restatement of libxgboost 1.6.0: exact TreeSHAP within the per-row bar of
contribs_forests.assert_shap_close, approximate contributions bit for bit; additivity, determinism, shapes, and the
kernel family that served."""
import os

import numpy as np
import pytest

from conftest import inject_specials
import oracle_contribs as oc
from contribs_forests import NF, assert_shap_close, few_feature_forest, sklearn_forest
from quickchem_b200 import synth, xgbmodel

pytestmark = pytest.mark.gpu

CFG = {"type": 2, "training": False, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}


@pytest.fixture(scope="module")
def gpu(capi):
    if capi.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return capi


@pytest.fixture(scope="module")
def boosters(tmp_path_factory, small_forest):
    """name -> (legacy model path for the oracle, model path for the library, forest)"""
    d = tmp_path_factory.mktemp("contribs")
    out = {}

    def add(name, forest, fmt="model"):
        legacy = str(d / f"{name}.model")
        xgbmodel.write_legacy_binary(forest, legacy)
        path = legacy
        if fmt == "json":
            path = str(d / f"{name}.json")
            xgbmodel.write_json(forest, path)
        elif fmt == "ubj":
            path = str(d / f"{name}.ubj")
            xgbmodel.write_ubj(forest, path)
        out[name] = (legacy, path, forest)

    add("small", small_forest)
    add("small_json", small_forest, "json")
    add("small_ubj", small_forest, "ubj")
    add("sklearn", sklearn_forest([0, 1, 2, 4, 18, 20, 22, 26], n_trees=5, max_depth=8)[0])
    add("prod10x18", synth.prod_like_booster(n_trees=10, max_depth=18, n_sample=40000, grid_n=24, seed=11))
    add("many_trees", few_feature_forest(list(range(0, 27, 2)), 130, 6, seed=31, n_sample=4000))
    return out


def _rows(n, seed, specials, forest):
    x = synth.quick_features(synth.raw_fields(12, seed=seed))
    rng = np.random.default_rng(seed)
    x = x[rng.choice(x.shape[0], n, replace=x.shape[0] < n)]
    return inject_specials(x, forest, rng) if specials else x


def _check(gpu, oracle, legacy, path, forest, x, ntree_limit=0):
    b = gpu.Booster(path)
    m = oracle.Model(legacy)
    dm = gpu.DMatrix(x)
    exact = b.predict_contribs(dm, ntree_limit=ntree_limit)
    assert gpu.last_predict_kernel() == "shap"
    worst = assert_shap_close(exact, oc.predict_contribs(m, x, ntree_limit=ntree_limit), os.path.basename(path))
    approx = b.predict_contribs(dm, approximate=True, ntree_limit=ntree_limit)
    assert gpu.last_predict_kernel() == "shap_approx"
    assert np.array_equal(approx, oc.predict_contribs(m, x, approximate=True, ntree_limit=ntree_limit))
    # additivity, independent of the oracle: sum_f phi_f + bias is the margin
    margin = b.predict_from_dmatrix(dm, dict(CFG, type=1, iteration_end=ntree_limit)).astype(np.float64)
    for c in (exact, approx):
        s = c.astype(np.float64).sum(axis=1)
        assert np.all(np.abs(s - margin) <= 1e-5 * np.maximum(np.abs(c).sum(axis=1), 1.0)), np.abs(s - margin).max()
    return worst


@pytest.mark.parametrize("name", ["small", "small_json", "small_ubj", "sklearn", "prod10x18", "many_trees"])
@pytest.mark.parametrize("specials", [False, True], ids=["clean", "specials"])
def test_contribs_match_the_oracle(gpu, oracle, boosters, name, specials):
    legacy, path, forest = boosters[name]
    x = _rows(700, 3, specials, forest)
    before = gpu.kernel_launches("shap_reduce")
    _check(gpu, oracle, legacy, path, forest, x)
    assert gpu.kernel_launches("shap_reduce") == before + 1


@pytest.mark.parametrize("nrow", [1, 255, 257, 1000])
def test_row_counts_and_tree_limits(gpu, oracle, boosters, nrow):
    legacy, path, forest = boosters["small"]
    x = _rows(nrow, 5, True, forest)
    for ntree in (0, 1, 5):
        _check(gpu, oracle, legacy, path, forest, x, ntree_limit=ntree)


def test_many_trees_with_a_limit(gpu, oracle, boosters):
    legacy, path, forest = boosters["many_trees"]
    x = _rows(300, 9, True, forest)
    for ntree in (121, 130, 500):
        _check(gpu, oracle, legacy, path, forest, x, ntree_limit=ntree)


def test_fewer_columns_than_features(gpu, oracle, boosters):
    legacy, path, forest = boosters["small"]
    x = _rows(600, 7, True, forest)[:, :19]
    _check(gpu, oracle, legacy, path, forest, x)


def test_bench_booster_on_c90_rows(gpu, oracle):
    import bench

    path = bench.booster_path()
    x = synth.quick_features(synth.raw_fields(90, seed=2024))
    x = x[np.random.default_rng(1).choice(x.shape[0], 300, replace=False)]
    oracle.use_all_cores()
    worst = _check(gpu, oracle, path, path, None, x)
    print(f"bench booster: max |dphi| / (sum |phi| + |bias|) = {worst:.2e}")


def test_deterministic_across_calls_and_row_shardings(gpu, boosters):
    legacy, path, forest = boosters["prod10x18"]
    b = gpu.Booster(path)
    x = _rows(5000, 13, True, forest)
    full = b.predict_contribs(gpu.DMatrix(x))
    assert np.array_equal(full.view(np.uint32), b.predict_contribs(gpu.DMatrix(x)).view(np.uint32))
    for k in (1, 777, 2600):
        parts = [b.predict_contribs(gpu.DMatrix(x[:k])), b.predict_contribs(gpu.DMatrix(x[k:]))]
        assert np.array_equal(full.view(np.uint32), np.concatenate(parts).view(np.uint32)), k
    # the device variant writes the same bits
    dm = gpu.DMatrix(x)
    for approximate in (False, True):
        out = gpu.DeviceArray(x.shape[0] * (NF + 1))
        b.predict_contribs_device(dm, out, approximate=approximate)
        gpu.synchronize()
        host = b.predict_contribs(dm, approximate=approximate)
        assert np.array_equal(out.get().reshape(-1, NF + 1).view(np.uint32), host.view(np.uint32))
        out.free()


def test_predict_from_dmatrix_types_and_shapes(gpu, boosters):
    legacy, path, forest = boosters["small"]
    b = gpu.Booster(path)
    x = _rows(500, 17, True, forest)
    dm = gpu.DMatrix(x)
    n, nt = x.shape[0], forest.num_trees
    for strict in (False, True):
        for ty, mask, shape in ((0, 0, (n,)), (1, 1, (n,)), (6, 2, (n, nt))):
            got = b.predict_from_dmatrix(dm, dict(CFG, type=ty, strict_shape=strict))
            want = b.predict(dm, option_mask=mask)
            assert got.shape == (((n, 1) if ty != 6 else (n, nt, 1, 1)) if strict else shape)
            assert np.array_equal(got.reshape(want.shape).view(np.uint32), want.view(np.uint32))
            assert gpu.last_predict_kernel().startswith(("duo", "nodes8"))
        for ty in (2, 3):
            got = b.predict_from_dmatrix(dm, dict(CFG, type=ty, strict_shape=strict))
            assert got.shape == ((n, 1, NF + 1) if strict else (n, NF + 1))
    got = b.predict_from_dmatrix(dm, dict(CFG, type=6, iteration_end=4))
    assert np.array_equal(got, b.predict(dm, option_mask=2, ntree_limit=4))
    with pytest.raises(gpu.QcohError, match="interaction"):
        b.predict_from_dmatrix(dm, dict(CFG, type=4))
