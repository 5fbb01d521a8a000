"""SHAP interaction values on the GPU (qcoh_booster_predict_interactions_device) against the C oracle's restatement of
libxgboost 1.6.0 PredictInteractionContributions: exact values within the per-row bar of
interactions_forests.assert_interactions_close (and against the Shapley interaction index where few features are used),
approximate values bit for bit; row sums, margin, symmetry, the bias entries, determinism across calls, row shardings
and chunks, and the kernel families that served."""
import numpy as np
import pytest

import oracle_interactions as oi
from contribs_forests import NF
from interactions_forests import assert_interactions_close
from quickchem_b200 import synth
from test_gpu_contribs import CFG, _rows, boosters, gpu  # noqa: F401  (fixtures)

pytestmark = pytest.mark.gpu

def _check(gpu, oracle, legacy, path, forest, x, ntree_limit=0, brute=False):
    b = gpu.Booster(path)
    m = oracle.Model(legacy)
    dm = gpu.DMatrix(x)
    n = x.shape[0]
    launches = {f: gpu.kernel_launches(f) for f in ("shap", "shap_inter", "shap_inter_reduce", "shap_approx", "shap_inter_expand")}
    exact = b.predict_interactions(dm, ntree_limit=ntree_limit)
    assert gpu.last_predict_kernel() == "shap_inter"
    chunks = -(-n // 4096)
    for f in ("shap", "shap_inter", "shap_inter_reduce"):
        assert gpu.kernel_launches(f) == launches[f] + chunks, f
    assert exact.shape == (n, NF + 1, NF + 1)
    worst = assert_interactions_close(exact, oi.predict_interactions(m, x, ntree_limit=ntree_limit), path)
    if brute:
        assert_interactions_close(exact, oi.shapley_interactions_brute_force(forest, x, ntree_limit=ntree_limit), path)
    approx = b.predict_interactions(dm, approximate=True, ntree_limit=ntree_limit)
    assert gpu.last_predict_kernel() == "shap_approx"
    assert gpu.kernel_launches("shap_approx") == launches["shap_approx"] + 1
    assert gpu.kernel_launches("shap_inter_expand") == launches["shap_inter_expand"] + 1
    want = oi.predict_interactions(m, x, approximate=True, ntree_limit=ntree_limit)
    assert np.array_equal(approx.view(np.uint32), want.view(np.uint32))
    # independent of the oracle: rows sum to the contributions, the matrix to the margin, M is symmetric, and the
    # bias row and column are 0 but for the contributions' bias
    phi = b.predict_contribs(dm, ntree_limit=ntree_limit)
    margin = b.predict_from_dmatrix(dm, dict(CFG, type=1, iteration_end=ntree_limit)).astype(np.float64)
    e = exact.astype(np.float64)
    scale = np.maximum(np.abs(e).sum(axis=(1, 2)), 1.0)
    assert np.all(np.abs(e.sum(axis=2) - phi).max(axis=1) <= 1e-5 * scale)
    assert np.all(np.abs(e.sum(axis=(1, 2)) - margin) <= 1e-5 * scale)
    assert np.all(np.abs(e - e.transpose(0, 2, 1)).max(axis=(1, 2)) <= 1e-5 * scale)
    assert np.array_equal(exact[:, NF, NF].view(np.uint32), phi[:, NF].view(np.uint32))
    assert np.all(exact[:, NF, :NF] == 0) and np.all(exact[:, :NF, NF] == 0)
    return worst


@pytest.mark.parametrize("name,nrow,brute", [("small", 300, False), ("small_json", 100, False), ("small_ubj", 100, False),
                                             ("sklearn", 300, True), ("prod10x18", 24, False), ("many_trees", 60, False)])  # fmt: skip
@pytest.mark.parametrize("specials", [False, True], ids=["clean", "specials"])
def test_interactions_match_the_oracle(gpu, oracle, boosters, name, nrow, brute, specials):
    legacy, path, forest = boosters[name]
    worst = _check(gpu, oracle, legacy, path, forest, _rows(nrow, 3, specials, forest), brute=brute)
    print(f"{name}: max |dM| / sum |M| = {worst:.2e}")


@pytest.mark.parametrize("nrow", [1, 255, 257, 4500])
def test_row_counts_and_tree_limits(gpu, oracle, boosters, nrow):
    legacy, path, forest = boosters["small"]
    x = _rows(nrow, 5, True, forest)
    for ntree in (0, 1, 5):
        _check(gpu, oracle, legacy, path, forest, x, ntree_limit=ntree)


def test_many_trees_with_a_limit(gpu, oracle, boosters):
    legacy, path, forest = boosters["many_trees"]
    x = _rows(40, 9, True, forest)
    for ntree in (121, 130, 500):
        _check(gpu, oracle, legacy, path, forest, x, ntree_limit=ntree)


def test_fewer_columns_than_features(gpu, oracle, boosters):
    legacy, path, forest = boosters["small"]
    _check(gpu, oracle, legacy, path, forest, _rows(300, 7, True, forest)[:, :19])


def test_bench_booster_on_c90_rows(gpu, oracle):
    import bench

    path = bench.booster_path()
    x = synth.quick_features(synth.raw_fields(90, seed=2024))
    x = x[np.random.default_rng(1).choice(x.shape[0], 16, replace=False)]
    oracle.use_all_cores()
    worst = _check(gpu, oracle, path, path, None, x)
    print(f"bench booster: max |dM| / sum |M| = {worst:.2e}")


def test_deterministic_across_calls_shardings_and_chunks(gpu, boosters):
    """4 500 rows are two chunks of the exact path; the shardings put the chunk boundary at other rows."""
    legacy, path, forest = boosters["prod10x18"]
    b = gpu.Booster(path)
    x = _rows(4500, 13, True, forest)
    full = b.predict_interactions(gpu.DMatrix(x))
    assert np.array_equal(full.view(np.uint32), b.predict_interactions(gpu.DMatrix(x)).view(np.uint32))
    for k in (1, 777, 2600):
        parts = [b.predict_interactions(gpu.DMatrix(x[:k])), b.predict_interactions(gpu.DMatrix(x[k:]))]
        assert np.array_equal(full.view(np.uint32), np.concatenate(parts).view(np.uint32)), k
    # the device call writes what the host wrapper returns, and contributions calls in between change nothing
    dm = gpu.DMatrix(x)
    for approximate in (False, True):
        out = gpu.DeviceArray(x.shape[0] * (NF + 1) ** 2)
        b.predict_contribs(dm, approximate=not approximate)
        b.predict_interactions_device(dm, out, approximate=approximate)
        gpu.synchronize()
        host = b.predict_interactions(dm, approximate=approximate)
        assert np.array_equal(out.get().reshape(host.shape).view(np.uint32), host.view(np.uint32))
        out.free()
    with pytest.raises(gpu.QcohError, match="Invalid DMatrix handle"):
        b.predict_interactions_device(None, None)
    with pytest.raises(gpu.QcohError, match="interaction"):
        b.predict_from_dmatrix(dm, dict(CFG, type=5))
