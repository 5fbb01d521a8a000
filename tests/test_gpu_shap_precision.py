"""Exact contributions and interaction values on the GPU held entry by entry to the extended-precision reference
(tests/oracle_shap_exact.c), at the edges of the path tables: every path length up to a full bin, repeated splits at
signed zeros, denormals and +-FLT_MAX, 1 / 15 / 16 / 17 bins against the 16 slices, extreme cover ratios, row counts
around the tile and chunk sizes, absent columns, and every entry point.

The kernels compute in float64 and round each output once, so against the reference run on the zero fractions the
tables hold (z~, float32):   |got - ref| <= 1/2 ulp32(max(|got|, |ref|)) + 2^-30 A,
and against the exact zero fractions:   |got - ref| <= 1/2 ulp32 + (D_max + 1) 2^-24 A,
A the entry's magnitude from the reference and D_max the most elements on one path: the float32 storage of z is the
only approximation.  2^-30 and not float64's 2^-52: unwinding (UnwoundPathSum) loses bits on long paths.  The path
form replayed in numpy float64 (contribs_forests.replay_paths, interactions_forests.replay_interactions) is off the
reference by up to 2^-37.8 A (contributions) and 2^-32.2 A (interaction values) on the 31-level caterpillar, and the
kernels by no more.  A float32 path weight or row sum is off by about 2^-24 A and fails.  The bias entries are
bit-equal to the float32 oracle's."""

import numpy as np
import pytest

import oracle_contribs as oc
import oracle_shap_exact as se
import shap_edge_forests as ef
from conftest import inject_specials
from contribs_forests import NF, few_feature_forest, sklearn_forest
from quickchem_b200 import synth, xgbmodel

pytestmark = pytest.mark.gpu

CFG = {"type": 2, "training": False, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}


@pytest.fixture(scope="module")
def gpu(capi):
    if capi.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return capi


@pytest.fixture(scope="module")
def models(tmp_path_factory, small_forest, oracle):
    """name -> (legacy model path, forest, oracle model); the grown boosters of test_gpu_contribs.py and the edge
    boosters of shap_edge_forests.py."""
    d = tmp_path_factory.mktemp("shap_precision")
    forests = {
        "small": small_forest,
        "prod10x18": synth.prod_like_booster(n_trees=10, max_depth=18, n_sample=40000, grid_n=24, seed=11),
        "many_trees": few_feature_forest(list(range(0, 27, 2)), 130, 6, seed=31, n_sample=4000),
        "sklearn": sklearn_forest([0, 1, 2, 4, 18, 20, 22, 26], n_trees=5, max_depth=8)[0],
        "caterpillar": ef.caterpillar()[0],
        "caterpillar_mirror": ef.caterpillar(mirror=True)[0],
        "repeats": ef.repeats(),
        "covers": ef.covers(),
        "leaves": ef.single_leaves(),
        **{f"stumps{nb}": ef.stumps(nb, seed=nb) for nb in (1, 15, 16, 17)},
    }
    out = {}
    for name, f in forests.items():
        p = str(d / f"{name}.model")
        xgbmodel.write_legacy_binary(f, p)
        out[name] = (p, f, oracle.Model(p))
    return out


def _grown_rows(n, seed, forest, ncol=NF):
    x = synth.quick_features(synth.raw_fields(12, seed=seed))
    rng = np.random.default_rng(seed)
    x = inject_specials(x[rng.choice(x.shape[0], n, replace=x.shape[0] < n)], forest, rng)
    return np.ascontiguousarray(x[:, :ncol])


def _rows(name, forest, n, seed):
    if name.startswith("caterpillar"):
        _, thr, cont = ef.caterpillar(mirror=name.endswith("mirror"))
        return ef.caterpillar_rows(thr, cont, n, seed)
    if name in ("repeats", "covers") or name.startswith("stumps") or name == "leaves":
        return ef.special_rows(forest if name != "leaves" else ef.stumps(3), n, seed)
    return _grown_rows(n, seed, forest)


def _ulp32(a):
    return np.spacing(np.abs(np.asarray(a, np.float64)).astype(np.float32)).astype(np.longdouble)


def assert_entries_close(got, ref, mag, dmax, what):
    """Both bars above, entry by entry (bias entries excluded); prints and returns the worst ratio to each bar."""
    g = np.asarray(got, np.float32).astype(np.longdouble)
    worst = []
    for (r, a), rel in zip(((ref[0], mag[0]), (ref[1], mag[1])), (np.longdouble(2.0**-30), np.longdouble((dmax + 1) * 2.0**-24))):
        h = 0.5 * _ulp32(np.maximum(np.abs(g), np.abs(r)))
        ratio = np.abs(g - r) / (h + rel * a)
        i = np.unravel_index(int(np.argmax(ratio)), ratio.shape) if ratio.size else ()
        w = float(ratio.max()) if ratio.size else 0.0
        worst.append(w)
        assert w <= 1.0, f"{what}: |got - ref| / bar = {w:.3g} at {i}: got {g[i]!r} ref {r[i]!r} A {a[i]!r}"
    print(f"{what}: worst |got - ref| / bar = {worst[0]:.3g} (z~), {worst[1]:.3g} (exact z); D_max {dmax}")
    return worst


def check_contribs(got, m, x, what, ntree_limit=0):
    """Exact contributions against the reference in both modes; the bias column bit-equal to the float32 oracle's."""
    nf = m.num_feature
    ref, mag, dmax = se.contributions(m, x, ntree_limit=ntree_limit)
    refx, magx, _ = se.contributions(m, x, ntree_limit=ntree_limit, exact_z=True)
    assert got.shape == ref.shape
    bias = oc.predict_contribs(m, x[:1], ntree_limit=ntree_limit)[0, nf]
    assert np.all(got[:, nf].view(np.uint32) == np.float32(bias).view(np.uint32)), what
    assert np.all(ref[:, nf].astype(np.float32) == bias)
    return assert_entries_close(got[:, :nf], (ref[:, :nf], refx[:, :nf]), (mag[:, :nf], magx[:, :nf]), dmax, what)


def check_interactions(got, m, x, what, ntree_limit=0, contribs=None):
    nf = m.num_feature
    ref, mag, dmax = se.interactions(m, x, ntree_limit=ntree_limit)
    refx, magx, _ = se.interactions(m, x, ntree_limit=ntree_limit, exact_z=True)
    assert got.shape == ref.shape
    assert np.all(got[:, nf, :nf] == 0) and np.all(got[:, :nf, nf] == 0)
    if contribs is not None:
        assert np.array_equal(got[:, nf, nf].view(np.uint32), contribs[:, nf].view(np.uint32))
    return assert_entries_close(got[:, :nf, :nf], (ref[:, :nf, :nf], refx[:, :nf, :nf]),
                                (mag[:, :nf, :nf], magx[:, :nf, :nf]), dmax, what)  # fmt: skip


def _contribs(gpu, path, x, ntree_limit=0):
    b = gpu.Booster(path)
    dm = gpu.DMatrix(x)
    got = b.predict_contribs(dm, ntree_limit=ntree_limit)
    assert gpu.last_predict_kernel() == "shap"
    return b, dm, got


EDGE = ["caterpillar", "caterpillar_mirror", "repeats", "covers", "stumps1", "stumps15", "stumps16", "stumps17"]


@pytest.mark.parametrize("name", EDGE + ["small", "sklearn", "prod10x18", "many_trees"])
def test_contributions_entry_by_entry(gpu, oracle, models, name):
    path, forest, m = models[name]
    n = 300 if name not in ("prod10x18", "many_trees") else 200
    x = _rows(name, forest, n, seed=5)
    b, dm, got = _contribs(gpu, path, x)
    check_contribs(got, m, x, name)


@pytest.mark.parametrize("name", EDGE + ["small", "sklearn", "prod10x18", "many_trees"])
def test_interactions_entry_by_entry(gpu, oracle, models, name):
    path, forest, m = models[name]
    n = {"prod10x18": 12, "many_trees": 24, "caterpillar": 48, "caterpillar_mirror": 48}.get(name, 120)
    x = _rows(name, forest, n, seed=6)
    b, dm, phi = _contribs(gpu, path, x)
    got = b.predict_interactions(dm)
    assert gpu.last_predict_kernel() == "shap_inter"
    check_interactions(got, m, x, name, contribs=phi)


def test_tree_limits(gpu, oracle, models):
    path, forest, m = models["many_trees"]
    x = _rows("many_trees", forest, 64, seed=7)
    b, dm, _ = _contribs(gpu, path, x)
    for ntree in (1, 121, 130, 500):
        check_contribs(b.predict_contribs(dm, ntree_limit=ntree), m, x, f"many_trees ntree_limit {ntree}", ntree)
        xi = x[:16]
        dmi = gpu.DMatrix(xi)
        phi = b.predict_contribs(dmi, ntree_limit=ntree)
        check_interactions(b.predict_interactions(dmi, ntree_limit=ntree), m, xi, f"many_trees interactions ntree_limit {ntree}",
                           ntree, contribs=phi)  # fmt: skip


def test_single_leaf_trees_give_positive_zeros(gpu, oracle, models):
    path, forest, m = models["leaves"]
    x = _rows("leaves", forest, 257, seed=8)
    b, dm, got = _contribs(gpu, path, x)
    assert np.all(got[:, :NF].view(np.uint32) == 0)
    want = oc.predict_contribs(m, x)
    assert np.array_equal(got[:, NF].view(np.uint32), want[:, NF].view(np.uint32))
    inter = b.predict_interactions(dm)
    z = inter.copy()
    z[:, NF, NF] = 0
    assert np.all(z.view(np.uint32) == 0)
    assert np.array_equal(inter[:, NF, NF].view(np.uint32), want[:, NF].view(np.uint32))


@pytest.mark.parametrize("nrow", [1, 255, 256, 257, 4096, 4097, 32768, 32769])
def test_row_counts(gpu, oracle, models, nrow):
    """Tiles of 256 rows, 4 096-row interaction chunks and 32 768-row contribution chunks, on the repeats booster."""
    path, forest, m = models["repeats"]
    x = _rows("repeats", forest, nrow, seed=nrow)
    b, dm, got = _contribs(gpu, path, x)
    check_contribs(got, m, x, f"repeats {nrow} rows")
    if nrow <= 4097:
        check_interactions(b.predict_interactions(dm), m, x, f"repeats interactions {nrow} rows", contribs=got)


@pytest.mark.parametrize("ncol", [19, 1])
def test_absent_columns(gpu, oracle, models, ncol):
    for name in ("small", "caterpillar"):
        path, forest, m = models[name]
        x = np.ascontiguousarray(_rows(name, forest, 300, seed=9)[:, :ncol])
        b, dm, got = _contribs(gpu, path, x)
        check_contribs(got, m, x, f"{name} ncol {ncol}")
        xi = x[:40]
        dmi = gpu.DMatrix(xi)
        check_interactions(b.predict_interactions(dmi), m, xi, f"{name} interactions ncol {ncol}", contribs=b.predict_contribs(dmi))


def test_entry_points(gpu, oracle, models):
    """predict_contribs, the device call and XGBoosterPredictFromDMatrix type 2; interactions through the host wrapper
    and the device call; and a DMatrix built from device columns."""
    import torch

    path, forest, m = models["caterpillar_mirror"]
    x = _rows("caterpillar_mirror", forest, 700, seed=10)
    b, dm, host = _contribs(gpu, path, x)
    nc = forest.num_feature + 1
    out = gpu.DeviceArray(x.shape[0] * nc)
    b.predict_contribs_device(dm, out)
    gpu.synchronize()
    dev = out.get().reshape(-1, nc)
    out.free()
    typed = b.predict_from_dmatrix(dm, CFG)
    for what, got in (("predict_contribs", host), ("predict_contribs_device", dev), ("predict_from_dmatrix type 2", typed)):
        check_contribs(got, m, x, f"caterpillar_mirror {what}")
    xi = x[:64]
    dmi = gpu.DMatrix(xi)
    phi = b.predict_contribs(dmi)
    out = gpu.DeviceArray(xi.shape[0] * nc * nc)
    b.predict_interactions_device(dmi, out)
    gpu.synchronize()
    dev = out.get().reshape(-1, nc, nc)
    out.free()
    for what, got in (("predict_interactions", b.predict_interactions(dmi)), ("predict_interactions_device", dev)):
        check_interactions(got, m, xi, f"caterpillar_mirror {what}", contribs=phi)
    # a DMatrix from device columns (XGDMatrixCreateFromCudaColumnar)
    t = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    dmc = gpu.DMatrix.from_columns([t[c] for c in range(x.shape[1])], -999.0)
    check_contribs(b.predict_contribs(dmc), m, x, "caterpillar_mirror from device columns")
    torch.cuda.synchronize()


def test_bench_booster_on_c90_rows(gpu, oracle):
    """The 100 x 18 production-shape booster on 32 C90 rows, contributions only."""
    import bench

    path = bench.booster_path()
    x = synth.quick_features(synth.raw_fields(90, seed=2024))
    x = x[np.random.default_rng(1).choice(x.shape[0], 32, replace=False)]
    oracle.use_all_cores()
    m = oracle.Model(path)
    b, dm, got = _contribs(gpu, path, x)
    check_contribs(got, m, x, "bench booster")


@pytest.mark.parametrize("name", ["underflow", "overflow"])
def test_unrepresentable_zero_fractions_are_refused(gpu, tmp_path, name):
    """A product of cover ratios that float32 holds as +0 or +inf is refused with a message, not explained wrongly."""
    p = str(tmp_path / f"{name}.model")
    xgbmodel.write_legacy_binary(getattr(ef, name)(), p)
    b = gpu.Booster(p)
    dm = gpu.DMatrix(ef.special_rows(getattr(ef, name)(), 8, seed=1))
    with pytest.raises(gpu.QcohError, match="tree 0 leaf 3 has .* on feature 0"):
        b.predict_contribs(dm)
    with pytest.raises(gpu.QcohError, match="positive, finite float32"):
        b.predict_interactions(dm)
    assert b.predict(dm).shape == (8,)  # prediction itself needs no path tables
