"""GPU parity: XGDMatrixCreateFromMat + XGBoosterPredict of libqcoh.so (through the C ABI the
reference's xgb_fortran_api binds) against the CPU oracle on the same seeded inputs.

Bars: leaf indices bit-exact; the float32 margin is summed in the reference's tree order, so it
is compared bit-exactly too (stricter than the 1e-6 relative of BASELINE.json); the fused
10**x epilogue within 1e-6 relative (float64 exp10 on the device vs libm powf in the oracle)."""
import numpy as np
import pytest

from conftest import inject_specials
from quickchem_b200 import synth, xgbmodel

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("duo_mode")]

REL_TOL_OH = 1e-6  # BASELINE.json north_star: summed OH within max relative error 1e-6


def _both(capi, oracle, forest, x, tmp_path, missing=-999.0, **kw):
    p = str(tmp_path / "m.model")
    xgbmodel.write_legacy_binary(forest, p)
    b = capi.Booster(p)
    d = capi.DMatrix(x, missing)
    got = b.predict(d, **kw)
    ref = oracle.Model(p).predict(x, missing=missing, **kw)
    return got, ref


def test_known_answer_stump(capi, oracle, tmp_path):
    # one split on feature 3 at 0.5, default left; leaves -1 / +2; base_score 0.5
    f = xgbmodel.Forest(trees=[xgbmodel.tree_from_nested((3, 0.5, True, -1.0, 2.0))], base_score=0.5, num_feature=27)
    x = np.zeros((6, 27), np.float32)
    x[:, 3] = [0.0, 0.5, np.nextafter(np.float32(0.5), np.float32(0)), 1.0, -999.0, np.nan]
    got, ref = _both(capi, oracle, f, x, tmp_path)
    expect = np.float32(0.5) + np.array([-1, 2, -1, 2, -1, -1], np.float32)  # == threshold goes right
    assert np.array_equal(got, expect)
    assert np.array_equal(ref, expect)
    leaf, _ = _both(capi, oracle, f, x, tmp_path, option_mask=2)
    assert np.array_equal(leaf[:, 0], np.array([1, 2, 1, 2, 1, 1], np.float32))


def test_known_answer_defaults_and_signed_zero(capi, oracle, tmp_path):
    # depth-2 tree: root default-right, left child default-left; -0.0 vs 0.0 threshold; denormal
    t = xgbmodel.tree_from_nested((0, 0.0, False, (1, np.float32(1e-40), True, 10.0, 20.0), (2, -0.0, False, 30.0, 40.0)))
    f = xgbmodel.Forest(trees=[t], base_score=0.0, num_feature=27)
    rows = [
        (-1.0, 0.0, 0.0, 10.0),        # f0 < 0 -> left; f1=0 < 1e-40 -> 10
        (-1.0, 1e-40, 0.0, 20.0),      # equal to denormal threshold -> right
        (-1.0, np.nan, 0.0, 10.0),     # missing at default-left node
        (-0.0, 0.0, -1.0, 30.0),       # -0.0 < 0.0 is false -> right; f2=-1 < -0.0 -> 30
        (0.0, 0.0, 0.0, 40.0),         # 0.0 < -0.0 false -> 40
        (-999.0, 0.0, -0.0, 40.0),     # missing at root -> default right; -0.0 < -0.0 false
        (np.nan, 0.0, np.nan, 40.0),   # missing, missing -> right, right
    ]
    x = np.zeros((len(rows), 27), np.float32)
    for i, r in enumerate(rows):
        x[i, :3] = r[:3]
    got, ref = _both(capi, oracle, f, x, tmp_path)
    expect = np.array([r[3] for r in rows], np.float32)
    assert np.array_equal(ref, expect)
    assert np.array_equal(got, expect)


def test_known_answer_sum_order(capi, oracle, tmp_path):
    # 100 single-leaf trees whose float32 sum depends on the order of addition
    vals = [1e8, 1.0, -1e8, 1.0] * 25
    f = xgbmodel.Forest(trees=[xgbmodel.tree_from_nested(float(v)) for v in vals], base_score=0.5, num_feature=27)
    x = np.zeros((3, 27), np.float32)
    got, ref = _both(capi, oracle, f, x, tmp_path)
    acc = np.float32(0.5)
    for v in vals:
        acc = np.float32(acc + np.float32(v))
    assert np.all(got == acc) and np.all(ref == acc)
    assert acc != np.float32(0.5 + 50.0)  # a tree-reduced sum would give 50.5


@pytest.mark.parametrize("nrow", [1, 31, 255, 256, 257, 1000, 4099])
def test_ragged_sizes(capi, oracle, tmp_path, small_forest, nrow):
    rng = np.random.default_rng(nrow)
    raw = synth.raw_fields(8, seed=3)
    x = synth.quick_features(raw)
    x = x[rng.choice(x.shape[0], nrow, replace=False)]
    got, ref = _both(capi, oracle, small_forest, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_empty_matrix(capi, small_model_path):
    b = capi.Booster(small_model_path)
    d = capi.DMatrix(np.zeros((0, 27), np.float32))
    assert d.num_row == 0 and d.num_col == 27
    assert b.predict(d).shape == (0,)


def test_c24_leaf_indices_and_sums(capi, oracle, tmp_path, small_forest):
    """configs[0]/[1]-style check at C24 x 72 with missing / NaN / on-threshold injections."""
    rng = np.random.default_rng(7)
    x = synth.quick_features(synth.raw_fields(24))
    x = inject_specials(x, small_forest, rng)
    got, ref = _both(capi, oracle, small_forest, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    leaf, leaf_ref = _both(capi, oracle, small_forest, x, tmp_path, option_mask=2)
    assert leaf.shape == (x.shape[0], small_forest.num_trees)
    assert np.array_equal(leaf, leaf_ref)


def test_clean_matrix_takes_no_missing_path_and_matches(capi, oracle, tmp_path, small_forest):
    x = synth.quick_features(synth.raw_fields(12))
    assert not np.isnan(x).any() and not (x == -999.0).any()
    got, ref = _both(capi, oracle, small_forest, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    margin, _ = _both(capi, oracle, small_forest, x, tmp_path, option_mask=1)
    assert np.array_equal(margin, got)  # reg:squarederror: value == margin


def test_deep_forest_uncorrelated_rows(capi, oracle, tmp_path):
    f = synth.random_forest_structure(40, 14, seed=11, p_leaf=0.05)
    rng = np.random.default_rng(12)
    x = rng.normal(0, 1, (20000, 27)).astype(np.float32)
    x[rng.random(x.shape) < 0.02] = np.nan
    got, ref = _both(capi, oracle, f, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    leaf, leaf_ref = _both(capi, oracle, f, x, tmp_path, option_mask=2)
    assert np.array_equal(leaf, leaf_ref)


def test_ntree_limit(capi, oracle, tmp_path, small_forest):
    x = synth.quick_features(synth.raw_fields(6))
    for lim in (1, 5, 12, 100):
        got, ref = _both(capi, oracle, small_forest, x, tmp_path, ntree_limit=lim)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    leaf, leaf_ref = _both(capi, oracle, small_forest, x, tmp_path, option_mask=2, ntree_limit=5)
    assert leaf.shape[1] == 5 and np.array_equal(leaf, leaf_ref)


def test_fewer_columns_than_features(capi, oracle, tmp_path, small_forest):
    """Columns the matrix does not have count as missing (xgboost FVec::Fill)."""
    x = synth.quick_features(synth.raw_fields(6))[:, :20]
    got, ref = _both(capi, oracle, small_forest, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_other_missing_values(capi, oracle, tmp_path, small_forest):
    x = synth.quick_features(synth.raw_fields(6))
    x[::7, 2] = 0.0
    for missing in (0.0, np.nan, np.inf):
        xx = x.copy()
        if np.isinf(missing):
            xx[::5, 4] = np.inf
        got, ref = _both(capi, oracle, small_forest, xx, tmp_path, missing=missing)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_error_behaviour(capi, small_model_path, tmp_path):
    b = capi.Booster(small_model_path)
    x = np.zeros((4, 27), np.float32)
    x[1, 1] = np.inf
    with pytest.raises(capi.QcohError, match="inf"):
        capi.DMatrix(x)  # finite missing + inf data: libxgboost's CreateFromMat fails too
    with pytest.raises(capi.QcohError, match="Number of columns"):
        b.predict(capi.DMatrix(np.zeros((2, 28), np.float32)))
    with pytest.raises(capi.QcohError, match="columns"):
        capi.DMatrix(np.zeros((2, 500), np.float32))
    with pytest.raises(capi.QcohError, match="option_mask"):
        b.predict(capi.DMatrix(np.zeros((2, 27), np.float32)), option_mask=4)
    empty = capi.Booster()
    with pytest.raises(capi.QcohError, match="no model"):
        empty.predict(capi.DMatrix(np.zeros((2, 27), np.float32)))
    with pytest.raises(capi.QcohError):
        capi.Booster(str(tmp_path / "does_not_exist.model"))


def test_model_formats_agree_on_device(capi, tmp_path, small_forest):
    x = synth.quick_features(synth.raw_fields(6))
    outs = []
    for ext, wr in (("model", xgbmodel.write_legacy_binary), ("json", xgbmodel.write_json), ("ubj", xgbmodel.write_ubj)):
        p = str(tmp_path / ("m." + ext))
        wr(small_forest, p)
        outs.append(capi.Booster(p).predict(capi.DMatrix(x)))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


def test_device_resident_predict_and_epilogue(capi, oracle, small_model_path, small_forest):
    x = synth.quick_features(synth.raw_fields(12))
    b = capi.Booster(small_model_path)
    d = capi.DMatrix.device(x.shape[0], 27)
    d.upload(x[: x.shape[0] // 2], 0)
    d.upload(x[x.shape[0] // 2 :], x.shape[0] // 2)
    d.seal()
    out = capi.DeviceArray(x.shape[0])
    b.predict_device(d, out)
    capi.synchronize()
    ref = oracle.Model(small_model_path).predict(x)
    assert np.array_equal(out.get().view(np.uint32), ref.view(np.uint32))
    b.predict_device(d, out, exp10=True, scale=0.85)
    capi.synchronize()
    oh_ref = (np.float32(10.0) ** ref).astype(np.float32) * np.float32(0.85)
    rel = np.abs(out.get().astype(np.float64) - oh_ref) / np.abs(oh_ref)
    assert rel.max() <= REL_TOL_OH


def test_launch_shapes_agree(capi, oracle, tmp_path, small_model_path, small_forest, duo_mode):
    """Every launch shape of the predict kernels gives the oracle's bits, on both layouts of the duo_mode fixture.
    The two-level records run in the shallow shape on the small forest and in the default 6-wide shape on a forest
    whose records average more than 4 KB per tree; the 8-byte nodes run with the constant-memory table.
    ntree_limit 1, 5, 7 and 11 end the walks in the narrower groups (6-wide, 3-wide, single tree), and a matrix
    with missing entries takes the default-direction walk.  The 8-byte nodes without the table and the LSU-only
    fetch are covered by test_wide_tree_records_without_default_bits (nodes8_missing) and by the single-tree tail
    of every group walk."""
    deep = synth.random_forest_structure(13, 11, seed=6, p_leaf=0.12)
    deep_path = str(tmp_path / "deep.model")
    xgbmodel.write_legacy_binary(deep, deep_path)
    family = "duo" if duo_mode else "nodes8"
    rng = np.random.default_rng(5)
    for path, forest, x in ((small_model_path, small_forest, synth.quick_features(synth.raw_fields(8))),
                            (deep_path, deep, rng.normal(0, 1, (20000, 27)).astype(np.float32))):  # fmt: skip
        b, om = capi.Booster(path), oracle.Model(path)
        if forest is deep:
            assert b.duo()[0].nbytes >= 4096 * deep.num_trees  # not a shallow forest: the default launch shape
        d = capi.DMatrix(x)
        for nt in (0, 1, 5, 7, 11):
            assert np.array_equal(b.predict(d, ntree_limit=nt).view(np.uint32), om.predict(x, ntree_limit=nt).view(np.uint32)), (path, nt)
            assert capi.last_predict_kernel() == family
        xm = inject_specials(x, forest, rng)
        assert np.array_equal(b.predict(capi.DMatrix(xm)).view(np.uint32), om.predict(xm).view(np.uint32)), path
        assert capi.last_predict_kernel() == family + "_missing"


def test_pipelined_create_matches_plain_path(capi, oracle, tmp_path, small_model_path, small_forest):
    """XGDMatrixCreateFromMat pipelines H2D chunks with prediction by the process's booster; the
    answer must be the same as the plain path, and any other booster / option must not see it."""
    rng = np.random.default_rng(9)
    x = inject_specials(synth.quick_features(synth.raw_fields(8)), small_forest, rng)
    ref = oracle.Model(small_model_path).predict(x)
    other = synth.random_forest_structure(7, 6, seed=21)
    p2 = str(tmp_path / "other.model")
    xgbmodel.write_legacy_binary(other, p2)
    ref2 = oracle.Model(p2).predict(x)
    try:
        for chunk in (256, 1024, 1 << 21):
            capi.set_param("chunk_rows", chunk)
            for spec in (0, 1):
                capi.set_param("speculate", spec)
                b = capi.Booster(small_model_path)  # becomes the process's booster
                d = capi.DMatrix(x)
                assert np.array_equal(b.predict(d).view(np.uint32), ref.view(np.uint32)), (chunk, spec)
                assert np.array_equal(b.predict(d).view(np.uint32), ref.view(np.uint32))  # second call: plain path
                leaf = b.predict(capi.DMatrix(x), option_mask=2)  # options the pipeline did not assume
                assert leaf.shape == (x.shape[0], small_forest.num_trees)
                lim = b.predict(capi.DMatrix(x), ntree_limit=3)
                assert np.array_equal(lim.view(np.uint32), oracle.Model(small_model_path).predict(x, ntree_limit=3).view(np.uint32))
                b2 = capi.Booster(p2)  # now the last-loaded booster
                d2 = capi.DMatrix(x)   # pipelined for b2 ...
                assert np.array_equal(b.predict(d2).view(np.uint32), ref.view(np.uint32))   # ... asked of b
                assert np.array_equal(b2.predict(d2).view(np.uint32), ref2.view(np.uint32))
        capi.set_param("speculate", 1)
        xi = x.copy()
        xi[-1, 3] = np.inf  # inf in the last chunk still fails the create call
        capi.set_param("chunk_rows", 1024)
        with pytest.raises(capi.QcohError, match="inf"):
            capi.DMatrix(xi)
    finally:
        capi.set_param("chunk_rows", 0)
        capi.set_param("speculate", 1)


def test_result_buffer_lifetime(capi, small_model_path):
    """The prediction buffer belongs to the booster and stays valid until its next predict — also
    across the creation of the next matrix (which is pipelined into another pinned buffer)."""
    x1 = synth.quick_features(synth.raw_fields(6))
    x2 = x1[::-1].copy()
    b = capi.Booster(small_model_path)
    d1 = capi.DMatrix(x1)
    n, p = b.predict_raw(d1)
    first = np.ctypeslib.as_array(p, (n,)).copy()
    d2 = capi.DMatrix(x2)  # must not clobber p
    assert np.array_equal(np.ctypeslib.as_array(p, (n,)), first)
    d1.free()
    assert np.array_equal(np.ctypeslib.as_array(p, (n,)), first)
    assert np.array_equal(b.predict(d2), first[::-1])


def test_dmatrix_file_roundtrip(capi, tmp_path, small_model_path):
    x = synth.quick_features(synth.raw_fields(4))
    d = capi.DMatrix(x)
    p = str(tmp_path / "x.qcdm")
    d.save_binary(p)
    d2 = capi.DMatrix.from_file(p)
    assert (d2.num_row, d2.num_col) == x.shape
    b = capi.Booster(small_model_path)
    assert np.array_equal(b.predict(d), b.predict(d2))


def test_more_trees_than_the_constant_table_holds(capi, oracle, tmp_path, duo_mode):
    """The constant-memory table of tree tops holds 7680 nodes (480 trees x 16); a bigger forest runs on the
    two-level records (or, with duo = 0, the 8-byte nodes) in launches of 120 trees, the table re-filled with the
    next window of 480 trees when a launch leaves it, and still matches, with and without missing entries."""
    family = "duo" if duo_mode else "nodes8"
    rng = np.random.default_rng(8)
    trees = [xgbmodel.tree_from_nested((int(rng.integers(27)), float(rng.normal()), bool(rng.random() < 0.5),
                                        float(rng.normal()), (int(rng.integers(27)), float(rng.normal()), False, 1.0, -1.0)))
             for _ in range(650)]  # fmt: skip
    f = xgbmodel.Forest(trees=trees, base_score=0.25, num_feature=27)
    x = rng.normal(0, 1, (3000, 27)).astype(np.float32)
    got, ref = _both(capi, oracle, f, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert capi.last_predict_kernel() == family
    x[::3, 5] = np.nan
    got, ref = _both(capi, oracle, f, x, tmp_path)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert capi.last_predict_kernel() == family + "_missing"


def test_dmatrix_from_libsvm_and_csv(capi, oracle, tmp_path, small_model_path):
    """XGDMatrixCreateFromFile's text inputs: libsvm (absent entries are missing) and csv with a label column."""
    rng = np.random.default_rng(4)
    x = synth.quick_features(synth.raw_fields(4))[:300]
    x[rng.random(x.shape) < 0.1] = np.nan
    svm, csv = tmp_path / "x.libsvm", tmp_path / "x.csv"
    with open(svm, "w") as f:
        for r in x:
            f.write("0 " + " ".join(f"{j}:{float(v)!r}" for j, v in enumerate(r) if not np.isnan(v)) + "\n")
    with open(csv, "w") as f:
        for r in x:
            f.write("1.5," + ",".join("" if np.isnan(v) else repr(float(v)) for v in r) + "\n")
    x[:, -1] = np.where(np.isnan(x[:, -1]), x[:, -1], x[:, -1])  # (libsvm infers ncol from the largest index)
    ref = oracle.Model(small_model_path).predict(x, missing=np.nan)
    b = capi.Booster(small_model_path)
    d1 = capi.DMatrix.from_file(str(svm))
    d2 = capi.DMatrix.from_file(str(csv) + "?format=csv&label_column=0")
    assert d2.num_row == 300 and d2.num_col == 27 and d1.num_row == 300 and d1.num_col <= 27
    assert np.array_equal(b.predict(d1).view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(b.predict(d2).view(np.uint32), ref.view(np.uint32))
    with pytest.raises(capi.QcohError):
        capi.DMatrix.from_file(str(tmp_path / "missing_file.libsvm"))


def test_linearity_property_full_size(capi, small_model_path):
    """Size-independent property at a BASELINE-sized slab (C90 x 72 = 3.5 M rows): predicting the
    matrix in one call equals predicting its halves (rows are independent), and a permutation of
    rows permutes the output."""
    x = synth.quick_features(synth.raw_fields(90))
    b = capi.Booster(small_model_path)
    full = b.predict(capi.DMatrix(x))
    h = x.shape[0] // 2 + 13
    a = b.predict(capi.DMatrix(x[:h]))
    c = b.predict(capi.DMatrix(x[h:]))
    assert np.array_equal(full, np.concatenate([a, c]))
    perm = np.random.default_rng(0).permutation(x.shape[0])[:500000]
    assert np.array_equal(b.predict(capi.DMatrix(x[perm])), full[perm])


def test_replication_property_c360_size(capi, small_model_path):
    """BASELINE.json configs[2] size (C360 x 72 = 55 987 200 rows, 6 GB of features) without
    generating 6 GB on the host: the C90 matrix is uploaded 16 times into one device-resident
    DMatrix; every replica must reproduce the first one's predictions bit for bit (rows are
    independent, tiles and chunk boundaries fall differently in every replica)."""
    x = synth.quick_features(synth.raw_fields(90))
    n = x.shape[0]
    reps = 16
    b = capi.Booster(small_model_path)
    d = capi.DMatrix.device(n * reps, 27)
    for r in range(reps):
        d.upload(x, r * n)
    d.seal()
    assert d.num_row == 55987200
    out = capi.DeviceArray(n * reps)
    b.predict_device(d, out)
    capi.synchronize()
    got = out.get().reshape(reps, n)
    first = b.predict(capi.DMatrix(x))
    for r in range(reps):
        assert np.array_equal(got[r].view(np.uint32), first.view(np.uint32)), r

