"""Inplace prediction on the GPU (XGBoosterPredictFromDense / XGBoosterPredictFromCudaArray, predict_dense_kernel): the
margins are bit-equal to the C oracle's and to XGDMatrixCreateFromMat + XGBoosterPredictFromDMatrix on the same array
and `missing`, for every layout of the array, both node layouts (duo_mode), forests that need several tree ranges and
the host path's chunked copy; the dense families serve, and no key tiles are sealed."""
import ctypes as C

import numpy as np
import pytest

from conftest import inject_specials
from quickchem_b200 import synth, xgbmodel

pytestmark = pytest.mark.gpu

CFG = {"type": 1, "training": False, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}


@pytest.fixture(scope="module")
def gpu(capi):
    if capi.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return capi


@pytest.fixture(scope="module")
def deep_path(tmp_path_factory):
    p = str(tmp_path_factory.mktemp("inplace") / "deep13x11.model")
    xgbmodel.write_legacy_binary(synth.random_forest_structure(13, 11, seed=6, p_leaf=0.12), p)
    return p


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _via_dmatrix(capi, b, x, missing=-999.0, iteration_end=0):
    d = capi.DMatrix(x, missing)
    out = b.predict_from_dmatrix(d, dict(CFG, iteration_end=iteration_end))
    d.free()
    return out


def _family(capi, b, duo_mode):
    try:
        b.duo_info()
        records = True
    except capi.QcohError:
        records = False
    return "dense_duo" if duo_mode and records else "dense_nodes8"


def _inplace_all(capi, b, x, missing=-999.0, **kw):
    """FromCudaArray on a row-major device copy and FromDense on the host array: both, checked equal, and the family."""
    dev = capi.DeviceArray(x)
    got = b.inplace_predict(dev, missing, shape=x.shape, **kw)
    host = b.inplace_predict(np.ascontiguousarray(x), missing, **kw)
    dev.free()
    assert np.array_equal(_u32(got), _u32(host)), kw
    return got


@pytest.mark.parametrize("which", ["small", "deep13x11", "bench"])
@pytest.mark.parametrize("specials", [False, True], ids=["clean", "specials"])
def test_bits_match_the_oracle_and_the_dmatrix_path(gpu, oracle, small_model_path, deep_path, duo_mode, which, specials):
    import bench

    rng = np.random.default_rng(3)
    if which == "bench":
        path = bench.booster_path()
        x = synth.quick_features(synth.raw_fields(90, seed=2024))
        x = x[rng.choice(x.shape[0], 30000, replace=False)]
        oracle.use_all_cores()
    else:
        path = small_model_path if which == "small" else deep_path
        x = synth.quick_features(synth.raw_fields(24, seed=7))
    b, om = gpu.Booster(path), oracle.Model(path)
    if specials:
        x = inject_specials(x, xgbmodel.read_legacy_binary(path), rng)
    fam = _family(gpu, b, duo_mode)
    for it in (0, 1, 5, 7, 11):
        ref = om.predict(x, ntree_limit=it)
        assert np.array_equal(_u32(_via_dmatrix(gpu, b, x, iteration_end=it)), _u32(ref)), it
        seals = gpu.kernel_launches("seal_tiles")
        for ty in (0, 1):
            for strict in (False, True):
                got = _inplace_all(gpu, b, x, type=ty, iteration_end=it, strict_shape=strict)
                assert got.shape == ((x.shape[0], 1) if strict else (x.shape[0],))
                assert np.array_equal(_u32(got.reshape(-1)), _u32(ref)), (it, ty, strict)
                assert gpu.last_predict_kernel() == fam
        assert gpu.kernel_launches("seal_tiles") == seals


@pytest.mark.parametrize("nrow", [0, 1, 255, 256, 257, 100_003])
def test_layouts_of_the_array_give_the_same_bits(gpu, oracle, small_model_path, small_forest, duo_mode, nrow):
    rng = np.random.default_rng(nrow)
    base = synth.quick_features(synth.raw_fields(24, seed=11))
    x = inject_specials(base[rng.choice(base.shape[0], nrow, replace=True)], small_forest, rng) if nrow else base[:0]
    b, om = gpu.Booster(small_model_path), oracle.Model(small_model_path)
    for xc in (x, np.ascontiguousarray(x[:, :19])):
        n, nc = xc.shape
        ref = _u32(om.predict(xc) if n else np.zeros(0, np.float32))
        assert np.array_equal(_u32(b.inplace_predict(xc)), ref)
        if n:
            assert gpu.last_predict_kernel() == ("dense_duo" if duo_mode else "dense_nodes8")
        layouts = {
            "row-major": (gpu.DeviceArray(xc), None, 0),
            "padded rows": (gpu.DeviceArray(np.pad(xc, ((0, 0), (0, 5)))), (4 * (nc + 5), 4), 0),
            "feature-major": (gpu.DeviceArray(np.ascontiguousarray(xc.T)), (4, 4 * n), 0),
            "offset by one float": (gpu.DeviceArray(np.concatenate([np.zeros(1, np.float32), xc.ravel()])), None, 1),
        }
        for name, (dev, strides, offset) in layouts.items():
            got = b.inplace_predict(dev, shape=(n, nc), strides=strides, offset=offset)
            assert np.array_equal(_u32(got), ref), (name, nc)
            dev.free()


def test_many_trees_in_ranges_and_the_wide_tree_booster(gpu, oracle, tmp_path, small_model_path, duo_mode):
    """The 1 100-tree forest walks ranges of 120 trees and moves the constant-table window; the small forest takes the
    table over in between.  The wide-tree booster's records carry no default bits: rows with missing entries walk
    the 8-byte nodes (MissingWalk)."""
    big = synth.random_forest_structure(1100, 7, seed=77, p_leaf=0.1)
    big_path = str(tmp_path / "many.model")
    xgbmodel.write_legacy_binary(big, big_path)
    rng = np.random.default_rng(11)
    xb = rng.normal(0, 1, (3000, 27)).astype(np.float32)
    xb[rng.random(xb.shape) < 0.01] = np.nan
    xs = synth.quick_features(synth.raw_fields(4))
    b_big, b_small = gpu.Booster(big_path), gpu.Booster(small_model_path)
    om_big, om_small = oracle.Model(big_path), oracle.Model(small_model_path)
    fam = "dense_duo" if duo_mode else "dense_nodes8"
    for it in (0, 121, 481):
        n0 = gpu.kernel_launches(fam)
        got = _inplace_all(gpu, b_big, xb, iteration_end=it)
        assert np.array_equal(_u32(got), _u32(om_big.predict(xb, ntree_limit=it))), it
        assert gpu.kernel_launches(fam) - n0 == 2 * -(-(it or 1100) // 120)  # one launch per range, two calls
        assert np.array_equal(_u32(_inplace_all(gpu, b_small, xs)), _u32(om_small.predict(xs)))
    wide = synth.random_forest_structure(2, 17, seed=5, p_leaf=0.0)
    p = str(tmp_path / "wide.model")
    xgbmodel.write_legacy_binary(wide, p)
    b, om = gpu.Booster(p), oracle.Model(p)
    assert b.duo_info() == (15, False)
    x = rng.normal(0, 1, (20000, 27)).astype(np.float32)
    x[rng.random(x.shape) < 0.02] = -999.0
    got = _inplace_all(gpu, b, x)
    assert np.array_equal(_u32(got), _u32(om.predict(x)))
    assert gpu.last_predict_kernel() == fam


@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_host_path_in_chunks(gpu, oracle, small_model_path, small_forest, pinned):
    rng = np.random.default_rng(5)
    base = synth.quick_features(synth.raw_fields(24, seed=5))
    x = inject_specials(base[:5000], small_forest, rng)
    b = gpu.Booster(small_model_path)
    dev = gpu.DeviceArray(x)
    want = _u32(b.inplace_predict(dev, shape=x.shape))
    dev.free()
    src = x
    if pinned:
        src = gpu.pinned_empty(x.shape)
        src[:] = x
    gpu.set_param("chunk_rows", 512)  # 10 chunks, the last one 392 rows
    try:
        for it in (0, 5):
            got = b.inplace_predict(src, iteration_end=it)
            assert np.array_equal(_u32(got), _u32(oracle.Model(small_model_path).predict(x, ntree_limit=it)))
        assert np.array_equal(_u32(b.inplace_predict(src)), want)
    finally:
        gpu.set_param("chunk_rows", 0)


def test_contract(gpu, small_model_path, tmp_path):
    import torch

    b = gpu.Booster(small_model_path)
    rng = np.random.default_rng(9)
    x = synth.quick_features(synth.raw_fields(8, seed=9))[:3000].copy()
    ref = _u32(_via_dmatrix(gpu, b, x))
    # +-inf with a finite missing fails like XGDMatrixCreateFromMat; with missing = inf it is a missing entry
    xi = x.copy()
    xi[17, 3] = np.inf
    dev = gpu.DeviceArray(xi)
    for call in (lambda: b.inplace_predict(xi), lambda: b.inplace_predict(dev, shape=xi.shape)):
        with pytest.raises(gpu.QcohError, match="Input data contains `inf` or `nan`"):
            call()
    want = _u32(_via_dmatrix(gpu, b, xi, missing=np.inf))
    assert np.array_equal(_u32(b.inplace_predict(xi, missing=np.inf)), want)
    assert np.array_equal(_u32(b.inplace_predict(dev, missing=np.inf, shape=xi.shape)), want)
    # NaN as `missing`
    assert np.array_equal(_u32(b.inplace_predict(x, missing=np.nan)), _u32(_via_dmatrix(gpu, b, x, missing=np.nan)))
    dev.free()
    # "stream": 1 (legacy default) and 2 (per-thread default) are waited for; 0 is invalid
    dev = gpu.DeviceArray(x)
    for s in (1, 2):
        shape_, p, on_device = b.inplace_predict_raw(dev, shape=x.shape, stream=s)
        assert on_device
        out = np.empty(x.shape[0], np.float32)
        gpu.check(gpu.lib().qcoh_memcpy_d2h(out.ctypes.data_as(C.c_void_p), C.cast(p, C.c_void_p), out.nbytes))
        assert np.array_equal(_u32(out), ref)
    with pytest.raises(gpu.QcohError, match="stream 0"):
        b.inplace_predict_raw(dev, shape=x.shape, stream=0)
    # the device result stays valid until the next predict on that booster: a predict on another booster leaves it
    _, p, _ = b.inplace_predict_raw(dev, shape=x.shape)
    other = gpu.Booster(small_model_path)
    other.inplace_predict(gpu.DeviceArray(x[::-1].copy()), shape=x.shape)
    out = np.empty(x.shape[0], np.float32)
    gpu.check(gpu.lib().qcoh_memcpy_d2h(out.ctypes.data_as(C.c_void_p), C.cast(p, C.c_void_p), out.nbytes))
    assert np.array_equal(_u32(out), ref)
    dev.free()
    # a torch CUDA tensor through __cuda_array_interface__, contiguous and as a transposed view of a feature-major copy
    t = torch.from_numpy(x).cuda()
    tf = torch.from_numpy(np.ascontiguousarray(x.T)).cuda().T
    torch.cuda.synchronize()
    assert not tf.is_contiguous()
    for tt in (t, tf):
        assert np.array_equal(_u32(b.inplace_predict(tt)), ref)
