"""Array-interface DMatrix constructors and the columnar inplace predict on the GPU.  Whatever the layout of the source
(device row-major, padded rows, feature-major, every other column of a wider array, a torch transposed view, separate
columns, views into one feature-major tensor, a strided column, pinned and pageable host memory), the DMatrix is the one
XGDMatrixCreateFromMat makes from np.ascontiguousarray of the same values: the same key tiles, the same X (SaveBinary
files byte-equal), NumRow / NumCol and missing flags; predictions equal the oracle's bit for bit, and contributions and
interaction values equal those on the CreateFromMat DMatrix bit for bit.  The columnar inplace predict equals
XGBoosterPredictFromCudaArray on the stacked array and the oracle, on both node layouts and over several tree ranges."""
import ctypes as C

import numpy as np
import pytest

from conftest import inject_specials
from quickchem_b200 import synth, xgbmodel

pytestmark = pytest.mark.gpu

NROWS = [0, 1, 255, 256, 257, 3 * 256 + 17, 48600]  # 48 600 = one C90 level slab
NCOLS = [27, 19, 1]


@pytest.fixture(scope="module")
def gpu(capi):
    if capi.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return capi


def _u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _values(nrow, ncol, forest, seed):
    rng = np.random.default_rng(seed)
    base = synth.quick_features(synth.raw_fields(24, seed=11))
    x = inject_specials(base[rng.choice(base.shape[0], max(nrow, 1), replace=True)], forest, rng)[:nrow]
    x[rng.random(x.shape) < 0.01] = np.float32(-0.0)
    return np.ascontiguousarray(x[:, :ncol])


def _tiles(gpu, d):
    p, nt = gpu.vp(), gpu.u64()
    gpu.check(gpu.lib().qcoh_dmatrix_tiles_ptr(d.handle, C.byref(p), C.byref(nt)))
    out = np.empty(nt.value * (d.num_col + 1) * 256, np.uint32)
    if out.size:
        gpu.check(gpu.lib().qcoh_memcpy_d2h(out.ctypes.data_as(C.c_void_p), p, out.nbytes))
    return out


def _saved(d, path):
    d.save_binary(path)
    with open(path, "rb") as f:
        return f.read()


def _family_of(gpu, build):
    s0, c0 = gpu.kernel_launches("seal_tiles"), gpu.kernel_launches("seal_columns")
    d = build()
    return d, {"seal_tiles": gpu.kernel_launches("seal_tiles") - s0, "seal_columns": gpu.kernel_launches("seal_columns") - c0}


def _transposed_view(x):
    """a torch transposed view of a feature-major device copy of x"""
    import torch

    return torch.from_numpy(np.ascontiguousarray(x.T)).cuda().T


def _layouts(gpu, x):
    """name -> (build(missing) of the DMatrix, family that seals it, keep-alive)"""
    import torch

    n, nc = x.shape
    D = gpu.DMatrix
    t = torch.from_numpy(x).cuda()
    fm = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    padded = gpu.DeviceArray(np.pad(x, ((0, 0), (0, 5))))
    feature_major = gpu.DeviceArray(np.ascontiguousarray(x.T))
    wide = np.zeros((n, 2 * nc), np.float32)
    wide[:, ::2] = x
    every_other = gpu.DeviceArray(wide)
    separate = [torch.from_numpy(x[:, c].copy()).cuda() for c in range(nc)]
    strided = [t[:, 0]] + [fm[c] for c in range(1, nc)]
    pinned = gpu.pinned_empty(x.shape)
    pinned[:] = x
    torch.cuda.synchronize()

    def seal(strides):  # a C-contiguous array is copied and sealed by seal_tiles, any other layout by seal_columns
        return "seal_tiles" if strides is None or tuple(strides) == (4 * nc, 4) else "seal_columns"

    tv = fm.T
    tv_strides = tv.__cuda_array_interface__["strides"]
    out = {
        "device row-major": (lambda m: D.from_array(t, m), "seal_tiles"),
        "padded rows": (lambda m: D.from_array(padded, m, shape=(n, nc), strides=(4 * (nc + 5), 4)), "seal_columns"),
        "feature-major": (lambda m: D.from_array(feature_major, m, shape=(n, nc), strides=(4, 4 * n)), seal((4, 4 * n))),
        "every other column": (lambda m: D.from_array(every_other, m, shape=(n, nc), strides=(8 * nc, 8)), "seal_columns"),
        "torch transposed view": (lambda m: D.from_array(tv, m), seal(tv_strides)),
        "columns: separate": (lambda m: D.from_columns(separate, m), "seal_columns"),
        "columns: views of [ncol][nrow]": (lambda m: D.from_columns([fm[c] for c in range(nc)], m), "seal_columns"),
        "columns: one strided": (lambda m: D.from_columns(strided, m), "seal_columns"),
        "host pinned": (lambda m: D.from_array(pinned, m), "seal_tiles"),
        "host pageable": (lambda m: D.from_array(x, m), "seal_tiles"),
    }
    keep = [t, fm, padded, feature_major, every_other, separate, strided, pinned]
    return out, keep


@pytest.mark.parametrize("ncol", NCOLS)
@pytest.mark.parametrize("nrow", NROWS)
def test_every_layout_gives_the_create_from_mat_dmatrix(gpu, oracle, small_model_path, small_forest, tmp_path, nrow, ncol):
    x = _values(nrow, ncol, small_forest, seed=nrow * 31 + ncol)
    b, om = gpu.Booster(small_model_path), oracle.Model(small_model_path)
    ref = gpu.DMatrix(np.ascontiguousarray(x), -999.0)
    ref_tiles, ref_bin = _tiles(gpu, ref), _saved(ref, str(tmp_path / "ref.bin"))
    want = {}
    if nrow:
        for mask in (0, 1, 2):
            want[mask] = _u32(om.predict(x, option_mask=mask))
            assert np.array_equal(_u32(b.predict(ref, option_mask=mask)), want[mask])
        b.predict(ref)
        ref_kernel = gpu.last_predict_kernel()
        ref_contribs = {a: _u32(b.predict_contribs(ref, approximate=a)) for a in (False, True)}
        few = min(nrow, 40)
        ref_inter = {a: _u32(b.predict_interactions(gpu.DMatrix(x[:few], -999.0), approximate=a)) for a in (False, True)}
    layouts, keep = _layouts(gpu, x)
    for name, (build, family) in layouts.items():
        d, fams = _family_of(gpu, lambda: build(-999.0))
        assert (d.num_row, d.num_col) == (nrow, ncol), name
        assert np.array_equal(_tiles(gpu, d), ref_tiles), name
        assert _saved(d, str(tmp_path / "got.bin")) == ref_bin, name
        if nrow:
            assert fams[family] == 1 and sum(fams.values()) == 1, (name, fams)
            for mask in (0, 1, 2):
                assert np.array_equal(_u32(b.predict(d, option_mask=mask)), want[mask]), (name, mask)
            b.predict(d)
            assert gpu.last_predict_kernel() == ref_kernel, name  # the same missing flags
            for a in (False, True):
                assert np.array_equal(_u32(b.predict_contribs(d, approximate=a)), ref_contribs[a]), (name, a)
            if name in ("feature-major", "columns: separate"):
                few_d = gpu.DMatrix.from_array(_transposed_view(x[:few]), -999.0)
                for a in (False, True):
                    assert np.array_equal(_u32(b.predict_interactions(few_d, approximate=a)), ref_inter[a]), (name, a)
                few_d.free()
        d.free()
    del keep
    ref.free()


def test_inf_raises_and_creates_nothing_and_nan_missing(gpu, small_forest, tmp_path):
    import torch

    x = _values(3000, 27, small_forest, seed=4)
    xi = x.copy()
    xi[1234, 5] = np.inf
    ti = torch.from_numpy(np.ascontiguousarray(xi.T)).cuda()
    builds = [lambda: gpu.DMatrix.from_array(ti.T, -999.0), lambda: gpu.DMatrix.from_columns([ti[c] for c in range(27)], -999.0),
              lambda: gpu.DMatrix.from_array(xi, -999.0), lambda: gpu.DMatrix.from_array(torch.from_numpy(xi).cuda(), -999.0)]
    for build in builds:
        with pytest.raises(gpu.QcohError, match="Input data contains `inf` or `nan`"):
            build()
    # with missing = inf it is a missing entry; the pooled buffers serve the next create
    ref = gpu.DMatrix(xi, np.inf)
    for build_inf in (lambda: gpu.DMatrix.from_array(ti.T, np.inf), lambda: gpu.DMatrix.from_columns([ti[c] for c in range(27)], np.inf)):
        d = build_inf()
        assert np.array_equal(_tiles(gpu, d), _tiles(gpu, ref))
        assert _saved(d, str(tmp_path / "a.bin")) == _saved(ref, str(tmp_path / "b.bin"))
        d.free()
    # NaN as `missing` (the default of from_array / from_columns)
    t = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    ref = gpu.DMatrix(x, np.nan)
    d = gpu.DMatrix.from_columns([t[c] for c in range(27)])
    assert np.array_equal(_tiles(gpu, d), _tiles(gpu, ref))
    assert _saved(d, str(tmp_path / "a.bin")) == _saved(ref, str(tmp_path / "b.bin"))


def test_streams_and_determinism(gpu, small_forest):
    """Columns written on a torch side stream behind queued work: the interface's stream is waited for, and the
    DMatrix holds the written values.  Building the same DMatrix twice gives identical tiles."""
    import torch

    x = _values(48600, 27, small_forest, seed=8)
    ref = _tiles(gpu, gpu.DMatrix(x, -999.0))
    src = torch.from_numpy(np.ascontiguousarray(x.T)).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for kind in ("columns", "array"):
        dst = torch.zeros_like(src)
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(200_000_000)  # queued work ahead of the writes
            dst.copy_(src)
        if kind == "columns":
            d = gpu.DMatrix.from_columns([dst[c] for c in range(27)], -999.0, stream=side.cuda_stream)
        else:
            d = gpu.DMatrix.from_array(dst.T, -999.0, stream=side.cuda_stream)
        assert np.array_equal(_tiles(gpu, d), ref), kind
        d.free()
        torch.cuda.synchronize()
    a = gpu.DMatrix.from_columns([src[c] for c in range(27)], -999.0)
    b = gpu.DMatrix.from_columns([src[c] for c in range(27)], -999.0)
    assert np.array_equal(_tiles(gpu, a), _tiles(gpu, b))


@pytest.mark.parametrize("which", ["small", "many"])
def test_columnar_inplace_predict(gpu, oracle, small_model_path, tmp_path, duo_mode, which):
    import torch

    rng = np.random.default_rng(12)
    if which == "many":  # 1 100 trees: ten ranges of 120 trees
        path = str(tmp_path / "many.model")
        xgbmodel.write_legacy_binary(synth.random_forest_structure(1100, 7, seed=77, p_leaf=0.1), path)
        x = rng.normal(0, 1, (3000, 27)).astype(np.float32)
        x[rng.random(x.shape) < 0.01] = np.nan
        x[rng.random(x.shape) < 0.01] = -999.0
    else:
        path = small_model_path
        x = synth.quick_features(synth.raw_fields(24, seed=3))[:48600].copy()
        x[rng.random(x.shape) < 0.01] = -999.0
    b, om = gpu.Booster(path), oracle.Model(path)
    try:
        b.duo_info()
        records = True
    except gpu.QcohError:
        records = False
    fam = "columns_duo" if duo_mode and records else "columns_nodes8"
    for nc in (27, 19, 1):
        xc = np.ascontiguousarray(x[:, :nc])
        fm = torch.from_numpy(np.ascontiguousarray(xc.T)).cuda()
        rm = torch.from_numpy(xc).cuda()
        torch.cuda.synchronize()
        column_sets = {"views": [fm[c] for c in range(nc)], "strided": [rm[:, c] for c in range(nc)]}
        for it in (0, 121) if which == "many" else (0, 5):
            ref = _u32(om.predict(xc, ntree_limit=it, option_mask=1))
            stacked = _u32(b.inplace_predict(rm, type=1, iteration_end=it))
            assert np.array_equal(stacked, ref), (nc, it)
            for name, cols in column_sets.items():
                n0 = gpu.kernel_launches(fam)
                got = b.inplace_predict_columns(cols, type=1, iteration_end=it)
                assert got.shape == (xc.shape[0],)
                assert np.array_equal(_u32(got), ref), (name, nc, it)
                assert gpu.last_predict_kernel() == fam
                assert gpu.kernel_launches(fam) - n0 == -(-(it or b.info().num_trees) // 120)
        strict = b.inplace_predict_columns(column_sets["views"], type=0, strict_shape=True)
        assert strict.shape == (xc.shape[0], 1)
        assert np.array_equal(_u32(strict.reshape(-1)), _u32(om.predict(xc)))
