"""Array-interface DMatrix constructors (XGDMatrixCreateFromDense / FromCudaArrayInterface / FromCudaColumnar) and the
columnar inplace predict (XGBoosterPredictFromCudaColumnar) without a GPU: the four symbols are exported; every refusal
of the interfaces and the config comes before any device work and names the caller (and the column); without a device
valid inputs fail with "no CPU fallback"."""
import ctypes as C
import json

import numpy as np
import pytest

ARR = {"data": [0x1000, False], "shape": [4, 27], "strides": None, "typestr": "<f4", "version": 3}
COL = {"data": [0x1000, False], "shape": [4], "strides": None, "typestr": "<f4", "version": 3}
DCFG = {"missing": -999.0, "nthread": 4}
PCFG = {"type": 0, "missing": -999.0, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}
CTORS = ["XGDMatrixCreateFromDense", "XGDMatrixCreateFromCudaArrayInterface"]
NEW = CTORS + ["XGDMatrixCreateFromCudaColumnar", "XGBoosterPredictFromCudaColumnar"]


def _create(capi, name, data, cfg=DCFG):
    h = capi.vp()
    data = data if isinstance(data, (str, bytes)) else json.dumps(data)
    data = data if isinstance(data, bytes) else data.encode()
    cfg = cfg if isinstance(cfg, str) else json.dumps(cfg)
    rc = getattr(capi.lib(), name)(data, cfg.encode(), C.byref(h))
    if rc != 0:
        raise capi.QcohError(capi.last_error())
    assert h.value
    capi.check(capi.lib().XGDMatrixFree(h))


def _predict_columns(capi, booster, cols, cfg=PCFG, m=None):
    shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
    rc = capi.lib().XGBoosterPredictFromCudaColumnar(booster.handle, json.dumps(cols).encode(), json.dumps(cfg).encode(), m,
                                                     C.byref(shp), C.byref(dim), C.byref(p))  # fmt: skip
    if rc != 0:
        raise capi.QcohError(capi.last_error())


@pytest.fixture(scope="module")
def parsed(capi, small_model_path):
    return capi.Booster(small_model_path, parse_only=True)


def test_the_four_symbols_are_declared_and_exported(capi):
    import os

    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "qcoh.h")).read()
    for name in NEW:
        assert name in capi.XGB_SYMBOLS and hasattr(capi.lib(), name)
        assert f"int {name}(" in header


@pytest.mark.parametrize("name", CTORS)
def test_array_interface_refusals_name_the_constructor(capi, name):
    cases = [
        (dict(ARR, typestr="<f8"), "typestr '<f8'"),
        (dict(ARR, typestr="<i4"), "typestr '<i4'"),
        (dict(ARR, mask=None), "'mask'"),
        (dict(ARR, shape=[108]), "2-D.*1 dimensions"),
        (dict(ARR, strides=[-108, 4]), r"strides \[-108, 4\]"),
        (dict(ARR, strides=[110, 4]), r"strides \[110, 4\]"),
        (dict(ARR, data=[0, False]), "NULL for a 4 x 27 array"),
        (dict(ARR, shape=[4, 193]), "193 columns; libqcoh's tile form holds at most 192"),
        (dict(ARR, stream=0), "stream 0"),
        ({k: v for k, v in ARR.items() if k != "typestr"}, "missing the key 'typestr'"),
    ]
    for iface, msg in cases:
        with pytest.raises(capi.QcohError, match=f"{name}: .*{msg}"):
            _create(capi, name, iface)
    with pytest.raises(capi.QcohError, match=f"{name}: .*not valid JSON"):
        _create(capi, name, "{data: 1")


@pytest.mark.parametrize("name", NEW[:3])
def test_config_refusals(capi, name):
    data = [COL] if "Columnar" in name else ARR
    with pytest.raises(capi.QcohError, match=f"{name}: config is missing the key 'missing'"):
        _create(capi, name, data, {"nthread": 1})
    with pytest.raises(capi.QcohError, match=f"{name}: config: 'missing' must be a number"):
        _create(capi, name, data, {"missing": None})
    with pytest.raises(capi.QcohError, match=f"{name}: config must be a JSON object"):
        _create(capi, name, data, "[1]")


def _columnar_cases():
    return [
        (dict(COL), "the columnar interface must be a JSON list"),
        ([], "the list of columns is empty"),
        ([COL, 3], "column 1: must be an array interface"),
        ([COL, dict(COL, shape=[2, 2])], "column 1: a column must be 1-D.*2 dimensions"),
        ([COL, COL, dict(COL, shape=[5])], "column 2: the columns differ in length: column 2 has 5 rows, column 0 has 4"),
        ([COL] * 193, "193 columns; libqcoh's tile form holds at most 192"),
        ([COL, dict(COL, data=[0, False])], "column 1: the data address is NULL for a column of 4 rows"),
        ([dict(COL, typestr="<f8")], "column 0: typestr '<f8'"),
        ([COL, dict(COL, mask=None)], "column 1: masked arrays are not supported"),
        ([COL, dict(COL, strides=[0])], r"column 1: strides \[0\]"),
        ([COL, dict(COL, strides=[6])], r"column 1: strides \[6\]"),
        ([COL, dict(COL, strides=[-4])], r"column 1: strides \[-4\]"),
        ([COL, dict(COL, strides=[4, 4])], "column 1: strides must be null or \\[bytes\\]"),
        ([COL, dict(COL, stream=0)], "column 1: stream 0"),
        ([{k: v for k, v in COL.items() if k != "data"}], "column 0: array interface is missing the key 'data'"),
    ]


def test_columnar_refusals(capi):
    name = "XGDMatrixCreateFromCudaColumnar"
    for cols, msg in _columnar_cases():
        with pytest.raises(capi.QcohError, match=f"{name}: {msg}"):
            _create(capi, name, cols)
    # a host address in a Cuda call (without a device every address is host memory)
    x = np.zeros(8, np.float32)
    host = [dict(COL, data=[x.ctypes.data, False], shape=[8])] * 2
    with pytest.raises(capi.QcohError, match=f"{name}: column 0 is in host memory"):
        _create(capi, name, host)


def test_columnar_predict_refusals(capi, parsed):
    name = "XGBoosterPredictFromCudaColumnar"
    for cols, msg in _columnar_cases():
        if "193 columns" in msg:
            continue  # more columns than the booster has features fails first (below)
        with pytest.raises(capi.QcohError, match=f"{name}: {msg}"):
            _predict_columns(capi, parsed, cols)
    with pytest.raises(capi.QcohError, match="Columns: 28 Features: 27"):
        _predict_columns(capi, parsed, [COL] * 28)
    for ty in (2, 3, 6):
        with pytest.raises(capi.QcohError, match=f"{name}: prediction type {ty} is not supported inplace"):
            _predict_columns(capi, parsed, [COL] * 27, dict(PCFG, type=ty))
    with pytest.raises(capi.QcohError, match=f"{name}: iteration_begin = 3 is not supported"):
        _predict_columns(capi, parsed, [COL] * 27, dict(PCFG, iteration_begin=3))
    with pytest.raises(capi.QcohError, match=f"{name}: the proxy DMatrix must be NULL"):
        _predict_columns(capi, parsed, [COL] * 27, m=C.c_void_p(0x1234))
    with pytest.raises(capi.QcohError, match=f"{name}: config is missing the key 'missing'"):
        _predict_columns(capi, parsed, [COL] * 27, {k: v for k, v in PCFG.items() if k != "missing"})
    x = np.zeros(8, np.float32)
    with pytest.raises(capi.QcohError, match=f"{name}: column 0 is in host memory"):
        _predict_columns(capi, parsed, [dict(COL, data=[x.ctypes.data, False], shape=[8])] * 27)


def test_host_memory_refusals(capi):
    x = np.zeros((8, 27), np.float32)
    with pytest.raises(capi.QcohError, match=r"XGDMatrixCreateFromDense: a host array must be C-contiguous.*got \[216, 8\]"):
        capi.DMatrix.from_array(np.zeros((8, 54), np.float32)[:, ::2])
    with pytest.raises(capi.QcohError, match=r"XGDMatrixCreateFromDense: a host array must be C-contiguous.*got \[4, 32\]"):
        capi.DMatrix.from_array(np.asfortranarray(x))
    with pytest.raises(capi.QcohError, match="XGDMatrixCreateFromCudaArrayInterface: the array is in host memory"):
        _create(capi, "XGDMatrixCreateFromCudaArrayInterface", dict(ARR, data=[x.ctypes.data, False], shape=[8, 27]))


def test_without_a_device_there_is_no_cpu_fallback(capi, parsed):
    if capi.device_count() > 0:
        pytest.skip("checks the behaviour without a device")
    x = np.zeros((8, 27), np.float32)
    cfg = json.dumps(dict(DCFG, extra=1)).replace("-999.0", "NaN")  # NaN `missing` and unknown keys are accepted
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _create(capi, "XGDMatrixCreateFromDense", dict(ARR, data=[x.ctypes.data, False], shape=[8, 27]), cfg)
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        capi.DMatrix.from_array(x, -999.0)
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _create(capi, "XGDMatrixCreateFromCudaArrayInterface", dict(ARR, data=[0, False], shape=[0, 27]))
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _create(capi, "XGDMatrixCreateFromCudaColumnar", [dict(COL, data=[0, False], shape=[0])] * 3)
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _predict_columns(capi, parsed, [dict(COL, data=[0, False], shape=[0])] * 27)
