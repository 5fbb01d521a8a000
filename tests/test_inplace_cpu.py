"""Inplace prediction (XGBoosterPredictFromDense / XGBoosterPredictFromCudaArray) without a GPU: every refusal of the
array interface, the config and the memory kinds comes before any device work and names what it got; both symbols are
exported; without a device both calls fail with "no CPU fallback"."""
import ctypes as C
import json

import numpy as np
import pytest

ARR = {"data": [0x1000, False], "shape": [4, 27], "strides": None, "typestr": "<f4", "version": 3}
CFG = {"type": 0, "missing": -999.0, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}


def _call(capi, booster, name, iface, cfg=CFG, m=None):
    shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
    cfg = cfg if isinstance(cfg, str) else json.dumps(cfg)
    rc = getattr(capi.lib(), name)(booster.handle, json.dumps(iface).encode(), cfg.encode(), m, C.byref(shp), C.byref(dim), C.byref(p))
    if rc != 0:
        raise capi.QcohError(capi.last_error())
    return rc


@pytest.fixture(scope="module")
def parsed(capi, small_model_path):
    return capi.Booster(small_model_path, parse_only=True)


def test_both_symbols_are_exported(capi):
    for name in ("XGBoosterPredictFromDense", "XGBoosterPredictFromCudaArray"):
        assert name in capi.XGB_SYMBOLS and hasattr(capi.lib(), name)


@pytest.mark.parametrize("name", ["XGBoosterPredictFromDense", "XGBoosterPredictFromCudaArray"])
def test_array_interface_refusals(capi, parsed, name):
    cases = [
        (dict(ARR, typestr="<f8"), "typestr '<f8'"),
        (dict(ARR, typestr="<i4"), "typestr '<i4'"),
        (dict(ARR, mask=None), "'mask'"),
        (dict(ARR, shape=[108]), "2-D.*1 dimensions"),
        (dict(ARR, shape=[2, 2, 27]), "2-D.*3 dimensions"),
        (dict(ARR, strides=[-108, 4]), r"strides \[-108, 4\]"),
        (dict(ARR, strides=[108, 2]), r"strides \[108, 2\]"),
        (dict(ARR, strides=[110, 4]), r"strides \[110, 4\]"),
        (dict(ARR, data=[0, False]), "NULL for a 4 x 27 array"),
        (dict(ARR, shape=[4, 28]), "Columns: 28 Features: 27"),
        (dict(ARR, stream=0), "stream 0"),
        ({k: v for k, v in ARR.items() if k != "typestr"}, "missing the key 'typestr'"),
    ]
    for iface, msg in cases:
        with pytest.raises(capi.QcohError, match=f"{name}: .*{msg}" if "Columns" not in msg else msg):
            _call(capi, parsed, name, iface)
    with pytest.raises(capi.QcohError, match="not valid JSON"):
        shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
        capi.check(getattr(capi.lib(), name)(parsed.handle, b"{data: 1", json.dumps(CFG).encode(), None, C.byref(shp), C.byref(dim), C.byref(p)))


@pytest.mark.parametrize("name", ["XGBoosterPredictFromDense", "XGBoosterPredictFromCudaArray"])
def test_config_and_proxy_refusals(capi, parsed, name):
    for k in CFG:
        with pytest.raises(capi.QcohError, match=f"{name}: config is missing the key '{k}'"):
            _call(capi, parsed, name, ARR, {kk: v for kk, v in CFG.items() if kk != k})
    for ty in (2, 3, 4, 5, 6):
        with pytest.raises(capi.QcohError, match=f"prediction type {ty} is not supported inplace"):
            _call(capi, parsed, name, ARR, dict(CFG, type=ty))
    with pytest.raises(capi.QcohError, match="iteration_begin = 2 is not supported"):
        _call(capi, parsed, name, ARR, dict(CFG, iteration_begin=2))
    with pytest.raises(capi.QcohError, match="'missing' must be a number"):
        _call(capi, parsed, name, ARR, dict(CFG, missing=None))
    with pytest.raises(capi.QcohError, match="proxy DMatrix must be NULL"):
        _call(capi, parsed, name, ARR, m=C.c_void_p(0x1234))


def test_memory_kind_refusals(capi, parsed):
    x = np.zeros((8, 27), np.float32)
    with pytest.raises(capi.QcohError, match="XGBoosterPredictFromDense: a host array must be C-contiguous.*got \\[216, 8\\]"):
        parsed.inplace_predict(np.zeros((8, 54), np.float32)[:, ::2])
    with pytest.raises(capi.QcohError, match="XGBoosterPredictFromDense: a host array must be C-contiguous.*got \\[4, 32\\]"):
        parsed.inplace_predict(np.asfortranarray(x))
    with pytest.raises(capi.QcohError, match="XGBoosterPredictFromCudaArray: the array is in host memory"):
        _call(capi, parsed, "XGBoosterPredictFromCudaArray", dict(ARR, data=[x.ctypes.data, False]))


def test_the_config_accepts_nan_and_ignores_other_keys(capi, parsed):
    """NaN as `missing`, and xgboost's own keys (training, cache_id) are accepted: the call reaches the device."""
    if capi.device_count() > 0:
        pytest.skip("checks how far a call gets without a device")
    x = np.zeros((8, 27), np.float32)
    cfg = json.dumps(dict(CFG, training=False, cache_id=0)).replace("-999.0", "NaN")
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _call(capi, parsed, "XGBoosterPredictFromDense", dict(ARR, data=[x.ctypes.data, False], shape=[8, 27]), cfg)


def test_without_a_device_there_is_no_cpu_fallback(capi, parsed):
    if capi.device_count() > 0:
        pytest.skip("checks the behaviour without a device")
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        parsed.inplace_predict(np.zeros((8, 27), np.float32))
    with pytest.raises(capi.QcohError, match="no CPU fallback"):
        _call(capi, parsed, "XGBoosterPredictFromCudaArray", dict(ARR, data=[0, False], shape=[0, 27]))
