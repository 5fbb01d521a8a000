"""Inplace prediction against create -> predict -> free, on one GPU.  Two workloads: C360 x 72 rows with the seeded
100 x 18 bench booster, and C180 x 72 rows with a seeded 10 x 6 booster (the HBM-bound end, where the seal and the
copy weigh most).  The rows are C90 x 72 features (synth.quick_features) repeated to the grid's size.  Per workload:

  (a)  XGDMatrixCreateFromMat from a device pointer -> XGBoosterPredict -> XGDMatrixFree (result to pinned host)
  (a2) the same with XGBoosterPredictFromDMatrix
  (b)  XGBoosterPredictFromCudaArray on the same row-major device buffer (result stays on the device)
  (b2) XGBoosterPredictFromDense on that device address (the same kernels, plus the D2H of the result)
  (c)  XGBoosterPredictFromCudaArray on a feature-major [27][N] copy
  (d)  XGBoosterPredictFromDense from pinned and from pageable host memory (whole call, host to host)

Times are CUDA events on the library stream (qcoh_timer_start / stop) around a window of at least a second of
back-to-back calls, after a warm-up call; every call ends in a stream synchronise.  The margins of all calls are
compared bit for bit.  Writes profiles/inplace_<grid>_<booster>.json (or --out-dir) and prints one JSON line each.

  python tools/bench_inplace.py [--out-dir DIR] [--only c360|c180]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from quickchem_b200 import capi, synth, xgbmodel  # noqa: E402

KM = 72


def gpu_name_and_power_limit():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()  # fmt: skip
    return [s.strip() for s in q.split(",")]


def timed(fn, min_ms=1000.0):
    """(ms per call, calls): CUDA events around back-to-back calls until the window holds at least min_ms."""
    fn()
    capi.synchronize()
    calls, total = 0, 0.0
    while total < min_ms:
        n = max(1, calls)
        capi.timer_start()
        for _ in range(n):
            fn()
        total += capi.timer_stop()
        calls += n
    return total / calls, calls


def d2h(p, n, on_device):
    out = np.empty(n, np.float32)
    if on_device:
        capi.check(capi.lib().qcoh_memcpy_d2h(out.ctypes.data_as(C.c_void_p), C.cast(p, C.c_void_p), out.nbytes))
    else:
        out[:] = np.ctypeslib.as_array(p, (n,))
    return out


def workload(grid, booster_path, x90):
    reps = (grid // 90) ** 2
    n = x90.shape[0] * reps
    L = capi.lib()
    b = capi.Booster(booster_path)
    X = capi.DeviceArray(n * 27)
    Xf = capi.DeviceArray(n * 27)
    xt = np.ascontiguousarray(x90.T)
    for r in range(reps):  # row-major and feature-major device copies of the repeated rows
        capi.check(L.qcoh_memcpy_h2d(C.c_void_p(X.ptr.value + r * x90.nbytes), x90.ctypes.data_as(C.c_void_p), x90.nbytes))
        for f in range(27):
            dst = Xf.ptr.value + (f * n + r * x90.shape[0]) * 4
            capi.check(L.qcoh_memcpy_h2d(C.c_void_p(dst), xt[f].ctypes.data_as(C.c_void_p), xt.shape[1] * 4))
    outs, res = {}, {}

    def create_predict_free(api):
        def run():
            h = C.c_void_p()
            capi.check(L.XGDMatrixCreateFromMat(X.ptr, n, 27, -999.0, C.byref(h)))
            d = capi.DMatrix(handle=h)
            if api == "predict":
                ln, p = b.predict_raw(d)
                outs["a"] = (p, ln, False)
            else:
                cfg = json.dumps({"type": 0, "training": False, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False})
                shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
                capi.check(L.XGBoosterPredictFromDMatrix(b.handle, d.handle, cfg.encode(), C.byref(shp), C.byref(dim), C.byref(p)))
                outs["a2"] = (p, n, False)
            d.free()

        return run

    def inplace(key, data, **kw):
        def run():
            shape_, p, on_device = b.inplace_predict_raw(data, **kw)
            outs[key] = (p, n, on_device)

        return run

    def from_dense_device():
        iface = {"data": [X.ptr.value, False], "shape": [n, 27], "strides": None, "typestr": "<f4", "version": 3}
        cfg = {"type": 0, "missing": -999.0, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}
        shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
        capi.check(L.XGBoosterPredictFromDense(b.handle, json.dumps(iface).encode(), json.dumps(cfg).encode(), None, C.byref(shp), C.byref(dim), C.byref(p)))
        outs["b2"] = (p, n, False)

    cases = [("a", create_predict_free("predict")), ("a2", create_predict_free("from_dmatrix")),
             ("b", inplace("b", X, shape=(n, 27))), ("b2", from_dense_device),
             ("c", inplace("c", Xf, shape=(n, 27), strides=(4, 4 * n)))]  # fmt: skip
    bits = {}
    for key, fn in cases:
        ms, calls = timed(fn)
        res[key] = {"ms": round(ms, 4), "calls": calls, "family": capi.last_predict_kernel()}
        p, ln, dev = outs[key]
        bits[key] = d2h(p, ln, dev).view(np.uint32)
    Xf.free()
    host = np.empty((n, 27), np.float32)
    capi.check(L.qcoh_memcpy_d2h(host.ctypes.data_as(C.c_void_p), X.ptr, host.nbytes))
    X.free()
    pinned = capi.pinned_empty((n, 27))
    pinned[:] = host
    for key, src in (("d_pinned", pinned), ("d_pageable", host)):
        ms, calls = timed(inplace(key, src))
        res[key] = {"ms": round(ms, 4), "calls": calls, "family": capi.last_predict_kernel()}
        p, ln, dev = outs[key]
        bits[key] = d2h(p, ln, dev).view(np.uint32)
    ref = bits["a"]
    res["bit_equal_to_a"] = {k: bool(np.array_equal(v, ref)) for k, v in bits.items()}
    res["rows"] = n
    b.free()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--only", choices=["c360", "c180"])
    args = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("bench_inplace needs a CUDA device")
    name, limit, clock = gpu_name_and_power_limit()
    x90 = synth.quick_features(synth.raw_fields(90, seed=2024))
    with tempfile.TemporaryDirectory() as d:
        p10 = os.path.join(d, "b10x6.model")
        xgbmodel.write_legacy_binary(synth.prod_like_booster(n_trees=10, max_depth=6, seed=18), p10)
        runs = [("c360", 360, "100x18", bench.booster_path()), ("c180", 180, "10x6", p10)]
        for tag, grid, bname, path in runs:
            if args.only and args.only != tag:
                continue
            r = workload(grid, path, x90)
            out = {"gpu": name, "power_limit": limit, "sm_clock_max": clock, "grid": f"C{grid}x{KM}", "booster": bname, **r}
            print(json.dumps(out), flush=True)
            os.makedirs(args.out_dir, exist_ok=True)
            with open(os.path.join(args.out_dir, f"inplace_{tag}_{bname}.json"), "w") as f:
                json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
