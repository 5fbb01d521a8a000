"""DMatrix from device arrays without a transpose, on one GPU, at C360 x 72 (55 987 200 rows x 27 features; the rows
are C90 x 72 features of synth.quick_features repeated to the grid's size).  Times one create -> free per call:

  (a) XGDMatrixCreateFromCudaColumnar from 27 separate device fields (seal_columns)
  (b) XGDMatrixCreateFromCudaArrayInterface from a feature-major [27][N] array (seal_columns)
  (c) a caller transpose (torch .contiguous() of the [N][27] view) + XGDMatrixCreateFromMat on its device pointer
      (D2D copy + seal_tiles)

and the columnar inplace predict (XGBoosterPredictFromCudaColumnar on the 27 fields) against
XGBoosterPredictFromCudaArray on the feature-major array, both with the seeded 100 x 18 bench booster.  The matrices of
(a), (b) and (c) are compared on the device (X and key tiles), and the margins of the two predicts bit for bit.

Times are CUDA events on the caller's stream around a window of at least a second of back-to-back calls, after a
warm-up call; every library call ends in a synchronise of its stream, so the window covers it.  Every input is larger
than the 126 MB L2 (one field is 224 MB).  Achieved GB/s are over the bytes the algorithm moves: 4 B read + 4 B X +
4 B key per entry for (a) and (b); for (c) 8 B for the transpose, 8 B for the D2D copy and 8 B for the seal.  The copy
bandwidth is that of a device-to-device torch copy of the feature-major array (read + write).  Writes
profiles/array_dmatrix_c360.json (or --out) and prints it as one JSON line.

  python tools/bench_array_dmatrix.py [--out PATH] [--grid 360]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from quickchem_b200 import capi, synth  # noqa: E402

KM = 72
NF = 27


def gpu_name_and_power_limit():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()  # fmt: skip
    return [s.strip() for s in q.split(",")]


def timed(fn, min_ms=1000.0):
    """(ms per call, calls): CUDA events around back-to-back calls until the window holds at least min_ms."""
    import torch

    fn()
    torch.cuda.synchronize()
    calls, total = 0, 0.0
    while total < min_ms:
        n = max(1, calls)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        calls += n
    return total / calls, calls


class _Dev:
    """a device buffer as a torch tensor, through the CUDA Array Interface"""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": (n,), "strides": None, "typestr": typestr, "version": 2}


def dmatrix_views(d):
    """(X, key tiles) of a DMatrix as device tensors"""
    import torch

    L = capi.lib()
    x, t, nt = capi.vp(), capi.vp(), capi.u64()
    capi.check(L.qcoh_dmatrix_device_ptr(d.handle, C.byref(x)))
    capi.check(L.qcoh_dmatrix_tiles_ptr(d.handle, C.byref(t), C.byref(nt)))
    X = torch.as_tensor(_Dev(x.value, d.num_row * d.num_col, "<f4"), device="cuda").view(torch.int32)
    Xt = torch.as_tensor(_Dev(t.value, nt.value * (d.num_col + 1) * 256, "<i4"), device="cuda")
    return X, Xt


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "array_dmatrix_c360.json"))
    ap.add_argument("--grid", type=int, default=360)
    args = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("bench_array_dmatrix needs a CUDA device")
    name, limit, clock = gpu_name_and_power_limit()
    L = capi.lib()
    x90 = synth.quick_features(synth.raw_fields(90, seed=2024))
    reps = (args.grid // 90) ** 2
    n = x90.shape[0] * reps
    fm = torch.from_numpy(np.ascontiguousarray(x90.T)).cuda().repeat(1, reps)  # feature-major [27][N]
    fields = [fm[f].clone() for f in range(NF)]  # 27 separate allocations
    torch.cuda.synchronize()
    entries = n * NF
    res = {"gpu": name, "power_limit": limit, "sm_clock_max": clock, "grid": f"C{args.grid}x{KM}", "rows": n, "features": NF}

    # copy bandwidth: device-to-device copy of the feature-major array
    dst = torch.empty_like(fm)
    ms, calls = timed(lambda: dst.copy_(fm))
    res["copy_d2d"] = {"ms": round(ms, 4), "calls": calls, "GBps": round(8 * entries / ms / 1e6, 1)}
    del dst

    def create_columnar():
        capi.DMatrix.from_columns(fields, -999.0).free()

    def create_feature_major():
        capi.DMatrix.from_array(fm.T, -999.0).free()

    def transpose_then_create_from_mat():
        rm = fm.T.contiguous()
        torch.cuda.current_stream().synchronize()
        h = capi.vp()
        capi.check(L.XGDMatrixCreateFromMat(C.c_void_p(rm.data_ptr()), n, NF, -999.0, C.byref(h)))
        capi.DMatrix(handle=h).free()

    for key, fn, nbytes, family in (("a_columnar_fields", create_columnar, 12, "seal_columns"),
                                    ("b_feature_major_array", create_feature_major, 12, "seal_columns"),
                                    ("c_transpose_create_from_mat", transpose_then_create_from_mat, 24, "seal_tiles")):  # fmt: skip
        f0 = capi.kernel_launches(family)
        ms, calls = timed(fn)
        assert capi.kernel_launches(family) - f0 == calls + 1, key
        gb = nbytes * entries / 1e9
        res[key] = {"ms": round(ms, 4), "calls": calls, "family": family, "algorithmic_GB": round(gb, 2),
                    "GBps": round(gb / ms * 1e3, 1)}  # fmt: skip

    # the three matrices are the same, bit for bit
    ref = capi.DMatrix(handle=capi.vp())
    rm = fm.T.contiguous()
    torch.cuda.synchronize()
    capi.check(L.XGDMatrixCreateFromMat(C.c_void_p(rm.data_ptr()), n, NF, -999.0, C.byref(ref.handle)))
    del rm
    rX, rT = dmatrix_views(ref)
    same = {}
    for key, build in (("a", lambda: capi.DMatrix.from_columns(fields, -999.0)), ("b", lambda: capi.DMatrix.from_array(fm.T, -999.0))):
        d = build()
        X, T = dmatrix_views(d)
        same[key] = bool(torch.equal(X, rX) and torch.equal(T, rT))
        d.free()
    res["matrix_bit_equal_to_c"] = same
    ref.free()

    # columnar inplace predict against FromCudaArray on the same values (the bench booster)
    b = capi.Booster(bench.booster_path())
    cfg = json.dumps({"type": 0, "missing": -999.0, "iteration_begin": 0, "iteration_end": 0, "strict_shape": False}).encode()
    cols = capi._columns_interface(fields).encode()
    outs = {}

    def predict_columnar():
        shp, dim, p = C.POINTER(capi.u64)(), capi.u64(), capi.f32p()
        capi.check(L.XGBoosterPredictFromCudaColumnar(b.handle, cols, cfg, None, C.byref(shp), C.byref(dim), C.byref(p)))
        outs["columnar"] = p

    def predict_cuda_array():
        outs["cuda_array"] = b.inplace_predict_raw(fm.T)[1]

    bits = {}
    for key, fn in (("predict_columnar", predict_columnar), ("predict_cuda_array", predict_cuda_array)):
        ms, calls = timed(fn)
        res[key] = {"ms": round(ms, 4), "calls": calls, "family": capi.last_predict_kernel()}
        out = np.empty(n, np.float32)
        k = key.split("_", 1)[1]
        capi.check(L.qcoh_memcpy_d2h(out.ctypes.data_as(C.c_void_p), C.cast(outs[k], C.c_void_p), out.nbytes))
        bits[key] = out.view(np.uint32)
    res["predict_bit_equal"] = bool(np.array_equal(bits["predict_columnar"], bits["predict_cuda_array"]))
    b.free()
    print(json.dumps(res), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
