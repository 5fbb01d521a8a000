"""Per-feature contribution rates on one GPU: exact (TreeSHAP) and approximate (Saabas) contributions of the seeded
100 x 18 bench booster on a fixed, seeded sample of C90 x 72 rows, plain prediction of the same rows for scale, and
the CPU oracle's contribution rate on a subsample.  Device times are CUDA events on the library stream around
qcoh_booster_predict_contribs_device / qcoh_booster_predict_device after a warm-up call of the same shape; each
timed window is at least a second.  Prints one JSON line (and writes it to --out when given).

  python tools/bench_contribs.py [--rows 32768] [--oracle-rows 64] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # the contributions oracle is test infrastructure

import bench  # noqa: E402
import oracle_contribs  # noqa: E402
from oracle import cpu as oracle  # noqa: E402
from quickchem_b200 import capi, synth  # noqa: E402


def gpu_name_and_power_limit():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()  # fmt: skip
    name, limit = (s.strip() for s in q.split(",", 1))
    return name, limit


def timed(fn, min_seconds=1.0):
    """(seconds per call, calls) over a window of at least `min_seconds` of device time, after one warm-up call."""
    fn()
    capi.synchronize()
    calls, total = 0, 0.0
    while total < min_seconds * 1e3:
        capi.timer_start()
        fn()
        total += capi.timer_stop()
        calls += 1
    return total / 1e3 / calls, calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=32768)
    ap.add_argument("--oracle-rows", type=int, default=64)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("bench_contribs needs a CUDA device")
    gpu, power_limit = gpu_name_and_power_limit()
    path = bench.booster_path()
    x = synth.quick_features(synth.raw_fields(90, seed=2024))  # C90 x 72
    x = np.ascontiguousarray(x[np.random.default_rng(90).choice(x.shape[0], args.rows, replace=False)])
    b = capi.Booster(path)
    info = b.info()
    nf = info.num_feature
    bins, tree_bin, _ = b.shap_paths()
    # a path's length = its elements, the bias element included; the bias lane of each path carries it
    lens = (bins[:, :, 2] >> 24).astype(np.int64)
    bias_lane = (lens > 0) & ((bins[:, :, 2] & 0xFF) == 0xFF)
    n_paths, path_elements = int(bias_lane.sum()), int(lens[bias_lane].sum())
    dm = capi.DMatrix(x)
    out = capi.DeviceArray(args.rows * (nf + 1))
    t_exact, n_exact = timed(lambda: b.predict_contribs_device(dm, out, approximate=False))
    assert capi.last_predict_kernel() == "shap"
    exact = out.get().reshape(args.rows, nf + 1)
    t_approx, n_approx = timed(lambda: b.predict_contribs_device(dm, out, approximate=True))
    assert capi.last_predict_kernel() == "shap_approx"
    approx = out.get().reshape(args.rows, nf + 1)
    pred = capi.DeviceArray(args.rows)
    t_pred, n_pred = timed(lambda: b.predict_device(dm, pred))
    # the CPU oracle on a subsample (all cores), and the agreement there
    cores = oracle.use_all_cores()
    m = oracle.Model(path)
    oracle_contribs.build()  # compiled before the timed calls
    xs = x[: args.oracle_rows]
    t0 = time.perf_counter()
    ref = oracle_contribs.predict_contribs(m, xs)
    t_orc = time.perf_counter() - t0
    t0 = time.perf_counter()
    ref_a = oracle_contribs.predict_contribs(m, xs, approximate=True)
    t_orc_a = time.perf_counter() - t0
    scale = np.abs(ref.astype(np.float64)).sum(axis=1)
    ratio = float((np.abs(exact[: len(xs)].astype(np.float64) - ref).max(axis=1) / scale).max())
    res = {
        "gpu": gpu, "power_limit": power_limit,
        "booster": f"{info.num_trees} trees, max depth {info.max_depth}, {info.num_nodes} nodes (bench.py seeded booster)",
        "rows": args.rows, "sample": "C90 x 72 rows, seeded (synth.raw_fields(90, seed=2024), rng 90)",
        "paths": n_paths, "path_elements": path_elements, "bins": int(len(bins)),
        "exact_rows_per_s": args.rows / t_exact, "exact_s_per_call": t_exact, "exact_calls": n_exact,
        "exact_path_elements_per_s": path_elements * args.rows / t_exact,
        "approx_rows_per_s": args.rows / t_approx, "approx_s_per_call": t_approx, "approx_calls": n_approx,
        "predict_rows_per_s": args.rows / t_pred, "predict_s_per_call": t_pred, "predict_calls": n_pred,
        "oracle_cores": cores, "oracle_rows": len(xs),
        "oracle_exact_rows_per_s": len(xs) / t_orc, "oracle_approx_rows_per_s": len(xs) / t_orc_a,
        "exact_vs_oracle_max_ratio": ratio,
        "approx_bit_equal_to_oracle": bool(np.array_equal(approx[: len(xs)], ref_a)),
    }  # fmt: skip
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
