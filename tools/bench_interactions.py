"""SHAP interaction value rates on one GPU: exact and approximate interaction values of the seeded 100 x 18 bench
booster on a fixed, seeded sample of C90 x 72 rows, and exact contributions of the same rows in the same run for
scale, with the CPU oracle's interaction rate and agreement on a subsample.  Device times are CUDA events on the
library stream around qcoh_booster_predict_interactions_device / qcoh_booster_predict_contribs_device after a warm-up
call of the same shape (tools/bench_contribs.py timed).  Prints one JSON line (and writes it to --out when given).

  python tools/bench_interactions.py [--rows 2048] [--oracle-rows 8] [--out FILE]
"""
import argparse
import json
import os
import time

import numpy as np

from bench_contribs import bench, gpu_name_and_power_limit, oracle, timed  # also puts tests/ on the path
import oracle_interactions  # noqa: E402
from quickchem_b200 import capi, synth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=2048)
    ap.add_argument("--oracle-rows", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("bench_interactions needs a CUDA device")
    gpu, power_limit = gpu_name_and_power_limit()
    path = bench.booster_path()
    x = synth.quick_features(synth.raw_fields(90, seed=2024))  # C90 x 72
    x = np.ascontiguousarray(x[np.random.default_rng(90).choice(x.shape[0], args.rows, replace=False)])
    b = capi.Booster(path)
    info = b.info()
    nc = info.num_feature + 1
    bins, _, _ = b.shap_paths()
    # (path, condition) pairs: every feature element of every path conditions the path once
    lens = (bins[:, :, 2] >> 24).astype(np.int64)
    bias_lane = (lens > 0) & ((bins[:, :, 2] & 0xFF) == 0xFF)
    n_paths = int(bias_lane.sum())
    pairs = int(lens[bias_lane].sum()) - n_paths
    dm = capi.DMatrix(x)
    out = capi.DeviceArray(args.rows * nc * nc)
    t_exact, n_exact = timed(lambda: b.predict_interactions_device(dm, out, approximate=False))
    assert capi.last_predict_kernel() == "shap_inter"
    exact = out.get().reshape(args.rows, nc, nc)
    t_approx, n_approx = timed(lambda: b.predict_interactions_device(dm, out, approximate=True))
    assert capi.last_predict_kernel() == "shap_approx"
    approx = out.get().reshape(args.rows, nc, nc)
    out.free()
    cout = capi.DeviceArray(args.rows * nc)
    t_contribs, n_contribs = timed(lambda: b.predict_contribs_device(dm, cout, approximate=False))
    cout.free()
    cores = oracle.use_all_cores()
    m = oracle.Model(path)
    oracle_interactions.build()  # compiled before the timed calls
    xs = x[: args.oracle_rows]
    t0 = time.perf_counter()
    ref = oracle_interactions.predict_interactions(m, xs)
    t_orc = time.perf_counter() - t0
    ref_a = oracle_interactions.predict_interactions(m, xs, approximate=True)
    n = len(xs)
    scale = np.abs(ref.astype(np.float64)).reshape(n, -1).sum(axis=1)
    ratio = float((np.abs(exact[:n].astype(np.float64) - ref).reshape(n, -1).max(axis=1) / scale).max())
    res = {
        "gpu": gpu, "power_limit": power_limit,
        "booster": f"{info.num_trees} trees, max depth {info.max_depth}, {info.num_nodes} nodes (bench.py seeded booster)",
        "rows": args.rows, "sample": "C90 x 72 rows, seeded (synth.raw_fields(90, seed=2024), rng 90)",
        "paths": n_paths, "path_condition_pairs": pairs, "bins": int(len(bins)),
        "exact_rows_per_s": args.rows / t_exact, "exact_s_per_call": t_exact, "exact_calls": n_exact,
        "exact_path_condition_pairs_per_s": pairs * args.rows / t_exact,
        "approx_rows_per_s": args.rows / t_approx, "approx_s_per_call": t_approx, "approx_calls": n_approx,
        "contribs_exact_rows_per_s": args.rows / t_contribs, "contribs_exact_s_per_call": t_contribs,
        "contribs_exact_calls": n_contribs,
        "oracle_cores": cores, "oracle_rows": n, "oracle_exact_rows_per_s": n / t_orc,
        "exact_vs_oracle_max_ratio": ratio,
        "approx_bit_equal_to_oracle": bool(np.array_equal(approx[:n].view(np.uint32), ref_a.view(np.uint32))),
    }  # fmt: skip
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
