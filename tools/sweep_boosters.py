#!/usr/bin/env python
"""BASELINE.json configs[4]: C180 x 72 with device-resident fields —
(a) booster sweep trees x depth (SURVEY.md 8d: trees in {10, 100, 500, 1000} x depth in {6, 10, 14, 18}, plus 30):
    cells/s, node visits per cell, fraction of the HBM roofline (112 B/cell) of the predict kernel, the kernel
    family that served it, forest bytes in both layouts.  10 / 30 / 100 trees are grown (seeded); 500 / 1000 are
    the 100-tree booster of that depth replicated 5 x / 10 x with jittered thresholds (synth.replicate_forest);
(b) forests larger than the 126 MB L2: a 20-tree booster with ~1e5 nodes per tree (grown on 700 k samples,
    min_leaf 2) replicated to 100 trees; both node layouts are timed (`duo` = 0 / 1);
(d) the production-shape booster on a matrix with 1 % missing entries (-999.0): the same two-level kernel with the
    default-direction test, against the clean matrix;
(c) one model day of 24 hourly steps with compute_once_per_day (1 boost step + 23 steps that reuse the persistent
    OH_ML), fields resident in HBM.
    python tools/sweep_boosters.py [--grid 180] [--grow-only] [--part a,b,c]"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from quickchem_b200 import synth, xgbmodel  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--grid", type=int, default=180)
ap.add_argument("--grow-only", action="store_true")
ap.add_argument("--trees", default="10,30,100,500,1000")
ap.add_argument("--depths", default="6,10,14,18")
ap.add_argument("--part", default="a,b,d,c")
ap.add_argument("--iters", type=int, default=10)
a = ap.parse_args()
os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
parts = set(a.part.split(","))
GROWN = (10, 30, 100)


def grown_path(t, d):
    p = os.path.join(ROOT, "build", f"oh_booster_{t}x{d}.model")
    if not os.path.exists(p):
        t0 = time.time()
        f = synth.prod_like_booster(n_trees=t, max_depth=d)
        xgbmodel.write_legacy_binary(f, p)
        print(f"grew {t}x{d}: {f.total_nodes()} nodes in {time.time() - t0:.0f}s", file=sys.stderr, flush=True)
    return p


def big_seed_path():
    p = os.path.join(ROOT, "build", "oh_booster_big20.model")
    if not os.path.exists(p):
        t0 = time.time()
        f = synth.prod_like_booster(n_trees=20, max_depth=18, n_sample=700000, min_leaf=2, seed=28, grid_n=48)
        xgbmodel.write_legacy_binary(f, p)
        print(f"grew big20: {f.total_nodes()} nodes in {time.time() - t0:.0f}s", file=sys.stderr, flush=True)
    return p


combos = [(t, d) for t in map(int, a.trees.split(",")) for d in map(int, a.depths.split(","))]
for t, d in combos:
    grown_path(t if t in GROWN else 100, d)
if "b" in parts:
    big_seed_path()
if a.grow_only:
    sys.exit(0)

from quickchem_b200 import capi  # noqa: E402

pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
peak = json.load(open(pk)).get("hbm_gbs", 6650.0) if os.path.exists(pk) else 6650.0
fields = synth.raw_fields(a.grid)
km, ncol = fields["T"].shape
ncell = km * ncol
dev = {k: capi.DeviceArray(v) for k, v in fields.items()}
out = capi.DeviceArray(ncell)
tmp = tempfile.mkdtemp(prefix="qcoh_sweep_")
state = {}


def matrix(b):
    """X assembled once on the device with the fused path, sealed (key tiles)."""
    if "dX" not in state:
        oh = capi.OhRun1(b, ncol, km, synth.MAPL, tropp_min=0.0)
        dX = capi.DMatrix.device(ncell, 27)
        xp = capi.vp()
        capi.check(capi.lib().qcoh_dmatrix_device_ptr(dX.handle, capi.C.byref(xp)))
        ro = capi.Run1Out()
        oh_out = capi.DeviceArray(ncell)
        ro.OH, ro.X = oh_out.ptr, xp
        capi.check(capi.lib().qcoh_oh_run1(oh.handle, capi.C.byref(oh.make_in(dev)), capi.C.byref(ro)))
        dX.seal()
        hx = np.empty((1 << 16, 27), np.float32)
        capi.check(capi.lib().qcoh_memcpy_d2h(hx.ctypes.data_as(capi.vp), xp, hx.nbytes))
        oh.free()
        state.update(dX=dX, hx=hx, oh_out=oh_out)
    return state["dX"], state["hx"]


def time_predict(b, dX):
    for _ in range(3):
        b.predict_device(dX, out, exp10=True, scale=0.85)
    capi.synchronize()
    capi.timer_start()
    for _ in range(a.iters):
        b.predict_device(dX, out, exp10=True, scale=0.85)
    ms = capi.timer_stop() / a.iters
    state["kernel"] = capi.last_predict_kernel()
    return ms


def model_file(t, d):
    if t in GROWN:
        return grown_path(t, d)
    p = os.path.join(tmp, f"rep_{t}x{d}.model")
    f = synth.replicate_forest(xgbmodel.read_legacy_binary(grown_path(100, d)), t // 100, seed=t + d)
    xgbmodel.write_legacy_binary(f, p)
    return p


def row(b, dX, hx, ms, **extra):
    info = b.info()
    visits = capi.node_visits_per_cell(b, hx[:2048])
    gbs = ncell * 112 / 1e9 / (ms * 1e-3)
    try:
        rec = b.duo()[0]
        duo_mb, (shift, has_dl) = rec.nbytes / 1e6, b.duo_info()
    except capi.QcohError:
        duo_mb, shift, has_dl = None, None, None
    r = dict(trees=info.num_trees, max_depth=info.max_depth, nodes=int(info.num_nodes), nodes8_mb=round(info.num_nodes * 8 / 1e6, 1),
             duo_mb=None if duo_mb is None else round(duo_mb, 1), duo_blk_shift=shift, visits_per_cell=round(visits, 1),
             kernel=state.get("kernel"), ms=round(ms, 3), cells_per_s=ncell / (ms * 1e-3), hbm_gbs=round(gbs, 1),
             hbm_frac=round(gbs / peak, 4), **extra)  # fmt: skip
    print(json.dumps(r), flush=True)
    return r


if "a" in parts:
    for t, d in combos:
        p = model_file(t, d)
        b = capi.Booster(p)
        dX, hx = matrix(b)
        ms = time_predict(b, dX)
        row(b, dX, hx, ms, sweep="trees x depth", grown=t in GROWN)
        b.free()
        if t not in GROWN:
            os.remove(p)

if "b" in parts:
    seed = xgbmodel.read_legacy_binary(big_seed_path())
    for times in (1, 7):
        f = synth.replicate_forest(seed, times, seed=99)
        p = os.path.join(tmp, f"big_{times}.model")
        xgbmodel.write_legacy_binary(f, p)
        b = capi.Booster(p)
        os.remove(p)
        dX, hx = matrix(b)
        for duo in (1, 0):
            capi.set_param("duo", duo)
            ms = time_predict(b, dX)
            row(b, dX, hx, ms, sweep="forest vs L2 (126 MB)", duo=duo, nodes_per_tree=int(b.info().num_nodes // b.info().num_trees))
        capi.set_param("duo", -1)
        b.free()

if "d" in parts:
    b = capi.Booster(grown_path(100, 18))
    dX, hx = matrix(b)
    ms_clean = time_predict(b, dX)
    row(b, dX, hx, ms_clean, sweep="missing entries", missing_frac=0.0)
    xp = capi.vp()
    capi.check(capi.lib().qcoh_dmatrix_device_ptr(dX.handle, capi.C.byref(xp)))
    full = np.empty((ncell, 27), np.float32)
    capi.check(capi.lib().qcoh_memcpy_d2h(full.ctypes.data_as(capi.vp), xp, full.nbytes))
    rng = np.random.default_rng(4)
    idx = rng.integers(0, full.size, full.size // 100)
    full.reshape(-1)[idx] = np.float32(-999.0)
    dM = capi.DMatrix.device(ncell, 27)
    dM.upload(full)
    dM.seal()
    ms_miss = time_predict(b, dM)
    row(b, dM, hx, ms_miss, sweep="missing entries", missing_frac=0.01, slowdown=round(ms_miss / ms_clean, 4))
    dM.free()
    del full
    b.free()

if "c" in parts:
    # one model day: 24 hourly steps, compute_once_per_day
    b = capi.Booster(grown_path(100, 18))
    matrix(b)
    oh = capi.OhRun1(b, ncol, km, synth.MAPL)  # 40 hPa slab as in production
    ro = capi.Run1Out()
    ro.OH = state["oh_out"].ptr
    k1 = 0
    for day in range(2):  # day 0 warms up (allocations, lazy kernel load, SZA cache); day 1 is timed
        t_steps = []
        for hour in range(24):
            rin = oh.make_in(dev, nymd=20220701 + day, need_to_call_boost=(hour == 0))
            capi.synchronize()
            t0 = time.perf_counter()
            capi.check(capi.lib().qcoh_oh_run1(oh.handle, capi.C.byref(rin), capi.C.byref(ro)))
            t_steps.append((time.perf_counter() - t0) * 1e3)
            if hour == 0:
                k1 = ro.k1
    print(json.dumps(dict(day="24 hourly steps, compute_once_per_day, device-resident fields (2nd day timed)", grid=a.grid, k1=k1,
                          boost_step_ms=round(t_steps[0], 2), other_step_ms=round(float(np.median(t_steps[1:])), 3),
                          day_ms=round(sum(t_steps), 2))), flush=True)  # fmt: skip
