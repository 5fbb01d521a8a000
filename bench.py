#!/usr/bin/env python
"""bench.py — OH grid-cell predictions/sec of the B200 path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--grid 360] [--dump-outputs DIR]

A *step* is one pass of the hot path over the whole C<grid> x 72-level slab: the dense feature
matrix X[N x 27] (resident in HBM) -> tree-ensemble prediction -> 10**x * OHscale -> OH_ML, i.e.
what `predict_OH_with_XGB` does per call after packing (OH_GridCompMod.F90:347-374, :1569).
`value` times that with CUDA events on the library's stream (the DMatrix resident in HBM in its device
form, as XGDMatrixCreateFromMat leaves it); `e2e` times the same through the xgb_fortran_api C ABI
(XGDMatrixCreateFromMat + XGBoosterPredict + XGDMatrixFree) from pinned HOST buffers, H2D / D2H inside the
timed region, `e2e_pageable` from plain malloc'ed memory (what the reference's ALLOCATE gives), `h2d_floor_ms`
is the bare copy of the same buffer; `run1` (extra) times the fused device-resident Run1 (feature assembly +
predict + export transform + diagnostic partial sums).
N > 1: columns are sharded over ranks (one process per GPU, no collective on the data path;
the build-defined diagnostic is all-reduced over NCCL in the `run1` leg) — total work is fixed,
so scaling is "strong".  The synthetic fields are a function of the global column only, so every N
computes the same global OH: the line carries a checksum of the result bits that must not depend on N.

`--impl reference` times the reference's CPU algorithm (the libxgboost-1.6.0-equivalent oracle
restatement, OpenMP over all host cores) on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import atexit
import functools
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KM = 72
NFEAT = 27
ALGO_BYTES_PER_CELL = NFEAT * 4 + 4  # SURVEY.md 8(d): 27 float32 in + 1 float32 out
BOOSTER = dict(n_trees=100, max_depth=18)  # "Depth18_eta1_100Trees", OH_GridCompMod.F90:224
DUMP_CELLS = 1 << 22  # --dump-outputs keeps at most this many cells (16 MB of float32)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


@functools.lru_cache(maxsize=None)
def booster_path():
    """Seeded prod-like booster (100 trees, depth <= 18, 27 features); grown once and cached under build/.  A
    read-only checkout without it gets one grown into a temporary directory for this process."""
    from quickchem_b200 import synth, xgbmodel

    d = os.path.join(ROOT, "build")
    name = f"oh_booster_{BOOSTER['n_trees']}x{BOOSTER['max_depth']}.model"
    if os.path.exists(os.path.join(d, name)):
        return os.path.join(d, name)
    try:
        os.makedirs(d, exist_ok=True)
    except OSError:
        pass
    if not os.access(d, os.W_OK):
        d = tempfile.mkdtemp(prefix="qcoh_bench_")
        atexit.register(shutil.rmtree, d, True)
    p = os.path.join(d, name)
    if not os.path.exists(p):
        t0 = time.time()
        f = synth.prod_like_booster(**BOOSTER)
        xgbmodel.write_legacy_binary(f, p + ".tmp%d" % os.getpid())
        os.replace(p + ".tmp%d" % os.getpid(), p)
        log(f"[bench] grew booster: {f.total_nodes()} nodes in {time.time() - t0:.0f}s -> {p}")
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")  # fmt: skip

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)  # fmt: skip
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Summarise the samples taken inside [t0, t1] (the timed region)."""
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, reasons, smax = [], set(), None
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        inside = [r for ts, r in self.rows if (t0 is None or ts >= t0) and (t1 is None or ts <= t1 + 0.1)]
        for r in inside or [r for _, r in self.rows[-3:]]:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        hi = [v for v in sm if smax and v > 0.5 * smax] or sm
        return {"sm_mhz": statistics.median(hi) if hi else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}  # fmt: skip


def shard_rows(grid, rank, world):
    """This rank's range of j-rows of the (N, 6N) index space: whole blocks of synth.raw_fields_blocked."""
    from quickchem_b200 import synth

    rows = synth.field_block_rows(grid)
    nblk = 6 * grid // rows
    if nblk % world:
        raise SystemExit(f"C{grid}: {nblk} field blocks do not split over {world} ranks")
    return rows * (nblk * rank // world), rows * (nblk * (rank + 1) // world)


def shard_fields(grid, rank, world):
    """This rank's contiguous column range of C<grid> (whole j-rows) and its synthetic fields — the same global
    fields for every world size."""
    from quickchem_b200 import synth

    j0, j1 = shard_rows(grid, rank, world)
    col0, ncol = j0 * grid, (j1 - j0) * grid
    t0 = time.time()
    f = synth.raw_fields_blocked(grid, 20220726 + grid, j0, j1)
    log(f"[bench r{rank}] synthetic fields C{grid} cols [{col0},{col0 + ncol}) in {time.time() - t0:.0f}s")
    return col0, ncol, f


def run_reference(args):
    """The reference's CPU algorithm (oracle restatement) on a bounded sample; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu as oracle
    from quickchem_b200 import synth

    oracle.build()
    model = oracle.Model(booster_path())
    grid = args.grid
    nrows_j = max(1, min(6 * grid, args.ref_cols // grid))
    rows = synth.field_block_rows(grid)
    nrows_j = max(rows, nrows_j // rows * rows)
    f = synth.raw_fields_blocked(grid, 20220726 + grid, 0, nrows_j)
    r = oracle.run1(model, f, synth.MAPL, tropp_min=0.0, want_features=True)
    X = np.ascontiguousarray(r["X"])
    n = X.shape[0]
    out = np.empty(n, np.float32)
    cores = oracle.use_all_cores()

    def step():
        p = model.predict(X)  # orc_dmatrix_from_mat + orc_predict (:347-356)
        np.power(np.float32(10.0), p, out=out)  # :369

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    sample = f"{n} rows = first {nrows_j * grid} columns x {KM} levels of C{grid}, per step"
    print(json.dumps({
        "impl": "reference", "metric": "OH grid-cell predictions/sec", "value": v, "unit": "cells/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(grid, args.gpus), sample=sample,
                       note="rate-based: each step times the CPU algorithm on this bounded sample of the workload's rows"),
        "cpu_baseline": {"value": v, "unit": "cells/s", "cores": cores, "kind": "port", "sample": sample,
                         "build": oracle.build_flags()},
        "e2e": {"value": v, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)  # fmt: skip


def workload_config(grid, world):
    which = {90: "configs[1]", 360: "configs[2]", 720: "configs[3]", 180: "configs[4]"}.get(grid, "other grid")
    return {"workload": f"C{grid}x{KM}L OH prediction, {6 * grid * grid * KM} cells, dense X[Nx27] f32 (BASELINE {which})",
            "booster": f"{BOOSTER['n_trees']} trees, max depth {BOOSTER['max_depth']}, 27 features (synthetic, seeded)",
            "sharding": f"{world} rank(s), contiguous column blocks, no halo",
            "cache": "inputs (>= 0.75 GB per GPU) exceed the 126 MB L2; forest stays L2-resident by design"}  # fmt: skip


def dump_outputs(out_dir, grid, col0, ncol, oh, rank, world, dist):
    """--dump-outputs: this rank's OH values `oh` (the last timed step's result, rows k * ncol + local column) at a
    fixed set of global cells, gathered on rank 0 into DIR/oh.npy in global cell order (k * 6 grid^2 + column), so
    that two builds run with the same arguments can be compared value for value at any number of GPUs."""
    ncol_g = 6 * grid * grid
    n = ncol_g * KM
    cells = np.arange(n) if n <= DUMP_CELLS else np.unique(np.random.default_rng(0).integers(0, n, DUMP_CELLS))
    k, col = np.divmod(cells, ncol_g)
    mine = (col >= col0) & (col < col0 + ncol)
    part = (np.nonzero(mine)[0], oh[k[mine] * ncol + col[mine] - col0])
    parts = [part]
    if dist:
        parts = [None] * world
        dist.all_gather_object(parts, part)
    if rank != 0:
        return
    sample = np.full(cells.size, np.nan, np.float32)
    for pos, v in parts:
        sample[pos] = v
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "oh.npy"), sample)
    log(f"[bench] wrote {sample.size} of {n} OH values to {os.path.join(out_dir, 'oh.npy')}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="qcoh", choices=["qcoh", "reference"])
    ap.add_argument("--grid", type=int, default=360, help="cubed-sphere C<grid> (BASELINE configs[2] = 360)")
    ap.add_argument("--ref-cols", type=int, default=7200, help="columns in the CPU sample")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU-baseline time")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--param", action="append", default=[], help="name=value forwarded to qcoh_set_param")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the OH values of the last timed step to DIR/oh.npy (float32; every cell of a grid of "
                         f"at most {DUMP_CELLS} cells, else a fixed seeded sample of about that many)")  # fmt: skip
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "qcoh":
        ap.error("--dump-outputs writes the outputs of the qcoh path")
    args.warmup = max(args.warmup, 3) if args.impl == "qcoh" else args.warmup

    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch  # plumbing only: process group, barrier, max-over-ranks

    dist = None
    if world > 1:
        # keep stdout to the one JSON line: NCCL's banner / logs go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from quickchem_b200 import capi, synth

    L = capi.lib()
    capi.check(L.qcoh_set_device(local))
    for kv in args.param:
        k, v = kv.split("=")
        capi.set_param(k, v)
    if rank == 0:
        booster_path()
    if dist:
        dist.barrier()
        # the library's own NCCL communicator for the diagnostic all-reduce: rank 0's id travels over the
        # process group (a MAPL host would MPI_Bcast it)
        uid = [capi.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        capi.comm_init(world, rank, uid[0])
    booster = capi.Booster(booster_path())
    info = booster.info()

    col0, ncol, fields = shard_fields(args.grid, rank, world)
    ncell = ncol * KM
    area = np.full(ncol, 5.1e14 / (6 * args.grid * args.grid), np.float32)
    dev = {k: capi.DeviceArray(v) for k, v in fields.items()}
    d_area = capi.DeviceArray(area)
    # tropp_min = 0 Pa: the slab is all 72 levels, as BASELINE.json's cell counts require
    oh = capi.OhRun1(booster, ncol, KM, synth.MAPL, tropp_min=0.0)
    rin = oh.make_in(dev, area=d_area)
    dX = capi.DMatrix.device(ncell, NFEAT)
    xptr = capi.vp()
    capi.check(L.qcoh_dmatrix_device_ptr(dX.handle, capi.C.byref(xptr)))
    d_out = {n: capi.DeviceArray(ncell) for n in ("OH", "OH_boost")}
    ro = capi.Run1Out()
    ro.OH, ro.OH_boost, ro.X = d_out["OH"].ptr, d_out["OH_boost"].ptr, xptr
    capi.check(L.qcoh_oh_run1(oh.handle, capi.C.byref(rin), capi.C.byref(ro)))
    assert ro.k1 == 1, ro.k1
    dX.seal()  # XGDMatrixCreateFromMat's device work: missing / inf scan + key tiles (the DMatrix's device form)
    ro.X = None
    d_pred = capi.DeviceArray(ncell)

    def barrier():
        capi.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize() if world > 1 else None

    def max_over_ranks(ms):
        if not dist:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    window = [0.0, 0.0]

    def timed(fn, steps, warm):
        """CUDA events on the library's stream around exactly `steps` calls, max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        n0 = capi.launch_count()
        window[0] = time.time()
        capi.timer_start()
        for _ in range(steps):
            fn()
        ms = capi.timer_stop()
        window[1] = time.time()
        barrier()
        return max_over_ranks(ms) / steps, capi.launch_count() - n0

    def wall(fn, steps, warm):
        """Host clock around `steps` blocking calls (they end with the result on the host), max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        capi.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        barrier()
        return max_over_ranks(dt) / steps

    total_cells = 6 * args.grid * args.grid * KM
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)  # let nvidia-smi start sampling before the warm-up

    # ---- value: predict step on the resident DMatrix (K2b + fused export transform)
    step = lambda: booster.predict_device(dX, d_pred, exp10=True, scale=0.85)
    ms_step, launches = timed(step, args.steps, args.warmup)
    clocks = sampler.stop(*window) if rank == 0 else None
    value = total_cells / (ms_step * 1e-3)
    served_by = capi.last_predict_kernel()

    # ---- the result itself: a checksum of the OH bits that must not depend on the number of ranks (the fields are
    # a function of the global column only), and the raw margins for the bit-level parity check below
    oh_host = d_pred.get()
    oh_bits = oh_host.view(np.uint32)
    local_ck = [int(np.bitwise_xor.reduce(oh_bits)), int(oh_bits.sum(dtype=np.uint64)), int(oh_bits.size)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, args.grid, col0, ncol, oh_host, rank, world, dist)
    del oh_bits, oh_host
    all_ck = [local_ck]
    if dist:
        all_ck = [None] * world
        dist.all_gather_object(all_ck, local_ck)
    ck_xor, ck_sum, ck_n = 0, 0, 0
    for x_, s_, n_ in all_ck:
        ck_xor ^= x_
        ck_sum = (ck_sum + s_) % (1 << 64)
        ck_n += n_
    d_margin = capi.DeviceArray(ncell)
    booster.predict_device(dX, d_margin, option_mask=1)
    capi.synchronize()

    # ---- create: XGDMatrixCreateFromMat's device work on the resident matrix, timed for the record
    ms_seal, _ = timed(lambda: dX.seal(), 3, 1)

    # ---- run1: fused device-resident Run1 (+ NCCL all-reduce of the diagnostic at N > 1)
    diag_sum = [list(ro.diag)]

    def run1_step():
        capi.check(L.qcoh_oh_run1(oh.handle, capi.C.byref(rin), capi.C.byref(ro)))
        if dist:  # ncclAllReduce(sum, float64, count = 4) inside libqcoh, over NVLink / NVSwitch
            diag_sum[0] = capi.comm_allreduce_sum(list(ro.diag)).tolist()

    ms_run1 = wall(run1_step, max(3, args.steps // 2), 2)
    diag = list(ro.diag) if not dist else diag_sum[0]
    run1_bits = d_out["OH_boost"].get().view(np.uint32)
    run1_ck = [int(np.bitwise_xor.reduce(run1_bits)), int(run1_bits.size)]
    del run1_bits
    all_r1 = [run1_ck]
    if dist:
        all_r1 = [None] * world
        dist.all_gather_object(all_r1, run1_ck)
    r1_xor = 0
    for x_, _n in all_r1:
        r1_xor ^= x_

    # ---- e2e: xgb_fortran_api C ABI from host buffers
    e2e = e2e_pageable = None
    h2d_floor_ms = None
    hX = None
    if not args.no_e2e:
        hX = capi.pinned_empty((ncell, NFEAT))
        capi.check(L.qcoh_memcpy_d2h(hX.ctypes.data_as(capi.vp), xptr, hX.nbytes))
        sink = np.zeros(1, np.float64)

        def e2e_step_on(host_x):
            def f():
                d = capi.DMatrix(host_x, -999.0)         # XGDMatrixCreateFromMat_f (:347)  H2D
                n, p = booster.predict_raw(d)            # XGBoosterPredict_f (:356)        kernel + D2H
                res = np.ctypeslib.as_array(p, (n,))
                sink[0] = float(res[0]) + float(res[n - 1])  # the host reads the result it was handed
                d.free()                                 # XGDMatrixFree_f (:377)
            return f

        nsteps = max(3, args.steps // 2)
        ms_e2e = wall(e2e_step_on(hX), nsteps, 3)
        # the bare H2D of the same pinned buffer into HBM (one cudaMemcpyAsync): the PCIe floor under e2e
        h2d_floor_ms = wall(lambda: capi.check(L.qcoh_memcpy_h2d(xptr, hX.ctypes.data_as(capi.vp), hX.nbytes)), 3, 1)
        dX.seal()
        e2e = {"value": total_cells / (ms_e2e * 1e-3), "unit": "cells/s", "h2d_bytes_per_step": ncell * NFEAT * 4 * world,
               "d2h_bytes_per_step": ncell * 4 * world, "ms_per_step": ms_e2e, "h2d_floor_ms": h2d_floor_ms,
               "fraction_of_h2d_floor": h2d_floor_ms / ms_e2e,
               "h2d_gbs_per_rank": ncell * NFEAT * 4 / 1e9 / (h2d_floor_ms * 1e-3),
               "path": "XGDMatrixCreateFromMat+XGBoosterPredict+XGDMatrixFree, pinned host X, result read on host"}  # fmt: skip
        # pageable host memory: what the unmodified Fortran caller's ALLOCATE(xx_carr) gives (:306)
        try:
            pX = np.empty((ncell, NFEAT), np.float32)
            np.copyto(pX, hX)
            ms_pg = wall(e2e_step_on(pX), nsteps, 2)
            e2e_pageable = {"value": total_cells / (ms_pg * 1e-3), "unit": "cells/s", "ms_per_step": ms_pg,
                            "fraction_of_pinned": ms_e2e / ms_pg,
                            "path": "same calls, pageable (malloc) host X staged through the library's pinned ring"}
            del pX
        except MemoryError:
            e2e_pageable = {"unavailable": "not enough host memory for a second copy of X"}

    # ---- cpu_baseline: oracle on a bounded sample of the same X (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import cpu as oracle

        oracle.build()
        oracle.use_all_cores()
        om = oracle.Model(booster_path())
        hs = np.empty((1 << 18, NFEAT), np.float32)
        stride = max(1, ncell // hs.shape[0])
        probe_rows = np.arange(hs.shape[0]) * stride
        full = hX
        if full is None:
            full = capi.pinned_empty((ncell, NFEAT))
            capi.check(L.qcoh_memcpy_d2h(full.ctypes.data_as(capi.vp), xptr, full.nbytes))
        hs[:] = full[probe_rows]
        t0 = time.perf_counter()
        om.predict(hs)
        probe_dt = time.perf_counter() - t0
        nsamp = int(min(ncell, max(hs.shape[0], hs.shape[0] * args.cpu_seconds / max(probe_dt, 1e-3))))
        nsamp = min(nsamp, 1 << 25)
        stride = max(1, ncell // nsamp)
        rows = np.arange(nsamp) * stride
        xs = np.ascontiguousarray(full[rows])
        t0 = time.perf_counter()
        ref = om.predict(xs)
        oh_ref = np.power(np.float32(10.0), ref) * np.float32(0.85)
        cpu_dt = time.perf_counter() - t0
        # parity on the sampled rows: the raw float32 margins bit for bit (a wrong leaf anywhere changes them),
        # and the fused 10**x * OHscale within the 1e-6 of BASELINE.json
        m_gpu = d_margin.get()[rows]
        ulp = np.abs(m_gpu.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
        got = d_pred.get()[rows]
        rel = float(np.max(np.abs(got.astype(np.float64) - oh_ref) / np.abs(oh_ref)))
        cpu = {"value": nsamp / cpu_dt, "unit": "cells/s", "cores": oracle.omp_threads(), "kind": "port",
               "sample": f"{nsamp} rows (every {stride}th row of the C{args.grid}x{KM} matrix): dense->CSR + predict + 10**x",
               "seconds": cpu_dt, "build": oracle.build_flags(),
               "margin_bits_equal": bool(np.array_equal(m_gpu.view(np.uint32), ref.view(np.uint32))),
               "margin_max_ulp": int(ulp.max()), "max_rel_err_gpu_vs_cpu": rel}  # fmt: skip

    if rank != 0:
        if dist:
            capi.comm_destroy()
            dist.destroy_process_group()
        return
    # compute-side view of the same kernel: node visits per second (SURVEY.md 8d "compute-side bound")
    xs_v = np.empty((4096, NFEAT), np.float32)
    capi.check(L.qcoh_memcpy_d2h(xs_v.ctypes.data_as(capi.vp), xptr, xs_v.nbytes))
    visits = capi.node_visits_per_cell(booster, xs_v)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    achieved = (ncell * ALGO_BYTES_PER_CELL / 1e9) / (ms_step * 1e-3)  # per GPU: this rank's launch
    traffic = traffic_src = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture, scaled to this launch
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) / tj["cells_per_launch"] * ncell
        traffic_src = tj["source"]
    except (OSError, KeyError, ValueError):
        pass
    out = {
        "metric": "OH grid-cell predictions/sec", "value": value, "unit": "cells/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.grid, world),
        "value_scope": "predict step (XGBoosterPredict + 10**x * OHscale) on the resident DMatrix; `run1` below is the full "
                       "Run1-equivalent step from raw fields (assembly + predict + finalize + diagnostic)",
        "clocks": clocks, "e2e": e2e, "e2e_pageable": e2e_pageable, "gpu_launches": launches,
        "kernel": served_by,
        "checksum": {"oh_xor": f"0x{ck_xor:08x}", "oh_sum_u32": ck_sum, "cells": ck_n, "run1_oh_boost_xor": f"0x{r1_xor:08x}",
                     "note": "XOR / sum of the float32 bit patterns of all predicted OH values over all ranks: independent of n_gpus"},
        "roofline": {"bound": "hbm", "kernel": "predict_tiles_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6.65 TB/s",
                     "algorithmic_bytes_per_cell": ALGO_BYTES_PER_CELL, "cells_per_launch": ncell,
                     "compute_side": {"node_visits_per_cell": round(visits, 1), "node_visits_per_s_per_gpu": ncell * visits / (ms_step * 1e-3),
                                      "note": "one visit = one tree level of one row; a 16-byte record gather decides two of them"},
                     "note": "traversal is bound by the L1TEX data pipes (record gathers + feature fetches) and issue slots, not HBM "
                             "(profiles/README.md); the HBM-bound end of the booster sweep is in profiles/r2_sweep_*.jsonl"},
        "cpu_baseline": cpu,
        "create_device": {"ms": ms_seal, "what": "XGDMatrixCreateFromMat's device work on a resident matrix: scan + key tiles"},
        "run1": {"value": total_cells / (ms_run1 * 1e-3), "unit": "cells/s", "ms_per_step": ms_run1,
                 "what": "fused device-resident Run1: assembly + predict + export transform + diagnostic"
                         + (" + NCCL all-reduce" if dist else ""),
                 "global_mean_oh_molec_cm3": diag[0] / diag[1] if diag[1] else None,
                 "ch4_lifetime_years": diag[2] / diag[3] / 3.15576e7 if diag[3] else None,
                 "diag_sums": diag},
        "booster": {"trees": info.num_trees, "nodes": int(info.num_nodes), "max_depth": info.max_depth},
    }  # fmt: skip
    print(json.dumps(out), flush=True)
    if dist:
        capi.comm_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
