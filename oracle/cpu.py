"""ctypes binding of oracle/libqc_oracle.so (TEST INFRASTRUCTURE ONLY; PARITY UNPINNED — see
oracle/qc_oracle.h).  Builds the library with oracle/Makefile on first use if it is missing."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

f32p = C.POINTER(C.c_float)


class _Node(C.Structure):
    _fields_ = [("parent", C.c_int32), ("cleft", C.c_int32), ("cright", C.c_int32), ("sindex", C.c_uint32),
                ("info", C.c_float)]  # fmt: skip


class _Stat(C.Structure):
    _fields_ = [("loss_chg", C.c_float), ("sum_hess", C.c_float), ("base_weight", C.c_float),
                ("leaf_child_cnt", C.c_int32)]  # fmt: skip


class _Tree(C.Structure):
    _fields_ = [("num_nodes", C.c_int32), ("nodes", C.POINTER(_Node)), ("stats", C.POINTER(_Stat))]


class _Model(C.Structure):
    _fields_ = [("base_score", C.c_float), ("num_feature", C.c_uint32), ("major_version", C.c_uint32),
                ("minor_version", C.c_uint32), ("num_trees", C.c_int32), ("trees", C.POINTER(_Tree)),
                ("tree_info", C.POINTER(C.c_int32)), ("objective", C.c_char * 64), ("booster", C.c_char * 32)]  # fmt: skip


class _DMat(C.Structure):
    _fields_ = [("nrow", C.c_uint64), ("ncol", C.c_uint64), ("offset", C.POINTER(C.c_uint64)),
                ("index", C.POINTER(C.c_uint32)), ("value", f32p)]  # fmt: skip


class Run1In(C.Structure):
    _fields_ = (
        [("ncol", C.c_int), ("km", C.c_int)]
        + [(n, C.c_float) for n in ("mapl_epsilon", "mapl_avogad", "mapl_runiv", "mapl_radians_to_degrees",
                                    "mapl_degrees_to_radians", "ohscale")]
        + [("compute_once_per_day", C.c_int), ("tropp_min", C.c_float), ("nymd", C.c_int), ("missing", C.c_float)]
        + [(n, f32p) for n in ("T_MOD", "Q_MOD", "PLE_MOD", "TROPP", "T_BST", "Q_BST", "PLE_BST", "ZLE_BST",
                               "TAUCLW", "TAUCLI", "FCLD", "CH4", "CO")]
        + [("SCA", f32p * 7)]
        + [(n, f32p) for n in ("NO2", "O3", "ISOP", "ACET", "C2H6", "C3H8", "PRPE", "ALK4", "MP", "H2O2", "CH2O",
                               "GMITO3", "GMITTO3", "ALBUV", "LATS", "LONS", "OH_CLIM")]
    )  # fmt: skip


class Run1Out(C.Structure):
    _fields_ = [("OH", f32p), ("OH_boost", f32p), ("X", f32p), ("feat3d", f32p * 27), ("NDWET", f32p),
                ("pred", f32p), ("k1", C.c_int)]  # fmt: skip


def _cpu_id() -> str:
    """The host CPU as far as -march=native cares: model name + ISA flags."""
    try:
        model = flags = ""
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and not model:
                model = line.split(":", 1)[1].strip()
            if line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
            if model and flags:
                break
        import hashlib

        return model + " " + hashlib.sha1(flags.encode()).hexdigest()[:12]
    except OSError:
        return "unknown"


def build_flags() -> str:
    try:
        return subprocess.check_output(["make", "-s", "-C", _HERE, "flags"], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def build(force=False):
    """Compile the C restatement (-O3 -march=native) next to its source, and rebuild it if the host's CPU is not
    the one it was built for (oracle/.cpu_stamp).  In a read-only checkout a library that has to be (re)built is
    built into a temporary directory for this process instead."""
    so = os.path.join(_HERE, "libqc_oracle.so")
    src = os.path.join(_HERE, "qc_oracle.c")
    stamp = os.path.join(_HERE, ".cpu_stamp")
    cpu = _cpu_id()
    try:
        built_for = open(stamp).read()
    except OSError:
        built_for = ""
    stale = not os.path.exists(so) or any(os.path.exists(f) and os.path.getmtime(f) > os.path.getmtime(so)
                                          for f in (src, os.path.join(_HERE, "Makefile")))  # fmt: skip
    if force or stale or built_for != cpu:
        writable = os.access(_HERE, os.W_OK) and (not os.path.exists(so) or os.access(so, os.W_OK))
        if not writable:
            tmp = tempfile.mkdtemp(prefix="qc_oracle_")
            atexit.register(shutil.rmtree, tmp, True)
            so = os.path.join(tmp, "libqc_oracle.so")
        subprocess.check_call(["make", "-C", _HERE, "-B", "OUT=" + so], stdout=subprocess.DEVNULL)
        if writable:
            with open(stamp, "w") as f:
                f.write(cpu)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.orc_last_error.restype = C.c_char_p
        L.orc_num_threads.restype = C.c_int
        L.orc_model_load.restype = C.POINTER(_Model)
        L.orc_model_load.argtypes = [C.c_char_p]
        L.orc_model_free.argtypes = [C.POINTER(_Model)]
        L.orc_dmatrix_from_mat.restype = C.POINTER(_DMat)
        L.orc_dmatrix_from_mat.argtypes = [f32p, C.c_uint64, C.c_uint64, C.c_float]
        L.orc_dmatrix_free.argtypes = [C.POINTER(_DMat)]
        L.orc_predict.restype = C.c_uint64
        L.orc_predict.argtypes = [C.POINTER(_Model), C.POINTER(_DMat), C.c_int, C.c_uint, f32p]
        L.orc_julian_day.argtypes = [C.c_int]
        L.orc_noon_sza.argtypes = [C.c_int, f32p, f32p, C.c_int, C.c_float, C.c_float, f32p]
        L.orc_run1.argtypes = [C.POINTER(_Model), C.POINTER(Run1In), C.POINTER(Run1Out)]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(f32p)


class OracleError(RuntimeError):
    pass


class Model:
    def __init__(self, path):
        self._m = lib().orc_model_load(os.fsencode(path))
        if not self._m:
            raise OracleError(lib().orc_last_error().decode())

    def __del__(self):
        if getattr(self, "_m", None):
            lib().orc_model_free(self._m)
            self._m = None

    @property
    def num_trees(self):
        return self._m.contents.num_trees

    @property
    def num_feature(self):
        return self._m.contents.num_feature

    @property
    def base_score(self):
        return self._m.contents.base_score

    @property
    def objective(self):
        return self._m.contents.objective.decode()

    def tree_arrays(self, t):
        tr = self._m.contents.trees[t]
        n = tr.num_nodes
        dt = np.dtype([("parent", "<i4"), ("cleft", "<i4"), ("cright", "<i4"), ("sindex", "<u4"), ("info", "<f4")])
        return np.ctypeslib.as_array(C.cast(tr.nodes, C.POINTER(C.c_uint8)), (n * 20,)).view(dt).copy()

    def predict(self, x, missing=-999.0, option_mask=0, ntree_limit=0):
        """XGDMatrixCreateFromMat + XGBoosterPredict on a host matrix."""
        x = np.ascontiguousarray(x, np.float32)
        nrow, ncol = x.shape
        d = lib().orc_dmatrix_from_mat(_p(x), nrow, ncol, missing)
        if not d:
            raise OracleError(lib().orc_last_error().decode())
        try:
            nt = self.num_trees if ntree_limit == 0 else min(ntree_limit, self.num_trees)
            out = np.empty(nrow * nt if option_mask & 2 else nrow, np.float32)
            n = lib().orc_predict(self._m, d, option_mask, ntree_limit, _p(out))
            if n != out.size and out.size:
                raise OracleError(lib().orc_last_error().decode())
        finally:
            lib().orc_dmatrix_free(d)
        return out.reshape(nrow, nt) if option_mask & 2 else out


def omp_threads() -> int:
    return lib().orc_num_threads()


def use_all_cores() -> int:
    """All host cores this process may run on, whatever OMP_NUM_THREADS says (torchrun exports 1)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    lib().orc_set_num_threads(n)
    return lib().orc_num_threads()


def julian_day(nymd):
    return lib().orc_julian_day(nymd)


def noon_sza(jday, lat, lon, r2d, d2r):
    lat = np.ascontiguousarray(lat, np.float32)
    lon = np.ascontiguousarray(lon, np.float32)
    out = np.empty_like(lat)
    lib().orc_noon_sza(jday, _p(lat), _p(lon), lat.size, r2d, d2r, _p(out))
    return out


def run1(model: Model, fields: dict, consts: dict, *, ohscale=0.85, compute_once_per_day=True, tropp_min=4000.0,
         nymd=20220701, missing=-999.0, mod_fields: dict | None = None, want_features=False):  # fmt: skip
    """One Run1 pass.  `fields` uses the import names of synth.raw_fields (ONLINE_INST aliasing:
    model-state T/Q/PLE are the boost-state ones unless `mod_fields` overrides them)."""
    km, ncol = fields["T"].shape
    keep = []

    def P(a):
        a = np.ascontiguousarray(a, np.float32)
        keep.append(a)
        return _p(a)

    mod = mod_fields or fields
    i = Run1In()
    i.ncol, i.km = ncol, km
    i.mapl_epsilon, i.mapl_avogad, i.mapl_runiv = consts["EPSILON"], consts["AVOGAD"], consts["RUNIV"]
    i.mapl_radians_to_degrees, i.mapl_degrees_to_radians = consts["RADIANS_TO_DEGREES"], consts["DEGREES_TO_RADIANS"]
    i.ohscale, i.compute_once_per_day, i.tropp_min, i.nymd, i.missing = ohscale, int(compute_once_per_day), tropp_min, nymd, missing
    i.T_MOD, i.Q_MOD, i.PLE_MOD, i.TROPP = P(mod["T"]), P(mod["Q"]), P(mod["PLE"]), P(mod["TROPP"])
    i.T_BST, i.Q_BST, i.PLE_BST, i.ZLE_BST = P(fields["T"]), P(fields["Q"]), P(fields["PLE"]), P(fields["ZLE"])
    i.TAUCLW, i.TAUCLI, i.FCLD, i.CH4, i.CO = (P(fields[k]) for k in ("TAUCLW", "TAUCLI", "FCLD", "CH4", "CO"))
    for s, sp in enumerate(("BC", "OC", "BR", "DU", "SU", "SS", "NI")):
        i.SCA[s] = P(fields[sp + "SCACOEF"])
    for g in ("NO2", "O3", "ISOP", "ACET", "C2H6", "C3H8", "PRPE", "ALK4", "MP", "H2O2", "CH2O"):
        setattr(i, g, P(fields["oh_" + g]))
    i.GMITO3, i.GMITTO3, i.ALBUV = P(fields["oh_GMITO3"]), P(fields["oh_GMITTO3"]), P(fields["oh_ALBUV"])
    i.LATS, i.LONS, i.OH_CLIM = P(fields["LATS"]), P(fields["LONS"]), P(fields["oh_OH"])
    o = Run1Out()
    res = {"OH": np.empty((km, ncol), np.float32), "OH_boost": np.empty((km, ncol), np.float32),
           "NDWET": np.empty((km, ncol), np.float32)}  # fmt: skip
    o.OH, o.OH_boost, o.NDWET = _p(res["OH"]), _p(res["OH_boost"]), _p(res["NDWET"])
    if want_features:
        res["feat"] = [np.empty(ncol if f in (0, 21, 22, 26) else (km, ncol), np.float32) for f in range(27)]
        for f in range(27):
            o.feat3d[f] = _p(res["feat"][f])
        res["X"] = np.empty((km * ncol, 27), np.float32)
        res["pred"] = np.empty(km * ncol, np.float32)
        o.X, o.pred = _p(res["X"]), _p(res["pred"])
    rc = lib().orc_run1(model._m, C.byref(i), C.byref(o))
    if rc != 0:
        raise OracleError(lib().orc_last_error().decode())
    res["k1"] = o.k1
    if want_features:
        n = (km - o.k1 + 1) * ncol
        res["X"], res["pred"] = res["X"][:n], res["pred"][:n]
    return res
