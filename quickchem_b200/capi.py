"""ctypes binding of libqcoh.so (include/qcoh.h) for the test-suite and bench.py.

Python is harness only: everything numerical happens inside the shared library on the GPU.
There is no fallback — if the library is missing this module raises, and every compute call
fails with the library's own error on a box without a CUDA device.

Names mirror the reference's Fortran interface module (`Shared/xgb_fortran_api.F90`): the
`XG*` wrappers take the same arguments in the same order and return the same `rc`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QCOH_LIB") or os.path.join(_HERE, "libqcoh.so")  # QCOH_LIB: load another build, e.g. to compare two side by side

f32p = C.POINTER(C.c_float)
u64 = C.c_uint64
vp = C.c_void_p


class QcohError(RuntimeError):
    pass


class BoosterInfo(C.Structure):
    _fields_ = [("num_trees", C.c_int32), ("num_feature", C.c_int32), ("max_depth", C.c_int32),
                ("num_nodes", C.c_int64), ("base_score", C.c_float), ("format", C.c_int32),
                ("version", C.c_uint32 * 3)]  # fmt: skip


class Epilogue(C.Structure):
    _fields_ = [("exp10", C.c_int), ("scale", C.c_float)]


class OhConfig(C.Structure):
    _fields_ = [("ncol", C.c_int), ("km", C.c_int), ("mapl_epsilon", C.c_float), ("mapl_avogad", C.c_float),
                ("mapl_runiv", C.c_float), ("mapl_radians_to_degrees", C.c_float),
                ("mapl_degrees_to_radians", C.c_float), ("ohscale", C.c_float), ("compute_once_per_day", C.c_int),
                ("tropp_min", C.c_float), ("missing", C.c_float)]  # fmt: skip


_IN_PTRS = ("T_MOD", "Q_MOD", "PLE_MOD", "TROPP", "T_BST", "Q_BST", "PLE_BST", "ZLE_BST", "TAUCLW", "TAUCLI",
            "FCLD", "CH4", "CO")  # fmt: skip
_IN_PTRS2 = ("NO2", "O3", "ISOP", "ACET", "C2H6", "C3H8", "PRPE", "ALK4", "MP", "H2O2", "CH2O", "GMITO3",
             "GMITTO3", "ALBUV", "LATS", "LONS", "OH_CLIM", "AREA")  # fmt: skip


class Run1In(C.Structure):
    _fields_ = ([("nymd", C.c_int), ("need_to_call_boost", C.c_int)] + [(n, vp) for n in _IN_PTRS]
                + [("SCA", vp * 7)] + [(n, vp) for n in _IN_PTRS2])  # fmt: skip


class Run1Out(C.Structure):
    _fields_ = [("OH", vp), ("OH_boost", vp), ("NDWET", vp), ("X", vp), ("pred", vp),
                ("LOSS_CH4", vp), ("LOSS_CO", vp), ("k1", C.c_int),
                ("diag", C.c_double * 4)]  # fmt: skip


# every symbol include/qcoh.h declares (tests check the library exports all of them)
XGB_SYMBOLS = ("XGBoosterLoadModel", "XGBoosterSaveModel", "XGDMatrixSaveBinary", "XGDMatrixFree",
               "XGDMatrixCreateFromFile", "XGBoosterPredict", "XGBoosterCreate", "XGDMatrixCreateFromMat",
               "XGDMatrixNumRow", "XGDMatrixNumCol", "XGBoosterFree", "XGBGetLastError", "XGBoosterPredictFromDMatrix",
               "XGBoosterPredictFromDense", "XGBoosterPredictFromCudaArray", "XGBoosterPredictFromCudaColumnar",
               "XGDMatrixCreateFromDense", "XGDMatrixCreateFromCudaArrayInterface", "XGDMatrixCreateFromCudaColumnar")  # fmt: skip
QCOH_SYMBOLS = ("qcoh_version", "qcoh_device_count", "qcoh_set_device", "qcoh_host_alloc", "qcoh_host_free",
                "qcoh_device_alloc", "qcoh_device_free", "qcoh_memcpy_h2d", "qcoh_memcpy_d2h",
                "qcoh_device_synchronize", "qcoh_timer_start", "qcoh_timer_stop", "qcoh_flush_l2",
                "qcoh_booster_parse", "qcoh_booster_get_info", "qcoh_booster_get_flat", "qcoh_booster_get_duo",
                "qcoh_booster_get_duo_info", "qcoh_booster_get_shap_paths", "qcoh_booster_predict_contribs_device",
                "qcoh_booster_predict_interactions_device",
                "qcoh_dmatrix_create_device", "qcoh_dmatrix_device_ptr", "qcoh_dmatrix_upload", "qcoh_dmatrix_seal",
                "qcoh_booster_predict_device", "qcoh_set_param", "qcoh_launch_count", "qcoh_kernel_launches",
                "qcoh_last_predict_kernel", "qcoh_dmatrix_tiles_ptr", "qcoh_oh_invalidate_sza", "qcoh_oh_create",
                "qcoh_oh_run1", "qcoh_oh_free", "qcoh_oh_get_diag", "qcoh_predict_OH_with_XGB", "qcoh_predict_OH_reset",
                "qcoh_predict_OH_reload_on_file_change", "qcoh_oh_set_booster", "qcoh_oh_get_booster",
                "qcoh_expand_template", "qcoh_model_cache_get", "qcoh_model_cache_size", "qcoh_model_cache_clear",
                "qcoh_oh_select_model", "qcoh_data_source_from_name", "qcoh_need_to_call_boost", "qcoh_use_inst_values",
                "qcoh_import_name",
                "qcoh_partition_columns", "qcoh_comm_get_unique_id", "qcoh_comm_init",
                "qcoh_comm_allreduce_sum_f64", "qcoh_comm_destroy")  # fmt: skip

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise QcohError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(make -C quickchem_b200/csrc); there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.XGBGetLastError.restype = C.c_char_p
        L.qcoh_version.restype = C.c_char_p
        L.qcoh_launch_count.restype = C.c_uint64
        L.qcoh_kernel_launches.restype = C.c_uint64
        L.qcoh_kernel_launches.argtypes = [C.c_char_p]
        L.qcoh_last_predict_kernel.restype = C.c_char_p
        L.qcoh_dmatrix_tiles_ptr.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
        L.qcoh_oh_invalidate_sza.argtypes = [vp]
        L.XGBoosterCreate.argtypes = [vp, u64, C.POINTER(vp)]
        L.XGBoosterFree.argtypes = [vp]
        L.XGBoosterLoadModel.argtypes = [vp, C.c_char_p]
        L.XGBoosterSaveModel.argtypes = [vp, C.c_char_p]
        L.XGDMatrixCreateFromMat.argtypes = [vp, u64, u64, C.c_float, C.POINTER(vp)]
        L.XGDMatrixCreateFromFile.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
        L.XGDMatrixSaveBinary.argtypes = [vp, C.c_char_p, C.c_int]
        L.XGDMatrixFree.argtypes = [vp]
        L.XGDMatrixNumRow.argtypes = [vp, C.POINTER(u64)]
        L.XGDMatrixNumCol.argtypes = [vp, C.POINTER(u64)]
        L.XGBoosterPredict.argtypes = [vp, vp, C.c_int, C.c_uint, C.c_int, C.POINTER(u64), C.POINTER(f32p)]
        L.qcoh_set_device.argtypes = [C.c_int]
        L.qcoh_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
        L.qcoh_host_free.argtypes = [vp]
        L.qcoh_device_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
        L.qcoh_device_free.argtypes = [vp]
        L.qcoh_memcpy_h2d.argtypes = [vp, vp, C.c_size_t]
        L.qcoh_memcpy_d2h.argtypes = [vp, vp, C.c_size_t]
        L.qcoh_timer_stop.argtypes = [C.POINTER(C.c_float)]
        L.qcoh_booster_parse.argtypes = [vp, C.c_char_p]
        L.qcoh_booster_get_info.argtypes = [vp, C.POINTER(BoosterInfo)]
        L.qcoh_booster_get_flat.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.POINTER(C.c_uint32)),
                                            C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32))]  # fmt: skip
        L.qcoh_booster_get_duo.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.POINTER(C.c_uint32)),
                                           C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.c_int64)]  # fmt: skip
        L.qcoh_booster_get_duo_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.qcoh_dmatrix_create_device.argtypes = [u64, u64, C.c_float, C.POINTER(vp)]
        L.qcoh_dmatrix_device_ptr.argtypes = [vp, C.POINTER(vp)]
        L.qcoh_dmatrix_upload.argtypes = [vp, vp, u64, u64]
        L.qcoh_dmatrix_seal.argtypes = [vp]
        L.qcoh_booster_predict_device.argtypes = [vp, vp, C.c_int, C.c_uint, C.POINTER(Epilogue), vp]
        L.XGBoosterPredictFromDMatrix.argtypes = [vp, vp, C.c_char_p, C.POINTER(C.POINTER(u64)), C.POINTER(u64),
                                                  C.POINTER(f32p)]  # fmt: skip
        for name in ("XGDMatrixCreateFromDense", "XGDMatrixCreateFromCudaArrayInterface", "XGDMatrixCreateFromCudaColumnar"):
            getattr(L, name).argtypes = [C.c_char_p, C.c_char_p, C.POINTER(vp)]
        for name in ("XGBoosterPredictFromDense", "XGBoosterPredictFromCudaArray", "XGBoosterPredictFromCudaColumnar"):
            getattr(L, name).argtypes = [vp, C.c_char_p, C.c_char_p, vp, C.POINTER(C.POINTER(u64)), C.POINTER(u64), C.POINTER(f32p)]
        L.qcoh_booster_predict_contribs_device.argtypes = [vp, vp, C.c_int, C.c_uint, vp]
        L.qcoh_booster_predict_interactions_device.argtypes = [vp, vp, C.c_int, C.c_uint, vp]
        L.qcoh_booster_get_shap_paths.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.POINTER(C.c_int64)),
                                                  C.POINTER(C.POINTER(C.c_float)), C.POINTER(C.c_int64)]  # fmt: skip
        L.qcoh_set_param.argtypes = [C.c_char_p, C.c_char_p]
        L.qcoh_oh_create.argtypes = [vp, C.POINTER(OhConfig), C.POINTER(vp)]
        L.qcoh_oh_run1.argtypes = [vp, C.POINTER(Run1In), C.POINTER(Run1Out)]
        L.qcoh_oh_free.argtypes = [vp]
        L.qcoh_oh_get_diag.argtypes = [vp, C.c_char_p, vp]
        L.qcoh_predict_OH_with_XGB.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp,
                                               C.POINTER(vp), C.POINTER(C.c_int), vp]  # fmt: skip
        L.qcoh_partition_columns.argtypes = [C.c_int64, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.qcoh_comm_get_unique_id.argtypes = [C.c_char_p]
        L.qcoh_comm_init.argtypes = [C.c_int, C.c_int, C.c_char_p]
        L.qcoh_comm_allreduce_sum_f64.argtypes = [C.POINTER(C.c_double), C.c_int]
        L.qcoh_oh_set_booster.argtypes = [vp, vp]
        L.qcoh_oh_get_booster.argtypes = [vp, C.POINTER(vp)]
        L.qcoh_expand_template.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t]
        L.qcoh_model_cache_get.argtypes = [C.c_char_p, C.POINTER(vp)]
        L.qcoh_oh_select_model.argtypes = [vp, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.qcoh_data_source_from_name.argtypes = [C.c_char_p]
        L.qcoh_need_to_call_boost.argtypes = [C.c_int, C.c_int]
        L.qcoh_use_inst_values.argtypes = [C.c_int, C.c_float]
        L.qcoh_import_name.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_int)]
        L.qcoh_predict_OH_reload_on_file_change.argtypes = [C.c_int]
        L.qcoh_predict_OH_reload_on_file_change.restype = None
        _LIB = L
    return _LIB


def last_error() -> str:
    return lib().XGBGetLastError().decode(errors="replace")


def check(rc: int):
    if rc != 0:
        raise QcohError(last_error())


def device_count() -> int:
    return lib().qcoh_device_count()


def set_param(name: str, value) -> None:
    check(lib().qcoh_set_param(name.encode(), str(value).encode()))


def launch_count() -> int:
    return int(lib().qcoh_launch_count())


def kernel_launches(family: str) -> int:
    """Launches of one kernel family since load ("duo", "duo_missing", "duo_leaf", "nodes8", ...)."""
    return int(lib().qcoh_kernel_launches(family.encode()))


def last_predict_kernel() -> str:
    return lib().qcoh_last_predict_kernel().decode()


def partition_columns(ncol_global: int, nranks: int, rank: int):
    c0, n = C.c_int64(), C.c_int64()
    check(lib().qcoh_partition_columns(ncol_global, nranks, rank, C.byref(c0), C.byref(n)))
    return c0.value, n.value


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    check(lib().qcoh_comm_get_unique_id(buf))
    return buf.raw


def comm_init(nranks: int, rank: int, uid: bytes) -> None:
    check(lib().qcoh_comm_init(nranks, rank, uid))


def comm_allreduce_sum(values) -> np.ndarray:
    """NCCL all-reduce (sum) of a few float64 values, in the library, without torch."""
    a = np.ascontiguousarray(values, np.float64).copy()
    check(lib().qcoh_comm_allreduce_sum_f64(a.ctypes.data_as(C.POINTER(C.c_double)), a.size))
    return a


def comm_destroy() -> None:
    check(lib().qcoh_comm_destroy())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(vp)


def pinned_empty(shape, dtype=np.float32) -> np.ndarray:
    """numpy array backed by cudaHostAlloc'ed memory (kept alive for the life of the process)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = vp()
    check(lib().qcoh_host_alloc(n, C.byref(p)))
    buf = (C.c_char * n).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


class DeviceArray:
    """Raw HBM buffer (float32) managed through the C ABI."""

    def __init__(self, n_or_array):
        self.ptr = vp()
        if isinstance(n_or_array, np.ndarray):
            a = np.ascontiguousarray(n_or_array, np.float32)
            self.n = a.size
            check(lib().qcoh_device_alloc(max(a.nbytes, 4), C.byref(self.ptr)))
            check(lib().qcoh_memcpy_h2d(self.ptr, _ptr(a), a.nbytes))
        else:
            self.n = int(n_or_array)
            check(lib().qcoh_device_alloc(max(self.n * 4, 4), C.byref(self.ptr)))

    def get(self, n=None) -> np.ndarray:
        out = np.empty(self.n if n is None else n, np.float32)
        check(lib().qcoh_memcpy_d2h(_ptr(out), self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().qcoh_device_free(self.ptr)
            self.ptr = vp()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _array_interface(data, shape=None, strides=None, offset=0):
    """(interface dict, on device) of a numpy array, a DeviceArray (explicit `shape`, `strides` in bytes or None for
    C-contiguous, `offset` in floats) or anything with __cuda_array_interface__ (e.g. a torch CUDA tensor or view)."""
    if isinstance(data, np.ndarray):
        if data.dtype != np.float32:
            raise TypeError("float32 arrays only")
        iface, cuda = dict(data.__array_interface__), False
    elif isinstance(data, DeviceArray):
        iface = {"data": [data.ptr.value + 4 * offset if data.ptr.value else 0, False], "shape": list(shape),
                 "strides": None if strides is None else list(strides), "typestr": "<f4", "version": 3}  # fmt: skip
        cuda = True
    else:
        iface, cuda = dict(data.__cuda_array_interface__), True
    iface["data"] = list(iface["data"])
    iface["shape"] = list(iface["shape"])
    if iface.get("strides") is not None:
        iface["strides"] = list(iface["strides"])
    return iface, cuda


def _columns_interface(cols, stream=None):
    """JSON list of the 1-D interfaces of `cols`: objects with __cuda_array_interface__ (e.g. torch CUDA tensors or views)
    or (DeviceArray, nrow, stride in bytes or None, offset in floats) tuples."""
    import json

    out = []
    for c in cols:
        if isinstance(c, tuple):
            dev, n, st, off = (tuple(c) + (None, 0))[:4]
            iface, _ = _array_interface(dev, shape=(n,), strides=None if st is None else (st,), offset=off)
        else:
            iface, _ = _array_interface(c)
        if stream is not None:
            iface["stream"] = stream
        out.append(iface)
    return json.dumps(out)


class DMatrix:
    def __init__(self, data: np.ndarray | None = None, missing=-999.0, *, handle=None):
        self.handle = vp()
        if handle is not None:
            self.handle = handle
            return
        data = np.ascontiguousarray(data, np.float32)
        assert data.ndim == 2
        # XGDMatrixCreateFromMat_f(data, nrow, ncol, missing, out)
        check(lib().XGDMatrixCreateFromMat(_ptr(data), data.shape[0], data.shape[1], missing, C.byref(self.handle)))

    @classmethod
    def device(cls, nrow, ncol, missing=-999.0):
        h = vp()
        check(lib().qcoh_dmatrix_create_device(nrow, ncol, missing, C.byref(h)))
        return cls(handle=h)

    @classmethod
    def from_array(cls, data, missing=float("nan"), *, shape=None, strides=None, offset=0, stream=None):
        """xgboost's DMatrix(array): a numpy float32 array through XGDMatrixCreateFromDense, a DeviceArray (explicit
        `shape`, `strides` in bytes, `offset` in floats) or anything with __cuda_array_interface__ (e.g. a torch CUDA
        tensor or a transposed view of one) through XGDMatrixCreateFromCudaArrayInterface, read in place with its
        strides.  `stream` adds a "stream" entry to a device array's interface."""
        import json

        iface, cuda = _array_interface(data, shape, strides, offset)
        if stream is not None:
            iface["stream"] = stream
        fn = lib().XGDMatrixCreateFromCudaArrayInterface if cuda else lib().XGDMatrixCreateFromDense
        h = vp()
        check(fn(json.dumps(iface).encode(), json.dumps({"missing": float(missing), "nthread": 0}).encode(), C.byref(h)))
        return cls(handle=h)

    @classmethod
    def from_columns(cls, cols, missing=float("nan"), *, stream=None):
        """xgboost's DMatrix(cuDF): one device column per feature (torch CUDA tensors or views, or (DeviceArray, nrow,
        stride in bytes, offset in floats) tuples) through XGDMatrixCreateFromCudaColumnar, each read in place."""
        import json

        h = vp()
        cfg = json.dumps({"missing": float(missing), "nthread": 0}).encode()
        check(lib().XGDMatrixCreateFromCudaColumnar(_columns_interface(cols, stream).encode(), cfg, C.byref(h)))
        return cls(handle=h)

    @classmethod
    def from_file(cls, path):
        h = vp()
        check(lib().XGDMatrixCreateFromFile(os.fsencode(path), 1, C.byref(h)))
        return cls(handle=h)

    def upload(self, rows: np.ndarray, row0=0):
        rows = np.ascontiguousarray(rows, np.float32)
        check(lib().qcoh_dmatrix_upload(self.handle, _ptr(rows), row0, rows.shape[0]))

    def seal(self):
        check(lib().qcoh_dmatrix_seal(self.handle))

    def save_binary(self, path):
        check(lib().XGDMatrixSaveBinary(self.handle, os.fsencode(path), 1))

    @property
    def num_row(self):
        v = u64()
        check(lib().XGDMatrixNumRow(self.handle, C.byref(v)))
        return v.value

    @property
    def num_col(self):
        v = u64()
        check(lib().XGDMatrixNumCol(self.handle, C.byref(v)))
        return v.value

    def free(self):
        if self.handle:
            check(lib().XGDMatrixFree(self.handle))
            self.handle = vp()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def expand_template(pattern: str, nymd: int, nhms: int = 0) -> str:
    """fill_grads_template for the XGBoostFile pattern (OH_GridCompMod.F90:1187, OH_instance_OH.rc:20)."""
    buf = C.create_string_buffer(4096)
    check(lib().qcoh_expand_template(os.fsencode(pattern), nymd, nhms, buf, C.c_size_t(len(buf))))
    return os.fsdecode(buf.value)


def import_name(field: str, data_source: int, use_inst_values: bool = False):
    """(import name, is_4d) feeding a boost-state field (OH_GridCompMod.F90:1326-1548)."""
    buf, four_d = C.create_string_buffer(64), C.c_int(0)
    check(lib().qcoh_import_name(field.encode(), data_source, int(use_inst_values), buf, len(buf), C.byref(four_d)))
    return buf.value.decode(), bool(four_d.value)


def model_cache_size() -> int:
    return int(lib().qcoh_model_cache_size())


def model_cache_clear() -> None:
    check(lib().qcoh_model_cache_clear())


class Booster:
    def __init__(self, model_file=None, *, parse_only=False, handle=None):
        self.handle = vp()
        self.owned = handle is None
        if handle is not None:
            self.handle = handle
            return
        check(lib().XGBoosterCreate(None, 0, C.byref(self.handle)))
        if model_file is not None:
            if parse_only:
                check(lib().qcoh_booster_parse(self.handle, os.fsencode(model_file)))
            else:
                check(lib().XGBoosterLoadModel(self.handle, os.fsencode(model_file)))

    def load_model(self, path):
        check(lib().XGBoosterLoadModel(self.handle, os.fsencode(path)))

    def save_model(self, path):
        check(lib().XGBoosterSaveModel(self.handle, os.fsencode(path)))

    def info(self) -> BoosterInfo:
        i = BoosterInfo()
        check(lib().qcoh_booster_get_info(self.handle, C.byref(i)))
        return i

    def flat(self):
        """(nodes_xy[n,2] uint32, tree_offset[T+1], tree_depth[T], orig_id[n]) copies."""
        i = self.info()
        pn, po = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint32)()
        pd, pi = C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
        check(lib().qcoh_booster_get_flat(self.handle, C.byref(pn), C.byref(po), C.byref(pd), C.byref(pi)))
        n, t = i.num_nodes, i.num_trees
        nodes = np.ctypeslib.as_array(pn, (n * 2,)).reshape(n, 2).copy() if n else np.zeros((0, 2), np.uint32)
        off = np.ctypeslib.as_array(po, (t + 1,)).copy()
        depth = np.ctypeslib.as_array(pd, (t,)).copy() if t else np.zeros(0, np.int32)
        orig = np.ctypeslib.as_array(pi, (n,)).copy() if n else np.zeros(0, np.int32)
        return nodes, off, depth, orig

    def duo(self):
        """(records[nslots,4] uint32, tree_slot[T], top_xy[T,16,2]) copies of the two-level record layout; raises
        if the booster does not qualify."""
        pr, ps, pt, n = C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint32)(), C.c_int64()
        check(lib().qcoh_booster_get_duo(self.handle, C.byref(pr), C.byref(ps), C.byref(pt), C.byref(n)))
        nt = self.info().num_trees
        rec = np.ctypeslib.as_array(pr, (n.value * 4,)).reshape(n.value, 4).copy()
        return rec, np.ctypeslib.as_array(ps, (nt,)).copy(), np.ctypeslib.as_array(pt, (nt * 32,)).reshape(nt, 16, 2).copy()

    def duo_info(self):
        """(blk_shift, has_default_bits) of the two-level records."""
        sh, dl = C.c_int(), C.c_int()
        check(lib().qcoh_booster_get_duo_info(self.handle, C.byref(sh), C.byref(dl)))
        return sh.value, bool(dl.value)

    def predict(self, dmat: DMatrix, option_mask=0, ntree_limit=0, training=0) -> np.ndarray:
        """XGBoosterPredict_f(handle, dmat, option_mask, ntree_limit, training, length, prediction).
        Returns a copy of the library-owned result."""
        n, p = u64(), f32p()
        check(lib().XGBoosterPredict(self.handle, dmat.handle, option_mask, ntree_limit, training, C.byref(n), C.byref(p)))
        out = np.ctypeslib.as_array(p, (n.value,)).copy() if n.value else np.zeros(0, np.float32)
        if option_mask & 2:
            nt = self.info().num_trees if ntree_limit == 0 else min(ntree_limit, self.info().num_trees)
            out = out.reshape(-1, nt) if nt else np.zeros((dmat.num_row, 0), np.float32)
        return out

    def predict_raw(self, dmat: DMatrix, option_mask=0, ntree_limit=0):
        """As predict(), but returns (length, borrowed pointer) without copying (bench)."""
        n, p = u64(), f32p()
        check(lib().XGBoosterPredict(self.handle, dmat.handle, option_mask, ntree_limit, 0, C.byref(n), C.byref(p)))
        return n.value, p

    def predict_device(self, dmat: DMatrix, out: DeviceArray, option_mask=0, ntree_limit=0, exp10=False, scale=1.0):
        epi = Epilogue(int(exp10), float(scale))
        check(lib().qcoh_booster_predict_device(self.handle, dmat.handle, option_mask, ntree_limit, C.byref(epi), out.ptr))

    def predict_from_dmatrix(self, dmat: DMatrix, config) -> np.ndarray:
        """XGBoosterPredictFromDMatrix(handle, dmat, config, shape, dim, result): `config` is a dict or a JSON string
        (type, training, iteration_begin, iteration_end, strict_shape).  Returns a copy shaped as the library says."""
        import json

        cfg = config if isinstance(config, str) else json.dumps(config)
        shp, dim, p = C.POINTER(u64)(), u64(), f32p()
        check(lib().XGBoosterPredictFromDMatrix(self.handle, None if dmat is None else dmat.handle, cfg.encode(), C.byref(shp), C.byref(dim), C.byref(p)))
        shape = tuple(int(shp[i]) for i in range(dim.value))
        n = int(np.prod(shape)) if shape else 0
        out = np.ctypeslib.as_array(p, (n,)).copy() if n else np.zeros(0, np.float32)
        return out.reshape(shape)

    def inplace_predict(self, data, missing=-999.0, type=0, iteration_end=0, strict_shape=False, *, shape=None,
                        strides=None, offset=0) -> np.ndarray:
        """xgboost's Booster.inplace_predict: value (type 0) or margin (1) straight from a dense float32 array, without a
        DMatrix.  A numpy array goes through XGBoosterPredictFromDense, a DeviceArray or anything with
        __cuda_array_interface__ (e.g. a torch CUDA tensor) through XGBoosterPredictFromCudaArray.  A DeviceArray takes
        an explicit `shape` (nrow, ncol), `strides` in bytes (None: C-contiguous) and `offset` in floats.  Returns a copy
        of the margins, shaped as the library says."""
        shape_, p, on_device = self.inplace_predict_raw(data, missing, type, iteration_end, strict_shape, shape=shape,
                                                        strides=strides, offset=offset)  # fmt: skip
        n = int(np.prod(shape_))
        out = np.empty(n, np.float32)
        if n and on_device:
            check(lib().qcoh_memcpy_d2h(_ptr(out), C.cast(p, vp), out.nbytes))
        elif n:
            out[:] = np.ctypeslib.as_array(p, (n,))
        return out.reshape(shape_)

    def inplace_predict_raw(self, data, missing=-999.0, type=0, iteration_end=0, strict_shape=False, *, shape=None,
                            strides=None, offset=0, stream=None):
        """As inplace_predict(), but returns (shape, borrowed result pointer, whether it points at device memory)
        without copying; `stream` adds a "stream" entry to the interface of a device array."""
        import json

        if isinstance(data, np.ndarray) and data.dtype != np.float32:
            raise TypeError("inplace_predict takes float32 arrays")
        iface, cuda = _array_interface(data, shape, strides, offset)
        if stream is not None:
            iface["stream"] = stream
        cfg = {"type": int(type), "training": False, "missing": float(missing), "iteration_begin": 0,
               "iteration_end": int(iteration_end), "strict_shape": bool(strict_shape)}  # fmt: skip
        shp, dim, p = C.POINTER(u64)(), u64(), f32p()
        fn = lib().XGBoosterPredictFromCudaArray if cuda else lib().XGBoosterPredictFromDense
        check(fn(self.handle, json.dumps(iface).encode(), json.dumps(cfg).encode(), None, C.byref(shp), C.byref(dim), C.byref(p)))
        return tuple(int(shp[i]) for i in range(dim.value)), p, cuda

    def inplace_predict_columns(self, cols, missing=-999.0, type=0, iteration_end=0, strict_shape=False, *,
                                stream=None) -> np.ndarray:  # fmt: skip
        """xgboost's Booster.inplace_predict(cuDF): value (type 0) or margin (1) straight from one device column per
        feature (as DMatrix.from_columns takes them) through XGBoosterPredictFromCudaColumnar.  Returns a copy of the
        margins, shaped as the library says."""
        import json

        cfg = {"type": int(type), "training": False, "missing": float(missing), "iteration_begin": 0,
               "iteration_end": int(iteration_end), "strict_shape": bool(strict_shape)}  # fmt: skip
        shp, dim, p = C.POINTER(u64)(), u64(), f32p()
        check(lib().XGBoosterPredictFromCudaColumnar(self.handle, _columns_interface(cols, stream).encode(), json.dumps(cfg).encode(),
                                                     None, C.byref(shp), C.byref(dim), C.byref(p)))  # fmt: skip
        shape_ = tuple(int(shp[i]) for i in range(dim.value))
        n = int(np.prod(shape_))
        out = np.empty(n, np.float32)
        if n:
            check(lib().qcoh_memcpy_d2h(_ptr(out), C.cast(p, vp), out.nbytes))
        return out.reshape(shape_)

    def predict_contribs(self, dmat: DMatrix, approximate=False, ntree_limit=0) -> np.ndarray:
        """[nrow, num_feature + 1] per-feature contributions, last column the bias: exact TreeSHAP, or Saabas when
        `approximate` (XGBoosterPredictFromDMatrix type 2 / 3, iteration_end = ntree_limit)."""
        cfg = {"type": 3 if approximate else 2, "training": False, "iteration_begin": 0,
               "iteration_end": int(ntree_limit), "strict_shape": False}  # fmt: skip
        return self.predict_from_dmatrix(dmat, cfg)

    def predict_contribs_device(self, dmat: DMatrix, out: DeviceArray, approximate=False, ntree_limit=0):
        """qcoh_booster_predict_contribs_device: the same into a device buffer of nrow * (num_feature + 1) floats,
        asynchronous on the library stream."""
        check(lib().qcoh_booster_predict_contribs_device(self.handle, dmat.handle, int(approximate), ntree_limit, out.ptr))

    def predict_interactions(self, dmat: DMatrix, approximate=False, ntree_limit=0) -> np.ndarray:
        """[nrow, num_feature + 1, num_feature + 1] SHAP interaction values (libxgboost's pred_interactions, type 4 /
        5): M[i][j] is the part of feature i's contribution shared with feature j, index num_feature the bias; each row
        of M sums to the contribution, the whole matrix to the margin."""
        nc = self.info().num_feature + 1
        nrow = dmat.num_row
        out = DeviceArray(nrow * nc * nc)
        try:
            self.predict_interactions_device(dmat, out, approximate, ntree_limit)
            synchronize()
            return out.get().reshape(nrow, nc, nc)
        finally:
            out.free()

    def predict_interactions_device(self, dmat: DMatrix | None, out: DeviceArray | None, approximate=False, ntree_limit=0):
        """qcoh_booster_predict_interactions_device: the same into a device buffer of nrow * (num_feature + 1)**2
        floats, asynchronous on the library stream."""
        check(lib().qcoh_booster_predict_interactions_device(self.handle, None if dmat is None else dmat.handle,
                                                             int(approximate), ntree_limit, None if out is None else out.ptr))  # fmt: skip

    def shap_paths(self):
        """(bins[nbins,32,4] uint32, tree_bin[T+1] int64, node_mean[num_nodes] float32) copies of the contribution
        tables (host only; raises when the booster has no covers)."""
        pb, pt, pm, nb = C.POINTER(C.c_uint32)(), C.POINTER(C.c_int64)(), C.POINTER(C.c_float)(), C.c_int64()
        check(lib().qcoh_booster_get_shap_paths(self.handle, C.byref(pb), C.byref(pt), C.byref(pm), C.byref(nb)))
        i = self.info()
        bins = np.ctypeslib.as_array(pb, (nb.value * 128,)).reshape(nb.value, 32, 4).copy() if nb.value else np.zeros((0, 32, 4), np.uint32)
        tree_bin = np.ctypeslib.as_array(pt, (i.num_trees + 1,)).copy()
        mean = np.ctypeslib.as_array(pm, (i.num_nodes,)).copy() if i.num_nodes else np.zeros(0, np.float32)
        return bins, tree_bin, mean

    @classmethod
    def cached(cls, model_file):
        """The process-wide cache's booster for this file (loaded on first request); owned by the cache."""
        h = vp()
        check(lib().qcoh_model_cache_get(os.fsencode(model_file), C.byref(h)))
        return cls(handle=h)

    def free(self):
        if self.handle and self.owned:
            check(lib().XGBoosterFree(self.handle))
        self.handle = vp()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def node_visits_per_cell(booster: "Booster", x_sample: np.ndarray) -> float:
    """Mean number of node fetches per row (sum over trees of leaf depth + 1), from the device's own per-tree
    leaf ids on a sample of rows and the flattened (depth-ordered) layout."""
    leaf = booster.predict(DMatrix(x_sample), option_mask=2).astype(np.int64)
    nodes, off, _, orig = booster.flat()
    visits = 0.0
    for t in range(len(off) - 1):
        n0, n1 = int(off[t]), int(off[t + 1])
        rel = (nodes[n0:n1, 1] & ((1 << 23) - 1)).astype(np.int64)
        dep = np.zeros(n1 - n0, np.int32)
        for i in np.nonzero(rel)[0]:  # breadth-first order: parents come before their children
            dep[i + rel[i]] = dep[i] + 1
            dep[i + rel[i] + 1] = dep[i] + 1
        lut = np.empty(n1 - n0, np.int64)
        lut[orig[n0:n1]] = np.arange(n1 - n0)
        visits += float(dep[lut[leaf[:, t]]].mean()) + 1.0
    return visits


def synchronize():
    check(lib().qcoh_device_synchronize())


def timer_start():
    check(lib().qcoh_timer_start())


def timer_stop() -> float:
    ms = C.c_float()
    check(lib().qcoh_timer_stop(C.byref(ms)))
    return ms.value


def flush_l2():
    check(lib().qcoh_flush_l2())


class OhRun1:
    """Fused device-resident Run1 (qcoh_oh_*): the call a patched OH_GridCompMod Run1 makes."""

    def __init__(self, booster: Booster, ncol, km, consts, *, ohscale=0.85, compute_once_per_day=True,
                 tropp_min=4000.0, missing=-999.0):  # fmt: skip
        self.booster = booster
        self.ncol, self.km = ncol, km
        cfg = OhConfig(ncol, km, consts["EPSILON"], consts["AVOGAD"], consts["RUNIV"], consts["RADIANS_TO_DEGREES"],
                       consts["DEGREES_TO_RADIANS"], ohscale, int(compute_once_per_day), tropp_min, missing)  # fmt: skip
        self.handle = vp()
        check(lib().qcoh_oh_create(booster.handle, C.byref(cfg), C.byref(self.handle)))
        self._keep = []

    @staticmethod
    def _addr(a):
        if a is None:
            return None
        if isinstance(a, DeviceArray):
            return a.ptr
        return a.ctypes.data_as(vp)

    def make_in(self, fields: dict, nymd=20220701, need_to_call_boost=True, mod_fields: dict | None = None,
                area=None) -> Run1In:  # fmt: skip
        """Bind a synth.raw_fields-style dict (ONLINE_INST aliasing: the model-state T/Q/PLE are the
        boost-state ones unless `mod_fields` overrides them).  Values: numpy arrays or DeviceArrays."""
        mod = mod_fields or fields
        i = Run1In()
        i.nymd, i.need_to_call_boost = nymd, int(need_to_call_boost)
        A = self._addr
        i.T_MOD, i.Q_MOD, i.PLE_MOD, i.TROPP = A(mod["T"]), A(mod["Q"]), A(mod["PLE"]), A(mod["TROPP"])
        i.T_BST, i.Q_BST, i.PLE_BST, i.ZLE_BST = A(fields["T"]), A(fields["Q"]), A(fields["PLE"]), A(fields["ZLE"])
        for k in ("TAUCLW", "TAUCLI", "FCLD", "CH4", "CO"):
            setattr(i, k, A(fields[k]))
        for s, sp in enumerate(("BC", "OC", "BR", "DU", "SU", "SS", "NI")):
            i.SCA[s] = A(fields[sp + "SCACOEF"])
        for g_ in ("NO2", "O3", "ISOP", "ACET", "C2H6", "C3H8", "PRPE", "ALK4", "MP", "H2O2", "CH2O", "GMITO3",
                   "GMITTO3", "ALBUV"):  # fmt: skip
            setattr(i, g_, A(fields["oh_" + g_]))
        i.LATS, i.LONS, i.OH_CLIM = A(fields["LATS"]), A(fields["LONS"]), A(fields["oh_OH"])
        i.AREA = A(area)
        self._keep = [fields, mod, area]
        return i

    def run(self, rin: Run1In, *, want=("OH", "OH_boost", "NDWET"), device_out: dict | None = None) -> dict:
        km, ncol = self.km, self.ncol
        o = Run1Out()
        res = {}
        for name in ("OH", "OH_boost", "NDWET", "LOSS_CH4", "LOSS_CO"):
            if device_out and name in device_out:
                setattr(o, name, device_out[name].ptr)
            elif name in want or name == "OH":
                res[name] = np.empty((km, ncol), np.float32)
                setattr(o, name, _ptr(res[name]))
        if "X" in want:
            res["X"] = np.empty((km * ncol, 27), np.float32)
            o.X = _ptr(res["X"])
        if "pred" in want:
            res["pred"] = np.empty(km * ncol, np.float32)
            o.pred = _ptr(res["pred"])
        check(lib().qcoh_oh_run1(self.handle, C.byref(rin), C.byref(o)))
        res["k1"] = o.k1
        if o.k1 > 0:
            n = (km - o.k1 + 1) * ncol
            if "X" in res:
                res["X"] = res["X"][:n]
            if "pred" in res:
                res["pred"] = res["pred"][:n]
        res["diag"] = np.array(list(o.diag))
        return res

    def set_booster(self, booster: Booster) -> None:
        check(lib().qcoh_oh_set_booster(self.handle, booster.handle))
        self.booster = booster

    def select_model(self, pattern: str, nymd: int, nhms: int = 0) -> bool:
        """Opt-in month roll-over (SURVEY.md 0.5): switch to the cached booster of the expanded file name."""
        ch = C.c_int(0)
        check(lib().qcoh_oh_select_model(self.handle, os.fsencode(pattern), nymd, nhms, C.byref(ch)))
        return bool(ch.value)

    def get_diag(self, name: str) -> np.ndarray:
        """DIAG_<name> export of the last boost step (OH_StateSpecs.rc:41-73)."""
        two_d = name in ("LAT", "SZA", "stratO3")
        out = np.empty(self.ncol if two_d else (self.km, self.ncol), np.float32)
        check(lib().qcoh_oh_get_diag(self.handle, name.encode(), _ptr(out)))
        return out

    def free(self):
        if self.handle:
            check(lib().qcoh_oh_free(self.handle))
            self.handle = vp()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def predict_OH_with_XGB(xgb_fname, icount, jcount, kcount, dynamic_k_range, tropp_min, pl, tropp, bb, OH_ML):
    """Host mirror of the reference subroutine (OH_GridCompMod.F90:123-398), same argument order.
    `bb` is the list of 27 arrays in OH_BOOST_INPUT_DATA order; 2-D members have ndim == 1 here
    (flattened (i,j)).  OH_ML is updated in place.  Returns rc."""
    arrs = [np.ascontiguousarray(a, np.float32) for a in bb]
    ptrs = (vp * 27)(*[_ptr(a) for a in arrs])
    is2d = (C.c_int * 27)(*[int(f in (0, 21, 22, 26)) for f in range(27)])  # LAT, GMISTRATO3, ALBUV, SZA
    pl = np.ascontiguousarray(pl, np.float32)
    tropp = np.ascontiguousarray(tropp, np.float32)
    assert OH_ML.dtype == np.float32 and OH_ML.flags.c_contiguous
    return lib().qcoh_predict_OH_with_XGB(os.fsencode(xgb_fname), icount, jcount, kcount, int(dynamic_k_range),
                                          tropp_min, _ptr(pl), _ptr(tropp), ptrs, is2d, _ptr(OH_ML))  # fmt: skip
