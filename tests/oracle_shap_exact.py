"""Exact TreeSHAP contributions and SHAP interaction values in extended precision, for the tests (TEST INFRASTRUCTURE
ONLY; parity unpinned, like oracle/).

`contributions` / `interactions` bind tests/oracle_shap_exact.c: per path, the Shapley values of its product game from
the coefficients of the product polynomial, in long double, on the model and DMatrix the C oracle (oracle/cpu.py)
loads and builds.  Each value comes with its magnitude A (what a relative perturbation of the path's fractions and
weights can move it by), so that a comparison can be held to a bar per entry.  `exact_z=False` uses the zero fractions
the library's path tables hold, (float) of the float64 product of cover ratios; `exact_z=True` the product itself.
Compiled on first use into a temporary directory of this process, so a read-only checkout works.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle_contribs import OracleContribsError

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None

assert np.finfo(np.longdouble).nmant >= 63, "the reference needs the x87 80-bit long double"


def build():
    """Compile and load the C reference (once per process)."""
    global _LIB
    if _LIB is None:
        from oracle import cpu

        cpu.lib()  # the oracle proper (model loader, DMatrix) is loaded first
        tmp = tempfile.mkdtemp(prefix="oracle_shap_exact_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "liboracle_shap_exact.so")
        cflags = ["-O3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-Wall", "-Wextra", "-std=gnu11"]
        subprocess.check_call(["gcc", *cflags, "-shared", "-I", _ORACLE, "-o", so,
                               os.path.join(_HERE, "oracle_shap_exact.c"), "-lm"])  # fmt: skip
        L = C.CDLL(so)
        L.se_last_error.restype = C.c_char_p
        ld = np.ctypeslib.ndpointer(np.longdouble, flags="C_CONTIGUOUS")
        L.se_shap.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_int, C.c_int, ld, ld, C.POINTER(C.c_int)]
        _LIB = L
    return _LIB


def _run(model, x, missing, ntree_limit, exact_z, interactions):
    from oracle import cpu

    L = build()
    x = np.ascontiguousarray(x, np.float32)
    nrow, ncol = x.shape
    nc = model.num_feature + 1
    shape = (nrow, nc, nc) if interactions else (nrow, nc)
    d = cpu.lib().orc_dmatrix_from_mat(x.ctypes.data_as(C.POINTER(C.c_float)), nrow, ncol, missing)
    if not d:
        raise OracleContribsError(cpu.lib().orc_last_error().decode())
    try:
        val, mag, dmax = np.empty(shape, np.longdouble), np.empty(shape, np.longdouble), C.c_int(0)
        if L.se_shap(C.cast(model._m, C.c_void_p), C.cast(d, C.c_void_p), ntree_limit, int(exact_z), int(interactions),
                     val, mag, C.byref(dmax)) != 0:  # fmt: skip
            raise OracleContribsError(L.se_last_error().decode())
    finally:
        cpu.lib().orc_dmatrix_free(d)
    return val, mag, dmax.value


def contributions(model, x, missing=-999.0, ntree_limit=0, exact_z=False):
    """(phi, A, D_max): phi [nrow, num_feature + 1] long double, last column the float32 bias; A the magnitude of each
    entry (0 for the bias); D_max the most distinct features on one path of the trees used."""
    return _run(model, x, missing, ntree_limit, exact_z, False)


def interactions(model, x, missing=-999.0, ntree_limit=0, exact_z=False):
    """(M, A, D_max): M [nrow, num_feature + 1, num_feature + 1] long double SHAP interaction values, M[F][F] the float32
    bias; A the magnitude of each entry."""
    return _run(model, x, missing, ntree_limit, exact_z, True)
