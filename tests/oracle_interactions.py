"""SHAP interaction values restated for the tests (TEST INFRASTRUCTURE ONLY; parity unpinned, like oracle/):

* `predict_interactions`: libxgboost 1.6.0's PredictInteractionContributions in C (tests/oracle_interactions.c: the
  conditioned recursive TreeShap on top of tests/oracle_contribs.c, in float32), run on the model and DMatrix the C
  oracle (oracle/cpu.py) loads and builds.  Compiled on first use into a temporary directory of this process, so a
  read-only checkout works.
* `shapley_interactions_brute_force`: the Shapley interaction index straight from its definition (the independent pin
  of the conditioned TreeShap: it needs only the definition), on the v(S) of oracle_contribs.shapley_brute_force.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle_contribs import OracleContribsError, shapley_brute_force

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None


def build():
    """Compile and load the C restatement (once per process)."""
    global _LIB
    if _LIB is None:
        from oracle import cpu

        cpu.lib()  # the oracle proper (model loader, DMatrix) is loaded first
        tmp = tempfile.mkdtemp(prefix="oracle_interactions_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "liboracle_interactions.so")
        cflags = ["-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-Wall", "-Wextra",
                  "-std=gnu11"]  # fmt: skip
        subprocess.check_call(["gcc", *cflags, "-shared", "-I", _ORACLE, "-o", so,
                               os.path.join(_HERE, "oracle_interactions.c"), "-lm"])  # fmt: skip
        L = C.CDLL(so)
        L.oc_last_error.restype = C.c_char_p
        L.oc_predict_interactions.restype = C.c_uint64
        L.oc_predict_interactions.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.POINTER(C.c_float)]
        _LIB = L
    return _LIB


def predict_interactions(model, x, missing=-999.0, approximate=False, ntree_limit=0) -> np.ndarray:
    """[nrow, num_feature + 1, num_feature + 1] float32 SHAP interaction values of an oracle.cpu.Model (libxgboost's
    loop over conditioned TreeShap; approximate passes the flag through, which makes on == off), index num_feature
    the bias.  About 2 (num_feature + 1) + 1 TreeShap passes per row: keep the rows few on deep boosters."""
    from oracle import cpu

    L = build()
    x = np.ascontiguousarray(x, np.float32)
    nrow, ncol = x.shape
    nc = model.num_feature + 1
    d = cpu.lib().orc_dmatrix_from_mat(x.ctypes.data_as(C.POINTER(C.c_float)), nrow, ncol, missing)
    if not d:
        raise OracleContribsError(cpu.lib().orc_last_error().decode())
    try:
        out = np.empty((nrow, nc, nc), np.float32)
        n = L.oc_predict_interactions(C.cast(model._m, C.c_void_p), C.cast(d, C.c_void_p), int(approximate), ntree_limit,
                                      out.ctypes.data_as(C.POINTER(C.c_float)))  # fmt: skip
        if n != out.size and out.size:
            raise OracleContribsError(L.oc_last_error().decode())
    finally:
        cpu.lib().orc_dmatrix_free(d)
    return out


def _coalition_values(forest, x, missing, ntree_limit):
    """(the features the forest splits on, v[mask, row]): the path-dependent v(S) of shapley_brute_force — base_score
    plus, per tree, the expectation that follows x at a split on a feature in S (the default child when the entry is
    missing) and weighs both children by cover(child) / cover(node) otherwise — for every subset S of those features,
    bit i of mask standing for the i-th of them."""
    x = np.asarray(x, np.float32)
    miss = np.isnan(x) | (x == np.float32(missing))
    nrow, ncol = x.shape
    nt = len(forest.trees) if ntree_limit == 0 else min(ntree_limit, len(forest.trees))
    trees = forest.trees[:nt]
    used = sorted({int(f) for t in trees for f in np.asarray(t.split_index)[np.asarray(t.left) != -1]})
    pos = {f: i for i, f in enumerate(used)}

    def expect(t, n, mask):
        if t.left[n] == -1:
            return np.full(nrow, float(t.split_cond[n]))
        l, r, f = int(t.left[n]), int(t.right[n]), int(t.split_index[n])
        el, er = expect(t, l, mask), expect(t, r, mask)
        if (mask >> pos[f]) & 1:
            if f < ncol:
                with np.errstate(invalid="ignore"):
                    go_left = np.where(miss[:, f], bool(t.default_left[n]), x[:, f] < np.float32(t.split_cond[n]))
            else:
                go_left = np.full(nrow, bool(t.default_left[n]))
            return np.where(go_left, el, er)
        c = np.asarray(t.sum_hess, np.float64)
        return (c[l] * el + c[r] * er) / c[n]

    v = np.zeros((1 << len(used), nrow))
    for mask in range(1 << len(used)):
        v[mask] = float(np.float32(forest.base_score)) + sum(expect(t, 0, mask) for t in trees)
    return used, v


def shapley_interactions_brute_force(forest, x, missing=-999.0, ntree_limit=0) -> np.ndarray:
    """SHAP interaction values straight from the definition of the Shapley interaction index, float64: for i != j,
        Phi_ij = sum over S in N minus {i, j} of |S|! (M - |S| - 2)! / (2 (M - 1)!) [v(S+ij) - v(S+i) - v(S+j) + v(S)],
    Phi_ii = phi_i - sum_{j != i} Phi_ij (phi from shapley_brute_force), and the bias entry v({}).
    [nrow, num_feature + 1, num_feature + 1].  Exponential in the number of features used: keep it below ~12."""
    from math import factorial

    used, v = _coalition_values(forest, x, missing, ntree_limit)
    M, nrow, nf = len(used), v.shape[1], forest.num_feature
    phi = shapley_brute_force(forest, x, missing, ntree_limit)
    out = np.zeros((nrow, nf + 1, nf + 1))
    for a, fi in enumerate(used):
        for b, fj in enumerate(used):
            if a == b:
                continue
            for mask in range(1 << M):
                if (mask >> a) & 1 or (mask >> b) & 1:
                    continue
                s = bin(mask).count("1")
                w = factorial(s) * factorial(M - s - 2) / (2 * factorial(M - 1))
                ia, ib = 1 << a, 1 << b
                out[:, fi, fj] += w * (v[mask | ia | ib] - v[mask | ia] - v[mask | ib] + v[mask])
        out[:, fi, fi] = phi[:, fi] - out[:, fi, :nf].sum(axis=1)
    out[:, nf, nf] = v[0]
    return out
