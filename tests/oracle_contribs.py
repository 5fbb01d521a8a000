"""Per-feature contributions restated for the tests (TEST INFRASTRUCTURE ONLY; parity unpinned, like oracle/):

* `predict_contribs`: libxgboost 1.6.0's PredictContribution in C (tests/oracle_contribs.c: recursive TreeShap and
  CalculateContributionsApprox in float32), run on the model and DMatrix the C oracle (oracle/cpu.py) loads and builds.
  The library is compiled on first use into a temporary directory of this process, so a read-only checkout works.
* `node_means`, `saabas`, `shapley_brute_force`: deliberately naive numpy restatements — the Saabas walk, and Shapley
  values straight from their definition (the independent pin of TreeSHAP: it needs only the definition).
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None


def build():
    """Compile and load the C restatement (once per process)."""
    global _LIB
    if _LIB is None:
        from oracle import cpu

        cpu.lib()  # the oracle proper (model loader, DMatrix) is loaded first
        tmp = tempfile.mkdtemp(prefix="oracle_contribs_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "liboracle_contribs.so")
        cflags = ["-O3", "-march=native", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-Wall", "-Wextra",
                  "-std=gnu11"]  # fmt: skip
        subprocess.check_call(["gcc", *cflags, "-shared", "-I", _ORACLE, "-o", so, os.path.join(_HERE, "oracle_contribs.c"),
                               "-lm"])  # fmt: skip
        L = C.CDLL(so)
        L.oc_last_error.restype = C.c_char_p
        L.oc_predict_contribs.restype = C.c_uint64
        L.oc_predict_contribs.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint, C.POINTER(C.c_float)]
        _LIB = L
    return _LIB


class OracleContribsError(RuntimeError):
    pass


def predict_contribs(model, x, missing=-999.0, approximate=False, ntree_limit=0) -> np.ndarray:
    """[nrow, num_feature + 1] float32 contributions of an oracle.cpu.Model (exact recursive TreeShap, or approximate),
    last column the bias."""
    from oracle import cpu

    L = build()
    x = np.ascontiguousarray(x, np.float32)
    nrow, ncol = x.shape
    d = cpu.lib().orc_dmatrix_from_mat(x.ctypes.data_as(C.POINTER(C.c_float)), nrow, ncol, missing)
    if not d:
        raise OracleContribsError(cpu.lib().orc_last_error().decode())
    try:
        out = np.empty((nrow, model.num_feature + 1), np.float32)
        n = L.oc_predict_contribs(C.cast(model._m, C.c_void_p), C.cast(d, C.c_void_p), int(approximate), ntree_limit,
                                  out.ctypes.data_as(C.POINTER(C.c_float)))  # fmt: skip
        if n != out.size and out.size:
            raise OracleContribsError(L.oc_last_error().decode())
    finally:
        cpu.lib().orc_dmatrix_free(d)
    return out


def _missing(x, missing):
    x = np.asarray(x, np.float32)
    return x, np.isnan(x) | (x == np.float32(missing))


# These take an in-memory forest with covers (quickchem_b200.xgbmodel.Forest, or anything with `trees` whose members
# carry left / right / split_index / split_cond / default_left / sum_hess, `base_score` and `num_feature`).
def node_means(tree) -> np.ndarray:
    """libxgboost 1.6.0 FillNodeMeanValue in float32: mean(n) = (mean(l) * cover(l) + mean(r) * cover(r)) / cover(n)."""
    cov = np.asarray(tree.sum_hess, np.float32)
    mean = np.zeros(len(tree.left), np.float32)

    def fill(n):
        if tree.left[n] == -1:
            mean[n] = np.float32(tree.split_cond[n])
        else:
            l, r = int(tree.left[n]), int(tree.right[n])
            a = np.float32(fill(l) * cov[l])
            a = np.float32(a + np.float32(fill(r) * cov[r]))
            mean[n] = np.float32(a / cov[n])
        return mean[n]

    fill(0)
    return mean


def saabas(forest, x, missing=-999.0, ntree_limit=0) -> np.ndarray:
    """Approximate contributions (CalculateContributionsApprox), float32 in libxgboost's order: per tree a zeroed
    vector gets mean(root) on the bias and mean(next) - mean(node) on each split feature of the row's path (plus
    leaf - mean(leaf) at the end), and is added into the row; base_score goes to the bias last."""
    x, miss = _missing(x, missing)
    nrow, ncol = x.shape
    nf = forest.num_feature
    nt = len(forest.trees) if ntree_limit == 0 else min(ntree_limit, len(forest.trees))
    out = np.zeros((nrow, nf + 1), np.float32)
    ar = np.arange(nrow)
    for t in forest.trees[:nt]:
        mean = node_means(t)
        left, right = np.asarray(t.left, np.int64), np.asarray(t.right, np.int64)
        sidx, cond = np.asarray(t.split_index, np.int64), np.asarray(t.split_cond, np.float32)
        tc = np.zeros((nrow, nf + 1), np.float32)
        tc[:, nf] += mean[0]
        nid = np.zeros(nrow, np.int64)
        node_value = np.full(nrow, mean[0], np.float32)
        last = np.zeros(nrow, np.int64)
        while True:
            act = np.nonzero(left[nid] != -1)[0]
            if act.size == 0:
                break
            n = nid[act]
            f = sidx[n]
            fin = np.minimum(f, ncol - 1)
            is_miss = miss[act, fin] | (f >= ncol)
            with np.errstate(invalid="ignore"):
                go_right = np.where(is_miss, np.asarray(t.default_left, np.int64)[n] == 0, ~(x[act, fin] < cond[n]))
            nxt = left[n] + go_right.astype(np.int64)
            new = mean[nxt]
            tc[act, f] = tc[act, f] + (new - node_value[act])
            node_value[act], last[act], nid[act] = new, f, nxt
        deep = left[0] != -1
        if deep:
            tc[ar, last] = tc[ar, last] + (cond[nid] - node_value)
        out += tc
    out[:, nf] += np.float32(forest.base_score)
    return out


def shapley_brute_force(forest, x, missing=-999.0, ntree_limit=0) -> np.ndarray:
    """Exact Shapley values straight from the definition, float64: over every subset S of the features the forest
    splits on, v(S) = base_score + sum_t E_t[f | x_S], where the expectation follows x at a split on a feature in S
    (the default child when the entry is missing) and weighs both children by cover(child) / cover(node) otherwise.
    [nrow, num_feature + 1], last column v({}).  Exponential in the number of features used: keep it below ~12."""
    from math import factorial

    x, miss = _missing(x, missing)
    nrow, ncol = x.shape
    nf = forest.num_feature
    nt = len(forest.trees) if ntree_limit == 0 else min(ntree_limit, len(forest.trees))
    trees = forest.trees[:nt]
    used = sorted({int(f) for t in trees for f in np.asarray(t.split_index)[np.asarray(t.left) != -1]})
    M = len(used)
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

    v = np.zeros((1 << M, nrow))
    for mask in range(1 << M):
        v[mask] = float(np.float32(forest.base_score)) + sum(expect(t, 0, mask) for t in trees)
    out = np.zeros((nrow, nf + 1))
    for i, f in enumerate(used):
        for mask in range(1 << M):
            if (mask >> i) & 1:
                continue
            s = bin(mask).count("1")
            w = factorial(s) * factorial(M - s - 1) / factorial(M)
            out[:, f] += w * (v[mask | (1 << i)] - v[mask])
    out[:, nf] = v[0]
    return out
