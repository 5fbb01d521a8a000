"""The extended-precision SHAP reference (tests/oracle_shap_exact.c) pinned without a GPU: against the Shapley values and
the Shapley interaction index from their definitions, against exact rational arithmetic on the edge boosters, against
the float32 oracle, and its bias bit for bit.  Also the library's refusal of a zero fraction that float32 cannot hold."""
from fractions import Fraction
from math import factorial

import numpy as np
import pytest

import oracle_contribs as oc
import oracle_interactions as oi
import oracle_shap_exact as se
import shap_edge_forests as ef
from contribs_forests import NF, assert_shap_close, few_feature_forest, on_thresholds, sklearn_forest, with_missing
from interactions_forests import assert_interactions_close
from quickchem_b200 import synth, xgbmodel


def _model(oracle, forest, tmp_path, name):
    p = str(tmp_path / f"{name}.model")
    xgbmodel.write_legacy_binary(forest, p)
    return oracle.Model(p), p


def _grown(case):
    rng = np.random.default_rng(7)
    if case == "sklearn":
        f, x = sklearn_forest([1, 2, 4, 18, 20, 22], n_trees=4, max_depth=6)
    else:
        i = int(case[-1])
        cols, nt, d = (([2, 4, 20], 3, 4), ([0, 1, 2, 5, 15, 26], 6, 6), ([3, 7, 11, 19, 23, 24, 25, 26], 4, 9))[i]
        f, x = few_feature_forest(cols, nt, d, seed=20 + i), synth.quick_features(synth.raw_fields(6, seed=40 + i))
    return f, with_missing(on_thresholds(x[:200], f, rng), rng)


def _within(got, ref, mag, rel, what):
    """|got - ref| <= rel * A entry by entry (long double); returns the worst |got - ref| / A."""
    err = np.abs(np.asarray(got, np.longdouble) - ref)
    bad = err > rel * mag
    assert not bad.any(), f"{what}: {int(bad.sum())} entries off, first at {np.argwhere(bad)[0]}"
    return float((err / np.maximum(mag, np.longdouble(1e-300))).max())


@pytest.mark.parametrize("case", ["grown0", "grown1", "grown2", "sklearn"])
def test_reference_is_the_brute_force_definition(oracle, tmp_path, case):
    """With the exact zero fractions the reference is the Shapley value / interaction index of the path-dependent
    coalition game, computed here from its definition in float64, within 1e-12 of each entry's magnitude."""
    forest, x = _grown(case)
    m, _ = _model(oracle, forest, tmp_path, case)
    for ntree in (0, 2):
        phi, mag, _ = se.contributions(m, x, ntree_limit=ntree, exact_z=True)
        bf = oc.shapley_brute_force(forest, x, ntree_limit=ntree)
        _within(bf[:, :NF], phi[:, :NF], mag[:, :NF], 1e-12, case)
        xi = x[:40]
        M, magm, _ = se.interactions(m, xi, ntree_limit=ntree, exact_z=True)
        bfi = oi.shapley_interactions_brute_force(forest, xi, ntree_limit=ntree)
        _within(bfi[:, :NF, :NF], M[:, :NF, :NF], magm[:, :NF, :NF], 1e-12, case)
        assert np.all(M[:, NF, :NF] == 0) and np.all(M[:, :NF, NF] == 0)
        # rows of M sum to phi
        _within(M[:, :NF, :NF].sum(axis=2), phi[:40, :NF], mag[:40, :NF] + magm[:, :NF, :NF].sum(axis=2), 2.0**-60, case)


# ---- exact rational arithmetic ----------------------------------------------------------------------------------
def _rational_paths(forest, ntree):
    """Per path: (leaf value, [(feature, [(threshold, right)], missing flag, z~, z)]) with z~ / z Fractions."""
    out = []
    for t in forest.trees[:ntree]:
        cov = [float(c) for c in np.asarray(t.sum_hess, np.float32)]

        def walk(n, route):
            if t.left[n] == -1:
                elems = {}
                for nd, right in route:
                    f = int(t.split_index[nd])
                    child = int(t.right[nd] if right else t.left[nd])
                    e = elems.setdefault(f, {"splits": [], "miss": True, "zd": 1.0, "z": Fraction(1)})
                    e["splits"].append((float(t.split_cond[nd]), right))
                    e["miss"] &= bool(t.default_left[nd]) == (not right)
                    e["zd"] *= cov[child] / cov[nd]  # float64, root to leaf, as the tables multiply
                    e["z"] *= Fraction(cov[child]) / Fraction(cov[nd])
                with np.errstate(over="ignore"):
                    zt = {f: np.float32(e["zd"]) for f, e in elems.items()}  # +inf in the overflow booster
                out.append((Fraction(float(t.split_cond[n])),
                            [(f, e["splits"], e["miss"], Fraction(float(zt[f])) if np.isfinite(zt[f]) else None, e["z"])
                             for f, e in elems.items()]))  # fmt: skip
                return
            walk(int(t.left[n]), route + [(n, False)])
            walk(int(t.right[n]), route + [(n, True)])

        walk(0, [])
    return out


def _one(row, f, splits, miss):
    v = row[f] if f < len(row) else np.float32(np.nan)
    if np.isnan(v) or v == np.float32(-999.0):
        return Fraction(int(miss))
    return Fraction(int(all((v < np.float32(thr)) != right for thr, right in splits)))


def _weights(o, z):
    """W_e = sum_k k! (D-1-k)! / D! c_k, c the coefficients of prod_{j != e}(z_j + o_j t), exactly."""
    D = len(o)
    W = []
    for e in range(D):
        c = [Fraction(1)]
        for j in range(D):
            if j != e:
                c = [(c[k] if k < len(c) else 0) * z[j] + (c[k - 1] * o[j] if k else 0) for k in range(len(c) + 1)]
        W.append(sum(Fraction(factorial(k) * factorial(D - 1 - k), factorial(D)) * ck for k, ck in enumerate(c)))
    return W


def rational_shap(forest, x, exact_z, interactions, ntree=None):
    """Contributions [nrow][nf] or interaction values [nrow][nf][nf] (no bias entries) in exact rational arithmetic."""
    paths = _rational_paths(forest, ntree or len(forest.trees))
    nf = forest.num_feature
    out = []
    for row in np.asarray(x, np.float32):
        phi = [Fraction(0)] * nf
        M = [[Fraction(0)] * nf for _ in range(nf)]
        for v, elems in paths:
            o = [_one(row, f, s, miss) for f, s, miss, _, _ in elems]
            z = [ze if exact_z else zt for _, _, _, zt, ze in elems]
            feats = [e[0] for e in elems]
            for e, w in enumerate(_weights(o, z)):
                phi[feats[e]] += v * (o[e] - z[e]) * w
            if interactions:
                for c in range(len(elems)):
                    keep = [j for j in range(len(elems)) if j != c]
                    W = _weights([o[j] for j in keep], [z[j] for j in keep])
                    for k, j in enumerate(keep):
                        M[feats[c]][feats[j]] += Fraction(1, 2) * v * (o[c] - z[c]) * W[k] * (o[j] - z[j])
        if interactions:
            for c in range(nf):
                M[c][c] = phi[c] - sum(M[c][k] for k in range(nf) if k != c)
            out.append(M)
        else:
            out.append(phi)
    return out


def _edge(name):
    """(forest, rows, rows for the interactions) of an edge booster."""
    if name in ("caterpillar", "caterpillar_mirror"):
        f, thr, cont = ef.caterpillar(mirror=name.endswith("mirror"))
        return f, ef.caterpillar_rows(thr, cont, 3, seed=2), None
    f = {"repeats": ef.repeats, "covers": ef.covers, "underflow": ef.underflow, "overflow": ef.overflow,
         "stumps17": lambda: ef.stumps(17)}[name]()  # fmt: skip
    x = ef.special_rows(f, 6, seed=3)
    return f, x, x[:3]


def _exact_diff(ref, want, mag):
    """max over entries of |ref - want| / A, in exact arithmetic; 0 where A = 0 requires ref == want."""
    worst = Fraction(0)
    for r, w, a in zip(np.asarray(ref).ravel(), want, np.asarray(mag).ravel()):
        n, d = np.longdouble(r).as_integer_ratio()
        diff = abs(Fraction(n, d) - w)
        if a == 0:
            assert diff == 0, (r, w)
            continue
        n, d = np.longdouble(a).as_integer_ratio()
        worst = max(worst, diff / Fraction(n, d))
    return worst


@pytest.mark.parametrize("name", ["caterpillar", "caterpillar_mirror", "repeats", "covers", "underflow", "overflow", "stumps17"])
def test_reference_is_exact_rational_arithmetic(oracle, tmp_path, name):
    """Both modes (the float32 zero fractions of the tables, and the exact products) agree with Fraction arithmetic
    within 2^-58 of each entry's magnitude — also where the library refuses the booster (+0 / +inf zero fractions)."""
    forest, x, xi = _edge(name)
    m, _ = _model(oracle, forest, tmp_path, name)
    nf = forest.num_feature
    for exact_z in (False, True):
        if name == "overflow" and not exact_z:
            continue  # z~ = +inf is no game
        phi, mag, _ = se.contributions(m, x, exact_z=exact_z)
        want = [q for row in rational_shap(forest, x, exact_z, False) for q in row]
        assert _exact_diff(phi[:, :nf], want, mag[:, :nf]) <= Fraction(1, 2**58), name
        if xi is not None:
            M, magm, _ = se.interactions(m, xi, exact_z=exact_z)
            want = [q for row in rational_shap(forest, xi, exact_z, True) for line in row for q in line]
            assert _exact_diff(M[:, :nf, :nf], want, magm[:, :nf, :nf]) <= Fraction(1, 2**58), name


@pytest.mark.parametrize("name", ["grown1", "sklearn", "caterpillar", "caterpillar_mirror", "repeats", "covers", "stumps17"])
def test_reference_is_the_float32_oracle_within_its_bar(oracle, tmp_path, name):
    """The float32 recursive TreeShap of libxgboost, restated in tests/oracle_contribs.c / oracle_interactions.c, is
    within the existing per-row bar of the reference, and the bias entries are bit-equal."""
    if name in ("grown1", "sklearn"):
        forest, x = _grown(name)
    else:
        forest, x, _ = _edge(name)
        x = np.concatenate([x, ef.special_rows(forest, 60, seed=4)]) if name != "caterpillar" else x
    m, _ = _model(oracle, forest, tmp_path, name)
    nf = forest.num_feature
    phi, _, _ = se.contributions(m, x)
    f32 = oc.predict_contribs(m, x)
    assert_shap_close(f32, phi.astype(np.float64), name)
    assert np.array_equal(f32[:, nf].view(np.uint32), phi[:, nf].astype(np.float32).view(np.uint32))
    xi = x[:30]
    M, _, _ = se.interactions(m, xi)
    i32 = oi.predict_interactions(m, xi)
    assert_interactions_close(i32, M.astype(np.float64), name)
    assert np.array_equal(M[:, nf, nf].astype(np.float32).view(np.uint32), f32[:30, nf].view(np.uint32))
    for ntree in (1, 2):
        b = se.contributions(m, x, ntree_limit=ntree)[0][:, nf].astype(np.float32)
        assert np.array_equal(b.view(np.uint32), oc.predict_contribs(m, x, ntree_limit=ntree)[:, nf].view(np.uint32))


def test_single_leaf_trees_explain_nothing(oracle, tmp_path):
    m, _ = _model(oracle, ef.single_leaves(), tmp_path, "leaves")
    x = ef.special_rows(ef.stumps(3), 5, seed=1)
    phi, mag, dmax = se.contributions(m, x)
    assert dmax == 0 and np.all(phi[:, :NF] == 0) and np.all(mag == 0)
    assert np.array_equal(phi[:, NF].astype(np.float32), oc.predict_contribs(m, x)[:, NF])


@pytest.mark.parametrize("name", ["underflow", "overflow"])
def test_unrepresentable_zero_fractions_are_refused(capi, tmp_path, name):
    """The kernels keep an element's one fraction in the sign of its float32 zero fraction: a product of cover
    ratios that rounds to +0 or +inf in float32 would be read as a wrong one fraction (or divide by zero), so the
    path tables refuse such a booster, naming the tree, the leaf and the feature, before any device work."""
    forest = getattr(ef, name)()
    p = str(tmp_path / f"{name}.model")
    xgbmodel.write_legacy_binary(forest, p)
    b = capi.Booster(p, parse_only=True)
    with pytest.raises(capi.QcohError, match=r"tree 0 leaf 3 has .* on feature 0: this booster cannot be explained"):
        b.shap_paths()
    with pytest.raises(capi.QcohError, match="positive, finite float32"):
        b.predict_contribs(None)
    with pytest.raises(capi.QcohError, match="positive, finite float32"):
        b.predict_interactions_device(None, None)
