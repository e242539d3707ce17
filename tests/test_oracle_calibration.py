"""CPU: the calibration oracle (tests/_calib_oracle.py) against independent forms of its definitions: an exact-rational
PAV loop (minCllr), BOSARIS' max-over-segments rocch2eer, scipy.optimize on C(a, b), brute-force actual-DCF counts and,
loosely, sklearn's isotonic and logistic regressions."""
import math
import warnings
from fractions import Fraction

import numpy as np
import pytest

import _calib_oracle as O
import _verif_oracle as V


def cases():
    out = []
    for seed in range(12):
        r = np.random.RandomState(seed)
        n = int(r.randint(2, 400))
        lab = r.rand(n) < r.uniform(0.05, 0.95)
        lab[0], lab[-1] = True, False
        s = r.standard_normal(n) * r.uniform(0.3, 3) + r.uniform(0, 3) * lab
        if seed % 3 == 1:
            s = np.round(s, 1)                                  # ties within and across classes
        out.append((s.astype(np.float32), lab))
    r = np.random.RandomState(99)
    lab = r.rand(300) < 0.3
    lab[0], lab[1] = True, False
    out.append((r.randint(0, 6, 300).astype(np.float32), lab))  # few distinct values
    out.append((np.array([0.0, -0.0, 1e-40, -1e-40, 2.0, 2.0], np.float32), np.array([1, 0, 0, 1, 1, 0], bool)))
    return out


def pav_min_cllr(s, lab):
    """Pool-adjacent-violators over groups of equal scores in exact fractions; min Cllr of the pooled LLRs."""
    s = np.where(s == 0, np.float32(0), s)
    Nt, Nn = int(lab.sum()), int((~lab).sum())
    blocks = []                                                 # [targets, trials]
    for v in np.unique(s):
        m = s == v
        blocks.append([int(lab[m].sum()), int(m.sum())])
        while len(blocks) >= 2 and Fraction(blocks[-2][0], blocks[-2][1]) >= Fraction(blocks[-1][0], blocks[-1][1]):
            t, n = blocks.pop()
            blocks[-1][0] += t
            blocks[-1][1] += n
    ts, ns = [], []
    for t, m in blocks:
        f = m - t
        if t and f:
            ts.append(t * math.log2(1 + Fraction(f * Nt, t * Nn)))
            ns.append(f * math.log2(1 + Fraction(t * Nn, f * Nt)))
    return 0.5 * (math.fsum(ts) / Nt + math.fsum(ns) / Nn)


def bosaris_rocch2eer(pmiss, pfa):
    eer = 0.0
    for i in range(len(pfa) - 1):
        xx, yy = pfa[i:i + 2], pmiss[i:i + 2]
        if min(abs(xx[0] - xx[1]), abs(yy[0] - yy[1])) == 0:
            seg = 0.0
        else:
            XY = np.array([[xx[0], yy[0]], [xx[1], yy[1]]], np.float64)
            c = np.linalg.solve(XY, np.ones(2))
            seg = 1.0 / c.sum()
        eer = max(eer, seg)
    return eer


@pytest.mark.parametrize("k", range(len(cases())))
def test_min_cllr_matches_exact_pav(k):
    s, lab = cases()[k]
    got = O.metrics(s, lab, V.operating_points(0.01))
    assert abs(got[1] - pav_min_cllr(s, lab)) <= 1e-13
    assert got[1] <= got[0] + 1e-15 and got[1] <= 1 + 1e-15


@pytest.mark.parametrize("k", range(len(cases())))
def test_hull_forms_agree(k):
    s, lab = cases()[k]
    X, Y = O.group_points(s, lab)
    hx, hy = O.lower_hull(X, Y)
    assert list(zip(hx.tolist(), hy.tolist())) == O.lower_hull_serial(X, Y)


@pytest.mark.parametrize("k", range(len(cases())))
def test_rocch_eer_matches_bosaris_and_fractions(k):
    s, lab = cases()[k]
    _, _, Nt, Nn = O._canon(s, lab)
    hx, hy = O.lower_hull(*O.group_points(s, lab))
    e = O.rocch_eer(hx, hy, Nt, Nn)
    assert abs(e - float(O.rocch_eer(hx, hy, Nt, Nn, exact=True))) <= 1e-15
    pmiss = hy / Nt
    pfa = (Nn - (hx - hy)) / Nn
    if np.all(np.diff(pmiss) > 0) and np.all(np.diff(pfa) < 0):   # BOSARIS' form needs non-axis-parallel segments
        assert abs(e - bosaris_rocch2eer(pmiss, pfa)) <= 1e-12


def test_min_cllr_extremes():
    lab = np.array([0, 0, 0, 1, 1], bool)
    sep = O.metrics(np.array([1, 2, 3, 4, 5], np.float32), lab, V.operating_points(0.5))
    assert sep[1] == 0.0 and sep[2] == 0.0
    flat = O.metrics(np.full(5, 0.3, np.float32), lab, V.operating_points(0.5))
    assert abs(flat[1] - 1.0) <= 1e-15 and flat[6] == 2 and flat[7] == 1
    rev = O.metrics(np.array([5, 4, 3, 2, 1], np.float32), lab, V.operating_points(0.5))
    assert abs(rev[1] - 1.0) <= 1e-15 and rev[2] == 0.5


@pytest.mark.parametrize("k", range(len(cases())))
def test_actual_dcf_by_brute_force(k):
    s, lab = cases()[k]
    pts = V.operating_points([0.01, 0.3, 0.5, 0.9], 2.0, 0.5)
    l = np.where(s == 0, 0.0, s.astype(np.float64))
    Nt, Nn = int(lab.sum()), int((~lab).sum())
    for (w_miss, w_fa, c_def), (dcf, th, pm, pf) in zip(pts, O.act_dcf(s, lab, pts)):
        assert th == math.log(w_fa / w_miss)
        miss = sum(1 for x, t in zip(l, lab) if t and not x >= th)
        fa = sum(1 for x, t in zip(l, lab) if not t and x >= th)
        assert (pm, pf) == (miss / Nt, fa / Nn)
        assert dcf == (w_miss * (miss / Nt) + w_fa * (fa / Nn)) / c_def


def test_cllr_definition():
    s = np.array([-2.0, 0.5, 3.0, -1.0, 1.0], np.float32)
    lab = np.array([0, 1, 1, 0, 0], bool)
    sp = lambda x: math.log(1 + math.exp(x))
    ref = 0.5 * ((sp(-0.5) + sp(-3.0)) / 2 + (sp(-2.0) + sp(-1.0) + sp(1.0)) / 3) / math.log(2)
    assert abs(O.cllr(s, lab) - ref) <= 1e-15


@pytest.mark.parametrize("prior", [0.5, 0.1, 0.9])
@pytest.mark.parametrize("k", [0, 4, 7, 12])
def test_train_matches_scipy(prior, k):
    scipy_opt = pytest.importorskip("scipy.optimize")
    s, lab = cases()[k]
    a, b, c, iters, status = O.train(s, lab, prior)
    assert status == 0 and iters < 30
    x64, Nt, Nn = s.astype(np.float64), int(lab.sum()), int((~lab).sum())
    w = np.where(lab, prior / Nt, (1 - prior) / Nn)

    def grad(x):                                                # sum w (sigmoid(z) - y) (s, 1)
        r = w * (1 / (1 + np.exp(-(x[0] * x64 + x[1] + math.log(prior / (1 - prior))))) - lab)
        return np.array([np.sum(r * x64), np.sum(r)])

    res = scipy_opt.minimize(lambda x: O.objective(x[0], x[1], s, lab, prior), np.zeros(2), jac=grad, method="BFGS",
                             options={"gtol": 1e-13, "xrtol": 1e-15})
    ra, rb = res.x
    assert abs(a - ra) <= 1e-7 * max(1.0, abs(ra)) and abs(b - rb) <= 1e-7 * (1 + abs(rb))
    assert abs(c * math.log(2) - O.objective(a, b, s, lab, prior)) <= 1e-14
    assert O.objective(a, b, s, lab, prior) <= res.fun + 1e-15


def test_train_at_half_prior_gives_cllr():
    s, lab = cases()[3]
    a, b, c, _, status = O.train(s, lab, 0.5)
    assert status == 0
    assert abs(c - O.cllr((a * s.astype(np.float64) + b), lab)) <= 1e-6      # float32 rounding of the LLRs
    m = O.metrics(s, lab, V.operating_points(0.5))
    assert m[1] <= c <= 1 + 1e-12


def test_train_separable_and_single_value():
    lab = np.array([0, 0, 1, 1], bool)
    assert O.train(np.array([0, 1, 2, 3], np.float32), lab)[4] == 1
    assert O.train(np.array([0, 1, 1, 3], np.float32), lab)[4] == 1          # touching, not overlapping
    assert O.train(np.array([3, 2, 1, 0], np.float32), lab)[4] == 1
    assert O.train(np.full(4, 2.0, np.float32), lab)[4] == 1
    assert O.train(np.array([0, 2, 1, 3], np.float32), lab)[4] == 0


def test_sklearn_cross_checks():
    iso = pytest.importorskip("sklearn.isotonic")
    lm = pytest.importorskip("sklearn.linear_model")
    for k in (0, 1, 4, 12):
        s, lab = cases()[k]
        Nt, Nn = int(lab.sum()), int((~lab).sum())
        p = iso.IsotonicRegression(out_of_bounds="clip").fit(s.astype(np.float64), lab.astype(np.float64)).predict(
            s.astype(np.float64))
        with np.errstate(divide="ignore"):
            t = np.where(p[lab] > 0, -np.log2(np.where(p[lab] > 0, p[lab], 1) * Nn /
                                               (np.where(p[lab] > 0, p[lab], 1) * Nn + (1 - p[lab]) * Nt)), np.inf)
            f = np.where(p[~lab] < 1, -np.log2(np.where(p[~lab] < 1, 1 - p[~lab], 1) * Nt /
                                                (p[~lab] * Nn + np.where(p[~lab] < 1, 1 - p[~lab], 1) * Nt)), np.inf)
        ref = 0.5 * (t.sum() / Nt + f.sum() / Nn)
        got = O.metrics(s, lab, V.operating_points(0.5))[1]
        assert abs(got - ref) <= 1e-7
        prior = 0.3
        w = np.where(lab, prior / Nt, (1 - prior) / Nn)
        with warnings.catch_warnings():                        # newer sklearn deprecates penalty=None
            warnings.simplefilter("ignore", FutureWarning)
            clf = lm.LogisticRegression(penalty=None, tol=1e-12, max_iter=10000).fit(
                s.astype(np.float64).reshape(-1, 1), lab, sample_weight=w * len(s))
        a, b, _, _, status = O.train(s, lab, prior)
        assert status == 0
        assert abs(a - clf.coef_[0, 0]) <= 1e-5 * abs(a)
        assert abs(b - (clf.intercept_[0] - math.log(prior / (1 - prior)))) <= 1e-5 * (1 + abs(b))
