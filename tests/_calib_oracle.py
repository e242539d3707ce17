"""Float64 numpy restatement of the calibration definitions (DESIGN.md 4.5.3; the kernels: csrc/calib.cu).

Scores are float32 natural-log LLRs; -0.0 counts as +0.0.  Sums use math.fsum, hull tests exact integer cross products
(int64 numpy, every product < 2^62), and ``rocch_eer(..., exact=True)`` takes the crossing in Python fractions.
"""
import math
from fractions import Fraction

import numpy as np

LN2 = math.log(2.0)


def _canon(scores, labels):
    s = np.asarray(scores, np.float32).ravel().copy()
    s[s == 0] = 0.0                                             # -0 -> +0 (denormals compare unequal to 0)
    lab = np.asarray(labels).ravel() != 0
    if not np.isfinite(s).all():
        raise ValueError("non-finite score")
    Nt, Nn = int(lab.sum()), int((~lab).sum())
    if Nt == 0 or Nn == 0:
        raise ValueError("empty class")
    return s, lab, Nt, Nn


def softplus(x):
    return np.maximum(x, 0.0) + np.log1p(np.exp(-np.abs(x)))


def cllr(scores, labels):
    s, lab, Nt, Nn = _canon(scores, labels)
    l = s.astype(np.float64)
    return 0.5 * (math.fsum(softplus(-l[lab])) / Nt + math.fsum(softplus(l[~lab])) / Nn) / LN2


def thresholds(points):
    return [math.log(w_fa / w_miss) for w_miss, w_fa, _ in points]


def act_dcf(scores, labels, points):
    """-> [(act_dcf, theta, p_miss, p_fa)] per operating point (w_miss, w_fa, c_def)."""
    s, lab, Nt, Nn = _canon(scores, labels)
    l = s.astype(np.float64)
    out = []
    for (w_miss, w_fa, c_def), th in zip(points, thresholds(points)):
        miss = int(np.sum(lab & (l < th)))
        fa = int(np.sum(~lab & (l >= th)))
        pm, pf = miss / Nt, fa / Nn
        out.append(((w_miss * pm + w_fa * pf) / c_def, th, pm, pf))
    return out


def group_points(scores, labels):
    """-> (X, Y) int64: trials and targets up to and including each group of equal scores, ascending."""
    s, lab, _, _ = _canon(scores, labels)
    order = np.argsort(s, kind="stable")
    ss, ll = s[order], lab[order]
    ends = np.flatnonzero(np.append(ss[1:] != ss[:-1], True))
    return (ends + 1).astype(np.int64), np.cumsum(ll, dtype=np.int64)[ends]


def _cross(ox, oy, ax, ay, bx, by):
    return (ax - ox) * (by - oy) - (ay - oy) * (bx - ox)


def lower_hull(X, Y):
    """Strictly convex lower hull of (0, 0) and the points (X, Y) (X ascending): vertices as int64 arrays.  Points on or
    above the segment joining their neighbours are dropped, all at once, until none is; every dropped point lies on or
    above the final chain, which is convex, so it is the lower hull."""
    hx = np.concatenate([[0], X]).astype(np.int64)
    hy = np.concatenate([[0], Y]).astype(np.int64)
    while hx.size > 2:
        c = _cross(hx[:-2], hy[:-2], hx[1:-1], hy[1:-1], hx[2:], hy[2:])
        drop = c <= 0
        if not drop.any():
            break
        keep = np.concatenate([[True], ~drop, [True]])
        hx, hy = hx[keep], hy[keep]
    return hx, hy


def lower_hull_serial(X, Y):
    """The same hull by Andrew's monotone chain in Python integers (for small inputs)."""
    h = [(0, 0)]
    for p in zip((int(v) for v in X), (int(v) for v in Y)):
        while len(h) >= 2 and _cross(*h[-2], *h[-1], *p) <= 0:
            h.pop()
        h.append(p)
    return h


def min_cllr(hx, hy, Nt, Nn):
    ts, ns = [], []
    for k in range(1, hx.size):
        t = int(hy[k] - hy[k - 1])
        f = int(hx[k] - hx[k - 1]) - t
        if t > 0 and f > 0:
            ts.append(t * math.log1p((f * Nt) / (t * Nn)))
            ns.append(f * math.log1p((t * Nn) / (f * Nt)))
    return 0.5 * (math.fsum(ts) / Nt + math.fsum(ns) / Nn) / LN2


def rocch_eer(hx, hy, Nt, Nn, exact=False):
    """Where the hull's ROC polyline (P_miss = Y/Nt, P_fa = (Nn - (X - Y))/Nn) crosses P_miss = P_fa."""
    d = hy * Nn - (Nn - hx + hy) * Nt                           # sign of P_miss - P_fa, exact
    m = int(np.argmax(d >= 0))
    if d[m] == 0:
        return Fraction(int(hy[m]), Nt) if exact else int(hy[m]) / Nt
    dp, dq = int(d[m - 1]), int(d[m])
    if exact:
        pm0, pm1 = Fraction(int(hy[m - 1]), Nt), Fraction(int(hy[m]), Nt)
        return pm0 + Fraction(-dp, dq - dp) * (pm1 - pm0)
    pm0, pm1 = int(hy[m - 1]) / Nt, int(hy[m]) / Nt
    return pm0 + (float(-dp) / float(dq - dp)) * (pm1 - pm0)


def metrics(scores, labels, points):
    """-> float64 array laid out as svb_calib_metrics' `out`: cllr, min_cllr, rocch_eer, Nt, Nn, #non-finite (0),
    #hull vertices, K, then per point act_dcf, theta, p_miss, p_fa."""
    _, _, Nt, Nn = _canon(scores, labels)
    X, Y = group_points(scores, labels)
    hx, hy = lower_hull(X, Y)
    out = [cllr(scores, labels), min_cllr(hx, hy, Nt, Nn), rocch_eer(hx, hy, Nt, Nn), Nt, Nn, 0, hx.size, X.size]
    for row in act_dcf(scores, labels, points):
        out += list(row)
    return np.array(out, np.float64)


# ------------------------------------------------------------------------------------------------ calibration
def objective(a, b, scores, labels, prior=0.5):
    """C(a, b) = (pi/Nt) sum_tar softplus(-(a s + b + tau)) + ((1 - pi)/Nn) sum_non softplus(a s + b + tau)."""
    s, lab, Nt, Nn = _canon(scores, labels)
    z = a * s.astype(np.float64) + b + math.log(prior / (1.0 - prior))
    return prior / Nt * math.fsum(softplus(-z[lab])) + (1.0 - prior) / Nn * math.fsum(softplus(z[~lab]))


def train(scores, labels, prior=0.5, max_iter=100, tol=1e-12):
    """Damped Newton from (0, 0) on centred scores u = (s - c0) * scale, as the kernels run it: a step is accepted when
    the objective decreases (else halved), and once half the squared Newton decrement is <= tol the last step is taken
    without a line search.  -> (a, b, C / ln 2, evaluations, status) as svb_calib_train's `out`."""
    s, lab, Nt, Nn = _canon(scores, labels)
    tmin, tmax, nmin, nmax = s[lab].min(), s[lab].max(), s[~lab].min(), s[~lab].max()
    if not (tmin < nmax and nmin < tmax):
        return (math.nan, math.nan, math.nan, 0, 1)
    lo, hi = float(min(tmin, nmin)), float(max(tmax, nmax))
    c0, scale = 0.5 * lo + 0.5 * hi, 2.0 / (hi - lo)
    u = (s.astype(np.float64) - c0) * scale
    w = np.where(lab, prior / Nt, (1.0 - prior) / Nn)
    tau = math.log(prior / (1.0 - prior))

    def evaluate(a, b):
        z = a * u + b + tau
        e = np.exp(-np.abs(z))
        sig = np.where(z >= 0, 1.0 / (1.0 + e), e / (1.0 + e))
        f = np.where(lab, np.maximum(-z, 0.0), np.maximum(z, 0.0)) + np.log1p(e)
        g = w * np.where(lab, sig - 1.0, sig)
        h = w * (e / ((1.0 + e) * (1.0 + e)))
        return (np.sum(w * f), np.sum(g * u), np.sum(g), np.sum(h * u * u), np.sum(h * u), np.sum(h))

    a = b = c = 0.0
    ta = tb = 0.0
    t, da, db, have, final, halvings = 1.0, 0.0, 0.0, False, False, 0
    for it in range(1, max_iter + 1):
        C, ga, gb, haa, hab, hbb = evaluate(ta, tb)
        if final:
            a, b, c = ta, tb, C
            return (a * scale, b - a * scale * c0, c / LN2, it, 0)
        if not have or C < c:
            a, b, c, have = ta, tb, C, True
            det = haa * hbb - hab * hab
            da, db = -(hbb * ga - hab * gb) / det, -(haa * gb - hab * ga) / det
            t, halvings = 1.0, 0
            ta, tb = a + da, b + db
            final = 0.5 * -(ga * da + gb * db) <= tol
        else:
            halvings += 1
            if halvings > 40:
                return (a * scale, b - a * scale * c0, c / LN2, it, 0)
            t *= 0.5
            ta, tb = a + t * da, b + t * db
    return (a * scale, b - a * scale * c0, c / LN2, max_iter, 2)
