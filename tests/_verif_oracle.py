"""Float64 numpy restatement of the exact EER / minDCF definitions (DESIGN.md 4.5; the kernels: csrc/verif.cu).

Operating point k in {0, ..., K} of the distinct scores v_1 < ... < v_K accepts the scores >= v_{k+1} (point K accepts
nothing, threshold +inf).  miss_k = targets below v_{k+1}, fa_k = non-targets at or above it.  EER: the first k of the
smallest |miss_k * Nn - fa_k * Nt| (exact integers), reported as (p_miss + p_fa) / 2.  minDCF per (w_miss, w_fa, c_def):
the first k of the smallest (w_miss * p_miss + w_fa * p_fa) / c_def, numpy's separately rounded float64 operations.
"""
import numpy as np


def operating_points(p_target=0.01, c_miss=1.0, c_fa=1.0):
    """-> [(w_miss, w_fa, c_def)] in float64, one per target prior."""
    priors = [p_target] if np.ndim(p_target) == 0 else list(p_target)
    out = []
    for p in priors:
        w_miss, w_fa = float(c_miss) * float(p), float(c_fa) * (1.0 - float(p))
        out.append((w_miss, w_fa, min(w_miss, w_fa)))
    return out


def curve(scores, labels):
    """-> (thr, miss, fa, Nt, Nn) over the K + 1 operating points: thr float64 (+inf last), miss / fa int64."""
    s = np.asarray(scores, np.float32).ravel().copy()
    s[s == 0] = 0.0                                             # -0 -> +0 (denormals compare unequal to 0)
    lab = np.asarray(labels).ravel() != 0
    if not np.isfinite(s).all():
        raise ValueError("non-finite score")
    t, nt = np.sort(s[lab]), np.sort(s[~lab])
    v = np.unique(s)                                            # v_1 < ... < v_K
    miss = np.append(np.searchsorted(t, v, "left"), t.size).astype(np.int64)         # targets < v_{k+1}
    fa = np.append(nt.size - np.searchsorted(nt, v, "left"), 0).astype(np.int64)     # non-targets >= v_{k+1}
    thr = np.append(v.astype(np.float64), np.inf)
    return thr, miss, fa, int(t.size), int(nt.size)


def metrics(scores, labels, points):
    """-> float64 array laid out as svb_verif_metrics' `out`: eer, threshold, p_miss, p_fa, Nt, Nn, #non-finite (0), K,
    then per point min_dcf, threshold, p_miss, p_fa."""
    thr, miss, fa, Nt, Nn = curve(scores, labels)
    if Nt == 0 or Nn == 0:
        raise ValueError("empty class")
    crit = np.abs(miss * Nn - fa * Nt)                          # int64: < 2^62 for n < 2^31
    k = int(np.argmin(crit))                                    # first index of the minimum
    pm, pf = miss / Nt, fa / Nn
    out = [(pm[k] + pf[k]) / 2, thr[k], pm[k], pf[k], Nt, Nn, 0, thr.size - 1]
    for w_miss, w_fa, c_def in points:
        dcf = (w_miss * pm + w_fa * pf) / c_def
        j = int(np.argmin(dcf))
        out += [dcf[j], thr[j], pm[j], pf[j]]
    return np.array(out, np.float64)


def sim_labels(N, Mv):
    """Target mask of a TI-SV similarity matrix (N, Mv, N): [j, m, k] is a target iff k == j."""
    lab = np.zeros((N, Mv, N), bool)
    lab[np.arange(N), :, np.arange(N)] = True
    return lab


def metrics_sim(sim, points):
    sim = np.asarray(sim, np.float32)
    return metrics(sim, sim_labels(sim.shape[0], sim.shape[1]), points)


def brute_force(scores, labels, points):
    """Every candidate threshold (each score value, then +inf) with counts by direct comparison: the definitions
    without np.unique / searchsorted, for small inputs."""
    s = np.asarray(scores, np.float32).ravel().astype(np.float64)
    s[s == 0] = 0.0
    lab = np.asarray(labels).ravel() != 0
    Nt, Nn = int(lab.sum()), int((~lab).sum())
    cands = sorted(set(s.tolist())) + [np.inf]
    rows = []
    for c in cands:
        miss = int(np.sum(lab & (s < c)))
        fa = int(np.sum(~lab & (s >= c)))
        rows.append((c, miss, fa))
    best = None
    for k, (c, miss, fa) in enumerate(rows):
        crit = abs(miss * Nn - fa * Nt)
        if best is None or crit < best[0]:
            best = (crit, k)
    c, miss, fa = rows[best[1]]
    out = [(miss / Nt + fa / Nn) / 2, c, miss / Nt, fa / Nn, Nt, Nn, 0, len(cands) - 1]
    for w_miss, w_fa, c_def in points:
        bd = None
        for c, miss, fa in rows:
            d = (w_miss * (miss / Nt) + w_fa * (fa / Nn)) / c_def
            if bd is None or d < bd[0]:
                bd = (d, c, miss / Nt, fa / Nn)
        out += list(bd)
    return np.array(out, np.float64)
