"""float64 numpy restatement of cohort score normalization (DESIGN.md 4.5.2, include/svb200.h svb_cohort_stats).

Statistics of a row against a cohort with top-K: S_K = the K largest cosines, mean, sample std (ddof = 1) and the K-th
largest value v_K.  A row with a non-finite cohort score has NaN statistics.  Normalized score of a trial (e, t):
1/2 ((s - mean_e) / std_e + (s - mean_t) / std_t).
"""
import numpy as np


def unit(X):
    X = np.asarray(X, np.float64)
    return X / np.linalg.norm(X, axis=-1, keepdims=True)


def cosine(X, Y):
    return unit(X) @ unit(Y).T


def stats_from_scores(S, K):
    """S (n, Nc) -> (n, 3) float64: mean, std, v_K."""
    S = np.asarray(S, np.float64)
    Nc = S.shape[1]
    top = np.partition(S, Nc - K, axis=1)[:, Nc - K:]      # v_K at column 0, every other column >= it
    with np.errstate(invalid="ignore"):                     # rows with inf / NaN scores are set to NaN below
        out = np.stack([top.mean(axis=1), top.std(axis=1, ddof=1), top[:, 0]], axis=1)
    out[~np.isfinite(S).all(axis=1)] = np.nan
    return out


def stats(X, C, K):
    return stats_from_scores(cosine(X, C), K)


def normalized(s, st_e, st_t):
    return 0.5 * ((s - st_e[..., 0]) / st_e[..., 1] + (s - st_t[..., 0]) / st_t[..., 1])


def trial_scores(E, T, ei, ti, C=None, K=None):
    """Raw cosines of the trials, or their normalized scores with a cohort C (K None: all of it)."""
    s = np.sum(unit(E)[ei] * unit(T)[ti], axis=1)
    if C is None:
        return s
    K = len(C) if K is None else K
    return normalized(s, stats(E, C, K)[ei], stats(T, C, K)[ti])


def normalize_sim(sim, centroids, ver, C, K=None):
    """TI-SV matrix sim (N, M, N): centroids (N, D) are the enrollment side, ver (N, M, D) the test side."""
    N, M = sim.shape[:2]
    K = len(C) if K is None else K
    sc = stats(centroids, C, K)
    sv = stats(np.asarray(ver).reshape(N * M, -1), C, K).reshape(N, M, 1, 3)
    return normalized(np.asarray(sim, np.float64), sc[None, None, :, :], sv)
