"""CPU: the cohort score normalization oracle (tests/_asnorm_oracle.py) against an independent float64 torch
composition and a brute-force sorted loop."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _asnorm_oracle as A


def torch_stats(X, C, K):
    S = F.normalize(torch.tensor(X, dtype=torch.float64), dim=1) @ F.normalize(torch.tensor(C, dtype=torch.float64),
                                                                               dim=1).T
    top = torch.topk(S, K, dim=1).values
    return torch.stack([top.mean(1), top.std(1), top[:, -1]], 1).numpy()


def brute_stats(S, K):
    out = []
    for row in np.asarray(S, np.float64):
        top = sorted(row.tolist(), reverse=True)[:K]
        mu = sum(top) / K
        out.append([mu, (sum((v - mu) ** 2 for v in top) / (K - 1)) ** 0.5, top[-1]])
    return np.array(out)


@pytest.mark.parametrize("n,Nc,D,K", [(7, 50, 16, 2), (5, 300, 64, 37), (3, 31, 13, 31), (4, 1001, 100, 300)])
def test_oracle_matches_torch_composition(n, Nc, D, K):
    r = np.random.RandomState(n * 1000 + Nc)
    X, C = r.standard_normal((n, D)), r.standard_normal((Nc, D))
    np.testing.assert_allclose(A.stats(X, C, K), torch_stats(X, C, K), rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("case", ["ties", "two_values", "k_equals_nc", "signed_zero"])
def test_oracle_matches_brute_force(case):
    r = np.random.RandomState(3)
    if case == "ties":
        S, K = np.round(r.standard_normal((6, 40)), 1), 7
    elif case == "two_values":
        S, K = np.where(r.rand(6, 20) < 0.3, 0.25, -0.5), 9
    elif case == "k_equals_nc":
        S, K = r.standard_normal((6, 9)), 9
    else:
        S, K = np.where(r.rand(6, 12) < 0.5, 0.0, -0.0), 3
        S[:, 0] = 1.0
    got, ref = A.stats_from_scores(S, K), brute_stats(S, K)
    np.testing.assert_allclose(got[:, :2], ref[:, :2], rtol=1e-12, atol=1e-15)
    np.testing.assert_array_equal(got[:, 2], ref[:, 2])


def test_non_finite_score_gives_nan_statistics():
    S = np.zeros((3, 5))
    S[1, 2] = np.inf
    S[2, 0] = np.nan
    got = A.stats_from_scores(S + np.arange(5), 2)
    assert np.isfinite(got[0]).all() and np.isnan(got[1:]).all()


def test_normalized_forms_agree():
    """The trial form and the TI-SV matrix form give the same score for the same (centroid, utterance) pair."""
    r = np.random.RandomState(5)
    N, M, D = 5, 3, 24
    cen, ver, C = r.standard_normal((N, D)), r.standard_normal((N, M, D)), r.standard_normal((40, D))
    sim = A.cosine(ver.reshape(N * M, D), cen).reshape(N, M, N)
    mat = A.normalize_sim(sim, cen, ver, C, 10)
    ei = np.tile(np.arange(N), N * M)
    ti = np.repeat(np.arange(N * M), N)
    trials = A.trial_scores(cen, ver.reshape(N * M, D), ei, ti, C, 10)
    np.testing.assert_allclose(mat.reshape(-1), trials, rtol=1e-12, atol=1e-12)
    st = A.stats(cen, C, 10)
    sv = A.stats(ver.reshape(N * M, D), C, 10)
    j, m, k = 2, 1, 4
    ref = 0.5 * ((sim[j, m, k] - st[k, 0]) / st[k, 1] + (sim[j, m, k] - sv[j * M + m, 0]) / sv[j * M + m, 1])
    assert abs(mat[j, m, k] - ref) < 1e-12
