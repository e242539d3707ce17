"""CPU: the matmul-form float64 get_cossim of tests/_ge2e_oracle.py (used by tests/test_gpu_ge2e_routes.py at sizes
where oracle.ge2e.get_cossim's broadcast does not fit) is oracle.ge2e.get_cossim, values and gradient."""
import numpy as np
import pytest

import _ge2e_oracle as G
import _inputs as I
from oracle import ge2e as oge2e


def foreign(N, M, D, kind, seed):
    """(E, C): a batch and the centroids of a different batch of the same speakers count."""
    E = I.ge2e_embeddings(N, M, D, kind, seed=seed).astype(np.float64)
    C = oge2e.get_centroids(I.ge2e_embeddings(N, M + 1, D, kind, seed=seed + 1).astype(np.float64))
    return E, C


CASES = [(7, 3, 16, "raw"), (5, 2, 64, "unit"), (12, 4, 20, "clustered"), (9, 17, 8, "raw")]


@pytest.mark.parametrize("N,M,D,kind", CASES)
def test_matmul_restatement_is_the_oracle(N, M, D, kind):
    """Own centroids and foreign centroids, including a zero centroid row and a zero embedding row (each norm is
    clamped on its own)."""
    E, C = foreign(N, M, D, kind, 5 * N + M)
    np.testing.assert_allclose(G.cossim(E, oge2e.get_centroids(E)), oge2e.get_cossim(E, oge2e.get_centroids(E)),
                               rtol=0, atol=1e-14)
    np.testing.assert_allclose(G.cossim(E, C), oge2e.get_cossim(E, C), rtol=0, atol=1e-14)
    C[1] = 0.0
    E[2, 0] = 0.0
    np.testing.assert_allclose(G.cossim(E, C), oge2e.get_cossim(E, C), rtol=0, atol=1e-14)
    # float32 inputs are taken as float64 values
    np.testing.assert_array_equal(G.cossim(E.astype(np.float32), C.astype(np.float32)),
                                  G.cossim(E.astype(np.float32).astype(np.float64), C.astype(np.float32).astype(np.float64)))


@pytest.mark.parametrize("N,M,D,kind", CASES[:3])
def test_gradient_is_the_oracles_derivative(N, M, D, kind):
    """dE and dC of (cos * V).sum() against central differences of oracle.ge2e.get_cossim, element by element."""
    E, C = foreign(N, M, D, kind, 7 * N + M)
    V = np.random.RandomState(N + M + D).standard_normal((N, M, N))
    cos, dE, dC = G.cossim_grads(E, C, V)
    np.testing.assert_allclose(cos, oge2e.get_cossim(E, C), rtol=0, atol=1e-14)
    f = lambda E_, C_: float((oge2e.get_cossim(E_, C_) * V).sum())
    h = 1e-6

    def numeric(X, other_first):
        g = np.zeros_like(X)
        for i in np.ndindex(X.shape):
            Xp, Xm = X.copy(), X.copy()
            Xp[i] += h
            Xm[i] -= h
            g[i] = ((f(Xp, C) - f(Xm, C)) if other_first else (f(E, Xp) - f(E, Xm))) / (2 * h)
        return g
    nE, nC = numeric(E, True), numeric(C, False)
    assert np.abs(dE - nE).max() < 1e-6 * np.abs(nE).max(), np.abs(dE - nE).max()
    assert np.abs(dC - nC).max() < 1e-6 * np.abs(nC).max(), np.abs(dC - nC).max()


def test_own_column_takes_no_centroid_gradient():
    """Column j of speaker j's rows is the leave-one-out cosine: an upstream gradient there reaches E only."""
    E, C = foreign(6, 3, 10, "raw", 3)
    V = np.zeros((6, 3, 6))
    V[np.arange(6), :, np.arange(6)] = 1.0
    _, dE, dC = G.cossim_grads(E, C, V)
    assert not np.any(dC) and np.abs(dE).max() > 0
