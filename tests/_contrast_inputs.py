"""Seeded inputs for the GE2E contrast loss tests.

The contrast loss picks, per row, the most similar OTHER centroid k*; its gradient jumps where two off-diagonal
similarities tie.  Random embeddings at realistic sizes nearly always hold such near-ties, and an fp32 kernel may then
pick a different k* than the fp64 oracle.  Twin-structured batches avoid that: speakers come in pairs whose centres
share a component, so every speaker has one clear nearest impostor (its twin).
"""
import numpy as np

from _ge2e_oracle import cossim
from oracle import ge2e as oge2e


def top2_gap(E, w, b):
    """Smallest gap, over all rows, between the largest and the second largest off-diagonal S = w cos + b (float64)."""
    E = np.asarray(E, dtype=np.float64)
    S = w * cossim(E, oge2e.get_centroids(E)) + b                    # (matmul form: fits at N = 512, D = 768)
    N = S.shape[0]
    idx = np.arange(N)
    S[idx, :, idx] = -np.inf
    top = np.sort(S, axis=2)
    return float((top[:, :, -1] - top[:, :, -2]).min())


def twin_embeddings(N, M, D, seed=0, raw=False, min_cos_gap=2e-3):
    """(N, M, D) float32.  Speakers 2p and 2p+1 have centres normalize(g_p + 0.8 r): each one's nearest impostor is its
    twin (an odd last speaker stands alone).  Utterances are normalize(centre + noise); raw=True scales each row by a
    factor in [0.5, 3].  Seeds are tried from ``seed`` on until every row's top-two off-diagonal cosine gap exceeds
    ``min_cos_gap`` (deterministic: the same arguments give the same batch)."""
    for s in range(seed, seed + 1000):
        r = np.random.RandomState(s * 7919 + N * 1000 + M * 10 + D)
        g = r.standard_normal(((N + 1) // 2, D))
        g = np.repeat(g / np.linalg.norm(g, axis=1, keepdims=True), 2, axis=0)[:N]
        c = g + 0.8 * r.standard_normal((N, D)) / np.sqrt(D)
        c /= np.linalg.norm(c, axis=1, keepdims=True)
        x = c[:, None, :] + 0.3 * r.standard_normal((N, M, D)) / np.sqrt(D)
        x /= np.linalg.norm(x, axis=2, keepdims=True)
        if raw:
            x *= r.uniform(0.5, 3.0, size=(N, M, 1))
        x = x.astype(np.float32)
        if N < 2 or top2_gap(x, 1.0, 0.0) > min_cos_gap:
            return x
    raise RuntimeError("no twin batch with a clear nearest impostor")


def twin_logmel(N, M, T, seed, nmels=40):
    """(N * M, T, nmels) float32 log-mel-like input (as _inputs.logmel) with the twin structure: speakers 2p and 2p+1
    share a (T, nmels) component, so that even an untrained embedder gives every speaker a clear nearest impostor."""
    r = np.random.RandomState(seed)
    g = np.repeat(r.standard_normal(((N + 1) // 2, 1, T, nmels)), 2, axis=0)[:N]
    c = g + 0.6 * r.standard_normal((N, 1, T, nmels))
    x = -3.0 + 1.5 * (c + 0.2 * r.standard_normal((N, M, T, nmels)))
    return np.maximum(x, -6.0).astype(np.float32).reshape(N * M, T, nmels)
