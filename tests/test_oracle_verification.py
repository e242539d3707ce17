"""CPU: the float64 restatement of the exact EER / minDCF (tests/_verif_oracle.py) against a brute-force loop over every
candidate threshold, its structural properties, and its counts pinned to the reference's 50-threshold sweep
(oracle.eer.eer_counts) on the C5 similarity matrix."""
import numpy as np
import pytest

import _inputs as I
import _verif_oracle as V
from oracle import eer as oeer

POINTS = V.operating_points([0.01, 0.05, 0.5], 1.0, 1.0) + V.operating_points(0.2, 3.0, 0.5)


def _case(kind, n, seed):
    r = np.random.RandomState(seed)
    if kind == "random":
        s = r.standard_normal(n).astype(np.float32)
    elif kind == "ties":
        s = r.randint(0, 7, n).astype(np.float32) * np.float32(0.25)
    else:                                                      # signed zeros and a few distinct values
        s = r.choice(np.array([-0.0, 0.0, -1.0, 1.0, 1e-40], np.float32), n)
    lab = r.rand(n) < 0.3
    lab[0], lab[1] = True, False
    return s, lab


@pytest.mark.parametrize("kind", ["random", "ties", "zeros"])
@pytest.mark.parametrize("n,seed", [(2, 1), (7, 2), (40, 3), (257, 4)])
def test_oracle_equals_brute_force(kind, n, seed):
    s, lab = _case(kind, n, seed)
    got, ref = V.metrics(s, lab, POINTS), V.brute_force(s, lab, POINTS)
    np.testing.assert_array_equal(got, ref)


@pytest.mark.parametrize("kind", ["random", "ties", "zeros"])
def test_criterion_strictly_increasing(kind):
    s, lab = _case(kind, 500, 9)
    _, miss, fa, Nt, Nn = V.curve(s, lab)
    d = miss * Nn - fa * Nt
    assert (np.diff(d) > 0).all()
    assert miss[0] == 0 and fa[-1] == 0 and miss[-1] == Nt and fa[0] == Nn


def test_perfect_separation_is_zero():
    r = np.random.RandomState(5)
    s = np.concatenate([r.rand(50) + 2.0, r.rand(70)]).astype(np.float32)
    lab = np.arange(120) < 50
    out = V.metrics(s, lab, POINTS)
    assert out[0] == 0.0 and out[2] == 0.0 and out[3] == 0.0
    assert out[1] == float(s[:50].min())
    assert all(out[8 + 4 * p] == 0.0 for p in range(len(POINTS)))


def test_scale_invariance_where_the_grid_sweep_reports_zero():
    """Scores below 0.5 everywhere: the 50-threshold sweep returns EER 0, the exact EER is that of the unscaled
    scores (a positive scale keeps the order)."""
    enr, ver = I.eer_embeddings(64, 6, 0.06, 0.5, 7)
    cen = enr.mean(1)
    cen /= np.linalg.norm(cen, axis=1, keepdims=True)
    sim = np.einsum("nmd,kd->nmk", ver, cen).astype(np.float32)
    assert oeer.eer_sweep(sim * np.float32(0.4))[0] == 0
    a, b = V.metrics_sim(sim, POINTS), V.metrics_sim(sim * np.float32(0.25), POINTS)
    assert a[0] == b[0] and a[0] > 0


def test_counts_match_reference_grid_c5():
    """At every float32 grid threshold tau, the point whose v_{k+1} is the smallest distinct value above tau has the
    reference's pooled counts: fa = sum(cnt_all - cnt_diag), miss = N * Mv - sum(cnt_diag)."""
    enr, ver = I.eer_embeddings(1024, 6, 0.06, 0.5, 4242)
    cen = enr.mean(1)
    cen /= np.linalg.norm(cen, axis=1, keepdims=True)
    sim = np.einsum("nmd,kd->nmk", ver, cen).astype(np.float32)
    N, Mv, _ = sim.shape
    thr, miss, fa, Nt, Nn = V.curve(sim, V.sim_labels(N, Mv))
    assert Nt == N * Mv and Nn == N * Mv * (N - 1)
    v = thr[:-1].astype(np.float32)
    call, cdiag = oeer.eer_counts(sim)
    for t, tau in enumerate(oeer.THRESHOLDS):
        k = int(np.searchsorted(v, np.float32(tau), "right"))
        assert fa[k] == call[t].sum() - cdiag[t].sum(), tau
        assert miss[k] == N * Mv - cdiag[t].sum(), tau
    out = V.metrics_sim(sim, V.operating_points(0.01))
    assert abs(out[0] - 0.04) < 5e-4                         # the grid sweep reports 0.0403 at threshold 0.57
