"""CPU: the GE2E contrast loss oracle (Wan et al. eq. 7, tests/_contrast_oracle.py).  Its closed form shares every step
but G with oracle.ge2e.ge2e_fwd_bwd (its softmax branch reproduces that function) and equals float64 torch autograd
(ge2e_torch), which is itself pinned by reproducing the reference's softmax fixtures."""
import os

import numpy as np
import pytest

import _inputs as I
from _contrast_inputs import top2_gap, twin_embeddings
import _contrast_oracle as ge2e
from oracle import ge2e as oge2e

G = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize("name", list(I.GE2E_CASES))
def test_torch_restatement_reproduces_the_softmax_fixtures(name):
    """ge2e_torch's get_cossim / calc_loss restatement gives the reference's own float64 results."""
    g = load(f"ge2e_{name}.npz")
    N, M, D, kind, w, b = I.GE2E_CASES[name]
    E = I.ge2e_embeddings(N, M, D, kind)
    t = ge2e.ge2e_torch(E.astype(np.float64), w, b, "softmax")
    assert rel(t["loss"], g["loss_f64"]) < 1e-12
    assert rel(t["dw"], g["dw_f64"]) < 1e-10
    assert rel(t["db"], g["db_f64"]) < 1e-7
    assert rel(t["dE"], g["dE_f64"]) < 2e-6


@pytest.mark.parametrize("name", list(I.GE2E_CASES))
def test_closed_form_softmax_branch_is_the_oracle(name):
    """Everything but G is shared: with the softmax G the restated closed form is oracle.ge2e.ge2e_fwd_bwd, exactly."""
    N, M, D, kind, w, b = I.GE2E_CASES[name]
    for E in (I.ge2e_embeddings(N, M, D, kind), I.ge2e_embeddings(N, M, D, kind).astype(np.float64)):
        a, o = ge2e.ge2e_fwd_bwd(E, w, b, "softmax"), oge2e.ge2e_fwd_bwd(E, w, b)
        for k in ("loss", "per", "cos", "dE", "dw", "db"):
            np.testing.assert_array_equal(a[k], o[k])


def _cases():
    out = {}
    for name in ("c1", "nonunit", "clustered"):
        N, M, D, kind, w, b = I.GE2E_CASES[name]
        out[name] = (I.ge2e_embeddings(N, M, D, kind), w, b)
    out["twins"] = (twin_embeddings(64, 10, 256), 10.0, -5.0)
    return out


@pytest.mark.parametrize("name", ["c1", "nonunit", "clustered", "twins"])
def test_contrast_closed_form_matches_autograd(name):
    E, w, b = _cases()[name]
    E = E.astype(np.float64)
    o = ge2e.ge2e_fwd_bwd(E, w, b, "contrast")
    t = ge2e.ge2e_torch(E, w, b, "contrast")
    assert rel(o["loss"], t["loss"]) < 1e-10
    assert rel(o["per"], t["per"]) < 1e-10
    assert rel(o["dE"], t["dE"]) < 1e-10
    assert rel(o["dw"], t["dw"]) < 1e-10
    assert rel(o["db"], t["db"]) < 1e-10
    loss, per = ge2e.calc_loss_contrast(w * oge2e.get_cossim(E, oge2e.get_centroids(E)) + b)
    assert rel(loss, o["loss"]) < 1e-12 and rel(per, o["per"]) < 1e-12


def test_contrast_loss_values():
    """per = 1 - sigmoid(S_jj) + sigmoid(max_{k != j} S_jk) on a hand-made S."""
    S = np.array([[[2.0, 0.5, -1.0]], [[0.3, -0.2, 0.3]], [[1.0, 4.0, 0.0]]])
    sig = lambda x: 1 / (1 + np.exp(-x))
    exp = [1 - sig(2.0) + sig(0.5), 1 - sig(-0.2) + sig(0.3), 1 - sig(0.0) + sig(4.0)]
    loss, per = ge2e.calc_loss_contrast(S)
    np.testing.assert_allclose(per[:, 0], exp, rtol=1e-14)
    assert abs(loss - sum(exp)) < 1e-14
    np.testing.assert_array_equal(ge2e.contrast_kstar(S)[:, 0], [1, 0, 1])


def test_exact_ties_go_to_the_lowest_index():
    """tests/golden/toy.npz holds exact ties between off-diagonal cosines (rows (0, 1) and (2, *)): the gradient goes to
    the lowest tied column, as torch.max's does."""
    E = load("toy.npz")["E"].astype(np.float64)
    S = oge2e.get_cossim(E, oge2e.get_centroids(E))
    np.testing.assert_array_equal(ge2e.contrast_kstar(S), [[1, 1], [0, 0], [0, 0]])
    G = ge2e.contrast_grad(S)
    assert G[0, 1, 1] > 0 and G[0, 1, 2] == 0 and G[2, 0, 0] > 0 and G[2, 0, 1] == 0
    o = ge2e.ge2e_fwd_bwd(E, 1.0, 0.0, "contrast")
    t = ge2e.ge2e_torch(E, 1.0, 0.0, "contrast")
    assert rel(o["dE"], t["dE"]) < 1e-12 and rel(o["loss"], t["loss"]) < 1e-12


def test_twin_batches_have_a_clear_nearest_impostor():
    for N, M, D in [(3, 2, 4), (33, 7, 20), (64, 10, 256), (512, 10, 256)]:
        E = twin_embeddings(N, M, D)
        assert E.shape == (N, M, D) and E.dtype == np.float32
        assert top2_gap(E, 10.0, -5.0) > 1e-3
    np.testing.assert_array_equal(twin_embeddings(8, 4, 32, seed=3), twin_embeddings(8, 4, 32, seed=3))


def test_unknown_method_is_rejected():
    E = I.ge2e_embeddings(4, 5, 256, "unit").astype(np.float64)
    with pytest.raises(ValueError):
        ge2e.ge2e_fwd_bwd(E, 10.0, -5.0, "angular")
    with pytest.raises(ValueError):
        ge2e.ge2e_torch(E, 10.0, -5.0, "angular")
