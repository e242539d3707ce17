"""Test-support oracle of the GE2E contrast loss (Wan et al., arXiv 1710.10467, eq. 7), in numpy and float64 torch.

The reference implements only the softmax loss (eq. 6); oracle/ge2e.py restates it.  The contrast loss is defined on
the same similarity matrix S = w cos + b (cos as get_cossim returns it: + 1e-6, leave-one-out diagonal):

    k*  = argmax_{k != j} S[j,i,k]                     (lowest index among exact ties, the element torch.max picks)
    per = 1 - sigmoid(S[j,i,j]) + sigmoid(S[j,i,k*])   (1 - sigmoid(x) evaluated as sigmoid(-x)),  loss = sum per

Only G = dL/dS differs from the softmax loss; ``ge2e_fwd_bwd`` takes either G through one copy of the closed form of
oracle.ge2e.ge2e_fwd_bwd (SURVEY.md section 7.3), and tests/test_oracle_contrast.py checks that its softmax branch
reproduces oracle.ge2e.ge2e_fwd_bwd and its contrast branch float64 autograd (``ge2e_torch``).
"""
import numpy as np

from oracle.ge2e import COS_BIAS, COS_EPS, LOG_BIAS

METHODS = ("softmax", "contrast")


def _sigmoid(x):
    return 1 / (1 + np.exp(-x))


def contrast_kstar(S):
    """k* of every row of S (N, M, Nc): the arg-max over the off-diagonal columns, lowest index among exact ties."""
    N = S.shape[0]
    Soff = S.copy()
    idx = np.arange(N)
    Soff[idx, :, idx] = -np.inf
    return Soff.argmax(axis=2)                                  # numpy's argmax returns the first maximum


def calc_loss_contrast(S):
    """Contrast loss of S (N, M, Nc), Nc >= 2 -> (loss, per_embedding_loss (N, M))."""
    N = S.shape[0]
    idx = np.arange(N)
    ks = contrast_kstar(S)
    sk = np.take_along_axis(S, ks[:, :, None], axis=2)[:, :, 0]
    per = _sigmoid(-S[idx, :, idx]) + _sigmoid(sk)
    return per.sum(), per


def contrast_grad(S):
    """dL/dS of the contrast loss: -sigmoid(S_jj) sigmoid(-S_jj) on the diagonal, sigmoid(S_jk*) sigmoid(-S_jk*) at k*,
    zero elsewhere."""
    N = S.shape[0]
    idx = np.arange(N)
    G = np.zeros_like(S)
    sd = S[idx, :, idx]
    G[idx, :, idx] = -_sigmoid(sd) * _sigmoid(-sd)
    ks = contrast_kstar(S)
    sk = np.take_along_axis(S, ks[:, :, None], axis=2)
    np.put_along_axis(G, ks[:, :, None], _sigmoid(sk) * _sigmoid(-sk), axis=2)
    return G


def ge2e_fwd_bwd(E, w, b, loss="softmax"):
    """Closed-form loss and gradient of the GE2E loss of either method -> dict(loss, per, cos, G, dE, dw, db).  The
    forward up to S and everything after G are oracle.ge2e.ge2e_fwd_bwd's, operation for operation."""
    if loss not in METHODS:
        raise ValueError(loss)
    dt = E.dtype.type
    N, M, D = E.shape
    eps = dt(COS_EPS)
    ne = np.maximum(np.sqrt((E * E).sum(-1, keepdims=True)), eps)
    Eh = E / ne
    s = E.sum(axis=1, keepdims=True)
    c = s[:, 0, :] / dt(M)
    nc = np.maximum(np.sqrt((c * c).sum(-1, keepdims=True)), eps)
    Ch = c / nc
    U = (s - E) / dt(M - 1)
    nu = np.maximum(np.sqrt((U * U).sum(-1, keepdims=True)), eps)
    Uh = U / nu
    cos0 = np.einsum('jid,kd->jik', Eh, Ch)
    idx = np.arange(N)
    cosd0 = (Eh * Uh).sum(-1)
    cos0[idx, :, idx] = cosd0
    cos = cos0 + dt(COS_BIAS)
    S = dt(w) * cos + dt(b)
    if loss == "contrast":
        total, per = calc_loss_contrast(S)
        G = contrast_grad(S)
    else:
        ex = np.exp(S)
        den = ex.sum(axis=2) + dt(LOG_BIAS)
        per = -(S[idx, :, idx] - np.log(den))
        total = per.sum()
        G = ex / den[:, :, None]
        G[idx, :, idx] -= dt(1)
    dw = (G * cos).sum()
    db = G.sum()
    A = dt(w) * G
    a = A[idx, :, idx].copy()
    Aoff = A.copy()
    Aoff[idx, :, idx] = 0
    cos_off = cos0.copy()
    cos_off[idx, :, idx] = 0
    r = (Aoff * cos_off).sum(axis=2)
    R = np.einsum('jik,kd->jid', Aoff, Ch)
    dE = (R - r[:, :, None] * Eh) / ne
    dE += a[:, :, None] * (Uh - cosd0[:, :, None] * Eh) / ne
    P = np.einsum('jik,jid->kd', Aoff, Eh)
    q = (Aoff * cos_off).sum(axis=(0, 1))
    dC = (P - q[:, None] * Ch) / nc
    dE += dC[:, None, :] / dt(M)
    dU = a[:, :, None] * (Eh - cosd0[:, :, None] * Uh) / nu
    dE += (dU.sum(axis=1, keepdims=True) - dU) / dt(M - 1)
    return dict(loss=total, per=per, cos=cos, G=G, dE=dE, dw=dw, db=db)


def ge2e_torch(E, w, b, loss="softmax"):
    """Independent float64 restatement through torch autograd: get_cossim as utils.py:72-115 writes it
    (F.cosine_similarity against the centroids and the leave-one-out centroids, diagonal overwrite, + 1e-6), S = w cos
    + b, then the softmax loss (utils.py:126-132) or the contrast loss (sigmoid, and a gather at the first arg-max of
    the off-diagonal S).  Returns dict(loss, per, dE, dw, db) as float64 numpy."""
    import torch
    import torch.nn.functional as F
    if loss not in METHODS:
        raise ValueError(loss)
    Et = torch.tensor(np.asarray(E), dtype=torch.float64, requires_grad=True)
    wt = torch.tensor(float(w), dtype=torch.float64, requires_grad=True)
    bt = torch.tensor(float(b), dtype=torch.float64, requires_grad=True)
    N, M, D = Et.shape
    C = Et.mean(dim=1)                                                          # utils.py:27-29
    U = (Et.sum(dim=1, keepdim=True) - Et) / (M - 1)                            # utils.py:40-58
    cos_same = F.cosine_similarity(Et.reshape(N * M, D), U.reshape(N * M, D), dim=1, eps=COS_EPS).reshape(N, M)
    cos_diff = F.cosine_similarity(Et.reshape(N * M, 1, D), C.reshape(1, N, D), dim=2, eps=COS_EPS).reshape(N, M, N)
    idx = torch.arange(N)
    cos_diff = cos_diff.clone()
    cos_diff[idx, :, idx] = cos_same                                            # utils.py:112-113
    S = wt * (cos_diff + COS_BIAS) + bt                                         # utils.py:114, speech_embedder_net.py:45
    if loss == "softmax":
        per = -(S[idx, :, idx] - torch.log(torch.exp(S).sum(dim=2) + LOG_BIAS))  # utils.py:126-130
    else:
        if N < 2:
            raise ValueError("the contrast loss needs at least 2 speakers")
        mask = torch.zeros(N, 1, N, dtype=torch.bool)
        mask[idx, 0, idx] = True
        ks = S.masked_fill(mask, float("-inf")).detach().numpy().argmax(axis=2)  # first arg-max (lowest index)
        sk = torch.gather(S, 2, torch.tensor(ks)[:, :, None])[:, :, 0]
        per = torch.sigmoid(-S[idx, :, idx]) + torch.sigmoid(sk)
    total = per.sum()
    total.backward()
    return dict(loss=total.item(), per=per.detach().numpy(), dE=Et.grad.numpy(), dw=wt.grad.item(), db=bt.grad.item())
