"""Float64 get_cossim (utils.py:72-115) in matmul form, with its gradient, for shapes where oracle.ge2e.get_cossim's
(N, M, Nc, D) broadcast does not fit in memory (the C5 similarity matrix: 6.4 GB of float64) and which it has no
gradient for.

The restatement: rows of E and C normalised (each norm clamped at 1e-8 on its own, as F.cosine_similarity does),
cos = E^ C^T, column j of speaker j's rows replaced by the cosine to the leave-one-out centroid of speaker j's
utterances, then + 1e-6.  tests/test_oracle_ge2e_routes.py pins it, values and gradient, to oracle.ge2e.get_cossim.
"""
import numpy as np
import torch

from oracle.ge2e import COS_BIAS, COS_EPS


def _unit(x):
    return x / torch.clamp(torch.linalg.vector_norm(x, dim=-1, keepdim=True), min=COS_EPS)


def cossim_t(E, C):
    """get_cossim(E (N, M, D), C (Nc, D)), Nc >= N, on float64 torch tensors (differentiable)."""
    N, M, D = E.shape
    U = (E.sum(dim=1, keepdim=True) - E) / (M - 1)
    Eh = _unit(E)
    cosd = (Eh * _unit(U)).sum(-1)                                     # (N, M)
    cos = (Eh.reshape(N * M, D) @ _unit(C).T).reshape(N, M, C.shape[0])
    own = torch.zeros(N, 1, C.shape[0], dtype=torch.bool)
    own[torch.arange(N), 0, torch.arange(N)] = True
    return torch.where(own, cosd[:, :, None], cos) + COS_BIAS


def cossim(E, C):
    """get_cossim(E, C) as float64 numpy."""
    with torch.no_grad():
        return cossim_t(torch.as_tensor(np.asarray(E, dtype=np.float64)),
                        torch.as_tensor(np.asarray(C, dtype=np.float64))).numpy()


def cossim_grads(E, C, V):
    """-> (cos, dE, dC): get_cossim(E, C) and the gradient of (cos * V).sum() w.r.t. E and C (C an independent input),
    float64 numpy, by torch autograd through the restatement."""
    Et = torch.tensor(np.asarray(E, dtype=np.float64), requires_grad=True)
    Ct = torch.tensor(np.asarray(C, dtype=np.float64), requires_grad=True)
    cos = cossim_t(Et, Ct)
    (cos * torch.as_tensor(np.asarray(V, dtype=np.float64))).sum().backward()
    return cos.detach().numpy(), Et.grad.numpy(), Ct.grad.numpy()
