"""The float64 oracle (oracle.embedder.embedder_explicit) at every model shape of tests/_embedder_shapes.py, against
torch.nn.LSTM + nn.Linear + L2 norm in float64: forward and the autograd gradient of every parameter.

The golden fixtures pin the oracle at the default dimensions only (40 / 768 / 3 / 256); this is what lets the GPU
shape tests trust it at one, two and four layers, odd nmels and a projection width that is not a multiple of 32.
Biases are nonzero here (nn.LSTM's default init), so the b_ih + b_hh sum of the oracle is exercised too.
"""
import numpy as np
import pytest
import torch
import torch.nn as nn

from _embedder_shapes import CASES, param_names
from oracle import embedder as oemb


def rel_l2(a, b):
    a = a.detach().double().ravel()
    b = b.detach().double().ravel()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_oracle_matches_torch_lstm_in_float64(case):
    I, H, L, P = case.nmels, case.hidden, case.num_layer, case.proj
    B, T = 3, 5
    torch.manual_seed(1000 + I + H + L + P)
    lstm = nn.LSTM(I, H, num_layers=L, batch_first=True).double()
    lin = nn.Linear(H, P).double()
    x = torch.randn(B, T, I, dtype=torch.float64) * 1.5 - 3.0
    v = torch.randn(B, P, dtype=torch.float64)

    y, _ = lstm(x)
    y = lin(y[:, T - 1])
    e_lib = y / torch.norm(y, dim=1).unsqueeze(1)
    (e_lib * v).sum().backward()
    lib_grads = {f"LSTM_stack.{k}": p.grad for k, p in lstm.named_parameters()}
    lib_grads["projection.weight"] = lin.weight.grad
    lib_grads["projection.bias"] = lin.bias.grad

    sd = {f"LSTM_stack.{k}": p.detach().clone().requires_grad_(True) for k, p in lstm.named_parameters()}
    sd["projection.weight"] = lin.weight.detach().clone().requires_grad_(True)
    sd["projection.bias"] = lin.bias.detach().clone().requires_grad_(True)
    e = oemb.embedder_explicit(x, sd, num_layer=L, keep_f64=True)
    assert e.dtype == torch.float64 and e.shape == (B, P)
    (e * v).sum().backward()

    assert rel_l2(e, e_lib) < 1e-10, rel_l2(e, e_lib)
    names = param_names(L)
    assert sorted(names) == sorted(lib_grads)
    for k in names:
        assert sd[k].grad is not None and lib_grads[k] is not None, k
        assert float(lib_grads[k].norm()) > 0, k
        assert rel_l2(sd[k].grad, lib_grads[k]) < 1e-10, (k, rel_l2(sd[k].grad, lib_grads[k]))


def test_oracle_weight_hh_gradient_is_zero_at_one_frame():
    """h_{-1} = 0, so with T = 1 the recurrent weights receive exactly no gradient: the GPU test holds the kernels to
    exact zeros there instead of a relative bar."""
    torch.manual_seed(7)
    lstm = nn.LSTM(13, 128, num_layers=2, batch_first=True).double()
    lin = nn.Linear(128, 32).double()
    sd = {f"LSTM_stack.{k}": p.detach().clone().requires_grad_(True) for k, p in lstm.named_parameters()}
    sd["projection.weight"] = lin.weight.detach().clone().requires_grad_(True)
    sd["projection.bias"] = lin.bias.detach().clone().requires_grad_(True)
    x = torch.randn(4, 1, 13, dtype=torch.float64)
    oemb.embedder_explicit(x, sd, num_layer=2, keep_f64=True).sum().backward()
    for l in range(2):
        g = sd[f"LSTM_stack.weight_hh_l{l}"].grad
        assert g is not None and np.count_nonzero(g.numpy()) == 0
        assert float(sd[f"LSTM_stack.weight_ih_l{l}"].grad.norm()) > 0
