"""Oracle (test infrastructure): SpeechEmbedder restated on the CPU.

Follows /root/reference/speech_embedder_net.py:15-33:
  :19    nn.LSTM(nmels, hidden, num_layers, batch_first=True)  gate order i,f,g,o; h0=c0=0
  :20-24 biases 0, LSTM weights xavier_normal_
  :25    nn.Linear(hidden, proj) default init
  :28    x.float() -> LSTM            :30 last frame only
  :31    projection                   :32 x / ||x||_2 (no epsilon)

The LSTM arithmetic itself lives in third-party torch (aten::lstm -> oneDNN on CPU,
cuDNN on CUDA); ``lstm_explicit`` restates the published cell equations
    g_t = W_ih x_t + b_ih + W_hh h_{t-1} + b_hh      (rows i|f|g|o)
    c_t = sig(f) c_{t-1} + sig(i) tanh(g);   h_t = sig(o) tanh(c_t)
with plain matmuls so that autograd yields the BPTT gradients.  tests/golden pins it
against the reference's nn.LSTM.

``ReferenceLibraryStep`` calls the same torch library entry points the reference calls
(nn.LSTM / nn.Linear / F.cosine_similarity / clip_grad_norm_ / SGD); it is what
bench.py times as the CPU baseline.

``Emu`` lets tests/experiments emulate the CUDA path's operand rounding (bf16 operands,
fp32 accumulate) to budget the 1e-3 embedding tolerance.
"""
from dataclasses import dataclass

import torch
import torch.nn as nn
import torch.nn.functional as F

PARAM_NAMES = [f"LSTM_stack.{k}_l{l}" for l in range(3)
               for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")] + \
              ["projection.weight", "projection.bias"]


def init_state_dict(nmels=40, hidden=768, num_layer=3, proj=256, seed=0):
    """Same RNG consumption order as speech_embedder_net.py:17-25 under torch.manual_seed(seed)."""
    torch.manual_seed(seed)
    lstm = nn.LSTM(nmels, hidden, num_layers=num_layer, batch_first=True)
    for name, param in lstm.named_parameters():
        if 'bias' in name:
            nn.init.constant_(param, 0.0)
        elif 'weight' in name:
            nn.init.xavier_normal_(param)
    lin = nn.Linear(hidden, proj)
    sd = {f"LSTM_stack.{k}": v.detach().clone() for k, v in lstm.state_dict().items()}
    sd["projection.weight"] = lin.weight.detach().clone()
    sd["projection.bias"] = lin.bias.detach().clone()
    return sd


@dataclass
class Emu:
    """Which operands are rounded to bf16 (hi), to a hi+lo bf16 pair ("split") or to fp16 (the operand format of the
    forward GEMMs)."""
    x_in: str = "fp32"      # activations entering the input-projection GEMM: fp32|bf16|split|fp16
    w_in: str = "fp32"      # W_ih
    h_rec: str = "fp32"     # h_{t-1} entering the recurrent GEMM
    w_rec: str = "fp32"     # W_hh
    gin_store: str = "fp32" # storage of the input-projection output


def _rnd(t, mode):
    if mode == "fp32":
        return t
    if mode == "fp16":
        return t.to(torch.float16).to(t.dtype)
    hi = t.to(torch.bfloat16).to(t.dtype)
    if mode == "bf16":
        return hi
    if mode == "split":
        lo = (t - hi).to(torch.bfloat16).to(t.dtype)
        return hi + lo
    raise ValueError(mode)


def lstm_explicit(x, sd, num_layer=3, emu=None, return_all=False):
    """x (B,T,I) -> top-layer h sequence (B,T,H) (or list per layer)."""
    emu = emu or Emu()
    inp = x
    outs = []
    for l in range(num_layer):
        w_ih = sd[f"LSTM_stack.weight_ih_l{l}"].to(x.dtype)
        w_hh = sd[f"LSTM_stack.weight_hh_l{l}"].to(x.dtype)
        bias = (sd[f"LSTM_stack.bias_ih_l{l}"] + sd[f"LSTM_stack.bias_hh_l{l}"]).to(x.dtype)
        H = w_hh.shape[1]
        B, T, _ = inp.shape
        gin = _rnd(inp, emu.x_in) @ _rnd(w_ih, emu.w_in).t() + bias          # (B,T,4H)
        gin = _rnd(gin, emu.gin_store)
        w_hh_r = _rnd(w_hh, emu.w_rec).t()
        h = x.new_zeros(B, H)
        c = x.new_zeros(B, H)
        hs = []
        for t in range(T):
            g = gin[:, t] + _rnd(h, emu.h_rec) @ w_hh_r
            i, f, gg, o = g.split(H, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            hs.append(h)
        inp = torch.stack(hs, dim=1)
        outs.append(inp)
    return outs if return_all else inp


def embedder_explicit(x, sd, emu=None, num_layer=3, keep_f64=False):
    """speech_embedder_net.py:27-33 with the explicit LSTM.  Like the reference (:28
    ``x.float()``) any input is computed in float32 unless keep_f64 asks for the
    high-precision oracle on a float64 input."""
    dt = torch.float64 if (keep_f64 and x.dtype == torch.float64) else torch.float32
    x = x.to(dt)
    y = lstm_explicit(x, sd, num_layer=num_layer, emu=emu)
    y = y[:, y.size(1) - 1]
    y = y @ sd["projection.weight"].to(dt).t() + sd["projection.bias"].to(dt)
    return y / torch.norm(y, dim=1).unsqueeze(1)


class LibraryEmbedder(nn.Module):
    """The third-party calls of speech_embedder_net.py:15-33 (nn.LSTM + nn.Linear)."""

    def __init__(self, nmels=40, hidden=768, num_layer=3, proj=256):
        super().__init__()
        self.LSTM_stack = nn.LSTM(nmels, hidden, num_layers=num_layer, batch_first=True)
        for name, param in self.LSTM_stack.named_parameters():
            if 'bias' in name:
                nn.init.constant_(param, 0.0)
            elif 'weight' in name:
                nn.init.xavier_normal_(param)
        self.projection = nn.Linear(hidden, proj)

    def forward(self, x):
        x, _ = self.LSTM_stack(x.float())
        x = x[:, x.size(1) - 1]
        x = self.projection(x.float())
        return x / torch.norm(x, dim=1).unsqueeze(1)


def library_ge2e_loss(E, w, b):
    """utils.py:27-29,40-58,72-115,126-132 + speech_embedder_net.py:43-49 as torch calls
    (kept op-for-op so that the CPU baseline pays what the reference pays, including the
    two repeat() expansions of utils.py:99-104)."""
    N, M, D = E.shape
    C = E.mean(dim=1)
    U = (E.sum(dim=1).reshape(N, 1, D) - E) / (M - 1)
    Ef = E.reshape(N * M, D)
    cos_same = F.cosine_similarity(Ef, U.reshape(N * M, D))
    C_exp = C.repeat((M * N, 1))
    E_exp = Ef.unsqueeze(1).repeat(1, N, 1).reshape(N * M * N, D)
    cos = F.cosine_similarity(E_exp, C_exp).view(N, M, N)
    idx = list(range(N))
    cos[idx, :, idx] = cos_same.view(N, M)
    cos = cos + 1e-6
    S = w * cos + b
    pos = S[idx, :, idx]
    neg = (torch.exp(S).sum(dim=2) + 1e-6).log_()
    return (-1 * (pos - neg)).sum()


class ReferenceLibraryStep:
    """One training step as train_speech_embedder.py:45-65 runs it on the CPU."""

    def __init__(self, N, M, lr=0.01, seed=0):
        torch.manual_seed(seed)
        self.N, self.M = N, M
        self.net = LibraryEmbedder()
        self.w = nn.Parameter(torch.tensor(10.0))
        self.b = nn.Parameter(torch.tensor(-5.0))
        self.opt = torch.optim.SGD([{'params': self.net.parameters()},
                                    {'params': [self.w, self.b]}], lr=lr)

    def step(self, batch):
        """batch (N*M, T, 40) float32 on the CPU."""
        self.opt.zero_grad()
        emb = self.net(batch).reshape(self.N, self.M, -1)
        loss = library_ge2e_loss(emb, self.w, self.b)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.net.parameters(), 3.0)
        torch.nn.utils.clip_grad_norm_([self.w, self.b], 1.0)
        self.opt.step()
        return float(loss)
