"""Drop-in for the reference's speech_embedder_net.py: SpeechEmbedder and GE2ELoss (same constructor
signatures, attribute names, parameter order and state_dict keys), computed by hand-written sm_100a kernels.
"""
import torch
import torch.nn as nn

from . import hparam as _hp
from . import ops
from .utils import calc_loss, get_centroids, get_cossim  # noqa: F401  (re-exported like speech_embedder_net.py:13)


class SpeechEmbedder(nn.Module):
    """3-layer LSTM(nmels -> hidden) + Linear(hidden -> proj) on the last frame + L2 norm
    (speech_embedder_net.py:15-33).  ``LSTM_stack`` is a real nn.LSTM used purely as the parameter container, so
    initialisation (RNG order), ``state_dict`` keys/shapes and checkpoints are identical to the reference's; its
    own forward (cuDNN/oneDNN) is never called."""

    def __init__(self, nmels=None, hidden=None, num_layer=None, proj=None):
        super(SpeechEmbedder, self).__init__()
        d = _hp.model_dims()
        nmels, hidden = nmels or d[0], hidden or d[1]
        num_layer, proj = num_layer or d[2], proj or d[3]
        self.LSTM_stack = nn.LSTM(nmels, hidden, num_layers=num_layer, batch_first=True)
        for name, param in self.LSTM_stack.named_parameters():
            if 'bias' in name:
                nn.init.constant_(param, 0.0)
            elif 'weight' in name:
                nn.init.xavier_normal_(param)
        self.projection = nn.Linear(hidden, proj)
        self._dims = (nmels, hidden, num_layer, proj)
        self._cache = ops.PackedWeights()
        # Split-bf16 terms of the recurrent GEMM: 1 (h_hi W_hi) holds the 1e-3 embedding tolerance for the
        # reference initialisation; 3 (+ h_hi W_lo + h_lo W_hi) is near-fp32 for large-magnitude weights.
        self.recurrent_terms = 1

    def _ordered_params(self):
        ps = []
        for l in range(self._dims[2]):
            for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"):
                ps.append(getattr(self.LSTM_stack, f"{k}_l{l}"))
        return ps + [self.projection.weight, self.projection.bias]

    def repack(self):
        """Rebuild the fp16/bf16 weight shadows on the next call.  Only needed after in-place surgery that bypasses
        autograd's version counter (``p.data.copy_()``, ``p.data.add_()``); optimizers, ``load_state_dict`` and
        ``.to()`` / ``.cpu()`` are detected automatically."""
        self._cache.invalidate()

    def forward(self, x):
        return ops.embedder_forward(x, self._cache, (*self._dims, int(self.recurrent_terms)), self._ordered_params())


class GE2ELoss(nn.Module):
    """GE2E loss with learnable w, b (speech_embedder_net.py:35-49).  ``loss_method``: "softmax" (default, the
    reference's loss, Wan et al. eq. 6) or "contrast" (eq. 7: 1 - sigmoid(S_jj) + sigmoid of the most similar other
    centroid, summed over the embeddings).  Like ``fused``, it is a plain attribute: ``state_dict`` holds w and b only."""

    def __init__(self, device, loss_method="softmax"):
        super(GE2ELoss, self).__init__()
        ops.loss_code(loss_method)                       # ValueError for an unknown method
        self.w = nn.Parameter(torch.tensor(10.0).to(device), requires_grad=True)
        self.b = nn.Parameter(torch.tensor(-5.0).to(device), requires_grad=True)
        self.device = device
        self.fused = True
        self.loss_method = loss_method

    def forward(self, embeddings):
        # speech_embedder_net.py:44 `torch.clamp(self.w, 1e-6)` discards its result: w is NOT clamped.
        return ops.ge2e_loss(embeddings, self.w, self.b, int(self.fused), self.loss_method)
