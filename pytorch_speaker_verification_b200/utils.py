"""Drop-in for the loss math of the reference's utils.py (lines 27-29, 40-58, 72-115, 126-132).

Same names, argument meaning and return types; the arithmetic runs in the CUDA kernels of csrc/ge2e.cu behind the
``torch.ops.svb200`` custom ops (no CPU path).  All four functions are differentiable like the reference's.
"""
from . import ops


def get_centroids(embeddings):
    """(N, M, D) -> (N, D): mean over each speaker's utterances (utils.py:27-29)."""
    return ops.get_centroids(embeddings)


def get_utterance_centroids(embeddings):
    """(N, M, D) -> (N, M, D) leave-one-out centroids (utils.py:40-58): (sum over the speaker's utterances - the
    utterance itself) / (M - 1), the reference's float32 operations in the reference's order."""
    return ops.get_utterance_centroids(embeddings)


def get_cossim(embeddings, centroids):
    """(N, M, D), (N, D) -> (N, M, N) cosine similarity + 1e-6 with the diagonal computed against the
    leave-one-out centroid of ``embeddings`` (utils.py:72-115), also when ``centroids`` is foreign
    (train_speech_embedder.py:129)."""
    return ops.get_cossim(embeddings, centroids)


def calc_loss(sim_matrix, loss_method="softmax"):
    """(N, M, N) -> (loss, per_embedding_loss (N, M)); loss is the SUM over rows (utils.py:126-132).
    ``loss_method="contrast"``: the GE2E contrast loss (Wan et al. eq. 7) instead of the softmax loss (eq. 6)."""
    return ops.calc_loss(sim_matrix, loss_method)
