"""TI-SV equal-error-rate sweep: host mirror of train_speech_embedder.py:127-149; exact EER and minDCF over every
score threshold."""
import collections
import math
import numbers

import torch

from . import ops
from .scoring import normalize_sim
from .utils import get_centroids, get_cossim

THRESHOLDS = [0.01 * i + 0.5 for i in range(50)]          # train_speech_embedder.py:134
_thr_cache = {}


def _thresholds_f32(device, thresholds):
    key = (str(device), tuple(thresholds))
    if key not in _thr_cache:
        t = torch.tensor(list(thresholds), dtype=torch.float64).to(torch.float32)   # torch rounds the double to fp32
        if not bool((t[1:] >= t[:-1]).all()):
            raise ValueError("thresholds must be ascending")
        _thr_cache[key] = t.to(device)
    return _thr_cache[key]


def eer_sweep(sim_matrix, thresholds=None):
    """sim_matrix (N, M/2, N) -> (EER, EER_thresh, EER_FAR, EER_FRR) exactly as the loop at
    train_speech_embedder.py:132-149 leaves them: float32 0-dim tensors on sim_matrix's device and the Python
    double threshold, or the integers 0 when no threshold ever satisfied ``diff > |FAR-FRR|``."""
    thresholds = THRESHOLDS if thresholds is None else list(thresholds)
    out_device = sim_matrix.device
    dev = ops._target_device(sim_matrix)
    with torch.cuda.device(dev):
        sim = ops._stage(sim_matrix.detach(), torch.float32, dev)
        thr = _thresholds_f32(sim.device, thresholds)
        if sim.shape[0] == sim.shape[2] and sim.shape[0] >= 2 and len(thresholds) < 64 and sim.shape[1] * sim.shape[2] < (1 << 23):
            out_d, ca, cd = ops.eer_sweep_fused(sim, thr)
            out = out_d.cpu()
            if int(out[1]) == -2:                       # totals beyond 2^24: sequential float32 emulation
                out = ops.eer_finish(ca, cd, sim.shape[1]).cpu()
        else:
            ca, cd = ops.eer_counts(sim, thr)
            out = ops.eer_finish(ca, cd, sim.shape[1]).cpu()
    sel = int(out[1])
    if sel < 0:
        return 0, 0, 0, 0
    return (out[0].clone().to(out_device), thresholds[sel], out[2].clone().to(out_device),
            out[3].clone().to(out_device))


def compute_eer(enrollment_embeddings, verification_embeddings):
    """train_speech_embedder.py:127-149 from the two (N, M/2, D) embedding blocks."""
    enrollment_centroids = get_centroids(enrollment_embeddings)
    sim_matrix = get_cossim(verification_embeddings, enrollment_centroids)
    return eer_sweep(sim_matrix), sim_matrix


# ---------------------------------------------------------------------------- exact EER and minDCF (DESIGN.md 4.5)
MAX_OPERATING_POINTS = 8

VerificationMetrics = collections.namedtuple("VerificationMetrics", [
    "eer", "eer_threshold", "eer_p_miss", "eer_p_fa",
    "min_dcf", "min_dcf_threshold", "min_dcf_p_miss", "min_dcf_p_fa",
    "n_target", "n_nontarget"])
VerificationMetrics.__doc__ = """Exact verification metrics over every score threshold.

eer: (p_miss + p_fa) / 2 at the threshold where miss * Nn - fa * Nt is closest to zero; a trial is accepted when its
score is >= the threshold (+inf: nothing is accepted).  min_dcf and its threshold / p_miss / p_fa are tuples, one entry
per target prior of p_target, in its order.  n_target / n_nontarget: the trial counts."""


def _operating_points(p_target, c_miss, c_fa):
    """-> flat [w_miss, w_fa, c_def] * P in float64, the normalisation of NIST SRE / VoxSRC minDCF."""
    priors = [p_target] if isinstance(p_target, numbers.Real) else list(p_target)
    if not 1 <= len(priors) <= MAX_OPERATING_POINTS:
        raise ValueError(f"p_target must be a float or a sequence of 1 to {MAX_OPERATING_POINTS} floats")
    c_miss, c_fa = float(c_miss), float(c_fa)
    if not (0.0 < c_miss < math.inf and 0.0 < c_fa < math.inf):
        raise ValueError(f"the costs must be positive and finite (c_miss={c_miss}, c_fa={c_fa})")
    ops = []
    for p in priors:
        p = float(p)
        if not 0.0 < p < 1.0:
            raise ValueError(f"every p_target must lie in (0, 1), got {p}")
        w_miss, w_fa = c_miss * p, c_fa * (1.0 - p)
        ops += [w_miss, w_fa, min(w_miss, w_fa)]
    return ops


def _metrics_from_out(out, P):
    v = out.cpu().tolist()
    n_target, n_nontarget, nonfinite = int(v[4]), int(v[5]), int(v[6])
    if nonfinite:
        raise ValueError(f"{nonfinite} score(s) are not finite")
    if n_target == 0 or n_nontarget == 0:
        raise ValueError(f"need at least one target and one non-target trial (got {n_target} targets, "
                         f"{n_nontarget} non-targets)")
    pts = [v[8 + 4 * p: 12 + 4 * p] for p in range(P)]
    return VerificationMetrics(v[0], v[1], v[2], v[3], tuple(p[0] for p in pts), tuple(p[1] for p in pts),
                               tuple(p[2] for p in pts), tuple(p[3] for p in pts), n_target, n_nontarget)


def _check_n(n):
    if n < 2:
        raise ValueError("need at least one target and one non-target trial")
    if n >= 1 << 31:
        raise ValueError(f"at most 2^31 - 1 scores per call, got {n}")


def verification_metrics(scores, labels, p_target=0.01, c_miss=1.0, c_fa=1.0):
    """Exact EER and minDCF of trial scores: ``scores`` (any float dtype, any device) and ``labels`` of the same shape
    (bool or integer, nonzero = target trial).  ``p_target``: one target prior or up to 8 of them.  Higher scores mean
    "same speaker".  Returns VerificationMetrics; raises ValueError on a non-finite score or an empty class."""
    if tuple(scores.shape) != tuple(labels.shape):
        raise ValueError(f"scores {tuple(scores.shape)} and labels {tuple(labels.shape)} differ in shape")
    ops_ = _operating_points(p_target, c_miss, c_fa)
    _check_n(scores.numel())
    dev = ops._target_device(scores, labels)
    with torch.cuda.device(dev):
        s = ops._stage(scores.detach(), torch.float32, dev).reshape(-1)
        lab = labels.detach()
        lab = lab if lab.dtype == torch.bool else lab != 0
        lab = ops._stage(lab, None, dev).reshape(-1).view(torch.uint8)
        out = ops.verif_metrics(s, lab, ops_)
    return _metrics_from_out(out, len(ops_) // 3)


def verification_metrics_from_sim(sim_matrix, p_target=0.01, c_miss=1.0, c_fa=1.0):
    """Exact EER and minDCF of a TI-SV similarity matrix (N, M/2, N) as eer_sweep takes it: element [j, m, k] is a
    target trial iff k == j.  These are the pooled trials of the reference's FAR and FRR, scored at every threshold
    instead of the 50-point grid."""
    if sim_matrix.dim() != 3 or sim_matrix.shape[0] != sim_matrix.shape[2]:
        raise ValueError(f"expected a similarity matrix (N, M, N), got {tuple(sim_matrix.shape)}")
    if sim_matrix.shape[0] < 2:
        raise ValueError("the similarity matrix needs at least 2 speakers (a non-target trial)")
    ops_ = _operating_points(p_target, c_miss, c_fa)
    _check_n(sim_matrix.numel())
    dev = ops._target_device(sim_matrix)
    with torch.cuda.device(dev):
        out = ops.verif_metrics_sim(ops._stage(sim_matrix.detach(), torch.float32, dev), ops_)
    return _metrics_from_out(out, len(ops_) // 3)


def compute_verification_metrics(enrollment_embeddings, verification_embeddings, p_target=0.01, c_miss=1.0, c_fa=1.0,
                                 *, cohort=None, top_k=None):
    """compute_eer's similarity matrix scored exactly: (VerificationMetrics, sim_matrix).  With a ``cohort`` (Nc, D) of
    impostor embeddings the matrix is first S-norm (top_k None) or AS-norm normalized (scoring.normalize_sim), and the
    normalized matrix is returned."""
    enrollment_centroids = get_centroids(enrollment_embeddings)
    sim_matrix = get_cossim(verification_embeddings, enrollment_centroids)
    if cohort is not None:
        sim_matrix = normalize_sim(sim_matrix, enrollment_centroids, verification_embeddings, cohort, top_k)
    return verification_metrics_from_sim(sim_matrix, p_target, c_miss, c_fa), sim_matrix
