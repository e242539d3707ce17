"""Score calibration and calibration metrics, computed on the GPU (csrc/calib.cu, DESIGN.md 4.5.3).

``verification_metrics`` picks its thresholds after seeing the labels.  A deployed verifier fixes its threshold in
advance, so its scores are reported as log-likelihood ratios (LLRs) and judged by the actual DCF at the Bayes threshold
and by Cllr.  ``train_calibration`` fits the linear logistic-regression map llr = scale * s + offset that turns raw or
S-norm scores into LLRs, ``apply_calibration`` applies it and ``calibration_metrics`` scores LLRs:

- cllr: 1/2 [mean over targets of log2(1 + e^-l) + mean over non-targets of log2(1 + e^l)];
- min_cllr: the Cllr left after the best non-decreasing recalibration (PAV, tied scores pooled);
- rocch_eer: the EER of the ROC convex hull;
- act_dcf: the detection cost at the Bayes threshold log(w_fa / w_miss) of each target prior, normalised as
  ``verification_metrics`` normalises minDCF.

Inputs may live on any device and have any float dtype (scores are used as float32); labels are bool or integer,
nonzero = target.  Each call reads its result back once and raises ValueError for a shape mismatch, a non-finite score,
an empty class, a prior outside (0, 1), training data whose classes do not overlap, and a fit that hits ``max_iter``.
"""
import collections
import math
import numbers

import torch

from . import ops
from .eer import _check_n, _operating_points

CalibrationMetrics = collections.namedtuple("CalibrationMetrics", [
    "cllr", "min_cllr", "rocch_eer", "n_target", "n_nontarget",
    "act_dcf", "act_dcf_threshold", "act_dcf_p_miss", "act_dcf_p_fa"])
CalibrationMetrics.__doc__ = """Calibration metrics of LLR scores.  act_dcf and its threshold / p_miss / p_fa are
tuples, one entry per target prior of p_target, in its order; a trial is accepted when its score is >= the threshold."""

Calibration = collections.namedtuple("Calibration", ["scale", "offset", "iterations"])
Calibration.__doc__ = """llr = scale * score + offset; iterations: objective evaluations the fit used."""

_CONVERGED, _SEPARABLE, _ITERATION_CAP, _BAD_INPUT = 0, 1, 2, 3


def _stage(scores, labels):
    if tuple(scores.shape) != tuple(labels.shape):
        raise ValueError(f"scores {tuple(scores.shape)} and labels {tuple(labels.shape)} differ in shape")
    _check_n(scores.numel())
    dev = ops._target_device(scores, labels)
    s = ops._stage(scores.detach(), torch.float32, dev).reshape(-1)
    lab = labels.detach()
    lab = lab if lab.dtype == torch.bool else lab != 0
    return dev, s, ops._stage(lab, None, dev).reshape(-1).view(torch.uint8)


def calibration_metrics(llrs, labels, p_target=0.01, c_miss=1.0, c_fa=1.0):
    """Cllr, minCllr, ROCCH-EER and the actual DCF of LLR scores ``llrs`` with ``labels`` of the same shape.
    ``p_target``: one target prior or up to 8 of them.  Returns CalibrationMetrics."""
    points = _operating_points(p_target, c_miss, c_fa)
    dev, s, lab = _stage(llrs, labels)
    with torch.cuda.device(dev):
        v = ops.calib_metrics(s, lab, points).cpu().tolist()
    n_target, n_nontarget, nonfinite = int(v[3]), int(v[4]), int(v[5])
    if nonfinite:
        raise ValueError(f"{nonfinite} score(s) are not finite")
    if n_target == 0 or n_nontarget == 0:
        raise ValueError(f"need at least one target and one non-target trial (got {n_target} targets, "
                         f"{n_nontarget} non-targets)")
    pts = [v[8 + 4 * p: 12 + 4 * p] for p in range(len(points) // 3)]
    return CalibrationMetrics(v[0], v[1], v[2], n_target, n_nontarget, tuple(p[0] for p in pts),
                              tuple(p[1] for p in pts), tuple(p[2] for p in pts), tuple(p[3] for p in pts))


def train_calibration(scores, labels, prior=0.5, max_iter=100):
    """Linear logistic-regression calibration at target prior ``prior``: the (scale, offset) minimising
    prior * mean_tar softplus(-(l + logit(prior))) + (1 - prior) * mean_non softplus(l + logit(prior)) with
    l = scale * s + offset.  Damped Newton from (0, 0), at most ``max_iter`` objective evaluations.  Returns
    Calibration."""
    prior = float(prior)
    if not 0.0 < prior < 1.0:
        raise ValueError(f"prior must lie in (0, 1), got {prior}")
    if isinstance(max_iter, bool) or not isinstance(max_iter, numbers.Integral) or max_iter < 1:
        raise ValueError(f"max_iter must be a positive integer, got {max_iter!r}")
    dev, s, lab = _stage(scores, labels)
    with torch.cuda.device(dev):
        a, b, _, iters, status = ops.calib_train(s, lab, prior, int(max_iter)).cpu().tolist()
    status = int(status)
    if status == _BAD_INPUT:
        raise ValueError("every score must be finite and both classes non-empty")
    if status == _SEPARABLE:
        raise ValueError("the target and non-target scores do not overlap (or take a single value): the likelihood "
                         "has no finite maximum")
    if status == _ITERATION_CAP:
        raise ValueError(f"the calibration fit did not converge in max_iter = {max_iter} objective evaluations")
    return Calibration(a, b, int(iters))


def apply_calibration(scores, calibration):
    """scale * scores + offset in float64, rounded once to float32, on the scores' device."""
    if not (math.isfinite(calibration.scale) and math.isfinite(calibration.offset)):
        raise ValueError(f"calibration parameters must be finite, got {calibration}")
    s = scores.detach().to(torch.float32).to(torch.float64)
    return (s * calibration.scale + calibration.offset).to(torch.float32)
