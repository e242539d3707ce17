"""Cohort score normalization of cosine trial scores: S-norm and adaptive S-norm (AS-norm), computed on the GPU
(csrc/asnorm.cu, DESIGN.md 4.5.2).

The statistics of a row x against a cohort of Nc impostor embeddings with top-K (2 <= K <= Nc, default K = Nc, plain
S-norm) are the mean and the sample standard deviation (divisor K - 1) of the K largest cosines cos(x, c).  A trial
(e, t) with cosine s scores 1/2 ((s - mean(e)) / std(e) + (s - mean(t)) / std(t)).  Statistics are float64, scores
float32 (what ``verification_metrics`` consumes).  The functions accept CPU and float64 inputs, run on the GPU and return
on the caller's device.  They raise ValueError for mismatched dimensions, a K outside [2, Nc], a cohort of fewer than
two rows, an index out of range, a non-finite input or statistic (a zero-norm row has no cosine) and a zero std.
"""
import numbers

import torch

from . import ops


def _top_k(top_k, Nc):
    if Nc < 2:
        raise ValueError(f"the cohort needs at least 2 rows, got {Nc}")
    if top_k is None:
        return Nc
    if isinstance(top_k, bool) or not isinstance(top_k, numbers.Integral):
        raise ValueError(f"top_k must be an integer or None, got {top_k!r}")
    if not 2 <= int(top_k) <= Nc:
        raise ValueError(f"top_k must lie in [2, {Nc}] (the cohort size), got {top_k}")
    return int(top_k)


def _rows(x, what):
    if x.dim() != 2:
        raise ValueError(f"{what} must be a matrix (rows, D), got shape {tuple(x.shape)}")
    return x


def _check(flags, messages):
    """One host read of every validity flag; raises the first failed check's message."""
    ok = torch.stack(flags).cpu().tolist()
    for good, msg in zip(ok, messages):
        if not good:
            raise ValueError(msg)


def _stats_flags(stats, what):
    finite = torch.isfinite(stats).all()
    return ([finite, (stats[:, 1] > 0).all()],
            [f"non-finite cohort statistic of the {what}: a row or cohort score is not finite, or a row has zero norm",
             f"zero cohort std of the {what}: every selected cohort score of a row is equal"])


def _input_flags(tensors, names):
    return [torch.isfinite(t).all() for t in tensors], [f"{n} contains a non-finite value" for n in names]


def cohort_stats(embeddings, cohort, top_k=None):
    """(mean, std) of every row of ``embeddings`` (n, D) against ``cohort`` (Nc, D): float64 tensors (n,) on the
    embeddings' device.  ``top_k``: K of AS-norm, None = Nc (S-norm)."""
    _rows(embeddings, "embeddings")
    _rows(cohort, "cohort")
    if embeddings.shape[1] != cohort.shape[1]:
        raise ValueError(f"embeddings have D = {embeddings.shape[1]}, the cohort D = {cohort.shape[1]}")
    K = _top_k(top_k, cohort.shape[0])
    out_device = embeddings.device
    dev = ops._target_device(embeddings, cohort)
    with torch.cuda.device(dev):
        X = ops._stage(embeddings.detach(), torch.float32, dev)
        C = ops._stage(cohort.detach(), torch.float32, dev)
        st = ops.cohort_stats(X, C, K)
        f1, m1 = _input_flags([X, C], ["embeddings", "cohort"])
        f2, m2 = _stats_flags(st, "embeddings")
        _check(f1 + f2, m1 + m2)
    return ops._back(st[:, 0], out_device), ops._back(st[:, 1], out_device)


def score_trials(enrollment, test, enroll_idx, test_idx, cohort=None, top_k=None):
    """float32 scores of the trials (enrollment[enroll_idx[i]], test[test_idx[i]]): raw cosines without a cohort,
    S-norm (top_k None) or AS-norm scores with one.  enrollment (ne, D), test (nt, D), integer index vectors of one
    length.  Returned on the enrollment's device."""
    _rows(enrollment, "enrollment")
    _rows(test, "test")
    if enrollment.shape[1] != test.shape[1]:
        raise ValueError(f"enrollment has D = {enrollment.shape[1]}, test D = {test.shape[1]}")
    for idx, name in ((enroll_idx, "enroll_idx"), (test_idx, "test_idx")):
        if idx.dtype.is_floating_point or idx.dtype.is_complex or idx.dtype == torch.bool or idx.dim() != 1:
            raise ValueError(f"{name} must be a 1-D integer tensor")
    if enroll_idx.shape != test_idx.shape:
        raise ValueError(f"enroll_idx {tuple(enroll_idx.shape)} and test_idx {tuple(test_idx.shape)} differ in length")
    if enrollment.shape[0] < 1 or test.shape[0] < 1:
        raise ValueError("enrollment and test need at least one row each")
    if cohort is not None:
        _rows(cohort, "cohort")
        if cohort.shape[1] != enrollment.shape[1]:
            raise ValueError(f"the cohort has D = {cohort.shape[1]}, the embeddings D = {enrollment.shape[1]}")
        K = _top_k(top_k, cohort.shape[0])
    out_device = enrollment.device
    dev = ops._target_device(enrollment, test, enroll_idx, test_idx, cohort)
    with torch.cuda.device(dev):
        E = ops._stage(enrollment.detach(), torch.float32, dev)
        T = ops._stage(test.detach(), torch.float32, dev)
        ei = ops._stage(enroll_idx.detach(), None, dev)
        ti = ops._stage(test_idx.detach(), None, dev)
        flags = [((ei >= 0) & (ei < E.shape[0])).all(), ((ti >= 0) & (ti < T.shape[0])).all()]
        msgs = [f"enroll_idx out of range [0, {E.shape[0]})", f"test_idx out of range [0, {T.shape[0]})"]
        f, m = _input_flags([E, T], ["enrollment", "test"])
        flags, msgs = flags + f, msgs + m
        se = st = None
        if cohort is not None:
            C = ops._stage(cohort.detach(), torch.float32, dev)
            se, st = ops.cohort_stats(E, C, K), ops.cohort_stats(T, C, K)
            f, m = _input_flags([C], ["cohort"])
            flags, msgs = flags + f, msgs + m
            for s, what in ((se, "enrollment"), (st, "test")):
                f, m = _stats_flags(s, what)
                flags, msgs = flags + f, msgs + m
        out = ops.score_trials(E, T, ei.to(torch.int32), ti.to(torch.int32), se, st)
        flags.append(torch.isfinite(out).all())
        msgs.append("a trial score is not finite (a row has zero norm)")
        _check(flags, msgs)
    return ops._back(out, out_device)


def normalize_sim(sim_matrix, enrollment_centroids, verification_embeddings, cohort, top_k=None):
    """The TI-SV similarity matrix (N, M, N) of get_cossim / eer_sweep normalized against ``cohort`` (Nc, D):
    out[j, m, k] = 1/2 ((sim - mean_c[k]) / std_c[k] + (sim - mean_v[j, m]) / std_v[j, m]), the centroids (N, D)
    being the enrollment side and the verification utterances (N, M, D) the test side.  float32, on sim's device."""
    if sim_matrix.dim() != 3 or sim_matrix.shape[0] != sim_matrix.shape[2]:
        raise ValueError(f"expected a similarity matrix (N, M, N), got {tuple(sim_matrix.shape)}")
    N, M = sim_matrix.shape[0], sim_matrix.shape[1]
    _rows(enrollment_centroids, "enrollment_centroids")
    _rows(cohort, "cohort")
    D = cohort.shape[1]
    if tuple(enrollment_centroids.shape) != (N, D):
        raise ValueError(f"enrollment_centroids {tuple(enrollment_centroids.shape)}: expected ({N}, {D})")
    if tuple(verification_embeddings.shape) != (N, M, D):
        raise ValueError(f"verification_embeddings {tuple(verification_embeddings.shape)}: expected ({N}, {M}, {D})")
    K = _top_k(top_k, cohort.shape[0])
    out_device = sim_matrix.device
    dev = ops._target_device(sim_matrix, enrollment_centroids, verification_embeddings, cohort)
    with torch.cuda.device(dev):
        sim = ops._stage(sim_matrix.detach(), torch.float32, dev)
        Cen = ops._stage(enrollment_centroids.detach(), torch.float32, dev)
        V = ops._stage(verification_embeddings.detach(), torch.float32, dev).reshape(N * M, D)
        C = ops._stage(cohort.detach(), torch.float32, dev)
        sc, sv = ops.cohort_stats(Cen, C, K), ops.cohort_stats(V, C, K)
        flags, msgs = _input_flags([sim, Cen, V, C], ["sim_matrix", "enrollment_centroids",
                                                      "verification_embeddings", "cohort"])
        for s, what in ((sc, "enrollment centroids"), (sv, "verification embeddings")):
            f, m = _stats_flags(s, what)
            flags, msgs = flags + f, msgs + m
        _check(flags, msgs)
        out = ops.asnorm_sim(sim, sc, sv)
    return ops._back(out, out_device)
