"""GPU: cohort score normalization (csrc/asnorm.cu) against the float64 restatement (tests/_asnorm_oracle.py).

From scores the selection is exact: v_K must equal the oracle (==) and the float64 mean / std agree to 1e-12.  From
embeddings the cohort cosines are 3-term split-fp16 tensor-core products (about 2^-22 relative), so the mean and std
are held to bars measured on the B200 (see DESIGN.md 4.5.2); v_K is not compared there, because a near-tie at the K-th
position may swap, which moves the mean by at most |gap| / K."""
import ctypes

import numpy as np
import pytest
import torch

import _asnorm_oracle as A
import _inputs as I
import pytorch_speaker_verification_b200 as svb
from pytorch_speaker_verification_b200 import _lib

pytestmark = pytest.mark.gpu

# bars of the tensor-core route (DESIGN.md 4.5.2: about 3x the worst error measured on the B200)
COS_BAR = 2e-6          # cohort cosine (absolute; worst measured 6.0e-7, D = 512)
MEAN_BAR = 1.5e-6       # mean of the top-K cohort cosines (absolute; worst measured 4.8e-7, D = 512, K = 10)
STD_BAR = 1e-4          # std of the top-K cohort cosines (relative; worst measured 2.5e-5, D = 512, K = 10)
SCORE_BAR = 1e-5        # normalized score, |error| / (1 + |score|), worst measured 2.9e-6: the std's error scales the z-score


def score_err(got, ref):
    return (np.abs(np.asarray(got, np.float64) - ref) / (1 + np.abs(ref))).max()


def chunk_rows(Nc):
    """Rows per chunk of svb_cohort_stats (csrc/asnorm.cu chunk_rows at the default 48 MB slab)."""
    Ncp = (Nc + 7) // 8 * 8
    return max(128, (48 << 20) // (Ncp * 4) // 128 * 128)


def raw_stats(S, K):
    return torch.ops.svb200.cohort_stats_scores(S, K).cpu().numpy()


def check_exact(S, K):
    """S: CUDA float32 (n, Nc) (any row pitch)."""
    got = raw_stats(S, K)
    ref = A.stats_from_scores(S.cpu().numpy(), K)
    np.testing.assert_array_equal(got[:, 2], ref[:, 2])
    scale = np.abs(S.cpu().numpy().astype(np.float64)).max(axis=1)
    assert (np.abs(got[:, 0] - ref[:, 0]) <= 1e-12 * scale).all()
    assert (np.abs(got[:, 1] - ref[:, 1]) <= 1e-12 * ref[:, 1]).all()
    return got


def clustered(n, D, seed, spread=0.6):
    """Trained-like unit embeddings: a shared component plus a per-row direction (cosines mostly in [-0.2, 0.8])."""
    r = np.random.RandomState(seed)
    g = r.standard_normal(D)
    x = spread * r.standard_normal((n, D)) / np.sqrt(D) + g / np.linalg.norm(g) * 0.5
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


# ------------------------------------------------------------------------------------------------- from scores, exact
@pytest.mark.parametrize("Nc", [2, 3, 31, 300, 4097, 6000, 65537])
@pytest.mark.parametrize("kk", ["2", "7", "Nc"])
def test_stats_from_scores_exact(Nc, kk):
    K = {"2": 2, "7": 7, "Nc": Nc}[kk]
    if K > Nc:
        pytest.skip("K > Nc")
    n = 3 if Nc > 10000 else 257
    r = np.random.RandomState(Nc + K)
    S = np.clip(r.standard_normal((n, Nc)) * 0.3 + 0.2, -1, 1).astype(np.float32)
    check_exact(torch.tensor(S).cuda(), K)


@pytest.mark.parametrize("n", [1, 2, 3000])
def test_stats_rows(n):
    r = np.random.RandomState(n)
    check_exact(torch.tensor(r.standard_normal((n, 1000)).astype(np.float32)).cuda(), 100)


@pytest.mark.parametrize("case", ["rounded", "two_values", "specials", "all_equal_but_one"])
@pytest.mark.parametrize("Nc", [300, 20000])
def test_stats_ties_and_special_values(case, Nc):
    r = np.random.RandomState(7)
    n = 64
    if case == "rounded":
        S = np.round(r.standard_normal((n, Nc)) * 0.3, 2)
    elif case == "two_values":
        S = np.where(r.rand(n, Nc) < 0.1, 0.375, -0.125)
    elif case == "specials":
        vals = np.array([0.0, -0.0, 1.0, -1.0, 1e-40, -1e-40, 1.4e-45, -1.4e-45, 0.5, -0.5], np.float32)
        S = vals[r.randint(len(vals), size=(n, Nc))]
    else:
        S = np.full((n, Nc), 0.25)
        S[:, 5] = 0.75
    S = S.astype(np.float32)
    for K in (2, 7, 150, Nc):
        check_exact(torch.tensor(S).cuda(), K)


def test_stats_row_pitch_larger_than_the_cohort():
    r = np.random.RandomState(9)
    wide = torch.tensor(r.standard_normal((100, 1300)).astype(np.float32)).cuda()
    S = wide[:, 3:1003]
    assert S.stride(0) == 1300
    check_exact(S, 50)


def test_non_finite_score_gives_nan_statistics():
    r = np.random.RandomState(4)
    S = r.standard_normal((4, 500)).astype(np.float32)
    S[1, 17] = np.nan
    S[2, 400] = np.inf
    S[3, 0] = -np.inf
    got = raw_stats(torch.tensor(S).cuda(), 10)
    assert np.isfinite(got[0]).all() and np.isnan(got[1:]).all()


# ------------------------------------------------------------------------------------ from embeddings (tensor cores)
def embedding_errors(X, C, K):
    st = torch.ops.svb200.cohort_stats(torch.tensor(X).cuda(), torch.tensor(C).cuda(), K).cpu().numpy()
    ref = A.stats(X, C, K)
    return np.abs(st[:, 0] - ref[:, 0]).max(), (np.abs(st[:, 1] - ref[:, 1]) / ref[:, 1]).max(), st, ref


def test_tensor_core_cohort_cosines():
    """With two cohort rows and K = 2, v_K = the smaller cosine: the GEMM's error on its own."""
    for D in (13, 100, 256, 512):
        X = clustered(3000, D, D)
        C = clustered(2, D, D + 1)
        st = torch.ops.svb200.cohort_stats(torch.tensor(X).cuda(), torch.tensor(C).cuda(), 2).cpu().numpy()
        ref = A.cosine(X, C).min(axis=1)
        err = np.abs(st[:, 2] - ref).max()
        print(f"asnorm cohort cosine D={D}: worst abs error {err:.3e}")
        assert err < COS_BAR


@pytest.mark.parametrize("D", [13, 100, 256, 512])
@pytest.mark.parametrize("K", [10, 300, 1001])
def test_stats_from_embeddings(D, K):
    X, C = clustered(700, D, 11 + D), clustered(1001, D, 12 + D)
    em, es, _, _ = embedding_errors(X, C, K)
    print(f"asnorm stats D={D} Nc=1001 K={K}: mean {em:.3e}, std rel {es:.3e}")
    assert em < MEAN_BAR and es < STD_BAR


@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_stats_at_chunk_boundaries(delta):
    Nc = 1001
    n = chunk_rows(Nc) + delta
    X, C = clustered(n, 256, 21), clustered(Nc, 256, 22)
    em, es, st, _ = embedding_errors(X, C, 300)
    print(f"asnorm stats n={n} (chunk {chunk_rows(Nc)}): mean {em:.3e}, std rel {es:.3e}")
    assert em < MEAN_BAR and es < STD_BAR
    # the chunks are independent: the last chunk's rows agree with a call on those rows alone
    tail = torch.ops.svb200.cohort_stats(torch.tensor(X[-3:]).cuda(), torch.tensor(C).cuda(), 300).cpu().numpy()
    np.testing.assert_array_equal(tail, st[-3:])


# ------------------------------------------------------------------------------------------------- trials and matrices
def trial_case(seed=5, ne=400, nt=900, n=20000, D=256, Nc=1001):
    r = np.random.RandomState(seed)
    E, T, C = clustered(ne, D, seed), clustered(nt, D, seed + 1), clustered(Nc, D, seed + 2)
    return E, T, C, r.randint(ne, size=n), r.randint(nt, size=n)


def test_raw_trial_cosines():
    E, T, _, ei, ti = trial_case()
    got = svb.score_trials(torch.tensor(E).cuda(), torch.tensor(T).cuda(), torch.tensor(ei).cuda(),
                           torch.tensor(ti).cuda()).cpu().numpy()
    err = np.abs(got - A.trial_scores(E, T, ei, ti)).max()
    print(f"asnorm raw trial cosine: worst abs error {err:.3e}")
    assert got.dtype == np.float32 and err < 1e-6


@pytest.mark.parametrize("K", [None, 300])
def test_normalized_trial_scores(K):
    E, T, C, ei, ti = trial_case(D=100)
    got = svb.score_trials(torch.tensor(E).cuda(), torch.tensor(T).cuda(), torch.tensor(ei).cuda(),
                           torch.tensor(ti).cuda(), cohort=torch.tensor(C).cuda(), top_k=K).cpu().numpy()
    err = score_err(got, A.trial_scores(E, T, ei, ti, C, K))
    print(f"asnorm normalized trial score K={K}: worst error {err:.3e}")
    assert err < SCORE_BAR


def ti_sv_case(N=64, Mv=3, Nc=500):
    enr, ver = I.eer_embeddings(N, 2 * Mv, 0.06, 0.5, 17)
    C = clustered(Nc, 256, 18)
    return torch.tensor(enr).cuda(), torch.tensor(ver).cuda(), torch.tensor(C).cuda()


def test_normalize_sim_against_oracle():
    enr, ver, C = ti_sv_case()
    cen = svb.get_centroids(enr)
    sim = svb.get_cossim(ver, cen)
    got = svb.normalize_sim(sim, cen, ver, C, top_k=100).cpu().numpy()
    ref = A.normalize_sim(sim.cpu().numpy(), cen.cpu().numpy(), ver.cpu().numpy(), C.cpu().numpy(), 100)
    err = score_err(got, ref)
    print(f"asnorm normalized TI-SV matrix: worst error {err:.3e}")
    assert err < SCORE_BAR


def test_compute_verification_metrics_with_cohort():
    enr, ver, C = ti_sv_case()
    m, nsim = svb.compute_verification_metrics(enr, ver, cohort=C, top_k=50)
    cen = svb.get_centroids(enr)
    ref_sim = svb.normalize_sim(svb.get_cossim(ver, cen), cen, ver, C, top_k=50)
    assert torch.equal(nsim, ref_sim)
    assert m == svb.verification_metrics_from_sim(ref_sim)
    plain, sim = svb.compute_verification_metrics(enr, ver, cohort=None)
    assert torch.equal(sim, svb.get_cossim(ver, cen))
    assert plain == svb.verification_metrics_from_sim(sim)


# ------------------------------------------------------------------------------------------------- interface
def test_cpu_float64_noncontiguous_and_integer_inputs():
    E, T, C, ei, ti = trial_case(n=3000)
    ref = svb.score_trials(torch.tensor(E).cuda(), torch.tensor(T).cuda(), torch.tensor(ei, dtype=torch.int32).cuda(),
                           torch.tensor(ti, dtype=torch.int32).cuda(), cohort=torch.tensor(C).cuda(), top_k=64)
    E64 = torch.tensor(E, dtype=torch.float64)
    Tnc = torch.tensor(T).t().contiguous().t()                      # column-major: non-contiguous rows
    assert not Tnc.is_contiguous()
    got = svb.score_trials(E64, Tnc, torch.tensor(ei, dtype=torch.int64), torch.tensor(ti, dtype=torch.int16),
                           cohort=torch.tensor(C), top_k=64)
    assert got.device.type == "cpu" and got.dtype == torch.float32
    assert torch.equal(got, ref.cpu())
    mean, std = svb.cohort_stats(E64, torch.tensor(C), top_k=64)
    assert mean.device.type == "cpu" and mean.dtype == torch.float64
    st = torch.ops.svb200.cohort_stats(torch.tensor(E).cuda(), torch.tensor(C).cuda(), 64).cpu()
    assert torch.equal(mean, st[:, 0]) and torch.equal(std, st[:, 1])


def test_value_errors():
    E, T, C, ei, ti = trial_case(n=100)
    E, T, C = torch.tensor(E).cuda(), torch.tensor(T).cuda(), torch.tensor(C).cuda()
    ei, ti = torch.tensor(ei).cuda(), torch.tensor(ti).cuda()
    with pytest.raises(ValueError, match="D ="):
        svb.score_trials(E, T[:, :100], ei, ti)
    with pytest.raises(ValueError, match="D ="):
        svb.cohort_stats(E, C[:, :13])
    with pytest.raises(ValueError, match="top_k"):
        svb.cohort_stats(E, C, top_k=1)
    with pytest.raises(ValueError, match="top_k"):
        svb.cohort_stats(E, C, top_k=C.shape[0] + 1)
    with pytest.raises(ValueError, match="at least 2"):
        svb.cohort_stats(E, C[:1])
    bad = ei.clone()
    bad[7] = E.shape[0]
    with pytest.raises(ValueError, match="enroll_idx out of range"):
        svb.score_trials(E, T, bad, ti)
    bad = ti.clone()
    bad[3] = -1
    with pytest.raises(ValueError, match="test_idx out of range"):
        svb.score_trials(E, T, ei, bad, cohort=C)
    En = E.clone()
    En[5, 3] = float("nan")
    with pytest.raises(ValueError, match="non-finite"):
        svb.cohort_stats(En, C)
    with pytest.raises(ValueError, match="non-finite"):
        svb.score_trials(En, T, ei, ti)
    Ez = E.clone()
    Ez[2] = 0
    with pytest.raises(ValueError, match="non-finite cohort statistic"):
        svb.cohort_stats(Ez, C)
    Cn = C.clone()
    Cn[10, 0] = float("inf")
    with pytest.raises(ValueError, match="non-finite"):
        svb.score_trials(E, T, ei, ti, cohort=Cn)
    with pytest.raises(ValueError, match="zero cohort std"):
        svb.cohort_stats(E, C[:1].repeat(50, 1), top_k=10)     # every cohort cosine of a row is equal
    enr, ver, Ct = ti_sv_case(N=8)
    cen = svb.get_centroids(enr)
    sim = svb.get_cossim(ver, cen)
    with pytest.raises(ValueError, match="verification_embeddings"):
        svb.normalize_sim(sim, cen, ver[:, :2], Ct)
    with pytest.raises(ValueError, match="zero cohort std"):
        svb.compute_verification_metrics(enr, ver, cohort=Ct[:1].repeat(5, 1))


def test_determinism_and_streams():
    X, C = clustered(5000, 256, 31), clustered(6000, 256, 32)
    Xt, Ct = torch.tensor(X).cuda(), torch.tensor(C).cuda()
    a = torch.ops.svb200.cohort_stats(Xt, Ct, 300)
    b = torch.ops.svb200.cohort_stats(Xt, Ct, 300)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = torch.ops.svb200.cohort_stats(Xt, Ct, 300)
    side.synchronize()
    assert torch.equal(a.view(torch.int64), b.view(torch.int64))
    assert torch.equal(a.view(torch.int64), c.view(torch.int64))
    ei = torch.arange(5000, device="cuda", dtype=torch.int32)
    s1 = torch.ops.svb200.score_trials(Xt, Xt, ei, ei.flip(0), a, a)
    s2 = torch.ops.svb200.score_trials(Xt, Xt, ei, ei.flip(0), b, c)
    assert torch.equal(s1.view(torch.int32), s2.view(torch.int32))


def test_opcheck():
    r = np.random.RandomState(2)
    X, C = torch.tensor(clustered(40, 64, 1)).cuda(), torch.tensor(clustered(50, 64, 2)).cuda()
    S = torch.tensor(r.standard_normal((30, 70)).astype(np.float32)).cuda()
    st = torch.ops.svb200.cohort_stats(X, C, 5)
    idx = torch.tensor(r.randint(40, size=90), dtype=torch.int32).cuda()
    sim = torch.tensor(r.standard_normal((4, 10, 4)).astype(np.float32)).cuda()
    utils = ("test_schema", "test_faketensor")
    torch.library.opcheck(torch.ops.svb200.cohort_stats.default, (X, C, 5), test_utils=utils)
    torch.library.opcheck(torch.ops.svb200.cohort_stats_scores.default, (S, 9), test_utils=utils)
    torch.library.opcheck(torch.ops.svb200.score_trials.default, (X, X, idx, idx.flip(0), st, st), test_utils=utils)
    torch.library.opcheck(torch.ops.svb200.score_trials.default, (X, X, idx, idx, None, None), test_utils=utils)
    torch.library.opcheck(torch.ops.svb200.asnorm_sim.default, (sim, st[:4], st[:40]), test_utils=utils)


def test_cuda_graph_capture_of_the_c_abi():
    """A captured svb_cohort_stats (two chunks) + svb_score_trials replays correctly on new data."""
    L = _lib.lib()
    n, Nc, D, K = 3000, 6000, 256, 300
    X = torch.empty(n, D, device="cuda")
    C = torch.empty(Nc, D, device="cuda")
    nb = ctypes.c_size_t(0)
    assert L.svb_cohort_stats_workspace_bytes(ctypes.c_int64(n), Nc, D, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    st = torch.empty(n, 3, dtype=torch.float64, device="cuda")
    idx = torch.arange(n, dtype=torch.int32, device="cuda")
    out = torch.empty(n, device="cuda")
    side = torch.cuda.Stream()

    def call():
        s = ctypes.c_void_p(side.cuda_stream)
        rc = L.svb_cohort_stats(_lib.ptr(X), ctypes.c_int64(n), _lib.ptr(C), Nc, D, K, _lib.ptr(ws),
                                ctypes.c_size_t(nb.value), _lib.ptr(st), s)
        assert rc == 0, L.svb_last_error()
        rc = L.svb_score_trials(_lib.ptr(X), ctypes.c_int64(n), _lib.ptr(X), ctypes.c_int64(n), D, _lib.ptr(idx),
                                _lib.ptr(idx), ctypes.c_int64(n),
                                _lib.ptr(st), _lib.ptr(st), _lib.ptr(out), s)
        assert rc == 0, L.svb_last_error()

    X.copy_(torch.tensor(clustered(n, D, 41)))
    C.copy_(torch.tensor(clustered(Nc, D, 42)))
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            call()
    torch.cuda.synchronize()
    for seed in (43, 45):
        Xn, Cn = clustered(n, D, seed), clustered(Nc, D, seed + 1)
        X.copy_(torch.tensor(Xn))
        C.copy_(torch.tensor(Cn))
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        direct = torch.ops.svb200.cohort_stats(X, C, K)
        assert torch.equal(st, direct)
        assert torch.equal(out, torch.ops.svb200.score_trials(X, X, idx, idx, direct, direct))
        ref = A.stats(Xn, Cn, K)
        assert np.abs(st.cpu().numpy()[:, 0] - ref[:, 0]).max() < MEAN_BAR
