"""GPU: calibration metrics and the calibration fit (svb_calib_metrics / svb_calib_train, csrc/calib.cu) against the
float64 numpy restatement (tests/_calib_oracle.py).  Counts, K, hull vertices, thresholds, p_miss, p_fa and act_dcf
must be equal (==); cllr and min_cllr agree to BAR_CLLR relative, rocch_eer to BAR_EER absolute; the fit's a to
BAR_A * |a|, b to BAR_B * (1 + |b|) and its objective to BAR_OBJ relative (DESIGN.md 4.5.3 records the worst errors
measured on the B200 behind these bars)."""
import ctypes
import math

import numpy as np
import pytest
import torch

import _calib_oracle as O
import _inputs as I
import _verif_oracle as V
import pytorch_speaker_verification_b200 as svb

pytestmark = pytest.mark.gpu

# About 3x the worst errors measured on the B200 (cllr 3.5e-16, min_cllr 2.7e-16, rocch_eer 0, a 1.6e-15, b 1.5e-15,
# objective 4.2e-16); the ROCCH-EER bar is a few ulps of 0.5 since its measured error was 0.
BAR_CLLR, BAR_EER = 1e-15, 1e-15
BAR_A, BAR_B, BAR_OBJ = 5e-15, 5e-15, 1.5e-15
P1 = V.operating_points(0.01)
P8 = V.operating_points([0.001, 0.005, 0.01, 0.05, 0.1, 0.3, 0.5, 0.9], 2.0, 0.75)
WORST = {"cllr": 0.0, "min_cllr": 0.0, "rocch_eer": 0.0, "a": 0.0, "b": 0.0, "objective": 0.0}


def flat(points):
    return [w for p in points for w in p]


def run_metrics(s, lab, points=P1):
    st = torch.as_tensor(np.asarray(s, np.float32)).cuda()
    lt = torch.as_tensor(np.asarray(lab) != 0).cuda().view(torch.uint8)
    return torch.ops.svb200.calib_metrics(st, lt, flat(points)).cpu().numpy()


def compare(got, ref):
    exact = [3, 4, 5, 6, 7] + list(range(8, got.size))
    np.testing.assert_array_equal(got[exact], ref[exact])
    for k, name in ((0, "cllr"), (1, "min_cllr")):
        err = abs(got[k] - ref[k]) / max(abs(ref[k]), 1e-300)
        WORST[name] = max(WORST[name], err)
        assert err <= BAR_CLLR, (name, got[k], ref[k])
    err = abs(got[2] - ref[2])
    WORST["rocch_eer"] = max(WORST["rocch_eer"], err)
    assert err <= BAR_EER, (got[2], ref[2])


def check_metrics(s, lab, points=P1):
    got, ref = run_metrics(s, lab, points), O.metrics(s, lab, points)
    compare(got, ref)
    return got


def check_train(s, lab, prior=0.5):
    st = torch.as_tensor(np.asarray(s, np.float32)).cuda()
    lt = torch.as_tensor(np.asarray(lab) != 0).cuda().view(torch.uint8)
    a, b, c, iters, status = torch.ops.svb200.calib_train(st, lt, prior, 100).cpu().tolist()
    ra, rb, rc, _, rstatus = O.train(s, lab, prior)
    assert status == rstatus == 0 and iters <= 30
    ea, eb, ec = abs(a - ra) / abs(ra), abs(b - rb) / (1 + abs(rb)), abs(c - rc) / abs(rc)
    WORST["a"], WORST["b"], WORST["objective"] = max(WORST["a"], ea), max(WORST["b"], eb), max(WORST["objective"], ec)
    assert ea <= BAR_A and eb <= BAR_B and ec <= BAR_OBJ, (a, ra, b, rb, c, rc)
    return a, b, c


def labels_with(n, kind, r):
    if kind == "one_target":
        lab = np.zeros(n, bool); lab[r.randint(n)] = True
    elif kind == "one_nontarget":
        lab = np.ones(n, bool); lab[r.randint(n)] = False
    else:
        lab = r.rand(n) < kind
        lab[0], lab[-1] = True, False
    return lab


# ------------------------------------------------------------------------------------------------ metrics
@pytest.mark.parametrize("n", [2, 3, 31, 1000, 4097, 65537, 1_000_003])
@pytest.mark.parametrize("kind", ["one_target", 0.01, 0.5, "one_nontarget"])
def test_metrics_random_sizes(n, kind):
    r = np.random.RandomState(n % 1000 + 23)
    lab = labels_with(n, kind, r)
    s = (r.standard_normal(n) * 2 + 2.5 * lab - 1).astype(np.float32)
    check_metrics(s, lab, P8 if n in (1000, 65537) else P1)


@pytest.mark.parametrize("case", ["round2", "all_equal", "two_values", "cross_class_ties"])
def test_metrics_ties(case):
    r = np.random.RandomState(3)
    n = 50_001
    lab = r.rand(n) < 0.1
    lab[0], lab[1] = True, False
    s = (r.standard_normal(n) * 0.3 + 0.5 + 0.4 * lab).astype(np.float32)
    if case == "round2":
        s = np.round(s, 2).astype(np.float32)
    elif case == "all_equal":
        s = np.full(n, 0.7, np.float32)
    elif case == "two_values":
        s = np.where(r.rand(n) < 0.5, 0.25, 0.75).astype(np.float32)
    else:
        s = r.randint(0, 20, n).astype(np.float32)
    out = check_metrics(s, lab, P8)
    if case == "all_equal":
        assert out[7] == 1 and out[6] == 2 and abs(out[1] - 1.0) <= 1e-15


def test_metrics_special_values():
    r = np.random.RandomState(8)
    n = 20_000
    vals = np.array([0.0, -0.0, -1.5, -1e-3, 1e-40, -1e-40, 1.4e-45, -1.4e-45, 3e38, -3e38, 2.0, -2.0], np.float32)
    s = np.concatenate([vals, r.choice(vals, n // 2), r.standard_normal(n // 2).astype(np.float32) - 1.0])
    lab = r.rand(s.size) < 0.3
    lab[0], lab[1] = True, False
    check_metrics(s, lab, P8)
    z = np.array([0.0, -0.0, -0.0, 0.0, 1.0], np.float32)
    assert check_metrics(z, np.array([1, 0, 1, 0, 1]))[7] == 2


@pytest.mark.parametrize("reverse", [False, True])
def test_metrics_separation(reverse):
    r = np.random.RandomState(11)
    lab = r.rand(30_000) < 0.2
    lab[0], lab[1] = True, False
    s = (r.rand(lab.size) + np.where(lab != reverse, 3.0, 0.0)).astype(np.float32)
    out = check_metrics(s, lab, P8)
    if reverse:
        assert abs(out[1] - 1.0) <= 1e-15 and out[2] == 0.5
    else:
        assert out[1] == 0.0 and out[2] == 0.0


def test_metrics_adversarial_convex_csd():
    """Group g holds g + 1 trials, g of them targets: every group end is a hull vertex (about 2,000 over 500 tiles)."""
    G = 2000
    g = np.repeat(np.arange(G), np.arange(G) + 1)
    s = g.astype(np.float32)
    lab = np.ones(s.size, bool)
    lab[np.cumsum(np.arange(G) + 1) - 1] = False               # the last trial of each group is the non-target
    out = check_metrics(s, lab, P8)
    assert out[6] == G + 1 and out[7] == G and s.size > 4096 * 400


def test_metrics_large_input_beyond_l2():
    n = (1 << 25) + 7
    r = np.random.RandomState(99)
    lab = r.rand(n) < 0.01
    s = (r.standard_normal(n).astype(np.float32) * np.float32(3) + np.float32(4.0) * lab - np.float32(5)).astype(np.float32)
    check_metrics(s, lab, P8)


def test_act_dcf_is_at_least_min_dcf():
    r = np.random.RandomState(5)
    lab = r.rand(200_000) < 0.05
    s = (r.standard_normal(lab.size) * 1.5 + 3 * lab - 4).astype(np.float32)
    pt = [0.001, 0.01, 0.05, 0.1, 0.3, 0.5, 0.7, 0.9]
    m = svb.calibration_metrics(torch.tensor(s).cuda(), torch.tensor(lab).cuda(), p_target=pt)
    v = svb.verification_metrics(torch.tensor(s).cuda(), torch.tensor(lab).cuda(), p_target=pt)
    assert all(a >= b for a, b in zip(m.act_dcf, v.min_dcf)), (m.act_dcf, v.min_dcf)
    assert m.min_cllr <= m.cllr and m.rocch_eer <= v.eer


# ------------------------------------------------------------------------------------------------ calibration
@pytest.mark.parametrize("n", [31, 1000, 65537, 1_000_003])
@pytest.mark.parametrize("prior", [0.5, 0.1, 0.9])
def test_train_against_oracle(n, prior):
    r = np.random.RandomState(n % 997 + int(prior * 10))
    lab = labels_with(n, 0.3, r)
    s = (r.standard_normal(n) * 0.2 + 0.3 * lab + 0.4).astype(np.float32)
    check_train(s, lab, prior)


@pytest.mark.parametrize("kind", ["one_target", "one_nontarget", "round2"])
def test_train_edge_cases(kind):
    r = np.random.RandomState(7)
    n = 4097
    lab = labels_with(n, kind, r) if kind != "round2" else labels_with(n, 0.2, r)
    s = (r.standard_normal(n) + lab).astype(np.float32)
    if kind == "round2":
        s = np.round(s, 2).astype(np.float32)
    check_train(s, lab, 0.5)


def test_calibrating_a_set_on_itself():
    r = np.random.RandomState(17)
    lab = r.rand(300_000) < 0.1
    s = torch.tensor((r.standard_normal(lab.size) * 0.15 + 0.25 * lab + 0.3).astype(np.float32)).cuda()
    lt = torch.tensor(lab).cuda()
    cal = svb.train_calibration(s, lt)
    llr = svb.apply_calibration(s, cal)
    assert llr.dtype == torch.float32 and llr.device == s.device
    assert torch.equal(llr, (s.double() * cal.scale + cal.offset).float())
    m = svb.calibration_metrics(llr, lt)
    assert m.min_cllr <= m.cllr <= 1 + 1e-12
    a, b, c = check_train(s.cpu().numpy(), lab)
    assert abs(m.cllr - c) <= 1e-6                                # the LLRs are rounded to float32


def test_end_to_end_with_cohort_scoring():
    """score_trials with a cohort, a fit on half the trials, applied to the other half, then the metrics."""
    enr, ver = I.eer_embeddings(300, 4, 0.08, 0.5, 31)
    E = torch.tensor(enr.reshape(-1, enr.shape[-1])).cuda()
    T = torch.tensor(ver.reshape(-1, ver.shape[-1])).cuda()
    cohort = torch.tensor(I.unit_rows(400, enr.shape[-1], 5)).cuda()
    r = np.random.RandomState(2)
    ne, nt = E.shape[0], T.shape[0]
    ei = torch.tensor(r.randint(0, ne, 200_000)).cuda()
    ti = torch.tensor(r.randint(0, nt, 200_000)).cuda()
    ei[::10] = ti[::10] // ver.shape[1] * enr.shape[1]           # a tenth of the trials are same-speaker
    lab = (ei // enr.shape[1]) == (ti // ver.shape[1])
    s = svb.score_trials(E, T, ei, ti, cohort=cohort, top_k=100)
    half = s.numel() // 2
    cal = svb.train_calibration(s[:half], lab[:half])
    llr = svb.apply_calibration(s[half:], cal)
    m = svb.calibration_metrics(llr, lab[half:], p_target=[0.01, 0.05])
    ref = O.metrics(llr.cpu().numpy(), lab[half:].cpu().numpy(), V.operating_points([0.01, 0.05]))
    compare(np.array([m.cllr, m.min_cllr, m.rocch_eer, m.n_target, m.n_nontarget, 0, ref[6], ref[7]] +
                     [x for p in range(2) for x in (m.act_dcf[p], m.act_dcf_threshold[p], m.act_dcf_p_miss[p],
                                                     m.act_dcf_p_fa[p])]), ref)
    assert m.min_cllr <= m.cllr < 1.0


# ------------------------------------------------------------------------------------------------ Python API
def test_value_errors():
    s = torch.randn(100, device="cuda")
    lab = torch.arange(100, device="cuda") % 3 == 0
    for bad in (float("nan"), float("inf"), -float("inf")):
        s2 = s.clone()
        s2[17] = bad
        with pytest.raises(ValueError, match="not finite"):
            svb.calibration_metrics(s2, lab)
        with pytest.raises(ValueError, match="finite"):
            svb.train_calibration(s2, lab)
    for empty in (torch.zeros_like(lab), torch.ones_like(lab)):
        with pytest.raises(ValueError, match="target"):
            svb.calibration_metrics(s, empty)
        with pytest.raises(ValueError, match="classes"):
            svb.train_calibration(s, empty)
    for f in (svb.calibration_metrics, svb.train_calibration):
        with pytest.raises(ValueError, match="shape"):
            f(s, lab[:99])
        with pytest.raises(ValueError):
            f(s[:1], lab[:1])
    for p in (0.0, 1.0, -0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="prior"):
            svb.train_calibration(s, lab, prior=p)
        with pytest.raises(ValueError):
            svb.calibration_metrics(s, lab, p_target=p)
    with pytest.raises(ValueError):
        svb.calibration_metrics(s, lab, p_target=[0.1] * 9)
    sep = torch.where(lab, s.abs() + 1, -s.abs())
    with pytest.raises(ValueError, match="overlap"):
        svb.train_calibration(sep, lab)
    with pytest.raises(ValueError, match="overlap"):
        svb.train_calibration(torch.full_like(s, 0.5), lab)
    with pytest.raises(ValueError, match="max_iter"):
        svb.train_calibration(s + lab * 0.5, lab, max_iter=1)
    with pytest.raises(ValueError, match="max_iter"):
        svb.train_calibration(s, lab, max_iter=0)


def test_input_handling():
    r = np.random.RandomState(6)
    base = (r.standard_normal((300, 200)) * 2).astype(np.float32)
    lab_i = r.randint(-2, 3, (300, 200)).astype(np.int64)
    lab_i[0, 0], lab_i[0, 1] = 1, 0
    base += 1.5 * (lab_i != 0)
    ref = O.metrics(base, lab_i, P1)

    def arr(m):
        return np.array([m.cllr, m.min_cllr, m.rocch_eer, m.n_target, m.n_nontarget, 0, ref[6], ref[7],
                         m.act_dcf[0], m.act_dcf_threshold[0], m.act_dcf_p_miss[0], m.act_dcf_p_fa[0]])
    compare(arr(svb.calibration_metrics(torch.tensor(base), torch.tensor(lab_i))), ref)          # CPU, int64 labels
    compare(arr(svb.calibration_metrics(torch.tensor(base).cuda(), torch.tensor(lab_i != 0).cuda())), ref)
    st = torch.tensor(base.T.copy()).cuda().t()
    lt = torch.tensor(lab_i.T.copy().astype(np.int32)).cuda().t()
    assert not st.is_contiguous() and not lt.is_contiguous()
    compare(arr(svb.calibration_metrics(st, lt)), ref)
    compare(arr(svb.calibration_metrics(torch.tensor(base.astype(np.float64)), torch.tensor(lab_i))), ref)
    fits = [svb.train_calibration(torch.tensor(base), torch.tensor(lab_i)),
            svb.train_calibration(st, lt),
            svb.train_calibration(torch.tensor(base.astype(np.float64)).cuda(), torch.tensor(lab_i != 0))]
    assert fits[0] == fits[1] == fits[2]
    llr = svb.apply_calibration(torch.tensor(base.astype(np.float64)), fits[0])
    assert llr.dtype == torch.float32 and llr.device.type == "cpu" and llr.shape == (300, 200)


def test_determinism_and_streams():
    r = np.random.RandomState(12)
    lab = r.rand(2_000_000) < 0.02
    s = np.round(r.standard_normal(lab.size) + lab, 3).astype(np.float32)
    st = torch.tensor(s).cuda()
    lt = torch.tensor(lab).cuda().view(torch.uint8)
    runs = []
    for k in range(3):
        side = torch.cuda.Stream() if k == 2 else torch.cuda.current_stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            runs.append((torch.ops.svb200.calib_metrics(st, lt, flat(P8)), torch.ops.svb200.calib_train(st, lt, 0.3, 100)))
        side.synchronize()
    for m, t in runs[1:]:
        assert torch.equal(m.view(torch.int64), runs[0][0].view(torch.int64))
        assert torch.equal(t.view(torch.int64), runs[0][1].view(torch.int64))
    compare(runs[0][0].cpu().numpy(), O.metrics(s, lab, P8))


def test_opcheck():
    r = np.random.RandomState(2)
    s = torch.tensor(r.standard_normal(5000).astype(np.float32)).cuda()
    lab = torch.tensor(r.rand(5000) < 0.3).cuda().view(torch.uint8)
    utils = ("test_schema", "test_faketensor")
    torch.library.opcheck(torch.ops.svb200.calib_metrics.default, (s, lab, flat(P8)), test_utils=utils)
    torch.library.opcheck(torch.ops.svb200.calib_train.default, (s, lab, 0.5, 100), test_utils=utils)


def test_cuda_graph_capture_of_the_c_abi():
    """Both entry points in one captured graph, replayed on two new data sets."""
    from pytorch_speaker_verification_b200 import _lib
    L = _lib.lib()
    n = 300_001
    r = np.random.RandomState(31)
    data = []
    for k in range(2):
        lab = r.rand(n) < (0.05 if k == 0 else 0.3)
        s = np.round(r.standard_normal(n) * (1 + k) + (1 + k) * lab - 2, 2 + k).astype(np.float32)
        data.append((s, lab))
    scores = torch.empty(n, dtype=torch.float32, device="cuda")
    labels = torch.empty(n, dtype=torch.uint8, device="cuda")
    nb = ctypes.c_size_t(0)
    assert L.svb_calib_workspace_bytes(ctypes.c_int64(n), ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(8 + 4 * len(P8), dtype=torch.float64, device="cuda")
    fit = torch.empty(5, dtype=torch.float64, device="cuda")
    ops = (ctypes.c_double * (3 * len(P8)))(*flat(P8))
    side = torch.cuda.Stream()

    def call():
        st = ctypes.c_void_p(side.cuda_stream)
        rc = L.svb_calib_metrics(_lib.ptr(scores), _lib.ptr(labels), ctypes.c_int64(n), ops, len(P8), _lib.ptr(ws),
                                 ctypes.c_size_t(nb.value), _lib.ptr(out), st)
        assert rc == 0, L.svb_last_error()
        rc = L.svb_calib_train(_lib.ptr(scores), _lib.ptr(labels), ctypes.c_int64(n), ctypes.c_double(0.5), 100,
                               _lib.ptr(ws), ctypes.c_size_t(nb.value), _lib.ptr(fit), st)
        assert rc == 0, L.svb_last_error()

    scores.copy_(torch.tensor(data[1][0]))
    labels.copy_(torch.tensor(data[1][1]).view(torch.uint8))
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            call()
    torch.cuda.synchronize()
    for s, lab in data:
        scores.copy_(torch.tensor(s))
        labels.copy_(torch.tensor(lab).view(torch.uint8))
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        compare(out.cpu().numpy(), O.metrics(s, lab, P8))
        a, b, c, _, status = fit.cpu().tolist()
        ra, rb, rc, _, _ = O.train(s, lab, 0.5)
        assert status == 0 and abs(a - ra) <= BAR_A * abs(ra) and abs(b - rb) <= BAR_B * (1 + abs(rb))


def test_zz_worst_errors():
    """Prints the worst error of each compared quantity over this module's tests (DESIGN.md 4.5.3 records them)."""
    print("\nworst errors: " + ", ".join(f"{k} {v:.2e}" for k, v in WORST.items()))
