"""GPU: exact EER and minDCF (svb_verif_metrics / svb_verif_metrics_sim, csrc/verif.cu) against the float64 numpy
restatement (tests/_verif_oracle.py).  Every integer and float64 step is fixed by the definitions, so every field must
equal the oracle exactly (==), including K (the number of distinct scores)."""
import ctypes

import numpy as np
import pytest
import torch

import _inputs as I
import _verif_oracle as V
import pytorch_speaker_verification_b200  # noqa: F401  (registers torch.ops.svb200.*)

pytestmark = pytest.mark.gpu

P1 = V.operating_points(0.01)
P8 = V.operating_points([0.001, 0.005, 0.01, 0.05, 0.1, 0.3, 0.5, 0.9], 2.0, 0.75)


def flat(points):
    return [w for p in points for w in p]


def run_flat(s, lab, points=P1):
    """Raw op on CUDA float32 scores / uint8 labels -> numpy float64 out."""
    st = torch.as_tensor(np.asarray(s, np.float32)).cuda()
    lt = torch.as_tensor(np.asarray(lab) != 0).cuda().view(torch.uint8)
    return torch.ops.svb200.verif_metrics(st, lt, flat(points)).cpu().numpy()


def run_sim(sim, points=P1):
    return torch.ops.svb200.verif_metrics_sim(torch.as_tensor(np.asarray(sim, np.float32)).cuda(),
                                              flat(points)).cpu().numpy()


def check_flat(s, lab, points=P1):
    got, ref = run_flat(s, lab, points), V.metrics(s, lab, points)
    np.testing.assert_array_equal(got, ref)
    return got


def api_array(m):
    """VerificationMetrics -> the out layout without the #non-finite and K fields."""
    out = [m.eer, m.eer_threshold, m.eer_p_miss, m.eer_p_fa, m.n_target, m.n_nontarget]
    for p in range(len(m.min_dcf)):
        out += [m.min_dcf[p], m.min_dcf_threshold[p], m.min_dcf_p_miss[p], m.min_dcf_p_fa[p]]
    return np.array(out, np.float64)


def strip(ref):
    return np.concatenate([ref[:6], ref[8:]])


def labels_with(n, kind, r):
    if kind == "one_target":
        lab = np.zeros(n, bool); lab[r.randint(n)] = True
    elif kind == "one_nontarget":
        lab = np.ones(n, bool); lab[r.randint(n)] = False
    else:
        lab = r.rand(n) < kind
        lab[0], lab[-1] = True, False
    return lab


def c5_sim():
    enr, ver = I.eer_embeddings(1024, 6, 0.06, 0.5, 4242)
    cen = enr.mean(1)
    cen /= np.linalg.norm(cen, axis=1, keepdims=True)
    return np.einsum("nmd,kd->nmk", ver, cen).astype(np.float32)


# ------------------------------------------------------------------------------------------------ flat form
@pytest.mark.parametrize("n", [2, 3, 31, 1000, 4097, 65537, 1_000_003])
@pytest.mark.parametrize("kind", ["one_target", 0.01, 0.5, "one_nontarget"])
def test_flat_random_sizes(n, kind):
    r = np.random.RandomState(n % 1000 + 17)
    lab = labels_with(n, kind, r)
    s = (r.standard_normal(n) + 1.5 * lab).astype(np.float32)
    check_flat(s, lab, P8 if n in (1000, 65537) else P1)


@pytest.mark.parametrize("case", ["round2", "round4", "all_equal", "two_values", "cross_class_ties"])
def test_ties(case):
    r = np.random.RandomState(3)
    n = 50_001
    lab = r.rand(n) < 0.1
    lab[0], lab[1] = True, False
    s = (r.standard_normal(n) * 0.3 + 0.5 + 0.4 * lab).astype(np.float32)
    if case == "round2":
        s = np.round(s, 2).astype(np.float32)
    elif case == "round4":
        s = np.round(s, 4).astype(np.float32)
    elif case == "all_equal":
        s = np.full(n, 0.7, np.float32)
    elif case == "two_values":
        s = np.where(r.rand(n) < 0.5, 0.25, 0.75).astype(np.float32)
    else:                                                      # every value held by both classes
        s = r.randint(0, 20, n).astype(np.float32)
    out = check_flat(s, lab, P8)
    if case == "all_equal":
        assert out[7] == 1


def test_special_values():
    r = np.random.RandomState(8)
    n = 20_000
    vals = np.array([0.0, -0.0, -1.5, -1e-3, 1e-40, -1e-40, 1.4e-45, -1.4e-45, 3e38, -3e38, 2.0, -2.0], np.float32)
    s = np.concatenate([vals, r.choice(vals, n // 2), r.standard_normal(n // 2).astype(np.float32) - 1.0])
    lab = r.rand(s.size) < 0.3
    lab[0], lab[1] = True, False
    check_flat(s, lab, P8)
    # -0 and +0 are one distinct value
    z = np.array([0.0, -0.0, -0.0, 0.0, 1.0], np.float32)
    out = check_flat(z, np.array([1, 0, 1, 0, 1]))
    assert out[7] == 2


@pytest.mark.parametrize("reverse", [False, True])
def test_extreme_separation(reverse):
    r = np.random.RandomState(11)
    lab = r.rand(30_000) < 0.2
    lab[0], lab[1] = True, False
    s = (r.rand(lab.size) + np.where(lab != reverse, 3.0, 0.0)).astype(np.float32)
    out = check_flat(s, lab, P8)
    if not reverse:
        assert out[0] == 0.0 and all(out[8 + 4 * p] == 0.0 for p in range(len(P8)))
    else:
        assert out[0] > 0.49


# ------------------------------------------------------------------------------------------------ sim form
@pytest.mark.parametrize("N,Mv", [(2, 1), (3, 5), (17, 3), (64, 10)])
def test_sim_small(N, Mv):
    r = np.random.RandomState(N * 100 + Mv)
    sim = r.uniform(-1, 1, (N, Mv, N)).astype(np.float32)
    sim[np.arange(N), :, np.arange(N)] += 0.5
    got = run_sim(sim, P8)
    np.testing.assert_array_equal(got, V.metrics_sim(sim, P8))
    np.testing.assert_array_equal(got, run_flat(sim.ravel(), V.sim_labels(N, Mv).ravel(), P8))


def test_sim_c5_and_flat_form_agree():
    sim = c5_sim()
    got = run_sim(sim, P8)
    np.testing.assert_array_equal(got, V.metrics_sim(sim, P8))
    np.testing.assert_array_equal(got, run_flat(sim.ravel(), V.sim_labels(*sim.shape[:2]).ravel(), P8))
    assert abs(got[0] - 0.04) < 5e-4
    # the scale that makes the 50-threshold sweep report 0 leaves the exact EER where it was (K may shrink: the
    # float32 product merges some neighbouring values)
    scaled = sim * np.float32(0.4)
    got_scaled = run_sim(scaled)
    np.testing.assert_array_equal(got_scaled, V.metrics_sim(scaled, P1))
    np.testing.assert_array_equal(got_scaled[[0, 2, 3, 4, 5]], got[[0, 2, 3, 4, 5]])


def test_compute_verification_metrics_matches_compute_eer_sim():
    import pytorch_speaker_verification_b200 as svb
    enr, ver = I.eer_embeddings(200, 8, 0.08, 0.5, 21)
    e, v = torch.tensor(enr).cuda(), torch.tensor(ver).cuda()
    m, sim = svb.compute_verification_metrics(e, v, p_target=[0.01, 0.05])
    _, sim_eer = svb.compute_eer(e, v)
    assert torch.equal(sim, sim_eer)
    ref = V.metrics_sim(sim.cpu().numpy(), V.operating_points([0.01, 0.05]))
    np.testing.assert_array_equal(api_array(m), strip(ref))


# ------------------------------------------------------------------------------------------------ Python API
def test_operating_points_and_costs():
    import pytorch_speaker_verification_b200 as svb
    r = np.random.RandomState(4)
    lab = r.rand(100_000) < 0.05
    s = (r.standard_normal(lab.size) + 2.0 * lab).astype(np.float32)
    m1 = svb.verification_metrics(torch.tensor(s).cuda(), torch.tensor(lab).cuda())
    np.testing.assert_array_equal(api_array(m1), strip(V.metrics(s, lab, V.operating_points(0.01))))
    assert isinstance(m1.min_dcf, tuple) and len(m1.min_dcf) == 1
    pt = [0.001, 0.01, 0.02, 0.05, 0.1, 0.25, 0.5, 0.75]
    m8 = svb.verification_metrics(torch.tensor(s).cuda(), torch.tensor(lab).cuda(), p_target=pt, c_miss=10.0, c_fa=0.3)
    np.testing.assert_array_equal(api_array(m8), strip(V.metrics(s, lab, V.operating_points(pt, 10.0, 0.3))))
    assert m8.min_dcf[1] != m1.min_dcf[0]


def test_value_errors():
    import pytorch_speaker_verification_b200 as svb
    s = torch.randn(100, device="cuda")
    lab = torch.arange(100, device="cuda") % 3 == 0
    for bad in (float("nan"), float("inf"), -float("inf")):
        s2 = s.clone()
        s2[17] = bad
        with pytest.raises(ValueError, match="not finite"):
            svb.verification_metrics(s2, lab)
    with pytest.raises(ValueError, match="target"):
        svb.verification_metrics(s, torch.zeros_like(lab))
    with pytest.raises(ValueError, match="target"):
        svb.verification_metrics(s, torch.ones_like(lab))
    with pytest.raises(ValueError):
        svb.verification_metrics(s[:1], lab[:1])
    with pytest.raises(ValueError, match="shape"):
        svb.verification_metrics(s, lab[:99])
    with pytest.raises(ValueError, match="shape"):
        svb.verification_metrics(s.reshape(10, 10), lab)
    with pytest.raises(ValueError):
        svb.verification_metrics_from_sim(torch.randn(1, 3, 1, device="cuda"))
    with pytest.raises(ValueError):
        svb.verification_metrics_from_sim(torch.randn(4, 3, 5, device="cuda"))
    for p in (0.0, 1.0, -0.1, 1.5, [0.01, 1.0], []):
        with pytest.raises(ValueError):
            svb.verification_metrics(s, lab, p_target=p)
    for cm, cf in ((0.0, 1.0), (1.0, 0.0), (-1.0, 1.0), (1.0, -2.0)):
        with pytest.raises(ValueError):
            svb.verification_metrics(s, lab, c_miss=cm, c_fa=cf)
    with pytest.raises(ValueError):
        svb.verification_metrics(s, lab, p_target=[0.1] * 9)
    with pytest.raises(ValueError):
        svb.verification_metrics_from_sim(torch.full((3, 2, 3), float("nan"), device="cuda"))


def test_input_handling():
    import pytorch_speaker_verification_b200 as svb
    r = np.random.RandomState(6)
    base = r.standard_normal((300, 200)).astype(np.float32)
    lab_i = r.randint(-2, 3, (300, 200)).astype(np.int64)        # nonzero = target
    lab_i[0, 0], lab_i[0, 1] = 1, 0
    ref = strip(V.metrics(base, lab_i, P1))
    # CPU tensors, integer labels
    np.testing.assert_array_equal(api_array(svb.verification_metrics(torch.tensor(base), torch.tensor(lab_i))), ref)
    np.testing.assert_array_equal(api_array(svb.verification_metrics(torch.tensor(base),
                                                                      torch.tensor(lab_i.astype(np.int32)).cuda())), ref)
    # non-contiguous views
    st = torch.tensor(base.T.copy()).cuda().t()
    lt = torch.tensor(lab_i.T.copy() != 0).cuda().t()
    assert not st.is_contiguous() and not lt.is_contiguous()
    np.testing.assert_array_equal(api_array(svb.verification_metrics(st, lt)), ref)
    sl = torch.tensor(base).cuda()[:, ::2]
    ll = torch.tensor(lab_i).cuda()[:, ::2]
    np.testing.assert_array_equal(api_array(svb.verification_metrics(sl, ll)),
                                  strip(V.metrics(base[:, ::2], lab_i[:, ::2], P1)))
    # float64 scores are staged to float32
    s64 = r.standard_normal(5000)
    l64 = r.rand(5000) < 0.2
    np.testing.assert_array_equal(api_array(svb.verification_metrics(torch.tensor(s64), torch.tensor(l64))),
                                  strip(V.metrics(s64.astype(np.float32), l64, P1)))
    # sim form from the CPU and from a non-contiguous CUDA view
    sim = np.ascontiguousarray(c5_sim()[:100, :, :100])
    ref_sim = strip(V.metrics_sim(sim, P1))
    np.testing.assert_array_equal(api_array(svb.verification_metrics_from_sim(torch.tensor(sim))), ref_sim)
    sim_view = torch.tensor(np.ascontiguousarray(sim.transpose(2, 1, 0))).cuda().permute(2, 1, 0)
    assert not sim_view.is_contiguous()
    np.testing.assert_array_equal(api_array(svb.verification_metrics_from_sim(sim_view)), ref_sim)


@pytest.mark.parametrize("offset", [1, 2, 3])
def test_misaligned_scores_take_the_scalar_path(offset):
    """A contiguous view at a 4-byte offset stays unaligned after staging: the key kernel reads it element by element."""
    import pytorch_speaker_verification_b200 as svb
    r = np.random.RandomState(40 + offset)
    n = 70_001
    lab = r.rand(n) < 0.1
    s = np.round(r.standard_normal(n) + lab, 3).astype(np.float32)
    st, lt = torch.tensor(s).cuda(), torch.tensor(lab).cuda()
    view = st[offset:]
    assert view.data_ptr() % 16 != 0
    m = svb.verification_metrics(view, lt[offset:], p_target=[0.01, 0.1])
    np.testing.assert_array_equal(api_array(m), strip(V.metrics(s[offset:], lab[offset:], V.operating_points([0.01, 0.1]))))
    # the raw op on an unaligned view, including K
    got = torch.ops.svb200.verif_metrics(view, lt[offset:].view(torch.uint8), flat(P8)).cpu().numpy()
    np.testing.assert_array_equal(got, V.metrics(s[offset:], lab[offset:], P8))


def test_raw_op_rejects_labels_on_another_device():
    s = torch.randn(100, device="cuda")
    lab = (torch.arange(100) % 2).to(torch.uint8)
    with pytest.raises((ValueError, RuntimeError), match="device"):
        torch.ops.svb200.verif_metrics(s, lab, flat(P1))


def test_determinism_and_streams():
    r = np.random.RandomState(12)
    lab = r.rand(2_000_000) < 0.02
    s = np.round(r.standard_normal(lab.size) + lab, 3).astype(np.float32)
    st = torch.tensor(s).cuda()
    lt = torch.tensor(lab).cuda().view(torch.uint8)
    a = torch.ops.svb200.verif_metrics(st, lt, flat(P8))
    b = torch.ops.svb200.verif_metrics(st, lt, flat(P8))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = torch.ops.svb200.verif_metrics(st, lt, flat(P8))
    side.synchronize()
    assert torch.equal(a.view(torch.int64), b.view(torch.int64))
    assert torch.equal(a.view(torch.int64), c.view(torch.int64))
    np.testing.assert_array_equal(a.cpu().numpy(), V.metrics(s, lab, P8))


def test_large_input_beyond_l2():
    n = (1 << 25) + 7
    r = np.random.RandomState(99)
    lab = r.rand(n) < 0.01
    s = (r.standard_normal(n).astype(np.float32) + np.float32(2.0) * lab).astype(np.float32)
    got = run_flat(s, lab, P8)
    ref = V.metrics(s, lab, P8)
    np.testing.assert_array_equal(got, ref)
    assert ref[5] > (1 << 24)


def test_opcheck():
    r = np.random.RandomState(2)
    s = torch.tensor(r.standard_normal(5000).astype(np.float32)).cuda()
    lab = torch.tensor(r.rand(5000) < 0.3).cuda().view(torch.uint8)
    sim = torch.tensor(r.standard_normal((12, 3, 12)).astype(np.float32)).cuda()
    torch.library.opcheck(torch.ops.svb200.verif_metrics.default, (s, lab, flat(P8)),
                          test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(torch.ops.svb200.verif_metrics_sim.default, (sim, flat(P1)),
                          test_utils=("test_schema", "test_faketensor"))


def test_cuda_graph_capture_of_the_c_abi():
    """The entry point clears its own counters: two replays of one captured call on different data both match."""
    from pytorch_speaker_verification_b200 import _lib
    L = _lib.lib()
    n = 300_001
    r = np.random.RandomState(31)
    data = []
    for k in range(2):
        lab = r.rand(n) < (0.05 if k == 0 else 0.3)
        s = np.round(r.standard_normal(n) + (1 + k) * lab, 2 + k).astype(np.float32)
        data.append((s, lab))
    scores = torch.empty(n, dtype=torch.float32, device="cuda")
    labels = torch.empty(n, dtype=torch.uint8, device="cuda")
    nb = ctypes.c_size_t(0)
    assert L.svb_verif_workspace_bytes(ctypes.c_int64(n), ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(8 + 4 * len(P8), dtype=torch.float64, device="cuda")
    ops = (ctypes.c_double * (3 * len(P8)))(*flat(P8))
    side = torch.cuda.Stream()

    def call():
        rc = L.svb_verif_metrics(_lib.ptr(scores), _lib.ptr(labels), ctypes.c_int64(n), ops, len(P8), _lib.ptr(ws),
                                 ctypes.c_size_t(nb.value), _lib.ptr(out), ctypes.c_void_p(side.cuda_stream))
        assert rc == 0, L.svb_last_error()

    scores.copy_(torch.tensor(data[1][0]))
    labels.copy_(torch.tensor(data[1][1]).view(torch.uint8))
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()                                                 # warm-up outside the capture
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
        np.testing.assert_array_equal(out.cpu().numpy(), V.metrics(s, lab, P8))
