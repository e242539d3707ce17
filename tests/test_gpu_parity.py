"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures.

Tolerances (BASELINE.json north_star): embeddings 1e-3 per-vector L2-relative (bf16 recurrent GEMM, fp32
accumulate); GE2E loss / dE / dw 1e-5 relative (fp32); db against the float64 oracle (SURVEY 7.5: the fp32
reference itself is 1.7 % off there); EER bit-exact given identical similarity scores; LSTM parameter gradients
(bf16 BPTT operands, no tolerance stated by north_star) 1.2e-2 per-tensor L2-relative for weights, 3e-2 for biases.
"""
import os

import numpy as np
import pytest
import torch

import _inputs as I
from oracle import dvector as odv
from oracle import eer as oeer
from oracle import embedder as oemb
from oracle import ge2e as oge2e

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.fixture(scope="module")
def svb():
    import pytorch_speaker_verification_b200 as m
    return m


@pytest.fixture(scope="module")
def net(svb):
    torch.manual_seed(0)
    n = svb.SpeechEmbedder().cuda()
    g = load("embedder_c1.npz")
    sums = [float(v.double().sum()) for v in n.state_dict().values()]
    np.testing.assert_allclose(sums, g["w_sum"], atol=1e-9, rtol=0)     # same init as the reference's
    return n


# ----------------------------------------------------------------------------------------------- GE2E
@pytest.mark.parametrize("fused", [1, 2, 0])   # 1: per-speaker kernel (all cases are eligible), 2: general, 0: phases
@pytest.mark.parametrize("name", list(I.GE2E_CASES))
def test_ge2e_loss_and_gradients(svb, name, fused):
    N, M, D, kind, w0, b0 = I.GE2E_CASES[name]
    g = load(f"ge2e_{name}.npz")
    Enp = I.ge2e_embeddings(N, M, D, kind)
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    crit = svb.GE2ELoss("cuda")
    crit.fused = fused
    with torch.no_grad():
        crit.w.fill_(w0)
        crit.b.fill_(b0)
    loss = crit(E)
    loss.backward()
    o32 = oge2e.ge2e_fwd_bwd(Enp, w0, b0)
    assert rel(loss.item(), g["loss_f32"]) < 1e-5 and rel(loss.item(), g["loss_f64"]) < 1e-5
    assert rel(loss.item(), o32["loss"]) < 1e-5
    assert rel(E.grad.cpu().numpy(), g["dE_f64"]) < 1e-5
    assert rel(E.grad.cpu().numpy(), o32["dE"]) < 1e-5
    assert rel(crit.w.grad.item(), g["dw_f64"]) < 1e-5
    assert rel(crit.b.grad.item(), g["db_f64"]) < 2e-3     # ill-conditioned; fp32 reference is ~2e-2 off


@pytest.mark.parametrize("shape", [(3, 2, 4), (33, 7, 20), (20, 5, 24), (64, 10, 256), (70, 10, 256), (100, 16, 256), (120, 13, 64),
                                   (37, 9, 512), (74, 2, 8)])
def test_ge2e_speaker_kernel_matches_general_kernel(svb, shape):
    """The one-CTA-per-speaker kernel (small batches) against the general five-phase kernel and the fp64 oracle on
    shapes that exercise its padding (N % 4, N % 32, odd M, D < / > the block size) in both forms: 2-CTA clusters
    splitting D (D % 8 == 0 and 2N <= #SMs) and single CTAs."""
    N, M, D = shape
    r = np.random.RandomState(N * 1000 + M)
    Enp = (r.randn(N, 1, D) + 0.7 * r.randn(N, M, D)).astype(np.float32)
    o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0)
    res = []
    for fused in (1, 2):
        E = torch.tensor(Enp, device="cuda", requires_grad=True)
        crit = svb.GE2ELoss("cuda")
        crit.fused = fused
        loss = crit(E)
        loss.backward()
        assert rel(loss.item(), o["loss"]) < 1e-5
        assert rel(E.grad.cpu().numpy(), o["dE"]) < 1e-5
        assert rel(crit.w.grad.item(), o["dw"]) < 1e-5
        res.append((loss.item(), E.grad.clone()))
    assert rel(res[0][0], res[1][0]) < 1e-6 and rel(res[0][1].cpu().numpy(), res[1][1].cpu().numpy()) < 1e-5
    with torch.no_grad():                                   # forward-only mode of the speaker kernel
        crit = svb.GE2ELoss("cuda")
        assert rel(crit(torch.tensor(Enp, device="cuda")).item(), o["loss"]) < 1e-5


def test_ge2e_tensor_core_path_matches_fp32_path(svb):
    """Large batches (rows x centroids >= 2^18) run cos = E^ C^T, R = A_off C^, P = A_off^T E^ as 3-term split-fp16
    tcgen05 GEMMs between the phase kernels: same loss / dE / dw / db as the fp32 SIMT kernel and the float64 oracle
    (utils.py:72-115,126-132), in the full-batch form, the row-sharded form (svb_ge2e_rows) and get_cossim."""
    from pytorch_speaker_verification_b200 import ops
    N, M, D = 320, 7, 256                                    # 2240 rows x 320 centroids: ragged 128-row tiles
    r = np.random.RandomState(7)
    Enp = (r.randn(N, 1, D) + 0.8 * r.randn(N, M, D)).astype(np.float32)
    o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0)
    out = {}
    try:
        for tc in (True, False):
            ops.set_ge2e_tensor_cores(tc)
            E = torch.tensor(Enp, device="cuda", requires_grad=True)
            crit = svb.GE2ELoss("cuda")
            loss = crit(E)
            loss.backward()
            assert rel(loss.item(), o["loss"]) < 1e-5, tc
            assert rel(E.grad.cpu().numpy(), o["dE"]) < 1e-5, tc
            assert rel(crit.w.grad.item(), o["dw"]) < 1e-5, tc
            Cc = svb.get_centroids(E.detach())
            red, dEr = torch.ops.svb200.ge2e_rows(E.detach()[:160].contiguous(), Cc, crit.w.detach(), crit.b.detach(), 0)
            with torch.no_grad():
                cos = svb.get_cossim(E.detach(), Cc)
            out[tc] = (loss.item(), E.grad.clone(), red.clone(), dEr.clone(), cos.clone())
    finally:
        ops.set_ge2e_tensor_cores(True)
    a, b = out[True], out[False]
    assert rel(a[0], b[0]) < 1e-6
    assert rel(a[1].cpu().numpy(), b[1].cpu().numpy()) < 1e-5
    assert rel(a[2].cpu().numpy(), b[2].cpu().numpy()) < 1e-5 and rel(a[3].cpu().numpy(), b[3].cpu().numpy()) < 1e-5
    assert float((a[4] - b[4]).abs().max()) < 2e-6


def test_ge2e_upstream_scale_and_no_grad(svb):
    N, M, D, kind, w0, b0 = I.GE2E_CASES["c1"]
    Enp = I.ge2e_embeddings(N, M, D, kind)
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    crit = svb.GE2ELoss("cuda")
    (crit(E) * 0.25).backward()
    o = oge2e.ge2e_fwd_bwd(Enp, 10.0, -5.0)
    assert rel(E.grad.cpu().numpy(), 0.25 * o["dE"]) < 1e-5
    assert rel(crit.w.grad.item(), 0.25 * o["dw"]) < 1e-5
    with torch.no_grad():
        l2 = crit(E)
    assert rel(l2.item(), o["loss"]) < 1e-5 and not l2.requires_grad
    with pytest.raises(ValueError):
        crit(torch.randn(3, 1, 8, device="cuda"))          # M = 1: the reference divides by zero


def test_ge2e_large_w_is_stable(svb):
    """exp(S) overflows fp32 in the reference once w + b > 88; the kernel's max-subtraction must give the
    float64 value (quirk 4)."""
    enr, ver = I.eer_embeddings(16, 6, 0.06, 0.3, 99)       # overlapping speakers: cos ~0.9 everywhere
    Enp = np.concatenate([enr, ver], axis=1)
    crit = svb.GE2ELoss("cuda")
    with torch.no_grad():
        crit.w.fill_(100.0)
        crit.b.fill_(20.0)                                    # S ~ 110 > 88: exp overflows in fp32
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    loss = crit(E)
    loss.backward()
    o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 100.0, 20.0)
    assert o["loss"] > 10 and np.isfinite(loss.item())
    assert rel(loss.item(), o["loss"]) < 1e-4
    assert rel(E.grad.cpu().numpy(), o["dE"]) < 1e-4


def test_free_functions_match_reference_api(svb):
    """get_centroids / get_cossim / calc_loss (utils.py) forward and autograd, incl. foreign centroids."""
    g = load("toy.npz")
    E = torch.tensor(g["E"], device="cuda")
    C = svb.get_centroids(E)
    np.testing.assert_array_equal(C.cpu().numpy(), g["centroids"])
    cos = svb.get_cossim(E, C)
    np.testing.assert_allclose(cos.cpu().numpy(), g["cossim"], atol=2e-7, rtol=0)
    loss, per = svb.calc_loss(1.0 * cos + 0.0)
    np.testing.assert_allclose(per.cpu().numpy(), g["per"], rtol=1e-6)
    np.testing.assert_allclose(loss.item(), float(g["loss"]), rtol=1e-6)
    # autograd through the three free functions == closed form
    N, M, D, kind, w0, b0 = I.GE2E_CASES["nonunit"]
    Enp = I.ge2e_embeddings(N, M, D, kind)
    Et = torch.tensor(Enp, device="cuda", requires_grad=True)
    w = torch.tensor(w0, device="cuda", requires_grad=True)
    b = torch.tensor(b0, device="cuda", requires_grad=True)
    S = w * svb.get_cossim(Et, svb.get_centroids(Et)) + b
    l, _ = svb.calc_loss(S)
    l.backward()
    o = oge2e.ge2e_fwd_bwd(Enp, w0, b0)
    assert rel(l.item(), o["loss"]) < 1e-5
    assert rel(Et.grad.cpu().numpy(), o["dE"]) < 2e-5
    assert rel(w.grad.item(), o["dw"]) < 2e-5
    # CPU tensors are accepted and come back on the CPU
    cos_cpu = svb.get_cossim(torch.tensor(Enp), svb.get_centroids(torch.tensor(Enp)))
    assert cos_cpu.device.type == "cpu"
    np.testing.assert_allclose(cos_cpu.numpy(), oge2e.get_cossim(Enp, oge2e.get_centroids(Enp)), atol=3e-6)


# ----------------------------------------------------------------------------------------------- EER
@pytest.mark.parametrize("name", list(I.EER_CASES))
def test_eer_bit_exact(svb, name):
    g = load("eer.npz")
    N, M, sigma, alpha, seed = I.EER_CASES[name]
    enr, ver = I.eer_embeddings(N, M, sigma, alpha, seed)
    exp = [float(v) for v in g[f"{name}.tuple"]]
    if f"{name}.sim" in g:        # identical similarity scores in -> bit-exact tuple out
        got = svb.eer_sweep(torch.tensor(g[f"{name}.sim"]))
        assert [float(v) for v in got] == exp
        ca, cd = oeer.eer_counts(g[f"{name}.sim"])
        from pytorch_speaker_verification_b200 import eer as E, ops
        sim = torch.tensor(g[f"{name}.sim"], device="cuda")
        gca, gcd = ops.eer_counts(sim, E._thresholds_f32(sim.device, E.THRESHOLDS))
        np.testing.assert_array_equal(gca.cpu().numpy().T, ca)
        np.testing.assert_array_equal(gcd.cpu().numpy().T, cd)
    # end to end from embeddings (own similarity kernel): same tuple as the oracle fed the kernel's sim
    (tup, sim) = svb.compute_eer(torch.tensor(enr, device="cuda"), torch.tensor(ver, device="cuda"))
    sim_o = oge2e.get_cossim(ver, oge2e.get_centroids(enr))
    np.testing.assert_allclose(sim.cpu().numpy(), sim_o, atol=3e-6, rtol=0)
    assert [float(v) for v in tup] == [float(v) for v in oeer.eer_sweep(sim.cpu().numpy())]
    np.testing.assert_allclose([float(v) for v in tup], exp, atol=5e-3)


def test_eer_threshold_rounding_and_scale(svb):
    t = oeer.THRESHOLDS[7]
    sim = torch.full((2, 1, 2), float(np.float32(t)), dtype=torch.float32)
    from pytorch_speaker_verification_b200 import eer as E, ops
    sg = sim.cuda()
    ca, _ = ops.eer_counts(sg, E._thresholds_f32(sg.device, E.THRESHOLDS))
    assert ca[:, 7].sum().item() == 0 and ca[:, 6].sum().item() == 4
    # BASELINE config 5 size through size-independent properties: counts monotone in the threshold,
    # diagonal counts <= Mv, totals match a float64 numpy recount on a sample of thresholds
    N, Mv = 1024, 3
    enr, ver = I.eer_embeddings(N, 6, 0.06, 0.5, 4242)
    tup, sim = svb.compute_eer(torch.tensor(enr, device="cuda"), torch.tensor(ver, device="cuda"))
    ca, cd = ops.eer_counts(sim, E._thresholds_f32(sim.device, E.THRESHOLDS))
    ca, cd = ca.cpu().numpy(), cd.cpu().numpy()
    assert (np.diff(ca, axis=1) <= 0).all() and (np.diff(cd, axis=1) <= 0).all() and cd.max() <= Mv
    s = sim.cpu().numpy()
    for ti in (0, 13, 49):
        assert ca[:, ti].sum() == int((s > np.float32(oeer.THRESHOLDS[ti])).sum())
    assert [float(v) for v in tup] == [float(v) for v in oeer.eer_sweep(s)]


# ----------------------------------------------------------------------------------------------- d-vectors
def test_dvector_windows_alignment(svb):
    g = load("dvector.npz")
    for T in (37, 160):
        p = np.sqrt(I.power_spec(T, seed=T)) ** 2
        S = np.log10(np.dot(np.eye(40, dtype=np.float32), p) + 1e-6).astype(np.float32)
        np.testing.assert_array_equal(svb.get_windows(torch.tensor(S)).numpy(), g[f"win_T{T}"])
    assert tuple(svb.get_windows(torch.zeros(40, 24)).shape) == (0, 24, 40)
    for W in (1, 2, 3, 5, 13, 30, 82):
        out = svb.align_embeddings(I.unit_rows(W, 256, seed=W))
        assert out.dtype == np.float64
        np.testing.assert_array_equal(out, g[f"align_W{W}"])
    from pytorch_speaker_verification_b200 import dvector as D
    for T in list(range(0, 80)) + [160, 180, 301, 1000]:
        assert list(D.window_starts(T)) == odv.window_starts(T)
    for W in range(0, 90):
        offs = D.partition_offsets(W)
        if W:
            assert [(int(a), int(b)) for a, b in zip(offs[:-1], offs[1:])] == odv.partitions(W)


def test_extract_dvectors_batched_equals_per_file(svb, net):
    rng = np.random.RandomState(5)
    specs = [np.log10(I.power_spec(int(T), seed=int(T)) + 1e-6).astype(np.float32) for T in (20, 61, 130, 300)]
    outs = svb.extract_dvectors(net, specs)
    assert outs[0].shape == (0, 256)
    for S, o in zip(specs[1:], outs[1:]):
        with torch.no_grad():
            emb = net(svb.get_windows(torch.tensor(S)))                       # dvector_create.py:98-100 per file
        np.testing.assert_allclose(o, svb.align_embeddings(emb.cpu().numpy()), atol=2e-6)
        ref = odv.align_embeddings(emb.cpu().numpy())
        np.testing.assert_array_equal(svb.align_embeddings(emb.cpu().numpy()), ref)
    # chunked pipeline: many small chunks (incl. chunks whose utterances have no window) == one chunk, twice (the
    # pinned staging buffers are reused between calls)
    lens = [int(t) for t in rng.randint(10, 400, size=40)] + [24, 25, 12]
    many = [np.log10(I.power_spec(T, seed=T) + 1e-6).astype(np.float32) for T in lens]
    one = svb.extract_dvectors(net, many, chunk_frames=1 << 30)
    for _ in range(2):
        small = svb.extract_dvectors(net, many, chunk_frames=300)
        assert len(small) == len(one) == len(many)
        for a, b in zip(small, one):
            assert a.shape == b.shape
            np.testing.assert_allclose(a, b, atol=2e-6)
    assert svb.extract_dvectors(net, []) == []


# ----------------------------------------------------------------------------------------------- embedder
def emb_err(a, b):
    return (np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)).max()


def test_embedder_forward_matches_reference(svb, net):
    g = load("embedder_c1.npz")
    x = torch.tensor(I.logmel(20, 180, seed=1234))
    with torch.no_grad():
        e = net(x.cuda()).cpu().numpy()
        e24 = net(torch.tensor(I.logmel(7, 24, seed=4321)).cuda()).cpu().numpy()
        e64 = net(x[:3].double())                     # float64 CPU input: staged, computed in fp32, back on CPU
    assert emb_err(e, g["emb"]) < 1e-3, emb_err(e, g["emb"])
    assert emb_err(e24, g["emb_T24"]) < 1e-3
    assert e64.device.type == "cpu" and e64.dtype == torch.float32
    assert emb_err(e64.numpy(), g["emb_from_f64_input"]) < 1e-3
    np.testing.assert_allclose(np.linalg.norm(e, axis=1), 1.0, atol=1e-5)
    print("embedding err C1:", emb_err(e, g["emb"]), "T24:", emb_err(e24, g["emb_T24"]))


def test_persistent_and_per_frame_kernels_agree(svb, net):
    """The persistent wavefront kernel (weights stationary in tensor memory, all layers in one launch, flag-ordered
    tiles; MUFU.TANH activations, single-term fp16 layer-0 projection) and the per-frame kernels (3-term layer-0
    projection, ex2/rcp activations) both meet the 1e-3 embedding bar and agree with each other well inside it;
    their BPTT stashes give the same gradients within the gradient tolerance."""
    from pytorch_speaker_verification_b200 import ops
    g = load("embedder_c1.npz")
    x = torch.tensor(I.logmel(20, 180, seed=1234)).cuda()
    xb = torch.tensor(I.logmel(300, 50, seed=77)).cuda()          # 5 batch tiles, ragged last tile
    try:
        out = {}
        for mode in (True, False):
            ops.set_persistent(mode)
            with torch.no_grad():
                out[mode] = (net(x), net(xb))
            net.zero_grad()
            e = net(xb[:140])
            e.square().sum().mul(0.5).add(e.sum()).backward()
            out[mode] += (net.LSTM_stack.weight_hh_l0.grad.clone(), net.LSTM_stack.weight_ih_l2.grad.clone(),
                          net.LSTM_stack.bias_ih_l1.grad.clone(), net.LSTM_stack.weight_ih_l0.grad.clone())
    finally:
        ops.set_persistent(True)
    for mode in (True, False):
        assert emb_err(out[mode][0].cpu().numpy(), g["emb"]) < 1e-3, (mode, emb_err(out[mode][0].cpu().numpy(), g["emb"]))
    for a, b in zip(out[True][:2], out[False][:2]):
        assert emb_err(a.cpu().numpy(), b.cpu().numpy()) < 5e-4
    for a, b in zip(out[True][2:], out[False][2:]):
        assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) < 2e-2, rel_l2(a.cpu().numpy(), b.cpu().numpy())
    print("persistent vs golden:", emb_err(out[True][0].cpu().numpy(), g["emb"]),
          "per-frame vs golden:", emb_err(out[False][0].cpu().numpy(), g["emb"]))


@pytest.mark.parametrize("B,T", [(1540, 9), (1700, 6), (2100, 5), (3072, 4)])
def test_persistent_forward_chunked_tile_order(svb, net, B, T):
    """Batches of 24 or more 64-row tiles are walked in chunks of 16 tiles, all frames of a chunk before the next
    chunk (merged tail, ragged last tile): every row must equal the row computed in a small batch (bit for bit: the
    per-row arithmetic does not depend on the batch), inference and training forward, under a NaN-poisoned workspace;
    and the training stash written in that order must give the per-frame path's gradients."""
    from pytorch_speaker_verification_b200 import ops
    x = torch.tensor(I.logmel(B, T, seed=B)).cuda()
    try:
        ops.set_poison_workspace(True)
        with torch.no_grad():
            big = net(x)
            assert not torch.isnan(big).any()
            for lo in (0, 960, 1024, B - 70):
                assert torch.equal(net(x[lo:lo + 70]), big[lo:lo + 70]), lo
        grads = {}
        for mode in (True, False):
            ops.set_persistent(mode)
            ops.set_persistent_bwd(mode)
            net.zero_grad()
            e = net(x)
            if mode:
                assert torch.equal(e.detach(), big)
            e.square().sum().mul(0.5).add(e.sum()).backward()
            grads[mode] = [p.grad.clone() for p in net.parameters()]
        for a, b in zip(grads[True], grads[False]):
            assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) < 2e-2
    finally:
        ops.set_poison_workspace(False)
        ops.set_persistent(True)
        ops.set_persistent_bwd(True)


def test_persistent_bptt_matches_per_frame_bptt(svb, net):
    """The persistent wavefront BPTT kernel (split-K over 4-CTA clusters with a DSMEM reduction, dX products fused
    in) and the per-frame BPTT kernels + batched dX GEMMs consume the same stash and agree on every parameter
    gradient far inside the gradient tolerance."""
    from pytorch_speaker_verification_b200 import ops
    out = {}
    try:
        for (B, T) in ((20, 6), (140, 50), (300, 21)):
            x = torch.tensor(I.logmel(B, T, seed=B + T)).cuda()
            for mode in (True, False):
                ops.set_persistent_bwd(mode)
                net.zero_grad()
                e = net(x)
                e.square().sum().mul(0.5).add(e.sum()).backward()
                out[mode] = {k: p.grad.clone() for k, p in net.named_parameters()}
            for k in out[True]:
                assert torch.isfinite(out[True][k]).all(), k
                assert rel_l2(out[True][k].cpu().numpy(), out[False][k].cpu().numpy()) < 2e-3, (B, T, k)
    finally:
        ops.set_persistent_bwd(True)


def test_weight_gradient_overlap_matches_serial(svb, net):
    """Late-frame weight-gradient slices running beside the BPTT kernel (gated by its release counters) against the
    same products computed after it: identical up to the fp32 order of three partial sums; repeated, because a slice
    that started before its dG frames were complete would read gate activations instead of gradients."""
    from pytorch_speaker_verification_b200 import ops
    try:
        for (B, T) in ((640, 40), (128, 64), (70, 160)):
            x = torch.tensor(I.logmel(B, T, seed=B + T)).cuda()
            ref = None
            for mode, reps in ((False, 1), (True, 6)):
                ops.set_wgrad_overlap(mode)
                for _ in range(reps):
                    net.zero_grad()
                    e = net(x)
                    e.square().sum().mul(0.5).add(e.sum()).backward()
                    torch.cuda.synchronize()
                    got = {k: p.grad.clone() for k, p in net.named_parameters()}
                    if ref is None:
                        ref = got
                    for k in got:
                        assert rel_l2(got[k].cpu().numpy(), ref[k].cpu().numpy()) < 1e-5, (B, T, mode, k)
    finally:
        ops.set_wgrad_overlap(True)


def test_persistent_kernel_no_stale_reads(svb, net):
    """Flag protocol of the persistent kernel under a NaN-poisoned workspace: a tile read before its producer's
    stores are visible shows up as NaN (this is how the missing release on the h-tile counter was found).  Small
    batches keep producer and consumer closest in time; results must also be run-to-run identical and independent of
    the batch composition."""
    from pytorch_speaker_verification_b200 import ops
    try:
        ops.set_poison_workspace(True)
        for (B, T) in ((35, 24), (50, 40), (100, 40), (200, 30), (640, 20)):
            x = torch.tensor(I.logmel(B, T, seed=B)).cuda()
            with torch.no_grad():
                ref = net(x)
                assert not torch.isnan(ref).any()
                for _ in range(25):
                    assert torch.equal(net(x), ref)
                assert torch.equal(net(x[:B // 3]), ref[:B // 3])
            net.zero_grad()
            net(x).square().sum().backward()
            g1 = net.LSTM_stack.weight_hh_l1.grad.clone()
            net.zero_grad()
            net(x).square().sum().backward()
            assert torch.isfinite(g1).all() and torch.equal(g1, net.LSTM_stack.weight_hh_l1.grad)
    finally:
        ops.set_poison_workspace(False)


def test_embedder_saturated_weights(svb):
    g = load("embedder_saturated.npz")
    sat = I.saturating_weights({k: v.numpy() for k, v in oemb.init_state_dict(seed=0).items()})
    n = svb.SpeechEmbedder().cuda()
    n.load_state_dict({k: torch.tensor(v) for k, v in sat.items()})
    x = torch.tensor(I.logmel(20, 180, seed=1234)).cuda()
    errs = {}
    for terms in (1, 2, 3):
        n.recurrent_terms = terms
        with torch.no_grad():
            errs[terms] = emb_err(n(x).cpu().numpy(), g["emb"])
    print("embedding err, weights x2.5, recurrent terms 1/2/3:", errs)
    # x2.5 weights amplify the operand rounding of W_hh; with fp16 operands (11-bit significands) the default single
    # term holds north_star's 1e-3 bar on this stress case too (6.4e-4 measured), the residual terms stay inside it
    assert errs[3] < 1e-3 and errs[2] < 1e-3 and errs[1] < 1e-3, errs


def test_embedder_batch_independence_and_ragged_batch(svb, net):
    """Rows are independent (the caller's permutation at train_speech_embedder.py:48-57 is a no-op) and a batch
    that is not a multiple of the 128-row tile gives the same rows as a padded one."""
    x = torch.tensor(I.logmel(150, 40, seed=9)).cuda()
    with torch.no_grad():
        full = net(x)
        perm = torch.randperm(150, device="cuda")
        assert torch.equal(net(x[perm]), full[perm])
        assert torch.equal(net(x[:37]), full[:37])


def test_train_step_gradients(svb, net):
    """Full C1 train step (embedder + GE2E) against the explicit-cell oracle's autograd."""
    g = load("embedder_c1.npz")
    x = torch.tensor(I.logmel(20, 180, seed=1234))
    crit = svb.GE2ELoss("cuda")
    net.zero_grad()
    emb = net(x.cuda())
    loss = crit(emb.reshape(4, 5, -1))
    loss.backward()
    assert rel(loss.item(), g["loss"]) < 1e-3           # loss through bf16 embeddings
    sd = {k: v.clone().requires_grad_(True) for k, v in oemb.init_state_dict(seed=0).items()}
    e_o = oemb.embedder_explicit(x, sd)
    w = torch.tensor(10.0, requires_grad=True)
    b = torch.tensor(-5.0, requires_grad=True)
    oemb.library_ge2e_loss(e_o.reshape(4, 5, -1), w, b).backward()
    errs = {}
    for k, p in net.named_parameters():
        go = sd[k].grad.numpy()
        assert abs(np.linalg.norm(go) - float(g[f"gnorm.{k}"])) < 2e-3 * float(g[f"gnorm.{k}"])   # oracle == reference
        errs[k] = rel_l2(p.grad.cpu().numpy(), go)
    print("per-tensor grad rel-L2:", {k: round(float(v), 4) for k, v in errs.items()})
    # fp16 gate stash + bf16 dG / W^T operands (scripts/precision_study_bwd.py: weights 7e-3, biases 0.8-2.1e-2; the
    # bf16 gate stash of round 1 gave 1.4e-2 / 2-9e-2)
    for k, e in errs.items():
        assert e < (3e-2 if "bias" in k else 1.2e-2), (k, e)
    assert rel(crit.w.grad.item(), w.grad.item()) < 2e-2


def test_state_dict_roundtrip_and_cpu_module(svb):
    """Checkpoints are wire-compatible with the reference (14 keys) and a module left on the CPU (test(),
    dvector_create.py) still computes on the GPU."""
    torch.manual_seed(0)
    n = svb.SpeechEmbedder()
    assert list(n.state_dict().keys()) == oemb.PARAM_NAMES
    x = torch.tensor(I.logmel(5, 30, seed=3))
    with torch.no_grad():
        e_cpu_module = n(x)
        e_gpu_module = svb.SpeechEmbedder().cuda()
        e_gpu_module.load_state_dict(n.state_dict())
        e2 = e_gpu_module(x.cuda()).cpu()
    assert e_cpu_module.device.type == "cpu"
    assert torch.equal(e_cpu_module, e2)


def test_full_size_c2_parameter_gradients_vs_reference_library(svb, net):
    """BASELINE configs[1] (64 speakers x 10 utterances x 160 frames): every parameter gradient of the full train step
    against the reference's own library path on the CPU (nn.LSTM / nn.Linear / F.cosine_similarity autograd, float32:
    oracle.embedder.LibraryEmbedder + library_ge2e_loss, the calls speech_embedder_net.py:19-49 makes)."""
    xn = I.logmel(640, 160, seed=1234)
    crit = svb.GE2ELoss("cuda")
    net.zero_grad()
    loss = crit(net(torch.tensor(xn).cuda()).reshape(64, 10, -1))
    loss.backward()
    torch.manual_seed(0)
    ref = oemb.LibraryEmbedder()
    assert all(torch.equal(a, b.cpu()) for a, b in zip(ref.state_dict().values(), net.state_dict().values()))
    w = torch.tensor(10.0, requires_grad=True)
    b = torch.tensor(-5.0, requires_grad=True)
    torch.set_num_threads(os.cpu_count() or 8)
    lo = oemb.library_ge2e_loss(ref(torch.tensor(xn)).reshape(64, 10, -1), w, b)
    lo.backward()
    assert rel(loss.item(), lo.item()) < 1e-3
    errs = {k: rel_l2(p.grad.cpu().numpy(), dict(ref.named_parameters())[k].grad.numpy()) for k, p in net.named_parameters()}
    print("C2 per-tensor grad rel-L2:", {k: round(float(v), 4) for k, v in errs.items()})
    for k, e in errs.items():
        assert e < (3e-2 if "bias" in k else 1.2e-2), (k, e)
    assert rel(crit.w.grad.item(), w.grad.item()) < 2e-2


def test_bptt_is_invariant_to_the_gradient_scale(svb, net):
    """BPTT runs under a power-of-two scale taken from max |dL/dh_last| (csrc/lstm.cu grad_scale_kernel), so that the
    fp16 split-K partials of the persistent kernel never see a trained model's tiny gradients (or a huge SUM loss) in
    their subnormal / overflow range: gradients of c * loss are c * gradients -- bit for bit when c is a power of two,
    within rounding for any c -- from 1e-9 to 1e+6, on the persistent and the per-frame path."""
    from pytorch_speaker_verification_b200 import ops
    x = torch.tensor(I.logmel(140, 40, seed=21)).cuda()
    v = torch.tensor(np.random.RandomState(4).randn(140, 256).astype(np.float32)).cuda()

    def grads(c):
        net.zero_grad()
        ((net(x) * v).sum() * c).backward()
        return {k: p.grad.double().clone() for k, p in net.named_parameters()}

    try:
        for mode in (True, False):
            ops.set_persistent_bwd(mode)
            base = grads(1.0)
            for c in (2.0 ** -24, 2.0 ** 17):
                g = grads(c)
                for k in base:
                    assert torch.equal(g[k], base[k] * c), (mode, c, k)
            for c in (1e-9, 1e-4, 1e3, 1e6):
                g = grads(c)
                for k in base:
                    assert rel_l2(g[k].cpu().numpy(), (base[k] * c).cpu().numpy()) < 3e-3, (mode, c, k)
    finally:
        ops.set_persistent_bwd(True)
    net.zero_grad()
    (net(x) * 0.0).sum().backward()                          # zero upstream gradient: scale 1, gradients exactly 0
    assert all(float(p.grad.abs().max()) == 0.0 for p in net.parameters())


def test_second_backward_raises_and_repack(svb, net):
    """BPTT consumes the stash in place: a second backward through the same forward raises instead of returning
    garbage; weights changed behind autograd's back (``p.data``) are picked up after ``repack()``; a pending graph
    keeps the weight shadow it was built with when the weights change before its backward."""
    import copy
    m = copy.deepcopy(net)
    x = torch.tensor(I.logmel(12, 20, seed=7)).cuda()
    e = m(x)
    e.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="second backward"):
        e.sum().backward()
    with torch.no_grad():
        e0 = m(x)
        m.LSTM_stack.weight_hh_l1.data.mul_(1.5)              # bypasses the version counter
        assert torch.equal(m(x), e0)                          # documented: not seen ...
        m.repack()
        e1 = m(x)
        assert not torch.equal(e1, e0)                        # ... until repack()
        m.LSTM_stack.weight_hh_l1.mul_(1.0 / 1.5)             # a tracked in-place update is seen by itself
        assert emb_err(m(x).cpu().numpy(), e0.cpu().numpy()) < 1e-3
    # a pending graph keeps its own weight shadow: a weight update re-packs into a FRESH buffer
    m2 = copy.deepcopy(net)
    ea = m2(x)
    old = m2._cache.buf
    old_ptr, snapshot = old.data_ptr(), old.clone()
    with torch.no_grad():
        m2.LSTM_stack.weight_hh_l2.add_(0.05)
        m2(x)
    assert m2._cache.buf.data_ptr() != old_ptr and torch.equal(old, snapshot)
    del ea


def test_module_device_round_trip_like_the_checkpoint_code(svb):
    """train_speech_embedder.py:77-82: ``embedder_net.eval().cpu()`` -> ``torch.save(state_dict)`` ->
    ``.to(device).train()``; the weight shadows follow the parameters across the moves."""
    import io
    torch.manual_seed(0)
    m = svb.SpeechEmbedder().cuda()
    x = torch.tensor(I.logmel(9, 30, seed=5)).cuda()
    with torch.no_grad():
        e0 = m(x)
    m.eval().cpu()
    buf = io.BytesIO()
    torch.save(m.state_dict(), buf)
    with torch.no_grad():
        assert torch.equal(m(x.cpu()), e0.cpu())              # CPU-resident module, CPU input: computed on the GPU
    m.to("cuda").train()
    with torch.no_grad():
        assert torch.equal(m(x), e0)
    opt = torch.optim.SGD(m.parameters(), lr=0.5)
    m(x).sum().backward()
    opt.step()
    with torch.no_grad():
        e1 = m(x)
    assert not torch.equal(e1, e0)
    buf.seek(0)
    m.load_state_dict(torch.load(buf))
    with torch.no_grad():
        assert torch.equal(m(x), e0)
    # a module left on the CPU trains too: gradients arrive on the CPU parameters
    mc = svb.SpeechEmbedder()
    mc.load_state_dict(m.state_dict())
    mc(x.cpu()).square().sum().backward()
    m.zero_grad()
    m(x).square().sum().backward()
    for (k, a), b in zip(mc.named_parameters(), m.parameters()):
        assert a.grad.device.type == "cpu" and torch.equal(a.grad, b.grad.cpu()), k


def test_centroid_kernels_bit_exact(svb):
    """utils.get_centroids / get_utterance_centroids (utils.py:27-29, 40-58) against the reference's float32 bit
    patterns (tests/golden/centroids.npz), and the autograd of get_utterance_centroids."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from make_golden_centroids import CASES, bits_checksum, case_input
    g = load("centroids.npz")
    for (N, M, D, seed) in CASES:
        E = case_input(N, M, D, seed)
        tag = f"{N}x{M}x{D}"
        C = svb.get_centroids(torch.tensor(E, device="cuda")).cpu().numpy()
        U = svb.utils.get_utterance_centroids(torch.tensor(E, device="cuda")).cpu().numpy()
        assert (bits_checksum(C) == g[f"{tag}.C_sum"]).all(), tag
        assert (bits_checksum(U) == g[f"{tag}.U_sum"]).all(), tag
        np.testing.assert_array_equal(U.ravel()[g[f"{tag}.U_idx"]], g[f"{tag}.U_val"])
    E = torch.tensor(case_input(7, 3, 16, 3), requires_grad=True)             # CPU in -> CPU out, differentiable
    V = torch.tensor(np.random.RandomState(0).randn(7, 3, 16).astype(np.float32))
    U = svb.utils.get_utterance_centroids(E)
    assert U.device.type == "cpu"
    (U * V).sum().backward()
    want = (V.sum(dim=1, keepdim=True) - V) / 2.0
    np.testing.assert_allclose(E.grad.numpy(), want.numpy(), rtol=1e-6, atol=1e-6)
    with pytest.raises(ValueError):
        svb.utils.get_utterance_centroids(torch.randn(3, 1, 8))


@pytest.mark.parametrize("N,M,D,shards", [(8, 4, 32, 2), (64, 10, 256, 8), (512, 10, 256, 8), (12, 3, 20, 3),
                                          (264, 16, 192, 2)])
def test_ge2e_row_shards_sum_to_the_global_batch(svb, N, M, D, shards):
    """svb_ge2e_rows (multi-GPU design A: a rank's rows against the all-gathered centroids) on one GPU: the shards'
    partial losses / dw / db / centroid gradients sum to the global batch's (fp64 closed form), and
    dE_rows + dC_total[own speaker] / M is the global dL/dE."""
    Enp = I.ge2e_embeddings(N, M, D, "clustered" if N >= 64 else "raw")
    o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0)
    E = torch.tensor(Enp, device="cuda")
    w = torch.tensor(10.0, device="cuda")
    b = torch.tensor(-5.0, device="cuda")
    C = svb.get_centroids(E)
    nl = N // shards
    reds, dEs = [], []
    from pytorch_speaker_verification_b200 import ops
    try:
        ops.set_poison_workspace(True)              # workspace and outputs start as NaN: every element must be written
        for r in range(shards):
            red, dE = torch.ops.svb200.ge2e_rows(E[r * nl:(r + 1) * nl].contiguous(), C, w, b, r * nl)
            reds.append(red.double())
            dEs.append(dE)
    finally:
        ops.set_poison_workspace(False)
    red = torch.stack(reds).sum(dim=0)
    dC = red[:N * D].view(N, D).float()
    assert rel(red[N * D].item(), o["loss"]) < 1e-5
    assert rel(red[N * D + 1].item(), o["dw"]) < 1e-5
    assert rel(red[N * D + 2].item(), o["db"]) < 2e-3
    dE = torch.cat(dEs) + torch.ops.svb200.centroids_bwd(dC.contiguous(), M)
    assert rel(dE.cpu().numpy(), o["dE"]) < 1e-5


def test_torch_custom_ops_are_registered(svb, net):
    """The C ABI is reachable as torch.ops.svb200.* (schema, CUDA kernel, fake kernel, autograd): direct calls and
    torch.library.opcheck on the differentiable entry points."""
    from pytorch_speaker_verification_b200 import ops
    for name in ops.OP_NAMES:
        assert hasattr(torch.ops.svb200, name), name
    E = torch.tensor(I.ge2e_embeddings(6, 4, 32, "unit"), device="cuda")
    C = torch.ops.svb200.centroids(E)
    cos = torch.ops.svb200.cossim(E, C)
    loss, per = torch.ops.svb200.calc_loss(10.0 * cos - 5.0)
    o = oge2e.ge2e_fwd_bwd(E.cpu().numpy(), 10.0, -5.0)
    assert rel(loss.item(), o["loss"]) < 1e-5
    l2 = torch.ops.svb200.ge2e_loss(E, torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda"), 1, True)
    assert rel(l2[0].item(), o["loss"]) < 1e-5 and rel(l2[1].cpu().numpy(), o["dE"]) < 1e-5
    with pytest.raises((NotImplementedError, RuntimeError)):
        torch.ops.svb200.centroids(E.cpu())                   # no CPU kernel is registered
    Er = E.clone().requires_grad_(True)
    Cr = C.clone().requires_grad_(True)
    w = torch.tensor(10.0, device="cuda", requires_grad=True)
    b = torch.tensor(-5.0, device="cuda", requires_grad=True)
    chk = torch.library.opcheck
    chk(torch.ops.svb200.centroids.default, (Er,))
    chk(torch.ops.svb200.utterance_centroids.default, (Er,))
    chk(torch.ops.svb200.cossim.default, (Er, Cr))
    chk(torch.ops.svb200.calc_loss.default, ((10.0 * cos - 5.0).detach().requires_grad_(True),))
    chk(torch.ops.svb200.ge2e_loss.default, (Er, w, b, 1, True))
    chk(torch.ops.svb200.eer_sweep.default, (cos.detach()[:, :2].contiguous(), torch.tensor([0.5, 0.7], device="cuda")))
    chk(torch.ops.svb200.segment_mean.default, (E.reshape(24, 32), torch.tensor([0, 5, 24], dtype=torch.int32, device="cuda")))
    # embedder: schema / fake / autograd registration (the backward consumes its stash, so the two-run AOT comparison
    # of opcheck is left out for it)
    x = torch.tensor(I.logmel(12, 20, seed=7)).cuda()
    params = net._ordered_params()
    packed = torch.ops.svb200.pack_weights([p.detach() for p in params[:12]], 40, 768, 3)
    chk(torch.ops.svb200.embedder_fwd.default, (x, params, packed, 768, 3, True, 1),
        test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))
    emb, ws = torch.ops.svb200.embedder_fwd(x, params, packed, 768, 3, True, 1)
    with torch.no_grad():
        assert torch.equal(emb, net(x))


def test_overlapped_reducer_orders_reductions_before_autograd(svb, net):
    """dist.OverlappedGradReducer with a stand-in "all-reduce" that doubles each bucket asynchronously on another
    stream: the doubled values must be what autograd sees, whether it adopts the bucket views as p.grad
    (set_to_none=True) or ADDS them to existing gradients (set_to_none=False / gradient accumulation)."""
    from pytorch_speaker_verification_b200.dist import OverlappedGradReducer
    x = torch.tensor(I.logmel(70, 30, seed=3)).cuda()
    side = torch.cuda.Stream()

    class Work:
        def __init__(self, ev):
            self.ev = ev

        def wait(self):
            torch.cuda.current_stream().wait_event(self.ev)

    def fake_all_reduce(t):
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            torch.cuda._sleep(20_000_000)                     # ~10 ms: a late reduction would be seen as x1
            t.mul_(2.0)
            ev = torch.cuda.Event()
            ev.record()
        return Work(ev)

    net.zero_grad()
    net(x).square().sum().backward()
    base = [p.grad.clone() for p in net.parameters()]
    red = OverlappedGradReducer(all_reduce=fake_all_reduce)
    net.zero_grad(set_to_none=True)
    with red:
        net(x).square().sum().backward()
    assert red.buckets == 4
    for p, g in zip(net.parameters(), base):
        assert torch.equal(p.grad, 2.0 * g)
    for p in net.parameters():                                # existing gradients: autograd accumulates
        p.grad = torch.ones_like(p)
    with red:
        net(x).square().sum().backward()
    for p, g in zip(net.parameters(), base):
        assert torch.equal(p.grad, 1.0 + 2.0 * g)
    net.zero_grad()


# ----------------------------------------------------------------------------------------------- optimizer tail
def test_fused_clip_sgd_matches_clip_grad_norm_and_sgd(svb, net):
    """svb.FusedClipSGD (csrc/optim.cu) against the torch entry points train_speech_embedder.py:63-65 calls
    (oracle.optim.clip_sgd_library): updated parameters, clipped gradients and the returned norms."""
    from oracle import optim as ooptim
    import copy
    r = np.random.RandomState(3)
    m = copy.deepcopy(net)
    crit = svb.GE2ELoss("cuda")
    groups = []
    for params, mn, gscale in ((list(m.parameters()), 3.0, 0.02), (list(crit.parameters()), 1.0, 0.1)):
        pg = []
        for p in params:
            g = np.asarray(r.randn(*p.shape) * gscale, dtype=np.float32)
            p.grad = torch.tensor(g, device="cuda").reshape(p.shape)
            pg.append((p.detach().cpu().numpy().copy(), g))
        groups.append((pg, mn))
    versions = [p._version for p in m.parameters()]
    opt = svb.FusedClipSGD([{"params": m.parameters(), "max_norm": 3.0}, {"params": crit.parameters(), "max_norm": 1.0}],
                           lr=0.01)
    norms = opt.step().cpu().numpy()
    pl, gl, nl = ooptim.clip_sgd_library(groups, 0.01)
    assert nl[0] > 3.0 and nl[1] < 1.0                       # first group clips, second does not
    exact = [np.sqrt(sum(float((g.astype(np.float64) ** 2).sum()) for _, g in pg)) for pg, _ in groups]
    np.testing.assert_allclose(norms, exact, rtol=1e-6)      # fp64 above the per-thread sums
    np.testing.assert_allclose(norms, nl, rtol=2e-4)         # the library's own fp32 norm-of-norms (3.7e-5 off here)
    for ps, ref_p, ref_g in zip((list(m.parameters()), list(crit.parameters())), pl, gl):
        for p, rp, rg in zip(ps, ref_p, ref_g):
            np.testing.assert_allclose(p.grad.cpu().numpy(), rg, rtol=2e-4, atol=1e-9)     # inherits the norm difference
            np.testing.assert_allclose(p.detach().cpu().numpy(), rp, rtol=3e-7, atol=2e-9)
    assert all(p._version > v for p, v in zip(m.parameters(), versions))     # weight shadows get re-packed
    opt.zero_grad()
    assert all(p.grad is None for p in m.parameters())
    # a training step through the fused tail lowers the loss like the stock tail does
    x = torch.tensor(I.logmel(12, 20, seed=7)).cuda()
    l0 = crit(m(x).reshape(4, 3, -1))
    l0.backward()
    opt.step()
    with torch.no_grad():
        l1 = crit(m(x).reshape(4, 3, -1))
    assert l1.item() < l0.item()


def test_prefetch_yields_every_batch_in_order(svb):
    """staging.prefetch: (N, M, T, F) host batches arrive on the device reshaped to (N*M, T, F), in order, through
    reused page-locked buffers (more batches than buffers)."""
    r = np.random.RandomState(0)
    batches = [torch.tensor(r.randn(3, 2, 5 + i, 4).astype(np.float32)) for i in range(7)]
    got = list(svb.prefetch(batches, "cuda", depth=2))
    assert len(got) == len(batches)
    for b, g in zip(batches, got):
        assert g.is_cuda and g.shape == (6, b.shape[2], 4)
        assert torch.equal(g.cpu(), b.reshape(6, b.shape[2], 4))
    assert list(svb.prefetch([], "cuda")) == []


# ----------------------------------------------------------------------------------------------- BASELINE full sizes
def test_full_size_c2_embedder_properties(svb, net):
    """BASELINE configs[1] size (640 utterances x 160 frames): a sample of rows against the fp32 oracle, unit norms,
    batch independence at full size, and linearity of the parameter gradients in the batch (loss separable per row:
    grads(640 rows) = grads(first 320) + grads(last 320))."""
    xn = I.logmel(640, 160, seed=1234)
    x = torch.tensor(xn).cuda()
    with torch.no_grad():
        full = net(x)
        assert torch.equal(net(x[100:164]), full[100:164])
        np.testing.assert_allclose(full.norm(dim=1).cpu().numpy(), 1.0, atol=2e-6)
        sd = oemb.init_state_dict(seed=0)
        rows = [0, 77, 319, 320, 500, 639]
        e_ref = oemb.embedder_explicit(torch.tensor(xn[rows]), sd).numpy()
    assert emb_err(full[rows].cpu().numpy(), e_ref) < 1e-3
    grads = []
    for part in (x, x[:320], x[320:]):
        net.zero_grad()
        e = net(part)
        e.square().sum().mul(0.5).add(e[:, :7].sum()).backward()
        grads.append({k: p.grad.double().clone() for k, p in net.named_parameters()})
    for k in grads[0]:
        assert rel_l2((grads[1][k] + grads[2][k]).cpu().numpy(), grads[0][k].cpu().numpy()) < 2e-3, k


def test_full_size_c3_ge2e_and_c5_eer(svb):
    """BASELINE configs[2] loss (N = 512 x M = 10, the global batch every rank evaluates) against the fp64 closed form,
    and configs[4] (EER at N = 1024, M = 6): the kernel's tuple equals the oracle sweep over the same similarities."""
    Enp = I.ge2e_embeddings(512, 10, 256, "clustered")
    o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0)
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    crit = svb.GE2ELoss("cuda")
    loss = crit(E)
    loss.backward()
    assert rel(loss.item(), o["loss"]) < 1e-5
    assert rel(E.grad.cpu().numpy(), o["dE"]) < 1e-5
    assert rel(crit.w.grad.item(), o["dw"]) < 1e-5
    enr, ver = I.eer_embeddings(1024, 6, 0.06, 0.5, 4242)
    tup, sim = svb.compute_eer(torch.tensor(enr, device="cuda"), torch.tensor(ver, device="cuda"))
    assert sim.shape == (1024, 3, 1024)
    assert [float(v) for v in tup] == [float(v) for v in oeer.eer_sweep(sim.cpu().numpy())]
    assert 0.0 < float(tup[0]) < 0.5


# ----------------------------------------------------------------------------------------------- front end (8(f)-4)
def test_log_mel_front_end_matches_oracle(svb, net):
    """svb.log_mel_spectrogram (csrc/frontend.cu) against the float64 restatement of librosa's stft / filters.mel
    (oracle/frontend.py; PARITY UNPINNED: librosa itself is not available).  Tolerance 2e-3 in log10 units on
    speech-like signals (float32 direct DFT of 400 samples), frame count and reflect padding at both ends, and the
    result feeds the extraction path."""
    from oracle import frontend as ofe
    r = np.random.RandomState(11)
    for n in (16000, 24123, 400, 3 * 160 + 7):
        t = np.arange(n) / 16000.0
        y = (0.2 * np.sin(2 * np.pi * 220.0 * t) + 0.1 * np.sin(2 * np.pi * 3150.0 * t + 0.3)
             + 0.05 * r.randn(n) * (0.2 + np.abs(np.sin(2 * np.pi * 1.5 * t)))).astype(np.float32)
        S = svb.log_mel_spectrogram(y)
        ref = ofe.log_mel(y.astype(np.float64))
        assert S.shape == ref.shape == (40, 1 + n // 160)
        err = np.abs(S.cpu().numpy().astype(np.float64) - ref).max()
        assert err < 2e-3, (n, err)
    silent = svb.log_mel_spectrogram(np.zeros(8000, dtype=np.float32))
    assert torch.all(silent == -6.0)                                         # log10(0 + 1e-6)
    with pytest.raises(ValueError):
        svb.log_mel_spectrogram(np.zeros(200, dtype=np.float32))
    S = svb.log_mel_spectrogram(0.1 * r.randn(24000).astype(np.float32))          # 151 frames -> 11 windows
    out = svb.extract_dvectors(net, [S.cpu().numpy()])
    assert out[0].shape[1] == 256 and out[0].shape[0] >= 1


def test_train_step_is_bitwise_reproducible(svb):
    """Persistent forward + BPTT (bulk-copy DSMEM exchange, software-pipelined reduce / gate loop) + weight gradients
    beside BPTT + per-speaker GE2E: every hand-off is ordered by barriers and counters and every sum has a fixed order,
    so repeated steps on the same batch agree bit for bit (a lost hand-off or a stale read would show here)."""
    torch.manual_seed(0)
    net = svb.SpeechEmbedder().cuda()
    crit = svb.GE2ELoss("cuda")
    for (N, M, T, reps) in ((64, 10, 160, 12), (13, 10, 41, 12), (3, 7, 90, 12)):
        x = torch.tensor(I.logmel(N * M, T, seed=5)).cuda()
        ref = None
        for _ in range(reps):
            net.zero_grad(set_to_none=True)
            crit.zero_grad(set_to_none=True)
            loss = crit(net(x).reshape(N, M, -1))
            loss.backward()
            g = torch.cat([p.grad.reshape(-1) for p in net.parameters()] + [crit.w.grad.reshape(1), loss.detach().reshape(1)])
            assert torch.isfinite(g).all()
            if ref is None:
                ref = g.clone()
            else:
                assert torch.equal(g, ref), (N, M, T)
