"""GPU: the GE2E contrast loss (Wan et al. eq. 7, GE2ELoss(device, loss_method="contrast")) on every GE2E kernel path
against the float64 oracle (tests/_contrast_oracle.py, ge2e_fwd_bwd(..., "contrast")).

Tolerances as for the softmax loss (DESIGN.md section 2): loss, dE, dw 1e-5 relative; db within 1e-5 * sum |G|.
The contrast gradient jumps where two off-diagonal similarities tie, so every dE comparison runs on twin-structured
batches (tests/_contrast_inputs.py) whose top-two off-diagonal gap is asserted to exceed 1e-3 in S.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import _inputs as I
import _contrast_oracle as ocon
from _contrast_inputs import top2_gap, twin_embeddings, twin_logmel
from oracle import embedder as oemb
from oracle import ge2e as oge2e

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
SPEAKER_SHAPES = [(3, 2, 4), (33, 7, 20), (20, 5, 24), (64, 10, 256), (70, 10, 256), (100, 16, 256), (120, 13, 64),
                  (37, 9, 512), (74, 2, 8)]


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def oracle(Enp, w, b):
    """fp64 contrast closed form + sum |G| (the scale of db's tolerance)."""
    E = np.asarray(Enp, dtype=np.float64)
    o = ocon.ge2e_fwd_bwd(E, w, b, "contrast")
    o["gabs"] = float(np.abs(o["G"]).sum())
    return o


def twins(N, M, D, w=10.0, b=-5.0, **kw):
    E = twin_embeddings(N, M, D, **kw)
    if N >= 2:
        assert top2_gap(E, w, b) > 1e-3
    return E


def check(o, loss, dE, dw, db, tol=1e-5, scale=1.0):
    assert rel(loss, o["loss"]) < tol, (loss, o["loss"])
    assert rel(dE, scale * o["dE"]) < tol
    assert rel(dw, scale * o["dw"]) < tol
    assert abs(db - scale * o["db"]) <= tol * abs(scale) * o["gabs"], (db, o["db"])


@pytest.fixture(scope="module")
def svb():
    import pytorch_speaker_verification_b200 as m
    return m


def direct(Enp, w, b, fused):
    """svb_ge2e_ex through the op layer: dict(loss, per, dE, dw, db) as numpy."""
    from pytorch_speaker_verification_b200 import ops
    E = torch.tensor(Enp, device="cuda")
    wt, bt = torch.tensor(w, device="cuda"), torch.tensor(b, device="cuda")
    r = ops._ge2e_call(E, None, wt, bt, None, None, False, True, True, fused, 1)
    return {k: r[k].cpu().numpy() for k in ("loss", "per", "dE", "dw", "db")}


def module_step(svb, Enp, w, b, fused=1, scale=None):
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    crit = svb.GE2ELoss("cuda", loss_method="contrast")
    crit.fused = fused
    with torch.no_grad():
        crit.w.fill_(w)
        crit.b.fill_(b)
    loss = crit(E)
    (loss if scale is None else loss * scale).backward()
    return loss.item(), E.grad.cpu().numpy(), crit.w.grad.item(), crit.b.grad.item()


# ----------------------------------------------------------------------------------------------- kernel paths
@pytest.mark.parametrize("fused", [1, 2, 0])   # 1: per-speaker kernel, 2: general fused kernel, 0: one launch per phase
@pytest.mark.parametrize("name", list(I.GE2E_CASES))
def test_contrast_every_fused_mode(svb, name, fused):
    N, M, D, kind, w, b = I.GE2E_CASES[name]
    Enp = twins(N, M, D, w, b, raw=kind == "raw")
    o = oracle(Enp, w, b)
    r = direct(Enp, w, b, fused)
    check(o, r["loss"], r["dE"], r["dw"], r["db"])
    assert rel(r["per"], o["per"]) < 1e-5
    check(o, *module_step(svb, Enp, w, b, fused))


def test_contrast_loss_on_random_inputs(svb):
    """Loss and dw are continuous in the embeddings: plain random batches need no margin."""
    for name in ("c1", "clustered", "c2"):
        N, M, D, kind, w, b = I.GE2E_CASES[name]
        Enp = I.ge2e_embeddings(N, M, D, kind)
        o = oracle(Enp, w, b)
        for fused in (1, 2):
            r = direct(Enp, w, b, fused)
            assert rel(r["loss"], o["loss"]) < 1e-5 and rel(r["dw"], o["dw"]) < 1e-5


@pytest.mark.parametrize("shape", SPEAKER_SHAPES)
def test_contrast_speaker_kernel_matches_general_kernel(svb, shape):
    """Per-speaker kernel (2-CTA clusters where D % 8 == 0 and 2N <= #SMs, single CTAs otherwise) and general kernel,
    each against the oracle and against each other, on the padding shapes of the softmax test."""
    N, M, D = shape
    Enp = twins(N, M, D)
    o = oracle(Enp, 10.0, -5.0)
    res = [module_step(svb, Enp, 10.0, -5.0, fused) for fused in (1, 2)]
    for r in res:
        check(o, *r)
    assert rel(res[0][0], res[1][0]) < 1e-6 and rel(res[0][1], res[1][1]) < 1e-5
    with torch.no_grad():                                   # forward-only mode of the speaker kernel
        crit = svb.GE2ELoss("cuda", "contrast")
        assert rel(crit(torch.tensor(Enp, device="cuda")).item(), o["loss"]) < 1e-5


@pytest.mark.parametrize("shape", [(320, 7, 256), (512, 10, 256)])
def test_contrast_tensor_core_route(svb, shape):
    """rows x centroids >= 2^18: split-fp16 cos GEMM, contrast row phase, contrast phase D (no R / P products)."""
    from pytorch_speaker_verification_b200 import ops
    N, M, D = shape
    Enp = twins(N, M, D)
    o = oracle(Enp, 10.0, -5.0)
    out = {}
    try:
        for tc in (True, False):
            ops.set_ge2e_tensor_cores(tc)
            out[tc] = module_step(svb, Enp, 10.0, -5.0)
            check(o, *out[tc])
    finally:
        ops.set_ge2e_tensor_cores(True)
    assert rel(out[True][0], out[False][0]) < 1e-5 and rel(out[True][1], out[False][1]) < 1e-5


@pytest.mark.parametrize("N,M,D,shards", [(8, 4, 32, 2), (64, 10, 256, 8), (512, 10, 256, 8), (12, 3, 20, 3)])
def test_contrast_row_shards_sum_to_the_global_batch(svb, N, M, D, shards):
    """svb_ge2e_rows_ex with the contrast loss: the shards' losses / dw / db / centroid gradients sum to the global
    batch's, and dE_rows + dC_total[own speaker] / M is the global dL/dE."""
    Enp = twins(N, M, D)
    o = oracle(Enp, 10.0, -5.0)
    E = torch.tensor(Enp, device="cuda")
    w, b = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")
    C = svb.get_centroids(E)
    nl = N // shards
    reds, dEs = [], []
    for r in range(shards):
        red, dE = torch.ops.svb200.ge2e_rows(E[r * nl:(r + 1) * nl].contiguous(), C, w, b, r * nl, 1)
        reds.append(red.double())
        dEs.append(dE)
    red = torch.stack(reds).sum(dim=0)
    dC = red[:N * D].view(N, D).float()
    dE = torch.cat(dEs) + torch.ops.svb200.centroids_bwd(dC.contiguous(), M)
    check(o, red[N * D].item(), dE.cpu().numpy(), red[N * D + 1].item(), red[N * D + 2].item())


# ----------------------------------------------------------------------------------------------- public API
def test_contrast_composes_from_the_free_functions(svb):
    """get_cossim -> w cos + b -> calc_loss(S, "contrast") under autograd equals the fused GE2ELoss("cuda", "contrast");
    CPU tensors go in and come back on the CPU."""
    Enp = twins(4, 5, 256)
    o = oracle(Enp, 10.0, -5.0)
    Et = torch.tensor(Enp, requires_grad=True)
    w = torch.tensor(10.0, requires_grad=True)
    b = torch.tensor(-5.0, requires_grad=True)
    S = w * svb.get_cossim(Et, svb.get_centroids(Et)) + b
    loss, per = svb.calc_loss(S, "contrast")
    assert loss.device.type == "cpu" and per.device.type == "cpu"
    loss.backward()
    assert Et.grad.device.type == "cpu"
    fused = module_step(svb, Enp, 10.0, -5.0)
    assert rel(loss.item(), fused[0]) < 1e-6
    assert rel(Et.grad.numpy(), fused[1]) < 2e-5
    assert rel(w.grad.item(), fused[2]) < 2e-5
    assert rel(per.numpy(), o["per"]) < 1e-5
    check(o, loss.item(), Et.grad.numpy(), w.grad.item(), b.grad.item(), tol=2e-5)
    # the utils module's signature (the reference's name) and the softmax default are unchanged
    l_soft, _ = svb.utils.calc_loss(S.detach())
    assert rel(l_soft.item(), oge2e.calc_loss(S.detach().double().numpy())[0]) < 1e-5


def test_contrast_edge_cases(svb):
    Enp = twins(4, 5, 256)
    o = oracle(Enp, 10.0, -5.0)
    loss, dE, dw, db = module_step(svb, Enp, 10.0, -5.0, scale=0.25)     # upstream gradient 0.25
    assert rel(loss, o["loss"]) < 1e-5
    check(o, o["loss"], dE, dw, db, scale=0.25)
    crit = svb.GE2ELoss("cuda", "contrast")
    assert crit.loss_method == "contrast" and set(crit.state_dict()) == {"w", "b"}
    E = torch.tensor(Enp, device="cuda", requires_grad=True)
    with torch.no_grad():
        l2 = crit(E)
    assert rel(l2.item(), o["loss"]) < 1e-5 and not l2.requires_grad
    # w = 100, b = 20: sigmoid saturates; finite and within 1e-4 of float64
    Eb = twins(16, 6, 256, 100.0, 20.0)
    ob = oracle(Eb, 100.0, 20.0)
    r = module_step(svb, Eb, 100.0, 20.0)
    assert all(np.isfinite(np.asarray(v)).all() for v in r)
    assert rel(r[0], ob["loss"]) < 1e-4 and rel(r[1], ob["dE"]) < 1e-4
    with pytest.raises(ValueError):
        crit(torch.randn(1, 4, 8, device="cuda"))          # N = 1: no other centroid
    with pytest.raises(ValueError):
        svb.calc_loss(torch.randn(1, 4, 1, device="cuda"), "contrast")
    with pytest.raises(ValueError):
        svb.GE2ELoss("cuda", loss_method="angular")
    with pytest.raises(ValueError):
        svb.calc_loss(torch.randn(3, 2, 3, device="cuda"), "angular")
    with pytest.raises(ValueError):
        crit(torch.randn(3, 1, 8, device="cuda"))          # M = 1


def _toy(D):
    """tests/golden/toy.npz zero-padded to D dimensions (the cosines, and their exact ties, are unchanged)."""
    E = np.load(os.path.join(G, "toy.npz"))["E"]
    return np.ascontiguousarray(np.pad(E, ((0, 0), (0, 0), (0, D - E.shape[2])))).astype(np.float32)


def test_contrast_exact_ties_take_the_lowest_index(svb):
    """Rows (0, 1) and (2, *) of the toy batch tie exactly between two off-diagonal columns: every path sends the
    gradient to the lower index, as the oracle (and torch.max) does."""
    ks = ocon.contrast_kstar(oge2e.get_cossim(_toy(3).astype(np.float64), oge2e.get_centroids(_toy(3).astype(np.float64))))
    np.testing.assert_array_equal(ks, [[1, 1], [0, 0], [0, 0]])
    for D, fused in ((3, 2), (3, 0), (4, 1), (8, 1)):          # general, per-phase, speaker kernel (1-CTA, 2-CTA)
        Enp = _toy(D)
        o = oracle(Enp, 10.0, -5.0)
        check(o, *module_step(svb, Enp, 10.0, -5.0, fused))
    Enp = _toy(3)
    o = oracle(Enp, 10.0, -5.0)
    E = torch.tensor(Enp, device="cuda")
    C = svb.get_centroids(E)
    w, b = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")
    parts = [torch.ops.svb200.ge2e_rows(E[r:r + 1].contiguous(), C, w, b, r, 1) for r in range(3)]
    red = sum(p[0].double() for p in parts)
    dE = torch.cat([p[1] for p in parts]) + torch.ops.svb200.centroids_bwd(red[:9].view(3, 3).float().contiguous(), 2)
    check(o, red[9].item(), dE.cpu().numpy(), red[10].item(), red[11].item())
    S = (10.0 * oge2e.get_cossim(Enp.astype(np.float64), oge2e.get_centroids(Enp.astype(np.float64))) - 5.0)
    St = torch.tensor(S, dtype=torch.float32, device="cuda", requires_grad=True)
    loss, _ = svb.calc_loss(St, "contrast")
    loss.backward()
    np.testing.assert_allclose(St.grad.cpu().numpy(), ocon.contrast_grad(S), rtol=1e-5, atol=1e-7)


def test_contrast_is_deterministic(svb):
    """Two calls give bit-identical loss, dE, dw, db on every path."""
    from pytorch_speaker_verification_b200 import ops
    cases = [((64, 10, 256), 1), ((33, 7, 20), 1), ((64, 10, 256), 2), ((64, 10, 256), 0), ((512, 10, 256), 1)]
    for (N, M, D), fused in cases:
        Enp = twins(N, M, D)
        a, c = direct(Enp, 10.0, -5.0, fused), direct(Enp, 10.0, -5.0, fused)
        for k in a:
            assert np.array_equal(a[k], c[k]), (N, M, D, fused, k)
    E = torch.tensor(twins(512, 10, 256), device="cuda")
    C = svb.get_centroids(E)
    w, b = torch.tensor(10.0, device="cuda"), torch.tensor(-5.0, device="cuda")
    r1 = torch.ops.svb200.ge2e_rows(E[:64].contiguous(), C, w, b, 0, 1)
    r2 = torch.ops.svb200.ge2e_rows(E[:64].contiguous(), C, w, b, 0, 1)
    assert torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])
    S = (10.0 * svb.get_cossim(E, C) - 5.0).detach()
    g = torch.tensor(1.0, device="cuda")
    assert torch.equal(ops._calc_loss_bwd(S, g, 1), ops._calc_loss_bwd(S, g, 1))
    assert torch.equal(ops._calc_loss(S, 1)[0], ops._calc_loss(S, 1)[0])


def test_contrast_opcheck(svb):
    E = torch.tensor(twins(6, 4, 32), device="cuda")
    C = torch.ops.svb200.centroids(E)
    Er = E.clone().requires_grad_(True)
    w = torch.tensor(10.0, device="cuda", requires_grad=True)
    b = torch.tensor(-5.0, device="cuda", requires_grad=True)
    chk = torch.library.opcheck
    chk(torch.ops.svb200.ge2e_loss.default, (Er, w, b, 1, True, 1))
    chk(torch.ops.svb200.ge2e_rows.default, (E[:3].contiguous(), C, w.detach(), b.detach(), 0, 1))
    S = (10.0 * torch.ops.svb200.cossim(E, C) - 5.0).detach().requires_grad_(True)
    chk(torch.ops.svb200.calc_loss.default, (S, 1))
    chk(torch.ops.svb200.calc_loss_bwd.default, (S.detach(), torch.tensor(1.0, device="cuda"), 1))


# ----------------------------------------------------------------------------------------------- training step
def test_contrast_train_step_gradients(svb):
    """C1 step through SpeechEmbedder + GE2ELoss("cuda", "contrast").  The oracle takes the GPU's own embeddings (so
    that embedding error cannot flip a k*); every parameter gradient is checked against the reference's library
    embedder back-propagating the same dL/dE (DESIGN.md section 2 tolerances).  The untrained embedder maps random
    log-mels to nearly parallel embeddings (top-two gaps of 1e-5 in S), so the input has the twin structure."""
    torch.manual_seed(0)
    net = svb.SpeechEmbedder().cuda()
    x = torch.tensor(twin_logmel(4, 5, 180, seed=1))
    crit = svb.GE2ELoss("cuda", "contrast")
    emb = net(x.cuda())
    E = emb.reshape(4, 5, -1)
    E.retain_grad()
    loss = crit(E)
    loss.backward()
    Enp = E.detach().cpu().numpy()
    assert top2_gap(Enp, 10.0, -5.0) > 1e-3
    o = oracle(Enp, 10.0, -5.0)
    assert rel(loss.item(), o["loss"]) < 1e-5
    assert rel(E.grad.cpu().numpy(), o["dE"]) < 1e-5
    assert rel(crit.w.grad.item(), o["dw"]) < 1e-5
    torch.manual_seed(0)
    ref = oemb.LibraryEmbedder()
    assert all(torch.equal(a, b.cpu()) for a, b in zip(ref.state_dict().values(), net.state_dict().values()))
    ref(x).backward(torch.tensor(o["dE"].reshape(20, -1), dtype=torch.float32))
    refp = dict(ref.named_parameters())
    for k, p in net.named_parameters():
        e = rel_l2(p.grad.cpu().numpy(), refp[k].grad.numpy())
        assert e < (3e-2 if "bias" in k else 1.2e-2), (k, e)


# ----------------------------------------------------------------------------------------------- two GPUs
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, Enp, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import pytorch_speaker_verification_b200 as svb
    from pytorch_speaker_verification_b200.dist import GlobalGE2ELoss, speaker_shard
    N = Enp.shape[0]
    lo, hi = speaker_shard(N, rank, world)
    res = {}
    for mode in ("rows", "gather", "peer"):
        crit = svb.GE2ELoss("cuda", loss_method="contrast")
        E = torch.tensor(Enp[lo:hi], device="cuda", requires_grad=True)
        glob = GlobalGE2ELoss(crit, mode=mode)
        loss = glob(E)
        loss.backward()
        if mode == "peer":
            assert glob._px not in (None, False), "peer memory was not used"
        res[mode] = (loss.item(), E.grad.cpu(), crit.w.grad.item(), crit.b.grad.item())
    out[rank] = res
    dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_contrast_two_rank_step_equals_single_gpu(svb):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    Enp = twins(8, 4, 256)
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), Enp, out), nprocs=2, join=True)
    loss, dE, dw, db = module_step(svb, Enp, 10.0, -5.0)
    o = oracle(Enp, 10.0, -5.0)
    for rank in range(2):
        for mode, (l, g, gw, gb) in out[rank].items():
            assert abs(l - loss) < 1e-5 * abs(loss), (rank, mode)
            assert np.abs(g.numpy() - dE[4 * rank:4 * rank + 4]).max() < 1e-5 * np.abs(dE).max(), (rank, mode)
            assert abs(gw - dw) < 1e-4 * abs(dw), (rank, mode)
            assert abs(gb - o["db"]) <= 1e-5 * o["gabs"]
