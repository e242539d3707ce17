"""SpeechEmbedder kernels at non-default model dimensions against the float64 oracle, route by route.

Every model is built with constructor arguments (never hparam.configure, which is global) at the rows of
tests/_embedder_shapes.py, each row chosen for the kernel routes of csrc/lstm.cu it takes.  The oracle is
oracle.embedder.embedder_explicit in float64 on the module's own parameters (pinned to torch.nn.LSTM at these shapes by
tests/test_oracle_embedder_shapes.py), computed once per (row, B, T).  Everything runs under a NaN-poisoned workspace,
so that a slot read before it is written shows up.

Bars are the suite's (test_gpu_parity.py): embeddings 1e-3 worst per-row L2-relative; parameter gradients 1.2e-2
(weights) and 3e-2 (biases) per-tensor L2-relative, for the loss (e * v).sum() with a fixed random v.
"""
import os
from contextlib import contextmanager

import numpy as np
import pytest
import torch

import _inputs as I
from _embedder_shapes import BY_ID, CASES, narrow_kz6, param_names, wgrad_overlap
from _launches import count_launches, launched
from oracle import embedder as oemb

pytestmark = pytest.mark.gpu

EMB_BAR = 1e-3
W_BAR, B_BAR = 1.2e-2, 3e-2
# Row I (nmels = 768) on the persistent forward alone: its layer-0 input projection is ONE fp16 x fp16 term (the
# per-frame path splits x and W_ih into hi/lo terms), and at K = 768 the pre-activations are about 4x larger than at
# nmels = 40.  Measured on a B200, worst embedding error at B x T = 1x1, 65x2, 129x3, 130x32: 3.36e-4, 8.62e-4,
# 1.05e-3, 1.40e-3; the float32 oracle with the kernel's operand rounding emulated (oracle.embedder.Emu: x, W_ih, h,
# W_hh in fp16) is off the float64 oracle by 3.35e-4, 8.61e-4, 1.06e-3, 1.41e-3.  The per-frame kernels on the same
# row stay below 1.2e-4.
EMB_BAR_PERSISTENT = {"I": 2e-3}


def emb_err(a, b):
    return float((np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)).max())


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.fixture(scope="module")
def svb():
    import pytorch_speaker_verification_b200 as m
    torch.set_num_threads(os.cpu_count())
    return m


@pytest.fixture(scope="module")
def models(svb):
    cache = {}

    def get(case):
        if case.id not in cache:
            torch.manual_seed(17 + case.nmels + case.hidden + case.num_layer + case.proj)
            cache[case.id] = svb.SpeechEmbedder(nmels=case.nmels, hidden=case.hidden, num_layer=case.num_layer,
                                                proj=case.proj).cuda()
        return cache[case.id]
    return get


def inputs(case, B, T):
    """(x float32 (B, T, nmels), v float32 (B, proj)), seeded by the shape."""
    x = I.logmel(B, T, seed=1000 * B + T + case.nmels, nmels=case.nmels)
    v = np.random.RandomState(B + 7 * T + case.proj).standard_normal((B, case.proj)).astype(np.float32)
    return torch.tensor(x), torch.tensor(v)


@pytest.fixture(scope="module")
def oracle(models):
    """-> (embeddings (B, P), {parameter: gradient of (e * v).sum()}), float64 numpy, once per (row, B, T)."""
    cache = {}

    def get(case, B, T):
        key = (case.id, B, T)
        if key not in cache:
            net = models(case)
            x, v = inputs(case, B, T)
            sd = {k: p.detach().cpu().double().clone().requires_grad_(True) for k, p in net.state_dict().items()}
            e = oemb.embedder_explicit(x.double(), sd, num_layer=case.num_layer, keep_f64=True)
            (e * v.double()).sum().backward()
            cache[key] = (e.detach().numpy(), {k: sd[k].grad.numpy() for k in param_names(case.num_layer)})
        return cache[key]
    return get


@contextmanager
def poisoned(persistent=True):
    from pytorch_speaker_verification_b200 import ops
    try:
        ops.set_poison_workspace(True)
        ops.set_persistent(persistent)
        ops.set_persistent_bwd(persistent)
        yield
    finally:
        ops.set_poison_workspace(False)
        ops.set_persistent(True)
        ops.set_persistent_bwd(True)


def run(net, x, v):
    """One forward + backward of (e * v).sum() -> (embeddings, {parameter: gradient}) as numpy."""
    net.zero_grad(set_to_none=True)
    e = net(x)
    (e * v).sum().backward()
    torch.cuda.synchronize()
    return e.detach().cpu().numpy(), {k: p.grad.detach().cpu().numpy() for k, p in net.named_parameters()}


def check_against_oracle(case, T, got, ref, what, emb_bar=EMB_BAR):
    """Asserts the bars; returns (embedding error, worst weight-gradient error, worst bias-gradient error)."""
    e, grads = got
    e_ref, g_ref = ref
    assert np.isfinite(e).all(), what
    err = emb_err(e, e_ref)
    assert err < emb_bar, (what, err)
    worst_w = worst_b = 0.0
    for k in param_names(case.num_layer):
        g = grads[k]
        assert g.shape == g_ref[k].shape, (what, k)
        assert np.isfinite(g).all(), (what, k)
        if T == 1 and "weight_hh" in k:
            assert not np.any(g_ref[k]), k                  # h_{-1} = 0: exactly no gradient
            assert not np.any(g), (what, k, float(np.abs(g).max()))
            continue
        r = rel_l2(g, g_ref[k])
        if "bias" in k:
            worst_b = max(worst_b, r)
            assert r < B_BAR, (what, k, r)
        else:
            worst_w = max(worst_w, r)
            assert r < W_BAR, (what, k, r)
    return err, worst_w, worst_b


def persistent_eligible(case):
    return case.fwd == "wlstm" or case.bwd == "wbptt"


PARITY = [(c, B, T) for c in CASES for (B, T) in c.shapes]


@pytest.mark.parametrize("case,B,T", PARITY, ids=[f"{c.id}-B{B}-T{T}" for c, B, T in PARITY])
def test_embedder_matches_float64_oracle(svb, models, oracle, case, B, T):
    """Forward and every parameter gradient against the oracle, with the persistent kernels on and, where the row
    takes them, off; the default route also twice, bit for bit."""
    net = models(case)
    x, v = inputs(case, B, T)
    xg, vg = x.cuda(), v.cuda()
    ref = oracle(case, B, T)
    for persistent in ((True, False) if persistent_eligible(case) else (True,)):
        with poisoned(persistent):
            got = run(net, xg, vg)
            bar = EMB_BAR_PERSISTENT.get(case.id, EMB_BAR) if persistent else EMB_BAR
            err, ew, eb = check_against_oracle(case, T, got, ref, (case.id, B, T, persistent), bar)
            if persistent:
                again = run(net, xg, vg)
                assert np.array_equal(again[0], got[0]), (case.id, B, T)
                for k in got[1]:
                    assert np.array_equal(again[1][k], got[1][k]), (case.id, B, T, k)
        print(f"\n[{case.id} I={case.nmels} H={case.hidden} L={case.num_layer} P={case.proj} B={B} T={T} "
              f"{'persistent' if persistent else 'per-frame'}] emb {err:.2e}  worst weight grad {ew:.2e}  "
              f"worst bias grad {eb:.2e}")


def assert_routes(case, B, T, names):
    H, L = case.hidden, case.num_layer
    fwd_frame = launched(names, "tc_gemm_kernel", "EpiLstmFwd")
    bwd_frame = launched(names, "tc_gemm_kernel", "EpiLstmBwd")
    if case.fwd == "wlstm":
        assert launched(names, f"wlstm_fwd_kernelILi{H}E") and not fwd_frame, (case.id, sorted(names))
    else:
        assert fwd_frame and not launched(names, "wlstm_fwd_kernel"), (case.id, sorted(names))
    if case.bwd == "wbptt":
        assert launched(names, "wbptt_kernelILi768E") and not bwd_frame, (case.id, sorted(names))
    else:
        assert bwd_frame and not launched(names, "wbptt_kernel"), (case.id, sorted(names))
    assert launched(names, "wait_frames_kernel") == wgrad_overlap(case, B, T), (case.id, sorted(names))
    assert launched(names, "sumz_kernel") == narrow_kz6(case, B, T), (case.id, sorted(names))
    # per-frame recurrence on CTA pairs (128 x 5 stages, TWO_CTA = true) once the batch exceeds 1024 rows
    assert launched(names, "tc_gemm_kernel", "EpiLstmFwdELi8ELi1ELb1E") == (case.fwd == "frame" and B > 1024), case.id
    # dX on 128-wide tiles (H % 256 != 0) in the per-frame backward of a stack
    dx128 = case.bwd == "frame" and L > 1 and H % 256 != 0
    assert launched(names, "tc_gemm_kernelILi128ELi4ELb0ELb0ENS_11EpiStoreF32ILi128EEELi8ELi1ELb0E") == dx128, case.id


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_kernel_routes(svb, models, case):
    """The kernels each row claims to cover are the ones that launch (CUPTI callback count of one forward+backward at
    the row's largest shape); per-frame rows launch no persistent kernel."""
    net = models(case)
    B, T = max(case.shapes, key=lambda s: s[0] * s[1])
    x, v = inputs(case, B, T)
    xg, vg = x.cuda(), v.cuda()
    run(net, xg, vg)                                  # weights packed, modules loaded outside the counted window
    names = count_launches(lambda: run(net, xg, vg))
    if names is None:
        pytest.skip("launch counter unavailable (no CUPTI, or another CUPTI client is attached)")
    assert launched(names, "prep_x_kernelIfE"), sorted(names)
    assert_routes(case, B, T, names)


@pytest.mark.parametrize("terms", [2, 3])
def test_split_recurrent_terms_meet_the_oracle(svb, models, oracle, terms):
    """recurrent_terms 2 and 3 (residual fp16 terms of W_hh) force the per-frame forward on a persistent-eligible row."""
    case = BY_ID["B"]
    net = models(case)
    try:
        net.recurrent_terms = terms
        for (B, T) in case.shapes:
            x, v = inputs(case, B, T)
            with poisoned():
                err, ew, eb = check_against_oracle(case, T, run(net, x.cuda(), v.cuda()), oracle(case, B, T),
                                                   (case.id, B, T, terms))
            print(f"\n[B terms={terms} B={B} T={T}] emb {err:.2e}  worst weight grad {ew:.2e}  worst bias grad {eb:.2e}")
        B, T = case.shapes[-1]
        x, v = inputs(case, B, T)
        names = count_launches(lambda: run(net, x.cuda(), v.cuda()))
        if names is not None:
            assert launched(names, "tc_gemm_kernel", "EpiLstmFwd") and not launched(names, "wlstm_fwd_kernel")
    finally:
        net.recurrent_terms = 1


def test_float64_cpu_input_meets_the_oracle(svb, models, oracle):
    """A float64 CPU input (odd nmels) is staged to the device, converted by prep_x_kernel<double>, and the
    embeddings come back on the CPU."""
    case = BY_ID["C"]
    net = models(case)
    for (B, T) in case.shapes:
        x, v = inputs(case, B, T)
        with poisoned():
            net.zero_grad(set_to_none=True)
            e = net(x.double())
            assert e.device.type == "cpu"
            (e * v).sum().backward()
            got = (e.detach().numpy(), {k: p.grad.detach().cpu().numpy() for k, p in net.named_parameters()})
            err, ew, eb = check_against_oracle(case, T, got, oracle(case, B, T), (case.id, B, T, "float64"))
        print(f"\n[C float64 B={B} T={T}] emb {err:.2e}  worst weight grad {ew:.2e}  worst bias grad {eb:.2e}")
    x, _ = inputs(case, 65, 2)
    with torch.no_grad():
        names = count_launches(lambda: net(x.double()))
    if names is not None:
        assert launched(names, "prep_x_kernelIdE") and not launched(names, "prep_x_kernelIfE"), sorted(names)


def test_chunked_tile_order_at_hidden_256(svb, models, oracle):
    """B = 1540 is 25 tiles of 64 rows, so the persistent forward walks them in chunks (wlstm.cuh WL_FOR_TILES): every
    row equals the row computed in a small batch, bit for bit, and the batch meets the oracle."""
    case = BY_ID["A"]
    net = models(case)
    B, T = 1540, 4
    x, _ = inputs(case, B, T)
    xg = x.cuda()
    with poisoned(), torch.no_grad():
        big = net(xg)
        assert torch.isfinite(big).all()
        for lo in (0, 1024, B - 70):
            assert torch.equal(net(xg[lo:lo + 70]), big[lo:lo + 70]), lo
    sd = {k: p.detach().cpu().double() for k, p in net.state_dict().items()}
    with torch.no_grad():
        e_ref = oemb.embedder_explicit(x.double(), sd, num_layer=case.num_layer, keep_f64=True).numpy()
    assert emb_err(big.cpu().numpy(), e_ref) < EMB_BAR


def test_unsupported_dimensions_are_rejected(svb):
    """Shapes the kernels do not take raise with the reason, before any kernel runs."""
    from pytorch_speaker_verification_b200 import _lib
    x = torch.tensor(I.logmel(4, 3, seed=1)).cuda()
    with pytest.raises(_lib.SvbError, match="multiple of 128"):
        svb.SpeechEmbedder(nmels=40, hidden=100, num_layer=1, proj=64).cuda()(x)
    with pytest.raises(_lib.SvbError, match="num_layer"):
        svb.SpeechEmbedder(nmels=40, hidden=128, num_layer=9, proj=64).cuda()(x)
    net = svb.SpeechEmbedder(nmels=13, hidden=128, num_layer=1, proj=64).cuda()
    with pytest.raises(ValueError, match="expected input"):
        net(x)
    torch.cuda.synchronize()
