"""Every GE2E kernel route of csrc/ge2e.cu (ge2e_impl) at ragged shapes against the float64 oracle.

ge2e_impl picks the route from the shape:
  speaker  one CTA (or 2-CTA cluster) per speaker: fused == 1, own centroids, M <= 16, D % 4 == 0, N <= 148 (#SMs)
  tc       phase kernels around three 3-term split-fp16 tcgen05 GEMMs (cos = E^ C^T, R = A_off C^, P = A_off^T E^):
           D % 64 == 0, D <= 256, Nc % 8 == 0, N M >= 512, Nc >= 128, N M Nc >= 2^18, no upstream dcos.  The cos
           GEMM runs on 128 x 256 tiles when Nc % 256 == 0; P is reduced over `psplit` slices of `prows` rows (a
           multiple of 64).  Above D = 256 the tensor cores' accumulation bias (about -7.7e-9 D on cosines near 1)
           would exceed the 3e-6 cosine bar, so wider D takes the SIMT kernels
  general  the cooperative kernel: fused != 0 otherwise
  phases   one launch per phase: fused == 0 otherwise
The row table below names, per row, the routes it takes and what about it is ragged; CUPTI launch names prove the
route.  Everything numeric runs with ops.set_poison_workspace(True): workspace and outputs start as NaN, so a slot or
output element that no kernel writes fails the comparison instead of holding an earlier call's value.

Bars are the suite's: loss, dE, dw 1e-5 max-relative and db 2e-3 against oracle.ge2e.ge2e_fwd_bwd in float64
(test_gpu_parity.py); the contrast loss as tests/test_gpu_ge2e_contrast.py; cosines 3e-6 absolute (test_eer_bit_exact);
the get_cossim backward 2e-5 max-relative (test_free_functions_match_reference_api).  Each test prints its worst errors
per (row, route).
"""
import ctypes
from collections import namedtuple
from contextlib import contextmanager

import numpy as np
import pytest
import torch

import _contrast_oracle as ocon
import _ge2e_oracle as G
import _inputs as I
from _contrast_inputs import top2_gap, twin_embeddings
from _launches import count_launches, launched
from oracle import ge2e as oge2e

pytestmark = pytest.mark.gpu

Row = namedtuple("Row", "N M D kind w b tc speaker why")
ROWS = [
    Row(152, 12, 64, "unit", 10.0, -5.0, True, False,
        "D = one K tile; Nc = 152: K of R ragged by 24; psplit 15, last slice 32 rows"),
    Row(136, 17, 128, "raw", 3.0, -1.0, True, False,
        "M > 16 at N <= 148; Nc = 136: K ragged by 8; psplit 13, last slice 8 rows"),
    Row(256, 4, 192, "clustered", 10.0, -5.0, True, False,
        "N M Nc = 2^18 exactly; 128 x 256 cos tiles; R / P outputs 1.5 tiles wide"),
    Row(200, 7, 192, "raw", 10.0, -5.0, True, False, "Nc = 200; psplit 11, last slice 120 rows"),
    Row(768, 2, 256, "unit", 3.0, -1.0, True, False,
        "M = 2; three 256-wide cos tiles; D = 256, the widest D on tensor cores"),
    Row(200, 7, 320, "raw", 10.0, -5.0, False, False,
        "D = 320, one K tile over the tensor-core cut, otherwise eligible: SIMT; psplit 11, last slice 120 rows"),
    Row(512, 10, 768, "clustered", 10.0, -5.0, False, False, "D = 768 (the C3 batch at wide D): SIMT, psplit 16"),
    # The per-speaker kernel's single-CTA form needs 162 KB of shared memory at (144, 16, 128) but 251 KB at
    # (144, 16, 256), over its 220 KB limit: there fused = 1 falls through to the other routes.
    Row(144, 16, 128, "raw", 3.0, -1.0, True, True,
        "per-speaker kernel in its single-CTA form (2N > 148) with fused = 1; the same batch on tensor cores"),
    Row(148, 16, 192, "unit", 10.0, -5.0, False, True,
        "per-speaker kernel at N = 148 (206 KB); Nc % 8 = 4: general kernel and phases, never tensor cores"),
    Row(248, 4, 256, "clustered", 3.0, -1.0, False, False, "N M Nc one step below 2^18: no tcgen05 launch"),
    Row(300, 10, 200, "raw", 10.0, -5.0, False, False,
        "D % 64 != 0: general kernel and phases at large N; psplit 16, last slice 120 rows"),
    Row(201, 7, 256, "unit", 3.0, -1.0, False, False, "Nc % 8 != 0: SIMT although N M Nc > 2^18"),
]
TC_ROWS = [r for r in ROWS if r.tc]


def row_id(r):
    return f"{r.N}x{r.M}x{r.D}"


def arms(r):
    """(tensor cores on, fused, route) of every distinct route of the row."""
    out = [(True, 1, "speaker")] if r.speaker else []
    if r.tc:
        out += [(True, 2, "tc")] + ([(True, 0, "tc")] if r.speaker else [])
    return out + [(False, 2, "general"), (False, 0, "phases")]


CUPTI_MISSING = "launch counter unavailable (no CUPTI, or another CUPTI client is attached): route not verified"


def gemm_launches(names):
    return sum(n for k, n in names.items() if "tc_gemm_kernel" in k)


def route_of(names):
    """The route one call's launches show ('speaker', 'tc', 'general', 'phases'; a tuple if they mix), for either loss
    method: the contrast kernels share the prefixes."""
    phase = launched(names, "ge2e_phase_")
    gemms = gemm_launches(names)
    kinds = (("speaker", launched(names, "ge2e_speaker_")), ("general", launched(names, "ge2e_fused_")),
             ("tc", phase and gemms > 0), ("phases", phase and not gemms))
    found = [n for n, hit in kinds if hit]
    return found[0] if len(found) == 1 else tuple(found)


def rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.fixture(scope="module")
def svb():
    import pytorch_speaker_verification_b200 as m
    return m


@pytest.fixture(scope="module")
def oracle():
    """(embeddings float32, float64 closed form) per (row, loss method), computed once."""
    cache = {}

    def get(r, method="softmax"):
        key = (r, method)
        if key not in cache:
            if method == "softmax":
                E = I.ge2e_embeddings(r.N, r.M, r.D, r.kind)
                o = oge2e.ge2e_fwd_bwd(E.astype(np.float64), r.w, r.b)
            else:
                E = twin_embeddings(r.N, r.M, r.D, raw=r.kind == "raw")
                assert top2_gap(E, r.w, r.b) > 1e-3                   # a clear nearest impostor in every row
                o = ocon.ge2e_fwd_bwd(E.astype(np.float64), r.w, r.b, "contrast")
                o["gabs"] = float(np.abs(o["G"]).sum())
            o.pop("cos")
            o.pop("G", None)
            cache[key] = (E, o)
        return cache[key]
    return get


@contextmanager
def route(tc):
    from pytorch_speaker_verification_b200 import ops
    try:
        ops.set_poison_workspace(True)
        ops.set_ge2e_tensor_cores(tc)
        yield
    finally:
        ops.set_poison_workspace(False)
        ops.set_ge2e_tensor_cores(True)


def step(svb, Enp, w, b, fused, method="softmax", grad=True):
    """GE2ELoss forward (+ backward) -> (loss, dE, dw, db) as numpy (gradients None without grad)."""
    E = torch.tensor(Enp, device="cuda", requires_grad=grad)
    crit = svb.GE2ELoss("cuda", loss_method=method)
    crit.fused = fused
    with torch.no_grad():
        crit.w.fill_(w)
        crit.b.fill_(b)
    if not grad:
        with torch.no_grad():
            loss = crit(E)
        torch.cuda.synchronize()
        return loss.item(), None, None, None
    loss = crit(E)
    loss.backward()
    torch.cuda.synchronize()
    return loss.item(), E.grad.cpu().numpy(), crit.w.grad.item(), crit.b.grad.item()


def check_softmax(o, got, what):
    loss, dE, dw, db = got
    err = dict(loss=rel(loss, o["loss"]), dE=rel(dE, o["dE"]), dw=rel(dw, o["dw"]), db=rel(db, o["db"]))
    assert np.isfinite(dE).all(), what
    assert err["loss"] < 1e-5 and err["dE"] < 1e-5 and err["dw"] < 1e-5, (what, err)
    assert err["db"] < 2e-3, (what, err)       # ill-conditioned (SURVEY 7.5)
    return err


def fmt(err):
    return "  ".join(f"{k} {v:.2e}" for k, v in err.items())


# ----------------------------------------------------------------------------------------------- softmax, every route
@pytest.mark.parametrize("r", ROWS, ids=row_id)
def test_loss_and_gradients_on_every_route(svb, oracle, r):
    Enp, o = oracle(r)
    for tc, fused, name in arms(r):
        with route(tc):
            err = check_softmax(o, step(svb, Enp, r.w, r.b, fused), (row_id(r), name, fused))
        print(f"\n[{row_id(r)} {r.kind} w={r.w} {name} fused={fused}] {fmt(err)}")


@pytest.mark.parametrize("r", ROWS, ids=row_id)
def test_routes_are_the_claimed_ones(svb, oracle, r):
    """CUPTI launch names of one forward + backward per arm: the row's claimed kernels, and no other route's."""
    Enp, _ = oracle(r)
    for tc, fused, name in arms(r):
        with route(tc):
            step(svb, Enp, r.w, r.b, fused)                       # modules loaded outside the counted window
            names = count_launches(lambda: step(svb, Enp, r.w, r.b, fused))
        if names is None:
            pytest.skip(CUPTI_MISSING)
        what = (row_id(r), name, fused, sorted(names))
        assert route_of(names) == name, what
        if name == "speaker":                                       # single-CTA form: 2N > 148
            assert launched(names, f"ge2e_speaker_kernelILi{(r.M + 1) & ~1}ELi1EE"), what
        if name == "tc":
            assert gemm_launches(names) == 3, what                   # cos, R, P
            assert launched(names, "tc_gemm_kernel", "EpiStoreF32ILi256E") == (r.N % 256 == 0), what


@pytest.mark.parametrize("r", TC_ROWS, ids=row_id)
def test_no_grad_forward_on_tensor_cores(svb, oracle, r):
    """Loss only: the cos GEMM runs, the R / P GEMMs do not."""
    Enp, o = oracle(r)
    fused = 2 if r.speaker else 1
    with route(True):
        loss = step(svb, Enp, r.w, r.b, fused, grad=False)[0]
        names = count_launches(lambda: step(svb, Enp, r.w, r.b, fused, grad=False))
    err = rel(loss, o["loss"])
    print(f"\n[{row_id(r)} tc no-grad] loss {err:.2e}")
    assert err < 1e-5, err
    if names is None:
        pytest.skip(CUPTI_MISSING)
    assert route_of(names) == "tc" and gemm_launches(names) == 1, sorted(names)


# the tensor-core rows, and the rows that the D cut sends to the SIMT kernels although tensor cores are on
CONTRAST_ROWS = [r for r in ROWS if r.tc or (r.D > 256 and r.D % 64 == 0)]


@pytest.mark.parametrize("tc", [True, False], ids=["tc_on", "tc_off"])
@pytest.mark.parametrize("r", CONTRAST_ROWS, ids=row_id)
def test_contrast_loss_on_tensor_cores(svb, oracle, r, tc):
    """Contrast loss (cos GEMM, contrast row phase, contrast phase D; or the general kernel) on twin batches, against
    the float64 contrast closed form at tests/test_gpu_ge2e_contrast.py's bars."""
    Enp, o = oracle(r, "contrast")
    fused = 2 if r.speaker else 1
    with route(tc):
        loss, dE, dw, db = step(svb, Enp, r.w, r.b, fused, "contrast")
        names = count_launches(lambda: step(svb, Enp, r.w, r.b, fused, "contrast"))
    name = "tc" if tc and r.tc else "general"
    err = dict(loss=rel(loss, o["loss"]), dE=rel(dE, o["dE"]), dw=rel(dw, o["dw"]),
               db_over_sum_abs_G=abs(db - o["db"]) / o["gabs"])
    print(f"\n[{row_id(r)} contrast {name}] {fmt(err)}")
    assert err["loss"] < 1e-5 and err["dE"] < 1e-5 and err["dw"] < 1e-5, err
    assert err["db_over_sum_abs_G"] <= 1e-5, err
    if names is None:
        pytest.skip(CUPTI_MISSING)
    assert route_of(names) == name, sorted(names)


# ----------------------------------------------------------------------------------------------- foreign centroids
def enrollment_verification(N, M, D, seed):
    return I.eer_embeddings(N, 2 * M, 0.06, 0.5, seed, D=D)


@pytest.mark.parametrize("N,M,D,tc_route", [(1024, 3, 256, "tc"), (136, 17, 128, "tc"), (200, 7, 320, "general"),
                                             (512, 3, 512, "general")])
def test_foreign_centroid_cosine(svb, N, M, D, tc_route):
    """get_cossim(verification, centroids(enrollment)) -- the EER similarity matrix (C5 at N = 1024) -- with tensor
    cores on (D > 256 takes the SIMT kernel there too) and off, against the float64 restatement of the kernel's own
    float32 centroids."""
    enr, ver = enrollment_verification(N, M, D, 4242 + N)
    C = svb.get_centroids(torch.tensor(enr, device="cuda"))
    ref = G.cossim(ver, C.cpu().numpy())
    Vg = torch.tensor(ver, device="cuda")
    routes = []
    for tc in (True, False):
        with route(tc), torch.no_grad():
            cos = svb.get_cossim(Vg, C)
            names = count_launches(lambda: svb.get_cossim(Vg, C))
        err = float(np.abs(cos.cpu().numpy() - ref).max())
        name = tc_route if tc else "general"
        print(f"\n[get_cossim {N}x{M}x{D} {name}] max abs {err:.2e}")
        assert err < 3e-6, (name, err)
        routes.append((name, names))
    for name, names in routes:
        if names is None:
            pytest.skip(CUPTI_MISSING)
        assert route_of(names) == name and gemm_launches(names) == (name == "tc"), sorted(names)


@pytest.mark.parametrize("N,M,D", [(64, 10, 256), (200, 7, 320), (300, 10, 200)])
def test_foreign_centroid_cosine_backward(svb, N, M, D):
    """(cos * V).sum().backward() through get_cossim (the dcos mode: SIMT only, P over psplit > 1 slices into dC)
    against the float64 dE and dC."""
    enr, ver = enrollment_verification(N, M, D, 99 + N)
    V = np.random.RandomState(N + D).standard_normal((N, M, N)).astype(np.float32)
    with torch.no_grad():
        C = svb.get_centroids(torch.tensor(enr, device="cuda")).cpu().numpy()
    _, dE_ref, dC_ref = G.cossim_grads(ver, C, V)
    with route(True):
        E = torch.tensor(ver, device="cuda", requires_grad=True)
        Ct = torch.tensor(C, device="cuda", requires_grad=True)
        (svb.get_cossim(E, Ct) * torch.tensor(V, device="cuda")).sum().backward()
        torch.cuda.synchronize()
    eE, eC = rel(E.grad.cpu().numpy(), dE_ref), rel(Ct.grad.cpu().numpy(), dC_ref)
    print(f"\n[get_cossim backward {N}x{M}x{D}] dE {eE:.2e}  dC {eC:.2e}")
    assert eE < 2e-5 and eC < 2e-5, (eE, eC)


# ----------------------------------------------------------------------------------------------- shared-memory envelope
ENVELOPE = [("softmax", 65), ("contrast", 64)]           # the largest M at D = 256: smem_bytes() <= 200 KB


@pytest.mark.parametrize("method,M", ENVELOPE)
def test_shared_memory_envelope(svb, method, M):
    """At D = 256 the last M inside the 200 KB phase-D envelope runs on every route and meets the oracle; one more
    utterance is refused with the library's error before any launch, and the next valid call is still right."""
    from pytorch_speaker_verification_b200 import _lib
    N, D = 128, 256
    if method == "softmax":
        Enp = I.ge2e_embeddings(N, M, D, "raw")
        o = oge2e.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0)
    else:
        Enp = twin_embeddings(N, M, D)
        o = ocon.ge2e_fwd_bwd(Enp.astype(np.float64), 10.0, -5.0, "contrast")
        o["gabs"] = float(np.abs(o["G"]).sum())

    unverified = []

    def run(tc, fused, name):
        with route(tc):
            loss, dE, dw, db = step(svb, Enp, 10.0, -5.0, fused, method)
            names = count_launches(lambda: step(svb, Enp, 10.0, -5.0, fused, method))
        if names is None:
            unverified.append(name)
        else:
            assert route_of(names) == name, (method, name, sorted(names))
        err = dict(loss=rel(loss, o["loss"]), dE=rel(dE, o["dE"]), dw=rel(dw, o["dw"]))
        assert max(err.values()) < 1e-5, (method, M, tc, fused, err)
        if method == "softmax":
            assert rel(db, o["db"]) < 2e-3
        else:
            assert abs(db - o["db"]) <= 1e-5 * o["gabs"]
        return err

    for tc, fused, name in ((True, 1, "tc"), (False, 1, "general"), (False, 0, "phases")):
        print(f"\n[envelope {method} {N}x{M}x{D} {name}] {fmt(run(tc, fused, name))}")
    big = torch.tensor(np.concatenate([Enp, Enp[:, :1]], axis=1), device="cuda", requires_grad=True)
    crit = svb.GE2ELoss("cuda", loss_method=method)
    for tc in (True, False):
        def refused():
            with route(tc), pytest.raises(_lib.SvbError, match="M\\*D too large for one CTA's shared memory"):
                crit(big)
        names = count_launches(refused)
        if names is None:
            refused()
            unverified.append("refusal")
        else:
            assert not names, sorted(names)
    run(True, 1, "tc")
    if unverified:
        pytest.skip(CUPTI_MISSING)


# ----------------------------------------------------------------------------------------------- determinism, capture
def test_tensor_core_route_is_deterministic_and_graph_capturable(svb):
    """(512, 10, 256) on tensor cores: three calls agree bit for bit, and the raw svb_ge2e C ABI captured in a CUDA
    graph on a side stream (after a warm-up, as bench.py times it) replays to the eager bits for new embeddings copied
    into the captured input."""
    from pytorch_speaker_verification_b200 import _lib
    N, M, D = 512, 10, 256
    Enp = I.ge2e_embeddings(N, M, D, "clustered")
    with route(True):
        runs = [step(svb, Enp, 10.0, -5.0, 1) for _ in range(3)]
        names = count_launches(lambda: step(svb, Enp, 10.0, -5.0, 1))
    if names is not None:
        assert route_of(names) == "tc" and gemm_launches(names) == 3, sorted(names)
    for r in runs[1:]:
        assert r[0] == runs[0][0] and np.array_equal(r[1], runs[0][1]) and (r[2], r[3]) == runs[0][2:]

    L = _lib.lib()
    nb = ctypes.c_size_t(0)
    _lib.check(L.svb_ge2e_workspace_bytes(N, M, D, N, ctypes.byref(nb)), "svb_ge2e_workspace_bytes")
    w = torch.tensor(10.0, device="cuda")
    b = torch.tensor(-5.0, device="cuda")

    def buffers():
        ws = torch.full((nb.value,), 255, dtype=torch.uint8, device="cuda")
        return ws, [torch.full(s, float("nan"), device="cuda") for s in ((), (N, M, D), (), ())]

    def call(E, ws, out):
        loss, dE, dw, db = out
        _lib.check(L.svb_ge2e(_lib.ptr(E), None, N, M, D, N, _lib.ptr(w), _lib.ptr(b), None, None, None, None,
                              _lib.ptr(loss), _lib.ptr(dE), None, _lib.ptr(dw), _lib.ptr(db), _lib.ptr(ws),
                              ctypes.c_size_t(nb.value), 1, _lib.stream_ptr()), "svb_ge2e")

    Eg = torch.tensor(Enp, device="cuda")
    ws, out = buffers()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call(Eg, ws, out)                                       # warm-up
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            call(Eg, ws, out)
    torch.cuda.current_stream().wait_stream(side)
    E2 = torch.tensor(I.ge2e_embeddings(N, M, D, "raw"), device="cuda")
    ws2, ref = buffers()
    raw = count_launches(lambda: call(E2, ws2, ref))
    if raw is None:
        call(E2, ws2, ref)
    else:
        assert route_of(raw) == "tc" and gemm_launches(raw) == 3, sorted(raw)
    Eg.copy_(E2)
    g.replay()
    torch.cuda.synchronize()
    for a, e in zip(out, ref):
        assert torch.isfinite(e).all() and torch.equal(a, e)
    o = oge2e.ge2e_fwd_bwd(E2.cpu().numpy().astype(np.float64), 10.0, -5.0)
    assert rel(ref[0].item(), o["loss"]) < 1e-5 and rel(ref[1].cpu().numpy(), o["dE"]) < 1e-5
    if names is None or raw is None:
        pytest.skip(CUPTI_MISSING)
