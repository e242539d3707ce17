"""GPU: the tensor-core GEMM entry points element by element.

svb_gemm_bf16 (tc_gemm_kernel<128, 4, ...>, all four operand layouts) and svb_gemm_bf16_2cta (the CTA-pair
instantiations <256, 6, ..., TWO_CTA>, both layouts) are the instantiations that the LSTM input projection, the weight
gradients, the GE2E tensor-core route and the AS-norm cohort GEMM launch; svb_gemm_persistent is csrc/pgemm.cu.

Most cases use integer operands in [-3, 3], exact in bf16 and fp16, and integer-valued bias.  Every partial sum is then
an integer of magnitude <= 3 terms * 9 * K + |bias| < 2^19 (K <= 12800), exact in the fp32 accumulator in any order,
so C must equal the float64 product exactly.  A dropped or repeated k-block, a wrong term, a wrong tail or a bias added
twice all change some element.  Every output buffer carries pad columns and extra rows filled with a NaN sentinel:
the kernel must write every element of [0, M) x [0, N) and nothing else.  Operand pad columns hold NaN too, so a tensor
map that reads past K or past the rows of an MN-major operand poisons C.

Rounding is measured separately, on random-normal operands against float64 (test_rounding_*)."""
import ctypes

import pytest
import torch

from pytorch_speaker_verification_b200 import _lib

pytestmark = pytest.mark.gpu
i64 = ctypes.c_int64
SENTINEL = 0x7FC0DEAD            # a quiet-NaN bit pattern no kernel computes

# (entry point, A MN-major, B MN-major)
LAYOUTS = [("bf16", 0, 0), ("bf16", 1, 1), ("bf16", 0, 1), ("bf16", 1, 0), ("2cta", 0, 0), ("2cta", 1, 1)]
LAYOUT_IDS = ["%s-%s%s" % (e, "M" if a else "K", "M" if b else "K") for e, a, b in LAYOUTS]


@pytest.fixture(scope="module")
def L():
    return _lib.lib()


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ints(shape, g, dtype=torch.bfloat16):
    return torch.randint(-3, 4, shape, device="cuda", generator=g).to(dtype)


def round8(n):
    return (n + 7) // 8 * 8


class Operand:
    """Logical [rows, K] operand in the layout a kernel reads: K-major storage [rows, ld >= K] or MN-major storage
    [K, ld >= rows].  Storage outside the logical matrix is NaN."""

    def __init__(self, rows, K, mn, g=None, pad=0, dtype=torch.bfloat16, values=None):
        self.ld = (round8(rows) if mn else round8(K)) + pad
        self.storage = torch.full((K, self.ld) if mn else (rows, self.ld), float("nan"), dtype=dtype, device="cuda")
        self.view = self.storage[:, :rows].t() if mn else self.storage[:, :K]
        self.view.copy_(ints((rows, K), g, dtype) if values is None else values)

    def ptr(self):
        return self.storage.data_ptr()


class Output:
    """C[M, N] at element offset `offset` of a sentinel-filled buffer with row pitch ldc and `extra` rows below."""

    def __init__(self, M, N, ldc, extra=3, offset=0):
        self.M, self.N, self.ldc, self.offset = M, N, ldc, offset
        self.buf = torch.full((offset + (M + extra) * ldc,), SENTINEL, dtype=torch.int32, device="cuda")

    def ptr(self):
        return self.buf.data_ptr() + 4 * self.offset

    def c(self):
        return self.buf.view(torch.float32)[self.offset:self.offset + self.M * self.ldc].view(self.M, self.ldc)[:, :self.N]

    def check(self, ref, what=""):
        """C == ref (float64) on every element; every other word of the buffer still holds the sentinel."""
        c = self.c()
        bits = c.view(torch.int32)
        assert not (bits == SENTINEL).any(), f"{what}: {int((bits == SENTINEL).sum())} elements of C never written"
        bad = c.double() != ref
        if bad.any():
            i, j = (int(v) for v in bad.nonzero()[0])
            raise AssertionError(f"{what}: {int(bad.sum())} of {c.numel()} elements differ, first C[{i},{j}] = "
                                 f"{float(c[i, j])} vs {float(ref[i, j])}")
        outside = torch.ones_like(self.buf, dtype=torch.bool)
        outside[self.offset:self.offset + self.M * self.ldc].view(self.M, self.ldc)[:, :self.N] = False
        touched = int((self.buf[outside] != SENTINEL).sum())
        assert touched == 0, f"{what}: {touched} words outside C[0:{self.M}, 0:{self.N}] (ldc {self.ldc}) were written"


def product(As, Bs, bias=None):
    ref = sum(a.double() @ b.double().t() for a, b in zip(As, Bs))
    return ref + bias.double() if bias is not None else ref


def call(L, entry, a_mn, b_mn, As, Bs, C_ptr, bias_ptr, M, N, K, lda, ldb, ldc, stream=None):
    n = len(As)
    PA = (ctypes.c_void_p * n)(*As)
    PB = (ctypes.c_void_p * n)(*Bs)
    st = stream_ptr() if stream is None else stream
    if entry == "bf16":
        return L.svb_gemm_bf16(PA, PB, n, ctypes.c_void_p(C_ptr), ctypes.c_void_p(bias_ptr), M, N, K, i64(lda), i64(ldb),
                               i64(ldc), a_mn, b_mn, st)
    assert a_mn == b_mn
    return L.svb_gemm_bf16_2cta(PA, PB, n, ctypes.c_void_p(C_ptr), ctypes.c_void_p(bias_ptr), M, N, K, i64(lda),
                                i64(ldb), i64(ldc), a_mn, st)


def run_case(L, layout, M, N, K, nterms, bias, seed, pad=0, store="tma"):
    """One exact integer GEMM through `layout`; store picks the output layout: "tma" (ldc % 4 == 0, aligned C and
    bias: the TMA epilogue whenever N % 4 == 0), or one that forces direct stores: "ldc_odd", "c_off4" (C 4 bytes past
    an aligned address), "bias_off4" (bias likewise)."""
    entry, a_mn, b_mn = layout
    g = torch.Generator(device="cuda").manual_seed(seed)
    As = [Operand(M, K, a_mn, g, pad) for _ in range(nterms)]
    Bs = [Operand(N, K, b_mn, g, pad) for _ in range(nterms)]
    bias_buf = torch.randint(-40, 41, (N + 4,), device="cuda", generator=g).float() if bias else None
    boff = 1 if store == "bias_off4" else 0
    bias_t = bias_buf[boff:boff + N] if bias else None
    ldc = (N + 1 if N % 2 == 0 else N + 2) if store == "ldc_odd" else (N + 3) // 4 * 4 + 4
    out = Output(M, N, ldc, offset=1 if store == "c_off4" else 0)
    rc = call(L, entry, a_mn, b_mn, [a.ptr() for a in As], [b.ptr() for b in Bs], out.ptr(),
              bias_t.data_ptr() if bias else 0, M, N, K, As[0].ld, Bs[0].ld, ldc)
    assert rc == 0, L.svb_last_error()
    torch.cuda.synchronize()
    out.check(product([a.view for a in As], [b.view for b in Bs], bias_t),
              f"{entry} a_mn={a_mn} b_mn={b_mn} M={M} N={N} K={K} terms={nterms} bias={bias} store={store}")


# ----------------------------------------------------------------------------------------------- a. ragged shapes
# M: tails of a 128-row tile and of a 256-row pair tile (1, 127, 300 and 640 leave the second tile of a CTA pair
# wholly out of bounds, 385 leaves it one row); N: residues 4, 8 and 0 of 32, 128 and 256, and 129 (N % 4 != 0: the
# direct-store epilogue); K: a tail inside one 64-wide k-block (8, 40, 200) and rings that wrap over 4 or 6 stages (768).
MS = (1, 127, 129, 255, 300, 385, 640)
NS = (4, 100, 128, 129, 264, 520)
KS = (8, 40, 64, 200, 768)


def grid():
    """Every value of every axis with every layout; the offsets by layout index vary the combinations."""
    for li, lay in enumerate(LAYOUTS):
        for i in range(len(MS)):
            yield pytest.param(lay, MS[i], NS[(i + li) % len(NS)], KS[(i + 2 * li) % len(KS)], 1 + (i + li) % 3,
                               (i + li) % 2 == 0, 8 * (i % 2), id=f"{LAYOUT_IDS[li]}-{i}")


@pytest.mark.parametrize("layout,M,N,K,nterms,bias,pad", list(grid()))
def test_exact_ragged(L, layout, M, N, K, nterms, bias, pad):
    run_case(L, layout, M, N, K, nterms, bias, seed=M * 7 + N * 3 + K, pad=pad)


# ----------------------------------------------------------------------------------------------- b. direct stores
@pytest.mark.parametrize("store", ["ldc_odd", "c_off4", "bias_off4"])
@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("M,N,K,nterms", [(300, 264, 200, 2), (129, 100, 40, 3)])
def test_exact_direct_store(L, layout, M, N, K, nterms, store):
    run_case(L, layout, M, N, K, nterms, True, seed=N + K, store=store)


# ----------------------------------------------------------------------------------------------- c. rounding
# max |C - ref| / (|A| |B|^T) elementwise, against float64.  A dropped 16-wide k-step leaves an error of order 16 / K
# of |A| |B|^T (above 4e-3 at K = 3600), so the bars must stay far below 1e-4.  Measured worst on one NVIDIA B200 at
# its 1,000 W power limit, identical on all six layouts: 5.4e-7 (K = 3600) and 2.9e-7 (K = 1000) for one term;
# 1.85e-6 for the three-term split against the fp32 product, where one term leaves 5.9e-4.  The bars are about 3x.
ROUND_BAR = 1.6e-6
SPLIT_BAR = 5.5e-6


def rounding_error(C, ref, absprod):
    return float(((C.double() - ref).abs() / absprod.clamp_min(1e-300)).max())


@pytest.mark.parametrize("layout", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("M,N,K", [(256, 256, 3600), (300, 264, 1000)])
def test_rounding_normal_operands(L, layout, M, N, K):
    entry, a_mn, b_mn = layout
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = Operand(M, K, a_mn, values=torch.randn(M, K, device="cuda", generator=g).bfloat16())
    B = Operand(N, K, b_mn, values=torch.randn(N, K, device="cuda", generator=g).bfloat16())
    C = torch.full((M, N), float("nan"), device="cuda")
    rc = call(L, entry, a_mn, b_mn, [A.ptr()], [B.ptr()], C.data_ptr(), 0, M, N, K, A.ld, B.ld, N)
    assert rc == 0, L.svb_last_error()
    err = rounding_error(C, product([A.view], [B.view]), A.view.double().abs() @ B.view.double().abs().t())
    print(f"rounding {entry} a_mn={a_mn} b_mn={b_mn} M={M} N={N} K={K}: {err:.3e}")
    assert err < ROUND_BAR


def split_bf16(x):
    hi = x.bfloat16()
    return hi, (x - hi.float()).bfloat16()


@pytest.mark.parametrize("layout", [LAYOUTS[0], LAYOUTS[4]], ids=[LAYOUT_IDS[0], LAYOUT_IDS[4]])
def test_rounding_split_terms(L, layout):
    """fp32 X and W as bf16 hi + lo, three terms hi.hi + hi.lo + lo.hi (the input projection's split): the error
    against the float64 product of the fp32 matrices must be far below that of the one-term hi.hi product."""
    entry, a_mn, b_mn = layout
    M, N, K = 640, 520, 768
    g = torch.Generator(device="cuda").manual_seed(11)
    X = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g)
    (xh, xl), (wh, wl) = split_bf16(X), split_bf16(W)
    As = [Operand(M, K, a_mn, values=v) for v in (xh, xh, xl)]
    Bs = [Operand(N, K, b_mn, values=v) for v in (wh, wl, wh)]
    ref = X.double() @ W.double().t()
    absprod = X.double().abs() @ W.double().abs().t()
    errs = []
    for n in (1, 3):
        C = torch.full((M, N), float("nan"), device="cuda")
        rc = call(L, entry, a_mn, b_mn, [a.ptr() for a in As[:n]], [b.ptr() for b in Bs[:n]], C.data_ptr(), 0, M, N, K,
                  As[0].ld, Bs[0].ld, N)
        assert rc == 0, L.svb_last_error()
        errs.append(rounding_error(C, ref, absprod))
    print(f"split {entry}: 1 term {errs[0]:.3e}, 3 terms {errs[1]:.3e}")
    assert errs[1] < SPLIT_BAR and errs[1] < errs[0] / 100


# ----------------------------------------------------------------------------------------------- d. production shapes
@pytest.mark.parametrize("layout,M,N,K,nterms,bias", [
    pytest.param(LAYOUTS[4], 12800, 3072, 768, 3, True, id="input-projection"),
    pytest.param(LAYOUTS[5], 3072, 768, 12800, 1, False, id="wgrad-hh"),
    pytest.param(LAYOUTS[5], 3072, 40, 12800, 1, False, id="wgrad-ih"),
    pytest.param(LAYOUTS[0], 5120, 512, 256, 1, False, id="ge2e-KK"),
    pytest.param(LAYOUTS[2], 5120, 512, 256, 1, False, id="ge2e-KM"),
    pytest.param(LAYOUTS[1], 5120, 512, 256, 1, False, id="ge2e-MM"),
])
def test_exact_production_shapes(L, layout, M, N, K, nterms, bias):
    run_case(L, layout, M, N, K, nterms, bias, seed=M + N + K)


# ----------------------------------------------------------------------------------------------- e. ordering
# Every launch carries programmatic dependent launch and the kernel triggers its dependents first thing, so a GEMM
# enqueued behind another may start while the first still runs; only griddepcontrol.wait orders its reads and writes.
def big_operands(mn, g):
    """2048 x 2048 x 768: 256 CTAs of svb_gemm_bf16, two waves on 148 SMs."""
    return Operand(2048, 768, mn, g), Operand(2048, 768, mn, g)


def big_gemm(L, entry, mn, ops, out, stream=None):
    A, B = ops
    rc = call(L, entry, mn, mn, [A.ptr()], [B.ptr()], out.ptr(), 0, 2048, 2048, 768, A.ld, B.ld, out.ldc, stream)
    assert rc == 0, L.svb_last_error()
    return product([A.view], [B.view])


@pytest.mark.parametrize("second", [LAYOUTS[0], LAYOUTS[5]], ids=[LAYOUT_IDS[0], LAYOUT_IDS[5]])
def test_reads_wait_for_previous_kernel(L, second):
    """GEMM 2's bias is the last row of GEMM 1's output, enqueued behind it on one stream with no synchronisation."""
    g = torch.Generator(device="cuda").manual_seed(5)
    s = torch.cuda.Stream()
    ops1 = big_operands(0, g)
    out1 = Output(2048, 2048, 2048, extra=0)
    entry, mn, _ = second
    M, N, K = 384, 1024, 64
    A, B = Operand(M, K, mn, g), Operand(N, K, mn, g)
    out2 = Output(M, N, N + 4)
    torch.cuda.synchronize()                     # inputs ready before the side stream starts
    st = ctypes.c_void_p(s.cuda_stream)
    ref1 = big_gemm(L, "bf16", 0, ops1, out1, st)
    row = 2047
    rc = call(L, entry, mn, mn, [A.ptr()], [B.ptr()], out2.ptr(), out1.ptr() + 4 * row * 2048, M, N, K, A.ld, B.ld,
              out2.ldc, st)
    assert rc == 0, L.svb_last_error()
    s.synchronize()
    out1.check(ref1, "GEMM 1")
    out2.check(product([A.view], [B.view], ref1[row, :N]), "GEMM 2 (bias = GEMM 1 row)")


@pytest.mark.parametrize("layout", [LAYOUTS[0], LAYOUTS[4]], ids=[LAYOUT_IDS[0], LAYOUT_IDS[4]])
def test_writes_wait_for_previous_kernel(L, layout):
    """Two calls into the same C back to back: the second one's values win everywhere."""
    g = torch.Generator(device="cuda").manual_seed(6)
    out = Output(2048, 2048, 2052)
    entry, mn, _ = layout
    ops1, ops2 = big_operands(mn, g), big_operands(mn, g)
    big_gemm(L, entry, mn, ops1, out)
    ref2 = big_gemm(L, entry, mn, ops2, out)
    torch.cuda.synchronize()
    out.check(ref2, "second call")


@pytest.mark.parametrize("layout", [LAYOUTS[3], LAYOUTS[5]], ids=[LAYOUT_IDS[3], LAYOUT_IDS[5]])
def test_graph_replay_matches_eager(L, layout):
    entry, a_mn, b_mn = layout
    M, N, K = 300, 264, 200
    g = torch.Generator(device="cuda").manual_seed(7)
    As = [Operand(M, K, a_mn, g) for _ in range(2)]
    Bs = [Operand(N, K, b_mn, g) for _ in range(2)]
    bias = torch.randint(-9, 10, (N,), device="cuda", generator=g).float()
    out_g, out_e = Output(M, N, N + 4), Output(M, N, N + 4)
    args = ([a.ptr() for a in As], [b.ptr() for b in Bs])

    def run(out):
        rc = call(L, entry, a_mn, b_mn, *args, out.ptr(), bias.data_ptr(), M, N, K, As[0].ld, Bs[0].ld, out.ldc)
        assert rc == 0, L.svb_last_error()

    run(out_e)                                   # configures the kernel outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run(out_g)
    for op in As + Bs:                           # new operand data in the captured buffers
        op.view.copy_(ints(tuple(op.view.shape), g))
    bias.copy_(torch.randint(-9, 10, (N,), device="cuda", generator=g).float())
    graph.replay()
    run(out_e)
    torch.cuda.synchronize()
    ref = product([a.view for a in As], [b.view for b in Bs], bias)
    out_g.check(ref, "graph replay")
    assert torch.equal(out_g.buf, out_e.buf)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs a second GPU")
def test_second_device(L):
    """The kernels' shared-memory attribute is set per device: the first call on cuda:1 comes after calls on cuda:0."""
    run_case(L, LAYOUTS[0], 300, 264, 200, 2, True, seed=1)
    run_case(L, LAYOUTS[5], 300, 264, 200, 2, True, seed=1)
    pg_case(L, 300, 512, 192, 0, True, 0)
    with torch.cuda.device(1):
        run_case(L, LAYOUTS[0], 300, 264, 200, 2, True, seed=2)
        run_case(L, LAYOUTS[5], 300, 264, 200, 2, True, seed=2)
        pg_case(L, 300, 512, 192, 0, True, 0)


# ----------------------------------------------------------------------------------------------- f. persistent kernel
@pytest.mark.parametrize("M,N,K,f16,bias", [(256, 256, 64, 0, False), (1000, 512, 192, 1, True), (70, 256, 128, 1, False),
                                            (5000, 3072, 768, 0, True)])
def test_persistent_input_gemm(L, M, N, K, f16, bias):
    """svb_gemm_persistent (csrc/pgemm.cu: the LSTM input projection W_ih x_t as one batched GEMM) against fp32 matmul
    on the same bf16 / fp16-rounded operands: ragged M (rows clipped by TMA), bias, several tiles per CTA pair."""
    from pytorch_speaker_verification_b200._lib import ptr
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    dt = torch.float16 if f16 else torch.bfloat16
    A = torch.randn(M, K, device="cuda", generator=g).to(dt)
    B = (torch.randn(N, K, device="cuda", generator=g) * 0.05).to(dt)
    bs = torch.randn(N, device="cuda", generator=g) if bias else None
    C = torch.full((M, N), float("nan"), device="cuda")
    r = L.svb_gemm_persistent(ptr(A), ptr(B), ptr(C), ptr(bs), M, N, K, i64(K), i64(K), i64(N), f16, stream_ptr())
    assert r == 0
    ref = A.float() @ B.float().t() + (bs if bias else 0.0)
    assert not torch.isnan(C).any()
    assert float((C - ref).abs().max() / ref.abs().max()) < 2e-5
    assert L.svb_gemm_persistent(ptr(A), ptr(B), ptr(C), None, M, 100, K, i64(K), i64(K), i64(N), f16, None) != 0


def pg_case(L, M, N, K, f16, bias, pad):
    dt = torch.float16 if f16 else torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(M + N + K + f16)
    A, B = Operand(M, K, 0, g, pad, dt), Operand(N, K, 0, g, 2 * pad, dt)
    bias_t = torch.randint(-40, 41, (N,), device="cuda", generator=g).float() if bias else None
    out = Output(M, N, N + pad // 2)
    rc = L.svb_gemm_persistent(ctypes.c_void_p(A.ptr()), ctypes.c_void_p(B.ptr()), ctypes.c_void_p(out.ptr()),
                               ctypes.c_void_p(bias_t.data_ptr() if bias else 0), M, N, K, i64(A.ld), i64(B.ld),
                               i64(out.ldc), f16, stream_ptr())
    assert rc == 0, L.svb_last_error()
    torch.cuda.synchronize()
    out.check(product([A.view], [B.view], bias_t), f"persistent M={M} N={N} K={K} f16={f16} bias={bias} pad={pad}")


def pg_grid():
    """M: one row, tails of 128 and 256, and 8192 x 3072 (384 tiles on 74 pairs: more than 5 per pair, so both TMEM
    accumulators wrap their phase twice; at K = 320 the 5-stage ring ends each tile exactly on its boundary)."""
    ms, ns, ks = (1, 70, 128, 255, 257, 1000), (256, 512, 3072), (64, 192, 320, 768)
    for f16 in (0, 1):
        for i, M in enumerate(ms):
            yield pytest.param(M, ns[(i + f16) % 3], ks[(i + f16) % 4], f16, (i + f16) % 2 == 0, 8 * (i % 2),
                               id=f"f16={f16}-{i}")
        yield pytest.param(8192, 3072, 320, f16, f16 == 0, 8 * f16, id=f"f16={f16}-phase-wrap")


@pytest.mark.parametrize("M,N,K,f16,bias,pad", list(pg_grid()))
def test_persistent_exact(L, M, N, K, f16, bias, pad):
    pg_case(L, M, N, K, f16, bias, pad)
