"""CPU: the GEMM entry points (svb_gemm_bf16, svb_gemm_bf16_2cta, svb_gemm_persistent) reject bad arguments in host
code, before any CUDA call, with SVB_ERR_ARG / SVB_ERR_ALIGN and a message that names the function.

The pointers are fake device addresses: a rejected call must never reach the driver, let alone a device.  The file
skips where a CUDA device exists, so that a check that is missing can never launch a kernel with these arguments."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="GPU present: these calls must never reach a device")

ARG, ALIGN = -1, -4
i64 = ctypes.c_int64
P = 0x7F0000000000          # 16-byte aligned fake device addresses, never dereferenced
A0, A1, A2, B0, B1, B2, C, BIAS = (ctypes.c_void_p(P + 0x1000000 * i) for i in range(8))


@pytest.fixture(scope="module")
def L():
    import os
    from pytorch_speaker_verification_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def ptrs(*p):
    return (ctypes.c_void_p * max(len(p), 1))(*p)


# A valid call (M=300, N=264, K=200, two terms, K-major, ldc = N) and (id, overrides of it, expected code)
GOOD = dict(A=ptrs(A0, A1), B=ptrs(B0, B1), nterms=2, C=C, bias=BIAS, M=300, N=264, K=200, lda=200, ldb=200, ldc=264,
            mn=0)
REJECT = [
    ("M0", dict(M=0), ARG), ("Mneg", dict(M=-5), ARG),
    ("N0", dict(N=0), ARG), ("Nneg", dict(N=-1), ARG),
    ("K0", dict(K=0), ARG), ("Kneg", dict(K=-64), ARG),
    ("nterms0", dict(nterms=0), ARG), ("nterms4", dict(A=ptrs(A0, A1, A2, A0), B=ptrs(B0, B1, B2, B0), nterms=4), ARG),
    ("A_array_null", dict(A=None), ARG), ("B_array_null", dict(B=None), ARG),
    ("A1_null", dict(A=ptrs(A0, None)), ARG), ("B0_null", dict(B=ptrs(None, B1)), ARG),
    ("C_null", dict(C=None), ARG),
    ("lda_lt_K", dict(lda=192), ARG), ("ldb_lt_K", dict(ldb=192), ARG),
    ("ldc_lt_N", dict(ldc=260), ARG),
    ("lda_lt_M_mn", dict(mn=1, lda=296, ldb=264), ARG), ("ldb_lt_N_mn", dict(mn=1, lda=304, ldb=256), ARG),
    ("lda_unaligned", dict(lda=204), ALIGN), ("ldb_unaligned", dict(ldb=201), ALIGN),
    ("A0_unaligned", dict(A=ptrs(ctypes.c_void_p(P + 4), A1)), ALIGN),
    ("B1_unaligned", dict(B=ptrs(B0, ctypes.c_void_p(P + 8))), ALIGN),
]


def call_tc(L, fn, a):
    stream = None
    if fn == "svb_gemm_bf16":
        return L.svb_gemm_bf16(a["A"], a["B"], a["nterms"], a["C"], a["bias"], a["M"], a["N"], a["K"], i64(a["lda"]),
                               i64(a["ldb"]), i64(a["ldc"]), a["mn"], a["mn"], stream)
    return L.svb_gemm_bf16_2cta(a["A"], a["B"], a["nterms"], a["C"], a["bias"], a["M"], a["N"], a["K"], i64(a["lda"]),
                                i64(a["ldb"]), i64(a["ldc"]), a["mn"], stream)


@pytest.mark.parametrize("fn", ["svb_gemm_bf16", "svb_gemm_bf16_2cta"])
@pytest.mark.parametrize("name,over,code", REJECT, ids=[r[0] for r in REJECT])
def test_tc_gemm_rejects(L, fn, name, over, code):
    a = dict(GOOD, **over)
    assert call_tc(L, fn, a) == code
    assert L.svb_last_error().decode().startswith(fn + ":"), L.svb_last_error()


def test_tc_gemm_mixed_layouts_check_each_pitch(L):
    """svb_gemm_bf16 with one K-major and one MN-major operand holds each pitch to its own contiguous extent."""
    a = GOOD
    # A K-major (lda >= K = 200), B MN-major (ldb >= N = 264)
    rc = L.svb_gemm_bf16(a["A"], a["B"], 2, C, BIAS, 300, 264, 200, i64(200), i64(200), i64(264), 0, 1, None)
    assert rc == ARG and b"ldb" in L.svb_last_error()
    # A MN-major (lda >= M = 300), B K-major
    rc = L.svb_gemm_bf16(a["A"], a["B"], 2, C, BIAS, 300, 264, 200, i64(296), i64(200), i64(264), 1, 0, None)
    assert rc == ARG and b"lda" in L.svb_last_error()


@pytest.mark.parametrize("fn", ["svb_gemm_bf16", "svb_gemm_bf16_2cta"])
@pytest.mark.parametrize("over", [dict(), dict(mn=1, lda=304, ldb=264), dict(M=1, N=4, K=8, lda=8, ldb=8, ldc=4),
                                  dict(ldc=265, bias=ctypes.c_void_p(P + 4), C=ctypes.c_void_p(P + 4)),
                                  dict(K=8, mn=1, lda=304, ldb=264)])
def test_tc_gemm_accepts(L, fn, over):
    """Valid calls pass the checks (an MN-major pitch may be below K; C and bias need not be 16-byte aligned) and
    fail only later, at the missing driver or device."""
    rc = call_tc(L, fn, dict(GOOD, **over))
    assert rc not in (0, ARG, ALIGN)


PG_GOOD = dict(A=A0, B=B0, C=C, bias=BIAS, M=1000, N=512, K=192, lda=192, ldb=192, ldc=512)
PG_REJECT = [
    ("A_null", dict(A=None), ARG), ("B_null", dict(B=None), ARG), ("C_null", dict(C=None), ARG),
    ("M0", dict(M=0), ARG), ("Mneg", dict(M=-1), ARG),
    ("N0", dict(N=0), ARG), ("N100", dict(N=100), ARG), ("Nneg", dict(N=-256), ARG),
    ("K0", dict(K=0), ARG), ("K96", dict(K=96), ARG), ("Kneg", dict(K=-64), ARG),
    ("lda_lt_K", dict(lda=128), ARG), ("ldb_lt_K", dict(ldb=184), ARG),
    ("ldc_lt_N", dict(ldc=508), ARG), ("ldc_odd", dict(ldc=513), ARG),
    ("bias_unaligned", dict(bias=ctypes.c_void_p(P + 4)), ARG),
    ("lda_unaligned", dict(lda=196), ALIGN), ("ldb_unaligned", dict(ldb=193), ALIGN),
    ("A_unaligned", dict(A=ctypes.c_void_p(P + 2)), ALIGN), ("C_unaligned", dict(C=ctypes.c_void_p(P + 4)), ALIGN),
]


def call_pg(L, a):
    return L.svb_gemm_persistent(a["A"], a["B"], a["C"], a["bias"], a["M"], a["N"], a["K"], i64(a["lda"]),
                                 i64(a["ldb"]), i64(a["ldc"]), 0, None)


@pytest.mark.parametrize("name,over,code", PG_REJECT, ids=[r[0] for r in PG_REJECT])
def test_persistent_rejects(L, name, over, code):
    assert call_pg(L, dict(PG_GOOD, **over)) == code
    assert L.svb_last_error().decode().startswith("svb_gemm_persistent:"), L.svb_last_error()


@pytest.mark.parametrize("over", [dict(), dict(bias=None, lda=256, ldb=200, ldc=516)])
def test_persistent_accepts(L, over):
    assert call_pg(L, dict(PG_GOOD, **over)) not in (0, ARG, ALIGN)
