"""GPU dev timing: the tcgen05 GEMM core (svb_gemm_bf16, one CTA per 128 x 128 tile, and svb_gemm_bf16_2cta, CTA
pairs on 256 x 256 tiles) on the LSTM input-projection shape (B*T = 102400, 4H = 3072, K = 768), 1 and 3 terms, next
to cuBLAS.  Correctness is tests/test_gpu_gemm_core.py.  `python scripts/check_gemm.py 2cta` times the pair kernel
only."""
import ctypes
import sys

import torch

sys.path.insert(0, ".")
from pytorch_speaker_verification_b200 import _lib

L = _lib.lib()
dev = torch.device("cuda:0")
M, N, K = 102400, 3072, 768
A = torch.randn(M, K, device=dev).to(torch.bfloat16)
B = torch.randn(N, K, device=dev).to(torch.bfloat16)
C = torch.empty(M, N, device=dev)
i64 = ctypes.c_int64


def timed(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


entries = [("2cta 256x256", lambda PA, PB, nt: L.svb_gemm_bf16_2cta(PA, PB, nt, _lib.ptr(C), None, M, N, K, i64(K), i64(K),
                                                                     i64(N), 0, _lib.stream_ptr()))]
if not (len(sys.argv) > 1 and sys.argv[1] == "2cta"):
    entries.insert(0, ("input-proj GEMM", lambda PA, PB, nt: L.svb_gemm_bf16(PA, PB, nt, _lib.ptr(C), None, M, N, K,
                                                                             i64(K), i64(K), i64(N), 0, 0,
                                                                             _lib.stream_ptr())))
for name, fn in entries:
    for nt in (1, 3):
        PA = (ctypes.c_void_p * nt)(*[A.data_ptr()] * nt)
        PB = (ctypes.c_void_p * nt)(*[B.data_ptr()] * nt)
        assert fn(PA, PB, nt) == 0, L.svb_last_error()
        ms = timed(lambda: fn(PA, PB, nt))
        print(f"{name} terms={nt}: {ms:.3f} ms, {2 * M * N * K * nt / ms / 1e9:.1f} TFLOP/s", flush=True)
if len(entries) == 2:
    print(f"cuBLAS bf16 same shape: {timed(lambda: A @ B.t()):.3f} ms")
