"""Dev timing: the persistent CTA-pair GEMM (csrc/pgemm.cu) on the LSTM input-projection shape next to the
one-tile-per-CTA pair kernel.  Correctness is tests/test_gpu_gemm_core.py."""
import ctypes, sys
import torch
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from pytorch_speaker_verification_b200 import _lib
from pytorch_speaker_verification_b200._lib import ptr
L = _lib.lib()
st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
i64 = ctypes.c_int64
torch.manual_seed(0)
M, N, K = 102400, 3072, 768
A = torch.randn(M, K, device="cuda").to(torch.bfloat16)
B = (torch.randn(N, K, device="cuda") * 0.05).to(torch.bfloat16)
C = torch.empty(M, N, device="cuda")
PA = (ctypes.c_void_p * 1)(A.data_ptr()); PB = (ctypes.c_void_p * 1)(B.data_ptr())
def t(fn, n=10):
    assert fn() == 0, L.svb_last_error()
    for _ in range(2): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
ms_p = t(lambda: L.svb_gemm_persistent(ptr(A), ptr(B), ptr(C), None, M, N, K, i64(K), i64(K), i64(N), 0, st))
ms_o = t(lambda: L.svb_gemm_bf16_2cta(PA, PB, 1, ptr(C), None, M, N, K, i64(K), i64(K), i64(N), 0, st))
fl = 2.0 * M * N * K / 1e12
print(f"persistent pair kernel: {ms_p:.3f} ms = {fl / ms_p * 1e3:.0f} TFLOP/s;  one tile per CTA pair: {ms_o:.3f} ms = {fl / ms_o * 1e3:.0f} TFLOP/s")
