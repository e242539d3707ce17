// Host helpers for the tcgen05 GEMM core (tensor-map encoding) and the plain GEMM entry point.
#include "tc_gemm.cuh"
#include "epilogues.cuh"
#include "../../include/svb200.h"
#include <stdarg.h>
#include <stdio.h>

namespace svb {
void set_error(const char* what, cudaError_t e);

int host_error(int code, const char* fn, const char* fmt, ...) {
  char msg[384];
  int n = snprintf(msg, sizeof(msg), "%s: ", fn);
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(msg + n, sizeof(msg) - n, fmt, ap);
  va_end(ap);
  set_error(msg, cudaSuccess);
  return code;
}

PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

int make_tmap(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
              uint64_t stride1_elems, uint64_t stride2_elems, uint32_t box0, uint32_t box1, int swizzle) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return SVB_ERR_DRIVER;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_elems * elem_bytes, stride2_elems * elem_bytes};
  cuuint32_t box[3] = {box0, box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (strides[1] & 15)) return SVB_ERR_ALIGN;
  const CUtensorMapSwizzle sw = swizzle == 3 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : swizzle == 2 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "svb: cuTensorMapEncodeTiled failed (%d) elem=%d dims=(%llu,%llu,%llu) strides=(%llu,%llu) box=(%u,%u)\n",
            (int)r, elem_bytes, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
            (unsigned long long)strides[0], (unsigned long long)strides[1], box0, box1);
    return SVB_ERR_DRIVER;
  }
  return SVB_OK;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_elems,
                   uint64_t stride2_elems, uint32_t box_rows) {
  return make_tmap(out, base, 2, d0, d1, d2, stride1_elems, stride2_elems, 64, box_rows, 3);
}

// Operand descriptor for one GEMM side.  K-major: rows x K, ld = row pitch.  MN-major: K x rows, ld = k-row pitch.
int make_operand_map(CUtensorMap* out, const void* p, int rows, int K, int64_t ld, int mn_major, int box_rows_kmajor) {
  if (mn_major) return make_tmap_bf16(out, p, (uint64_t)rows, (uint64_t)K, 1, (uint64_t)ld, (uint64_t)ld * K, kBK);
  return make_tmap_bf16(out, p, (uint64_t)K, (uint64_t)rows, 1, (uint64_t)ld, (uint64_t)ld * rows, box_rows_kmajor);
}

}  // namespace svb

using namespace svb;

namespace {

// Validates the arguments shared by svb_gemm_bf16 and svb_gemm_bf16_2cta before any CUDA call.  An MN-major operand
// is stored [K, rows], so its pitch must span its rows; a K-major one is stored [rows, K], so its pitch must span K.
// The kernel does not need C or bias aligned: make_store_params falls back to direct stores.
int check_gemm_args(const char* fn, const void* const* A, const void* const* B, int nterms, const float* C, int M,
                    int N, int K, int64_t lda, int64_t ldb, int64_t ldc, int a_mn, int b_mn) {
  if (M < 1) return host_error(SVB_ERR_ARG, fn, "M = %d, needs M >= 1", M);
  if (N < 1) return host_error(SVB_ERR_ARG, fn, "N = %d, needs N >= 1", N);
  if (K < 1) return host_error(SVB_ERR_ARG, fn, "K = %d, needs K >= 1", K);
  if (nterms < 1 || nterms > kMaxTerms)
    return host_error(SVB_ERR_ARG, fn, "nterms = %d, needs 1 <= nterms <= %d", nterms, kMaxTerms);
  if (!A || !B) return host_error(SVB_ERR_ARG, fn, "A and B must be host arrays of nterms pointers");
  for (int t = 0; t < nterms; ++t) {
    if (!A[t]) return host_error(SVB_ERR_ARG, fn, "A[%d] is NULL", t);
    if (!B[t]) return host_error(SVB_ERR_ARG, fn, "B[%d] is NULL", t);
  }
  if (!C) return host_error(SVB_ERR_ARG, fn, "C is NULL");
  if (lda < (a_mn ? M : K))
    return host_error(SVB_ERR_ARG, fn, "lda = %lld, needs lda >= %s", (long long)lda, a_mn ? "M (A is MN-major)" : "K");
  if (ldb < (b_mn ? N : K))
    return host_error(SVB_ERR_ARG, fn, "ldb = %lld, needs ldb >= %s", (long long)ldb, b_mn ? "N (B is MN-major)" : "K");
  if (ldc < N) return host_error(SVB_ERR_ARG, fn, "ldc = %lld, needs ldc >= N = %d", (long long)ldc, N);
  // tensor-map operands: 16-byte aligned bases and pitches
  if (lda % 8) return host_error(SVB_ERR_ALIGN, fn, "lda = %lld is not a multiple of 8 elements", (long long)lda);
  if (ldb % 8) return host_error(SVB_ERR_ALIGN, fn, "ldb = %lld is not a multiple of 8 elements", (long long)ldb);
  for (int t = 0; t < nterms; ++t) {
    if (reinterpret_cast<uintptr_t>(A[t]) & 15) return host_error(SVB_ERR_ALIGN, fn, "A[%d] is not 16-byte aligned", t);
    if (reinterpret_cast<uintptr_t>(B[t]) & 15) return host_error(SVB_ERR_ALIGN, fn, "B[%d] is not 16-byte aligned", t);
  }
  return SVB_OK;
}

int make_gemm_operands(const char* fn, GemmOperands* ops, const void* const* A, const void* const* B, int nterms,
                       int M, int N, int K, int64_t lda, int64_t ldb, int a_mn, int b_mn) {
  memset(ops, 0, sizeof(*ops));
  ops->nterms = nterms; ops->M = M; ops->N = N; ops->K = K;
  for (int t = 0; t < nterms; ++t) {
    int e = make_operand_map(&ops->ta[t], A[t], M, K, lda, a_mn, kBM);
    if (e) return host_error(e, fn, "tensor map of A[%d] rejected", t);
    e = make_operand_map(&ops->tb[t], B[t], N, K, ldb, b_mn, 128);   // a CTA pair loads 128 of its 256 B rows per CTA
    if (e) return host_error(e, fn, "tensor map of B[%d] rejected", t);
  }
  return SVB_OK;
}

}  // namespace

extern "C" int svb_gemm_bf16(const void* const* A, const void* const* B, int nterms, float* C, const float* bias,
                             int M, int N, int K, int64_t lda, int64_t ldb, int64_t ldc, int a_mn, int b_mn,
                             void* stream) {
  const char* fn = "svb_gemm_bf16";
  int e = check_gemm_args(fn, A, B, nterms, C, M, N, K, lda, ldb, ldc, a_mn, b_mn);
  if (e) return e;
  GemmOperands ops;
  e = make_gemm_operands(fn, &ops, A, B, nterms, M, N, K, lda, ldb, a_mn, b_mn);
  if (e) return e;
  EpiStoreF32<128>::Params ep;
  e = make_store_params<128>(&ep, C, bias, M, N, ldc, 0);
  if (e) return host_error(e, fn, "tensor map of C rejected");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  cudaError_t err;
  if (!a_mn && !b_mn) err = launch_tc_gemm<128, 4, false, false, EpiStoreF32<128>>(ops, ep, s);
  else if (a_mn && b_mn) err = launch_tc_gemm<128, 4, true, true, EpiStoreF32<128>>(ops, ep, s);
  else if (!a_mn && b_mn) err = launch_tc_gemm<128, 4, false, true, EpiStoreF32<128>>(ops, ep, s);
  else err = launch_tc_gemm<128, 4, true, false, EpiStoreF32<128>>(ops, ep, s);
  if (err != cudaSuccess) { set_error("svb_gemm_bf16: launch", err); return SVB_ERR_CUDA; }
  return SVB_OK;
}

// CTA-pair variant (tcgen05.mma.cta_group::2, 256 x 256 pair tiles): both operands K-major (mn = 0) or both
// MN-major (mn = 1).
extern "C" int svb_gemm_bf16_2cta(const void* const* A, const void* const* B, int nterms, float* C, const float* bias,
                                  int M, int N, int K, int64_t lda, int64_t ldb, int64_t ldc, int mn, void* stream) {
  const char* fn = "svb_gemm_bf16_2cta";
  int e = check_gemm_args(fn, A, B, nterms, C, M, N, K, lda, ldb, ldc, mn, mn);
  if (e) return e;
  GemmOperands ops;
  e = make_gemm_operands(fn, &ops, A, B, nterms, M, N, K, lda, ldb, mn, mn);
  if (e) return e;
  EpiStoreF32<256>::Params ep;
  e = make_store_params<256>(&ep, C, bias, M, N, ldc, 0);
  if (e) return host_error(e, fn, "tensor map of C rejected");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const cudaError_t err = mn ? launch_tc_gemm<256, 6, true, true, EpiStoreF32<256>, 8, 1, true>(ops, ep, s)
                             : launch_tc_gemm<256, 6, false, false, EpiStoreF32<256>, 8, 1, true>(ops, ep, s);
  if (err != cudaSuccess) { set_error("svb_gemm_bf16_2cta: launch", err); return SVB_ERR_CUDA; }
  return SVB_OK;
}
