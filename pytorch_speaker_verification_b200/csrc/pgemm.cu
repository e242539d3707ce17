// Persistent CTA-pair GEMM for short reductions: C[M, N] = A[M, K] . B[N, K]^T (+ bias[n]), bf16 or fp16 operands
// (K-major), fp32 accumulate and output.
//
// Written for the LSTM input projection taken as a standalone batched GEMM over all frames (speech_embedder_net.py:19,28:
// the W_ih x_t half of nn.LSTM, [T*B = 102400 x 768] . [768 x 3072] at BASELINE configs[1]), the shape north_star's
// ">= 80 % tensor-pipe utilisation" target is stated on.  With K = 768 a 256 x 256 pair tile is only 12 k-blocks of
// tensor work (6144 cycles) followed by a 256 KB fp32 epilogue: the one-tile-per-CTA kernel (tc_gemm.cuh, 9600 CTAs)
// spent more time in prologues, epilogues and tails than in MMAs (tensor pipe 32 %).  Here:
//   * 74 CTA pairs (cluster 2, tcgen05.mma.cta_group::2, M = 256 x N = 256 per instruction) walk the tiles round-robin,
//     N-tile fastest, so that the 74 pairs in flight share 6-7 row blocks of A through L2;
//   * TWO accumulators (2 x 256 TMEM columns): the epilogue of tile i (tcgen05.ld -> +bias -> 128B-swizzled staging ->
//     TMA store, 32 columns at a time through double-buffered 16 KB buffers per warp group) runs under the MMAs of
//     tile i+1; the operand ring (5 x 32 KB per CTA) keeps streaming across tile boundaries;
//   * the MMA thread runs the whole loop itself (`if (elect_one())` around it, see wlstm.cuh).
// Roles per CTA (320 threads): warp 0 TMA producer, warp 1 MMA issuer (leader CTA only), warps 2-9 epilogue (two warps
// per TMEM lane quarter, each taking four of the eight 32-column chunks).
#include "tc_gemm.cuh"
#include "../../include/svb200.h"

namespace svb {
void set_error(const char* what, cudaError_t e);

constexpr int kPgStages = 5;
constexpr int kPgStageBytes = 2 * kBM * kBK * 2;          // A 128 x 64 + this CTA's half of B 128 x 64, 2-byte elements
constexpr int kPgRing = kPgStages * kPgStageBytes;        // 160 KB
constexpr int kPgStg = 4 * 16384;                         // 2 warp groups x 2 buffers of [128 rows x 32 fp32]
constexpr int kPgSmem = kPgRing + kPgStg + 1024 + 1024;
constexpr int kPgThreads = 64 + 256;

struct __align__(64) PgParams {
  CUtensorMap ta, tb;      // operands [rows][K], box {64, 128}, SW128
  CUtensorMap tc;          // fp32 C [M][N], box {32, 128}, SW128
  const float* bias;       // [N] or null
  int M, N, K, f16;
};

__global__ void __launch_bounds__(kPgThreads, 1) pgemm_kernel(const __grid_constant__ PgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stg = smem + kPgRing;
  uint64_t* full = reinterpret_cast<uint64_t*>(stg + kPgStg);
  uint64_t* empty = full + kPgStages;
  uint64_t* acc_full = empty + kPgStages;      // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2] (used in the leader CTA: 16 epilogue warps of the pair)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int ntn = p.N / 256;
  const int total = ((p.M + 255) / 256) * ntn;
  const int nkb = p.K / kBK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPgStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 16); }
    fence_mbar_init();
    tma_prefetch_desc(&p.ta);
    tma_prefetch_desc(&p.tb);
    tma_prefetch_desc(&p.tc);
  }
  if (warp == 1) tmem_alloc_2cta<512>(tmem_holder);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int ti = pair; ti < total; ti += npairs) {
        const int m0 = (ti / ntn) * 256 + rank * 128;          // this CTA's 128 rows of A
        const int n0 = (ti % ntn) * 256 + rank * 128;          // ... and its half of the 256 B rows
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kPgStageBytes;
          if (rank == 0) mbar_expect_tx(&full[stage], 2 * kPgStageBytes);     // both CTAs' bytes go to the leader
          tma_load_3d_2cta(sa, &p.ta, &full[stage], kb * kBK, m0, 0);
          tma_load_3d_2cta(sa + kBM * kBK * 2, &p.tb, &full[stage], kb * kBK, n0, 0);
          if (++stage == kPgStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA)
    if (rank == 0 && elect_one()) {
      const uint32_t idesc = p.f16 ? umma_idesc_f16(256, 256, 0, 0) : umma_idesc_bf16(256, 256, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int i = 0;
      for (int ti = pair; ti < total; ti += npairs, ++i) {
        const int b = i & 1;
        mbar_wait(&acc_empty[b], (uint32_t)(((i >> 1) & 1) ^ 1));      // both CTAs' epilogues have drained tile i-2
        tc_fence_after();
        const uint32_t dacc = tmem + b * 256;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kPgStageBytes);
          const uint32_t sb = sa + kBM * kBK * 2;
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_bf16_ss_2cta(dacc, umma_desc_kmajor_sw128(sa + k * 32), umma_desc_kmajor_sw128(sb + k * 32), idesc,
                              (kb | k) != 0 ? 1u : 0u);
          umma_commit_2cta(&empty[stage]);                       // frees the slot in both CTAs
          if (kb == nkb - 1) umma_commit_2cta(&acc_full[b]);     // accumulator complete in both CTAs
          if (++stage == kPgStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (both CTAs)
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;             // chunks [4 grp, 4 grp + 4)
    const int row = q * 32 + lane;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    const bool lead = (warp - 2) == grp * 4 && lane == 0;       // issues the group's TMA stores
    const uint32_t acc_empty_leader = map_to_cta(smem_u32(acc_empty), 0);
    int i = 0;
    for (int ti = pair; ti < total; ti += npairs, ++i) {
      const int b = i & 1;
      const int m0 = (ti / ntn) * 256 + rank * 128;
      const int n0 = (ti % ntn) * 256;
      mbar_wait(&acc_full[b], (uint32_t)((i >> 1) & 1));
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < 4; ++cc) {
        const int c = grp * 4 + cc;
        float acc[32];
        tmem_ld32(tmem + lane_base + b * 256 + c * 32, acc);
        tmem_ld_wait();
        if (cc == 3) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0)
            asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(acc_empty_leader + b * 8) : "memory");
        }
        uint8_t* o = stg + (grp * 2 + (cc & 1)) * 16384;
        if (lead) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");     // the store of 2 chunks ago has read `o`
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
        const int nc = n0 + c * 32;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 v = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
          if (p.bias) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + nc + 4 * j));
            v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
          }
          *reinterpret_cast<float4*>(o + sw128(row, j)) = v;
        }
        fence_proxy_async_smem();
        asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
        if (lead) {
          tma_store_3d(&p.tc, o, nc, m0, 0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
    }
    if (lead) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();                          // neither CTA leaves while its peer may still signal it
  if (warp == 1) tmem_dealloc_2cta<512>(tmem);
}

}  // namespace svb
using namespace svb;

// C[M, N] (fp32, row pitch ldc) = A[M, K] . B[N, K]^T + bias: persistent CTA-pair kernel for short K.  Operands
// K-major, 2-byte elements (f16 != 0: IEEE half, else bf16); K % 64 == 0, N % 256 == 0, 16-byte aligned pitches.
extern "C" int svb_gemm_persistent(const void* A, const void* B, float* C, const float* bias, int M, int N, int K,
                                   int64_t lda, int64_t ldb, int64_t ldc, int f16, void* stream) {
  const char* fn = "svb_gemm_persistent";
  if (!A) return host_error(SVB_ERR_ARG, fn, "A is NULL");
  if (!B) return host_error(SVB_ERR_ARG, fn, "B is NULL");
  if (!C) return host_error(SVB_ERR_ARG, fn, "C is NULL");
  if (M < 1) return host_error(SVB_ERR_ARG, fn, "M = %d, needs M >= 1", M);
  if (N < 256 || N % 256) return host_error(SVB_ERR_ARG, fn, "N = %d, needs a positive multiple of 256", N);
  if (K < 64 || K % 64) return host_error(SVB_ERR_ARG, fn, "K = %d, needs a positive multiple of 64", K);
  if (lda < K) return host_error(SVB_ERR_ARG, fn, "lda = %lld, needs lda >= K", (long long)lda);
  if (ldb < K) return host_error(SVB_ERR_ARG, fn, "ldb = %lld, needs ldb >= K", (long long)ldb);
  if (ldc < N) return host_error(SVB_ERR_ARG, fn, "ldc = %lld, needs ldc >= N", (long long)ldc);
  if (ldc % 4) return host_error(SVB_ERR_ARG, fn, "ldc = %lld is not a multiple of 4", (long long)ldc);
  if (bias && (reinterpret_cast<uintptr_t>(bias) & 15)) return host_error(SVB_ERR_ARG, fn, "bias is not 16-byte aligned");
  if (lda % 8) return host_error(SVB_ERR_ALIGN, fn, "lda = %lld is not a multiple of 8 elements", (long long)lda);
  if (ldb % 8) return host_error(SVB_ERR_ALIGN, fn, "ldb = %lld is not a multiple of 8 elements", (long long)ldb);
  if (reinterpret_cast<uintptr_t>(A) & 15) return host_error(SVB_ERR_ALIGN, fn, "A is not 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(B) & 15) return host_error(SVB_ERR_ALIGN, fn, "B is not 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(C) & 15) return host_error(SVB_ERR_ALIGN, fn, "C is not 16-byte aligned");
  PgParams p;
  memset(&p, 0, sizeof(p));
  int e = make_tmap_bf16(&p.ta, A, (uint64_t)K, (uint64_t)M, 1, (uint64_t)lda, (uint64_t)lda * M, kBM);
  if (e) return host_error(e, fn, "tensor map of A rejected");
  e = make_tmap_bf16(&p.tb, B, (uint64_t)K, (uint64_t)N, 1, (uint64_t)ldb, (uint64_t)ldb * N, kBM);
  if (e) return host_error(e, fn, "tensor map of B rejected");
  e = make_tmap(&p.tc, C, 4, (uint64_t)N, (uint64_t)M, 1, (uint64_t)ldc, (uint64_t)ldc * M, 32, 128, 3);
  if (e) return host_error(e, fn, "tensor map of C rejected");
  p.bias = bias; p.M = M; p.N = N; p.K = K; p.f16 = f16;
  static unsigned long long configured = 0;
  if (first_use_on_device(configured)) {
    cudaError_t ce = cudaFuncSetAttribute(pgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPgSmem);
    if (ce != cudaSuccess) { set_error("svb_gemm_persistent: cudaFuncSetAttribute", ce); return SVB_ERR_CUDA; }
  }
  const int total = ((M + 255) / 256) * (N / 256);
  int pairs = device_sm_count() / 2;
  if (pairs > total) pairs = total;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(kPgThreads);
  cfg.dynamicSmemBytes = kPgSmem;
  cfg.stream = reinterpret_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t ce = cudaLaunchKernelEx(&cfg, pgemm_kernel, p);
  if (ce != cudaSuccess) { set_error("svb_gemm_persistent: launch", ce); return SVB_ERR_CUDA; }
  return SVB_OK;
}
