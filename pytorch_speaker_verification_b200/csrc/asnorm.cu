// Cohort score normalization (S-norm and adaptive S-norm, DESIGN.md 4.5.2) for sm_100a.
//
// Cohort statistics of a row x against a cohort C of Nc rows with top-K: S_K(x) = the K largest cos(x, c); mu = mean,
// sigma = sample standard deviation (divisor K - 1) and v_K = the K-th largest value of S_K(x).  The normalized score of
// a trial (e, t) with raw cosine s is 1/2 ((s - mu(e)) / sigma(e) + (s - mu(t)) / sigma(t)).
//
// svb_cohort_stats, per chunk of rows (the chunk keeps its score slab L2-resident):
//   prepare   unit rows split into IEEE-half hi / lo, zero-padded to Dp = round64(D) columns (the cohort also to a
//             multiple of 8 rows); zero padding leaves every dot product unchanged
//   GEMM      slab = X^ C^T on tcgen05 as the 3-term split product hi hi + hi lo + lo hi (tc_gemm_kernel, as GE2E's)
//   stats     one CTA per row: radix select of v_K on order-preserving uint32 keys (11 + 11 + 10 bit digits, shared
//             digit histograms), then float64 sums over the selected values in a fixed thread assignment and tree order:
//             mu = v_K + sum_{v > v_K} (v - v_K) / K, sigma^2 = (sum_{v > v_K} (v - mu)^2 + (K - c_>) (v_K - mu)^2) / (K - 1)
// svb_cohort_stats_scores runs the stats kernel on caller-supplied scores.  svb_score_trials (one warp per trial, float64
// dot products) and svb_asnorm_sim (elementwise over the TI-SV matrix) apply the statistics.
// No float atomics, no allocation, no host synchronisation: every output is run-to-run identical and the calls can be
// captured in a CUDA graph.
#include <cuda_fp16.h>
#include "tc_gemm.cuh"
#include "epilogues.cuh"
#include "../../include/svb200.h"
#include "perdev.cuh"
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

namespace svb {
void set_error(const char* what, cudaError_t e);
int make_operand_map(CUtensorMap* out, const void* p, int rows, int K, int64_t ld, int mn_major, int box_rows_kmajor);

namespace asnorm {
constexpr int kMaxCohort = 1 << 20;
constexpr int kStatThreads = 256;
constexpr int kStatWarps = kStatThreads / 32;
constexpr int kBins = 2048;                             // 11-bit digits; the last pass uses 10 bits
constexpr int kBinsPerThread = kBins / kStatThreads;    // 8
constexpr int kStageMax = 12288;                        // rows up to 48 KB of keys are staged in shared memory
constexpr size_t kSlabBytes = (size_t)48 << 20;         // score slab per chunk (L2-resident: the B200 has 126 MB)

__device__ __forceinline__ uint32_t score_key(float x, unsigned& nonfinite) {
  uint32_t u = __float_as_uint(x);
  if (u == 0x80000000u) u = 0u;                         // -0 counts as +0 (bit test: denormals stay distinct)
  nonfinite += (u & 0x7f800000u) == 0x7f800000u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ double key_value(uint32_t key) {
  const uint32_t u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return (double)__uint_as_float(u);
}

// ------------------------------------------------------------------------------------------------- (a) prepare
// One warp per output row r < rows_out: rows r < rows_in are X[r0 + r] / |X[r0 + r]| split into hi + lo (float64 norm,
// so no finite row overflows); rows past rows_in and columns past D are zero.  A row with a zero or non-finite norm is
// written as NaN, so every cosine it takes part in, and every statistic, is NaN.
__global__ void __launch_bounds__(256) asnorm_prepare_kernel(const float* __restrict__ X, int64_t r0, int rows_in,
                                                             int rows_out, int D, int Dp, __half* __restrict__ hi,
                                                             __half* __restrict__ lo) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= rows_out) return;
  __half* h = hi + r * Dp;
  __half* l = lo + r * Dp;
  if (r >= rows_in) {
    for (int d = lane; d < Dp; d += 32) { h[d] = __float2half_rn(0.f); l[d] = __float2half_rn(0.f); }
    return;
  }
  const float* x = X + (r0 + r) * (int64_t)D;
  double ss = 0.0;
  for (int d = lane; d < D; d += 32) { const double v = x[d]; ss = fma(v, v, ss); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const double nrm = sqrt(ss);
  const double inv = (nrm > 0.0 && isfinite(nrm)) ? 1.0 / nrm : (double)NAN;
  for (int d = lane; d < Dp; d += 32) {
    const float v = d < D ? (float)((double)x[d] * inv) : 0.f;
    const __half vh = __float2half_rn(v);
    h[d] = vh;
    l[d] = __float2half_rn(v - __half2float(vh));
  }
}

// ------------------------------------------------------------------------------------------------- (b) statistics
// Exclusive scan of one value per thread in DESCENDING thread order (thread 255 first); *total = the block's sum.
__device__ __forceinline__ uint32_t scan_from_top(uint32_t v, uint32_t* warp_tot, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_down_sync(0xffffffffu, incl, o);
    if (lane + o < 32) incl += y;
  }
  if (lane == 0) warp_tot[warp] = incl;
  __syncthreads();
  uint32_t above = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kStatWarps; ++w) {
    const uint32_t t = warp_tot[w];
    above += w > warp ? t : 0u;
    all += t;
  }
  __syncthreads();
  *total = all;
  return above + incl - v;
}

// Fixed-order block sum of one double per thread (warp xor tree, then the warps in order); valid in every thread.
__device__ __forceinline__ double block_sum_f64(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
#pragma unroll
  for (int w = 1; w < kStatWarps; ++w) t += red[w];
  __syncthreads();
  return t;
}

// One CTA per row of S (row pitch ld): out[row] = {mu, sigma, v_K}.  kStaged: the row's keys live in dynamic shared
// memory (Nc <= kStageMax); otherwise every pass re-reads the row (from L2 when it comes from the chunk's slab).
// Thread t owns elements t, t + 256, ... in every pass.
template <bool kStaged>
__global__ void __launch_bounds__(kStatThreads) asnorm_stats_kernel(const float* __restrict__ S, int64_t ld, int Nc,
                                                                    int K, double inv_k, double inv_k1,
                                                                    double* __restrict__ out) {
  extern __shared__ uint32_t staged[];
  __shared__ uint32_t hist[kBins];
  __shared__ uint32_t warp_tot[kStatWarps];
  __shared__ double red[kStatWarps];
  __shared__ uint32_t s_bin, s_above;
  const int tid = threadIdx.x, lane = tid & 31;
  const float* row = S + (int64_t)blockIdx.x * ld;
  unsigned nonfinite = 0;
  if (kStaged) {
    for (int i = tid; i < Nc; i += kStatThreads) staged[i] = score_key(__ldg(row + i), nonfinite);
  }
  auto key_at = [&](int i, unsigned& nf) -> uint32_t { return kStaged ? staged[i] : score_key(__ldg(row + i), nf); };

  uint32_t prefix = 0, pmask = 0, krem = (uint32_t)K, cgt = 0;
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
    const int shift = pass == 0 ? 21 : pass == 1 ? 10 : 0;
    const uint32_t dmask = pass == 2 ? 0x3ffu : 0x7ffu;
    for (int b = tid; b < kBins; b += kStatThreads) hist[b] = 0;
    __syncthreads();                                    // also orders the staging stores before the first reads
    unsigned nf = 0;
    for (int i0 = 0; i0 < Nc; i0 += kStatThreads) {     // warp-uniform trip count for __match_any_sync
      const int i = i0 + tid;
      uint32_t d = 0xffffffffu;
      if (i < Nc) {
        const uint32_t key = key_at(i, nf);
        if ((key & pmask) == prefix) d = (key >> shift) & dmask;
      }
      const unsigned peers = __match_any_sync(0xffffffffu, d);   // one shared atomic per distinct digit in the warp
      if (d != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(&hist[d], (uint32_t)__popc(peers));
    }
    if (!kStaged && pass == 0) nonfinite = nf;
    __syncthreads();
    // the digit b whose run holds the krem-th largest candidate: (count above b) < krem <= (count above b) + hist[b]
    const int b0 = tid * kBinsPerThread;
    uint32_t mine = 0;
#pragma unroll
    for (int j = 0; j < kBinsPerThread; ++j) mine += hist[b0 + j];
    uint32_t total;
    uint32_t above = scan_from_top(mine, warp_tot, &total);
    if (above < krem && krem <= above + mine) {
#pragma unroll
      for (int j = kBinsPerThread - 1; j >= 0; --j) {
        const uint32_t c = hist[b0 + j];
        if (krem <= above + c) { s_bin = (uint32_t)(b0 + j); s_above = above; break; }
        above += c;
      }
    }
    __syncthreads();
    prefix |= s_bin << shift;
    pmask |= dmask << shift;
    cgt += s_above;
    krem -= s_above;
  }
  // prefix = key of v_K, cgt = number of values above it
  {
    uint32_t w = nonfinite;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
    if (lane == 0) warp_tot[tid >> 5] = w;
    __syncthreads();
    if (tid == 0) {
      uint32_t t = 0;
      for (int k = 0; k < kStatWarps; ++k) t += warp_tot[k];
      s_bin = t;
    }
    __syncthreads();
  }
  const bool bad = s_bin != 0;
  const double vK = key_value(prefix);
  unsigned dummy = 0;
  double sum = 0.0;
  for (int i = tid; i < Nc; i += kStatThreads) {
    const uint32_t key = key_at(i, dummy);
    if (key > prefix) sum += key_value(key) - vK;
  }
  sum = block_sum_f64(sum, red);
  const double mu = fma(sum, inv_k, vK);                // mu = v_K + sum(v - v_K) / K: exactly v_K when all are equal
  double sq = 0.0;
  for (int i = tid; i < Nc; i += kStatThreads) {
    const uint32_t key = key_at(i, dummy);
    if (key > prefix) { const double e = key_value(key) - mu; sq = fma(e, e, sq); }
  }
  sq = block_sum_f64(sq, red);
  if (tid == 0) {
    const double e = vK - mu;
    const double var = fma((double)(K - (int)cgt) * e, e, sq) * inv_k1;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    double* o = out + (size_t)blockIdx.x * 3;
    o[0] = bad ? qnan : mu;
    o[1] = bad ? qnan : sqrt(var);
    o[2] = bad ? qnan : vK;
  }
}

// ------------------------------------------------------------------------------------------------- (c) trials
__device__ __forceinline__ double normalize(double s, const double* st) { return (s - st[0]) / st[1]; }

// One warp per trial: s = cos(E[ei], T[ti]) from float64 dot products (each float product is exact in float64), then
// the normalized score when statistics are given.  An index out of range gives NaN and reads nothing.
__global__ void __launch_bounds__(256) asnorm_trials_kernel(const float* __restrict__ E, int64_t ne,
                                                            const float* __restrict__ T, int64_t nt, int D,
                                                            const int32_t* __restrict__ ei,
                                                            const int32_t* __restrict__ ti, int64_t n_trials,
                                                            const double* __restrict__ se,
                                                            const double* __restrict__ stt, float* __restrict__ out,
                                                            int vec) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (i >= n_trials) return;
  const int64_t a = __ldg(ei + i), b = __ldg(ti + i);
  if (a < 0 || a >= ne || b < 0 || b >= nt) {
    if (lane == 0) out[i] = __int_as_float(0x7fc00000);
    return;
  }
  const float* x = E + a * D;
  const float* y = T + b * D;
  double xx = 0.0, yy = 0.0, xy = 0.0;
  if (vec) {                                            // D % 4 == 0 and 16-byte aligned rows
    const float4* x4 = reinterpret_cast<const float4*>(x);
    const float4* y4 = reinterpret_cast<const float4*>(y);
    for (int q = lane; q < D / 4; q += 32) {
      const float4 u = __ldg(x4 + q), v = __ldg(y4 + q);
      const float us[4] = {u.x, u.y, u.z, u.w}, vs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const double p = us[k], r = vs[k];
        xx = fma(p, p, xx); yy = fma(r, r, yy); xy = fma(p, r, xy);
      }
    }
  } else {
    for (int d = lane; d < D; d += 32) {
      const double p = __ldg(x + d), r = __ldg(y + d);
      xx = fma(p, p, xx); yy = fma(r, r, yy); xy = fma(p, r, xy);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    xx += __shfl_xor_sync(0xffffffffu, xx, o);
    yy += __shfl_xor_sync(0xffffffffu, yy, o);
    xy += __shfl_xor_sync(0xffffffffu, xy, o);
  }
  if (lane == 0) {
    const double nx = sqrt(xx), ny = sqrt(yy);
    double s = (nx > 0.0 && ny > 0.0) ? xy / nx / ny : (double)NAN;
    if (se) s = 0.5 * (normalize(s, se + 3 * a) + normalize(s, stt + 3 * b));
    out[i] = (float)s;
  }
}

// ------------------------------------------------------------------------------------------------- (d) TI-SV matrix
// out[j, m, k] = 1/2 ((sim - mu_c[k]) / sigma_c[k] + (sim - mu_v[j, m]) / sigma_v[j, m]) for sim (N, Mv, N): rows
// [j, m] over the blocks, k over the threads.
__global__ void __launch_bounds__(256) asnorm_sim_kernel(const float* __restrict__ sim, int N, int rows,
                                                         const double* __restrict__ sc, const double* __restrict__ sv,
                                                         float* __restrict__ out) {
  for (int jm = blockIdx.x; jm < rows; jm += gridDim.x) {
    const double mv = __ldg(sv + 3 * (int64_t)jm), dv = __ldg(sv + 3 * (int64_t)jm + 1);
    const float* s_row = sim + (int64_t)jm * N;
    float* o_row = out + (int64_t)jm * N;
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
      const double s = __ldg(s_row + k);
      o_row[k] = (float)(0.5 * ((s - __ldg(sc + 3 * k)) / __ldg(sc + 3 * k + 1) + (s - mv) / dv));
    }
  }
}

// ------------------------------------------------------------------------------------------------- host side
inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Rows per chunk: the (rows x Ncp) fp32 slab stays within kSlabBytes (SVB_ASNORM_SLAB_MB overrides it for the chunk
// measurement of DESIGN.md 4.5.2), in whole 128-row GEMM tiles, at least one tile.
inline int chunk_rows(int Ncp) {
  static const size_t slab = getenv("SVB_ASNORM_SLAB_MB") ? (size_t)atoll(getenv("SVB_ASNORM_SLAB_MB")) << 20
                                                          : kSlabBytes;
  const size_t rows = slab / ((size_t)Ncp * 4) / 128 * 128;
  return (int)(rows < 128 ? 128 : rows > (1 << 20) ? (1 << 20) : rows);
}

// Workspace: cohort hi / lo (Ncp x Dp halves each), chunk hi / lo (rows x Dp halves each), score slab (rows x Ncp fp32).
struct Layout {
  size_t ch, cl, xh, xl, slab, total;
  int Ncp, Dp, rows;
};

inline Layout layout(int64_t n, int Nc, int D) {
  Layout L;
  L.Ncp = round_up(Nc, 8);
  L.Dp = round_up(D, 64);
  const int chunk = chunk_rows(L.Ncp);
  L.rows = (int)(n < chunk ? n : chunk);
  const size_t cb = align_up((size_t)L.Ncp * L.Dp * 2), xb = align_up((size_t)L.rows * L.Dp * 2);
  L.ch = 0;
  L.cl = cb;
  L.xh = 2 * cb;
  L.xl = L.xh + xb;
  L.slab = L.xl + xb;
  L.total = L.slab + align_up((size_t)L.rows * L.Ncp * 4);
  return L;
}

inline bool dims_ok(int64_t n, int Nc, int D) {
  return n >= 1 && n < (int64_t(1) << 31) && Nc >= 2 && Nc <= kMaxCohort && D >= 1 && D <= 65536;
}

int launch_stats(const float* S, int64_t n, int Nc, int64_t ld, int K, double* out, cudaStream_t st) {
  if (Nc <= kStageMax) {
    static unsigned long long attr_done = 0;
    if (first_use_on_device(attr_done)) {
      cudaError_t e = cudaFuncSetAttribute(asnorm_stats_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           kStageMax * 4);
      if (e != cudaSuccess) { attr_done = 0; set_error("asnorm stats kernel attribute", e); return SVB_ERR_CUDA; }
    }
    asnorm_stats_kernel<true><<<(unsigned)n, kStatThreads, (size_t)Nc * 4, st>>>(S, ld, Nc, K, 1.0 / K, 1.0 / (K - 1), out);
  } else {
    asnorm_stats_kernel<false><<<(unsigned)n, kStatThreads, 0, st>>>(S, ld, Nc, K, 1.0 / K, 1.0 / (K - 1), out);
  }
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("asnorm stats kernel launch", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

// slab[rows, Ncp] = Xh Ch^T + Xh Cl^T + Xl Ch^T (tc_gemm_kernel, 128 x 128 tiles, TMA store).
int cohort_gemm(const __half* Xh, const __half* Xl, int rows, const __half* Ch, const __half* Cl, int Ncp, int Dp,
                float* slab, cudaStream_t st) {
  GemmOperands g;
  memset(&g, 0, sizeof(g));
  g.nterms = 3; g.f16 = 1; g.M = rows; g.N = Ncp; g.K = Dp;
  const __half* As[3] = {Xh, Xh, Xl};
  const __half* Bs[3] = {Ch, Cl, Ch};
  for (int t = 0; t < 3; ++t) {
    int e = make_operand_map(&g.ta[t], As[t], rows, Dp, Dp, 0, kBM);
    if (e) return e;
    e = make_operand_map(&g.tb[t], Bs[t], Ncp, Dp, Dp, 0, 128);
    if (e) return e;
  }
  EpiStoreF32<128>::Params ep;
  int e = make_store_params<128>(&ep, slab, nullptr, rows, Ncp, (int64_t)Ncp, 0);
  if (e) return e;
  if (!ep.use_tma) { set_error("svb_cohort_stats: score slab is not 16-byte aligned", cudaSuccess); return SVB_ERR_ALIGN; }
  const cudaError_t ce = launch_tc_gemm<128, 4, false, false, EpiStoreF32<128>>(g, ep, st);
  if (ce != cudaSuccess) { set_error("svb_cohort_stats: tensor-core GEMM", ce); return SVB_ERR_CUDA; }
  return SVB_OK;
}

}  // namespace asnorm
}  // namespace svb

using namespace svb::asnorm;

extern "C" int svb_cohort_stats_workspace_bytes(int64_t n, int Nc, int D, size_t* bytes) {
  if (!bytes || !dims_ok(n, Nc, D)) {
    svb::set_error("svb_cohort_stats_workspace_bytes: need 1 <= n < 2^31, 2 <= Nc <= 2^20, 1 <= D <= 65536",
                   cudaSuccess);
    return SVB_ERR_ARG;
  }
  *bytes = layout(n, Nc, D).total;
  return SVB_OK;
}

extern "C" int svb_cohort_stats(const float* X, int64_t n, const float* cohort, int Nc, int D, int K, void* workspace,
                                size_t workspace_bytes, double* out, void* stream) {
  if (!X || !cohort || !workspace || !out || !dims_ok(n, Nc, D) || K < 2 || K > Nc ||
      (reinterpret_cast<uintptr_t>(workspace) & 255)) {
    svb::set_error("svb_cohort_stats: bad argument (1 <= n < 2^31, 2 <= K <= Nc <= 2^20, 1 <= D <= 65536, workspace "
                   "256-byte aligned)", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const Layout L = layout(n, Nc, D);
  if (workspace_bytes < L.total) {
    svb::set_error("svb_cohort_stats: workspace smaller than svb_cohort_stats_workspace_bytes", cudaSuccess);
    return SVB_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  __half* Ch = reinterpret_cast<__half*>(ws + L.ch);
  __half* Cl = reinterpret_cast<__half*>(ws + L.cl);
  __half* Xh = reinterpret_cast<__half*>(ws + L.xh);
  __half* Xl = reinterpret_cast<__half*>(ws + L.xl);
  float* slab = reinterpret_cast<float*>(ws + L.slab);
  asnorm_prepare_kernel<<<(L.Ncp + 7) / 8, 256, 0, st>>>(cohort, 0, Nc, L.Ncp, D, L.Dp, Ch, Cl);
  for (int64_t r0 = 0; r0 < n; r0 += L.rows) {
    const int rows = (int)(n - r0 < L.rows ? n - r0 : L.rows);
    asnorm_prepare_kernel<<<(rows + 7) / 8, 256, 0, st>>>(X, r0, rows, rows, D, L.Dp, Xh, Xl);
    int e = cohort_gemm(Xh, Xl, rows, Ch, Cl, L.Ncp, L.Dp, slab, st);
    if (e) return e;
    e = launch_stats(slab, rows, Nc, L.Ncp, K, out + r0 * 3, st);
    if (e) return e;
  }
  return SVB_OK;
}

extern "C" int svb_cohort_stats_scores(const float* scores, int64_t n, int Nc, int64_t ld, int K, double* out,
                                       void* stream) {
  if (!scores || !out || n < 1 || n >= (int64_t(1) << 31) || Nc < 2 || Nc > kMaxCohort || ld < Nc || K < 2 || K > Nc) {
    svb::set_error("svb_cohort_stats_scores: bad argument (1 <= n < 2^31, 2 <= K <= Nc <= 2^20, ld >= Nc)",
                   cudaSuccess);
    return SVB_ERR_ARG;
  }
  return launch_stats(scores, n, Nc, ld, K, out, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int svb_score_trials(const float* E, int64_t ne, const float* T, int64_t nt, int D, const int32_t* ei,
                                const int32_t* ti, int64_t n_trials, const double* stats_e, const double* stats_t,
                                float* out, void* stream) {
  if (!E || !T || !ei || !ti || !out || ne < 1 || nt < 1 || D < 1 || n_trials < 0 || (!stats_e != !stats_t)) {
    svb::set_error("svb_score_trials: bad argument (ne, nt, D >= 1; stats_e and stats_t both given or both NULL)",
                   cudaSuccess);
    return SVB_ERR_ARG;
  }
  if (n_trials == 0) return SVB_OK;
  const int vec = D % 4 == 0 && (reinterpret_cast<uintptr_t>(E) & 15) == 0 && (reinterpret_cast<uintptr_t>(T) & 15) == 0;
  const int64_t blocks = (n_trials + 7) / 8;
  if (blocks >= (int64_t(1) << 31)) { svb::set_error("svb_score_trials: too many trials", cudaSuccess); return SVB_ERR_ARG; }
  asnorm_trials_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      E, ne, T, nt, D, ei, ti, n_trials, stats_e, stats_t, out, vec);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { svb::set_error("svb_score_trials: launch", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

extern "C" int svb_asnorm_sim(const float* sim, int N, int Mv, const double* stats_c, const double* stats_v, float* out,
                              void* stream) {
  if (!sim || !stats_c || !stats_v || !out || N < 1 || Mv < 1) {
    svb::set_error("svb_asnorm_sim: bad argument (N, Mv >= 1, statistics of both sides)", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const int64_t rows = (int64_t)N * Mv;
  if (rows >= (int64_t(1) << 31)) { svb::set_error("svb_asnorm_sim: N * Mv must be below 2^31", cudaSuccess); return SVB_ERR_ARG; }
  const int grid = (int)(rows < 16 * (int64_t)svb::device_sm_count() ? rows : 16 * (int64_t)svb::device_sm_count());
  asnorm_sim_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sim, N, (int)rows, stats_c, stats_v, out);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { svb::set_error("svb_asnorm_sim: launch", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}
