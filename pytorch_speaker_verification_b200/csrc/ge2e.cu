// Fused GE2E loss forward + backward (fp32) for sm_100a.
//
// Replaces utils.py:27-29 (get_centroids), :40-58 (get_utterance_centroids), :72-115 (get_cossim),
// :126-132 (calc_loss), speech_embedder_net.py:43-49 (GE2ELoss.forward) and the autograd graph behind
// loss.backward() (train_speech_embedder.py:62) of the reference.  Closed form: SURVEY.md section 7.3,
// restated in oracle/ge2e.py::ge2e_fwd_bwd.
//
// One cooperative kernel, four phases separated by grid barriers; nothing of size N*M*N*D is ever
// materialised (the reference's repeat() expansions, utils.py:99-104, are 2 x 41.9 MB at N=64, M=10):
//   A  per speaker : utterance sum s_j, unit centroid c^_j, per-row 1/|e|, 1/|u| and leave-one-out cosine
//   B  per speaker : cos[j,i,:] = e^_ji . c^_k (diag replaced), S = w cos + b, stable log-sum-exp, G, A = wG;
//                    row-local part of dE (sum_k A_off c^_k, diagonal term)
//   C  per (8 centroids x 32 dims): dC_k = (sum_rows A_off e^ - q_k c^_k)/|c_k|
//   D  per speaker : dE += dC_j/M + leave-one-out chain; block 0 reduces loss, dw, db deterministically
// Reductions are warp shuffles + fixed-order shared-memory trees (no float atomics -> run-to-run identical).
#include <cuda_fp16.h>
#include "tc_gemm.cuh"
#include "epilogues.cuh"
#include "../../include/svb200.h"
#include "perdev.cuh"
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace svb {
void set_error(const char* what, cudaError_t e);
int make_operand_map(CUtensorMap* out, const void* p, int rows, int K, int64_t ld, int mn_major, int box_rows_kmajor);

constexpr float kCosEps = 1e-8f;    // F.cosine_similarity eps (utils.py:91,105)
constexpr float kCosBias = 1e-6f;   // utils.py:114
constexpr float kLogBias = 1e-6f;   // utils.py:129
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kSoftmax = SVB_GE2E_SOFTMAX;    // loss method of the row phase (template argument of the loss kernels)
constexpr int kContrast = SVB_GE2E_CONTRAST;

struct Ge2eArgs {
  const float* E;        // [N, M, D]
  const float* Cext;     // [Nc, D] foreign centroids or null (then Nc == N, centroids of E)
  const float* w;        // device scalars; null -> cosine only
  const float* b;
  const float* dcos;     // upstream gradient of the cosine matrix [N, M, Nc] (get_cossim backward) or null
  const float* gscale;   // device scalar multiplying all gradients (upstream dL) or null (= 1)
  int N, M, D, Nc;
  int col0;              // column of the centroid matrix that belongs to speaker 0 of E (row shard of a global batch)
  int need_grad;
  int psplit, prows;     // P = A_off^T E^ is accumulated over psplit slices of prows embedding rows
  // outputs (nullable)
  float* cos_out;        // [N, M, Nc]  cos + 1e-6
  float* per_out;        // [N, M]
  float* loss_out;       // scalar
  float* dE;             // [N, M, D]
  float* dCext;          // [Nc, D] gradient w.r.t. foreign centroids
  float* dw;
  float* db;
  // workspace
  float* Ehat;           // [N*M, D]
  float* Chat;           // [Nc, D]
  float* Ssum;           // [N, D]
  float* inv_ne;         // [N*M]
  float* inv_nu;         // [N*M]
  float* cosd;           // [N*M] leave-one-out cosine (no bias)
  float* inv_nc;         // [Nc]
  float* cosm;           // [N*M, Nc] cosine without bias, diagonal replaced
  float* Aoff;           // [N*M, Nc] upstream dL/dcos with the diagonal zeroed
  float* adiag;          // [N*M]
  float* rowstat;        // [3, N*M]: per-row loss, dw, db contributions
  float* dC;             // [Nc, D]  P = A_off^T E^ (numerator of the centroid gradient)
  float* R;              // [N*M, D] A_off C^
  // tensor-core path (large batches): fp16 hi / lo splits of E^, C^ and A_off (x = hi + lo to 22 bits), or null
  __half *Eh, *El;       // [N*M, D]
  __half *Ch, *Cl;       // [Nc, D]
  __half *Ah, *Al;       // [N*M, Nc]
  long long* trace;      // debug (SVB_GE2E_TRACE=1): [N, 16] clock64 stamps of the per-speaker kernel, else null
  unsigned* bar;         // per-speaker kernel, cluster form: the word of its own grid barrier
};

// x = hi + lo with two IEEE halves: 22 significant bits (|x| <= 65504; lo underflows below 6e-8 absolute)
__device__ __forceinline__ void split_h2(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Arg-max over (value, index) pairs across the warp: the larger value wins, equal values keep the lower index (the
// element torch.max returns); k < 0 marks a lane without a candidate.  Every lane ends with the same pair.
__device__ __forceinline__ void warp_argmax(float& v, int& k) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int ok = __shfl_xor_sync(0xffffffffu, k, o);
    if (ok >= 0 && (k < 0 || ov > v || (ov == v && ok < k))) { v = ov; k = ok; }
  }
}
__device__ __forceinline__ float sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }
// GE2E contrast loss of one row (Wan et al. eq. 7): per = 1 - sig(S_jj) + sig(S_jk*), k* = argmax_{k != j} S_jk.
// G_jj = -sig(S_jj) sig(-S_jj), G_jk* = sig(S_jk*) sig(-S_jk*), every other G is 0 (1 - sig(x) is evaluated as sig(-x)).
struct ContrastRow {
  float per, gd, gk;
};
__device__ __forceinline__ ContrastRow contrast_row(float sd, float sk) {
  const float pd = sigmoid(sd), nd = sigmoid(-sd), pk = sigmoid(sk), nk = sigmoid(-sk);
  return ContrastRow{nd + pk, -pd * nd, pk * nk};
}
// The contrast loss keeps one non-zero of A_off per row: its column k* and value w G_jk* live in the (otherwise unused)
// dense A_off slot of the workspace: [NM] ints, then [NM] floats.
__device__ __forceinline__ int* contrast_kstar(const Ge2eArgs& a) { return reinterpret_cast<int*>(a.Aoff); }
__device__ __forceinline__ float* contrast_gstar(const Ge2eArgs& a) { return a.Aoff + (size_t)a.N * a.M; }

// Block-wide sum, result broadcast to every thread.  red must hold kWarps floats.
__device__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < kWarps; ++i) t += red[i];
  return t;
}

// ---------------------------------------------------------------------------------------------- phase A
__device__ void phase_a(const Ge2eArgs& a, float* smem) {
  float* s = smem;                       // [D]
  float* red = smem + a.D;               // [kWarps]
  float* rows = red + kWarps;            // [M, D] the speaker's embeddings (one coalesced batch of loads)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int M = a.M, D = a.D;
  const float invM = 1.0f / (float)M;
  const float invM1 = 1.0f / (float)(M - 1);
  for (int j = blockIdx.x; j < a.N; j += gridDim.x) {
    const float* Ej = a.E + (size_t)j * M * D;
    for (int i = threadIdx.x; i < M * D; i += kThreads) rows[i] = Ej[i];
    __syncthreads();
    float cc = 0.f;
    for (int d = threadIdx.x; d < D; d += kThreads) {
      float acc = 0.f;
      for (int m = 0; m < M; ++m) acc += rows[m * D + d];
      s[d] = acc;
      a.Ssum[(size_t)j * D + d] = acc;
      const float c = acc * invM;
      cc += c * c;
    }
    if (!a.Cext) {
      cc = block_sum(cc, red);
      const float inc = 1.0f / fmaxf(sqrtf(cc), kCosEps);
      for (int d = threadIdx.x; d < D; d += kThreads) {
        const float c = s[d] * invM * inc;
        a.Chat[(size_t)j * D + d] = c;
        if (a.Ch) split_h2(c, a.Ch[(size_t)j * D + d], a.Cl[(size_t)j * D + d]);
      }
      if (threadIdx.x == 0) a.inv_nc[j] = inc;
    }
    __syncthreads();
    for (int m = warp; m < M; m += kWarps) {
      const float* e = rows + m * D;
      float ee = 0.f, uu = 0.f, eu = 0.f;
      for (int d = lane; d < D; d += 32) {
        const float x = e[d];
        const float u = (s[d] - x) * invM1;
        ee += x * x; uu += u * u; eu += x * u;
      }
      ee = warp_sum(ee); uu = warp_sum(uu); eu = warp_sum(eu);
      const float ine = 1.0f / fmaxf(sqrtf(ee), kCosEps);
      const float inu = 1.0f / fmaxf(sqrtf(uu), kCosEps);
      const size_t row = (size_t)j * M + m;
      for (int d = lane; d < D; d += 32) {
        const float x = e[d] * ine;
        a.Ehat[row * D + d] = x;
        if (a.Eh) split_h2(x, a.Eh[row * D + d], a.El[row * D + d]);
      }
      if (lane == 0) {
        a.inv_ne[row] = ine;
        a.inv_nu[row] = inu;
        a.cosd[row] = eu * ine * inu;
      }
    }
    __syncthreads();
  }
  if (a.Cext) {   // foreign centroids (EER: train_speech_embedder.py:127-129): normalise them once
    for (int k = blockIdx.x * kWarps + warp; k < a.Nc; k += gridDim.x * kWarps) {
      const float* c = a.Cext + (size_t)k * a.D;
      float cc = 0.f;
      for (int d = lane; d < a.D; d += 32) cc += c[d] * c[d];
      cc = warp_sum(cc);
      const float inc = 1.0f / fmaxf(sqrtf(cc), kCosEps);
      for (int d = lane; d < a.D; d += 32) {
        const float x = c[d] * inc;
        a.Chat[(size_t)k * a.D + d] = x;
        if (a.Ch) split_h2(x, a.Ch[(size_t)k * a.D + d], a.Cl[(size_t)k * a.D + d]);
      }
      if (lane == 0) a.inv_nc[k] = inc;
    }
  }
}

// ---------------------------------------------------------------------------------------------- tiled fp32 GEMM
// C[m, n] = sum_k A(m, k) * B(n, k) for one 64 x 64 tile; A(m,k) = A[m*sam + k*sak], B(n,k) = B[n*sbn + k*sbk]
// (one of each stride pair is 1).  256 threads, 4 x 4 register tile each, K staged 16 at a time in shared memory.
constexpr int kTM = 64, kTN = 64, kTK = 32;
constexpr int kLd = kTM * kTK / kThreads;        // elements per thread per operand per K chunk (8)
__device__ __forceinline__ void tile_fetch(const float* __restrict__ P, int64_t sr, int64_t sk, int R, int K, int r0,
                                           int k0, float (&v)[kLd]) {
#pragma unroll
  for (int i = 0; i < kLd; ++i) {
    const int e = threadIdx.x + i * kThreads;
    int r, k;
    if (sk == 1) { k = e % kTK; r = e / kTK; } else { r = e % kTM; k = e / kTM; }
    const int gr = r0 + r, gk = k0 + k;
    v[i] = (gr < R && gk < K) ? P[gr * sr + gk * sk] : 0.f;
  }
}
__device__ __forceinline__ void tile_stash(float (*S)[kTM + 4], int64_t sk, const float (&v)[kLd]) {
#pragma unroll
  for (int i = 0; i < kLd; ++i) {
    const int e = threadIdx.x + i * kThreads;
    int r, k;
    if (sk == 1) { k = e % kTK; r = e / kTK; } else { r = e % kTM; k = e / kTM; }
    S[k][r] = v[i];
  }
}
__device__ void gemm_tile_64(const float* __restrict__ A, int64_t sam, int64_t sak, const float* __restrict__ B,
                             int64_t sbn, int64_t sbk, float* __restrict__ C, int64_t ldc, int M, int N, int K, int m0,
                             int n0, float* smem) {
  float (*As)[kTM + 4] = reinterpret_cast<float (*)[kTM + 4]>(smem);                       // [kTK][kTM+4]
  float (*Bs)[kTN + 4] = reinterpret_cast<float (*)[kTN + 4]>(smem + kTK * (kTM + 4));     // [kTK][kTN+4]
  const int t = threadIdx.x;
  const int ty = t >> 4, tx = t & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float va[kLd], vb[kLd];
  tile_fetch(A, sam, sak, M, K, m0, 0, va);
  tile_fetch(B, sbn, sbk, N, K, n0, 0, vb);
  for (int k0 = 0; k0 < K; k0 += kTK) {
    __syncthreads();                                   // previous chunk fully consumed
    tile_stash(As, sak, va);
    tile_stash(Bs, sbk, vb);
    __syncthreads();
    if (k0 + kTK < K) {                                // next chunk's loads fly while this one is multiplied
      tile_fetch(A, sam, sak, M, K, m0, k0 + kTK, va);
      tile_fetch(B, sbn, sbk, N, K, n0, k0 + kTK, vb);
    }
#pragma unroll
    for (int k = 0; k < kTK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][4 * ty]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][4 * tx]);
      const float a4[4] = {av.x, av.y, av.z, av.w}, b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + 4 * ty + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + 4 * tx + j;
      if (gn < N) C[gm * ldc + gn] = acc[i][j];
    }
  }
}

// ---------------------------------------------------------------------------------------------- phase B1: cosine GEMM
__device__ void phase_b1(const Ge2eArgs& a, float* smem) {
  const int NM = a.N * a.M;
  const int mt = (NM + kTM - 1) / kTM, nt = (a.Nc + kTN - 1) / kTN;
  for (int tix = blockIdx.x; tix < mt * nt; tix += gridDim.x)
    gemm_tile_64(a.Ehat, a.D, 1, a.Chat, a.D, 1, a.cosm, a.Nc, NM, a.Nc, a.D, (tix / nt) * kTM, (tix % nt) * kTN, smem);
}

// ---------------------------------------------------------------------------------------------- phase B2: row softmax
// one warp per embedding row: diagonal overwrite, S = w cos + b, stable log-sum-exp, G, A = w G (diag split off).
// LOSS = kContrast: arg-max k* over the off-diagonal S instead, G has two non-zeros; no dense A_off is written, only
// (k*, w G_jk*) per row for the gather backward of phase D.
template <int LOSS>
__device__ void phase_b2(const Ge2eArgs& a) {
  const int M = a.M, Nc = a.Nc, NM = a.N * a.M;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float w = a.w ? *a.w : 0.f, b = a.b ? *a.b : 0.f;
  for (int row = blockIdx.x * kWarps + warp; row < NM; row += gridDim.x * kWarps) {
    const int j = row / M + a.col0;                     // this row's own column ("diagonal")
    float* t = a.cosm + (size_t)row * Nc;
    const float cd = a.cosd[row];
    if (lane == 0 && j < Nc) t[j] = cd;                 // diagonal overwrite (utils.py:113)
    __syncwarp();
    if (a.cos_out)
      for (int k = lane; k < Nc; k += 32) a.cos_out[(size_t)row * Nc + k] = t[k] + kCosBias;
    if (LOSS == kContrast) {                            // (loss mode only: the host requires w, b)
      float sk = -INFINITY;
      int ks = -1;
      for (int k = lane; k < Nc; k += 32) {
        if (k == j) continue;
        const float s = w * (t[k] + kCosBias) + b;
        if (ks < 0 || s > sk) { sk = s; ks = k; }
      }
      warp_argmax(sk, ks);
      if (lane == 0) {
        const float cd1 = cd + kCosBias, ck1 = t[ks] + kCosBias;
        const ContrastRow c = contrast_row(w * cd1 + b, sk);
        a.rowstat[row] = c.per;
        a.rowstat[NM + row] = c.gd * cd1 + c.gk * ck1;
        a.rowstat[2 * NM + row] = c.gd + c.gk;
        if (a.per_out) a.per_out[row] = c.per;
        a.adiag[row] = w * c.gd;
        contrast_kstar(a)[row] = ks;
        contrast_gstar(a)[row] = w * c.gk;
      }
    } else if (a.w) {
      float mx = -INFINITY;
      for (int k = lane; k < Nc; k += 32) mx = fmaxf(mx, w * (t[k] + kCosBias) + b);
      mx = warp_max(mx);
      float se = 0.f;
      for (int k = lane; k < Nc; k += 32) se += expf(w * (t[k] + kCosBias) + b - mx);
      se = warp_sum(se);
      // log(sum exp S + 1e-6) = mx + log(se + 1e-6 e^{-mx})  (reference has no max-subtraction: same value)
      const float tiny = kLogBias * expf(-mx);
      const float den = se + tiny;
      const float per = -(w * (cd + kCosBias) + b) + mx + logf(den);
      const float inv_den = 1.0f / den;
      float dwp = 0.f, ad = 0.f;
      for (int k = lane; k < Nc; k += 32) {
        const float c0 = t[k];
        float g = expf(w * (c0 + kCosBias) + b - mx) * inv_den;
        if (k == j) g -= 1.0f;
        dwp += g * (c0 + kCosBias);
        const float A = w * g;
        if (k == j) ad = A;
        const float ao = (k == j) ? 0.f : A;
        if (a.Ah) split_h2(ao, a.Ah[(size_t)row * Nc + k], a.Al[(size_t)row * Nc + k]);
        else a.Aoff[(size_t)row * Nc + k] = ao;
      }
      dwp = warp_sum(dwp); ad = warp_sum(ad);
      if (lane == 0) {
        a.rowstat[row] = per;
        a.rowstat[NM + row] = dwp;
        a.rowstat[2 * NM + row] = -tiny * inv_den;     // sum_k G = -1e-6/den exactly
        if (a.per_out) a.per_out[row] = per;
        a.adiag[row] = ad;
      }
    } else if (a.dcos) {   // get_cossim backward: upstream gradient given
      float ad = 0.f;
      for (int k = lane; k < Nc; k += 32) {
        const float A = a.dcos[(size_t)row * Nc + k];
        if (k == j) ad = A;
        a.Aoff[(size_t)row * Nc + k] = (k == j) ? 0.f : A;
      }
      ad = warp_sum(ad);
      if (lane == 0) a.adiag[row] = ad;
    }
  }
}

// ---------------------------------------------------------------------------------------------- phase C: two GEMMs
// R[row, d] = sum_k A_off[row, k] c^_k[d]   and   P[k, d] = sum_row A_off[row, k] e^_row[d]
__device__ void phase_c(const Ge2eArgs& a, float* smem) {
  const int NM = a.N * a.M, D = a.D, Nc = a.Nc;
  const int dt = (D + kTN - 1) / kTN;
  const int rt = ((NM + kTM - 1) / kTM) * dt;
  const int pk = (Nc + kTM - 1) / kTM;
  const int pt = a.psplit * pk * dt;                    // P is reduced over `psplit` slices of `prows` rows each
  for (int tix = blockIdx.x; tix < rt + pt; tix += gridDim.x) {
    if (tix < pt) {
      const int sl = tix / (pk * dt), u = tix % (pk * dt);
      const int r0 = sl * a.prows;
      const int rows = NM - r0 < a.prows ? NM - r0 : a.prows;
      gemm_tile_64(a.Aoff + (size_t)r0 * Nc, 1, Nc, a.Ehat + (size_t)r0 * D, 1, D, a.dC + (size_t)sl * Nc * D, D, Nc, D,
                   rows, (u / dt) * kTM, (u % dt) * kTN, smem);
    } else {
      const int u = tix - pt;
      gemm_tile_64(a.Aoff, Nc, 1, a.Chat, 1, D, a.R, D, NM, D, Nc, (u / dt) * kTM, (u % dt) * kTN, smem);
    }
  }
}

// ---------------------------------------------------------------------------------------------- phase D
// per speaker j: dC_j = (P_j - (P_j.c^_j) c^_j)/|c_j|;  per row: r = R.e^ (= sum_k A_off cos, since cos = e^.c^);
// dE = (R - r e^)/|e| + a (u^ - cosd e^)/|e| + dC_j/M + (sum_m dU_m - dU_i)/(M-1)
// fixed order (deterministic); the loads of four slices are in flight together (one dependent L2 round trip per slice
// made phase D the longest kernel of the tensor-core path: 16 slices x ~0.6 us)
__device__ float sum_slices(const float* p, size_t stride, int n) {
  float v = 0.f;
  int i = 0;
  for (; i + 4 <= n; i += 4) {
    const float x0 = p[(size_t)i * stride], x1 = p[(size_t)(i + 1) * stride], x2 = p[(size_t)(i + 2) * stride],
                x3 = p[(size_t)(i + 3) * stride];
    v += x0; v += x1; v += x2; v += x3;
  }
  for (; i < n; ++i) v += p[(size_t)i * stride];
  return v;
}
// Contrast loss, gather form of P_k = sum_rows A_off[row, k] e^_row: P[d] += sum of w G_jk* e^_row[d] over the rows whose
// k* is k, added in row order (one pass over k*; the matching rows of each 256-row chunk are compacted in order into
// lst / lg, then every thread adds them to its own dimensions).  Called by the whole block.
__device__ void contrast_gather_p(const Ge2eArgs& a, int k, float* P, int* lst, float* lg, int* wcnt) {
  const int NM = a.N * a.M, D = a.D;
  const int* ks = contrast_kstar(a);
  const float* gst = contrast_gstar(a);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r0 = 0; r0 < NM; r0 += kThreads) {
    const int r = r0 + threadIdx.x;
    const bool hit = r < NM && ks[r] == k;
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    __syncthreads();                                   // the previous chunk's list is consumed
    if (lane == 0) wcnt[warp] = __popc(bal);
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < kWarps; ++i) {
      base += i < warp ? wcnt[i] : 0;
      tot += wcnt[i];
    }
    if (tot == 0) continue;
    if (hit) {
      const int p = base + __popc(bal & ((1u << lane) - 1u));
      lst[p] = r;
      lg[p] = gst[r];
    }
    __syncthreads();
    for (int d = threadIdx.x; d < D; d += kThreads) {
      float v = P[d];
      for (int i = 0; i < tot; ++i) v += lg[i] * a.Ehat[(size_t)lst[i] * D + d];
      P[d] = v;
    }
  }
}
// LOSS = kContrast: R_row = w G_jk* c^_k* and P_j from contrast_gather_p (no phase C products)
template <int LOSS>
__device__ void phase_d(const Ge2eArgs& a, float* smem) {
  const int M = a.M, D = a.D, NM = a.N * a.M;
  float* red = smem;                 // [kWarps]
  float* rr = red + kWarps;          // [M]
  float* sc = rr + M;                // [4, M] inv_ne, inv_nu, cosd, adiag
  float* vec = sc + 4 * M;           // [3, D] P_j, c^_j, s_j
  float* rE = vec + 3 * D;           // [M, D] e
  float* rH = rE + (size_t)M * D;    // [M, D] e^
  float* rR = rH + (size_t)M * D;    // [M, D] R
  float* lg = rR + (size_t)M * D;    // contrast: [kThreads] w G_jk* of the compacted rows
  int* lst = reinterpret_cast<int*>(lg + kThreads);   // contrast: [kThreads] their row indices, then [kWarps] counts
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float gs = a.gscale ? *a.gscale : 1.0f;
  if (a.need_grad) {
    const float invM = 1.0f / (float)M, invM1 = 1.0f / (float)(M - 1);
    const size_t pstride = (size_t)a.Nc * D;
    for (int j = blockIdx.x; j < a.N; j += gridDim.x) {
      const size_t row0 = (size_t)j * M;
      // one coalesced batch of independent loads per speaker, everything else from shared memory
      for (int i = threadIdx.x; i < M * D; i += kThreads) {
        rE[i] = a.E[row0 * D + i];
        rH[i] = a.Ehat[row0 * D + i];
        if (LOSS == kContrast) {
          const size_t row = row0 + i / D;
          rR[i] = contrast_gstar(a)[row] * a.Chat[(size_t)contrast_kstar(a)[row] * D + i % D];
        } else {
          rR[i] = a.R[row0 * D + i];
        }
      }
      for (int d = threadIdx.x; d < D; d += kThreads) {
        if (LOSS == kContrast) vec[d] = 0.f;
        else vec[d] = a.Cext ? 0.f : sum_slices(a.dC + (size_t)j * D + d, pstride, a.psplit);
        vec[D + d] = a.Cext ? 0.f : a.Chat[(size_t)j * D + d];
        vec[2 * D + d] = a.Ssum[(size_t)j * D + d];
      }
      for (int m = threadIdx.x; m < M; m += kThreads) {
        sc[m] = a.inv_ne[row0 + m]; sc[M + m] = a.inv_nu[row0 + m];
        sc[2 * M + m] = a.cosd[row0 + m]; sc[3 * M + m] = a.adiag[row0 + m];
      }
      if (LOSS == kContrast && !a.Cext) contrast_gather_p(a, j, vec, lst, lg, lst + kThreads);
      __syncthreads();
      float q = 0.f;
      for (int d = threadIdx.x; d < D; d += kThreads) q += vec[d] * vec[D + d];
      q = block_sum(q, red);
      for (int m = warp; m < M; m += kWarps) {
        float r = 0.f;
        for (int d = lane; d < D; d += 32) r += rR[m * D + d] * rH[m * D + d];
        r = warp_sum(r);
        if (lane == 0) rr[m] = r;
      }
      __syncthreads();
      const float incj = a.Cext ? 0.f : a.inv_nc[j];
      for (int d = threadIdx.x; d < D; d += kThreads) {
        const float sj = vec[2 * D + d];
        float sumdu = 0.f;
        for (int m = 0; m < M; ++m) {
          const float eh = rH[m * D + d], inu = sc[M + m];
          const float uh = (sj - rE[m * D + d]) * invM1 * inu;
          sumdu += sc[3 * M + m] * (eh - sc[2 * M + m] * uh) * inu;
        }
        const float dc = (vec[d] - q * vec[D + d]) * incj * invM;
        for (int m = 0; m < M; ++m) {
          const float eh = rH[m * D + d];
          const float ine = sc[m], inu = sc[M + m], cd = sc[2 * M + m], ad = sc[3 * M + m];
          const float uh = (sj - rE[m * D + d]) * invM1 * inu;
          const float du = ad * (eh - cd * uh) * inu;
          const float local = (rR[m * D + d] - rr[m] * eh) * ine + ad * (uh - cd * eh) * ine;
          a.dE[(row0 + m) * D + d] = gs * (local + dc + (sumdu - du) * invM1);
        }
      }
      __syncthreads();
    }
    if (LOSS == kContrast && a.Cext && a.dCext) {   // the same for the contrast loss, one block per k
      for (int k = blockIdx.x; k < a.Nc; k += gridDim.x) {
        __syncthreads();                                   // vec is free
        for (int d = threadIdx.x; d < D; d += kThreads) vec[d] = 0.f;
        contrast_gather_p(a, k, vec, lst, lg, lst + kThreads);
        __syncthreads();
        float q = 0.f;
        for (int d = threadIdx.x; d < D; d += kThreads) q += vec[d] * a.Chat[(size_t)k * D + d];
        q = block_sum(q, red);
        for (int d = threadIdx.x; d < D; d += kThreads)
          a.dCext[(size_t)k * D + d] = gs * (vec[d] - q * a.Chat[(size_t)k * D + d]) * a.inv_nc[k];
      }
    } else if (a.Cext && a.dCext) {    // gradient w.r.t. foreign centroids: (P_k - (P_k.c^_k) c^_k)/|c_k|, one warp per k
      for (int k = blockIdx.x * kWarps + warp; k < a.Nc; k += gridDim.x * kWarps) {
        float q = 0.f;
        const size_t pstr = (size_t)a.Nc * D;
        for (int d = lane; d < D; d += 32) q += sum_slices(a.dC + (size_t)k * D + d, pstr, a.psplit) * a.Chat[(size_t)k * D + d];
        q = warp_sum(q);
        for (int d = lane; d < D; d += 32)
          a.dCext[(size_t)k * D + d] = gs * (sum_slices(a.dC + (size_t)k * D + d, pstr, a.psplit) - q * a.Chat[(size_t)k * D + d]) * a.inv_nc[k];
      }
    }
  }
  if (blockIdx.x == 0 && a.w) {
    float l = 0.f, dw = 0.f, db = 0.f;
    for (int r = threadIdx.x; r < NM; r += kThreads) {
      l += a.rowstat[r]; dw += a.rowstat[NM + r]; db += a.rowstat[2 * NM + r];
    }
    l = block_sum(l, red); dw = block_sum(dw, red); db = block_sum(db, red);
    if (threadIdx.x == 0) {
      if (a.loss_out) *a.loss_out = l;
      if (a.dw) *a.dw = gs * dw;
      if (a.db) *a.db = gs * db;
    }
  }
}

__global__ void __launch_bounds__(kThreads) ge2e_fused_kernel(const Ge2eArgs a) {
  extern __shared__ float smem[];
  cg::grid_group grid = cg::this_grid();
  phase_a(a, smem);
  grid.sync();
  phase_b1(a, smem);
  grid.sync();
  phase_b2<kSoftmax>(a);
  if (a.need_grad) {
    grid.sync();
    phase_c(a, smem);
  }
  grid.sync();
  phase_d<kSoftmax>(a, smem);
}
// Contrast loss: phase C (the two dense products R = A_off C^, P = A_off^T E^) is replaced by the gathers of phase D.
__global__ void __launch_bounds__(kThreads) ge2e_fused_contrast_kernel(const Ge2eArgs a) {
  extern __shared__ float smem[];
  cg::grid_group grid = cg::this_grid();
  phase_a(a, smem);
  grid.sync();
  phase_b1(a, smem);
  grid.sync();
  phase_b2<kContrast>(a);
  grid.sync();
  phase_d<kContrast>(a, smem);
}
// One kernel per phase (multi-launch forms): each phase gets its own register allocation and occupancy (as one kernel
// with a run-time phase switch every phase ran at the 164 registers of the widest one: one CTA per SM).
template <int PHASE>
__global__ void __launch_bounds__(kThreads) ge2e_phase_kernel(const Ge2eArgs a) {
  extern __shared__ float smem[];
  if (PHASE == 0) phase_a(a, smem);
  else if (PHASE == 1) phase_b1(a, smem);
  else if (PHASE == 2) phase_b2<kSoftmax>(a);
  else if (PHASE == 3) phase_c(a, smem);
  else phase_d<kSoftmax>(a, smem);
}
// Contrast loss: its row phase (PHASE 2) and phase D (PHASE 4); phases A and B1 are the kernels above.
template <int PHASE>
__global__ void __launch_bounds__(kThreads) ge2e_phase_contrast_kernel(const Ge2eArgs a) {
  extern __shared__ float smem[];
  if (PHASE == 2) phase_b2<kContrast>(a);
  else phase_d<kContrast>(a, smem);
}

// ---------------------------------------------------------------------------------------------- small-batch kernel
// One CTA (CL = 1) or one 2-CTA cluster (CL = 2, each CTA owning half of the D embedding dimensions) per speaker,
// three phases, two grid barriers.  The training batch of the reference (N = 64 x M = 10) is far too small for five
// phases of tiled GEMMs: the general kernel above spends its time in barriers and L2 round trips.
//   1  speaker j: its M rows -> utterance sum, unit centroid c^_j (published: N x D floats is all the other speakers
//      need), per-row norms, leave-one-out cosine, e^ (kept in shared memory for the whole kernel)
//   2  speaker j: all unit centroids -> shared memory; cos for its M rows, softmax, A = wG; R = A_off C^ stays on
//      chip; its contribution to every centroid's P_k = sum_rows A_off e^ goes to a [j][k][D] slab
//   3  speaker k: P_k = sum_j slab[j][k] (fixed order), dC_k, and dE of its own rows (the rest is still on chip)
// With CL = 2 every full-D dot product (row norms, cos, q, r) is the sum of the two CTAs' partial sums, exchanged
// through distributed shared memory and added in rank order by both, so the two halves see identical scalars.
// Eligibility (svb_ge2e, fused == 1): own centroids, loss mode, M <= 16, D % 4 == 0, CL * N <= #SMs.
constexpr int kST = 512;
constexpr int kSW = kST / 32;
constexpr int kSpkMaxN = 148;
constexpr int kSpkMaxM = 16;

__device__ float block_sum_s(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < kSW; ++i) t += red[i];
  return t;
}

struct SpkLayout {
  int Npad, LDC, KB, DS, KH, U, XB;   // U = floats of the aliased scratch region, XB = floats of one exchange slot
  size_t floats;
};
// DH = embedding dimensions owned by one CTA (D / CL), MP = compute rows (M rounded up to even)
__host__ __device__ inline SpkLayout spk_layout(int N, int DH, int MP) {
  SpkLayout l;
  const int MS = (MP + 3) & ~3;
  l.Npad = (N + 3) & ~3;
  l.LDC = DH + 4;
  l.KB = (N + 31) / 32;
  int ds = kSW / l.KB;
  if (ds < 1) ds = 1;
  if (ds > DH / 4) ds = DH / 4;
  l.DS = ds;
  l.KH = DH >= kST ? 1 : kST / DH;
  const int u1 = l.DS * MP * l.Npad;
  const int u2 = l.KH * MP * DH;
  l.U = u1 > u2 ? u1 : u2;
  l.XB = 3 * MS + 4;
  l.floats = (size_t)l.Npad * l.LDC          // Ch
             + 2 * (size_t)MS * DH           // rE, rH
             + (size_t)l.U                   // cos partials | R partials
             + 3 * (size_t)MS * l.Npad       // cosr, xcos[2]
             + (size_t)l.Npad * MS           // At
             + 2 * (size_t)DH                // s, Pv
             + (size_t)(l.KH * DH)           // Pq
             + 2 * (size_t)l.XB              // xb[2]
             + 5 * (size_t)MS + 32;          // ine, inu, cosd, adiag, rr, red
  return l;
}

// Grid barrier of the cluster form (a plain cluster launch: Nsight Compute refuses cooperative + cluster launches, and
// all CL * N <= #SMs CTAs are co-resident at one CTA per SM).  One word, self-resetting: every CTA adds 1, CTA 0 adds
// 2^31 - (nblocks - 1), so a complete round adds exactly 2^31: the top bit flips and the low bits return to where they
// were.  One release atomic + acquire polls per CTA (separate fences cost ~1000 cycles each with stores in flight);
// the other threads are ordered through the two CTA barriers.  The word is library-owned and zeroed once.
__device__ __forceinline__ void spk_grid_barrier(unsigned* bar, unsigned nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned inc = blockIdx.x == 0 ? 0x80000000u - (nblocks - 1) : 1u;
    unsigned old, v;
    asm volatile("atom.add.release.gpu.global.u32 %0, [%1], %2;" : "=r"(old) : "l"(bar), "r"(inc) : "memory");
    long long t0 = 0;
    while (true) {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
      if ((old ^ v) & 0x80000000u) break;
      if (t0 == 0) t0 = clock64();
      else if (clock64() - t0 > 4000000000LL) { printf("svb: ge2e grid barrier timeout block %d\n", blockIdx.x); __trap(); }
    }
  }
  __syncthreads();
}

// LOSS = kContrast replaces the softmax block of phase 2 by the contrast row block (one non-zero of A_off per row);
// everything else, the on-chip R and the P slab included, is shared.
template <int MP, int CL, int LOSS>
__device__ __forceinline__ void ge2e_speaker_body(const Ge2eArgs& a) {
  constexpr int MS = (MP + 3) & ~3;       // row stride of the [k][m] arrays (float4 loads)
  extern __shared__ float4 smem4[];
  float* smem = reinterpret_cast<float*>(smem4);
  auto grid_sync = [&]() {
    if constexpr (CL > 1) spk_grid_barrier(a.bar, gridDim.x); else cg::this_grid().sync();
  };
  const int N = a.N, M = a.M, D = a.D, NM = N * M;
  const int h = CL > 1 ? (int)(blockIdx.x % CL) : 0;           // rank in the cluster = which slice of D
  const int j = blockIdx.x / CL;
  const int DH = D / CL, d0 = h * DH, DH4 = DH / 4;
  const SpkLayout L = spk_layout(N, DH, MP);
  float* Ch = smem;
  float* rE = Ch + (size_t)L.Npad * L.LDC;
  float* rH = rE + MS * DH;
  float* U = rH + MS * DH;
  float* cosr = U + L.U;
  float* xcos = cosr + MS * L.Npad;       // [2][MS * Npad]
  float* At = xcos + 2 * MS * L.Npad;     // [Npad][MS]
  float* s = At + L.Npad * MS;
  float* Pv = s + DH;
  float* Pq = Pv + DH;
  float* xb = Pq + L.KH * DH;             // [2][XB]
  float* ine = xb + 2 * L.XB;
  float* inu = ine + MS;
  float* cosd = inu + MS;
  float* adiag = cosd + MS;
  float* rr = adiag + MS;
  float* red = rr + MS;
  float* xb_peer = xb;
  float* xcos_peer = xcos;
  if constexpr (CL > 1) {
    cg::cluster_group cluster = cg::this_cluster();
    xb_peer = cluster.map_shared_rank(xb, h ^ 1);
    xcos_peer = cluster.map_shared_rank(xcos, h ^ 1);
  }
  auto exchange_sync = [&]() {
    if constexpr (CL > 1) cg::this_cluster().sync(); else __syncthreads();
  };
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const size_t row0 = (size_t)j * M;
  const float invM = 1.0f / (float)M, invM1 = 1.0f / (float)(M - 1);
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 0] = clock64();

  // ------------------------------------------------------------------ phase 1
  {
    float4* rE4 = reinterpret_cast<float4*>(rE);
    for (int i = tid; i < MP * DH4; i += kST) {
      const int m = i / DH4, d4 = i - m * DH4;
      rE4[i] = (m < M) ? __ldg(reinterpret_cast<const float4*>(a.E + (row0 + m) * D + d0) + d4)
                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int i = tid; i < L.Npad * MS; i += kST) At[i] = 0.f;
  }
  __syncthreads();
  float cc = 0.f;
  for (int d = tid; d < DH; d += kST) {
    float acc = 0.f;
    for (int m = 0; m < M; ++m) acc += rE[m * DH + d];
    s[d] = acc;
    const float c = acc * invM;
    cc += c * c;
  }
  cc = block_sum_s(cc, red);
  if (tid == 0) { xb[h * L.XB + 3 * MS] = cc; if (CL > 1) xb_peer[h * L.XB + 3 * MS] = cc; }
  for (int m = warp; m < M; m += kSW) {
    const float* e = rE + m * DH;
    float ee = 0.f, uu = 0.f, eu = 0.f;
    for (int d = lane; d < DH; d += 32) {
      const float x = e[d];
      const float u = (s[d] - x) * invM1;
      ee += x * x; uu += u * u; eu += x * u;
    }
    ee = warp_sum(ee); uu = warp_sum(uu); eu = warp_sum(eu);
    if (lane == 0) {
      float* o = xb + h * L.XB + 3 * m;
      o[0] = ee; o[1] = uu; o[2] = eu;
      if (CL > 1) { float* p = xb_peer + h * L.XB + 3 * m; p[0] = ee; p[1] = uu; p[2] = eu; }
    }
  }
  exchange_sync();
  cc = xb[3 * MS];
  if (CL > 1) cc += xb[L.XB + 3 * MS];
  const float incj = 1.0f / fmaxf(sqrtf(cc), kCosEps);
  for (int d = tid; d < DH; d += kST) a.Chat[(size_t)j * D + d0 + d] = s[d] * invM * incj;
  for (int m = warp; m < MP; m += kSW) {
    if (m < M) {
      float ee = xb[3 * m], uu = xb[3 * m + 1], eu = xb[3 * m + 2];
      if (CL > 1) { ee += xb[L.XB + 3 * m]; uu += xb[L.XB + 3 * m + 1]; eu += xb[L.XB + 3 * m + 2]; }
      const float i_e = 1.0f / fmaxf(sqrtf(ee), kCosEps);
      const float i_u = 1.0f / fmaxf(sqrtf(uu), kCosEps);
      for (int d = lane; d < DH; d += 32) rH[m * DH + d] = rE[m * DH + d] * i_e;
      if (lane == 0) { ine[m] = i_e; inu[m] = i_u; cosd[m] = eu * i_e * i_u; }
    } else {
      for (int d = lane; d < DH; d += 32) rH[m * DH + d] = 0.f;
      if (lane == 0) { ine[m] = 0.f; inu[m] = 0.f; cosd[m] = 0.f; adiag[m] = 0.f; }
    }
  }
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 1] = clock64();
  grid_sync();
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 2] = clock64();

  // ------------------------------------------------------------------ phase 2
  for (int i = tid; i < L.Npad * DH4; i += kST) {
    const int k = i / DH4, d4 = i - k * DH4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k < N) v = __ldcg(reinterpret_cast<const float4*>(a.Chat + (size_t)k * D + d0) + d4);
    *reinterpret_cast<float4*>(Ch + (size_t)k * L.LDC + 4 * d4) = v;
  }
  __syncthreads();
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 3] = clock64();
  {   // cos partials: lane <-> centroid, warp task <-> (32 centroids, slice of the CTA's dimensions)
    const int chunk = (DH4 + L.DS - 1) / L.DS;
    for (int task = warp; task < L.KB * L.DS; task += kSW) {
      const int kb = task % L.KB, ds = task / L.KB;
      const int k = kb * 32 + lane;
      const int kk = k < L.Npad ? k : L.Npad - 1;
      float acc[MP];
#pragma unroll
      for (int m = 0; m < MP; ++m) acc[m] = 0.f;
      const int d4e = (ds + 1) * chunk < DH4 ? (ds + 1) * chunk : DH4;
      for (int d4 = ds * chunk; d4 < d4e; ++d4) {
        const float4 c = *reinterpret_cast<const float4*>(Ch + (size_t)kk * L.LDC + 4 * d4);
#pragma unroll
        for (int m = 0; m < MP; ++m) {
          const float4 e = *reinterpret_cast<const float4*>(rH + m * DH + 4 * d4);
          acc[m] = fmaf(c.x, e.x, acc[m]); acc[m] = fmaf(c.y, e.y, acc[m]);
          acc[m] = fmaf(c.z, e.z, acc[m]); acc[m] = fmaf(c.w, e.w, acc[m]);
        }
      }
      if (k < L.Npad) {
#pragma unroll
        for (int m = 0; m < MP; ++m) U[(ds * MP + m) * L.Npad + k] = acc[m];
      }
    }
  }
  __syncthreads();
  for (int i = tid; i < MP * L.Npad; i += kST) {
    float v = 0.f;
    for (int ds = 0; ds < L.DS; ++ds) v += U[ds * MP * L.Npad + i];
    if (CL > 1) { xcos[h * MS * L.Npad + i] = v; xcos_peer[h * MS * L.Npad + i] = v; } else cosr[i] = v;
  }
  exchange_sync();
  if (CL > 1) {
    for (int i = tid; i < MP * L.Npad; i += kST) cosr[i] = xcos[i] + xcos[MS * L.Npad + i];
    __syncthreads();
  }
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 4] = clock64();
  if constexpr (LOSS == kContrast) {   // contrast: one warp per row (both CTAs of a cluster see identical cosr -> same k*)
    const float w = *a.w, b = *a.b;
    for (int m = warp; m < M; m += kSW) {
      const float* t = cosr + m * L.Npad;
      float sk = -INFINITY;
      int ks = -1;
      for (int k = lane; k < N; k += 32) {
        if (k == j) continue;
        const float s = w * (t[k] + kCosBias) + b;
        if (ks < 0 || s > sk) { sk = s; ks = k; }
      }
      warp_argmax(sk, ks);
      if (lane == 0) {
        const float cd1 = cosd[m] + kCosBias, ck1 = t[ks] + kCosBias;
        const ContrastRow c = contrast_row(w * cd1 + b, sk);
        if (h == 0) {
          const size_t row = row0 + m;
          a.rowstat[row] = c.per;
          a.rowstat[NM + row] = c.gd * cd1 + c.gk * ck1;
          a.rowstat[2 * NM + row] = c.gd + c.gk;
          if (a.per_out) a.per_out[row] = c.per;
        }
        adiag[m] = w * c.gd;
        At[ks * MS + m] = w * c.gk;                   // At is zero elsewhere (phase 1)
      }
    }
  } else {   // softmax: one warp per row (both CTAs of a cluster, identical inputs -> identical A)
    const float w = *a.w, b = *a.b;
    for (int m = warp; m < M; m += kSW) {
      const float* t = cosr + m * L.Npad;
      const float cd = cosd[m];
      float mx = -INFINITY;
      for (int k = lane; k < N; k += 32) mx = fmaxf(mx, w * ((k == j ? cd : t[k]) + kCosBias) + b);   // utils.py:113
      mx = warp_max(mx);
      float se = 0.f;
      for (int k = lane; k < N; k += 32) se += expf(w * ((k == j ? cd : t[k]) + kCosBias) + b - mx);
      se = warp_sum(se);
      const float tiny = kLogBias * expf(-mx);
      const float den = se + tiny;
      const float per = -(w * (cd + kCosBias) + b) + mx + logf(den);
      const float inv_den = 1.0f / den;
      float dwp = 0.f, ad = 0.f;
      for (int k = lane; k < N; k += 32) {
        const float c0 = (k == j) ? cd : t[k];
        float g = expf(w * (c0 + kCosBias) + b - mx) * inv_den;
        if (k == j) g -= 1.0f;
        dwp += g * (c0 + kCosBias);
        const float A = w * g;
        if (k == j) ad = A;
        At[k * MS + m] = (k == j) ? 0.f : A;
      }
      dwp = warp_sum(dwp); ad = warp_sum(ad);
      if (lane == 0) {
        if (h == 0) {
          const size_t row = row0 + m;
          a.rowstat[row] = per;
          a.rowstat[NM + row] = dwp;
          a.rowstat[2 * NM + row] = -tiny * inv_den;
          if (a.per_out) a.per_out[row] = per;
        }
        adiag[m] = ad;
      }
    }
  }
  __syncthreads();
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 5] = clock64();
  if (a.need_grad) {
    // R[m, d] = sum_k A_off[m, k] c^_k[d] (on chip) and this speaker's slab of P[k, d] = sum_m A_off[m, k] e^_m[d]
    const int kc = (L.Npad + L.KH - 1) / L.KH;
    float* slab = a.dC + (size_t)j * N * D + d0;
    for (int idx = tid; idx < DH * L.KH; idx += kST) {
      const int kh = idx / DH, d = idx - kh * DH;
      const int k0 = kh * kc, k1 = (k0 + kc < L.Npad) ? k0 + kc : L.Npad;
      float eh[MP], acc[MP];
#pragma unroll
      for (int m = 0; m < MP; ++m) { eh[m] = rH[m * DH + d]; acc[m] = 0.f; }
      float* sp = slab + (size_t)k0 * D + d;
      for (int k = k0; k < k1; ++k, sp += D) {
        float at[MS];
#pragma unroll
        for (int m4 = 0; m4 < MS / 4; ++m4) {
          const float4 v = *reinterpret_cast<const float4*>(At + k * MS + 4 * m4);
          at[4 * m4] = v.x; at[4 * m4 + 1] = v.y; at[4 * m4 + 2] = v.z; at[4 * m4 + 3] = v.w;
        }
        const float c = Ch[(size_t)k * L.LDC + d];
        float p0 = 0.f, p1 = 0.f;
#pragma unroll
        for (int m = 0; m < MP; m += 2) {
          acc[m] = fmaf(at[m], c, acc[m]); acc[m + 1] = fmaf(at[m + 1], c, acc[m + 1]);
          p0 = fmaf(at[m], eh[m], p0); p1 = fmaf(at[m + 1], eh[m + 1], p1);
        }
        if (k < N) __stcg(sp, p0 + p1);
      }
#pragma unroll
      for (int m = 0; m < MP; ++m) U[(kh * MP + m) * DH + d] = acc[m];
    }
    __syncthreads();
    for (int i = tid; i < MP * DH; i += kST) {
      float v = U[i];
      for (int kh = 1; kh < L.KH; ++kh) v += U[kh * MP * DH + i];
      U[i] = v;                                     // rR = U[0 .. MP*DH)
    }
  }
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 6] = clock64();
  grid_sync();
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 7] = clock64();

  // ------------------------------------------------------------------ phase 3
  if (a.need_grad) {
    const float* rR = U;
    const float gs = a.gscale ? *a.gscale : 1.0f;
    const int jc = (N + L.KH - 1) / L.KH;
    for (int idx = tid; idx < DH * L.KH; idx += kST) {
      const int jh = idx / DH, d = idx - jh * DH;
      const int j0 = jh * jc, j1 = (j0 + jc < N) ? j0 + jc : N;
      const float* p = a.dC + ((size_t)j0 * N + j) * D + d0 + d;
      const size_t st = (size_t)N * D;
      float v = 0.f;
      int jj = j0;
      for (; jj + 8 <= j1; jj += 8) {
        float t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = __ldcg(p + (size_t)u * st);
#pragma unroll
        for (int u = 0; u < 8; ++u) v += t[u];
        p += 8 * st;
      }
      for (; jj < j1; ++jj) { v += __ldcg(p); p += st; }
      Pq[jh * DH + d] = v;
    }
    __syncthreads();
    if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 8] = clock64();
    float q = 0.f;
    for (int d = tid; d < DH; d += kST) {
      float v = Pq[d];
      for (int jh = 1; jh < L.KH; ++jh) v += Pq[jh * DH + d];
      Pv[d] = v;
      q += v * Ch[(size_t)j * L.LDC + d];
    }
    q = block_sum_s(q, red);
    if (tid == 0) { xb[h * L.XB + 3 * MS] = q; if (CL > 1) xb_peer[h * L.XB + 3 * MS] = q; }
    for (int m = warp; m < M; m += kSW) {
      float r = 0.f;
      for (int d = lane; d < DH; d += 32) r += rR[m * DH + d] * rH[m * DH + d];
      r = warp_sum(r);
      if (lane == 0) { xb[h * L.XB + m] = r; if (CL > 1) xb_peer[h * L.XB + m] = r; }
    }
    exchange_sync();
    q = xb[3 * MS];
    if (CL > 1) q += xb[L.XB + 3 * MS];
    if (tid < M) rr[tid] = CL > 1 ? xb[tid] + xb[L.XB + tid] : xb[tid];
    __syncthreads();
    for (int idx = tid; idx < DH * L.KH; idx += kST) {
      const int mh = idx / DH, d = idx - mh * DH;
      const float sj = s[d];
      const float chd = Ch[(size_t)j * L.LDC + d];
      float sumdu = 0.f;
      for (int m = 0; m < M; ++m) {
        const float eh = rH[m * DH + d], i_u = inu[m];
        const float uh = (sj - rE[m * DH + d]) * invM1 * i_u;
        sumdu += adiag[m] * (eh - cosd[m] * uh) * i_u;
      }
      const float dc = (Pv[d] - q * chd) * incj * invM;
      for (int m = mh; m < M; m += L.KH) {
        const float eh = rH[m * DH + d];
        const float i_e = ine[m], i_u = inu[m], cd = cosd[m], ad = adiag[m];
        const float uh = (sj - rE[m * DH + d]) * invM1 * i_u;
        const float du = ad * (eh - cd * uh) * i_u;
        const float local = (rR[m * DH + d] - rr[m] * eh) * i_e + ad * (uh - cd * eh) * i_e;
        a.dE[(row0 + m) * D + d0 + d] = gs * (local + dc + (sumdu - du) * invM1);
      }
    }
  }
  if (a.trace && tid == 0) a.trace[blockIdx.x * 16 + 9] = clock64();
  if (blockIdx.x == 0) {
    const float gs = a.gscale ? *a.gscale : 1.0f;
    float l = 0.f, dw = 0.f, db = 0.f;
    for (int r = tid; r < NM; r += kST) {
      l += __ldcg(a.rowstat + r); dw += __ldcg(a.rowstat + NM + r); db += __ldcg(a.rowstat + 2 * NM + r);
    }
    l = block_sum_s(l, red); dw = block_sum_s(dw, red); db = block_sum_s(db, red);
    if (tid == 0) {
      if (a.loss_out) *a.loss_out = l;
      if (a.dw) *a.dw = gs * dw;
      if (a.db) *a.db = gs * db;
    }
  }
}
template <int MP, int CL>
__global__ void __launch_bounds__(kST, 1) ge2e_speaker_kernel(const Ge2eArgs a) {
  ge2e_speaker_body<MP, CL, kSoftmax>(a);
}
template <int MP, int CL>
__global__ void __launch_bounds__(kST, 1) ge2e_speaker_contrast_kernel(const Ge2eArgs a) {
  ge2e_speaker_body<MP, CL, kContrast>(a);
}

static size_t align_up(size_t x) { return (x + 255) & ~size_t(255); }

static bool spk_candidate(int N, int M, int D, int Nc) {
  return Nc == N && M <= kSpkMaxM && D % 4 == 0 && N <= kSpkMaxN;
}
template <int CL>
static void* spk_kernel_cl(int MP) {
  switch (MP) {
    case 2: return (void*)ge2e_speaker_kernel<2, CL>;
    case 4: return (void*)ge2e_speaker_kernel<4, CL>;
    case 6: return (void*)ge2e_speaker_kernel<6, CL>;
    case 8: return (void*)ge2e_speaker_kernel<8, CL>;
    case 10: return (void*)ge2e_speaker_kernel<10, CL>;
    case 12: return (void*)ge2e_speaker_kernel<12, CL>;
    case 14: return (void*)ge2e_speaker_kernel<14, CL>;
    default: return (void*)ge2e_speaker_kernel<16, CL>;
  }
}
template <int CL>
static void* spk_contrast_kernel_cl(int MP) {
  switch (MP) {
    case 2: return (void*)ge2e_speaker_contrast_kernel<2, CL>;
    case 4: return (void*)ge2e_speaker_contrast_kernel<4, CL>;
    case 6: return (void*)ge2e_speaker_contrast_kernel<6, CL>;
    case 8: return (void*)ge2e_speaker_contrast_kernel<8, CL>;
    case 10: return (void*)ge2e_speaker_contrast_kernel<10, CL>;
    case 12: return (void*)ge2e_speaker_contrast_kernel<12, CL>;
    case 14: return (void*)ge2e_speaker_contrast_kernel<14, CL>;
    default: return (void*)ge2e_speaker_contrast_kernel<16, CL>;
  }
}
static void* spk_kernel(int MP, int CL, int loss) {
  if (loss == kContrast) return CL > 1 ? spk_contrast_kernel_cl<2>(MP) : spk_contrast_kernel_cl<1>(MP);
  return CL > 1 ? spk_kernel_cl<2>(MP) : spk_kernel_cl<1>(MP);
}

static size_t carve(Ge2eArgs& a, char* base) {
  const size_t NM = (size_t)a.N * a.M, D = a.D, Nc = a.Nc;
  {   // <= 16 slices, each a multiple of 64 rows
    int rows = (int)((NM + 15) / 16);
    rows = ((rows + 63) / 64) * 64;
    a.prows = rows;
    a.psplit = (int)((NM + rows - 1) / rows);
  }
  size_t off = 0;
  auto take = [&](size_t nfloats) { float* p = base ? reinterpret_cast<float*>(base + off) : nullptr; off += align_up(nfloats * 4); return p; };
  a.Ehat = take(NM * D); a.Chat = take(Nc * D); a.Ssum = take((size_t)a.N * D);
  a.inv_ne = take(NM); a.inv_nu = take(NM); a.cosd = take(NM); a.inv_nc = take(Nc);
  a.cosm = take(NM * Nc); a.Aoff = take(NM * Nc); a.adiag = take(NM); a.rowstat = take(3 * NM); a.dC = take((size_t)(spk_candidate(a.N, a.M, a.D, a.Nc) && a.N > a.psplit ? a.N : a.psplit) * Nc * D); a.R = take(NM * D);
  auto take_h = [&](size_t nhalfs) { return reinterpret_cast<__half*>(take((nhalfs + 1) / 2)); };
  a.Eh = take_h(NM * D); a.El = take_h(NM * D); a.Ch = take_h(Nc * D); a.Cl = take_h(Nc * D);
  a.Ah = take_h(NM * Nc); a.Al = take_h(NM * Nc);
  a.trace = reinterpret_cast<long long*>(take(2 * 16 * (size_t)kSpkMaxN));
  return off;
}

static size_t smem_bytes(const Ge2eArgs& a, int loss = kSoftmax) {
  size_t pa = (size_t)a.D + kWarps + (size_t)a.M * a.D;
  size_t pg = (size_t)kTK * (kTM + 4) + (size_t)kTK * (kTN + 4);
  size_t pd = (size_t)kWarps + 5 * (size_t)a.M + 3 * (size_t)a.D + 3 * (size_t)a.M * a.D;
  if (loss == kContrast) pd += 2 * (size_t)kThreads + kWarps;        // contrast_gather_p's row list and counts
  size_t m = pa > pg ? pa : pg;
  m = m > pd ? m : pd;
  return m * sizeof(float);
}

}  // namespace svb

using namespace svb;

extern "C" int svb_ge2e_workspace_bytes(int N, int M, int D, int Nc, size_t* bytes) {
  if (N < 1 || M < 1 || D < 1 || Nc < 1 || !bytes) return SVB_ERR_ARG;
  Ge2eArgs a{};
  a.N = N; a.M = M; a.D = D; a.Nc = Nc;
  *bytes = carve(a, nullptr);
  return SVB_OK;
}

// Debug: byte offset of the clock64 trace ([N, 16] int64) inside the workspace (written when SVB_GE2E_TRACE is set).
extern "C" int svb_ge2e_trace_offset(int N, int M, int D, int Nc, size_t* offset) {
  if (!offset) return SVB_ERR_ARG;
  Ge2eArgs a{};
  a.N = N; a.M = M; a.D = D; a.Nc = Nc;
  const size_t total = carve(a, nullptr);
  *offset = total - align_up(2 * 16 * (size_t)kSpkMaxN * 4);
  return SVB_OK;
}

// tensor-core path of the large-batch GE2E: 1 (default; env SVB_GE2E_TC=0 clears it) or 0 = fp32 SIMT contractions only
static int g_ge2e_tc = (getenv("SVB_GE2E_TC") != nullptr && atoi(getenv("SVB_GE2E_TC")) == 0) ? 0 : 1;
extern "C" int svb_set_ge2e_tensor_cores(int on) { g_ge2e_tc = on != 0; return SVB_OK; }

static int ge2e_impl(const float* E, const float* Cext, int N, int M, int D, int Nc, int col0, const float* w,
                     const float* b, const float* dcos, const float* gscale, float* cos_out, float* per_out,
                     float* loss_out, float* dE, float* dCext, float* dw, float* db, void* workspace,
                     size_t workspace_bytes, int fused, int loss, void* stream) {
  if (!E || N < 1 || M < 2 || D < 1 || !workspace) { set_error("svb_ge2e: bad argument (M must be >= 2)", cudaSuccess); return SVB_ERR_ARG; }
  if (loss != kSoftmax && loss != kContrast) { set_error("svb_ge2e: unknown loss method", cudaSuccess); return SVB_ERR_ARG; }
  if (loss == kContrast && (!w || dcos)) { set_error("svb_ge2e: the contrast loss method needs w and b (no cosine-only or dcos mode)", cudaSuccess); return SVB_ERR_ARG; }
  if (loss == kContrast && Nc < 2) { set_error("svb_ge2e: the contrast loss needs at least two centroid columns", cudaSuccess); return SVB_ERR_ARG; }
  if (col0 < 0 || (col0 > 0 && (!Cext || col0 + N > Nc))) { set_error("svb_ge2e: row shard outside the centroid matrix", cudaSuccess); return SVB_ERR_ARG; }
  if (!Cext && Nc != N) { set_error("svb_ge2e: Nc must equal N without foreign centroids", cudaSuccess); return SVB_ERR_ARG; }
  if ((w == nullptr) != (b == nullptr)) return SVB_ERR_ARG;
  Ge2eArgs a{};
  a.E = E; a.Cext = Cext; a.w = w; a.b = b; a.dcos = dcos; a.gscale = gscale;
  a.N = N; a.M = M; a.D = D; a.Nc = Nc; a.col0 = col0;
  a.need_grad = (dE != nullptr) ? 1 : 0;
  if (a.need_grad && !w && !dcos) { set_error("svb_ge2e: gradient requested without w/b or dcos", cudaSuccess); return SVB_ERR_ARG; }
  a.cos_out = cos_out; a.per_out = per_out; a.loss_out = loss_out; a.dE = dE; a.dCext = dCext; a.dw = dw; a.db = db;
  if (carve(a, static_cast<char*>(workspace)) > workspace_bytes) { set_error("svb_ge2e: workspace too small", cudaSuccess); return SVB_ERR_ARG; }
  static const bool trace_on = getenv("SVB_GE2E_TRACE") != nullptr;
  if (!trace_on) a.trace = nullptr;
  const size_t smem = smem_bytes(a);
  const size_t smem_ct = smem_bytes(a, loss);           // (== smem for the softmax loss)
  if (smem_ct > 200 * 1024) { set_error("svb_ge2e: M*D too large for one CTA's shared memory", cudaSuccess); return SVB_ERR_UNSUPPORTED; }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  static int max_smem_tab[kMaxDevices] = {};          // cudaFuncSetAttribute is per device
  const int dev_i = current_device_index();
  int& max_smem_set = max_smem_tab[dev_i];
  const int num_sms = device_sm_count();
  if ((int)smem > max_smem_set) {
    cudaError_t e = cudaFuncSetAttribute(ge2e_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_error("svb_ge2e: cudaFuncSetAttribute", e); return SVB_ERR_CUDA; }
    max_smem_set = (int)smem;
  }
  const bool contrast = loss == kContrast;
  static int max_smem_ct_tab[kMaxDevices] = {};       // the contrast kernels' own attribute
  if (contrast && (int)smem_ct > max_smem_ct_tab[dev_i]) {
    cudaError_t e = cudaFuncSetAttribute(ge2e_fused_contrast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ct);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_contrast_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ct);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ge2e_phase_contrast_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ct);
    if (e != cudaSuccess) { set_error("svb_ge2e: cudaFuncSetAttribute (contrast)", e); return SVB_ERR_CUDA; }
    max_smem_ct_tab[dev_i] = (int)smem_ct;
  }
  const int NMr = N * M;
  const int dtl = (D + kTN - 1) / kTN;
  const int b1tiles = ((NMr + kTM - 1) / kTM) * ((Nc + kTN - 1) / kTN);
  const int ctiles = (((NMr + kTM - 1) / kTM) + a.psplit * ((Nc + kTM - 1) / kTM)) * dtl;
  const int b2blocks = (NMr + kWarps - 1) / kWarps;
  int want = N;
  if (b1tiles > want) want = b1tiles;
  if (ctiles > want && a.need_grad && !contrast) want = ctiles;
  if (b2blocks > want) want = b2blocks;
  // contrast phase D with foreign centroids: one block per centroid gathers its P_k
  const int dblocks_ct = (Cext && a.need_grad && Nc > N) ? Nc : N;
  const int dgrid = dblocks_ct < 4 * num_sms ? dblocks_ct : 4 * num_sms;
  if (contrast && dblocks_ct > want) want = dblocks_ct;
  if (fused == 1 && spk_candidate(N, M, D, Nc) && !Cext && w && !dcos && !cos_out && N <= num_sms) {
    // small batch (the reference's training batch): one CTA or one 2-CTA cluster per speaker, three phases
    static int cluster_ok = 1;                       // cleared if the cluster launch is refused
    const int MP = (M + 1) & ~1;
    for (int CL = (cluster_ok && D % 8 == 0 && 2 * N <= num_sms) ? 2 : 1; CL >= 1; --CL) {
      const size_t sm = spk_layout(N, D / CL, MP).floats * sizeof(float);
      if (sm > 220 * 1024) break;
      void* fn = spk_kernel(MP, CL, loss);
      static int spk_smem_tab[kMaxDevices][2][2][kSpkMaxM / 2] = {};
      int (&spk_smem_set)[2][kSpkMaxM / 2] = spk_smem_tab[dev_i][contrast ? 1 : 0];
      if ((int)sm > spk_smem_set[CL - 1][MP / 2 - 1]) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) { set_error("svb_ge2e: cudaFuncSetAttribute (speaker kernel)", e); return SVB_ERR_CUDA; }
        spk_smem_set[CL - 1][MP / 2 - 1] = (int)sm;
      }
      if (CL > 1) {
        // barrier word per (device, stream): launches on one stream are serialised, launches on different streams
        // may overlap and must not share a word (256 B apart: separate L2 lines)
        struct BarSlot { int dev; cudaStream_t st; unsigned* word; };
        static BarSlot slots[32];
        static int nslots = 0;
        static unsigned* pool[64] = {};
        static int used[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64) continue;
        unsigned* word = nullptr;
        for (int i = 0; i < nslots; ++i)
          if (slots[i].dev == dev && slots[i].st == s) word = slots[i].word;
        if (!word) {
          if (!pool[dev]) {
            if (cudaMalloc(&pool[dev], 32 * 256) != cudaSuccess || cudaMemset(pool[dev], 0, 32 * 256) != cudaSuccess) {
              cudaGetLastError(); pool[dev] = nullptr; cluster_ok = 0; continue;
            }
          }
          if (nslots >= 32 || used[dev] >= 32) continue;          // too many streams: single-CTA form
          word = pool[dev] + 64 * used[dev]++;
          slots[nslots++] = BarSlot{dev, s, word};
        }
        a.bar = word;
      }
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3(N * CL); cfg.blockDim = dim3(kST); cfg.dynamicSmemBytes = sm; cfg.stream = s;
      cudaLaunchAttribute at[2];
      cfg.attrs = at; cfg.numAttrs = 1;
      if (CL > 1) {
        // cooperative cluster launch: the kernel's own grid barrier spins on all 2N CTAs, so their co-residency must be
        // guaranteed by the driver (another stream's kernel -- a second GE2E launch, NCCL -- may hold SMs).  Nsight
        // Compute refuses cooperative + cluster launches: profiling runs set SVB_PLAIN_CLUSTER_LAUNCH=1.
        static const bool plain = getenv("SVB_PLAIN_CLUSTER_LAUNCH") != nullptr;
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        at[1].id = cudaLaunchAttributeCooperative; at[1].val.cooperative = 1;
        cfg.numAttrs = plain ? 1 : 2;
      } else {
        at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
      }
      void* params[] = {&a};
      cudaError_t e = cudaLaunchKernelExC(&cfg, fn, params);
      if (e == cudaSuccess) return SVB_OK;
      if (CL == 1) { set_error("svb_ge2e: cooperative launch (speaker kernel)", e); return SVB_ERR_CUDA; }
      cudaGetLastError();                            // cluster form refused: remember, take the single-CTA form
      cluster_ok = 0;
    }
  }
  // ---- tensor-core path for large batches (C3: N = 512, the C5 similarity matrix): the three contractions
  //      cos = E^ C^T, R = A_off C^, P = A_off^T E^ run on tcgen05 as 3-term split-fp16 products
  //      (hi hi + hi lo + lo hi) between the phase kernels.  The SIMT GEMM phases are 95 % of the fused kernel's
  //      205 us at N = 512.  The split itself rounds to ~2^-22, but the products' fp32 accumulation in tensor memory is
  //      biased toward zero by about 7.7e-9 * D times the cosine (measured on a B200: cosines near 1 come out low by
  //      7.9e-7, 1.8e-6, 3.8e-6, 5.9e-6 at D = 128, 256, 512, 768; the SIMT kernel stays below 4e-8).  So only
  //      D <= kTcMaxD takes this path: there the bias stays under the 3e-6 cosine and 1e-5 loss tolerances, above it
  //      (D = 512: 3.8e-6) it would not (tests/test_gpu_ge2e_routes.py pins both sides).
  constexpr int kTcMaxD = 256;
  const bool tc_off = g_ge2e_tc == 0;
  static const size_t tc_min = getenv("SVB_GE2E_TC_MIN") ? (size_t)atoll(getenv("SVB_GE2E_TC_MIN")) : ((size_t)1 << 18);
  const bool tc_path = !tc_off && !dcos && D % 64 == 0 && D <= kTcMaxD && Nc % 8 == 0 && NMr >= 512 && Nc >= 128 &&
                       (size_t)NMr * Nc >= tc_min;
  if (tc_path) {
    auto gemm3 = [&](const __half* A0, const __half* A1, int a_rows, int64_t lda, int a_mn, const __half* B0, const __half* B1,
                     int b_rows, int64_t ldb, int b_mn, float* C, int Mo, int No, int K, int kz) -> int {
      GemmOperands g;
      memset(&g, 0, sizeof(g));
      g.nterms = 3; g.f16 = 1; g.M = Mo; g.N = No; g.K = K; g.kz = kz > 1 ? kz : 0;
      const __half* As[3] = {A0, A0, A1};
      const __half* Bs[3] = {B0, B1, B0};
      // the maps always describe the WHOLE reduction (kz slices address it by blockIdx.z; rows past the end are zero-filled)
      const int Ktot = a_mn ? a_rows : K;
      for (int t = 0; t < 3; ++t) {
        int e = make_operand_map(&g.ta[t], As[t], Mo, Ktot, lda, a_mn, kBM);
        if (e) return e;
        e = make_operand_map(&g.tb[t], Bs[t], No, Ktot, ldb, b_mn, 128);
        if (e) return e;
      }
      (void)b_rows;
      if (!a_mn && !b_mn && No % 256 == 0 && kz <= 1) {
        // wide output (cos = E^ C^T at N = 512: 40 x 2 tiles of 128 x 256 fill the machine in ONE wave; 128 x 128 tiles
        // are 160 CTAs = two waves for 148 SMs)
        EpiStoreF32<256>::Params ep2;
        int e2 = make_store_params<256>(&ep2, C, nullptr, Mo, No, (int64_t)No, 0);
        if (e2) return e2;
        if (ep2.use_tma) {
          for (int t = 0; t < 3; ++t) {
            e2 = make_operand_map(&g.tb[t], Bs[t], No, Ktot, ldb, 0, 256);
            if (e2) return e2;
          }
          cudaError_t ce2 = launch_tc_gemm<256, 4, false, false, EpiStoreF32<256>, 8>(g, ep2, s);
          if (ce2 != cudaSuccess) { set_error("svb_ge2e: tensor-core GEMM (128 x 256 tiles)", ce2); return SVB_ERR_CUDA; }
          return SVB_OK;
        }
      }
      EpiStoreF32<128>::Params ep;
      int e = make_store_params<128>(&ep, C, nullptr, Mo, No, (int64_t)No, 0);
      if (e) return e;
      if (!ep.use_tma) { set_error("svb_ge2e: tensor-core path needs 16-byte aligned outputs", cudaSuccess); return SVB_ERR_ARG; }
      if (kz > 1) {
        e = make_tmap(&ep.tc, C, 4, (uint64_t)No, (uint64_t)Mo, (uint64_t)kz, (uint64_t)No, (uint64_t)No * Mo, 32, 128, 3);
        if (e) return e;
        ep.tma_z = 1;
      }
      cudaError_t ce;
      if (!a_mn && !b_mn) ce = launch_tc_gemm<128, 4, false, false, EpiStoreF32<128>>(g, ep, s);
      else if (!a_mn && b_mn) ce = launch_tc_gemm<128, 4, false, true, EpiStoreF32<128>>(g, ep, s);
      else ce = launch_tc_gemm<128, 4, true, true, EpiStoreF32<128>>(g, ep, s);
      if (ce != cudaSuccess) { set_error("svb_ge2e: tensor-core GEMM", ce); return SVB_ERR_CUDA; }
      return SVB_OK;
    };
    ge2e_phase_kernel<0><<<N < 4 * num_sms ? N : 4 * num_sms, kThreads, smem, s>>>(a);
    int e = gemm3(a.Eh, a.El, NMr, D, 0, a.Ch, a.Cl, Nc, D, 0, a.cosm, NMr, Nc, D, 1);               // cos = E^ C^T
    if (e) return e;
    if (contrast) {          // contrast row phase, then phase D's gathers: no A_off split, no R / P products
      ge2e_phase_contrast_kernel<2><<<b2blocks, kThreads, 0, s>>>(a);
      ge2e_phase_contrast_kernel<4><<<dgrid, kThreads, smem_ct, s>>>(a);
      cudaError_t ce = cudaGetLastError();
      if (ce != cudaSuccess) { set_error("svb_ge2e: launch (tensor-core path, contrast)", ce); return SVB_ERR_CUDA; }
      return SVB_OK;
    }
    ge2e_phase_kernel<2><<<b2blocks, kThreads, 0, s>>>(a);
    if (a.need_grad) {
      e = gemm3(a.Ah, a.Al, NMr, Nc, 0, a.Ch, a.Cl, D, D, 1, a.R, NMr, D, Nc, 1);                   // R = A_off C^
      if (e) return e;
      // P = A_off^T E^ over psplit slices of prows rows (phase D adds the slices in order)
      e = gemm3(a.Ah, a.Al, NMr, Nc, 1, a.Eh, a.El, D, D, 1, a.dC, Nc, D, a.prows, a.psplit);
      if (e) return e;
    }
    ge2e_phase_kernel<4><<<N < 4 * num_sms ? N : 4 * num_sms, kThreads, smem, s>>>(a);
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) { set_error("svb_ge2e: launch (tensor-core path)", ce); return SVB_ERR_CUDA; }
    return SVB_OK;
  }
  a.Eh = a.El = a.Ch = a.Cl = a.Ah = a.Al = nullptr;      // (the fp32 paths do not write the splits)
  if (fused) {
    const void* fk = contrast ? (const void*)ge2e_fused_contrast_kernel : (const void*)ge2e_fused_kernel;
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fk, kThreads, smem_ct);
    if (per_sm < 1) { set_error("svb_ge2e: kernel does not fit", cudaSuccess); return SVB_ERR_UNSUPPORTED; }
    if (per_sm > 4) per_sm = 4;
    int grid = want < per_sm * num_sms ? want : per_sm * num_sms;
    void* params[] = {&a};
    cudaError_t e = cudaLaunchCooperativeKernel(fk, dim3(grid), dim3(kThreads), params, smem_ct, s);
    if (e != cudaSuccess) { set_error("svb_ge2e: cooperative launch", e); return SVB_ERR_CUDA; }
  } else if (contrast) {
    ge2e_phase_kernel<0><<<N, kThreads, smem, s>>>(a);
    ge2e_phase_kernel<1><<<b1tiles, kThreads, smem, s>>>(a);
    ge2e_phase_contrast_kernel<2><<<b2blocks, kThreads, 0, s>>>(a);
    ge2e_phase_contrast_kernel<4><<<dblocks_ct, kThreads, smem_ct, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("svb_ge2e: launch", e); return SVB_ERR_CUDA; }
  } else {
    ge2e_phase_kernel<0><<<N, kThreads, smem, s>>>(a);
    ge2e_phase_kernel<1><<<b1tiles, kThreads, smem, s>>>(a);
    ge2e_phase_kernel<2><<<b2blocks, kThreads, smem, s>>>(a);
    if (a.need_grad) ge2e_phase_kernel<3><<<ctiles, kThreads, smem, s>>>(a);
    ge2e_phase_kernel<4><<<N, kThreads, smem, s>>>(a);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { set_error("svb_ge2e: launch", e); return SVB_ERR_CUDA; }
  }
  return SVB_OK;
}

extern "C" int svb_ge2e_ex(const float* E, const float* Cext, int N, int M, int D, int Nc, const float* w,
                           const float* b, const float* dcos, const float* gscale, float* cos_out, float* per_out,
                           float* loss_out, float* dE, float* dCext, float* dw, float* db, void* workspace,
                           size_t workspace_bytes, int fused, int loss, void* stream) {
  return ge2e_impl(E, Cext, N, M, D, Nc, 0, w, b, dcos, gscale, cos_out, per_out, loss_out, dE, dCext, dw, db, workspace,
                   workspace_bytes, fused, loss, stream);
}
extern "C" int svb_ge2e(const float* E, const float* Cext, int N, int M, int D, int Nc, const float* w,
                        const float* b, const float* dcos, const float* gscale, float* cos_out, float* per_out,
                        float* loss_out, float* dE, float* dCext, float* dw, float* db, void* workspace,
                        size_t workspace_bytes, int fused, void* stream) {
  return svb_ge2e_ex(E, Cext, N, M, D, Nc, w, b, dcos, gscale, cos_out, per_out, loss_out, dE, dCext, dw, db, workspace,
                     workspace_bytes, fused, SVB_GE2E_SOFTMAX, stream);
}

// Row shard of a global GE2E batch (multi-GPU, SURVEY.md section 8e design A): E holds the M utterances of the N_local
// speakers [col0, col0 + N_local) of a batch of Nc speakers whose centroids C (Nc, D) have been gathered from all
// ranks.  Every row is scored against all Nc centroids, with its own column col0 + j replaced by the leave-one-out
// cosine (utils.py:91,113).  Outputs: the shard's part of the loss / dw / db (to be summed over the ranks), dE of the
// shard's rows WITHOUT the path through their own centroid, and dC (Nc, D): this shard's contribution to the gradient
// of every centroid (summed over the ranks, row j of the total is then spread over speaker j's utterances as dC_j / M).
extern "C" int svb_ge2e_rows_ex(const float* E, const float* C, int N_local, int M, int D, int Nc, int col0,
                                const float* w, const float* b, const float* gscale, float* per_out, float* loss_out,
                                float* dE, float* dC, float* dw, float* db, void* workspace, size_t workspace_bytes,
                                int loss, void* stream) {
  if (!C || !w || !b) { set_error("svb_ge2e_rows: centroids, w and b are required", cudaSuccess); return SVB_ERR_ARG; }
  return ge2e_impl(E, C, N_local, M, D, Nc, col0, w, b, nullptr, gscale, nullptr, per_out, loss_out, dE, dC, dw, db,
                   workspace, workspace_bytes, 2, loss, stream);
}
extern "C" int svb_ge2e_rows(const float* E, const float* C, int N_local, int M, int D, int Nc, int col0, const float* w,
                             const float* b, const float* gscale, float* per_out, float* loss_out, float* dE, float* dC,
                             float* dw, float* db, void* workspace, size_t workspace_bytes, void* stream) {
  return svb_ge2e_rows_ex(E, C, N_local, M, D, Nc, col0, w, b, gscale, per_out, loss_out, dE, dC, dw, db, workspace,
                          workspace_bytes, SVB_GE2E_SOFTMAX, stream);
}

// Sum over the utterance axis in the order torch's CPU sum kernel uses for this layout (reduction over a strided
// dimension with a contiguous inner dimension: ATen SumKernel.cpp, vectorized_outer_sum with 256-bit vectors, the
// kernel torch selects in the build image):
//   * columns [0, 32 (D / 32)): cascade summation -- rows are added sequentially into a level-0 accumulator that is
//     flushed into level 1 every 16 rows, level 1 into level 2 every 256, level 2 into level 3 every 4096; remaining
//     rows go to level 0 and the levels are added in order (plain sequential for M < 16, the reference's shapes);
//   * the remaining columns: four interleaved partial sums over rows i = k mod 4 (each a cascade over M / 4 rows), the
//     M % 4 tail rows added to partial 0, then p0 + p1 + p2 + p3.
// Bit-exact against the reference's `embeddings.sum(dim=1)` / `.mean(dim=1)` (tests/golden/centroids.npz).
__device__ __forceinline__ float cascade_sum_rows(const float* __restrict__ x, int M, size_t stride) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int i = 0;
  for (; i + 16 <= M;) {
    for (int j = 0; j < 16; ++j, ++i) a0 = __fadd_rn(a0, x[(size_t)i * stride]);
    a1 = __fadd_rn(a1, a0); a0 = 0.f;
    if ((i & 0xf0) == 0) {
      a2 = __fadd_rn(a2, a1); a1 = 0.f;
      if ((i & 0xf00) == 0) { a3 = __fadd_rn(a3, a2); a2 = 0.f; }
    }
  }
  for (; i < M; ++i) a0 = __fadd_rn(a0, x[(size_t)i * stride]);
  a0 = __fadd_rn(a0, a1);
  a0 = __fadd_rn(a0, a2);
  return __fadd_rn(a0, a3);
}
__device__ __forceinline__ float torch_order_sum_rows(const float* __restrict__ x, int M, int D, int d) {
  if (d < 32 * (D / 32)) return cascade_sum_rows(x, M, D);
  const int q = M / 4;
  float p[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) p[k] = cascade_sum_rows(x + (size_t)k * D, q, (size_t)4 * D);
  for (int i = 4 * q; i < M; ++i) p[0] = __fadd_rn(p[0], x[(size_t)i * D]);
  return __fadd_rn(__fadd_rn(__fadd_rn(p[0], p[1]), p[2]), p[3]);
}
// get_centroids (utils.py:27-29): C[j, d] = mean_m E[j, m, d]; backward: dE[j, m, d] = dC[j, d] / M.
__global__ void centroid_kernel(const float* __restrict__ E, float* __restrict__ C, int N, int M, int D) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)N * D) return;
  const int j = i / D, d = i % D;
  C[i] = __fdiv_rn(torch_order_sum_rows(E + (size_t)j * M * D + d, M, D, d), (float)M);
}
// get_utterance_centroids (utils.py:40-58): U[j, i, :] = (sum_m E[j, m, :] - E[j, i, :]) / (M - 1), the same three
// float32 operations (sum over dim 1, subtract, divide) in the same order.  The operator is linear and symmetric, so
// its backward is the same kernel applied to dL/dU.
__global__ void utterance_centroid_kernel(const float* __restrict__ E, float* __restrict__ U, int N, int M, int D) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)N * D) return;
  const int j = i / D, d = i % D;
  const float* e = E + (size_t)j * M * D + d;
  const float s = torch_order_sum_rows(e, M, D, d);
  const float den = (float)(M - 1);
  float* u = U + (size_t)j * M * D + d;
  for (int m = 0; m < M; ++m) u[(size_t)m * D] = __fdiv_rn(__fsub_rn(s, e[(size_t)m * D]), den);
}
__global__ void centroid_bwd_kernel(const float* __restrict__ dC, float* __restrict__ dE, int N, int M, int D) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)N * M * D) return;
  const int d = i % D;
  const int j = i / ((size_t)M * D);
  dE[i] = dC[(size_t)j * D + d] / (float)M;
}
extern "C" int svb_centroids(const float* E, float* C, int N, int M, int D, void* stream) {
  if (!E || !C || N < 1 || M < 1 || D < 1) return SVB_ERR_ARG;
  const size_t n = (size_t)N * D;
  centroid_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(E, C, N, M, D);
  return cudaGetLastError() == cudaSuccess ? SVB_OK : SVB_ERR_CUDA;
}
extern "C" int svb_utterance_centroids(const float* E, float* U, int N, int M, int D, void* stream) {
  if (!E || !U || N < 1 || M < 2 || D < 1) { set_error("svb_utterance_centroids: bad argument (M must be >= 2)", cudaSuccess); return SVB_ERR_ARG; }
  const size_t n = (size_t)N * D;
  utterance_centroid_kernel<<<(unsigned)((n + 127) / 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(E, U, N, M, D);
  return cudaGetLastError() == cudaSuccess ? SVB_OK : SVB_ERR_CUDA;
}
extern "C" int svb_centroids_bwd(const float* dC, float* dE, int N, int M, int D, void* stream) {
  if (!dC || !dE || N < 1 || M < 1 || D < 1) return SVB_ERR_ARG;
  const size_t n = (size_t)N * M * D;
  centroid_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(dC, dE, N, M, D);
  return cudaGetLastError() == cudaSuccess ? SVB_OK : SVB_ERR_CUDA;
}

// calc_loss (utils.py:126-132) on a caller-supplied similarity matrix S [N, M, Nc]; optional gradient
// dS = gscale * (softmax-with-bias - onehot).  One warp per row.
__global__ void calc_loss_kernel(const float* __restrict__ S, float* __restrict__ per, float* __restrict__ dS,
                                 const float* __restrict__ gscale, int N, int M, int Nc) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= N * M) return;
  const int j = row / M;
  const float* s = S + (size_t)row * Nc;
  float mx = -INFINITY;
  for (int k = lane; k < Nc; k += 32) mx = fmaxf(mx, s[k]);
  mx = warp_max(mx);
  float se = 0.f;
  for (int k = lane; k < Nc; k += 32) se += expf(s[k] - mx);
  se = warp_sum(se);
  const float den = se + kLogBias * expf(-mx);
  if (lane == 0) per[row] = -s[j] + mx + logf(den);
  if (dS) {
    const float gs = gscale ? *gscale : 1.0f;
    for (int k = lane; k < Nc; k += 32) dS[(size_t)row * Nc + k] = gs * (expf(s[k] - mx) / den - (k == j ? 1.f : 0.f));
  }
}
// The contrast loss on a caller-supplied S: per = 1 - sig(S_jj) + sig(S_jk*) (k* = argmax_{k != j} S_jk, lowest index
// among ties); dS = gscale * G with G_jj = -sig sig(-.), G_jk* = sig sig(-.), zero elsewhere.  One warp per row.
__global__ void calc_loss_contrast_kernel(const float* __restrict__ S, float* __restrict__ per, float* __restrict__ dS,
                                          const float* __restrict__ gscale, int N, int M, int Nc) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= N * M) return;
  const int j = row / M;
  const float* s = S + (size_t)row * Nc;
  float sk = -INFINITY;
  int ks = -1;
  for (int k = lane; k < Nc; k += 32) {
    if (k == j) continue;
    if (ks < 0 || s[k] > sk) { sk = s[k]; ks = k; }
  }
  warp_argmax(sk, ks);
  const ContrastRow c = contrast_row(s[j], sk);
  if (lane == 0) per[row] = c.per;
  if (dS) {
    const float gs = gscale ? *gscale : 1.0f;
    for (int k = lane; k < Nc; k += 32) dS[(size_t)row * Nc + k] = k == j ? gs * c.gd : (k == ks ? gs * c.gk : 0.f);
  }
}
__global__ void sum_kernel(const float* __restrict__ x, float* __restrict__ out, int n) {
  __shared__ float red[8];
  float v = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) v += x[i];
  v = block_sum(v, red);
  if (threadIdx.x == 0) *out = v;
}
extern "C" int svb_calc_loss_ex(const float* S, int N, int M, int Nc, float* per_out, float* loss_out, float* dS,
                                const float* gscale, int loss, void* stream) {
  if (!S || !per_out || N < 1 || M < 1 || Nc < N) return SVB_ERR_ARG;
  if (loss != kSoftmax && loss != kContrast) { set_error("svb_calc_loss: unknown loss method", cudaSuccess); return SVB_ERR_ARG; }
  if (loss == kContrast && Nc < 2) { set_error("svb_calc_loss: the contrast loss needs at least two columns", cudaSuccess); return SVB_ERR_ARG; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (loss == kContrast) calc_loss_contrast_kernel<<<(N * M + 7) / 8, 256, 0, st>>>(S, per_out, dS, gscale, N, M, Nc);
  else calc_loss_kernel<<<(N * M + 7) / 8, 256, 0, st>>>(S, per_out, dS, gscale, N, M, Nc);
  if (loss_out) sum_kernel<<<1, 256, 0, st>>>(per_out, loss_out, N * M);
  return cudaGetLastError() == cudaSuccess ? SVB_OK : SVB_ERR_CUDA;
}
extern "C" int svb_calc_loss(const float* S, int N, int M, int Nc, float* per_out, float* loss_out, float* dS,
                             const float* gscale, void* stream) {
  return svb_calc_loss_ex(S, N, M, Nc, per_out, loss_out, dS, gscale, SVB_GE2E_SOFTMAX, stream);
}
