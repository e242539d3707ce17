// Score calibration and calibration metrics (DESIGN.md 4.5.3) for sm_100a: Cllr, actual DCF, minCllr and ROCCH-EER of
// log-likelihood-ratio scores, and the linear logistic-regression calibration llr = a * s + b.
//
// - Cllr / actual DCF: one grid-stride pass (calib_stats_kernel) writes per-block float64 softplus sums and integer
//   counts; calib_metrics_finish_kernel adds the blocks in index order.
// - minCllr / ROCCH-EER: verif.cu's radix sort (verif_sort.cuh) puts the (key, label) elements in ascending order.
//   calib_tile_hull_kernel builds, per 4096-element tile, the lower convex hull of the cumulative points (trials, targets)
//   at the tile's group ends (last element of each run of equal keys) in tile-local coordinates.  calib_merge_kernel
//   joins neighbouring hulls pairwise, log2(tiles) launches, each join finding the bridge of the two hulls and
//   carrying the left node's (trials, targets) as the offset of the right one.  calib_hull_final_kernel adds the origin,
//   sums the segment terms and finds the ROCCH crossing.  Every hull test is an exact int64 cross product.
// - Calibration: damped Newton in float64 on centred scores.  Each iteration is a fused pass (objective, gradient,
//   2 x 2 Hessian as per-block partials) and a one-block update; the host enqueues max_iter pairs and the kernels after
//   convergence return at once, so the fit needs no host round trip.
// No float atomics and fixed reduction orders: every output is identical from run to run and across streams.  The
// entry points neither allocate nor synchronise, so a CUDA graph can capture them.
#include "../../include/svb200.h"
#include "verif_sort.cuh"
#include <cuda_runtime.h>
#include <math.h>
#include <algorithm>
#include <stdint.h>

namespace svb {
void set_error(const char* what, cudaError_t e);

namespace calib {
using verif::kSortTile;

constexpr int kMaxPoints = 8;
constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxBlocks = 512;              // per-block partials of the grid-stride passes
constexpr int kFinalThreads = 1024;
constexpr double kLn2 = 0.69314718055994530942;
// Newton stops once half the squared Newton decrement, g' H^-1 g / 2 (the predicted decrease of the objective), is at
// most this; the last Newton step is then taken without a line search, whose float64 objective comparison could not
// resolve decreases this small.
constexpr double kDecrementTol = 1e-12;
constexpr int kMaxHalvings = 40;

struct Points {
  double w[kMaxPoints][3];     // w_miss, w_fa, c_def
  double theta[kMaxPoints];    // Bayes threshold log(w_fa / w_miss)
  int P;
};

// Per-block partials of the stats pass.  [0] targets, [1] non-targets.
struct Stats {
  double sp[2];                // sum softplus(-l) over targets, softplus(l) over non-targets
  uint32_t nt, nonfinite;
  uint32_t miss[kMaxPoints], fa[kMaxPoints];
  uint32_t kmin[2], kmax[2];   // order-preserving keys of the class extremes
};

struct TrainState {
  double a, b, c;              // accepted point (centred parameters) and its objective
  double ta, tb;               // point the next pass evaluates
  double da, db, t;            // Newton direction and step fraction
  double c0, scale;            // centring: u = (s - c0) * scale
  double wt, wn, tau;          // pi / Nt, (1 - pi) / Nn, logit(pi)
  int have, phase, iters, halvings;   // phase 0: line search, 1: final evaluation, 2: done
};

__device__ __forceinline__ double softplus(double z) { return fmax(z, 0.0) + log1p(exp(-fabs(z))); }

// ------------------------------------------------------------------------------------------------ block reductions
struct Sum { template <typename T> __device__ T operator()(T a, T b) const { return a + b; } };
struct Min { __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a < b ? a : b; } };
struct Max { __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; } };

// Butterfly within each warp, then the warps in index order: a fixed order, so float sums are reproducible.  Every
// thread returns the block's value.
template <int kN, typename T, typename Op>
__device__ __forceinline__ T block_reduce(T v, Op op, T* scratch) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  T r = scratch[0];
  for (int w = 1; w < kN / 32; ++w) r = op(r, scratch[w]);
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------ (a) stats pass
// Grid-stride over the scores.  kSoftplus: also the Cllr sums (the training's first pass needs only counts and extremes).
template <bool kSoftplus>
__global__ void __launch_bounds__(kThreads) calib_stats_kernel(const float* __restrict__ s,
                                                               const uint8_t* __restrict__ lab, int n, Points pt,
                                                               Stats* __restrict__ part) {
  __shared__ double dscr[kWarps];
  __shared__ uint32_t uscr[kWarps];
  double sp0 = 0.0, sp1 = 0.0;
  uint32_t nt = 0, nf = 0, kmin0 = 0xffffffffu, kmin1 = 0xffffffffu, kmax0 = 0u, kmax1 = 0u;
  uint32_t miss[kMaxPoints], fa[kMaxPoints];
#pragma unroll
  for (int q = 0; q < kMaxPoints; ++q) miss[q] = fa[q] = 0;
  const int stride = gridDim.x * kThreads;
#pragma unroll 4
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const float x = __ldg(s + i);
    const bool t = __ldg(lab + i) != 0;
    const uint32_t key = verif::score_key(x, nf);
    const double l = (double)x;
    if (t) {
      ++nt;
      kmin0 = min(kmin0, key); kmax0 = max(kmax0, key);
      if (kSoftplus) sp0 += softplus(-l);
    } else {
      kmin1 = min(kmin1, key); kmax1 = max(kmax1, key);
      if (kSoftplus) sp1 += softplus(l);
    }
#pragma unroll
    for (int q = 0; q < kMaxPoints; ++q) {
      if (q < pt.P) {
        const bool below = l < pt.theta[q];
        miss[q] += t && below;
        fa[q] += !t && !below;
      }
    }
    if (i > n - stride) break;                         // keeps i + stride from overflowing int
  }
  Stats r;
  r.sp[0] = block_reduce<kThreads>(sp0, Sum(), dscr);
  r.sp[1] = block_reduce<kThreads>(sp1, Sum(), dscr);
  r.nt = block_reduce<kThreads>(nt, Sum(), uscr);
  r.nonfinite = block_reduce<kThreads>(nf, Sum(), uscr);
#pragma unroll
  for (int q = 0; q < kMaxPoints; ++q) {
    r.miss[q] = q < pt.P ? block_reduce<kThreads>(miss[q], Sum(), uscr) : 0u;
    r.fa[q] = q < pt.P ? block_reduce<kThreads>(fa[q], Sum(), uscr) : 0u;
  }
  r.kmin[0] = block_reduce<kThreads>(kmin0, Min(), uscr);
  r.kmin[1] = block_reduce<kThreads>(kmin1, Min(), uscr);
  r.kmax[0] = block_reduce<kThreads>(kmax0, Max(), uscr);
  r.kmax[1] = block_reduce<kThreads>(kmax1, Max(), uscr);
  if (threadIdx.x == 0) part[blockIdx.x] = r;
}

// The partials of G blocks, added in block order (thread t takes blocks t, t + 256, ...; then block_reduce).
__device__ Stats reduce_stats(const Stats* part, int G, int P, double* dscr, uint32_t* uscr) {
  Stats r;
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    double v = 0.0;
    for (int g = threadIdx.x; g < G; g += kThreads) v += part[g].sp[c];
    r.sp[c] = block_reduce<kThreads>(v, Sum(), dscr);
    uint32_t lo = 0xffffffffu, hi = 0u;
    for (int g = threadIdx.x; g < G; g += kThreads) { lo = min(lo, part[g].kmin[c]); hi = max(hi, part[g].kmax[c]); }
    r.kmin[c] = block_reduce<kThreads>(lo, Min(), uscr);
    r.kmax[c] = block_reduce<kThreads>(hi, Max(), uscr);
  }
  uint32_t nt = 0, nf = 0;
  for (int g = threadIdx.x; g < G; g += kThreads) { nt += part[g].nt; nf += part[g].nonfinite; }
  r.nt = block_reduce<kThreads>(nt, Sum(), uscr);
  r.nonfinite = block_reduce<kThreads>(nf, Sum(), uscr);
#pragma unroll
  for (int q = 0; q < kMaxPoints; ++q) {
    uint32_t m = 0, f = 0;
    if (q < P)
      for (int g = threadIdx.x; g < G; g += kThreads) { m += part[g].miss[q]; f += part[g].fa[q]; }
    r.miss[q] = block_reduce<kThreads>(m, Sum(), uscr);
    r.fa[q] = block_reduce<kThreads>(f, Sum(), uscr);
  }
  return r;
}

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000ll); }

// out: [0] cllr, [3] Nt, [4] Nn, [5] #non-finite, then per point act_dcf, theta, p_miss, p_fa (8 + 4p ...)
__global__ void __launch_bounds__(kThreads) calib_metrics_finish_kernel(const Stats* __restrict__ part, int G, int n,
                                                                        Points pt, double* __restrict__ out) {
  __shared__ double dscr[kWarps];
  __shared__ uint32_t uscr[kWarps];
  const Stats r = reduce_stats(part, G, pt.P, dscr, uscr);
  if (threadIdx.x != 0) return;
  const uint32_t Nt = r.nt, Nn = (uint32_t)n - r.nt;
  const bool bad = r.nonfinite != 0 || Nt == 0 || Nn == 0;
  const double dNt = (double)Nt, dNn = (double)Nn;
  out[0] = bad ? qnan() : 0.5 * (r.sp[0] / dNt + r.sp[1] / dNn) / kLn2;
  out[3] = dNt;
  out[4] = dNn;
  out[5] = (double)r.nonfinite;
#pragma unroll
  for (int q = 0; q < kMaxPoints; ++q) {
    if (q >= pt.P) break;
    const double pm = __ddiv_rn((double)r.miss[q], dNt), pf = __ddiv_rn((double)r.fa[q], dNn);
    const double dcf = __ddiv_rn(__dadd_rn(__dmul_rn(pt.w[q][0], pm), __dmul_rn(pt.w[q][1], pf)), pt.w[q][2]);
    double* o = out + 8 + 4 * q;
    o[0] = bad ? qnan() : dcf;
    o[1] = bad ? qnan() : pt.theta[q];
    o[2] = bad ? qnan() : pm;
    o[3] = bad ? qnan() : pf;
  }
}

// ------------------------------------------------------------------------------------------------ (b) convex hull
// Points are (x, y) = (trials, targets) at group ends.  cross > 0: o -> a -> b turns counter-clockwise.
__device__ __forceinline__ long long cross(int2 o, int2 a, int2 b) {
  return (long long)(a.x - o.x) * (b.y - o.y) - (long long)(a.y - o.y) * (b.x - o.x);
}

// Monotone chain: appends pts[start, start + len) (ascending x) to the lower hull pts[dst, dst + k).  In place: the
// hull never holds more points than were read, so every write lands at or before the point being read.
__device__ __forceinline__ void chain(int2* pts, int dst, int& k, int start, int len) {
  for (int i = start; i < start + len; ++i) {
    const int2 p = pts[i];
    while (k >= 2 && cross(pts[dst + k - 2], pts[dst + k - 1], p) <= 0) --k;   // collinear points are dropped
    pts[dst + k++] = p;
  }
}

// One 4096-element tile per CTA, 16 consecutive elements a thread.  The hull of the tile's group ends is built in three
// serial levels (each thread over its own points, lane 0 over its warp's hulls, thread 0 over the warps' hulls) and
// stored at hull[tile * 4096, + cnt[tile]) in tile-local coordinates: x = position in the tile + 1, y = targets in the
// tile up to and including the point.
__global__ void __launch_bounds__(kThreads) calib_tile_hull_kernel(const unsigned long long* __restrict__ sorted, int n,
                                                                   int2* __restrict__ hull, int* __restrict__ cnt,
                                                                   int* __restrict__ tgt, int* __restrict__ groups) {
  constexpr int kItems = kSortTile / kThreads;
  __shared__ int2 pts[kSortTile];
  __shared__ uint32_t wtot[kWarps];
  __shared__ int seg_start[kThreads], seg_len[kThreads], wseg_start[kWarps], wseg_len[kWarps], s_h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int base = blockIdx.x * kSortTile;
  const int lim = n - base;                            // tile-local positions below lim are elements
  const int lp = tid * kItems;
  unsigned long long e[kItems + 1];
#pragma unroll
  for (int j = 0; j <= kItems; ++j) e[j] = lp + j < lim ? __ldg(sorted + base + lp + j) : ~0ull;   // ~0: no next key
  uint32_t mine = 0, ends = 0;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (lp + j < lim) {
      mine += (uint32_t)(e[j] & 1ull);
      ends += (e[j] >> 1) != (e[j + 1] >> 1);
    }
  }
  uint32_t tile_tgt, tile_ends;
  uint32_t y = verif::block_excl_scan<kThreads>(mine, wtot, &tile_tgt);
  const uint32_t off = verif::block_excl_scan<kThreads>(ends, wtot, &tile_ends);
  int w = (int)off;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (lp + j < lim) {
      y += (uint32_t)(e[j] & 1ull);
      if ((e[j] >> 1) != (e[j + 1] >> 1)) pts[w++] = make_int2(lp + j + 1, (int)y);
    }
  }
  int k = 0;
  chain(pts, (int)off, k, (int)off, (int)ends);
  seg_start[tid] = (int)off;
  seg_len[tid] = k;
  __syncthreads();
  if (lane == 0) {
    int kw = 0;
    const int dst = seg_start[tid];
    for (int l = 0; l < 32; ++l) chain(pts, dst, kw, seg_start[tid + l], seg_len[tid + l]);
    wseg_start[warp] = dst;
    wseg_len[warp] = kw;
  }
  __syncthreads();
  if (tid == 0) {
    int kb = 0;
    for (int v = 0; v < kWarps; ++v) chain(pts, 0, kb, wseg_start[v], wseg_len[v]);
    s_h = kb;
    cnt[blockIdx.x] = kb;
    tgt[blockIdx.x] = (int)tile_tgt;
    groups[blockIdx.x] = (int)tile_ends;
  }
  __syncthreads();
  for (int i = tid; i < s_h; i += kThreads) hull[(size_t)base + i] = pts[i];
}

struct Bridge {
  long long num, den;          // slope num / den of the bridge candidate (num >= 0, den > 0)
  int i, j;
};

// a's slope is below b's (ties: the larger j).  j < 0 marks "no candidate", which loses to any candidate: a sentinel
// slope would overflow the cross-multiplication.
__device__ __forceinline__ bool lower_slope(const Bridge& a, const Bridge& b) {
  if (a.j < 0) return false;
  if (b.j < 0) return true;
  const long long l = a.num * b.den, r = b.num * a.den;
  return l < r || (l == r && a.j > b.j);
}

__device__ __forceinline__ Bridge warp_min(Bridge b) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    Bridge y;
    y.num = __shfl_xor_sync(0xffffffffu, b.num, o);
    y.den = __shfl_xor_sync(0xffffffffu, b.den, o);
    y.i = __shfl_xor_sync(0xffffffffu, b.i, o);
    y.j = __shfl_xor_sync(0xffffffffu, b.j, o);
    if (lower_slope(y, b)) b = y;
  }
  return b;
}

// Joins the hulls of nodes [l, l + s) and [l + s, l + 2s) of s tiles each (node data at its first tile).  The bridge
// touches R[j*], the vertex whose tangent to L has the smallest slope, and L[i*], that tangent's point of contact
// (binary search: the first i at which L[i + 1] is not strictly below the line L[i] -> R[j]).  The result L[0, i*] +
// R[j*, ...) is written in place over L, with R shifted by L's (trials, targets).
__global__ void __launch_bounds__(kThreads) calib_merge_kernel(int2* __restrict__ hull, int* __restrict__ cnt,
                                                               int* __restrict__ tgt, int T, int s) {
  __shared__ Bridge scr[kWarps];
  __shared__ Bridge s_best;
  const int l = 2 * s * blockIdx.x, r = l + s;
  if (r >= T) return;
  const int Lc = cnt[l], Rc = cnt[r];
  const int dx = s * kSortTile, dy = tgt[l];
  int2* L = hull + (size_t)l * kSortTile;
  const int2* R = hull + (size_t)r * kSortTile;
  Bridge best{1, 0, -1, 0};                            // Lc == 0: R is kept whole
  if (Lc > 0 && Rc > 0) {
    best = Bridge{0, 1, 0, -1};
    for (int j = threadIdx.x; j < Rc; j += kThreads) {
      const int2 q = make_int2(R[j].x + dx, R[j].y + dy);
      int lo = 0, hi = Lc - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cross(L[mid], q, L[mid + 1]) < 0) lo = mid + 1; else hi = mid;
      }
      const Bridge c{(long long)q.y - L[lo].y, (long long)q.x - L[lo].x, lo, j};
      if (lower_slope(c, best)) best = c;
    }
    best = warp_min(best);
    if ((threadIdx.x & 31) == 0) scr[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int v = 1; v < kWarps; ++v) if (lower_slope(scr[v], best)) best = scr[v];
      s_best = best;
    }
    __syncthreads();
    best = s_best;
  }
  if (Rc > 0) {
    // the destination L + i* + 1 + (j - j*) never passes the source R + j (i* < Lc <= s * 4096): chunk by chunk, all
    // reads of a chunk before its writes, is safe in place
    const int i0 = best.i + 1, j0 = best.j;
    for (int c0 = j0; c0 < Rc; c0 += kThreads) {
      const int j = c0 + threadIdx.x;
      int2 v = make_int2(0, 0);
      if (j < Rc) v = make_int2(R[j].x + dx, R[j].y + dy);
      __syncthreads();
      if (j < Rc) L[i0 + j - j0] = v;
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) {
    if (Rc > 0) cnt[l] = best.i + 1 + Rc - best.j;
    tgt[l] = dy + tgt[r];
  }
}

// One CTA.  The hull of every group end is hull[0, cnt[0]); the origin joins it at the vertex of smallest slope y / x
// (ties: the larger x).  out[1] min_cllr, out[2] rocch_eer, out[6] hull vertices (with the origin), out[7] K.
__global__ void __launch_bounds__(kFinalThreads) calib_hull_final_kernel(const int2* __restrict__ hull,
                                                                         const int* __restrict__ cnt,
                                                                         const int* __restrict__ groups, int T, int n,
                                                                         const unsigned long long* __restrict__ counts,
                                                                         double* __restrict__ out) {
  __shared__ double dscr[kFinalThreads / 32];
  __shared__ unsigned long long kscr[kFinalThreads / 32];
  __shared__ Bridge bscr[kFinalThreads / 32];
  __shared__ int iscr[kFinalThreads / 32];
  const int tid = threadIdx.x;
  const int c = cnt[0];
  const long long Nt = (long long)counts[0], Nn = (long long)n - Nt;
  const bool bad = counts[1] != 0 || Nt == 0 || Nn == 0;

  unsigned long long K = 0;
  for (int t = tid; t < T; t += kFinalThreads) K += (unsigned long long)groups[t];
  K = block_reduce<kFinalThreads>(K, Sum(), kscr);

  // the origin's tangent vertex k: smallest y / x, ties to the larger index
  Bridge b{0, 1, 0, -1};
  for (int m = tid; m < c; m += kFinalThreads) {
    const Bridge cand{hull[m].y, hull[m].x, m, m};
    if (lower_slope(cand, b)) b = cand;
  }
  b = warp_min(b);
  if ((tid & 31) == 0) bscr[tid >> 5] = b;
  __syncthreads();
  for (int v = 0; v < kFinalThreads / 32; ++v) if (lower_slope(bscr[v], b)) b = bscr[v];
  const int k = b.j;

  // segment m joins vertex m (the origin for m = k - 1) to vertex m + 1; natural-log terms, divided by ln 2 at the end
  const double dNt = (double)Nt, dNn = (double)Nn;
  double st = 0.0, sn = 0.0;
  for (int m = k - 1 + tid; m < c - 1; m += kFinalThreads) {
    const int2 p = m < k ? make_int2(0, 0) : hull[m], q = hull[m + 1];
    const long long t = q.y - p.y, f = (long long)(q.x - p.x) - t;
    if (t > 0 && f > 0) {
      st += (double)t * log1p(((double)f * dNt) / ((double)t * dNn));
      sn += (double)f * log1p(((double)t * dNn) / ((double)f * dNt));
    }
  }
  st = block_reduce<kFinalThreads>(st, Sum(), dscr);
  sn = block_reduce<kFinalThreads>(sn, Sum(), dscr);

  // ROCCH: the first hull vertex with d = y * Nn - (Nn - x + y) * Nt >= 0 (P_miss >= P_fa); the last vertex has d > 0
  int first = c;
  for (int m = k + tid; m < c; m += kFinalThreads) {
    const int2 v = hull[m];
    if ((long long)v.y * Nn - (Nn - v.x + v.y) * Nt >= 0) { first = m; break; }
  }
  first = block_reduce<kFinalThreads>(first, [](int a, int x) { return a < x ? a : x; }, iscr);
  if (tid != 0) return;
  double eer = qnan();
  if (first < c) {
    const int2 p = first == k ? make_int2(0, 0) : hull[first - 1], q = hull[first];
    const long long dp = (long long)p.y * Nn - (Nn - p.x + p.y) * Nt, dq = (long long)q.y * Nn - (Nn - q.x + q.y) * Nt;
    const double pm0 = (double)p.y / dNt, pm1 = (double)q.y / dNt;
    if (dq == 0) {
      eer = pm1;
    } else {
      const double u = (double)(-dp) / (double)(dq - dp);
      eer = pm0 + u * (pm1 - pm0);
    }
  }
  out[1] = bad ? qnan() : 0.5 * (st / dNt + sn / dNn) / kLn2;
  out[2] = bad ? qnan() : eer;
  out[6] = (double)(c - k + 1);
  out[7] = (double)K;
}

// ------------------------------------------------------------------------------------------------ (c) calibration
// out: a, b, C / ln 2, iterations, status (SVB_CALIB_*)
__device__ void write_fit(const TrainState& S, int status, double* out) {
  const bool ok = status == SVB_CALIB_CONVERGED || (status == SVB_CALIB_ITERATION_CAP && S.have);
  out[0] = ok ? S.a * S.scale : qnan();
  out[1] = ok ? S.b - S.a * S.scale * S.c0 : qnan();
  out[2] = ok ? S.c / kLn2 : qnan();
  out[3] = (double)S.iters;
  out[4] = (double)status;
}

__global__ void __launch_bounds__(kThreads) calib_train_init_kernel(const Stats* __restrict__ part, int G, int n,
                                                                    double prior, double tau,
                                                                    TrainState* __restrict__ state,
                                                                    double* __restrict__ out) {
  __shared__ double dscr[kWarps];
  __shared__ uint32_t uscr[kWarps];
  const Stats r = reduce_stats(part, G, 0, dscr, uscr);
  if (threadIdx.x != 0) return;
  TrainState S = {};
  S.phase = 2;
  const uint32_t Nt = r.nt, Nn = (uint32_t)n - r.nt;
  int status = -1;
  if (r.nonfinite != 0 || Nt == 0 || Nn == 0) {
    status = SVB_CALIB_BAD_INPUT;
  } else if (!(r.kmin[0] < r.kmax[1] && r.kmin[1] < r.kmax[0])) {   // no strict overlap (covers a single value)
    status = SVB_CALIB_SEPARABLE;
  } else {
    const double lo = verif::key_value(min(r.kmin[0], r.kmin[1])), hi = verif::key_value(max(r.kmax[0], r.kmax[1]));
    S.c0 = 0.5 * lo + 0.5 * hi;
    S.scale = 2.0 / (hi - lo);
    S.wt = prior / (double)Nt;
    S.wn = (1.0 - prior) / (double)Nn;
    S.tau = tau;
    S.t = 1.0;
    S.phase = 0;
  }
  *state = S;
  if (status >= 0) write_fit(S, status, out);
}

// Objective, gradient and Hessian at the trial point, as per-block partials [6 * block]:
// C, dC/da, dC/db, d2C/da2, d2C/dadb, d2C/db2 with z = ta * u + tb + tau.
__global__ void __launch_bounds__(kThreads) calib_newton_pass_kernel(const float* __restrict__ s,
                                                                     const uint8_t* __restrict__ lab, int n,
                                                                     const TrainState* __restrict__ state,
                                                                     double* __restrict__ part) {
  __shared__ double dscr[kWarps];
  const TrainState& S = *state;
  if (S.phase == 2) return;
  const double ta = S.ta, tb = S.tb, c0 = S.c0, scale = S.scale, tau = S.tau, wt = S.wt, wn = S.wn;
  double f = 0.0, ga = 0.0, gb = 0.0, haa = 0.0, hab = 0.0, hbb = 0.0;
  const int stride = gridDim.x * kThreads;
#pragma unroll 4
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const double u = ((double)__ldg(s + i) - c0) * scale;
    const bool t = __ldg(lab + i) != 0;
    const double z = ta * u + tb + tau;
    const double e = exp(-fabs(z));
    const double lg = log1p(e);
    const double sig = z >= 0.0 ? 1.0 / (1.0 + e) : e / (1.0 + e);     // sigmoid(z)
    const double w = t ? wt : wn;
    const double fz = t ? fmax(-z, 0.0) + lg : fmax(z, 0.0) + lg;      // softplus(-z) / softplus(z)
    const double gz = w * (t ? sig - 1.0 : sig);
    const double hz = w * (e / ((1.0 + e) * (1.0 + e)));              // sigmoid(z) sigmoid(-z)
    f += w * fz;
    ga += gz * u;
    gb += gz;
    haa += hz * u * u;
    hab += hz * u;
    hbb += hz;
    if (i > n - stride) break;
  }
  const double v[6] = {f, ga, gb, haa, hab, hbb};
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    const double r = block_reduce<kThreads>(v[c], Sum(), dscr);
    if (threadIdx.x == 0) part[6 * blockIdx.x + c] = r;
  }
}

__global__ void __launch_bounds__(kThreads) calib_newton_update_kernel(const double* __restrict__ part, int G,
                                                                       TrainState* __restrict__ state, int last,
                                                                       double* __restrict__ out) {
  __shared__ double dscr[kWarps];
  if (state->phase == 2) return;
  double v[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    double a = 0.0;
    for (int g = threadIdx.x; g < G; g += kThreads) a += part[6 * g + c];
    v[c] = block_reduce<kThreads>(a, Sum(), dscr);
  }
  if (threadIdx.x != 0) return;
  TrainState S = *state;
  ++S.iters;
  int status = -1;
  if (S.phase == 1) {                                  // the final Newton step, evaluated
    S.a = S.ta; S.b = S.tb; S.c = v[0];
    status = SVB_CALIB_CONVERGED;
  } else if (!S.have || v[0] < S.c) {                  // accept, then the next Newton step
    S.a = S.ta; S.b = S.tb; S.c = v[0]; S.have = 1;
    const double det = v[3] * v[5] - v[4] * v[4];
    const double da = -(v[5] * v[1] - v[4] * v[2]) / det, db = -(v[3] * v[2] - v[4] * v[1]) / det;
    const double lam2 = -(v[1] * da + v[2] * db);
    if (!(det > 0.0) || !isfinite(da) || !isfinite(db)) {
      status = SVB_CALIB_ITERATION_CAP;                // the Hessian lost its curvature in float64
    } else {
      S.da = da; S.db = db; S.t = 1.0; S.halvings = 0;
      S.ta = S.a + da; S.tb = S.b + db;
      if (0.5 * lam2 <= kDecrementTol) S.phase = 1;
    }
  } else if (++S.halvings > kMaxHalvings) {            // no decrease resolvable in float64: converged at the point
    status = SVB_CALIB_CONVERGED;
  } else {
    S.t *= 0.5;
    S.ta = S.a + S.t * S.da; S.tb = S.b + S.t * S.db;
  }
  if (status < 0 && last) status = SVB_CALIB_ITERATION_CAP;
  if (status >= 0) {
    S.phase = 2;
    write_fit(S, status, out);
  }
  *state = S;
}

// ------------------------------------------------------------------------------------------------ host side
inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }
inline bool n_ok(int64_t n) { return n >= 2 && n < (int64_t(1) << 31); }
inline int pass_blocks(int64_t n) {
  return (int)std::min<int64_t>(kMaxBlocks, (n + 4 * kThreads - 1) / (4 * kThreads));
}

// Workspace: the sort's two 8n-byte element buffers (the first holds the hulls once the sort is done: a node's hull
// has at most one vertex per element of its tiles), its digit table and cleared counters; per-tile hull counts,
// target counts and group counts; the per-block partials and the fit's state.
struct Layout {
  size_t a, b, offs, ctr, cnt, tgt, groups, stats, newton, state, total;
  int tiles;
};

inline Layout layout(int64_t n) {
  Layout L;
  L.tiles = verif::sort_tiles(n);
  L.a = 0;
  L.b = align_up(8 * (size_t)n);
  L.offs = L.b + align_up(8 * (size_t)n);
  L.ctr = L.offs + align_up(verif::sort_table_bytes(n));
  L.cnt = L.ctr + align_up(verif::kSortCounterBytes);
  L.tgt = L.cnt + align_up((size_t)L.tiles * 4);
  L.groups = L.tgt + align_up((size_t)L.tiles * 4);
  L.stats = L.groups + align_up((size_t)L.tiles * 4);
  L.newton = L.stats + align_up(kMaxBlocks * sizeof(Stats));
  L.state = L.newton + align_up(kMaxBlocks * 6 * sizeof(double));
  L.total = L.state + align_up(sizeof(TrainState));
  return L;
}

inline bool ws_ok(int64_t n, void* ws, size_t bytes) {
  return ws && bytes >= layout(n).total && (reinterpret_cast<uintptr_t>(ws) & 255) == 0;
}

int metrics(const float* llr, const uint8_t* labels, int64_t n64, const double* ops, int P, void* workspace,
            size_t workspace_bytes, double* out, void* stream) {
  const char* who = "svb_calib_metrics: bad argument (2 <= n < 2^31, 1 <= P <= 8, positive finite weights, workspace "
                    "of svb_calib_workspace_bytes, 256-byte aligned)";
  if (!llr || !labels || !ops || !out || !n_ok(n64) || P < 1 || P > kMaxPoints ||
      !ws_ok(n64, workspace, workspace_bytes)) {
    set_error(who, cudaSuccess);
    return SVB_ERR_ARG;
  }
  Points pt;
  pt.P = P;
  for (int p = 0; p < kMaxPoints; ++p) {
    for (int c = 0; c < 3; ++c) pt.w[p][c] = p < P ? ops[3 * p + c] : 1.0;
    if (!(pt.w[p][0] > 0.0) || !(pt.w[p][1] > 0.0) || !(pt.w[p][2] > 0.0) || !isfinite(pt.w[p][0]) ||
        !isfinite(pt.w[p][1]) || !isfinite(pt.w[p][2])) {
      set_error(who, cudaSuccess);
      return SVB_ERR_ARG;
    }
    pt.theta[p] = log(pt.w[p][1] / pt.w[p][0]);
  }
  const int n = (int)n64;
  const Layout L = layout(n64);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  auto* stats = reinterpret_cast<Stats*>(ws + L.stats);
  auto* cnt = reinterpret_cast<int*>(ws + L.cnt);
  auto* tgt = reinterpret_cast<int*>(ws + L.tgt);
  auto* groups = reinterpret_cast<int*>(ws + L.groups);
  verif::SortBuffers sb;
  sb.a = reinterpret_cast<unsigned long long*>(ws + L.a);
  sb.b = reinterpret_cast<unsigned long long*>(ws + L.b);
  sb.offs = reinterpret_cast<uint32_t*>(ws + L.offs);
  sb.hist = reinterpret_cast<uint32_t*>(ws + L.ctr);
  sb.counts = reinterpret_cast<unsigned long long*>(ws + L.ctr + verif::kPasses * verif::kBins * 4);
  auto* hull = reinterpret_cast<int2*>(ws + L.a);

  const int G = pass_blocks(n64);
  calib_stats_kernel<true><<<G, kThreads, 0, st>>>(llr, labels, n, pt, stats);
  calib_metrics_finish_kernel<<<1, kThreads, 0, st>>>(stats, G, n, pt, out);
  cudaError_t e = cudaMemsetAsync(ws + L.ctr, 0, verif::kSortCounterBytes, st);
  if (e == cudaSuccess) e = verif::sort_elements(llr, labels, n, 1, 1, sb, st);
  if (e != cudaSuccess) { set_error("svb_calib_metrics", e); return SVB_ERR_CUDA; }
  calib_tile_hull_kernel<<<L.tiles, kThreads, 0, st>>>(sb.b, n, hull, cnt, tgt, groups);
  for (int s = 1; s < L.tiles; s *= 2)
    calib_merge_kernel<<<(L.tiles - s + 2 * s - 1) / (2 * s), kThreads, 0, st>>>(hull, cnt, tgt, L.tiles, s);
  calib_hull_final_kernel<<<1, kFinalThreads, 0, st>>>(hull, cnt, groups, L.tiles, n, sb.counts, out);
  e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("svb_calib_metrics", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

int train(const float* s, const uint8_t* labels, int64_t n64, double prior, int max_iter, void* workspace,
          size_t workspace_bytes, double* out, void* stream) {
  if (!s || !labels || !out || !n_ok(n64) || !(prior > 0.0 && prior < 1.0) || max_iter < 1 ||
      !ws_ok(n64, workspace, workspace_bytes)) {
    set_error("svb_calib_train: bad argument (2 <= n < 2^31, 0 < prior < 1, max_iter >= 1, workspace of "
              "svb_calib_workspace_bytes, 256-byte aligned)", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const int n = (int)n64;
  const Layout L = layout(n64);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  auto* stats = reinterpret_cast<Stats*>(ws + L.stats);
  auto* part = reinterpret_cast<double*>(ws + L.newton);
  auto* state = reinterpret_cast<TrainState*>(ws + L.state);
  Points none = {};
  const int G = pass_blocks(n64);
  calib_stats_kernel<false><<<G, kThreads, 0, st>>>(s, labels, n, none, stats);
  calib_train_init_kernel<<<1, kThreads, 0, st>>>(stats, G, n, prior, log(prior / (1.0 - prior)), state, out);
  for (int k = 0; k < max_iter; ++k) {
    calib_newton_pass_kernel<<<G, kThreads, 0, st>>>(s, labels, n, state, part);
    calib_newton_update_kernel<<<1, kThreads, 0, st>>>(part, G, state, k == max_iter - 1, out);
  }
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("svb_calib_train", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

}  // namespace calib
}  // namespace svb

extern "C" int svb_calib_workspace_bytes(int64_t n, size_t* bytes) {
  if (!bytes || !svb::calib::n_ok(n)) {
    svb::set_error("svb_calib_workspace_bytes: need 2 <= n < 2^31", cudaSuccess);
    return SVB_ERR_ARG;
  }
  *bytes = svb::calib::layout(n).total;
  return SVB_OK;
}

extern "C" int svb_calib_metrics(const float* llr, const uint8_t* labels, int64_t n, const double* ops, int P,
                                 void* workspace, size_t workspace_bytes, double* out, void* stream) {
  return svb::calib::metrics(llr, labels, n, ops, P, workspace, workspace_bytes, out, stream);
}

extern "C" int svb_calib_train(const float* scores, const uint8_t* labels, int64_t n, double prior, int max_iter,
                               void* workspace, size_t workspace_bytes, double* out, void* stream) {
  return svb::calib::train(scores, labels, n, prior, max_iter, workspace, workspace_bytes, out, stream);
}
