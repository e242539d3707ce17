// Exact EER and minDCF over every score threshold (DESIGN.md 4.5) for sm_100a.
//
// Every score becomes one uint64 element (key << 1) | is_target, key being the order-preserving uint32 image of the
// float.  An LSD radix sort of the 33-bit elements (three 11-bit digits, reduce-then-scan: per-tile digit counts, a
// scan of each digit's column over the tiles, a stable scatter) puts the scores in ascending order; a sweep over the
// sorted elements evaluates the integer EER criterion and every detection cost at the first element of each run of
// equal keys (the operating point that accepts that value and everything above it) and at the point that accepts
// nothing.  Every count is an integer and every float64 expression is rounded operation by operation (__dmul_rn /
// __dadd_rn / __ddiv_rn), so the result equals the float64 numpy restatement (tests/_verif_oracle.py) bit for bit and is
// run-to-run identical.
//
// Launches: key kernel (elements + the three digit histograms), three passes of count / scan / scatter
// (A -> B -> A -> B), sweep (target prefix by decoupled look-back; the last block reduces the per-tile arg-mins and
// writes `out`).  The entry points clear the counter region of the workspace with one cudaMemsetAsync and neither
// allocate nor synchronise, so a CUDA graph can capture them.  DESIGN.md 4.5.1 explains why the sort is not onesweep.
#include "../../include/svb200.h"
#include "perdev.cuh"
#include "verif_sort.cuh"
#include <cuda_runtime.h>
#include <math.h>
#include <algorithm>
#include <stdint.h>

namespace svb {
void set_error(const char* what, cudaError_t e);

namespace verif {
constexpr int kMaxPoints = 8;

constexpr int kKeyThreads = 512;

constexpr int kBinsPerThread = kBins / kSortThreads;   // 8

constexpr int kSweepThreads = 256;
constexpr int kSweepItems = 16;
constexpr int kSweepTile = kSweepThreads * kSweepItems;

// Look-back status word: 0 = not published, 1 .. kTile + 1 = the tile's own count + 1, kPrefix | c = inclusive prefix c
// (c < 2^31).  One 32-bit word holds flag and count, so a reader never sees one without the other.
constexpr uint32_t kPrefix = 0x80000000u;

struct Points {
  double w[kMaxPoints][3];     // w_miss, w_fa, c_def
  int P;
};

// Per-tile arg-min of the sweep: the value as uint64 bits (the EER criterion, or a non-negative double whose bit pattern
// orders like its value), the position and the target count below it.
struct Best {
  unsigned long long v;
  uint32_t pos, miss;
};

__device__ __forceinline__ bool better(const Best& a, const Best& b) {
  return a.v < b.v || (a.v == b.v && a.pos < b.pos);
}

__device__ __forceinline__ uint32_t digit_of(unsigned long long e, int shift) {
  return (uint32_t)(e >> shift) & (kBins - 1);
}

__device__ __forceinline__ uint32_t ld_volatile(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ void st_volatile(uint32_t* p, uint32_t v) { *reinterpret_cast<volatile uint32_t*>(p) = v; }

// ---------------------------------------------------------------------------------------------------- (a) key kernel
// counters[0] = targets, counters[1] = non-finite scores; hist[3][kBins] = digit histograms of the three passes.
// Labels: `labels` (flat form, nonzero = target) or, with labels == NULL, the diagonal of sim (N, Mv, N): element
// i = (j * Mv + m) * N + k is a target iff k == j.
__device__ __forceinline__ void key_one(float x, bool tgt, bool valid, unsigned long long* out, int i, uint32_t* h,
                                        unsigned& nt, unsigned& nf) {
  unsigned long long e = 0;
  uint32_t d2 = 0xffffffffu;
  if (valid) {
    const uint32_t key = score_key(x, nf);
    e = ((unsigned long long)key << 1) | (tgt ? 1ull : 0ull);
    nt += tgt;
    out[i] = e;
    atomicAdd(&h[digit_of(e, 0)], 1u);
    atomicAdd(&h[kBins + digit_of(e, kDigitBits)], 1u);
    d2 = digit_of(e, 2 * kDigitBits);
  }
  // the top digit (sign, exponent, two mantissa bits) takes few values for real scores: one shared atomic per distinct
  // value in the warp instead of up to 32 on one address
  const unsigned peers = __match_any_sync(0xffffffffu, d2);
  if (valid && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[2 * kBins + d2], (uint32_t)__popc(peers));
}

__global__ void __launch_bounds__(kKeyThreads) verif_key_kernel(const float* __restrict__ scores,
                                                                const uint8_t* __restrict__ labels, int n, int N,
                                                                int MvN, unsigned long long* __restrict__ elems,
                                                                uint32_t* __restrict__ ghist,
                                                                unsigned long long* __restrict__ counters) {
  __shared__ uint32_t h[kPasses * kBins];
  __shared__ unsigned red[2][kKeyThreads / 32];
  for (int b = threadIdx.x; b < kPasses * kBins; b += blockDim.x) h[b] = 0;
  __syncthreads();
  unsigned nt = 0, nf = 0;
  auto label = [&](int i) -> bool {
    return labels ? labels[i] != 0 : (i % N) == (i / MvN);
  };
  const bool vec = ((reinterpret_cast<uintptr_t>(scores) & 15) == 0) &&
                   (!labels || (reinterpret_cast<uintptr_t>(labels) & 3) == 0);
  const int stride = gridDim.x * blockDim.x;
  int tail0 = 0;
  if (vec) {
    const int nq = n >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(scores);
    // warp-uniform trip count: __match_any_sync in key_one needs the whole warp
    for (int q0 = blockIdx.x * blockDim.x; q0 < nq; q0 += stride) {
      const int q = q0 + threadIdx.x;
      const bool ok = q < nq;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      uint32_t lab = 0;
      if (ok) {
        v = __ldg(s4 + q);
        if (labels) {
          lab = __ldg(reinterpret_cast<const uint32_t*>(labels) + q);
        } else {
          const int i = 4 * q;
#pragma unroll
          for (int e = 0; e < 4; ++e) lab |= (uint32_t)label(i + e) << (8 * e);
        }
      }
      const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e)
        key_one(vv[e], ((lab >> (8 * e)) & 0xffu) != 0, ok, elems, 4 * q + e, h, nt, nf);
    }
    tail0 = nq << 2;
  }
  for (long long i0 = tail0 + (long long)blockIdx.x * blockDim.x; i0 < n; i0 += stride) {   // 64-bit: n < 2^31
    const bool ok = i0 + threadIdx.x < n;
    const int i = ok ? (int)(i0 + threadIdx.x) : 0;
    key_one(ok ? scores[i] : 0.f, ok && label(i), ok, elems, i, h, nt, nf);
  }
  // one integer atomic per block for each count
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    nt += __shfl_xor_sync(0xffffffffu, nt, o);
    nf += __shfl_xor_sync(0xffffffffu, nf, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = nt; red[1][threadIdx.x >> 5] = nf; }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long a = 0, b = 0;
    for (int w = 0; w < kKeyThreads / 32; ++w) { a += red[0][w]; b += red[1][w]; }
    if (a) atomicAdd(&counters[0], a);
    if (b) atomicAdd(&counters[1], b);
  }
  for (int b = threadIdx.x; b < kPasses * kBins; b += blockDim.x)
    if (h[b]) atomicAdd(&ghist[b], h[b]);
}

// ------------------------------------------------------------------------------------- (b) sort passes
// Reduce-then-scan per digit: count (per-tile digit counts), scan (every digit's column over the tiles, offset by the
// digit's global start from the key kernel's histogram), scatter (stable, one tile per CTA).  No CTA waits on another,
// so the passes run at the rate of their traffic whatever the number of tiles.

// counts[tile][d] = elements of the tile with digit d
__global__ void __launch_bounds__(kSortThreads) verif_count_kernel(const unsigned long long* __restrict__ src, int n,
                                                                   int shift, uint32_t* __restrict__ counts) {
  __shared__ uint32_t h[kBins];
  const int tid = threadIdx.x, lane = tid & 31;
  for (int b = tid; b < kBins; b += kSortThreads) h[b] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortTile;
  const int lim = n - base;                            // tile-local offsets below lim are elements (no int overflow)
  unsigned long long e[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const int i = r * kSortThreads + tid;
    e[r] = i < lim ? __ldg(src + base + i) : 0ull;
  }
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const bool ok = r * kSortThreads + tid < lim;
    const uint32_t d = ok ? digit_of(e[r], shift) : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, d);    // one shared atomic per distinct digit in the warp
    if (ok && lane == __ffs(peers) - 1) atomicAdd(&h[d], (uint32_t)__popc(peers));
  }
  __syncthreads();
  uint32_t* row = counts + (size_t)blockIdx.x * kBins;
  for (int b = tid; b < kBins; b += kSortThreads) row[b] = h[b];
}

// In place: counts[t][d] -> global position of tile t's first element with digit d = (elements with a smaller digit)
// + (elements with digit d in tiles < t).  One CTA per 8 digits (one 32-byte sector of every tile's row).
constexpr int kScanDigits = 8;
__global__ void __launch_bounds__(kSortThreads) verif_scan_kernel(uint32_t* __restrict__ counts, int T,
                                                                  const uint32_t* __restrict__ ghist) {
  __shared__ uint32_t wtot[kSortWarps][kScanDigits];
  __shared__ uint32_t red[kSortWarps];
  __shared__ uint32_t base_s[kScanDigits];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int d0 = blockIdx.x * kScanDigits;
  uint32_t below = 0;
  for (int i = tid; i < d0; i += kSortThreads) below += __ldg(ghist + i);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) below += __shfl_xor_sync(0xffffffffu, below, o);
  if (lane == 0) red[warp] = below;
  __syncthreads();
  if (tid == 0) {
    uint32_t b = 0;
    for (int w = 0; w < kSortWarps; ++w) b += red[w];
    for (int k = 0; k < kScanDigits; ++k) { base_s[k] = b; b += __ldg(ghist + d0 + k); }
  }
  __syncthreads();
  uint32_t carry[kScanDigits];
#pragma unroll
  for (int k = 0; k < kScanDigits; ++k) carry[k] = base_s[k];
  for (int t0 = 0; t0 < T; t0 += kSortThreads) {
    const int t = t0 + tid;
    uint4* p = reinterpret_cast<uint4*>(counts + (size_t)t * kBins + d0);
    uint4 a = make_uint4(0, 0, 0, 0), b = a;
    if (t < T) { a = p[0]; b = p[1]; }
    uint32_t v[kScanDigits] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}, incl[kScanDigits];
#pragma unroll
    for (int k = 0; k < kScanDigits; ++k) {
      incl[k] = v[k];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl[k], o);
        if (lane >= o) incl[k] += y;
      }
      if (lane == 31) wtot[warp][k] = incl[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kScanDigits; ++k) {
      uint32_t before = 0, all = 0;
#pragma unroll
      for (int w = 0; w < kSortWarps; ++w) {
        const uint32_t x = wtot[w][k];
        before += w < warp ? x : 0u;
        all += x;
      }
      v[k] = carry[k] + before + incl[k] - v[k];
      carry[k] += all;
    }
    if (t < T) {
      p[0] = make_uint4(v[0], v[1], v[2], v[3]);
      p[1] = make_uint4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();                                   // wtot is rewritten by the next chunk
  }
}

struct SortSmem {
  uint16_t whist[kSortWarps][kBins];   // per-warp digit counts, then the exclusive prefix over the earlier warps
  unsigned long long elems[kSortTile]; // the tile in tile-local sorted order
  int tile_excl[kBins];                // exclusive prefix of the tile's digit counts
  int gbase[kBins];                    // global position of tile-local position 0 of each digit's run
  uint32_t warp_tot[kSortWarps];
};

// One tile of kSortTile elements per CTA, stable in input order: warp w ranks elements [w * 32 * kItems, ...) of the
// tile, kItems rounds of 32 in order, with __match_any_sync; the tile is reordered by digit in shared memory and written
// to offs[tile][digit] (verif_scan_kernel) + its rank within the digit.
__global__ void __launch_bounds__(kSortThreads, 2) verif_scatter_kernel(const unsigned long long* __restrict__ src,
                                                                      unsigned long long* __restrict__ dst, int n,
                                                                      int shift, const uint32_t* __restrict__ offs) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SortSmem& s = *reinterpret_cast<SortSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  {
    uint4* z = reinterpret_cast<uint4*>(&s.whist[0][0]);
    for (int i = tid; i < (int)(sizeof(s.whist) / sizeof(uint4)); i += kSortThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  const int tile = blockIdx.x;
  const int base = tile * kSortTile;
  const int lim = n - base;                            // tile-local offsets below lim are elements (no int overflow)
  const int wbase = warp * 32 * kSortItems;            // tile-local
  const unsigned lt = (1u << lane) - 1u;

  unsigned long long e[kSortItems];
  uint16_t off[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const int i = wbase + r * 32 + lane;
    e[r] = i < lim ? __ldcs(src + base + i) : 0ull;
  }
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const bool ok = wbase + r * 32 + lane < lim;
    const uint32_t d = ok ? digit_of(e[r], shift) : (uint32_t)kBins;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int leader = __ffs(peers) - 1;
    uint32_t b = 0;
    if (ok && lane == leader) {
      b = s.whist[warp][d];
      s.whist[warp][d] = (uint16_t)(b + __popc(peers));
    }
    b = __shfl_sync(0xffffffffu, b, leader);
    off[r] = (uint16_t)(b + __popc(peers & lt));
    __syncwarp();
  }
  __syncthreads();

  // digits [kBinsPerThread * tid, + kBinsPerThread): prefix over the warps and the tile's counts
  const int d0 = tid * kBinsPerThread;
  uint32_t tot[kBinsPerThread], sum = 0;
#pragma unroll
  for (int j = 0; j < kBinsPerThread; ++j) {
    uint32_t run = 0;
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
      const uint32_t c = s.whist[w][d0 + j];
      s.whist[w][d0 + j] = (uint16_t)run;
      run += c;
    }
    tot[j] = run;
    sum += run;
  }
  uint32_t tile_all;
  uint32_t texcl = block_excl_scan<kSortThreads>(sum, s.warp_tot, &tile_all);
  const uint4* o4 = reinterpret_cast<const uint4*>(offs + (size_t)tile * kBins + d0);
  const uint4 oa = __ldg(o4), ob = __ldg(o4 + 1);
  const uint32_t go[kBinsPerThread] = {oa.x, oa.y, oa.z, oa.w, ob.x, ob.y, ob.z, ob.w};
#pragma unroll
  for (int j = 0; j < kBinsPerThread; ++j) {
    s.tile_excl[d0 + j] = (int)texcl;
    s.gbase[d0 + j] = (int)go[j] - (int)texcl;
    texcl += tot[j];
  }
  __syncthreads();

#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    if (wbase + r * 32 + lane < lim) {
      const uint32_t d = digit_of(e[r], shift);
      s.elems[s.tile_excl[d] + s.whist[warp][d] + off[r]] = e[r];
    }
  }
  __syncthreads();
  const int cnt = min(kSortTile, lim);
  for (int i = tid; i < cnt; i += kSortThreads) {
    const unsigned long long x = s.elems[i];
    dst[s.gbase[digit_of(x, shift)] + i] = x;
  }
}

// ---------------------------------------------------------------------------------------------------- (c) sweep
__device__ __forceinline__ Best warp_min(Best b) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    Best y;
    y.v = __shfl_xor_sync(0xffffffffu, b.v, o);
    y.pos = __shfl_xor_sync(0xffffffffu, b.pos, o);
    y.miss = __shfl_xor_sync(0xffffffffu, b.miss, o);
    if (better(y, b)) b = y;
  }
  return b;
}

// lexicographic (value, position) minimum over the block; valid in thread 0
template <int kThreads>
__device__ __forceinline__ Best block_min(Best b, Best* scratch) {
  b = warp_min(b);
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = b;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w)
      if (better(scratch[w], b)) b = scratch[w];
  }
  __syncthreads();
  return b;
}

__device__ __forceinline__ double dcf_of(const Points& pt, int p, double pm, double pf) {
  return __ddiv_rn(__dadd_rn(__dmul_rn(pt.w[p][0], pm), __dmul_rn(pt.w[p][1], pf)), pt.w[p][2]);
}

// Tile results (not cleared between calls: every tile writes its slots before the last block reads them):
// best[tile * (1 + kMaxPoints) + 0] the EER criterion, + 1 + p the cost of point p; groups[tile] = distinct values that
// start in the tile.
__global__ void __launch_bounds__(kSweepThreads) verif_sweep_kernel(const unsigned long long* __restrict__ sorted,
                                                                    int n, const unsigned long long* __restrict__ counters,
                                                                    uint32_t* __restrict__ status,
                                                                    unsigned* __restrict__ tickets,
                                                                    Best* __restrict__ best,
                                                                    uint32_t* __restrict__ groups, Points pt,
                                                                    double* __restrict__ out) {
  __shared__ uint32_t warp_tot[kSweepThreads / 32];
  __shared__ Best scratch[kSweepThreads / 32];
  __shared__ uint32_t s_tile, s_prefix, s_groups[kSweepThreads / 32];
  __shared__ int s_last;
  const int tid = threadIdx.x;
  if (tid == 0) s_tile = atomicAdd(&tickets[0], 1u);
  __syncthreads();
  const int tile = (int)s_tile;
  const int ntiles = (n - 1) / kSweepTile + 1;
  const uint32_t Nt = (uint32_t)__ldcg(counters);
  const uint32_t Nn = (uint32_t)n - Nt;
  const double dNt = (double)Nt, dNn = (double)Nn;

  // blocked arrangement: the thread's kItems consecutive elements and the one before them
  // tile-local offsets are compared with lim, so no index passes 2^31
  const int lim = n - tile * kSweepTile;
  const int lp = tid * kSweepItems;
  const unsigned long long* my = sorted + (size_t)tile * kSweepTile + lp;
  unsigned long long e[kSweepItems];
#pragma unroll
  for (int j = 0; j < kSweepItems; j += 2) {
    if (lp + j + 1 < lim) {
      const ulonglong2 v = __ldcs(reinterpret_cast<const ulonglong2*>(my + j));
      e[j] = v.x; e[j + 1] = v.y;
    } else {
      e[j] = lp + j < lim ? my[j] : 0ull;
      e[j + 1] = 0ull;
    }
  }
  const bool first = tile == 0 && tid == 0;
  unsigned long long prev = (!first && lp < lim) ? my[-1] : ~0ull;   // ~0: no predecessor (key differs)
  uint32_t mine = 0;
#pragma unroll
  for (int j = 0; j < kSweepItems; ++j) mine += (lp + j < lim) ? (uint32_t)(e[j] & 1ull) : 0u;

  uint32_t tile_tgt;
  const uint32_t before = block_excl_scan<kSweepThreads>(mine, warp_tot, &tile_tgt);
  if (tid < 32) {            // decoupled look-back over the earlier tiles' target counts, 32 tiles per step (one a lane)
    const int lane = tid;
    uint32_t excl = 0;
    if (tile == 0) {
      if (lane == 0) st_volatile(status, kPrefix | tile_tgt);
    } else {
      if (lane == 0) st_volatile(status + tile, tile_tgt + 1u);
      for (int p = tile - 1;;) {                       // window: lane l reads tile p - l
        const int idx = p - lane;
        const uint32_t st = idx >= 0 ? ld_volatile(status + idx) : kPrefix;
        const unsigned inc = __ballot_sync(0xffffffffu, (st & kPrefix) != 0);
        const unsigned zero = __ballot_sync(0xffffffffu, st == 0);
        const unsigned upto = inc ? ((inc & (0u - inc)) | ((inc & (0u - inc)) - 1u)) : 0xffffffffu;
        if (zero & upto) continue;                     // a nearer tile has not published yet: poll the window again
        uint32_t v = ((upto >> lane) & 1u) ? ((st & kPrefix) ? (st & ~kPrefix) : st - 1u) : 0u;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        excl += v;
        if (inc) break;
        p -= 32;
      }
      if (lane == 0) st_volatile(status + tile, kPrefix | (excl + tile_tgt));
    }
    if (lane == 0) s_prefix = excl;
  }
  __syncthreads();

  Best b[1 + kMaxPoints];
#pragma unroll
  for (int q = 0; q <= kMaxPoints; ++q) { b[q].v = ~0ull; b[q].pos = 0xffffffffu; b[q].miss = 0; }
  uint32_t miss = s_prefix + before, ngroups = 0;
  auto eval = [&](uint32_t pos, uint32_t m) {
    const uint32_t fa = Nn - (pos - m);
    const unsigned long long a = (unsigned long long)m * Nn, c = (unsigned long long)fa * Nt;
    const Best cand{a > c ? a - c : c - a, pos, m};
    if (better(cand, b[0])) b[0] = cand;
    const double pm = __ddiv_rn((double)m, dNt), pf = __ddiv_rn((double)fa, dNn);
#pragma unroll
    for (int q = 0; q < kMaxPoints; ++q) {
      if (q < pt.P) {
        const Best cq{(unsigned long long)__double_as_longlong(dcf_of(pt, q, pm, pf)), pos, m};
        if (better(cq, b[1 + q])) b[1 + q] = cq;
      }
    }
  };
#pragma unroll
  for (int j = 0; j < kSweepItems; ++j) {
    if (lp + j < lim) {
      if ((e[j] >> 1) != (prev >> 1) || (first && j == 0)) {   // a group start: "accept >= this value"
        ++ngroups;
        eval((uint32_t)(tile * kSweepTile + lp + j), miss);
      }
      miss += (uint32_t)(e[j] & 1ull);
      prev = e[j];
    }
  }
  if (tile == ntiles - 1 && tid == kSweepThreads - 1) eval((uint32_t)n, Nt);   // point K: accept nothing

#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) ngroups += __shfl_xor_sync(0xffffffffu, ngroups, o);
  if ((tid & 31) == 0) s_groups[tid >> 5] = ngroups;
  Best* tb = best + (size_t)tile * (1 + kMaxPoints);
#pragma unroll
  for (int q = 0; q <= kMaxPoints; ++q) {
    if (q <= pt.P) {
      const Best r = block_min<kSweepThreads>(b[q], scratch);
      if (tid == 0) tb[q] = r;
    }
  }
  if (tid == 0) {
    uint32_t g = 0;
    for (int w = 0; w < kSweepThreads / 32; ++w) g += s_groups[w];
    groups[tile] = g;
    __threadfence();
    s_last = atomicAdd(&tickets[1], 1u) == (unsigned)ntiles - 1u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();

  // last block: (value, position) minimum over the tiles for every metric; the position is the operating point
  unsigned long long K = 0;
  for (int t = tid; t < ntiles; t += kSweepThreads) K += __ldcg(groups + t);
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) K += __shfl_xor_sync(0xffffffffu, K, o);
  __shared__ unsigned long long s_k[kSweepThreads / 32];
  if ((tid & 31) == 0) s_k[tid >> 5] = K;
  const unsigned long long nonfinite = __ldcg(counters + 1);
  const bool bad = nonfinite != 0 || Nt == 0 || Nn == 0;
  const double qnan = __longlong_as_double(0x7ff8000000000000ll);
  auto emit = [&](double* o, const Best& r) {          // value, threshold, p_miss, p_fa of the point at position pos
    const uint32_t fa = Nn - (r.pos - r.miss);
    const double thr = r.pos >= (uint32_t)n ? (double)INFINITY : key_value((uint32_t)(__ldcg(sorted + r.pos) >> 1));
    o[1] = bad ? qnan : thr;
    o[2] = bad ? qnan : __ddiv_rn((double)r.miss, dNt);
    o[3] = bad ? qnan : __ddiv_rn((double)fa, dNn);
  };
  for (int q = 0; q <= pt.P; ++q) {
    Best r;
    r.v = ~0ull; r.pos = 0xffffffffu; r.miss = 0;
    for (int t = tid; t < ntiles; t += kSweepThreads) {
      const Best* x = best + (size_t)t * (1 + kMaxPoints) + q;
      Best y;
      y.v = __ldcg(&x->v);
      y.pos = __ldcg(&x->pos);
      y.miss = __ldcg(&x->miss);
      if (better(y, r)) r = y;
    }
    r = block_min<kSweepThreads>(r, scratch);
    if (tid == 0) {
      double* o = q == 0 ? out : out + 8 + 4 * (q - 1);
      emit(o, r);
      if (q == 0) {
        o[0] = bad ? qnan : __ddiv_rn(__dadd_rn(o[2], o[3]), 2.0);
      } else {
        o[0] = bad ? qnan : __longlong_as_double((long long)r.v);
      }
    }
  }
  if (tid == 0) {
    unsigned long long k = 0;
    for (int w = 0; w < kSweepThreads / 32; ++w) k += s_k[w];
    out[4] = (double)Nt;
    out[5] = (double)Nn;
    out[6] = (double)nonfinite;
    out[7] = (double)k;
  }
}

// ---------------------------------------------------------------------------------------------------- host side
inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

// Workspace: elements A and B (8n bytes each); the per-tile digit counts / offsets of the sort passes (8 KB per
// 4096-score tile, 2 B a score, fully rewritten by every pass); the counter region cleared by every call (24 KB of digit
// histograms, the two counts and the tickets, then one sweep status word per 4096-score tile); the sweep's per-tile
// results (148 B per 4096-score tile, written before they are read).
struct Layout {
  size_t a, b, offs, ctr, hist, counts, tickets, sweep_status, ctr_bytes, best, groups, total;
  int sort_tiles, sweep_tiles;
};

inline Layout layout(int64_t n) {
  Layout L;
  L.sort_tiles = (int)((n + kSortTile - 1) / kSortTile);
  L.sweep_tiles = (int)((n + kSweepTile - 1) / kSweepTile);
  L.a = 0;
  L.b = align_up(8 * (size_t)n);
  L.offs = L.b + align_up(8 * (size_t)n);
  L.ctr = L.offs + align_up((size_t)L.sort_tiles * kBins * 4);
  L.hist = L.ctr;
  L.counts = L.hist + kPasses * kBins * 4;
  L.tickets = L.counts + 2 * 8;                        // [0] sweep tiles, [1] sweep done
  L.sweep_status = L.tickets + 8 * 4;
  L.ctr_bytes = L.sweep_status + (size_t)L.sweep_tiles * 4 - L.ctr;
  L.best = L.ctr + align_up(L.ctr_bytes);
  L.groups = L.best + align_up((size_t)L.sweep_tiles * (1 + kMaxPoints) * sizeof(Best));
  L.total = L.groups + align_up((size_t)L.sweep_tiles * 4);
  return L;
}

inline bool n_ok(int64_t n) { return n >= 2 && n < (int64_t(1) << 31); }

// After three passes (A -> B -> A -> B) the sorted elements are in B.
cudaError_t sort_elements(const float* scores, const uint8_t* labels, int n, int N, int MvN, const SortBuffers& sb,
                          cudaStream_t st) {
  static unsigned long long attr_done = 0;
  if (first_use_on_device(attr_done)) {
    const cudaError_t e = cudaFuncSetAttribute(verif_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)sizeof(SortSmem));
    if (e != cudaSuccess) { attr_done = 0; return e; }
  }
  const int tiles = sort_tiles(n);
  const int key_blocks = (int)std::min<int64_t>(2 * device_sm_count(), ((int64_t)n + 4 * kKeyThreads - 1) / (4 * kKeyThreads));
  verif_key_kernel<<<std::max(key_blocks, 1), kKeyThreads, 0, st>>>(scores, labels, n, N, MvN, sb.a, sb.hist, sb.counts);
  unsigned long long* src = sb.a;
  unsigned long long* dst = sb.b;
  for (int p = 0; p < kPasses; ++p) {
    verif_count_kernel<<<tiles, kSortThreads, 0, st>>>(src, n, p * kDigitBits, sb.offs);
    verif_scan_kernel<<<kBins / kScanDigits, kSortThreads, 0, st>>>(sb.offs, tiles, sb.hist + p * kBins);
    verif_scatter_kernel<<<tiles, kSortThreads, sizeof(SortSmem), st>>>(src, dst, n, p * kDigitBits, sb.offs);
    std::swap(src, dst);
  }
  return cudaGetLastError();
}

int run(const float* scores, const uint8_t* labels, int64_t n64, int N, int MvN, const double* ops, int P,
        void* workspace, size_t workspace_bytes, double* out, void* stream, const char* who) {
  if (!scores || !ops || !workspace || !out || !n_ok(n64) || P < 1 || P > kMaxPoints) {
    set_error(who, cudaSuccess);
    return SVB_ERR_ARG;
  }
  Points pt;
  pt.P = P;
  for (int p = 0; p < P; ++p) {
    for (int c = 0; c < 3; ++c) pt.w[p][c] = ops[3 * p + c];
    if (!(pt.w[p][0] > 0.0) || !(pt.w[p][1] > 0.0) || !(pt.w[p][2] > 0.0) || !isfinite(pt.w[p][0]) ||
        !isfinite(pt.w[p][1]) || !isfinite(pt.w[p][2])) {
      set_error(who, cudaSuccess);
      return SVB_ERR_ARG;
    }
  }
  for (int p = P; p < kMaxPoints; ++p) pt.w[p][0] = pt.w[p][1] = pt.w[p][2] = 1.0;
  const int n = (int)n64;
  const Layout L = layout(n64);
  if (workspace_bytes < L.total || (reinterpret_cast<uintptr_t>(workspace) & 255)) {
    set_error(who, cudaSuccess);
    return SVB_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  SortBuffers sb;
  sb.a = reinterpret_cast<unsigned long long*>(ws + L.a);
  sb.b = reinterpret_cast<unsigned long long*>(ws + L.b);
  sb.offs = reinterpret_cast<uint32_t*>(ws + L.offs);
  sb.hist = reinterpret_cast<uint32_t*>(ws + L.hist);
  sb.counts = reinterpret_cast<unsigned long long*>(ws + L.counts);
  auto* tickets = reinterpret_cast<unsigned*>(ws + L.tickets);
  auto* sweep_status = reinterpret_cast<uint32_t*>(ws + L.sweep_status);

  cudaError_t e = cudaMemsetAsync(ws + L.ctr, 0, L.ctr_bytes, st);
  if (e == cudaSuccess) e = sort_elements(scores, labels, n, N, MvN, sb, st);
  if (e != cudaSuccess) { set_error(who, e); return SVB_ERR_CUDA; }
  verif_sweep_kernel<<<L.sweep_tiles, kSweepThreads, 0, st>>>(sb.b, n, sb.counts, sweep_status, tickets,
                                                              reinterpret_cast<Best*>(ws + L.best),
                                                              reinterpret_cast<uint32_t*>(ws + L.groups), pt, out);
  e = cudaGetLastError();
  if (e != cudaSuccess) { set_error(who, e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

}  // namespace verif
}  // namespace svb

extern "C" int svb_verif_workspace_bytes(int64_t n, size_t* bytes) {
  if (!bytes || !svb::verif::n_ok(n)) {
    svb::set_error("svb_verif_workspace_bytes: need 2 <= n < 2^31", cudaSuccess);
    return SVB_ERR_ARG;
  }
  *bytes = svb::verif::layout(n).total;
  return SVB_OK;
}

extern "C" int svb_verif_metrics(const float* scores, const uint8_t* labels, int64_t n, const double* ops, int P,
                                 void* workspace, size_t workspace_bytes, double* out, void* stream) {
  if (!labels) {
    svb::set_error("svb_verif_metrics: labels is NULL", cudaSuccess);
    return SVB_ERR_ARG;
  }
  return svb::verif::run(scores, labels, n, 1, 1, ops, P, workspace, workspace_bytes, out, stream,
                         "svb_verif_metrics: bad argument (2 <= n < 2^31, 1 <= P <= 8, positive finite weights, "
                         "workspace of svb_verif_workspace_bytes, 256-byte aligned)");
}

extern "C" int svb_verif_metrics_sim(const float* sim, int N, int Mv, const double* ops, int P, void* workspace,
                                     size_t workspace_bytes, double* out, void* stream) {
  if (N < 2 || Mv < 1) {
    svb::set_error("svb_verif_metrics_sim: need N >= 2 and Mv >= 1", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const int64_t n = (int64_t)N * Mv * N;
  if (!svb::verif::n_ok(n)) {
    svb::set_error("svb_verif_metrics_sim: N * Mv * N must be below 2^31", cudaSuccess);
    return SVB_ERR_ARG;
  }
  return svb::verif::run(sim, nullptr, n, N, Mv * N, ops, P, workspace, workspace_bytes, out, stream,
                         "svb_verif_metrics_sim: bad argument (1 <= P <= 8, positive finite weights, workspace of "
                         "svb_verif_workspace_bytes, 256-byte aligned)");
}
