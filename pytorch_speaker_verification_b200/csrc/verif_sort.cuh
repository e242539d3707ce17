// The radix sort of verif.cu (DESIGN.md 4.5.1), shared with calib.cu: n scores with labels become uint64 elements
// (key << 1) | is_target, key the order-preserving uint32 image of the float (-0 counts as +0), sorted ascending by a
// key kernel and three LSD passes over 4096-element tiles.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace svb {
namespace verif {
constexpr int kDigitBits = 11;
constexpr int kBins = 1 << kDigitBits;                 // 2048
constexpr int kPasses = 3;                             // 33-bit elements

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortItems = 16;                         // per thread
constexpr int kSortTile = kSortThreads * kSortItems;   // 4096 elements

// hist (kPasses * kBins uint32) and counts (2 uint64) are adjacent, and the caller clears them before every sort
constexpr size_t kSortCounterBytes = kPasses * kBins * 4 + 2 * 8;

__device__ __forceinline__ uint32_t score_key(float x, unsigned& nonfinite) {
  uint32_t u = __float_as_uint(x);
  if (u == 0x80000000u) u = 0u;                        // -0 counts as +0 (bit test: denormals stay distinct)
  nonfinite += (u & 0x7f800000u) == 0x7f800000u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ double key_value(uint32_t key) {
  const uint32_t u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
  return (double)__uint_as_float(u);
}

// Exclusive scan of one value per thread over the block; returns the prefix, *total = the block's sum.
template <int kThreads>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* warp_tot, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  uint32_t before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    const uint32_t t = warp_tot[w];
    before += w < warp ? t : 0u;
    all += t;
  }
  __syncthreads();                                     // warp_tot may be reused by the caller's next scan
  *total = all;
  return before + incl - v;
}

struct SortBuffers {
  unsigned long long* a;       // n elements
  unsigned long long* b;       // n elements; holds the sorted elements afterwards
  uint32_t* offs;              // sort_table_bytes(n): per-tile digit counts / offsets
  uint32_t* hist;              // kPasses * kBins digit histograms, cleared by the caller
  unsigned long long* counts;  // [0] targets, [1] non-finite scores, cleared by the caller
};

inline int sort_tiles(int64_t n) { return (int)((n + kSortTile - 1) / kSortTile); }
inline size_t sort_table_bytes(int64_t n) { return (size_t)sort_tiles(n) * kBins * 4; }

// Enqueues the key kernel and the three passes on `st`.  Labels: `labels` (nonzero = target) or, with labels == NULL,
// the diagonal of a TI-SV matrix (N, Mv, N) with MvN = Mv * N.  Neither allocates nor synchronises.
cudaError_t sort_elements(const float* scores, const uint8_t* labels, int n, int N, int MvN, const SortBuffers& sb,
                          cudaStream_t st);
}  // namespace verif
}  // namespace svb
