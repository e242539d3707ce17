// Energy-based silence split of many PCM signals at once (librosa 0.6 effects.split with ref=np.max, frame_length 2048,
// hop_length 512; data_preprocess.py's `intervals = librosa.effects.split(utter, top_db=30)`), with the partial-utterance
// length filter of save_spectrogram_tisv.  Definitions in include/svb200.h and DESIGN.md 4.8.
//
// Two launches, no allocation, no synchronisation, no float atomics:
//   split_block_power_kernel: one warp per 512-sample block of a signal's reflect-padded copy writes the float64 sum
//     of its squares (lanes add 16 samples each in a fixed order, then a shuffle tree).  Frame t is the four blocks
//     t .. t+3, so every sample is read once although frames overlap four times.  Bound by the bytes of the samples.
//   split_select_kernel: one CTA per signal adds each frame's four block sums in a fixed order, takes the maximum, builds
//     the non-silent mask, finds the interval edges with a block-wide scan, writes the intervals into the signal's slot
//     range and compacts the ones at least min_len samples long in place.  A non-finite block sum (a non-finite
//     sample) makes the signal's count -1.
#include "../../include/svb200.h"
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace svb {
void set_error(const char* what, cudaError_t e);

namespace {
constexpr int kSpHop = 512, kSpPad = 1024, kSpWarps = 8, kSpThreads = 512;

// Workspace slot of signal i's first block: every signal owns 4 + (its length)/512 slots or more, which covers its
// 4 + n/512 padded blocks (n > 1024) or ceil(n/512) <= 2 raw blocks (n <= 1024).
__device__ __host__ __forceinline__ long long block_base(long long i, long long offset) { return 4 * i + offset / kSpHop; }

__device__ __forceinline__ long long n_blocks(long long n) {
  return n > kSpPad ? 4 + n / kSpHop : (n + kSpHop - 1) / kSpHop;
}

__global__ void __launch_bounds__(kSpWarps * 32) split_block_power_kernel(const float* __restrict__ y,
                                                                          const long long* __restrict__ offsets,
                                                                          int n_signals, long long n_slots,
                                                                          double* __restrict__ bsum) {
  const long long w = (long long)blockIdx.x * kSpWarps + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (w >= n_slots) return;
  int lo = 0, hi = n_signals - 1;                      // the last signal whose first slot is <= w
  while (lo < hi) {
    const int mid = (lo + hi + 1) / 2;
    if (block_base(mid, offsets[mid]) <= w) lo = mid; else hi = mid - 1;
  }
  const long long off = offsets[lo], n = offsets[lo + 1] - off, b = w - block_base(lo, off);
  if (b >= n_blocks(n)) return;
  const float* x = y + off;
  double s = 0.0;
  if (n > kSpPad) {
#pragma unroll 4
    for (int k = 0; k < kSpHop / 32; ++k) {
      long long idx = b * kSpHop + k * 32 + lane - kSpPad;          // np.pad(y, 1024, mode="reflect")
      if (idx < 0) idx = -idx;
      if (idx >= n) idx = 2 * (n - 1) - idx;
      const double v = x[idx];
      s = fma(v, v, s);                                             // exact square, one rounding of the sum
    }
  } else {
    for (int k = 0; k < kSpHop / 32; ++k) {
      const long long idx = b * kSpHop + k * 32 + lane;
      if (idx < n) { const double v = x[idx]; s = fma(v, v, s); }
    }
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) s += __shfl_down_sync(0xffffffffu, s, d);
  if (lane == 0) bsum[w] = s;
}

__device__ __forceinline__ double frame_power(const double* b, long long t) {
  return __dmul_rn(__dadd_rn(__dadd_rn(b[t], b[t + 1]), __dadd_rn(b[t + 2], b[t + 3])), 1.0 / 2048.0);
}

struct MaxOp {
  __device__ __forceinline__ double operator()(double a, double b) const { return a > b ? a : b; }
};

__global__ void __launch_bounds__(kSpThreads) split_select_kernel(const long long* __restrict__ offsets,
                                                                  const double* __restrict__ bsum, double top_db,
                                                                  long long min_len,
                                                                  const long long* __restrict__ slot_offsets,
                                                                  long long* __restrict__ intervals,
                                                                  long long* __restrict__ counts) {
  using Scan = cub::BlockScan<int, kSpThreads>;
  using Reduce = cub::BlockReduce<double, kSpThreads>;
  __shared__ union { typename Scan::TempStorage scan; typename Reduce::TempStorage reduce; } tmp;
  __shared__ double s_ref_db;
  __shared__ int s_carry;
  const int i = blockIdx.x, tid = threadIdx.x;
  const long long off = offsets[i], n = offsets[i + 1] - off;
  const double* b = bsum + block_base(i, off);
  const long long nb = n_blocks(n), F = n > kSpPad ? 1 + n / kSpHop : 0;

  int bad = 0;
  for (long long k = tid; k < nb; k += kSpThreads) bad |= !isfinite(b[k]);
  if (__syncthreads_or(bad)) {
    if (tid == 0) counts[i] = -1;
    return;
  }
  if (F == 0) {
    if (tid == 0) counts[i] = 0;
    return;
  }
  double pmax = 0.0;
  for (long long t = tid; t < F; t += kSpThreads) pmax = fmax(pmax, frame_power(b, t));
  pmax = Reduce(tmp.reduce).Reduce(pmax, MaxOp());
  if (tid == 0) { s_ref_db = __dmul_rn(10.0, log10(fmax(1e-10, pmax))); s_carry = 0; }
  __syncthreads();
  const double ref_db = s_ref_db, floor_db = -top_db;
  auto loud = [&](long long t) {
    // 10 log10(p) is rounded before the subtraction, as numpy does (a fused multiply-add would not round it, and the
    // loudest frame would come out a hair above 0 dB)
    return t >= 0 && t < F && __dsub_rn(__dmul_rn(10.0, log10(fmax(1e-10, frame_power(b, t)))), ref_db) > floor_db;
  };

  // Edges: the positions t in [0, F] where the mask changes (outside [0, F) it is silent); edge k is field k & 1 of
  // interval k / 2, at sample min(512 t, n).
  long long* out = intervals + 2 * slot_offsets[i];
  for (long long c = 0; c <= F; c += kSpThreads) {
    const long long t = c + tid;
    const int edge = t <= F && loud(t) != loud(t - 1);
    int pos, total;
    Scan(tmp.scan).ExclusiveSum(edge, pos, total);
    const int carry = s_carry;
    if (edge) out[carry + pos] = min(t * kSpHop, n);
    __syncthreads();
    if (tid == 0) s_carry = carry + total;
    __syncthreads();
  }
  const int n_int = s_carry / 2;
  if (min_len > 0) {                                   // keep the intervals of at least min_len samples, in order
    __syncthreads();
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int c = 0; c < n_int; c += kSpThreads) {
      const int j = c + tid;
      long long a = 0, e = 0;
      if (j < n_int) { a = out[2 * j]; e = out[2 * j + 1]; }
      const int keep = j < n_int && e - a >= min_len;
      int pos, total;
      Scan(tmp.scan).ExclusiveSum(keep, pos, total);
      const int carry = s_carry;
      __syncthreads();                                 // every read of this chunk precedes its writes
      if (keep) { out[2 * (carry + pos)] = a; out[2 * (carry + pos) + 1] = e; }
      __syncthreads();
      if (tid == 0) s_carry = carry + total;
      __syncthreads();
    }
    if (tid == 0) counts[i] = s_carry;
  } else if (tid == 0) {
    counts[i] = n_int;
  }
}

size_t workspace_bytes(int64_t total_samples, int n_signals) {
  return (size_t)block_base(n_signals, total_samples) * sizeof(double);
}
}  // namespace
}  // namespace svb
using namespace svb;

extern "C" int svb_split_workspace_bytes(int64_t total_samples, int n_signals, size_t* bytes) {
  if (total_samples < 0 || n_signals < 0 || !bytes) {
    set_error("svb_split_workspace_bytes: bad argument", cudaSuccess);
    return SVB_ERR_ARG;
  }
  *bytes = workspace_bytes(total_samples, n_signals);
  return SVB_OK;
}

extern "C" int svb_split_nonsilent(const float* y, const int64_t* offsets, int n_signals, int64_t total_samples,
                                   double top_db, int64_t min_len, const int64_t* slot_offsets, void* workspace,
                                   size_t workspace_bytes_, int64_t* intervals, int64_t* counts, void* stream) {
  if (n_signals < 0 || total_samples < 0 || min_len < 0 || isnan(top_db)) {
    set_error("svb_split_nonsilent: bad argument (n_signals >= 0, total_samples >= 0, min_len >= 0, top_db not NaN)",
              cudaSuccess);
    return SVB_ERR_ARG;
  }
  if (n_signals == 0) return SVB_OK;
  if (!y || !offsets || !slot_offsets || !workspace || !intervals || !counts) {
    set_error("svb_split_nonsilent: null pointer", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const size_t need = workspace_bytes(total_samples, n_signals);
  if (workspace_bytes_ < need || reinterpret_cast<uintptr_t>(workspace) % alignof(double) != 0) {
    set_error("svb_split_nonsilent: workspace smaller than svb_split_workspace_bytes or not 8-byte aligned",
              cudaSuccess);
    return SVB_ERR_ARG;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long n_slots = (long long)(need / sizeof(double));
  const auto* offs = reinterpret_cast<const long long*>(offsets);
  double* bsum = static_cast<double*>(workspace);
  if (n_slots > 0)
    split_block_power_kernel<<<(unsigned)((n_slots + kSpWarps - 1) / kSpWarps), kSpWarps * 32, 0, st>>>(
        y, offs, n_signals, n_slots, bsum);
  split_select_kernel<<<n_signals, kSpThreads, 0, st>>>(offs, bsum, top_db, (long long)min_len,
                                                        reinterpret_cast<const long long*>(slot_offsets),
                                                        reinterpret_cast<long long*>(intervals),
                                                        reinterpret_cast<long long*>(counts));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("svb_split_nonsilent", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}
