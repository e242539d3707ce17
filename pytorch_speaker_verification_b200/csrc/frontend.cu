// Log-mel front end for sm_100a (SURVEY.md section 8(f) rank 4): PCM -> (nmels, T) log10 mel power spectrogram, the
// input format of the hot path.  Replaces data_preprocess.py:41-45 / dvector_create.py:43-47 of the reference
// (librosa.core.stft with center=True reflect padding, periodic Hann window zero-padded to n_fft; |.|^2;
// librosa.filters.mel; log10(. + 1e-6)).  PARITY UNPINNED: librosa is not available in the build container, the
// oracle (oracle/frontend.py) restates its documented algorithm.
//
// One CTA = 8 frames.  The 512-point real DFT is evaluated directly (thread = frequency bin): per sample one complex
// rotation of the thread's running twiddle (re-seeded from an exact table every 32 samples, so the recurrence error
// stays below 1e-6) and 2 FMAs per frame, all frames read as shared-memory broadcasts; 205 k MACs per frame is
// ~0.03 % of what the LSTM spends on the same frame, so an FFT would buy nothing.  Then the 40 x 257 mel projection
// and the log from shared memory.
//
// Two kernels share that body (logmel_body): logmel_kernel frames one signal (svb_logmel), logmel_frames_kernel
// frames the partial utterances of a TI-SV training set, each output row a run of frames of one segment with the
// reflect padding taken at the segment's own bounds (svb_logmel_frames, DESIGN.md 4.8).  Only the sample gather and
// the output address differ, so a frame gets the same bits from either.
#include "../../include/svb200.h"
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

namespace svb {
void set_error(const char* what, cudaError_t e);

constexpr int kFeNfft = 512, kFeBins = kFeNfft / 2 + 1, kFeFrames = 8, kFeThreads = 288, kFeReseed = 32;

// Windowed DFT power, mel projection and log of this CTA's n_valid (<= 8) frames.  sample(f, m): the signal sample
// under window position m of local frame f (f < n_valid, w0 <= m < w1); store(mel, f, v) writes one output value.
template <class Sample, class Store>
__device__ __forceinline__ void logmel_body(Sample sample, Store store, int n_valid, const float* __restrict__ win,
                                            int w0, int w1, const float2* __restrict__ tw,
                                            const float* __restrict__ melw, int nmels) {
  __shared__ float fr[kFeFrames][kFeNfft];          // windowed frames
  __shared__ float pw[kFeFrames][kFeBins + 3];      // power spectra
  for (int i = threadIdx.x; i < kFeFrames * kFeNfft; i += kFeThreads) {
    const int f = i / kFeNfft, m = i % kFeNfft;
    float v = 0.f;
    if (f < n_valid && m >= w0 && m < w1) v = sample(f, m) * win[m];
    fr[f][m] = v;
  }
  __syncthreads();
  const int k = threadIdx.x;
  if (k < kFeBins) {
    float re[kFeFrames], im[kFeFrames];
#pragma unroll
    for (int f = 0; f < kFeFrames; ++f) { re[f] = 0.f; im[f] = 0.f; }
    const float2 step = tw[k];                                     // exp(-2 pi i k / 512) as (cos, sin)
    float2 z = make_float2(1.f, 0.f);
    for (int m = w0; m < w1; ++m) {
      if (((m - w0) & (kFeReseed - 1)) == 0) z = tw[(k * m) & (kFeNfft - 1)];     // exact table value
#pragma unroll
      for (int f = 0; f < kFeFrames; ++f) {
        const float v = fr[f][m];
        re[f] = fmaf(v, z.x, re[f]);
        im[f] = fmaf(-v, z.y, im[f]);
      }
      // the roundings are spelled out (no compiler contraction), so that both kernels give svb_logmel's bits
      const float zx = fmaf(z.x, step.x, -__fmul_rn(z.y, step.y));
      z.y = fmaf(z.y, step.x, __fmul_rn(z.x, step.y));
      z.x = zx;
    }
#pragma unroll
    for (int f = 0; f < kFeFrames; ++f) pw[f][k] = fmaf(re[f], re[f], __fmul_rn(im[f], im[f]));
  }
  __syncthreads();
  for (int o = threadIdx.x; o < nmels * kFeFrames; o += kFeThreads) {
    const int mel = o / kFeFrames, f = o % kFeFrames;
    if (f >= n_valid) continue;
    const float* wrow = melw + (size_t)mel * kFeBins;
    float s = 0.f;
    for (int b = 0; b < kFeBins; ++b) s = fmaf(__ldg(wrow + b), pw[f][b], s);
    store(mel, f, log10f(s + 1e-6f));
  }
}

__global__ void __launch_bounds__(kFeThreads) logmel_kernel(const float* __restrict__ y, long long n, int n_frames, int hop,
                                                            const float* __restrict__ win, int w0, int w1,
                                                            const float2* __restrict__ tw, const float* __restrict__ melw,
                                                            int nmels, float* __restrict__ out) {
  const int t0 = blockIdx.x * kFeFrames;
  auto sample = [&](int f, int m) {
    long long idx = (long long)(t0 + f) * hop + m - kFeNfft / 2;   // center=True: frame t is centred on sample t*hop
    if (idx < 0) idx = -idx;                                       // reflect padding (no edge repeat)
    if (idx >= n) idx = 2 * (n - 1) - idx;
    if (idx < 0) idx = 0;
    return y[idx];
  };
  auto store = [&](int mel, int f, float v) { out[(size_t)mel * n_frames + t0 + f] = v; };
  logmel_body(sample, store, min(kFeFrames, n_frames - t0), win, w0, w1, tw, melw, nmels);
}

// rows (P, 3) int64: segment start in y, segment length L >= 1, first frame.  Output frame g = p * T + j is frame
// rows[p][2] + j of the segment; out (P, nmels, T).  The padding reflects without repeating the edge sample, repeatedly
// when the frame reaches beyond the segment by more than L - 1 samples (np.pad(mode="reflect")).
__global__ void __launch_bounds__(kFeThreads) logmel_frames_kernel(const float* __restrict__ y,
                                                                   const long long* __restrict__ rows, long long P,
                                                                   int T, int hop, const float* __restrict__ win,
                                                                   int w0, int w1, const float2* __restrict__ tw,
                                                                   const float* __restrict__ melw, int nmels,
                                                                   float* __restrict__ out) {
  __shared__ long long seg[kFeFrames][3];           // start, length, frame index of each local frame
  const long long g0 = (long long)blockIdx.x * kFeFrames, total = P * T;
  if (threadIdx.x < kFeFrames && g0 + threadIdx.x < total) {
    const long long g = g0 + threadIdx.x, p = g / T;
    seg[threadIdx.x][0] = rows[3 * p];
    seg[threadIdx.x][1] = rows[3 * p + 1];
    seg[threadIdx.x][2] = rows[3 * p + 2] + g % T;
  }
  __syncthreads();
  auto sample = [&](int f, int m) {
    const long long L = seg[f][1];
    long long idx = seg[f][2] * hop + m - kFeNfft / 2;
    if (idx < 0 || idx >= L) {
      const long long period = 2 * (L - 1);
      if (period == 0) {
        idx = 0;
      } else {
        idx = (idx < 0 ? -idx : idx) % period;
        if (idx >= L) idx = period - idx;
      }
    }
    return y[seg[f][0] + idx];
  };
  auto store = [&](int mel, int f, float v) {
    const long long g = g0 + f;
    out[((g / T) * nmels + mel) * T + g % T] = v;
  };
  logmel_body(sample, store, (int)min((long long)kFeFrames, total - g0), win, w0, w1, tw, melw, nmels);
}
}  // namespace svb
using namespace svb;

extern "C" int svb_logmel(const float* y, int64_t n, int hop, const float* window, int w0, int w1, const float* twiddle,
                          const float* mel_w, int nmels, float* out, int n_frames, void* stream) {
  if (n_frames == 0) return SVB_OK;
  if (!y || !window || !twiddle || !mel_w || !out || n < 1 || hop < 1 || nmels < 1 || n_frames < 0 || w0 < 0 ||
      w1 > kFeNfft || w0 >= w1) {
    set_error("svb_logmel: bad argument (n_fft is fixed at 512)", cudaSuccess);
    return SVB_ERR_ARG;
  }
  logmel_kernel<<<(n_frames + kFeFrames - 1) / kFeFrames, kFeThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      y, (long long)n, n_frames, hop, window, w0, w1, reinterpret_cast<const float2*>(twiddle), mel_w, nmels, out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("svb_logmel", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}

extern "C" int svb_logmel_frames(const float* y, const int64_t* rows, int64_t P, int frames_per_row, int hop,
                                 const float* window, int w0, int w1, const float* twiddle, const float* mel_w,
                                 int nmels, float* out, void* stream) {
  if (P < 0 || frames_per_row < 1 || hop < 1 || nmels < 1 || w0 < 0 || w1 > kFeNfft || w0 >= w1) {
    set_error("svb_logmel_frames: bad size (P >= 0, frames_per_row >= 1, hop >= 1, nmels >= 1, "
              "0 <= w0 < w1 <= 512)", cudaSuccess);
    return SVB_ERR_ARG;
  }
  if (P == 0) return SVB_OK;
  if (!y || !rows || !window || !twiddle || !mel_w || !out) {
    set_error("svb_logmel_frames: null pointer", cudaSuccess);
    return SVB_ERR_ARG;
  }
  if (P > ((long long)INT_MAX * kFeFrames) / frames_per_row) {
    set_error("svb_logmel_frames: P * frames_per_row too large", cudaSuccess);
    return SVB_ERR_ARG;
  }
  const long long blocks = (P * (long long)frames_per_row + kFeFrames - 1) / kFeFrames;
  logmel_frames_kernel<<<(unsigned)blocks, kFeThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      y, reinterpret_cast<const long long*>(rows), (long long)P, frames_per_row, hop, window, w0, w1,
      reinterpret_cast<const float2*>(twiddle), mel_w, nmels, out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("svb_logmel_frames", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}
