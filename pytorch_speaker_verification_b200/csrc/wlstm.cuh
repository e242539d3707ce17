// Persistent wavefront LSTM forward kernel: weights stationary in TENSOR MEMORY (included by lstm.cu, namespace svb).
//
// Replaces, for the whole stack at once, nn.LSTM's forward (speech_embedder_net.py:19,28): one launch runs all T
// frames of all L layers.  2*L*(H/32) CTAs (144 at L=3, H=768), one per SM, two roles:
//
//   R(l, n)  recurrence of layer l, gate-column slice n (128 packed gate columns = 32 hidden units x 4 gates):
//            W_hh[slice] (128 x H fp16 = 192 KB at H=768) is loaded ONCE into tensor memory as the A operand of
//            tcgen05.mma (TS form).  Per frame t and 64-row batch tile j the CTA streams h^l_{t-1}[tile j] (K-major
//            fp16, TMA -> 128B-swizzled smem ring) as the B operand, so the accumulator is TRANSPOSED:
//            D[gate column (TMEM lane), batch row (TMEM column)].  Epilogue: + gin (from P(l, n)), sigma/tanh of the
//            thread's own gate column, a 4x4 register transpose across the four gate lanes of a unit (shuffles),
//            the cell update, and TMA stores of h_t (fp16 + bf16), c_t and the gate stash for BPTT.
//   P(l, n)  input projection of layer l, same slice: W_ih[slice] resident in tensor memory, streams
//            x_t (l = 0) or h^{l-1}_t (l > 0), writes gin = W_ih x + b_ih + b_hh (fp32) to a small L2-resident ring in
//            the epilogue's own fragment order (coalesced 16-byte stores/loads, no staging).
//
// Nothing is re-read per frame except the activations themselves: per frame a CTA pulls B*K*2 bytes (0.98 MB) and
// no weights, where the per-frame kernels pulled 393 KB of W_hh per 128x128 tile per frame (L2-throughput bound).
// Shared memory is free for a deep operand ring and double-buffered TMA staging.
//
// Ordering is by monotonically increasing counters in global memory (release/acquire at gpu scope), no grid barrier:
//   hcnt[l][j]     += 1 by every R(l, .) after its stores of (t, j) completed  -> h^l_t[tile j] complete at NS*(t+1)
//   gcnt[l][n][j]   = t+1 by P(l, n) after gin of (t, j) is written
// R(l,t,j) waits hcnt[l][j] >= NS*t and gcnt[l][n][j] >= t+1; P(l,t,j) waits hcnt[l-1][j] >= NS*(t+1) and (ring
// back-pressure) hcnt[l][j] >= NS*(t-D+1).  The dependency graph is acyclic in (t, l) and all CTAs are co-resident
// (cooperative launch), so the layers form a self-timed wavefront: layer l runs frame t while layer l+1 runs t-1.
// TMEM map (512 columns): [0, K/2) = weights, two fp16 per column; [384, 448) and [448, 512) = two accumulators.
// So K <= 768 (in 64-wide blocks): H <= 768, and nmels <= 768 for layer 0 (svb_embedder_forward checks it).
#pragma once

constexpr int kWlTile = 64;            // batch rows per tile (= MMA N)
// 64-wide K blocks per ring stage.  An mbarrier try_wait costs ~170 cycles even when the phase is already complete
// (scripts/ubench/mma_issue.cu: hidden behind queued MMAs in isolation, but visible as tensor-pipe bubbles in this
// kernel, where four epilogue warps share the issuer's scheduler), so waits are rare: 6 K blocks = 24 MMAs of N = 64
// (768 cycles of tensor work) per wait.
#ifdef SVB_WL_RING_ALT                 // experiment (make ALT=1): finer stages, same bytes
constexpr int kWlKbPerStage = 3;
constexpr int kWlStages = 6;
#else
constexpr int kWlKbPerStage = 6;
constexpr int kWlStages = 3;           // operand ring: 3 x 6 x [64 rows x 64 K] fp16 = 144 KB (1.5 tiles in flight)
#endif
constexpr int kWlKbBytes = kWlTile * 128;
constexpr int kWlStageBytes = kWlKbPerStage * kWlKbBytes;
constexpr int kWlGinRing = 3;          // frames of gin kept in flight per layer
constexpr int kWlChunk = 16;           // tile order: chunks of 16 tiles, frame-major inside a chunk (see WL_FOR_TILES)
#ifdef SVB_LAG_ALT
constexpr int kWlGinLagMax = 1 << 20;  // experiment: frame-granular back-pressure only (3 frames)
#else
constexpr int kWlGinLagMax = 24;       // ... and at most this many tiles (24 x 24 slices x 32 KB = 18 MB per layer: L2-resident)
#endif
#ifdef SVB_DEPS_ALT
constexpr int kWlDeps = 8;
#else
constexpr int kWlDeps = 4;             // tiles the dependency poller may run ahead
#endif
constexpr int kWlEpiWarps = 16;        // four warps per TMEM lane quarter, 16 batch rows of the tile each
// Warps 0..15 epilogue, 16 TMA producer, 17 MMA issuer, 18 store/signal, 19 dependency poller.  The single-thread
// roles get the HIGHEST warp ids: the SM sub-partition arbiter prefers the highest warp id among eligible warps, and
// as warp 1 the MMA issuer starved behind the four MUFU-heavy epilogue warps of its sub-partition (94 instead of 32
// cycles per tcgen05.mma, tensor pipe 31 % busy).
constexpr int kWlThreads = 32 * kWlEpiWarps + 128;
constexpr int kWlWarpTma = kWlEpiWarps, kWlWarpMma = kWlEpiWarps + 1, kWlWarpStore = kWlEpiWarps + 2,
              kWlWarpPoll = kWlEpiWarps + 3;   // lane 0: dependency poller, lane 1: c tile loader
constexpr int kWlAccCol = 384;
// staging buffer (per accumulator buffer): c tile (in place), h fp16, h bf16, two gate boxes
constexpr int kWlOffC = 0, kWlOffH16 = 8192, kWlOffHbf = 12288, kWlOffG = 16384, kWlStgBytes = 32768;
constexpr int kWlCinBytes = 8192;      // c_{t-1} tile, loaded ahead of time (double-buffered)
constexpr int kWlSmem = kWlStages * kWlStageBytes + 2 * kWlStgBytes + 2 * kWlCinBytes + 1024 + 1024;

struct __align__(64) WlstmLayer {
  CUtensorMap t_in;        // B operand of P: fp16 x [T][B][Ip] (l = 0) or h^{l-1} [T+1][B][H]; box {64, 64} SW128
  CUtensorMap t_h;         // B operand of R: fp16 h^l [T+1][B][H]; box {64, 64} SW128
  CUtensorMap t_h16_st;    // store h^l fp16, box {32, 64}, no swizzle
  CUtensorMap t_hbf_st;    // store h^l bf16 (training)
  CUtensorMap t_c;         // fp32 c [cslots][B][H], box {32, 64} SW128, load + store
  CUtensorMap t_gates;     // bf16 gates [T+1][B][4H], box {64, 64} SW128, store (training)
  const __half* whh;       // packed [4H][H]
  const __half* wih;       // packed [4H][Ip]
  const float* bias;       // packed [4H]
  float* gin;              // ring [kWlGinRing][nt][NS][64 x 128] fp32, fragment order
  int Ip;                  // K of the input projection (row pitch of wih)
  int in_slab0;            // slab of t_in that holds frame 0 (0 for x, 1 for h of the layer below)
};
struct __align__(64) WlstmParams {
  WlstmLayer layer[3];
  unsigned* hcnt;          // [L][nt]
  unsigned* gcnt;          // [L][NS][nt]
  float* h_last;           // [B][H] fp32: top layer, last frame
  long long* trace;        // debug: clock64 stamps of R(1,0) and P(1,0) at frame T/2 ([2][nt][16]), or null
  int B, T, L, H, nt, training;
  int ablate;              // debug: 1 skip MMAs, 2 skip epilogue math, 4 skip operand loads (results are garbage)
  int trace_mode;          // 1: per-tile stamps of frame T/2 (perturbs the traced CTAs); 2: wait accounting only
};
#define WL_STAMP(slot) do { if (tr) tr[(slot)] = clock64(); } while (0)
// wait accounting (debug; compile with -DSVB_WL_ACCOUNT and set trace_mode 2): cycles a role thread spends in a
// statement, accumulated in a register.  Off by default: the accumulators cost the epilogue warps registers (spills).
#ifdef SVB_WL_ACCOUNT
#define WL_ACC(var, ...) do { if (acct) { const long long a0_ = clock64(); __VA_ARGS__; var += clock64() - a0_; } else { __VA_ARGS__; } } while (0)
#else
#define WL_ACC(var, ...) do { __VA_ARGS__; } while (0)
#endif

// vector shared-memory accesses by 32-bit address (explicit LDS/STS: pointers derived from the aligned dynamic-smem base
// lose their address space and compile to generic LD/ST)
__device__ __forceinline__ uint4 lds_u4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float2 half2_to_float2(uint32_t h) {
  return __half22float2(*reinterpret_cast<const __half2*>(&h));
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts_u4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint2 lds_u2(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u2(uint32_t addr, uint2 v) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(v.x), "r"(v.y) : "memory");
}

__device__ __forceinline__ void red_release_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_relaxed_add(unsigned* p, unsigned v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed(unsigned* p, unsigned v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_relaxed(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
// Spin until *a >= ta and *b >= tb (null pointer = no condition); both loads are in flight together.  Bounded: a lost
// arrival traps instead of hanging the GPU.
// NO acquire / proxy fence follows on purpose.  Everything that is read after the flag bypasses L1 (TMA loads and
// ld.global.cg go to L2, the point of coherence) and is issued only after the flag value has come back (the poller
// arrives on an mbarrier that the consumers wait on), and the writers release their data at gpu scope before raising
// the flag (TMA stores: cp.async.bulk.wait_group + red.release; gin: fence.acq_rel.gpu in every writing thread).
// fence.acq_rel.gpu and fence.proxy.async cost ~1000 cycles EACH here and made this loop (3 fences per tile) the
// limiter of the whole kernel: 2.2 us per tile with all math, loads and stores switched off.  The poisoned-workspace
// stress test guards this protocol.
__device__ __forceinline__ void wait_two_counters(const unsigned* a, unsigned ta, const unsigned* b, unsigned tb) {
  long long t0 = 0;
  while (true) {
    const unsigned va = a ? ld_relaxed(a) : ta;
    const unsigned vb = b ? ld_relaxed(b) : tb;
    if (va >= ta && vb >= tb) break;
    if (t0 == 0) t0 = clock64();
    else if (clock64() - t0 > 4000000000LL) {
      printf("svb: wlstm dependency timeout cta %d have (%u, %u) want (%u, %u)\n", blockIdx.x, va, vb, ta, tb);
      __trap();
    }
  }
}

// Tile order of every role: the batch tiles are walked in chunks of kWlChunk, all T frames of a chunk before the next
// chunk (a tail shorter than half a chunk is merged into the last one).  The dependencies are per tile, so any order
// that keeps t ascending per tile is valid; this one keeps the live h / c / gin rows of a chunk in L2 when the batch
// is large (extraction, EER: hundreds of tiles per frame ran 10 % slower per tile in plain frame-major order) and is
// the plain frame-major order for nt <= 23.  `it` counts tiles in this order.
__device__ __forceinline__ int wl_chunk_end(int jc, int nt) {
  return (nt - (jc + kWlChunk) < kWlChunk / 2) ? nt : jc + kWlChunk;
}
#define WL_FOR_TILES(t, j, it)                                            \
  for (int jc_ = 0, je_ = wl_chunk_end(0, nt); jc_ < nt; jc_ = je_, je_ = wl_chunk_end(jc_, nt)) \
    for (int t = 0; t < T; ++t)                                           \
      for (int j = jc_; j < je_; ++j, ++it)
// one step of the same walk for code that carries (t, j) along
__device__ __forceinline__ void wl_advance(int& t, int& j, int& jc, int& je, int T, int nt) {
  if (++j == je) {
    if (++t == T) { t = 0; jc = je; je = wl_chunk_end(jc, nt); }
    j = jc;
  }
}

template <int kOff> __device__ __forceinline__ void wl_sts_u16_imm(uint32_t addr, uint16_t v) {
  asm volatile("st.shared.u16 [%0+%2], %1;" ::"r"(addr), "h"(v), "n"(kOff) : "memory");
}
// gate stash of one 16-row part: rows I, I + 1 of the thread's gate column, 128B-swizzled rows of 128 bytes
template <int I, int kBase> struct WlStash {
  static __device__ __forceinline__ void run(uint32_t gbase0, const float (&a)[16]) {
    const uint32_t pk = pack_f16x2(a[I], a[I + 1]);
    wl_sts_u16_imm<kBase + I * 128>(gbase0 ^ ((I & 7) << 4), (uint16_t)(pk & 0xffffu));
    wl_sts_u16_imm<kBase + (I + 1) * 128>(gbase0 ^ (((I + 1) & 7) << 4), (uint16_t)(pk >> 16));
    if constexpr (I + 2 < 16) WlStash<I + 2, kBase>::run(gbase0, a);
  }
};

template <int H>
__global__ void __launch_bounds__(kWlThreads, 1) wlstm_fwd_kernel(const __grid_constant__ WlstmParams p) {
  constexpr int NS = H / 32;                 // gate-column slices per layer
  constexpr int NKB_R = H / 64;
  static_assert(H % 64 == 0 && H / 2 <= kWlAccCol, "hidden size does not fit the tensor-memory weight slice");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  uint8_t* stg = smem + kWlStages * kWlStageBytes;
  uint8_t* cin = stg + 2 * kWlStgBytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(cin + 2 * kWlCinBytes);
  uint64_t* empty = full + kWlStages;
  uint64_t* acc_full = empty + kWlStages;      // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]
  uint64_t* cin_full = acc_empty + 2;          // [2]
  uint64_t* stg_full = cin_full + 2;           // [2]
  uint64_t* stg_free = stg_full + 2;           // [2]
  uint64_t* dep_ready = stg_free + 2;          // [kWlDeps]
  uint64_t* dep_free = dep_ready + kWlDeps;    // [kWlDeps]
  uint64_t* gin_done = dep_free + kWlDeps;     // [2] (P: gin tile written by all epilogue threads)
  uint64_t* gin_taken = gin_done + 2;          // [2] (P: the signal warp has seen gin_done; keeps the phases apart)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(gin_taken + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x;
  const bool is_R = cta < p.L * NS;
  const int l = (is_R ? cta : cta - p.L * NS) / NS;
  const int n = (is_R ? cta : cta - p.L * NS) % NS;
  const WlstmLayer& ly = p.layer[l];
  const int K = is_R ? H : ly.Ip;
  const int nkb = is_R ? NKB_R : (K + 63) / 64;
  const int ngroups = (nkb + kWlKbPerStage - 1) / kWlKbPerStage;
  const int nt = p.nt, T = p.T;
  const long long total = (long long)T * nt;
  long long* const trace_cta = (p.trace && p.trace_mode != 2 && l == 1 && n == 0) ? p.trace + (is_R ? 0 : (size_t)nt * 16) : nullptr;
  // accounting: CTAs R(0,0), R(1,0), P(1,0) -> rows 0, 1, 2 of 64 slots each at p.trace + 8192
  const int acct_row = (n == 0 && is_R && l == 0) ? 0 : (n == 0 && is_R && l == 1) ? 1 : (n == 0 && !is_R && l == 1) ? 2 : -1;
#ifdef SVB_WL_ACCOUNT
  const bool acct = p.trace && p.trace_mode == 2 && acct_row >= 0;
  long long* const acct_out = p.trace + 8192 + (acct_row < 0 ? 0 : acct_row) * 64;
  long long w0 = 0, w1 = 0, w2 = 0, w3 = 0;
#else
  constexpr bool acct = false;
  (void)acct_row;
#endif

  if (threadIdx.x == 0) {
    for (int s = 0; s < kWlStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], kWlEpiWarps / 2);        // one epilogue group (8 warps) per accumulator buffer
      mbar_init(&cin_full[b], 1);
      mbar_init(&stg_full[b], kWlEpiWarps / 2);         // one arrive per warp of the group (N arrivals on one mbarrier serialise)
      mbar_init(&stg_free[b], 1);
      mbar_init(&gin_done[b], kWlEpiWarps / 2);
      mbar_init(&gin_taken[b], 1);
    }
    for (int d = 0; d < kWlDeps; ++d) {
      mbar_init(&dep_ready[d], 1);
      mbar_init(&dep_free[d], is_R ? 2 + kWlEpiWarps / 2 : 1); // the producer (+ c loader + one epilogue group of R)
    }
    fence_mbar_init();
    tma_prefetch_desc(is_R ? &ly.t_h : &ly.t_in);
  }
  if (warp == kWlWarpMma) tmem_alloc<512>(tmem_holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_holder;

  // ---- weights -> tensor memory (once): lane r = packed gate row 128 n + r, two fp16 per column
  if (warp < 4) {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const __half* wrow = (is_R ? ly.whh : ly.wih) + (size_t)(n * 128 + r) * K;
    for (int kb = 0; kb < nkb; ++kb) {
      uint32_t v[32];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        uint4 x = make_uint4(0u, 0u, 0u, 0u);
        if (kb * 64 + u * 8 < K) x = __ldg(reinterpret_cast<const uint4*>(wrow + kb * 64 + u * 8));   // K % 8 == 0
        v[4 * u] = x.x; v[4 * u + 1] = x.y; v[4 * u + 2] = x.z; v[4 * u + 3] = x.w;
      }
      tmem_st32(tmem + (uint32_t(q * 32) << 16) + kb * 32, v);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  const long long t_cta0 = clock64();
  if (warp == kWlWarpPoll && lane == 0) {
    // ------------------------------------------------------------------ dependency poller (runs ahead of the rest)
    // A satisfied poll still costs an L2 round trip (~1000 clk); here it overlaps the previous tiles' work.
    {
      // P may run at most `lag` tiles ahead of its layer's recurrence: 3 frames is the capacity of the gin ring, but
      // with a large batch (extraction: hundreds of tiles per frame) a producer that far ahead pushes every gin tile
      // out of L2 before R reads it (80 GB of HBM traffic for 47 k windows); kWlGinLagMax tiles keep it resident.
      const long long lag = (long long)kWlGinRing * nt < kWlGinLagMax ? (long long)kWlGinRing * nt : kWlGinLagMax;
      int bt = 0, bj = 0, bjc = 0, bje = wl_chunk_end(0, nt);   // (frame, tile) of linear index it - lag
      long long it = 0;
      WL_FOR_TILES(t, j, it) {
        {
          const int d = (int)(it % kWlDeps);
          WL_ACC(w0, mbar_wait(&dep_free[d], (uint32_t)(((it / kWlDeps) & 1) ^ 1)));
#ifdef SVB_WL_ACCOUNT
          const long long pa0 = acct ? clock64() : 0;
#endif
          if (p.ablate & 8) {
          } else if (is_R) {
            wait_two_counters(t > 0 ? p.hcnt + l * nt + j : nullptr, (unsigned)(NS * t),
                              p.gcnt + ((size_t)l * NS + n) * nt + j, (unsigned)(t + 1));
          } else {
            const bool bp = it >= lag;          // every R(l, .) has finished tile it - lag (and, in order, all before)
            wait_two_counters(l > 0 ? p.hcnt + (l - 1) * nt + j : nullptr, (unsigned)(NS * (t + 1)),
                              bp ? p.hcnt + l * nt + bj : nullptr, (unsigned)(NS * (bt + 1)));
            if (bp) wl_advance(bt, bj, bjc, bje, T, nt);
          }
#ifdef SVB_WL_ACCOUNT
          if (acct) w1 += clock64() - pa0;
#endif
          mbar_arrive(&dep_ready[d]);
        }
      }
    }
  } else if (warp == kWlWarpPoll && lane == 1) {
    // ------------------------------------------------------------------ c_{t-1} tile loader (R only)
    // Its own thread: the wait for the c buffer (epilogue of tile it-2 finished) must not hold back the operand
    // loads of later tiles, or load latency + MMA + epilogue chain up into the per-tile period.
    if (is_R) {
      long long it = 0;
      WL_FOR_TILES(t, j, it) {
        {
          const int buf = (int)(it & 1);
          const uint32_t upar = (uint32_t)((it >> 1) & 1);
          const int d = (int)(it % kWlDeps);
          WL_ACC(w0, mbar_wait(&dep_ready[d], (uint32_t)((it / kWlDeps) & 1)));   // our own stores of frame t-1 are complete
          mbar_arrive(&dep_free[d]);
          WL_ACC(w1, mbar_wait(&stg_full[buf], upar ^ 1));                       // the epilogue of tile it-2 has read its c tile
          mbar_expect_tx(&cin_full[buf], kWlCinBytes);
          tma_load_3d(cin + buf * kWlCinBytes, &ly.t_c, &cin_full[buf], n * 32, j * kWlTile, p.training ? t : (t & 1));
        }
      }
    }
  } else if (warp == kWlWarpTma) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      long long it = 0;
      WL_FOR_TILES(t, j, it) {
        {
          const int buf = (int)(it & 1);
          const uint32_t upar = (uint32_t)((it >> 1) & 1);
          const int d = (int)(it % kWlDeps);
          long long* tr = (trace_cta && t == T / 2) ? trace_cta + j * 16 : nullptr;
          WL_STAMP(0);
          WL_ACC(w0, mbar_wait(&dep_ready[d], (uint32_t)((it / kWlDeps) & 1)));
          mbar_arrive(&dep_free[d]);
          WL_STAMP(1);
          const CUtensorMap* tm = is_R ? &ly.t_h : &ly.t_in;
          const int slab = is_R ? t : t + ly.in_slab0;
          for (int gi = 0; gi < ngroups; ++gi) {
            const int kb0 = gi * kWlKbPerStage;
            const int nk = nkb - kb0 < kWlKbPerStage ? nkb - kb0 : kWlKbPerStage;
            WL_ACC(w1, mbar_wait(&empty[stage], phase ^ 1));
            if (p.ablate & 4) {
              mbar_arrive(&full[stage]);
              if (++stage == kWlStages) { stage = 0; phase ^= 1; }
              continue;
            }
            mbar_expect_tx(&full[stage], nk * kWlKbBytes);
            for (int k = 0; k < nk; ++k)
              tma_load_3d(ring + stage * kWlStageBytes + k * kWlKbBytes, tm, &full[stage], (kb0 + k) * 64, j * kWlTile, slab);
            if (tr && gi < 3) tr[3 * nt * 16 + 13 + gi] = clock64();   // issue time of groups 0..2
            if (++stage == kWlStages) { stage = 0; phase ^= 1; }
          }
          WL_STAMP(2);
        }
      }
    }
  } else if (warp == kWlWarpMma) {
    // ------------------------------------------------------------------ MMA issuer (A = weights in TMEM)
    constexpr uint32_t idesc = umma_idesc_f16(128, kWlTile, 0, 0);
    const uint64_t desc0 = umma_desc_kmajor_sw128(smem_u32(ring));
    const uint32_t desc_lo0 = (uint32_t)desc0, desc_hi = (uint32_t)(desc0 >> 32);
    int stage = 0;
    uint32_t phase = 0;
    // ONE thread runs the whole loop (waits included): looping the whole warp with an election and a __syncwarp per
    // group costs +150 cycles per group of 8 MMAs (256 cycles of tensor work), scripts/ubench/mma_issue.cu
    // `if (elect_one())` around the loop, NOT a per-thread trip count: with `n = elect_one() ? total : 0; for (it < n)`
    // the compiler treats the body as divergent code and wraps EVERY tcgen05.mma in an elect / R2UR.BROADCAST /
    // BRA.U.ANY loop (~12 instructions, 60-70 cycles of issue per MMA instead of 32).
    if (elect_one())
    for (long long it = 0; it < total; ++it) {
      const int buf = (int)(it & 1);
      const uint32_t upar = (uint32_t)((it >> 1) & 1);
      long long* tr = (trace_cta && it / nt == T / 2) ? trace_cta + (it % nt) * 16 : nullptr;
      WL_STAMP(3);
      WL_ACC(w0, mbar_wait(&acc_empty[buf], upar ^ 1));
      tc_fence_after();
      WL_STAMP(4);
      for (int gi = 0; gi < ngroups; ++gi) {
        const int kb0 = gi * kWlKbPerStage;
        const int nk = nkb - kb0 < kWlKbPerStage ? nkb - kb0 : kWlKbPerStage;
        long long* trd = tr ? tr + 3 * nt * 16 : nullptr;      // MMA detail rows
        if (trd && gi < 6) trd[2 * gi] = clock64();
        WL_ACC(w1, mbar_wait(&full[stage], phase));
        tc_fence_after();
        if (trd && gi < 6) trd[2 * gi + 1] = clock64();
        if (gi == 0) WL_STAMP(5);
        if (gi == ngroups - 1) WL_STAMP(6);
        {
          // descriptor of stage s, K block kk, K step k = desc0 + ((s * stage + kk * 8192 + k * 32) >> 4) in the low half
          const uint32_t lo = desc_lo0 + stage * (kWlStageBytes >> 4);
          const uint32_t a0 = tmem + kb0 * 32;
          const uint32_t dacc = tmem + kWlAccCol + buf * kWlTile;
          if (p.ablate & 1) {
          } else if (nk == kWlKbPerStage) {
#pragma unroll
            for (int q = 0; q < 4 * kWlKbPerStage; ++q)
              umma_f16_ts_lohi(dacc, a0 + q * 8, lo + (q >> 2) * (kWlKbBytes >> 4) + (q & 3) * 2, desc_hi, idesc,
                               q == 0 ? (gi != 0 ? 1u : 0u) : 1u);
          } else {
            for (int q = 0; q < 4 * nk; ++q)
              umma_f16_ts_lohi(dacc, a0 + q * 8, lo + (q >> 2) * (kWlKbBytes >> 4) + (q & 3) * 2, desc_hi, idesc,
                               (gi | q) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (gi == ngroups - 1) umma_commit(&acc_full[buf]);
          if (trd && gi == ngroups - 1) trd[12] = clock64();
        }
        if (++stage == kWlStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp < kWlEpiWarps) {
    // ------------------------------------------------------------------ epilogue: thread = gate column (TMEM lane)
    // Two groups of 8 warps work on alternate tiles (group = accumulator buffer), so that one group's MUFU-bound
    // activation phase overlaps the other's shuffle / shared-memory phases and the ~170-cycle mbarrier waits.
    // Within a group two warps share a TMEM lane quarter; each takes two 16-row parts of the 64-row tile.  The
    // accumulator is drained into registers first so that the MMA of tile it+2 starts while this epilogue runs.
    const int grp = warp >> 3;                 // tiles it = grp, grp + 2, ... (accumulator / staging buffer = grp)
    const int q = warp & 3;                    // TMEM lane quarter
    const int sub = (warp >> 2) & 1;           // parts sub and sub + 2: rows [16 part, 16 part + 16)
    const int col = q * 32 + lane;             // packed gate column within the slice
    const int g = lane >> 3, ju = lane & 7;    // gate (i, f, g, o) and unit within the warp's 8 units
    const int unit = q * 8 + ju;               // unit within the CTA's 32
    const bool g0 = g & 1, g1 = g >> 1;
    const uint32_t lane_base = uint32_t(q * 32) << 16;
    // (P publishes gin' = cs (W_ih x + b), cs = 0.5 for the sigmoid gates: R's pre-activation scaling then folds into
    // one FFMA, fma(acc, cs, gin'), bit-identical to cs (acc + gin) because the scale is a power of two)
    const float bias = is_R ? 0.f : __ldg(ly.bias + n * 128 + col) * (g == 2 ? 1.0f : 0.5f);
    // activation of this thread's gate with one MUFU.TANH: sigmoid(x) = 0.5 tanh(0.5 x) + 0.5  (2^-11 relative:
    // embedding error 3.3e-4 instead of 2.3e-4 in the emulation of scripts/precision_study.py)
    const float cs = g == 2 ? 1.0f : 0.5f, ca = g == 2 ? 1.0f : 0.5f, cb = g == 2 ? 0.0f : 0.5f;
    const int buf = grp;
    // shared-memory addresses of this thread's slots, swizzle terms folded in (row & 7 is known at compile time below)
    const uint32_t sb_a = smem_u32(stg) + buf * kWlStgBytes;
    const int cb2 = (q & 1) * 32 + lane;                               // column within the 64-column gate box
    // gate stash: row i -> (gbase0 ^ ((i & 7) << 4)) + i * 128  (bits 4..6 of gbase0 hold only the 16-byte unit index)
    const uint32_t gbase0 = sb_a + kWlOffG + (q >> 1) * 8192 + ((cb2 >> 3) << 4) + (cb2 & 7) * 2 + sub * 2048;
    uint32_t cx[2];                                                    // c tile: row 4k + g -> cx[k & 1] + k * 512
#pragma unroll
    for (int e = 0; e < 2; ++e) cx[e] = sub * 2048 + g * 128 + ((((unit >> 2) ^ ((e << 2) | g))) << 4) + (unit & 3) * 4;
    const uint32_t cin_a = smem_u32(cin) + buf * kWlCinBytes;
    const uint32_t hx = sub * 1024 + g * 64 + unit * 2;                // h tiles: row 4k + g -> hx + k * 256
    // (t, j) of tile `it` are carried along: a 64-bit it / nt and it % nt by a run-time divisor is a ~70-instruction
    // subroutine call at the head of every tile's dependency chain
    int t = 0, j = 0, jc = 0, je = wl_chunk_end(0, nt);
    if (grp) wl_advance(t, j, jc, je, T, nt);
    for (long long it = grp; it < total; it += 2, wl_advance(t, j, jc, je, T, nt), wl_advance(t, j, jc, je, T, nt)) {
      const uint32_t upar = (uint32_t)((it >> 1) & 1);
      float4* gfrag = reinterpret_cast<float4*>(ly.gin) + ((size_t)((t % kWlGinRing) * nt + j) * NS + n) * 2048 +
                      (size_t)sub * 512 + col;      // + ps * 1024 + k * 128 float4
      float4 gv[4];
      long long* tr = (trace_cta && t == T / 2 && (warp & 7) == 0 && lane == 0) ? trace_cta + j * 16 : nullptr;
      WL_STAMP(7);
      if (is_R) {
        const int d = (int)(it % kWlDeps);
        WL_ACC(w0, mbar_wait(&dep_ready[d], (uint32_t)((it / kWlDeps) & 1)));     // gin of (t, j) is published
#pragma unroll
        for (int k = 0; k < 4; ++k) gv[k] = __ldcg(gfrag + k * 128);
      }
      WL_STAMP(8);
      WL_ACC(w1, mbar_wait(&acc_full[buf], upar));
      tc_fence_after();
      WL_STAMP(9);
      float a0[16], a1[16];
      tmem_ld16(tmem + lane_base + kWlAccCol + buf * kWlTile + sub * 16, a0);
      tmem_ld16(tmem + lane_base + kWlAccCol + buf * kWlTile + sub * 16 + 32, a1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      if (!is_R) {
        // gin = W_ih x + bias, in fragment order: float4 (rows 4r..4r+3) of column `col` at [r][col].  The tile is
        // staged in shared memory (P's staging buffers are otherwise unused) in exactly the ring's layout and leaves
        // through ONE bulk copy issued by the signal thread, whose completion + release publishes it.  Direct global
        // stores needed a gpu-scope fence in every epilogue thread before the flag (~2000 cycles in the chain of every
        // tile: P, not R, set the pace of layers 1 and 2 -- 3550 cycles per tile against 3070 for layer 0).
        mbar_wait(&gin_taken[buf], upar ^ 1);     // the bulk copy of tile it-2 has read this buffer
        const uint32_t gs = sb_a + (uint32_t)(sub * 512 + col) * 16;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          sts_f4(gs + k * 2048, make_float4(fmaf(a0[4 * k], cs, bias), fmaf(a0[4 * k + 1], cs, bias), fmaf(a0[4 * k + 2], cs, bias), fmaf(a0[4 * k + 3], cs, bias)));
          sts_f4(gs + 16384 + k * 2048, make_float4(fmaf(a1[4 * k], cs, bias), fmaf(a1[4 * k + 1], cs, bias), fmaf(a1[4 * k + 2], cs, bias), fmaf(a1[4 * k + 3], cs, bias)));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&gin_done[buf]);   // the signal warp copies and publishes the tile
        WL_STAMP(13);
        continue;
      }
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        float (&a)[16] = ps == 0 ? a0 : a1;
        // ---- activations of this thread's gate column for 16 rows
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          a[4 * k + 0] = fmaf(ca, tanh_approx(fmaf(a[4 * k + 0], cs, gv[k].x)), cb);
          a[4 * k + 1] = fmaf(ca, tanh_approx(fmaf(a[4 * k + 1], cs, gv[k].y)), cb);
          a[4 * k + 2] = fmaf(ca, tanh_approx(fmaf(a[4 * k + 2], cs, gv[k].z)), cb);
          a[4 * k + 3] = fmaf(ca, tanh_approx(fmaf(a[4 * k + 3], cs, gv[k].w)), cb);
        }
        if (ps == 0) {
          // gin of the second part: in flight while the first part is processed
#pragma unroll
          for (int k = 0; k < 4; ++k) gv[k] = __ldcg(gfrag + 1024 + k * 128);
          __syncwarp();
          if (lane == 0) mbar_arrive(&dep_free[(int)(it % kWlDeps)]);
          WL_STAMP(10);
          WL_ACC(w2, mbar_wait(&stg_free[buf], upar ^ 1));    // staging buffer drained by the store warp
          WL_STAMP(11);
        }
#ifndef SVB_NO_RING_DISCARD
        if (ps == 1) {
          // The gin tile has been consumed (both halves are in registers and have been used): drop its 32 lines of this
          // warp from L2 WITHOUT write-back.  The ring is consumed from L2 a few microseconds after it is written and
          // never read again, yet every dirty line was eventually written back to HBM: 3.8 GB per C2 step, as much as
          // the whole BPTT stash (the part is power-capped: forward 1.5 % faster without that traffic).  Ordering: the
          // ring slot is refilled only after this tile's h has been published, which follows this instruction through
          // the staging barrier and the store thread's gpu-scope release.  Lane -> (half, k, 128-byte line of the
          // warp's 512-byte row).
          const float4* dl = gfrag - lane + ((lane >> 4) * 1024 + ((lane >> 2) & 3) * 128) + (lane & 3) * 8;
          asm volatile("discard.global.L2 [%0], 128;" ::"l"(dl) : "memory");
        }
#endif
        if (p.ablate & 2) continue;
        if (p.training) {
          // gate stash [row][packed col] fp16 (see pack8_stash): two boxes of 64 columns, 128B-swizzled rows
          // (offsets as immediates: one XOR per store instead of XOR + two adds)
          if (ps == 0) WlStash<0, 0>::run(gbase0, a); else WlStash<0, 4096>::run(gbase0, a);
        }
        // 4 x 4 transposes across the lanes (g, ju), g = 0..3: afterwards this thread holds i, f, g, o of unit ju at
        // rows 16 part + 4k + g, k = 0..3
        float vi[4], vf[4], vg[4], vo[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float x0 = a[4 * k], x1 = a[4 * k + 1], x2 = a[4 * k + 2], x3 = a[4 * k + 3];
          const float r0 = __shfl_xor_sync(0xffffffffu, g0 ? x0 : x1, 8);
          const float r1 = __shfl_xor_sync(0xffffffffu, g0 ? x2 : x3, 8);
          const float p0lo = g0 ? r0 : x0, p0hi = g0 ? x1 : r0;     // (lo gate, hi gate) of row g0
          const float p1lo = g0 ? r1 : x2, p1hi = g0 ? x3 : r1;     // ... of row 2 + g0
          const float s0 = __shfl_xor_sync(0xffffffffu, g1 ? p0lo : p1lo, 16);
          const float s1 = __shfl_xor_sync(0xffffffffu, g1 ? p0hi : p1hi, 16);
          vi[k] = g1 ? s0 : p0lo; vf[k] = g1 ? s1 : p0hi;
          vg[k] = g1 ? p1lo : s0; vo[k] = g1 ? p1hi : s1;
        }
        if (ps == 0) {
          WL_ACC(w3, mbar_wait(&cin_full[buf], upar));        // c_{t-1} tile landed
          WL_STAMP(12);
        }
        // all loads, then the math, then all stores
        float cv[4], hv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) cv[k] = lds_f32(cin_a + ps * 4096 + k * 512 + cx[k & 1]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          cv[k] = vf[k] * cv[k] + vi[k] * vg[k];
          hv[k] = vo[k] * tanh_approx(cv[k]);
        }
#pragma unroll
        for (int k = 0; k < 4; k += 2) {
          sts_f32(sb_a + kWlOffC + ps * 4096 + k * 512 + cx[k & 1], cv[k]);
          sts_f32(sb_a + kWlOffC + ps * 4096 + (k + 1) * 512 + cx[(k + 1) & 1], cv[k + 1]);
          const uint32_t h16 = pack_f16x2(hv[k], hv[k + 1]);
          sts_u16(sb_a + kWlOffH16 + ps * 2048 + k * 256 + hx, (uint16_t)(h16 & 0xffffu));
          sts_u16(sb_a + kWlOffH16 + ps * 2048 + (k + 1) * 256 + hx, (uint16_t)(h16 >> 16));
          if (p.training) {
            const uint32_t hb = pack_bf16x2(hv[k], hv[k + 1]);
            sts_u16(sb_a + kWlOffHbf + ps * 2048 + k * 256 + hx, (uint16_t)(hb & 0xffffu));
            sts_u16(sb_a + kWlOffHbf + ps * 2048 + (k + 1) * 256 + hx, (uint16_t)(hb >> 16));
          }
        }
        if (p.h_last && l == p.L - 1 && t == T - 1) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int m = j * kWlTile + (sub + 2 * ps) * 16 + 4 * k + g;
            if (m < p.B) p.h_last[(size_t)m * H + n * 32 + unit] = hv[k];
          }
        }
      }
      if (p.ablate & 2) mbar_wait(&cin_full[buf], upar);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&stg_full[buf]);
      WL_STAMP(13);
    }
  } else if (warp == kWlWarpStore && !is_R) {
    // ------------------------------------------------------------------ signal thread (P): copy out + publish gin tiles
    // The completion of a bulk store (cp.async.bulk.wait_group, needed before the release that publishes the tile)
    // takes thousands of cycles under load.  A tile is therefore published LAZILY: if the next tile is already staged
    // its copy is issued first and the thread then waits for the older group only (wait_group 1: two tiles in flight);
    // if the next tile is not ready the pending one is completed and published at once, so a release never waits for
    // a later tile (with one tile per frame the next frame cannot start before it).
    if (lane == 0) {
      int t = 0, j = 0, jc = 0, je = wl_chunk_end(0, nt);
      bool pend = false;
      unsigned* pflag = nullptr;
      unsigned pval = 0;
      for (long long it = 0; it < total; ++it, wl_advance(t, j, jc, je, T, nt)) {
        const int buf = (int)(it & 1);
        const uint32_t upar = (uint32_t)((it >> 1) & 1);
        if (pend && !mbar_test_wait(&gin_done[buf], upar)) {
          asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
          asm volatile("red.release.gpu.global.max.u32 [%0], %1;" ::"l"(pflag), "r"(pval) : "memory");
          pend = false;
        }
        WL_ACC(w0, mbar_wait(&gin_done[buf], upar));
        float* dst = ly.gin + ((size_t)((t % kWlGinRing) * nt + j) * NS + n) * 8192;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
                     "r"(smem_u32(stg) + buf * kWlStgBytes), "n"(32768) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // the staging buffer may be refilled
        mbar_arrive(&gin_taken[buf]);
        if (pend) {
          WL_ACC(w1, asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"));   // the older tile is written: release its flag
          asm volatile("red.release.gpu.global.max.u32 [%0], %1;" ::"l"(pflag), "r"(pval) : "memory");
        }
        pend = true;
        pflag = p.gcnt + ((size_t)l * NS + n) * nt + j;
        pval = (unsigned)(t + 1);
      }
      if (pend) {
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        asm volatile("red.release.gpu.global.max.u32 [%0], %1;" ::"l"(pflag), "r"(pval) : "memory");
      }
    }
  } else if (warp == kWlWarpStore && is_R) {
    // ------------------------------------------------------------------ store + signal thread (R only): lazy publish,
    // two tiles in flight (see the P signal thread above)
    if (lane == 0) {
      int t = 0, j = 0, jc = 0, je = wl_chunk_end(0, nt);
      bool pend = false;
      unsigned* pflag = nullptr;
      for (long long it = 0; it < total; ++it, wl_advance(t, j, jc, je, T, nt)) {
        const int buf = (int)(it & 1);
        const uint32_t upar = (uint32_t)((it >> 1) & 1);
        if (pend && !mbar_test_wait(&stg_full[buf], upar)) {
          asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
          red_release_add(pflag, 1u);
          pend = false;
        }
        WL_ACC(w0, mbar_wait(&stg_full[buf], upar));
        long long* tr = (trace_cta && t == T / 2) ? trace_cta + j * 16 : nullptr;
        WL_STAMP(14);
        const uint8_t* sb = stg + buf * kWlStgBytes;
        const int row0 = j * kWlTile;
        tma_store_3d(&ly.t_h16_st, sb + kWlOffH16, n * 32, row0, t + 1);
        tma_store_3d(&ly.t_c, sb + kWlOffC, n * 32, row0, p.training ? t + 1 : ((t + 1) & 1));
        if (p.training) {
          tma_store_3d(&ly.t_hbf_st, sb + kWlOffHbf, n * 32, row0, t + 1);
          tma_store_3d(&ly.t_gates, sb + kWlOffG, n * 128, row0, t);
          tma_store_3d(&ly.t_gates, sb + kWlOffG + 8192, n * 128 + 64, row0, t);
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(&stg_free[buf]);          // the staging buffer has been read: the epilogue may refill it
        // complete, then a RELEASE increment publishes the tile.  The release is required: with a relaxed increment
        // other CTAs' TMA loads read stale rows of the tile (found with a NaN-poisoned workspace,
        // tests/test_gpu_parity.py::test_persistent_kernel_no_stale_reads).  One fence is enough; proxy fence +
        // __threadfence + release together cost ~3000 cycles per tile.
        if (pend) {
          WL_ACC(w1, asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"));
          WL_ACC(w2, red_release_add(pflag, 1u));
        }
        pend = true;
        pflag = p.hcnt + l * nt + j;
        WL_STAMP(15);
      }
      if (pend) {
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        red_release_add(pflag, 1u);
      }
    }
  }
#ifdef SVB_WL_ACCOUNT
  if (acct) {
    // slots: 8 per role thread: poller 0, c-loader 1, producer 2, mma 3, store/signal 4, epilogue warp 0 -> 5, warp 8 -> 6
    int role = -1;
    if (warp == kWlWarpPoll && lane == 0) role = 0;
    else if (warp == kWlWarpPoll && lane == 1) role = 1;
    else if (warp == kWlWarpTma && (w0 | w1)) role = 2;
    else if (warp == kWlWarpMma && (w0 | w1)) role = 3;
    else if (warp == kWlWarpStore && (w0 | w1 | w2)) role = 4;
    else if (threadIdx.x == 0) role = 5;
    else if (threadIdx.x == 256) role = 6;
    if (role >= 0) {
      acct_out[role * 8 + 0] = w0; acct_out[role * 8 + 1] = w1; acct_out[role * 8 + 2] = w2; acct_out[role * 8 + 3] = w3;
      acct_out[role * 8 + 4] = clock64() - t_cta0;
    }
  }
#endif
  tc_fence_before();
  __syncthreads();
  if (warp == kWlWarpMma) tmem_dealloc<512>(tmem);
  if (p.trace && threadIdx.x == 0) p.trace[4 * nt * 16 + cta] = clock64() - t_cta0;
}

template <int H>
static int launch_wlstm_fwd(WlstmParams& p, cudaStream_t s) {
  auto kern = wlstm_fwd_kernel<H>;
  for (int l = 0; l < p.L; ++l)                    // a wider W_ih slice would overlap the accumulators
    if ((p.layer[l].Ip + 63) / 64 * 32 > kWlAccCol) {
      set_error("wlstm: layer input wider than 768 does not fit tensor memory", cudaSuccess);
      return SVB_ERR_UNSUPPORTED;
    }
  static unsigned long long configured = 0;        // one bit per device
  if (first_use_on_device(configured)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kWlSmem);
    if (e != cudaSuccess) { set_error("wlstm: cudaFuncSetAttribute", e); return SVB_ERR_CUDA; }
  }
  void* args[] = {&p};
  cudaError_t e = cudaLaunchCooperativeKernel((void*)kern, dim3(2 * p.L * (H / 32)), dim3(kWlThreads), args, kWlSmem, s);
  if (e != cudaSuccess) { set_error("wlstm: cooperative launch", e); return SVB_ERR_CUDA; }
  return SVB_OK;
}
