// Warp-specialised tcgen05 GEMM core for sm_100a.
//
//   D[m, n] = sum_{term} sum_k A_term[m, k] * B_term[n, k]        (bf16 operands, fp32 accumulate in TMEM)
//
// One CTA computes one 128 x BN tile.  192 threads:
//   warp 0      TMA producer: first the epilogue's input tiles (Epi::issue_loads), then the operand ring
//               (cp.async.bulk.tensor into kStages 128B-swizzled stages)
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer
//   warps 2..5  epilogue: tcgen05.ld 32 lanes x 32 columns per warp -> Epi::apply, which reads its inputs from
//               swizzled shared memory (TMA-loaded) and writes its outputs to a staging area aliased on the
//               (by then idle) operand ring; one thread then issues TMA stores (Epi::issue_stores).
// All bulk global traffic of the epilogue is TMA: a thread-per-row epilogue doing 16-byte global accesses touches
// 32 cache lines per warp instruction and is L1TEX-wavefront bound (measured: 40 us of a 46 us BPTT frame).
// "Terms" accumulate several operand pairs into one accumulator; this is how the split-bf16 (hi/lo) input
// projection gets near-fp32 accuracy from bf16 tensor-core passes.
// Operands are K-major ([rows, K], K contiguous) or MN-major ([K, rows], rows contiguous; used by the
// weight-gradient GEMMs whose reduction runs over time*batch).
#pragma once
#include "sm100.cuh"

namespace svb {

constexpr int kBM = 128;
constexpr int kBK = 64;          // 64 bf16 = 128 B = one swizzle row
constexpr int kMaxTerms = 3;

struct __align__(64) GemmOperands {
  CUtensorMap ta[kMaxTerms];
  CUtensorMap tb[kMaxTerms];
  int za[kMaxTerms];             // slab (3rd tensor-map coordinate) of A per term
  int zb[kMaxTerms];
  int nterms;
  int f16;                       // operands are IEEE half instead of bf16 (same tensor maps: 2-byte elements)
  int kz;                        // > 1: gridDim.z = kz slices of the reduction, K = length of ONE slice; slice z writes
                                 // its partial product through Epi with blockIdx.z (see EpiStoreF32::z_stride)
  int M, N, K;                   // K = reduction length per term
  unsigned long long* trace;     // debug: 16 globaltimer stamps per CTA, or null
};

// Byte offset of 16-byte unit `u16` of row `row` in a TMA tile whose rows are 128 bytes (SWIZZLE_128B, tile base
// 1024-byte aligned): the unit index is XORed with (row mod 8).
__device__ __forceinline__ uint32_t sw128(int row, int u16) { return row * 128 + ((u16 ^ (row & 7)) << 4); }

template <int BN, int kStages, class Epi, int KSPLIT = 1, bool TWO_CTA = false>
struct GemmSmem {
  static constexpr int kABytes = kBM * kBK * 2;
  static constexpr int kBBytes = (TWO_CTA ? BN / 2 : BN) * kBK * 2;   // a CTA pair splits the B rows
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kRingBytes = kStages * kStageBytes;
  static_assert(kStageBytes % 1024 == 0, "stages must keep 1024-byte alignment");
  // split-K: the KSPLIT partial 32-column chunks (16 KB each) + the output staging live in the idle ring
  static constexpr int kRecvBytes = KSPLIT > 1 ? KSPLIT * 16384 : 0;
  static_assert(kRecvBytes + Epi::kOutBytes <= kRingBytes, "output staging is aliased on the operand ring");
  static constexpr int kInOffset = kRingBytes;
  static constexpr int kBarOffset = kInOffset + ((Epi::kInBytes + 1023) / 1024) * 1024;
  static constexpr int kTotal = kBarOffset + 256 + 1024;   // barriers + alignment slack
  static_assert(kTotal <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void trace_stamp(const GemmOperands& ops, int slot) {
  if (ops.trace) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    ops.trace[(size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 16 + slot] = t;
  }
}

// Epi interface:
//   struct Params;  static constexpr int kInBytes, kOutBytes;
//   static __device__ void issue_loads(const Params&, uint8_t* in, uint64_t* bar, int m0, int n0);   one thread
//   static __device__ void apply(const Params&, const uint8_t* in, uint8_t* out, int row, int m, int n0, int chunk,
//                                float (&acc)[32], bool valid);                                   128 threads
//   static __device__ void issue_stores(const Params&, const uint8_t* out, int m0, int n0);         one thread
// kEpiWarps = 4, 8 or 16 epilogue warps (kEpiWarps/4 warps per TMEM lane quarter share the column chunks).
// KSPLIT > 1 (requires BN == 32*KSPLIT, 4 epilogue warps, a (KSPLIT,1,1) cluster launch): the KSPLIT CTAs of a
// cluster each reduce a 1/KSPLIT slice of K for the same 128 x BN tile, exchange their partial 32-column chunks
// through distributed shared memory, and CTA r finishes columns [32r, 32r+32) with Epi.  Each SM then pulls only
// 1/KSPLIT of both operands from L2 -- the per-SM L2->SM port (~64 B/clk) is what bounds the BPTT frame.
// TWO_CTA (cluster (2,1,1): blockIdx.x = 2*n_tile + rank, K-major operands): the two CTAs of a pair own adjacent 128-row tiles and each holds half
// of the B rows; CTA 0 issues tcgen05.mma.cta_group::2 with M = 256, so every B byte is pulled from L2 once per 256
// rows and the operand traffic per SM halves relative to the arithmetic.
template <int BN, int kStages, bool A_MN, bool B_MN, class Epi, int kEpiWarps = 4, int KSPLIT = 1, bool TWO_CTA = false>
__global__ void __launch_bounds__(64 + 32 * kEpiWarps) tc_gemm_kernel(const __grid_constant__ GemmOperands ops,
                                                               const __grid_constant__ typename Epi::Params ep) {
  using S = GemmSmem<BN, kStages, Epi, KSPLIT, TWO_CTA>;
  static_assert(!TWO_CTA || KSPLIT == 1, "pair mode: no split-K");
  static_assert(KSPLIT == 1 || (BN == 32 * KSPLIT), "split-K layout");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* in_smem = smem + S::kInOffset;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::kBarOffset);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* accum_bar = empty_bar + kStages;
  uint64_t* in_bar = accum_bar + 1;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(in_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int kq = KSPLIT > 1 ? (int)cluster_ctarank() : 0;       // K slice (and finished column chunk) of this CTA
  const int pair_rank = TWO_CTA ? (int)cluster_ctarank() : 0;   // 0 = MMA leader
  const int n0 = (blockIdx.x / (TWO_CTA ? 2 : KSPLIT)) * BN;
  const int m0 = TWO_CTA ? (blockIdx.y * 2 + (blockIdx.x & 1)) * kBM : blockIdx.y * kBM;
  const int nkb = ((ops.K + kBK - 1) / kBK) / KSPLIT;            // host guarantees divisibility
  const int kbase = kq * nkb * kBK + (int)blockIdx.z * ops.K;
  const int iters = nkb * ops.nterms;
  const int n_epi = KSPLIT > 1 ? n0 + 32 * kq : n0;              // first column this CTA's epilogue owns
  uint8_t* out_smem = smem + S::kRecvBytes;

  // Programmatic dependent launch: let the next kernel of the stream begin its launch/prologue now; our own reads
  // of the previous kernel's results are ordered by griddepcontrol.wait below.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (threadIdx.x == 32) {
    tma_prefetch_desc(&ops.ta[0]);
    tma_prefetch_desc(&ops.tb[0]);
  }
  if (threadIdx.x == 0) {
    trace_stamp(ops, 0);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(accum_bar, 1);
    mbar_init(in_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    if (TWO_CTA) tmem_alloc_2cta<(BN < 32 ? 32 : BN)>(tmem_holder);
    else tmem_alloc<(BN < 32 ? 32 : BN)>(tmem_holder);
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");      // previous kernel complete and its writes visible
  tc_fence_before();
  if (TWO_CTA) cluster_sync_all();                         // both CTAs' barriers initialised before remote arrives
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_holder;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      trace_stamp(ops, 1);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < iters; ++it) {
        // the epilogue's input tiles are requested once the ring is primed, so that the first MMA is not queued
        // behind them in the TMA unit
        if (Epi::kInBytes > 0 && it == (kStages < iters ? kStages : iters - 1))
          Epi::issue_loads(ep, in_smem, in_bar, m0, n_epi);
        const int term = it / nkb;
        const int k0 = kbase + (it - term * nkb) * kBK;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * S::kStageBytes;
        uint8_t* sb = sa + S::kABytes;
        if constexpr (TWO_CTA) {
          // both CTAs load their own A rows and their half of the B rows; all bytes are credited to the leader
          if (pair_rank == 0) mbar_expect_tx(&full_bar[stage], 2 * S::kStageBytes);
          if (A_MN) {
            for (int j = 0; j < kBM / 64; ++j)
              tma_load_3d_2cta(sa + j * (kBK * 128), &ops.ta[term], &full_bar[stage], m0 + 64 * j, k0, ops.za[term]);
          } else {
            tma_load_3d_2cta(sa, &ops.ta[term], &full_bar[stage], k0, m0, ops.za[term]);
          }
          if (B_MN) {
            for (int j = 0; j < BN / 128; ++j)
              tma_load_3d_2cta(sb + j * (kBK * 128), &ops.tb[term], &full_bar[stage],
                               n0 + pair_rank * (BN / 2) + 64 * j, k0, ops.zb[term]);
          } else {
            tma_load_3d_2cta(sb, &ops.tb[term], &full_bar[stage], k0, n0 + pair_rank * (BN / 2), ops.zb[term]);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
          continue;
        }
        mbar_expect_tx(&full_bar[stage], S::kStageBytes);
        if (A_MN) {
          for (int j = 0; j < kBM / 64; ++j)
            tma_load_3d(sa + j * (kBK * 128), &ops.ta[term], &full_bar[stage], m0 + 64 * j, k0, ops.za[term]);
        } else {
          tma_load_3d(sa, &ops.ta[term], &full_bar[stage], k0, m0, ops.za[term]);
        }
        if (B_MN) {
          for (int j = 0; j < BN / 64; ++j)
            tma_load_3d(sb + j * (kBK * 128), &ops.tb[term], &full_bar[stage], n0 + 64 * j, k0, ops.zb[term]);
        } else {
          tma_load_3d(sb, &ops.tb[term], &full_bar[stage], k0, n0, ops.zb[term]);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      trace_stamp(ops, 2);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = ops.f16 ? umma_idesc_f16(TWO_CTA ? 2 * kBM : kBM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0)
                                   : umma_idesc_bf16(TWO_CTA ? 2 * kBM : kBM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < (TWO_CTA && pair_rank != 0 ? 0 : iters); ++it) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      if (elect_one()) {
        if (it == 0) trace_stamp(ops, 3);
        if (it == iters - 1) trace_stamp(ops, 4);
        const uint32_t sa = smem_u32(smem + stage * S::kStageBytes);
        const uint32_t sb = sa + S::kABytes;
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k) {
          // K-major: 16 bf16 = 32 B further along the swizzled row.  MN-major: 16 k-rows = 2 KB further.
          const uint64_t da = A_MN ? umma_desc_mnmajor_sw128(sa + k * 2048, kBK * 128)
                                   : umma_desc_kmajor_sw128(sa + k * 32);
          const uint64_t db = B_MN ? umma_desc_mnmajor_sw128(sb + k * 2048, kBK * 128)
                                   : umma_desc_kmajor_sw128(sb + k * 32);
          if (TWO_CTA) umma_bf16_ss_2cta(tmem_d, da, db, idesc, (it | k) != 0 ? 1u : 0u);
          else umma_bf16_ss(tmem_d, da, db, idesc, (it | k) != 0 ? 1u : 0u);
        }
        if (TWO_CTA) {
          umma_commit_2cta(&empty_bar[stage]);              // frees the slot in both CTAs
          if (it == iters - 1) umma_commit_2cta(accum_bar);
        } else {
          umma_commit(&empty_bar[stage]);               // frees the smem slot when these MMAs retire
          if (it == iters - 1) umma_commit(accum_bar);  // accumulator complete, operand ring idle
        }
      }
      __syncwarp();
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..)
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;            // 0 (or 1 with 8 epilogue warps)
    constexpr int kChunks = BN / 32;
    constexpr int kGroups = kEpiWarps / 4;                                   // warps per TMEM lane quarter
    constexpr int kPerWarp = (kChunks >= kGroups) ? kChunks / kGroups : kChunks;
    const int row = q * 32 + lane_id();
    const int m = m0 + row;
    const bool valid = m < ops.M;
    if (Epi::kInBytes > 0) mbar_wait(in_bar, 0);
    if (threadIdx.x == 64) trace_stamp(ops, 5);
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    if (threadIdx.x == 64) trace_stamp(ops, 6);
    if constexpr (KSPLIT == 1) {
      if (kChunks >= kGroups || half == 0) {
#pragma unroll 1
        for (int cc = 0; cc < kPerWarp; ++cc) {
          const int c = (kChunks >= kGroups) ? half * kPerWarp + cc : cc;
          float acc[32];
          tmem_ld32(tmem_d + (uint32_t(q * 32) << 16) + c * 32, acc);
          tmem_ld_wait();
          Epi::apply(ep, in_smem, out_smem, row, m, n0, c, acc, valid && (n0 + c * 32 < ops.N));
        }
      }
      if (threadIdx.x == 64) trace_stamp(ops, 7);
      if (Epi::kOutBytes > 0) {
        fence_proxy_async_smem();                  // staging writes -> visible to the TMA engine
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
        if (threadIdx.x == 64) {
          trace_stamp(ops, 8);
          Epi::issue_stores(ep, out_smem, m0, n0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          trace_stamp(ops, 9);
        }
      }
    }
  }
  if constexpr (KSPLIT > 1) {
    // ---- split-K exchange (pull): every CTA parks its four partial chunks in its own (idle) ring in the swizzled
    //      tile layout; after one cluster barrier the owner of chunk kq sums the three remote copies with
    //      lane-contiguous (coalesced) distributed-shared-memory loads, in place, then reads its rows back.
    const int q = warp & 3;
    const int row = q * 32 + lane_id();
    if (warp >= 2 && warp < 6) {
#pragma unroll 1
      for (int c = 0; c < KSPLIT; ++c) {
        float acc[32];
        tmem_ld32(tmem_d + (uint32_t(q * 32) << 16) + c * 32, acc);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(smem + c * 16384 + sw128(row, j)) =
              make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
      }
    }
    cluster_sync_all();                                              // all partials parked
    if (warp >= 2) {
      if (threadIdx.x == 64) trace_stamp(ops, 7);
      const int tix = threadIdx.x - 64;
      constexpr int kThreads = 32 * kEpiWarps;
      uint8_t* mine = smem + kq * 16384;
      uint32_t peer[KSPLIT - 1];
#pragma unroll
      for (int p = 0; p < KSPLIT - 1; ++p) peer[p] = map_to_cta(smem_u32(mine), (uint32_t)((kq + 1 + p) % KSPLIT));
      constexpr int kIter = 1024 / kThreads;
      float4 rv[kIter][KSPLIT - 1];
#pragma unroll
      for (int i = 0; i < kIter; ++i)                 // all remote loads in flight before the first use
#pragma unroll
        for (int p = 0; p < KSPLIT - 1; ++p) rv[i][p] = ld_cluster_f4(peer[p] + (uint32_t)(tix + kThreads * i) * 16);
#pragma unroll
      for (int i = 0; i < kIter; ++i) {
        const uint32_t off = (uint32_t)(tix + kThreads * i) * 16;
        float4 sacc = *reinterpret_cast<const float4*>(mine + off);
#pragma unroll
        for (int p = 0; p < KSPLIT - 1; ++p) {
          sacc.x += rv[i][p].x; sacc.y += rv[i][p].y; sacc.z += rv[i][p].z; sacc.w += rv[i][p].w;
        }
        *reinterpret_cast<float4*>(mine + off) = sacc;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
      Epi::apply_from_smem(ep, in_smem, out_smem, mine, tix & 127, tix >> 7, kEpiWarps / 4);
      if (Epi::kOutBytes > 0) {
        fence_proxy_async_smem();
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");
        if (threadIdx.x == 64) {
          trace_stamp(ops, 8);
          Epi::issue_stores(ep, out_smem, m0, n_epi);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          trace_stamp(ops, 9);
        }
      }
    }
    cluster_sync_all();                                              // peers are done reading my partials
  }
  tc_fence_before();
  if (TWO_CTA) cluster_sync_all();                         // neither CTA leaves while its peer may still signal it
  else __syncthreads();
  if (warp == 1) {
    if (TWO_CTA) tmem_dealloc_2cta<(BN < 32 ? 32 : BN)>(tmem_d);
    else tmem_dealloc<(BN < 32 ? 32 : BN)>(tmem_d);
  }
  if (threadIdx.x == 0) trace_stamp(ops, 10);
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_fn();

// Tensor viewed as [d2][d1][d0] (d0 contiguous), element size 2 (bf16) or 4 (fp32) bytes; box = {box0, box1, 1};
// swizzle: 0 none, 2 = 64B, 3 = 128B (box0 * elem_bytes must equal the swizzle span); OOB -> 0 / clipped.
int make_tmap(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
              uint64_t stride1_elems, uint64_t stride2_elems, uint32_t box0, uint32_t box1, int swizzle);
// bf16 operand tile map: box = {64, box_rows, 1}, 128B swizzle.
int make_tmap_bf16(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_elems,
                   uint64_t stride2_elems, uint32_t box_rows);
// Records "<fn>: <printf-formatted message>" for svb_last_error() and returns `code`.
int host_error(int code, const char* fn, const char* fmt, ...);

template <int BN, int kStages, bool A_MN, bool B_MN, class Epi, int kEpiWarps = 4, int KSPLIT = 1, bool TWO_CTA = false>
cudaError_t launch_tc_gemm(const GemmOperands& ops, const typename Epi::Params& ep, cudaStream_t stream) {
  using S = GemmSmem<BN, kStages, Epi, KSPLIT, TWO_CTA>;
  auto kern = tc_gemm_kernel<BN, kStages, A_MN, B_MN, Epi, kEpiWarps, KSPLIT, TWO_CTA>;
  static unsigned long long configured = 0;        // one bit per device
  if (first_use_on_device(configured)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(((ops.N + BN - 1) / BN) * KSPLIT, (ops.M + kBM - 1) / kBM, ops.kz > 1 ? ops.kz : 1);
  if (TWO_CTA) {       // x = 2 * n_tiles (pair rank in the low bit), y = pairs of 128-row tiles (odd tail: all OOB)
    cfg.gridDim.x *= 2;
    cfg.gridDim.y = (cfg.gridDim.y + 1) / 2;
  }
  cfg.blockDim = dim3(64 + 32 * kEpiWarps);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (KSPLIT > 1) {
    if (((ops.K + kBK - 1) / kBK) % KSPLIT != 0) return cudaErrorInvalidValue;
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = KSPLIT;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  if (TWO_CTA) {
    attr[1].id = cudaLaunchAttributeClusterDimension;
    attr[1].val.clusterDim.x = 2;
    attr[1].val.clusterDim.y = 1;
    attr[1].val.clusterDim.z = 1;
    cfg.numAttrs = 2;
  }
  return cudaLaunchKernelEx(&cfg, kern, ops, ep);
}

}  // namespace svb
