/* svb200.h -- C ABI of libsvb200.so, the B200 (sm_100a) GE2E speaker-verification hot path.
 *
 * Plain pointers, sizes and a cudaStream_t (as void*); no torch types.  All pointers are DEVICE pointers
 * unless a parameter is documented as host.  Every function returns SVB_OK (0) or a negative SVB_ERR_*;
 * svb_last_error() gives a message.  Nothing here synchronises the stream or touches the host copy of data.
 * Each entry point names the reference code it replaces (paths relative to
 * hwidong-na/PyTorch_Speaker_Verification).
 */
#ifndef SVB200_H
#define SVB200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SVB_OK 0
#define SVB_ERR_ARG (-1)
#define SVB_ERR_CUDA (-2)
#define SVB_ERR_DRIVER (-3)
#define SVB_ERR_ALIGN (-4)
#define SVB_ERR_UNSUPPORTED (-5)

/* Version / build info: returns 100 for sm_100a builds. */
int svb_arch(void);
const char* svb_last_error(void);

/* Generic tensor-core GEMM used by the LSTM: C[M,N] = sum_t A_t[M,K] * B_t[N,K]^T (+ bias[n]).
 * bf16 operands, fp32 accumulate/out.  a_mn/b_mn = 1 when the operand is stored [K, rows] instead of [rows, K].
 * A and B are HOST arrays of nterms DEVICE pointers (nterms <= 3). Replaces the aten::addmm / cuDNN GEMMs that
 * nn.LSTM / nn.Linear issue for speech_embedder_net.py:28,31.
 * Preconditions, checked before any CUDA call:
 *   SVB_ERR_ARG unless M, N, K >= 1; 1 <= nterms <= 3; A, B and every A[t], B[t] and C are non-null;
 *     lda >= K (A K-major) or lda >= M (a_mn); ldb >= K (B K-major) or ldb >= N (b_mn); ldc >= N.
 *   SVB_ERR_ALIGN unless every A[t], B[t] is 16-byte aligned and lda, ldb are multiples of 8 elements.
 * C and bias need only float alignment: when C, bias or ldc is not 16-byte aligned, or N % 4 != 0, the epilogue
 * stores directly instead of through TMA.  Elements of C outside [0, M) x [0, N) are never written. */
int svb_gemm_bf16(const void* const* A, const void* const* B, int nterms, float* C, const float* bias, int M, int N,
                  int K, int64_t lda, int64_t ldb, int64_t ldc, int a_mn, int b_mn, void* stream);

/* Same contract and preconditions computed by CTA pairs (tcgen05.mma.cta_group::2, 256 x 256 pair tiles); mn = 0:
 * both operands K-major, mn = 1: both MN-major (a_mn = b_mn = mn above). */
int svb_gemm_bf16_2cta(const void* const* A, const void* const* B, int nterms, float* C, const float* bias, int M,
                       int N, int K, int64_t lda, int64_t ldb, int64_t ldc, int mn, void* stream);

/* Persistent CTA-pair kernel for short reductions (the LSTM input projection W_ih x_t over all frames taken as one
 * batched GEMM, speech_embedder_net.py:19,28: [T*B x 768] . [768 x 3072] at BASELINE configs[1]): C[M,N] (fp32, pitch
 * ldc) = A[M,K] . B[N,K]^T + bias[n].  Operands K-major with 2-byte elements (f16 != 0: IEEE half, else bf16);
 * K % 64 == 0, N % 256 == 0.  74 CTA pairs walk the 256 x 256 tiles; two TMEM accumulators overlap each tile's
 * epilogue with the next tile's MMAs (csrc/pgemm.cu).
 * Preconditions, checked before any CUDA call:
 *   SVB_ERR_ARG unless A, B, C are non-null; M >= 1; N a positive multiple of 256; K a positive multiple of 64;
 *     lda >= K; ldb >= K; ldc >= N and a multiple of 4; bias null or 16-byte aligned.
 *   SVB_ERR_ALIGN unless A, B and C are 16-byte aligned and lda, ldb are multiples of 8 elements.
 * Elements of C outside [0, M) x [0, N) are never written. */
int svb_gemm_persistent(const void* A, const void* B, float* C, const float* bias, int M, int N, int K, int64_t lda,
                        int64_t ldb, int64_t ldc, int f16, void* stream);

/* ---- SpeechEmbedder (speech_embedder_net.py:15-33): 3-layer LSTM + last-frame Linear + L2 norm ------------------
 * Dimensions: B utterances, T frames, I mel bins, H hidden (multiple of 128), L layers (<= 8), P projection size. */

/* Bytes of the packed bf16 weight shadow and of the per-call workspace (training != 0 keeps the BPTT stash). */
int svb_embedder_sizes(int B, int T, int I, int H, int L, int P, int training, size_t* packed_bytes,
                       size_t* workspace_bytes);

/* Re-pack the fp32 master parameters of nn.LSTM (state_dict order: weight_ih, weight_hh, bias_ih, bias_hh per layer;
 * HOST array of 4L DEVICE pointers; speech_embedder_net.py:19-24) into gate-interleaved shadows: fp16 (+ fp16
 * residual) for the forward GEMMs, bf16 transposes for the BPTT GEMMs. */
int svb_embedder_pack_weights(const float* const* params, void* packed, int I, int H, int L, void* stream);

/* SpeechEmbedder.forward (speech_embedder_net.py:27-33). x: (B,T,I) batch-first, x_dtype 0=float32 1=float64
 * (":28 x.float()"); emb: (B,P) float32 unit rows.  rec_terms = number of weight terms of the forward GEMMs
 * (1: h16 W16, persistent kernel; 2 or 3: + h16 W16_residual, per-frame kernels).  With training != 0 the workspace afterwards holds the stash that
 * svb_embedder_backward consumes. */
int svb_embedder_forward(const void* x, int x_dtype, const void* packed, const float* proj_w, const float* proj_b,
                         float* emb, void* workspace, int B, int T, int I, int H, int L, int P, int training,
                         int rec_terms, void* stream);

/* BPTT for loss.backward() (train_speech_embedder.py:62).  demb: (B,P) dL/d(embeddings).  grads: HOST array of 4L+2
 * DEVICE pointers (nn.LSTM order, then projection.weight, projection.bias), fp32, parameter layout; overwritten. */
int svb_embedder_backward(const float* demb, const void* packed, const float* proj_w, float* const* grads,
                          void* workspace, int B, int T, int I, int H, int L, int P, void* stream);

/* Host callback invoked by svb_embedder_backward as gradient buckets have been ENQUEUED on the caller's stream:
 * bucket L = projection.weight/bias, then L-1 ... 0 = the four gradients of that LSTM layer (they are contiguous when
 * the grads array points into one flat buffer in state_dict order).  A data-parallel caller starts that bucket's
 * all-reduce immediately, overlapping it with the remaining weight-gradient GEMMs.  NULL clears it. */
int svb_set_grad_ready_callback(void (*cb)(int bucket, void* user), void* user);

/* LSTM forward path: 1 (default) = persistent wavefront kernel (csrc/wlstm.cuh: all layers and frames in one
 * cooperative launch, W_hh / W_ih slices stationary in tensor memory, fp16 operands, MUFU.TANH gates, tiles ordered by
 * release counters) when H is 256/512/768, L <= 3 and rec_terms == 1; 0 = batched input projection + one fused
 * GEMM+cell launch per frame (any H % 128 == 0, split terms). */
int svb_set_persistent(int on);
/* BPTT path: 1 (default) = persistent wavefront kernel (csrc/wbptt.cuh: recurrent and dX products of all layers in
 * one cooperative cluster launch, split-K over 4-CTA clusters with a DSMEM reduction) when H == 768 and L <= 3;
 * 0 = one fused GEMM + gate-backward launch per frame and batched dX GEMMs. */
int svb_set_persistent_bwd(int on);
/* Large-batch GE2E / get_cossim (rows x centroids >= 2^18, D % 64 == 0, D <= 256): 1 (default) = the three
 * contractions run on tensor cores as 3-term split-fp16 products between the phase kernels, 0 = fp32 SIMT contractions
 * (one cooperative launch).  Both agree with the float64 oracle to 1e-5 (utils.py:72-115,126-132).  Wider D always
 * takes the SIMT contractions: the tensor-core accumulation's bias grows with D (ge2e.cu, kTcMaxD). */
int svb_set_ge2e_tensor_cores(int on);

/* ---- multi-GPU GE2E exchange over NVLink peer memory (new: the reference, speech_embedder_net.py:43-49, is
 * single-device).  `peer_ptrs_dev` is a DEVICE array of `world` float pointers: the same symmetric buffer on every rank
 * (torch.distributed._symmetric_memory: handle.buffer_ptrs_dev).  The caller separates writes and reads of the buffers
 * with the handle's barrier.  Sums are taken in rank order (identical on every rank).
 *   svb_peer_gather: out[r * n + i] = peer_r[offset + r * rank_stride + i]    (centroid all-gather: rank_stride 0; second
 *                    shot of the gradient all-reduce: rank r's reduced slice lives at r * slice in ITS buffer)
 *   svb_peer_reduce: seg_out[i] = sum_r peer_r[offset + seg_offset + i], tail_out[k] = sum_r peer_r[offset + tail_offset + k]
 *                    (this rank's rows of the centroid gradient + the loss / dw / db scalars)
 * Lengths and offsets in floats, multiples of 4 except the tail (<= 256 floats). */
int svb_peer_gather(const void* peer_ptrs_dev, int world, size_t offset_floats, size_t rank_stride_floats, size_t n_floats,
                    float* out, void* stream);
int svb_peer_reduce(const void* peer_ptrs_dev, int world, size_t offset_floats, size_t seg_offset, size_t seg_floats,
                    size_t tail_offset, int tail_floats, float* seg_out, float* tail_out, void* stream);
/* Weight gradients of the late frames beside the persistent BPTT kernel (csrc/lstm.cu): 1 (default; env
 * SVB_WGRAD_OVERLAP=0 disables) = the products dW = dG^T X over the last `pct` percent of the frames run on a
 * library-owned second stream, gated by the BPTT kernel's release counters, on the SMs it leaves idle; 0 = all
 * weight-gradient GEMMs after it.  svb_wgrad_overlap_timing (SVB_WGRAD_DEBUG=1): ms since the fork of the last
 * backward for {gate of the top layer open, side stream done, BPTT done, backward done}; synchronises. */
int svb_set_wgrad_overlap(int on);
int svb_set_wgrad_late_pct(int pct);
int svb_wgrad_overlap_timing(float* out4);
/* Debug hooks of the persistent kernels (timing experiments only): ablation mask (results become garbage) and
 * clock64 trace buffers (device pointers, or NULL). */
int svb_set_ablate(int mask);
int svb_set_trace_mode(int mode);   /* 1: per-tile stamps of frame T/2, 2: per-role wait accounting (scripts/account_wlstm.py) */
int svb_set_trace(unsigned long long* device_buffer);
int svb_set_trace_bwd(unsigned long long* device_buffer);

/* Optional phase timing (CUDA events around the phases of forward/backward; none inside the per-frame loops).
 * Phases: 0 prep, 1 input GEMM, 2 recurrent fwd, 3 projection, 4 projection bwd, 5 recurrent bwd, 6 weight grads,
 * 7 bias grads, 8 dX.  svb_profile_read sums elapsed ms per phase since the last enable/read (sync the stream first). */
int svb_profile_enable(int on);
int svb_profile_read(float* ms_per_phase, int nphases);

/* Launch counter (measurement only; bench.py's gpu_launches): between begin and end, every kernel launch of the process
 * is seen through CUPTI's callback API; `ours` = launches whose host stub lives in this library, `other` = everyone
 * else's (torch, NCCL); names = "mangled_kernel_name=count;..." of ours.  SVB_ERR_UNSUPPORTED when libcupti cannot be
 * opened or another CUPTI client (a profiler) is attached. */
int svb_launch_count_begin(void);
int svb_launch_count_end(long long* ours, long long* other, char* names, size_t names_bytes);

/* ---- GE2E loss (speech_embedder_net.py:35-49, utils.py:27-132) ---------------------------------------------------- */

/* GE2E loss methods (Wan et al., arXiv 1710.10467):
 *   SVB_GE2E_SOFTMAX  eq. 6, the reference's calc_loss (utils.py:126-132): per = -S_jj + log(sum_k exp S_jk + 1e-6);
 *   SVB_GE2E_CONTRAST eq. 7: per = 1 - sigmoid(S_jj) + sigmoid(S_jk*), k* = argmax_{k != j} S_jk (lowest index among
 *                     ties).  Needs at least two centroid columns.  The loss is the SUM over rows for both. */
#define SVB_GE2E_SOFTMAX 0
#define SVB_GE2E_CONTRAST 1

int svb_ge2e_workspace_bytes(int N, int M, int D, int Nc, size_t* bytes);
/* Debug (env SVB_GE2E_TRACE=1): byte offset inside the workspace of the per-speaker kernel's clock64 phase stamps,
 * [CTA][16] int64 (scripts/trace_ge2e.py). */
int svb_ge2e_trace_offset(int N, int M, int D, int Nc, size_t* offset);

/* One fused kernel for get_centroids + get_utterance_centroids + get_cossim (+ w*cos+b, calc_loss and all gradients).
 *   E (N,M,D); Cext (Nc,D) foreign centroids or NULL (centroids of E, Nc == N);
 *   w,b device scalars (NULL,NULL: cosine matrix only); dcos (N,M,Nc) upstream gradient for get_cossim's backward;
 *   gscale device scalar multiplying every gradient or NULL.
 * Outputs (any may be NULL): cos_out (N,M,Nc) incl. the +1e-6 of utils.py:114; per_out (N,M) per-embedding loss;
 *   loss_out scalar (SUM, utils.py:131); dE (N,M,D); dCext (Nc,D); dw, db scalars.
 * fused = 1: single cooperative launch; loss batches with N <= #SMs, M <= 16, D % 4 == 0 (the reference's training
 *   batches) take the per-speaker kernel (3 phases, 2 grid barriers; one 2-CTA cluster per speaker, each CTA owning
 *   half of D, when D % 8 == 0 and 2N <= #SMs, else one CTA per speaker), everything else the general 5-phase
 *   kernel; fused = 2: always the general kernel; 0: one launch per phase (debug). */
int svb_ge2e(const float* E, const float* Cext, int N, int M, int D, int Nc, const float* w, const float* b,
             const float* dcos, const float* gscale, float* cos_out, float* per_out, float* loss_out, float* dE,
             float* dCext, float* dw, float* db, void* workspace, size_t workspace_bytes, int fused, void* stream);
/* svb_ge2e with a loss method (SVB_GE2E_*); svb_ge2e is svb_ge2e_ex(..., SVB_GE2E_SOFTMAX, stream).  The contrast
 * method is a loss: it needs w and b, and has no cosine-only or dcos mode.  Its backward gathers one centroid per row
 * (no dense A_off products); the workspace size is the same. */
int svb_ge2e_ex(const float* E, const float* Cext, int N, int M, int D, int Nc, const float* w, const float* b,
                const float* dcos, const float* gscale, float* cos_out, float* per_out, float* loss_out, float* dE,
                float* dCext, float* dw, float* db, void* workspace, size_t workspace_bytes, int fused, int loss,
                void* stream);

/* Row shard of a global GE2E batch (new: multi-GPU, one process per GPU; the reference is single-device).  E: the M
 * utterances of speakers [col0, col0 + N_local) of a batch of Nc speakers; C (Nc, D): all centroids (utils.py:27-29 of
 * every rank's shard, all-gathered).  Same arithmetic as svb_ge2e on the global batch restricted to these rows, with the
 * rows' own column col0 + j as the leave-one-out diagonal (utils.py:91,113).  loss_out / dw / db: the shard's partial
 * sums; dE (N_local, M, D): without the path through the rows' own centroid; dC (Nc, D): the shard's contribution to
 * every centroid's gradient.  The caller sums loss, dw, db, dC over the ranks and adds dC_total[col0 + j] / M to every
 * utterance of speaker j (svb_centroids_bwd). */
int svb_ge2e_rows(const float* E, const float* C, int N_local, int M, int D, int Nc, int col0, const float* w,
                  const float* b, const float* gscale, float* per_out, float* loss_out, float* dE, float* dC, float* dw,
                  float* db, void* workspace, size_t workspace_bytes, void* stream);
/* svb_ge2e_rows with a loss method (SVB_GE2E_*). */
int svb_ge2e_rows_ex(const float* E, const float* C, int N_local, int M, int D, int Nc, int col0, const float* w,
                     const float* b, const float* gscale, float* per_out, float* loss_out, float* dE, float* dC,
                     float* dw, float* db, void* workspace, size_t workspace_bytes, int loss, void* stream);

/* utils.get_centroids (utils.py:27-29) and its backward. */
int svb_centroids(const float* E, float* C, int N, int M, int D, void* stream);
int svb_centroids_bwd(const float* dC, float* dE, int N, int M, int D, void* stream);

/* utils.get_utterance_centroids (utils.py:40-58): U (N,M,D) = (sum over a speaker's utterances - the utterance itself)
 * / (M - 1), float32 operations in the reference's order (bit-exact for D >= 16).  The operator is its own adjoint: the
 * backward pass calls it on dL/dU. */
int svb_utterance_centroids(const float* E, float* U, int N, int M, int D, void* stream);

/* utils.calc_loss (utils.py:126-132) on a caller-supplied similarity matrix S (N,M,Nc); dS optional. */
int svb_calc_loss(const float* S, int N, int M, int Nc, float* per_out, float* loss_out, float* dS,
                  const float* gscale, void* stream);
/* svb_calc_loss with a loss method (SVB_GE2E_*): dS = gscale * dL/dS of that method. */
int svb_calc_loss_ex(const float* S, int N, int M, int Nc, float* per_out, float* loss_out, float* dS,
                     const float* gscale, int loss, void* stream);

/* x[i] *= *g for three buffers in one launch (autograd's upstream scalar). */
int svb_scale3(float* a, size_t na, float* b, size_t nb, float* c, size_t nc, const float* g, void* stream);

/* ---- optimizer tail of the training step (SURVEY.md section 8(f) rank 1; train_speech_embedder.py:33-36,63-65) ----- */

int svb_clip_sgd_workspace_bytes(size_t* bytes);
/* clip_grad_norm_ per clip group followed by the plain SGD step, two launches for all tensors:
 *   total_norm_g = sqrt(sum over the group's tensors of sum g^2); coef_g = min(1, max_norm_g / (total_norm_g + 1e-6));
 *   g <- coef_g * g (stored only if write_clipped_grads != 0, as clip_grad_norm_ does in place); p <- p - lr * g.
 * params/grads: HOST arrays of n_tensors (<= 32) DEVICE float32 pointers; numel, group (clip group of each tensor,
 * < n_groups <= 4) and max_norm (per group; <= 0 disables clipping) are HOST arrays; norms_out (device, n_groups
 * floats, may be NULL) receives the pre-clip total norms that clip_grad_norm_ returns. */
int svb_clip_sgd(void* const* params, void* const* grads, const int64_t* numel, const int32_t* group, int n_tensors,
                 const float* max_norm, int n_groups, float lr, int write_clipped_grads, float* norms_out,
                 void* workspace, size_t workspace_bytes, void* stream);

/* ---- TI-SV EER sweep (train_speech_embedder.py:132-149) ---------------------------------------------------------- */

/* Exact integer counts of sim > thresholds[t] for speakers [speaker0, speaker0+n_local): sim (n_local, Mv, Nc) float32,
 * thresholds ascending float32 (device, T <= 128); cnt_all/cnt_diag (n_local, T) int32. */
int svb_eer_counts(const float* sim, int n_local, int Mv, int Nc, int speaker0, const float* thresholds, int T,
                   int* cnt_all, int* cnt_diag, void* stream);
/* Reference float32 arithmetic on the counts of all N speakers -> out[0..3] = EER, selected threshold index (-1: none),
 * FAR, FRR; out[4..4+T) = FAR per threshold, out[4+T..4+2T) = FRR per threshold. */
int svb_eer_finish(const int* cnt_all, const int* cnt_diag, int N, int Mv, int T, float* out, void* stream);

/* Single-launch sweep for one GPU: per-speaker counts, integer totals (atomics) and the selection above, done by the
 * last block.  scratch: 1 + 16T uint64 zeroed by the caller.  out[1] == -2: a total exceeded 2^24, so float32 partial
 * sums are no longer exact -- call svb_eer_finish on the returned per-speaker counts instead. */
int svb_eer_sweep(const float* sim, int N, int Mv, const float* thresholds, int T, int* cnt_all, int* cnt_diag,
                  unsigned long long* scratch, float* out, void* stream);

/* ---- exact EER and minDCF over every score threshold (new; DESIGN.md 4.5) ----------------------------------------
 * Operating point k of the K distinct scores v_1 < ... < v_K accepts the scores >= v_{k+1} (point K accepts nothing,
 * threshold +inf).  EER: the point with the smallest |miss * Nn - fa * Nt| (exact integers, ties to the smaller k),
 * reported as (p_miss + p_fa) / 2.  minDCF of each operating point (w_miss, w_fa, c_def): the smallest
 * (w_miss * p_miss + w_fa * p_fa) / c_def, every float64 operation rounded separately, ties to the smaller k.  -0.0 counts
 * as +0.0.  Bit-exact and run-to-run identical.  2 <= n < 2^31.
 * The workspace (about 18.04 n bytes) holds two 8n-byte element buffers, the radix sort's per-tile digit count / offset
 * table (8 KB per 4096 scores, rewritten by every pass), a counter region that every call clears (cudaMemsetAsync on
 * `stream`: 24 KB plus 4 B per 4096 scores) and the sweep's per-tile results (148 B per 4096 scores).  No allocation
 * and no host synchronisation, so the calls can be captured in a CUDA graph. */
int svb_verif_workspace_bytes(int64_t n, size_t* bytes);
/* ops: HOST array of 3*P doubles {w_miss, w_fa, c_def} per operating point, 1 <= P <= 8.
 * out (device, 8 + 4P doubles): eer, eer threshold, eer p_miss, eer p_fa, Nt, Nn, #non-finite scores, K,
 * then per point: min_dcf, threshold, p_miss, p_fa.  With a non-finite score or an empty class the metrics are NaN.
 * labels: n bytes, nonzero = target. */
int svb_verif_metrics(const float* scores, const uint8_t* labels, int64_t n, const double* ops, int P,
                      void* workspace, size_t workspace_bytes, double* out, void* stream);
/* The same for a TI-SV similarity matrix sim (N, Mv, N) (svb_eer_sweep's input): element [j, m, k] is a target trial
 * iff k == j, the pooled trials behind the reference's FAR and FRR.  n = N * Mv * N, N >= 2. */
int svb_verif_metrics_sim(const float* sim, int N, int Mv, const double* ops, int P,
                          void* workspace, size_t workspace_bytes, double* out, void* stream);

/* ---- score calibration and calibration metrics (new; DESIGN.md 4.5.3) ---------------------------------------------
 * Scores are float32 natural-log likelihood ratios l; Nt / Nn are the target / non-target counts.  -0.0 counts as +0.0,
 * denormals stay distinct; a non-finite score makes every metric NaN.
 *   Cllr = 1/2 [ (1/Nt) sum_tar softplus(-l) + (1/Nn) sum_non softplus(l) ] / ln 2,  softplus(x) = log(1 + e^x).
 *   Actual DCF of an operating point (w_miss, w_fa, c_def) (as svb_verif_metrics takes them): threshold
 *   theta = log(w_fa / w_miss) (host float64); a trial is accepted iff (double)l >= theta; miss = targets below theta,
 *   fa = non-targets at or above it; act_dcf = (w_miss * miss/Nt + w_fa * fa/Nn) / c_def, every float64 operation
 *   rounded separately.
 *   minCllr: the Cllr after the optimal non-decreasing map from score to LLR (PAV, tied scores pooled).  With the
 *   cumulative points (X_g, Y_g) = (trials, targets in the groups of equal scores up to g), from (0, 0), it is read off
 *   their lower convex hull: a hull segment of m trials, t targets and f = m - t non-targets adds t log2(1 + f Nt/(t Nn))
 *   to the target sum and f log2(1 + t Nn/(f Nt)) to the non-target sum (a term with a zero count adds 0), and
 *   minCllr = 1/2 (target sum / Nt + non-target sum / Nn).  Hull tests are exact int64 cross products; collinear points
 *   are dropped.
 *   ROCCH-EER: the hull vertices as ROC points (P_miss = Y/Nt, P_fa = (Nn - (X - Y))/Nn); the value e where that
 *   polyline crosses P_miss = P_fa, in float64.
 *   Linear calibration at prior pi, tau = logit(pi): (a, b) minimises
 *   C(a, b) = (pi/Nt) sum_tar softplus(-(a s + b + tau)) + ((1 - pi)/Nn) sum_non softplus(a s + b + tau).  A finite,
 *   unique minimiser exists iff min_tar < max_non and min_non < max_tar.  At pi = 1/2, C / ln 2 is the Cllr of a s + b.
 * Float64 sums in a fixed order, no float atomics: run-to-run and stream-to-stream identical.  No allocation and no host
 * synchronisation, so both calls can be captured in a CUDA graph.  2 <= n < 2^31.
 * The workspace (about 18.04 n bytes, 256-byte aligned) serves both calls: svb_verif_metrics' sort buffers (the first
 * holds the convex hulls once the sort is done), 12 B per 4096 scores of hull bookkeeping, per-block partials. */
#define SVB_CALIB_CONVERGED 0
#define SVB_CALIB_SEPARABLE 1          /* the classes do not overlap strictly (includes fewer than two distinct scores) */
#define SVB_CALIB_ITERATION_CAP 2      /* max_iter passes without convergence */
#define SVB_CALIB_BAD_INPUT 3          /* an empty class or a non-finite score */
int svb_calib_workspace_bytes(int64_t n, size_t* bytes);
/* ops: HOST array of 3*P doubles {w_miss, w_fa, c_def}, 1 <= P <= 8.  out (device, 8 + 4P doubles): cllr, min_cllr,
 * rocch_eer, Nt, Nn, #non-finite scores, #hull vertices (with the origin), K (distinct scores), then per point:
 * act_dcf, theta, p_miss, p_fa.  labels: n bytes, nonzero = target. */
int svb_calib_metrics(const float* llr, const uint8_t* labels, int64_t n, const double* ops, int P,
                      void* workspace, size_t workspace_bytes, double* out, void* stream);
/* Damped Newton from (a, b) = (0, 0): one fused pass over the scores (objective, gradient, Hessian) and a one-block
 * update per iteration, max_iter >= 1 of them enqueued; it stops when half the squared Newton decrement is <= 1e-12
 * (then takes that last step without a line search).  0 < prior < 1.  out (device, 5 doubles): a, b, C(a, b) / ln 2,
 * iterations (objective evaluations), status (SVB_CALIB_*); a, b and C are NaN unless the status is CONVERGED or
 * ITERATION_CAP. */
int svb_calib_train(const float* scores, const uint8_t* labels, int64_t n, double prior, int max_iter,
                    void* workspace, size_t workspace_bytes, double* out, void* stream);

/* ---- cohort score normalization: S-norm and adaptive S-norm (new; DESIGN.md 4.5.2) --------------------------------
 * cos(x, y) = (x / |x|) . (y / |y|); a row with a zero or non-finite norm makes every score and statistic it takes part
 * in NaN.  Cohort statistics of a row x against a cohort C of Nc rows with top-K (2 <= K <= Nc; K = Nc is plain S-norm):
 * S_K(x) = the multiset of the K largest cos(x, c), mu = mean of S_K(x), sigma = sample standard deviation of S_K(x)
 * (divisor K - 1), v_K = the K-th largest value.  -0.0 counts as +0.0; a non-finite cohort score makes the row's three
 * statistics NaN.  Statistics are accumulated and returned in float64 (fixed reduction order, no float atomics:
 * run-to-run identical).  Normalized score of a trial (e, t) with raw score s:
 *   s' = 1/2 ((s - mu(e)) / sigma(e) + (s - mu(t)) / sigma(t)),  returned as float32.
 * No allocation and no host synchronisation, so every call can be captured in a CUDA graph. */

/* Workspace of svb_cohort_stats: the cohort's and one chunk's fp16 hi / lo splits (zero-padded to round64(D) columns,
 * the cohort to a multiple of 8 rows) and the chunk's fp32 score slab (about 48 MB).  1 <= n < 2^31, 2 <= Nc <= 2^20,
 * 1 <= D <= 65536. */
int svb_cohort_stats_workspace_bytes(int64_t n, int Nc, int D, size_t* bytes);
/* X (n, D), cohort (Nc, D) float32 row-major -> out (n, 3) float64: mu, sigma, v_K.  2 <= K <= Nc.  Cohort cosines are
 * 3-term split-fp16 tensor-core products (about 2^-22 relative); the workspace is 256-byte aligned. */
int svb_cohort_stats(const float* X, int64_t n, const float* cohort, int Nc, int D, int K, void* workspace,
                     size_t workspace_bytes, double* out, void* stream);
/* The same statistics of caller-supplied cohort scores: row i is scores[i * ld, i * ld + Nc).  ld >= Nc. */
int svb_cohort_stats_scores(const float* scores, int64_t n, int Nc, int64_t ld, int K, double* out, void* stream);
/* out[i] = cos(E[ei[i]], T[ti[i]]) for E (ne, D), T (nt, D), int32 indices (validated by the caller: an index out of
 * range gives NaN and reads nothing); with stats_e (ne, 3) and stats_t (nt, 3) from svb_cohort_stats the normalized
 * score instead.  stats_e and stats_t are both NULL (raw cosine) or both given. */
int svb_score_trials(const float* E, int64_t ne, const float* T, int64_t nt, int D, const int32_t* ei,
                     const int32_t* ti, int64_t n_trials, const double* stats_e, const double* stats_t, float* out,
                     void* stream);
/* TI-SV matrix sim (N, Mv, N) (svb_verif_metrics_sim's input): out[j, m, k] = the normalized score of sim[j, m, k] with
 * stats_c (N, 3) of the enrollment centroids k and stats_v (N * Mv, 3) of the verification utterances [j, m]. */
int svb_asnorm_sim(const float* sim, int N, int Mv, const double* stats_c, const double* stats_v, float* out,
                   void* stream);

/* ---- d-vector extraction (dvector_create.py:48-52,98-99 and :55-73) ----------------------------------------------- */

/* Sliding windows of a (nmels, Ttot) log-mel matrix (row pitch ldS) -> (W, win, nmels); win_start (W) int32 device. */
int svb_dvector_windows(const float* S, int64_t ldS, int nmels, const int* win_start, int W, int win, float* out,
                        void* stream);
/* align_embeddings: out[p,:] = float64(mean over rows [seg_offsets[p], seg_offsets[p+1]) of emb (W,D) float32). */
int svb_segment_mean(const float* emb, int D, const int* seg_offsets, int P, double* out, void* stream);

/* ---- log-mel front end (SURVEY.md section 8(f) rank 4; data_preprocess.py:41-45, dvector_create.py:43-47) ----------
 * PCM y (n float32 samples) -> out (nmels, n_frames) float32 = log10(mel_w . |STFT|^2 + 1e-6), n_frames = 1 + n/hop,
 * n_fft = 512, librosa.core.stft framing (center=True, reflect padding).  window: 512 floats (the analysis window
 * zero-padded to n_fft, non-zero on [w0, w1)); twiddle: 512 (cos, sin) pairs of 2 pi j / 512; mel_w: (nmels, 257).
 * All tables are device pointers (pytorch_speaker_verification_b200/frontend.py builds them in float64). */
int svb_logmel(const float* y, int64_t n, int hop, const float* window, int w0, int w1, const float* twiddle,
               const float* mel_w, int nmels, float* out, int n_frames, void* stream);

/* ---- TI-SV training-set preprocessing (data_preprocess.py save_spectrogram_tisv; new: DESIGN.md 4.8) ---------------
 * Silence split, librosa 0.6 effects.split(y, top_db, ref=np.max, frame_length=2048, hop_length=512), for a signal y of
 * n > 1024 samples:
 *   pad y with 1024 samples on each side, reflecting without repeating the edge sample (np.pad(mode="reflect"));
 *   F = 1 + n / 512 frames; frame t covers padded samples [512 t, 512 t + 2048) and p_t = the mean of their squares,
 *   in float64 (the squares of float32 samples are exact) with a fixed order: per 512-sample block a fixed sum, then
 *   p_t = ((B_t + B_t+1) + (B_t+2 + B_t+3)) / 2048;
 *   frame t is non-silent iff 10 log10(max(1e-10, p_t)) - 10 log10(max(1e-10, max_t p_t)) > -top_db;
 *   the interval edges are the frames t where the mask changes (frames outside [0, F) count as silent), times 512,
 *   clipped to n, paired as half-open [start, end).
 * So an all-zero signal is one interval [0, n), top_db <= 0 gives none, and a last interval may be empty ([n, n] when
 * n % 512 == 0).  librosa >= 0.10 pads with zeros instead, which can change frames 0 and F - 1 only.
 * Signals with n <= 1024 give no interval.  Interval counts of one signal are at most (F + 1) / 2. */

/* Bytes of svb_split_nonsilent's workspace: (4 n_signals + total_samples / 512) doubles of block sums. */
int svb_split_workspace_bytes(int64_t total_samples, int n_signals, size_t* bytes);
/* The intervals of n_signals signals concatenated in y: signal i is y[offsets[i], offsets[i+1]) (offsets: device,
 * n_signals + 1 ascending int64, offsets[0] = 0, offsets[n_signals] = total_samples).  Only intervals with
 * end - start >= min_len are kept (min_len = 0 keeps every one; data_preprocess.py's `> utter_min_len` is
 * min_len = floor(utter_min_len) + 1).  Signal i's kept intervals go, in order, to the int64 pairs
 * intervals[2 slot_offsets[i] ...] (sample offsets within the signal); slot_offsets (device, n_signals int64) must
 * leave (F_i + 1) / 2 pairs to signal i (F_i = 0 for n_i <= 1024).  counts[i] (device int64) = the number of kept
 * intervals, or -1 when signal i holds a non-finite sample.  Two launches; no allocation, synchronisation or float
 * atomics: identical from run to run and across streams.  SVB_ERR_ARG before any launch unless n_signals >= 0,
 * total_samples >= 0, min_len >= 0, top_db is not NaN, the pointers are non-null and the workspace is 8-byte aligned
 * and large enough. */
int svb_split_nonsilent(const float* y, const int64_t* offsets, int n_signals, int64_t total_samples, double top_db,
                        int64_t min_len, const int64_t* slot_offsets, void* workspace, size_t workspace_bytes,
                        int64_t* intervals, int64_t* counts, void* stream);
/* Log-mel frames of many segments of y in one launch, the same device code and bits as svb_logmel on the segment:
 * rows (device, P x 3 int64) = {segment start in y, segment length L >= 1, first frame f0}; out (P, nmels,
 * frames_per_row) float32, out[p, :, j] = frame f0 + j of svb_logmel(y + start, L, ...), the reflect padding taken at
 * the segment's bounds (repeatedly when a frame reaches more than L - 1 samples past them, as np.pad does).  The
 * caller keeps f0 + frames_per_row <= 1 + L / hop when it wants frames librosa would give.  Other arguments as
 * svb_logmel.  SVB_ERR_ARG before any launch unless P >= 0, frames_per_row >= 1, hop >= 1, nmels >= 1,
 * 0 <= w0 < w1 <= 512, the pointers are non-null (P > 0) and P * frames_per_row < 2^34. */
int svb_logmel_frames(const float* y, const int64_t* rows, int64_t P, int frames_per_row, int hop, const float* window,
                      int w0, int w1, const float* twiddle, const float* mel_w, int nmels, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif
