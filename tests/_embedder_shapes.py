"""Model dimensions at which the SpeechEmbedder kernels are checked against the float64 oracle, one row per set of
kernel routes (csrc/lstm.cu, svb_embedder_forward / svb_embedder_backward).

The reference's hparams (nmels, hidden, num_layer, proj) are honoured by the C ABI for any nmels, any hidden that is
a multiple of 128, 1 to 8 layers and any proj; the dispatch between the persistent kernels (wlstm.cuh, wbptt.cuh),
the per-frame kernels and the weight-gradient GEMM variants depends on exactly these four numbers and on the batch and
frame counts.  Each row names the routes it exists to cover.  The expected routes assume a full B200 (148 SMs); the
route test asserts them from the kernels that actually launched.

  fwd   "wlstm": persistent forward wlstm_fwd_kernel<H>;  "frame": per-frame GEMM + cell kernels (EpiLstmFwd)
  bwd   "wbptt": persistent BPTT wbptt_kernel<768>;       "frame": per-frame BPTT kernels (EpiLstmBwd)
"""
from collections import namedtuple

Case = namedtuple("Case", "id nmels hidden num_layer proj fwd bwd shapes covers")

# (B, T): batch 1 and frame 1; ragged batches of one and two 64-row tiles plus one row; and one long shape with
# T*B = 4160 >= 4096, T >= 16 and a ragged last tile, which switches on the 6-way split of the narrow dW_ih, the
# split-K pair tiles of dW_hh and (at H = 768) the weight-gradient overlap.
EDGES = ((1, 1), (65, 2), (129, 3))
LONG = (130, 32)
SHAPES = EDGES + (LONG,)

CASES = [
    Case("A", 40, 256, 1, 64, "wlstm", "frame", SHAPES,
         "wlstm<256> with L = 1; per-frame BPTT; dW_hh split-K pair tiles (split2); narrow dW_ih with kz = 6 (long) "
         "and kz = 1 (short); no dX"),
    Case("B", 80, 512, 2, 128, "wlstm", "frame", SHAPES,
         "wlstm<512> with L = 2 and two layer-0 K blocks; dX on 256-wide pair tiles; layer-1 dW_ih split2 (I = H)"),
    Case("C", 13, 384, 2, 100, "frame", "frame", SHAPES,
         "per-frame forward (H = 384); layer-0 padding Ip 13 -> 16; dW_hh on 256 x 128 pair tiles; 128-wide dX; "
         "layer-1 dW_ih on the I % 128 path; P = 100"),
    Case("D", 128, 768, 1, 256, "wlstm", "wbptt", SHAPES,
         "wlstm<768> and wbptt with L = 1; weight-gradient overlap with one layer; dW_ih on the I % 128 path"),
    Case("E", 40, 768, 2, 256, "wlstm", "wbptt", SHAPES,
         "wlstm<768> and wbptt with L = 2; overlap including the layer-1 dW_ih product"),
    Case("F", 256, 256, 4, 256, "frame", "frame", SHAPES,
         "L = 4: per-frame forward and BPTT; layer-0 dW_ih split2 (I % 256 == 0, I <= H)"),
    Case("G", 40, 1024, 1, 512, "frame", "frame", SHAPES,
         "per-frame at the widest gate row (4H = 4096)"),
    Case("H", 40, 128, 3, 32, "frame", "frame", SHAPES,
         "per-frame at the smallest H"),
    Case("I", 768, 256, 1, 64, "wlstm", "frame", SHAPES,
         "layer-0 weights of wlstm fill tensor memory exactly up to the accumulators (12 K blocks = 384 columns)"),
    Case("I+", 776, 256, 1, 64, "frame", "frame", SHAPES,
         "one layer-0 K block past that limit: must leave the persistent forward for the per-frame one"),
    Case("J", 40, 384, 1, 64, "frame", "frame", ((1100, 3),),
         "per-frame recurrence on CTA pairs (fwd_pair, B > 1024)"),
    Case("K", 40, 768, 3, 256, "wlstm", "wbptt", EDGES,
         "the default model at the edge shapes"),
]
BY_ID = {c.id: c for c in CASES}


def wgrad_overlap(case, B, T):
    """The late-frame weight-gradient slices run beside the persistent BPTT kernel (lstm.cu: H % 256 == 0, T >= 16,
    T*B >= 4096)."""
    return case.bwd == "wbptt" and T >= 16 and T * B >= 4096


def narrow_kz6(case, B, T):
    """Layer 0's dW_ih takes the narrow path (I % 128 != 0) with its reduction split six ways (summed by sumz_kernel)."""
    I, H = case.nmels, case.hidden
    return I % 128 != 0 and T * B >= 4096 and 6 * I <= 2 * H


def param_names(num_layer):
    return [f"LSTM_stack.{k}_l{l}" for l in range(num_layer)
            for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")] + ["projection.weight", "projection.bias"]
