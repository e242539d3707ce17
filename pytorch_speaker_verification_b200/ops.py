"""Host-side operators: the C ABI (include/svb200.h) registered as torch custom ops, namespace ``svb200``.

Every kernel entry point of libsvb200.so is wrapped once, here, as ``torch.ops.svb200.<name>`` (schema + CUDA
implementation + fake/meta implementation + autograd formula where the reference's function is differentiable).  The
implementations only allocate outputs and marshal pointers, sizes and the current stream of the tensors' device into
the C call; every arithmetic step runs in the library.  The ops are registered for the CUDA dispatch key only: there
is no CPU kernel behind them, so a CPU tensor reaching an op raises (no fallback).

The functions below the registrations are the thin boundary layer the drop-in modules call: they accept what the
reference's callers pass (CPU tensors in test() / dvector_create.py, float64 inputs), stage it to the GPU with
differentiable ``.to()`` calls and return results on the caller's device.
"""
import ctypes
import os
from typing import List, Optional, Tuple

import torch

from . import _lib
from ._lib import check, ptr

_POISON = os.environ.get("SVB_POISON_WORKSPACE", "0") == "1"
_i64 = ctypes.c_int64
_sz = ctypes.c_size_t
NS = "svb200"
_LIB = torch.library.Library(NS, "DEF")          # keeps the registrations alive for the life of the process


# ------------------------------------------------------------------------------------------ devices and streams
def _dev():
    if not torch.cuda.is_available():
        raise _lib.SvbError("a CUDA device (B200, sm_100a) is required: there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _target_device(*tensors):
    """The CUDA device the call runs on: the device of its CUDA tensors (they must agree), else the current device."""
    dev = None
    for t in tensors:
        if t is not None and t.is_cuda:
            if dev is None:
                dev = t.device
            elif t.device != dev:
                raise _lib.SvbError(f"tensors on different CUDA devices ({dev} and {t.device})")
    return dev if dev is not None else _dev()


def _stage(t, dtype=None, device=None):
    """-> contiguous CUDA tensor on ``device`` (default: its own CUDA device, else the current one), optionally cast.
    Differentiable: gradients flow back to a CPU tensor through the copy."""
    d = device if device is not None else (t.device if t.is_cuda else _dev())
    if t.device != d:
        t = t.to(d, non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _back(t, device):
    return t if t.device == device else t.to(device)


def _ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def _op(schema, impl, fake):
    name = schema.split("(")[0]
    _LIB.define(schema)
    _LIB.impl(name, impl, "CUDA")
    torch.library.register_fake(f"{NS}::{name}", fake)


def _f32(t, *shape):
    return torch.empty(shape, dtype=torch.float32, device=t.device)


# ------------------------------------------------------------------------------------------ debug switches
def set_poison_workspace(on):
    """Debug: NaN-fill every forward workspace (and the GE2E outputs), so that a kernel reading a slot before it is
    written, or leaving an output element unwritten, shows up."""
    global _POISON
    _POISON = bool(on)


def set_persistent(on):
    """Select the LSTM forward path: True (default) persistent wavefront kernel (csrc/wlstm.cuh), False per-frame
    launches (csrc/lstm.cu)."""
    check(_lib.lib().svb_set_persistent(int(bool(on))), "svb_set_persistent")


def set_persistent_bwd(on):
    """Select the BPTT path: True (default) persistent wavefront kernel (csrc/wbptt.cuh), False per-frame launches."""
    check(_lib.lib().svb_set_persistent_bwd(int(bool(on))), "svb_set_persistent_bwd")


def set_ge2e_tensor_cores(on):
    """True (default): large GE2E / get_cossim problems run their three contractions on tensor cores (3-term split
    fp16); False: the fp32 SIMT kernel."""
    check(_lib.lib().svb_set_ge2e_tensor_cores(int(bool(on))), "svb_set_ge2e_tensor_cores")


def set_wgrad_overlap(on):
    """True (default): the weight-gradient products over the late frames run on a second stream beside the persistent
    BPTT kernel (which leaves 28 SMs idle); False: all of them after it."""
    check(_lib.lib().svb_set_wgrad_overlap(int(bool(on))), "svb_set_wgrad_overlap")


_GRAD_CB = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.c_void_p)
_bucket_hook = None
_bucket_finish = None


def set_grad_bucket_hook(fn, finish=None):
    """fn(bucket: 1-D view of the flat gradient buffer) is called during backward as soon as a bucket's kernels are
    enqueued on the current stream (projection first, then the LSTM layers from the top); ``finish()`` is called once
    all buckets have been handed out and BEFORE the gradients are returned to autograd, so that whatever the hook
    started (asynchronous all-reduces) is ordered before autograd accumulates the buckets into ``p.grad``.
    None clears both."""
    global _bucket_hook, _bucket_finish
    _bucket_hook, _bucket_finish = fn, finish


# ------------------------------------------------------------------------------------------ embedder ops
def _embedder_sizes(B, T, I, H, L, P, training):
    packed, work = _sz(0), _sz(0)
    check(_lib.lib().svb_embedder_sizes(B, T, I, H, L, P, int(training), ctypes.byref(packed), ctypes.byref(work)),
          "svb_embedder_sizes")
    return packed.value, work.value


def _pack_weights(lstm_params: List[torch.Tensor], I: int, H: int, L: int) -> torch.Tensor:
    dev = lstm_params[0].device
    with torch.cuda.device(dev):
        ps = [p.detach().contiguous() for p in lstm_params]
        nbytes, _ = _embedder_sizes(1, 1, I, H, L, 1, 0)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        check(_lib.lib().svb_embedder_pack_weights(_ptr_array(ps), ptr(buf), I, H, L, stream_ptr(dev)),
              "svb_embedder_pack_weights")
    return buf


def _pack_weights_fake(lstm_params, I, H, L):
    return lstm_params[0].new_empty(_embedder_sizes(1, 1, I, H, L, 1, 0)[0], dtype=torch.uint8)


_op("pack_weights(Tensor[] lstm_params, int I, int H, int L) -> Tensor", _pack_weights, _pack_weights_fake)


def _embedder_fwd(x: torch.Tensor, params: List[torch.Tensor], packed: torch.Tensor, H: int, L: int, training: bool,
                  rec_terms: int) -> Tuple[torch.Tensor, torch.Tensor]:
    B, T, I = (int(s) for s in x.shape)
    proj_w, proj_b = params[4 * L].contiguous(), params[4 * L + 1].contiguous()
    P = int(proj_w.shape[0])
    dev = x.device
    with torch.cuda.device(dev):
        x = x.contiguous()
        _, wbytes = _embedder_sizes(B, T, I, H, L, P, training)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        if _POISON:          # debug: NaN-fill the workspace so that any read of a not-yet-written slot shows
            ws.fill_(255)
        emb = torch.empty(B, P, dtype=torch.float32, device=dev)
        check(_lib.lib().svb_embedder_forward(ptr(x), 0 if x.dtype == torch.float32 else 1, ptr(packed), ptr(proj_w),
                                              ptr(proj_b), ptr(emb), ptr(ws), B, T, I, H, L, P, int(training),
                                              int(rec_terms), stream_ptr(dev)), "svb_embedder_forward")
    return emb, ws


def _embedder_fwd_fake(x, params, packed, H, L, training, rec_terms):
    B, T, I = x.shape
    P = params[4 * L].shape[0]
    return x.new_empty(B, P, dtype=torch.float32), x.new_empty(_embedder_sizes(B, T, I, H, L, P, training)[1],
                                                               dtype=torch.uint8)


_op("embedder_fwd(Tensor x, Tensor[] params, Tensor packed, int H, int L, bool training, int rec_terms) -> "
    "(Tensor, Tensor)", _embedder_fwd, _embedder_fwd_fake)


def _embedder_bwd(demb: torch.Tensor, packed: torch.Tensor, proj_w: torch.Tensor, ws: torch.Tensor, numels: List[int],
                  T: int, I: int, H: int, L: int) -> torch.Tensor:
    B, P = (int(s) for s in demb.shape)
    dev = demb.device
    with torch.cuda.device(dev):
        dg = demb.contiguous()
        # one flat buffer, parameters as views: a single all-reduce covers every gradient (dist.py)
        flat = torch.empty(sum(numels), dtype=torch.float32, device=dev)
        offs = [0]
        for n in numels:
            offs.append(offs[-1] + n)
        grads = [flat[offs[i]:offs[i + 1]] for i in range(len(numels))]
        cb, errors = None, []
        hook, finish = _bucket_hook, _bucket_finish
        if hook is not None:
            def ready(bucket, _user):            # bucket L: projection, L-1 ... 0: LSTM layers (svb200.h)
                try:
                    lo, hi = (offs[4 * L], offs[4 * L + 2]) if bucket == L else (offs[4 * bucket], offs[4 * bucket + 4])
                    hook(flat[lo:hi])
                except BaseException as exc:         # exceptions cannot cross the C frame: re-raised below
                    errors.append(exc)

            cb = _GRAD_CB(ready)
            check(_lib.lib().svb_set_grad_ready_callback(cb, None), "svb_set_grad_ready_callback")
        try:
            check(_lib.lib().svb_embedder_backward(ptr(dg), ptr(packed), ptr(proj_w.contiguous()), _ptr_array(grads),
                                                   ptr(ws), B, T, I, H, L, P, stream_ptr(dev)), "svb_embedder_backward")
        finally:
            if cb is not None:
                _lib.lib().svb_set_grad_ready_callback(None, None)
        if errors:
            raise errors[0]
        if hook is not None and finish is not None:
            finish()          # the caller's stream now waits for whatever the hook started on the buckets
    return flat


def _embedder_bwd_fake(demb, packed, proj_w, ws, numels, T, I, H, L):
    return demb.new_empty(sum(numels), dtype=torch.float32)


# BPTT overwrites the gate stash inside the workspace with dG: `ws` is declared as mutated
_op("embedder_bwd(Tensor demb, Tensor packed, Tensor proj_w, Tensor(a!) ws, int[] numels, int T, int I, int H, int L) "
    "-> Tensor", _embedder_bwd, _embedder_bwd_fake)


def _embedder_setup(ctx, inputs, output):
    x, params, packed, H, L, training, rec_terms = inputs
    _, ws = output
    # no zero-filled "gradient" for the workspace output: materialising it costs a 5 GB fill per step at C2 (1.4 ms)
    ctx.set_materialize_grads(False)
    ctx.training = bool(training)
    if training:
        ctx.save_for_backward(packed, params[4 * L], ws)
        ctx.dims = (int(x.shape[1]), int(x.shape[2]), int(H), int(L))
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.consumed = False


def _embedder_backward(ctx, demb, _dws):
    if not ctx.training:
        raise RuntimeError("svb200::embedder_fwd was run with training=False: no BPTT stash was kept")
    if ctx.consumed:
        raise RuntimeError("svb200::embedder_fwd: backward was already run once for this forward; BPTT overwrites the "
                           "gate stash in place, so retain_graph / a second backward is not supported")
    if demb is None:                                     # the embeddings did not reach the loss
        return None, None, None, None, None, None, None
    ctx.consumed = True
    packed, proj_w, ws = ctx.saved_tensors
    T, I, H, L = ctx.dims
    numels = [int(torch.Size(s).numel()) for s in ctx.shapes]
    flat = torch.ops.svb200.embedder_bwd(demb, packed, proj_w, ws, numels, T, I, H, L)
    grads, off = [], 0
    for s, n in zip(ctx.shapes, numels):
        grads.append(flat[off:off + n].view(s))
        off += n
    return None, grads, None, None, None, None, None


torch.library.register_autograd(f"{NS}::embedder_fwd", _embedder_backward, setup_context=_embedder_setup)


class PackedWeights:
    """fp16 / bf16 gate-interleaved shadow of the fp32 master parameters (svb_embedder_pack_weights), rebuilt when a
    parameter's ``_version``, storage or device changes.

    Every rebuild goes to a FRESH buffer: a pending autograd graph may still hold the previous one for its BPTT.
    Updates that bypass the version counter (``p.data.add_()``, ``p.data.copy_()``) are not seen -- call
    ``invalidate()`` (``SpeechEmbedder.repack()``) after such surgery."""

    def __init__(self):
        self.key = None
        self.buf = None
        self.dev_params = None

    def invalidate(self):
        self.key = None

    def get(self, params, I, H, L, dev):
        key = tuple((p.data_ptr(), p._version, str(p.device)) for p in params) + (str(dev),)
        if key != self.key:
            with torch.no_grad():
                dev_params = [_stage(p.detach(), torch.float32, dev) for p in params]
                self.buf = torch.ops.svb200.pack_weights(dev_params[:4 * L], I, H, L)
            self.key = key
            self.dev_params = dev_params
        return self.buf, self.dev_params


class _StagedParam(torch.autograd.Function):
    """Plumbing only: hands the cached device copy of a parameter that lives elsewhere (a module left on the CPU, as
    in the reference's test() / dvector_create.py) to the op and routes its gradient back to the parameter's device."""

    @staticmethod
    def forward(ctx, p, staged):
        ctx.dev, ctx.dtype = p.device, p.dtype
        return staged.view_as(staged)

    @staticmethod
    def backward(ctx, g):
        return g.to(device=ctx.dev, dtype=ctx.dtype), None


def embedder_forward(x, cache, dims, params):
    """SpeechEmbedder.forward / BPTT (speech_embedder_net.py:27-33; train_speech_embedder.py:62)."""
    I, H, L, P, rec_terms = dims
    if x.dim() != 3 or x.shape[2] != I:
        raise ValueError(f"expected input (batch, frames, {I}), got {tuple(x.shape)}")
    dev = _target_device(x, *params)
    out_device = x.device
    with torch.cuda.device(dev):
        if x.dtype not in (torch.float32, torch.float64):
            x = x.float()                                          # speech_embedder_net.py:28
        xg = _stage(x.detach(), None, dev)
        packed, dev_params = cache.get(params, I, H, L, dev)
        training = torch.is_grad_enabled() and any(p.requires_grad for p in params)
        if training:
            # the op differentiates w.r.t. `params`: masters already on the device go in as they are, a module left
            # on the CPU goes in as its cached device copies (gradients flow back through _StagedParam)
            op_params = [p if (p.device == dev and p.dtype == torch.float32 and p.is_contiguous())
                         else _StagedParam.apply(p, s) for p, s in zip(params, dev_params)]
        else:
            op_params = dev_params
        emb, _ws = torch.ops.svb200.embedder_fwd(xg, op_params, packed, H, L, training, int(rec_terms))
    return _back(emb, out_device)


# ------------------------------------------------------------------------------------------ GE2E ops
# GE2E loss methods (include/svb200.h SVB_GE2E_*): Wan et al. eq. 6 (the reference's) and eq. 7
LOSS_METHODS = {"softmax": 0, "contrast": 1}


def loss_code(method):
    """'softmax' / 'contrast' (or their codes 0 / 1) -> the C ABI's SVB_GE2E_* code; anything else raises ValueError."""
    if isinstance(method, str) and method in LOSS_METHODS:
        return LOSS_METHODS[method]
    if not isinstance(method, (str, bool)) and method in LOSS_METHODS.values():
        return int(method)
    raise ValueError(f"unknown GE2E loss method {method!r}: expected one of {sorted(LOSS_METHODS)}")


def _check_loss(loss, columns):
    code = loss_code(loss)
    if code == LOSS_METHODS["contrast"] and columns < 2:
        raise ValueError("the GE2E contrast loss needs at least 2 centroid columns (speakers): it scores every row "
                         "against its most similar other centroid")
    return code


def _ge2e_call(E, Cext, w, b, dcos, gscale, want_cos, want_loss, need_grad, fused=1, loss=0):
    N, M, D = (int(s) for s in E.shape)
    Nc = N if Cext is None else int(Cext.shape[0])
    dev = E.device
    with torch.cuda.device(dev):
        nbytes = _sz(0)
        check(_lib.lib().svb_ge2e_workspace_bytes(N, M, D, Nc, ctypes.byref(nbytes)), "svb_ge2e_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        cos = torch.empty(N, M, Nc, **f32) if want_cos else None
        per = torch.empty(N, M, **f32) if want_loss else None
        dE = torch.empty(N, M, D, **f32) if need_grad else None
        dC = torch.empty(Nc, D, **f32) if (need_grad and Cext is not None) else None
        dw = torch.empty((), **f32) if (need_grad and w is not None) else None
        db = torch.empty((), **f32) if (need_grad and w is not None) else None
        lsum = torch.empty((), **f32) if want_loss else None
        if _POISON:          # debug: NaN-fill the workspace and every output, so that a slot no kernel writes shows
            for t in (ws, cos, per, dE, dC, dw, db, lsum):
                if t is not None:
                    t.view(-1).view(torch.uint8).fill_(255)
        check(_lib.lib().svb_ge2e_ex(ptr(E), ptr(Cext), N, M, D, Nc, ptr(w), ptr(b), ptr(dcos), ptr(gscale), ptr(cos),
                                     ptr(per), ptr(lsum), ptr(dE), ptr(dC), ptr(dw), ptr(db), ptr(ws), _sz(nbytes.value),
                                     int(fused), int(loss), stream_ptr(dev)), "svb_ge2e_ex")
    return dict(cos=cos, per=per, loss=lsum, dE=dE, dC=dC, dw=dw, db=db)


def _ge2e_loss(E: torch.Tensor, w: torch.Tensor, b: torch.Tensor, fused: int, need_grad: bool, loss: int = 0
               ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    if E.shape[1] < 2:
        raise ValueError("GE2E needs at least 2 utterances per speaker (leave-one-out centroid, utils.py:56-57)")
    loss = _check_loss(loss, E.shape[0])
    r = _ge2e_call(E.contiguous(), None, w.contiguous(), b.contiguous(), None, None, False, True, need_grad, fused, loss)
    if not need_grad:
        z = E.new_empty(0)
        return r["loss"], z, z.clone(), z.clone()
    return r["loss"], r["dE"], r["dw"], r["db"]


def _ge2e_loss_fake(E, w, b, fused, need_grad, loss=0):
    if not need_grad:
        return E.new_empty(()), E.new_empty(0), E.new_empty(0), E.new_empty(0)
    return E.new_empty(()), torch.empty_like(E), E.new_empty(()), E.new_empty(())


# forward AND gradients in one fused launch: loss plus d loss / d (E, w, b); autograd scales them by the upstream
_op("ge2e_loss(Tensor E, Tensor w, Tensor b, int fused, bool need_grad, int loss=0) -> (Tensor, Tensor, Tensor, Tensor)",
    _ge2e_loss, _ge2e_loss_fake)


def _ge2e_rows(E: torch.Tensor, C: torch.Tensor, w: torch.Tensor, b: torch.Tensor, col0: int, loss: int = 0
               ) -> Tuple[torch.Tensor, torch.Tensor]:
    N, M, D = (int(v) for v in E.shape)
    Nc = int(C.shape[0])
    loss = _check_loss(loss, Nc)
    dev = E.device
    with torch.cuda.device(dev):
        nbytes = _sz(0)
        check(_lib.lib().svb_ge2e_workspace_bytes(N, M, D, Nc, ctypes.byref(nbytes)), "svb_ge2e_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        # one buffer for everything that is summed over the ranks: dC (Nc, D), then loss, dw, db
        red = torch.empty(Nc * D + 3, dtype=torch.float32, device=dev)
        dE = torch.empty(N, M, D, dtype=torch.float32, device=dev)
        if _POISON:          # debug: NaN-fill the workspace and the outputs (see _ge2e_call)
            for t in (ws, red, dE):
                t.view(-1).view(torch.uint8).fill_(255)
        base = red.data_ptr()
        f = lambda off: ctypes.c_void_p(base + 4 * off)
        check(_lib.lib().svb_ge2e_rows_ex(ptr(E.contiguous()), ptr(C.contiguous()), N, M, D, Nc, int(col0),
                                          ptr(w.contiguous()), ptr(b.contiguous()), None, None, f(Nc * D), ptr(dE), f(0),
                                          f(Nc * D + 1), f(Nc * D + 2), ptr(ws), _sz(nbytes.value), int(loss),
                                          stream_ptr(dev)), "svb_ge2e_rows_ex")
    return red, dE


def _ge2e_rows_fake(E, C, w, b, col0, loss=0):
    return E.new_empty(C.shape[0] * C.shape[1] + 3), torch.empty_like(E)


# row shard of a global batch against all-gathered centroids: (reduction buffer [dC | loss, dw, db], dE of the shard)
_op("ge2e_rows(Tensor E, Tensor C, Tensor w, Tensor b, int col0, int loss=0) -> (Tensor, Tensor)", _ge2e_rows,
    _ge2e_rows_fake)


def _peer_gather(anchor: torch.Tensor, peer_ptrs_dev: int, world: int, offset: int, n: int) -> torch.Tensor:
    """out[r, i] = peer_r[offset + i]: `anchor` is this rank's symmetric buffer (device / stream of the launch)."""
    out = torch.empty(int(world), int(n), dtype=torch.float32, device=anchor.device)
    with torch.cuda.device(anchor.device):
        check(_lib.lib().svb_peer_gather(ctypes.c_void_p(int(peer_ptrs_dev)), int(world), _sz(int(offset)), _sz(0),
                                         _sz(int(n)), ptr(out), stream_ptr(anchor.device)), "svb_peer_gather")
    return out


def peer_allreduce_(flat, buf, peer_ptrs_dev, world, rank, barrier):
    """In-place SUM all-reduce of the contiguous float32 tensor ``flat`` through the symmetric buffer ``buf`` (>= numel
    padded to 4 * world floats) in two shots over NVLink peer memory: every rank sums ITS slice over all peers in place
    (svb_peer_reduce), then reads all reduced slices back (svb_peer_gather).  Sums in rank order: bit-identical on every
    rank.  ``barrier(channel)`` is the symmetric-memory handle's device-side barrier."""
    n = flat.numel()
    sl = (n + 4 * world - 1) // (4 * world) * 4                 # floats per slice
    if buf.numel() < sl * world:
        raise SvbError("peer_allreduce_: symmetric buffer too small")
    L = _lib.lib()
    with torch.cuda.device(flat.device):
        st = stream_ptr(flat.device)
        buf[:n].copy_(flat.reshape(-1))
        if sl * world > n:
            buf[n:sl * world].zero_()
        barrier(0)                                                  # every rank's gradients are in its buffer
        mine = ctypes.c_void_p(buf.data_ptr() + 4 * rank * sl)
        check(L.svb_peer_reduce(ctypes.c_void_p(int(peer_ptrs_dev)), int(world), _sz(0), _sz(rank * sl), _sz(sl), _sz(0), 0,
                                mine, None, st), "svb_peer_reduce")
        barrier(1)                                                  # every rank's slice is reduced
        if sl * world == n:
            out = flat.reshape(-1)
        else:
            out = torch.empty(sl * world, dtype=torch.float32, device=flat.device)
        check(L.svb_peer_gather(ctypes.c_void_p(int(peer_ptrs_dev)), int(world), _sz(0), _sz(sl), _sz(sl), ptr(out), st),
              "svb_peer_gather")
        if out.data_ptr() != flat.data_ptr():
            flat.reshape(-1).copy_(out[:n])
        barrier(2)                                                  # nobody still reads a buffer that the next call overwrites
    return flat


_op("peer_gather(Tensor anchor, int peer_ptrs_dev, int world, int offset, int n) -> Tensor", _peer_gather,
    lambda anchor, p, world, offset, n: anchor.new_empty(world, n))


def _peer_reduce(anchor: torch.Tensor, peer_ptrs_dev: int, world: int, offset: int, seg_offset: int, seg_n: int,
                 tail_offset: int, tail_n: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(sum over the ranks of peer_r[offset + seg_offset : + seg_n], of peer_r[offset + tail_offset : + tail_n]), in
    rank order."""
    seg = torch.empty(int(seg_n), dtype=torch.float32, device=anchor.device)
    tail = torch.empty(int(tail_n), dtype=torch.float32, device=anchor.device)
    with torch.cuda.device(anchor.device):
        check(_lib.lib().svb_peer_reduce(ctypes.c_void_p(int(peer_ptrs_dev)), int(world), _sz(int(offset)),
                                         _sz(int(seg_offset)), _sz(int(seg_n)), _sz(int(tail_offset)), int(tail_n),
                                         ptr(seg), ptr(tail), stream_ptr(anchor.device)), "svb_peer_reduce")
    return seg, tail


_op("peer_reduce(Tensor anchor, int peer_ptrs_dev, int world, int offset, int seg_offset, int seg_n, int tail_offset, "
    "int tail_n) -> (Tensor, Tensor)", _peer_reduce,
    lambda anchor, p, world, offset, so, sn, to, tn: (anchor.new_empty(sn), anchor.new_empty(tn)))


def _scale3(dE: torch.Tensor, dw: torch.Tensor, db: torch.Tensor, g: torch.Tensor
            ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    dE, dw, db = dE.clone(), dw.clone(), db.clone()
    with torch.cuda.device(dE.device):
        check(_lib.lib().svb_scale3(ptr(dE), _sz(dE.numel()), ptr(dw), _sz(dw.numel()), ptr(db), _sz(db.numel()),
                                    ptr(g.contiguous()), stream_ptr(dE.device)), "svb_scale3")
    return dE, dw, db


_op("scale3(Tensor a, Tensor b, Tensor c, Tensor g) -> (Tensor, Tensor, Tensor)", _scale3,
    lambda a, b, c, g: (torch.empty_like(a), torch.empty_like(b), torch.empty_like(c)))


def _ge2e_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)                     # outputs 1..3 are the saved gradients, never differentiated
    ctx.need = bool(inputs[4])
    if ctx.need:
        ctx.save_for_backward(output[1], output[2], output[3])


def _ge2e_backward(ctx, g, *_unused):
    if g is None:
        return None, None, None, None, None, None
    if not ctx.need:
        raise RuntimeError("svb200::ge2e_loss was run with need_grad=False")
    dE, dw, db = ctx.saved_tensors
    a, b, c = torch.ops.svb200.scale3(dE, dw, db, g.to(torch.float32))
    return a, b, c, None, None, None


torch.library.register_autograd(f"{NS}::ge2e_loss", _ge2e_backward, setup_context=_ge2e_setup)


def ge2e_loss(E, w, b, fused=1, loss_method="softmax"):
    """GE2ELoss.forward + backward in one fused kernel (speech_embedder_net.py:43-49, utils.py:27-132).
    ``loss_method``: "softmax" (the reference's, Wan et al. eq. 6) or "contrast" (eq. 7)."""
    if E.dim() != 3:
        raise ValueError("embeddings must be (speakers, utterances, dim)")
    if E.shape[1] < 2:
        raise ValueError("GE2E needs at least 2 utterances per speaker (leave-one-out centroid, utils.py:56-57)")
    code = _check_loss(loss_method, E.shape[0])
    dev = _target_device(E, w, b)
    need = torch.is_grad_enabled() and (E.requires_grad or w.requires_grad or b.requires_grad)
    with torch.cuda.device(dev):
        loss = torch.ops.svb200.ge2e_loss(_stage(E, torch.float32, dev), _stage(w, torch.float32, dev),
                                          _stage(b, torch.float32, dev), int(fused), bool(need), code)[0]
    return _back(loss, E.device)


def _centroids(E: torch.Tensor) -> torch.Tensor:
    N, M, D = (int(s) for s in E.shape)
    E = E.contiguous()
    C = _f32(E, N, D)
    with torch.cuda.device(E.device):
        check(_lib.lib().svb_centroids(ptr(E), ptr(C), N, M, D, stream_ptr(E.device)), "svb_centroids")
    return C


def _centroids_bwd(dC: torch.Tensor, M: int) -> torch.Tensor:
    N, D = (int(s) for s in dC.shape)
    dC = dC.contiguous()
    dE = _f32(dC, N, M, D)
    with torch.cuda.device(dC.device):
        check(_lib.lib().svb_centroids_bwd(ptr(dC), ptr(dE), N, M, D, stream_ptr(dC.device)), "svb_centroids_bwd")
    return dE


_op("centroids(Tensor E) -> Tensor", _centroids, lambda E: E.new_empty(E.shape[0], E.shape[2]))
_op("centroids_bwd(Tensor dC, int M) -> Tensor", _centroids_bwd, lambda dC, M: dC.new_empty(dC.shape[0], M, dC.shape[1]))
torch.library.register_autograd(
    f"{NS}::centroids", lambda ctx, g: torch.ops.svb200.centroids_bwd(g.to(torch.float32), ctx.M),
    setup_context=lambda ctx, inputs, output: setattr(ctx, "M", int(inputs[0].shape[1])))


def _utterance_centroids(E: torch.Tensor) -> torch.Tensor:
    N, M, D = (int(s) for s in E.shape)
    if M < 2:
        raise ValueError("get_utterance_centroids needs at least 2 utterances per speaker (utils.py:56-57 divides by M-1)")
    E = E.contiguous()
    U = torch.empty_like(E)
    with torch.cuda.device(E.device):
        check(_lib.lib().svb_utterance_centroids(ptr(E), ptr(U), N, M, D, stream_ptr(E.device)), "svb_utterance_centroids")
    return U


_op("utterance_centroids(Tensor E) -> Tensor", _utterance_centroids, lambda E: torch.empty_like(E))
# linear and symmetric: the adjoint is the operator itself
torch.library.register_autograd(f"{NS}::utterance_centroids",
                                lambda ctx, g: torch.ops.svb200.utterance_centroids(g.to(torch.float32)),
                                setup_context=lambda ctx, inputs, output: None)


def _cossim(E: torch.Tensor, C: torch.Tensor) -> torch.Tensor:
    return _ge2e_call(E.contiguous(), C.contiguous(), None, None, None, None, True, False, False)["cos"]


def _cossim_bwd(E: torch.Tensor, C: torch.Tensor, dcos: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    r = _ge2e_call(E.contiguous(), C.contiguous(), None, None, dcos.contiguous(), None, False, False, True)
    return r["dE"], r["dC"]


_op("cossim(Tensor E, Tensor C) -> Tensor", _cossim, lambda E, C: E.new_empty(E.shape[0], E.shape[1], C.shape[0]))
_op("cossim_bwd(Tensor E, Tensor C, Tensor dcos) -> (Tensor, Tensor)", _cossim_bwd,
    lambda E, C, dcos: (torch.empty_like(E), torch.empty_like(C)))
torch.library.register_autograd(
    f"{NS}::cossim", lambda ctx, g: torch.ops.svb200.cossim_bwd(*ctx.saved_tensors, g.to(torch.float32)),
    setup_context=lambda ctx, inputs, output: ctx.save_for_backward(inputs[0], inputs[1]))


def _calc_loss(S: torch.Tensor, loss: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    N, M, Nc = (int(s) for s in S.shape)
    code = _check_loss(loss, Nc)
    S = S.contiguous()
    per, lsum = _f32(S, N, M), _f32(S)
    with torch.cuda.device(S.device):
        check(_lib.lib().svb_calc_loss_ex(ptr(S), N, M, Nc, ptr(per), ptr(lsum), None, None, code, stream_ptr(S.device)),
              "svb_calc_loss_ex")
    return lsum, per


def _calc_loss_bwd(S: torch.Tensor, gloss: torch.Tensor, loss: int = 0) -> torch.Tensor:
    N, M, Nc = (int(s) for s in S.shape)
    code = _check_loss(loss, Nc)
    S = S.contiguous()
    per, dS = _f32(S, N, M), torch.empty_like(S)
    with torch.cuda.device(S.device):
        check(_lib.lib().svb_calc_loss_ex(ptr(S), N, M, Nc, ptr(per), None, ptr(dS), ptr(gloss.contiguous()), code,
                                          stream_ptr(S.device)), "svb_calc_loss_ex")
    return dS


_op("calc_loss(Tensor S, int loss=0) -> (Tensor, Tensor)", _calc_loss,
    lambda S, loss=0: (S.new_empty(()), S.new_empty(S.shape[0], S.shape[1])))
_op("calc_loss_bwd(Tensor S, Tensor gloss, int loss=0) -> Tensor", _calc_loss_bwd, lambda S, g, loss=0: torch.empty_like(S))


def _calc_loss_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    ctx.save_for_backward(inputs[0])
    ctx.loss = int(inputs[1]) if len(inputs) > 1 else 0
    ctx.mark_non_differentiable(output[1])       # the reference's per-embedding loss is used for logging only


def _calc_loss_backward(ctx, gloss, _gper):
    if gloss is None:
        return None, None
    return torch.ops.svb200.calc_loss_bwd(ctx.saved_tensors[0], gloss.to(torch.float32), ctx.loss), None


torch.library.register_autograd(f"{NS}::calc_loss", _calc_loss_backward, setup_context=_calc_loss_setup)


def get_centroids(E):
    """utils.get_centroids (utils.py:27-29)."""
    dev = _target_device(E)
    return _back(torch.ops.svb200.centroids(_stage(E, torch.float32, dev)), E.device)


def get_utterance_centroids(E):
    """utils.get_utterance_centroids (utils.py:40-58)."""
    if E.dim() != 3:
        raise ValueError("embeddings must be (speakers, utterances, dim)")
    if E.shape[1] < 2:
        raise ValueError("get_utterance_centroids needs at least 2 utterances per speaker (utils.py:56-57 divides by M-1)")
    dev = _target_device(E)
    return _back(torch.ops.svb200.utterance_centroids(_stage(E, torch.float32, dev)), E.device)


def get_cossim(E, C):
    """utils.get_cossim (utils.py:72-115), differentiable w.r.t. embeddings and centroids."""
    if E.dim() != 3 or C.dim() != 2 or C.shape[1] != E.shape[2]:
        raise ValueError("get_cossim expects embeddings (N,M,D) and centroids (N',D)")
    if C.shape[0] != E.shape[0]:
        # the reference's diagonal index_put (utils.py:112-113) requires N' >= N; it is only ever called with N' == N
        raise ValueError("get_cossim: centroids must have one row per speaker of embeddings")
    if E.shape[1] < 2:
        raise ValueError("get_cossim needs at least 2 utterances per speaker (leave-one-out centroid, utils.py:56-57)")
    dev = _target_device(E, C)
    return _back(torch.ops.svb200.cossim(_stage(E, torch.float32, dev), _stage(C, torch.float32, dev)), E.device)


def calc_loss(S, loss_method="softmax"):
    """utils.calc_loss (utils.py:126-132): (loss, per_embedding_loss); ``loss_method`` "contrast" gives the GE2E
    contrast loss (Wan et al. eq. 7) of the same similarity matrix."""
    if S.dim() != 3 or S.shape[2] < S.shape[0]:
        raise ValueError("calc_loss expects a similarity matrix (N, M, N)")
    code = _check_loss(loss_method, S.shape[2])
    dev = _target_device(S)
    loss, per = torch.ops.svb200.calc_loss(_stage(S, torch.float32, dev), code)
    return _back(loss, S.device), _back(per, S.device)


# ------------------------------------------------------------------------------------------ EER ops
def _eer_counts(sim: torch.Tensor, thresholds: torch.Tensor, speaker0: int) -> Tuple[torch.Tensor, torch.Tensor]:
    n, Mv, Nc = (int(s) for s in sim.shape)
    T = int(thresholds.numel())
    sim = sim.contiguous()
    ca = torch.empty(n, T, dtype=torch.int32, device=sim.device)
    cd = torch.empty(n, T, dtype=torch.int32, device=sim.device)
    with torch.cuda.device(sim.device):
        check(_lib.lib().svb_eer_counts(ptr(sim), n, Mv, Nc, int(speaker0), ptr(thresholds), T, ptr(ca), ptr(cd),
                                        stream_ptr(sim.device)), "svb_eer_counts")
    return ca, cd


def _counts_fake(sim, thresholds, speaker0=0):
    n, T = sim.shape[0], thresholds.numel()
    return sim.new_empty(n, T, dtype=torch.int32), sim.new_empty(n, T, dtype=torch.int32)


_op("eer_counts(Tensor sim, Tensor thresholds, int speaker0) -> (Tensor, Tensor)", _eer_counts, _counts_fake)


def _eer_sweep(sim: torch.Tensor, thresholds: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    N, Mv, Nc = (int(s) for s in sim.shape)
    T = int(thresholds.numel())
    sim = sim.contiguous()
    ca = torch.empty(N, T, dtype=torch.int32, device=sim.device)
    cd = torch.empty(N, T, dtype=torch.int32, device=sim.device)
    scratch = torch.zeros(1 + 16 * T, dtype=torch.int64, device=sim.device)
    out = torch.empty(4 + 2 * T, dtype=torch.float32, device=sim.device)
    with torch.cuda.device(sim.device):
        check(_lib.lib().svb_eer_sweep(ptr(sim), N, Mv, ptr(thresholds), T, ptr(ca), ptr(cd), ptr(scratch), ptr(out),
                                       stream_ptr(sim.device)), "svb_eer_sweep")
    return out, ca, cd


_op("eer_sweep(Tensor sim, Tensor thresholds) -> (Tensor, Tensor, Tensor)", _eer_sweep,
    lambda sim, thr: (sim.new_empty(4 + 2 * thr.numel()),) + _counts_fake(sim, thr))


def _eer_finish(cnt_all: torch.Tensor, cnt_diag: torch.Tensor, Mv: int) -> torch.Tensor:
    N, T = (int(s) for s in cnt_all.shape)
    out = torch.empty(4 + 2 * T, dtype=torch.float32, device=cnt_all.device)
    with torch.cuda.device(cnt_all.device):
        check(_lib.lib().svb_eer_finish(ptr(cnt_all.contiguous()), ptr(cnt_diag.contiguous()), N, int(Mv), T, ptr(out),
                                        stream_ptr(cnt_all.device)), "svb_eer_finish")
    return out


_op("eer_finish(Tensor cnt_all, Tensor cnt_diag, int Mv) -> Tensor", _eer_finish,
    lambda ca, cd, Mv: ca.new_empty(4 + 2 * ca.shape[1], dtype=torch.float32))


def eer_counts(sim, thresholds_f32, speaker0=0):
    """Exact counts of sim > t for the row blocks of speakers [speaker0, speaker0 + sim.shape[0])."""
    return torch.ops.svb200.eer_counts(sim, thresholds_f32, int(speaker0))


def eer_sweep_fused(sim, thresholds_f32):
    """One launch: (out[4 + 2T], cnt_all, cnt_diag); out[1] == -2 asks for the sequential eer_finish."""
    return torch.ops.svb200.eer_sweep(sim, thresholds_f32)


def eer_finish(cnt_all, cnt_diag, Mv):
    return torch.ops.svb200.eer_finish(cnt_all, cnt_diag, int(Mv))


# ------------------------------------------------------------------------------------------ exact EER / minDCF ops
# out (8 + 4P float64): eer, threshold, p_miss, p_fa, Nt, Nn, #non-finite, K, then per point min_dcf, threshold,
# p_miss, p_fa (include/svb200.h svb_verif_metrics)
def _verif_call(fn, what, n, args, ops, dev):
    P = len(ops) // 3
    with torch.cuda.device(dev):
        nbytes = _sz(0)
        check(_lib.lib().svb_verif_workspace_bytes(_i64(n), ctypes.byref(nbytes)), "svb_verif_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
        out = torch.empty(8 + 4 * P, dtype=torch.float64, device=dev)
        check(fn(*args, (ctypes.c_double * len(ops))(*ops), P, ptr(ws), _sz(nbytes.value), ptr(out), stream_ptr(dev)),
              what)
    return out


def _verif_metrics(scores: torch.Tensor, labels: torch.Tensor, ops: List[float]) -> torch.Tensor:
    if scores.dtype != torch.float32 or labels.dtype not in (torch.uint8, torch.bool) or scores.shape != labels.shape:
        raise ValueError("verif_metrics expects float32 scores and uint8 / bool labels of the same shape")
    if labels.device != scores.device:
        raise ValueError(f"verif_metrics: labels on {labels.device}, scores on {scores.device}: they must share the "
                         "CUDA device")
    s, lab = scores.contiguous(), labels.contiguous()
    n = s.numel()
    return _verif_call(_lib.lib().svb_verif_metrics, "svb_verif_metrics", n, (ptr(s), ptr(lab), _i64(n)), ops, s.device)


def _verif_metrics_sim(sim: torch.Tensor, ops: List[float]) -> torch.Tensor:
    if sim.dtype != torch.float32 or sim.dim() != 3 or sim.shape[0] != sim.shape[2]:
        raise ValueError("verif_metrics_sim expects a float32 similarity matrix (N, Mv, N)")
    s = sim.contiguous()
    N, Mv = int(s.shape[0]), int(s.shape[1])
    return _verif_call(_lib.lib().svb_verif_metrics_sim, "svb_verif_metrics_sim", N * Mv * N, (ptr(s), N, Mv), ops,
                       s.device)


_op("verif_metrics(Tensor scores, Tensor labels, float[] ops) -> Tensor", _verif_metrics,
    lambda scores, labels, ops: scores.new_empty(8 + 4 * (len(ops) // 3), dtype=torch.float64))
_op("verif_metrics_sim(Tensor sim, float[] ops) -> Tensor", _verif_metrics_sim,
    lambda sim, ops: sim.new_empty(8 + 4 * (len(ops) // 3), dtype=torch.float64))


def verif_metrics(scores, labels_u8, ops):
    return torch.ops.svb200.verif_metrics(scores, labels_u8, [float(v) for v in ops])


def verif_metrics_sim(sim, ops):
    return torch.ops.svb200.verif_metrics_sim(sim, [float(v) for v in ops])


# ------------------------------------------------------------------------------------------ score calibration
# metrics out (8 + 4P float64): cllr, min_cllr, rocch_eer, Nt, Nn, #non-finite, #hull vertices, K, then per point
# act_dcf, threshold, p_miss, p_fa; train out (5 float64): a, b, C / ln 2, iterations, status (include/svb200.h)
def _calib_args(what, scores, labels):
    if scores.dtype != torch.float32 or labels.dtype not in (torch.uint8, torch.bool) or scores.shape != labels.shape:
        raise ValueError(f"{what} expects float32 scores and uint8 / bool labels of the same shape")
    _same_device(what, scores, labels)
    s, lab = scores.contiguous(), labels.contiguous()
    n = s.numel()
    nbytes = _sz(0)
    with torch.cuda.device(s.device):
        check(_lib.lib().svb_calib_workspace_bytes(_i64(n), ctypes.byref(nbytes)), "svb_calib_workspace_bytes")
    return s, lab, n, torch.empty(nbytes.value, dtype=torch.uint8, device=s.device), nbytes.value


def _calib_metrics(llr: torch.Tensor, labels: torch.Tensor, ops: List[float]) -> torch.Tensor:
    s, lab, n, ws, nbytes = _calib_args("calib_metrics", llr, labels)
    P = len(ops) // 3
    out = torch.empty(8 + 4 * P, dtype=torch.float64, device=s.device)
    with torch.cuda.device(s.device):
        check(_lib.lib().svb_calib_metrics(ptr(s), ptr(lab), _i64(n), (ctypes.c_double * len(ops))(*ops), P, ptr(ws),
                                           _sz(nbytes), ptr(out), stream_ptr(s.device)), "svb_calib_metrics")
    return out


def _calib_train(scores: torch.Tensor, labels: torch.Tensor, prior: float, max_iter: int) -> torch.Tensor:
    s, lab, n, ws, nbytes = _calib_args("calib_train", scores, labels)
    out = torch.empty(5, dtype=torch.float64, device=s.device)
    with torch.cuda.device(s.device):
        check(_lib.lib().svb_calib_train(ptr(s), ptr(lab), _i64(n), ctypes.c_double(prior), int(max_iter), ptr(ws),
                                         _sz(nbytes), ptr(out), stream_ptr(s.device)), "svb_calib_train")
    return out


_op("calib_metrics(Tensor llr, Tensor labels, float[] ops) -> Tensor", _calib_metrics,
    lambda llr, labels, ops: llr.new_empty(8 + 4 * (len(ops) // 3), dtype=torch.float64))
_op("calib_train(Tensor scores, Tensor labels, float prior, int max_iter) -> Tensor", _calib_train,
    lambda scores, labels, prior, max_iter: scores.new_empty(5, dtype=torch.float64))


def calib_metrics(llr, labels_u8, ops):
    return torch.ops.svb200.calib_metrics(llr, labels_u8, [float(v) for v in ops])


def calib_train(scores, labels_u8, prior, max_iter):
    return torch.ops.svb200.calib_train(scores, labels_u8, float(prior), int(max_iter))


# ------------------------------------------------------------------------------------------ cohort score normalization
# statistics (n, 3) float64: mean, std (divisor K - 1), K-th largest cohort score (include/svb200.h svb_cohort_stats)
def _same_device(what, *tensors):
    for t in tensors:
        if t is not None and t.device != tensors[0].device:
            raise ValueError(f"{what}: tensors on {tensors[0].device} and {t.device}: they must share the CUDA device")


def _cohort_stats(X: torch.Tensor, cohort: torch.Tensor, top_k: int) -> torch.Tensor:
    if (X.dtype != torch.float32 or cohort.dtype != torch.float32 or X.dim() != 2 or cohort.dim() != 2
            or X.shape[1] != cohort.shape[1]):
        raise ValueError("cohort_stats expects float32 rows (n, D) and a float32 cohort (Nc, D)")
    _same_device("cohort_stats", X, cohort)
    x, c = X.contiguous(), cohort.contiguous()
    n, D, Nc = int(x.shape[0]), int(x.shape[1]), int(c.shape[0])
    out = torch.empty(n, 3, dtype=torch.float64, device=x.device)
    if n == 0:
        return out
    with torch.cuda.device(x.device):
        nbytes = _sz(0)
        check(_lib.lib().svb_cohort_stats_workspace_bytes(_i64(n), Nc, D, ctypes.byref(nbytes)),
              "svb_cohort_stats_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=x.device)
        check(_lib.lib().svb_cohort_stats(ptr(x), _i64(n), ptr(c), Nc, D, int(top_k), ptr(ws), _sz(nbytes.value),
                                          ptr(out), stream_ptr(x.device)), "svb_cohort_stats")
    return out


def _cohort_stats_scores(scores: torch.Tensor, top_k: int) -> torch.Tensor:
    if scores.dtype != torch.float32 or scores.dim() != 2:
        raise ValueError("cohort_stats_scores expects float32 cohort scores (n, Nc)")
    s = scores if scores.stride(1) == 1 and scores.stride(0) >= scores.shape[1] else scores.contiguous()
    n, Nc = int(s.shape[0]), int(s.shape[1])
    out = torch.empty(n, 3, dtype=torch.float64, device=s.device)
    if n == 0:
        return out
    with torch.cuda.device(s.device):
        check(_lib.lib().svb_cohort_stats_scores(ptr(s), _i64(n), Nc, _i64(s.stride(0)), int(top_k), ptr(out),
                                                 stream_ptr(s.device)), "svb_cohort_stats_scores")
    return out


def _score_trials(E: torch.Tensor, T: torch.Tensor, ei: torch.Tensor, ti: torch.Tensor,
                  stats_e: Optional[torch.Tensor], stats_t: Optional[torch.Tensor]) -> torch.Tensor:
    if (E.dtype != torch.float32 or T.dtype != torch.float32 or E.dim() != 2 or T.dim() != 2
            or E.shape[1] != T.shape[1]):
        raise ValueError("score_trials expects float32 rows E (ne, D) and T (nt, D)")
    if ei.dtype != torch.int32 or ti.dtype != torch.int32 or ei.shape != ti.shape or ei.dim() != 1:
        raise ValueError("score_trials expects int32 index vectors of one length")
    if (stats_e is None) != (stats_t is None):
        raise ValueError("score_trials: give the statistics of both sides or of neither")
    if stats_e is not None and (stats_e.dtype != torch.float64 or stats_t.dtype != torch.float64
                                or tuple(stats_e.shape) != (E.shape[0], 3) or tuple(stats_t.shape) != (T.shape[0], 3)):
        raise ValueError("score_trials expects float64 statistics (ne, 3) and (nt, 3)")
    _same_device("score_trials", E, T, ei, ti, stats_e, stats_t)
    e, t, a, b = E.contiguous(), T.contiguous(), ei.contiguous(), ti.contiguous()
    se = None if stats_e is None else stats_e.contiguous()
    st = None if stats_t is None else stats_t.contiguous()
    out = torch.empty(a.numel(), dtype=torch.float32, device=e.device)
    with torch.cuda.device(e.device):
        check(_lib.lib().svb_score_trials(ptr(e), _i64(e.shape[0]), ptr(t), _i64(t.shape[0]), int(e.shape[1]), ptr(a),
                                          ptr(b), _i64(a.numel()), ptr(se), ptr(st), ptr(out), stream_ptr(e.device)),
              "svb_score_trials")
    return out


def _asnorm_sim(sim: torch.Tensor, stats_c: torch.Tensor, stats_v: torch.Tensor) -> torch.Tensor:
    if sim.dtype != torch.float32 or sim.dim() != 3 or sim.shape[0] != sim.shape[2]:
        raise ValueError("asnorm_sim expects a float32 similarity matrix (N, Mv, N)")
    N, Mv = int(sim.shape[0]), int(sim.shape[1])
    if (stats_c.dtype != torch.float64 or stats_v.dtype != torch.float64 or tuple(stats_c.shape) != (N, 3)
            or tuple(stats_v.shape) != (N * Mv, 3)):
        raise ValueError("asnorm_sim expects float64 statistics (N, 3) and (N * Mv, 3)")
    _same_device("asnorm_sim", sim, stats_c, stats_v)
    s = sim.contiguous()
    out = torch.empty_like(s)
    if s.numel() == 0:
        return out
    with torch.cuda.device(s.device):
        check(_lib.lib().svb_asnorm_sim(ptr(s), N, Mv, ptr(stats_c.contiguous()), ptr(stats_v.contiguous()), ptr(out),
                                        stream_ptr(s.device)), "svb_asnorm_sim")
    return out


_op("cohort_stats(Tensor X, Tensor cohort, int top_k) -> Tensor", _cohort_stats,
    lambda X, cohort, top_k: X.new_empty(X.shape[0], 3, dtype=torch.float64))
_op("cohort_stats_scores(Tensor scores, int top_k) -> Tensor", _cohort_stats_scores,
    lambda scores, top_k: scores.new_empty(scores.shape[0], 3, dtype=torch.float64))
_op("score_trials(Tensor E, Tensor T, Tensor ei, Tensor ti, Tensor? stats_e, Tensor? stats_t) -> Tensor", _score_trials,
    lambda E, T, ei, ti, stats_e, stats_t: E.new_empty(ei.shape[0], dtype=torch.float32))
_op("asnorm_sim(Tensor sim, Tensor stats_c, Tensor stats_v) -> Tensor", _asnorm_sim,
    lambda sim, stats_c, stats_v: torch.empty_like(sim))


def cohort_stats(X, cohort, top_k):
    return torch.ops.svb200.cohort_stats(X, cohort, int(top_k))


def cohort_stats_scores(scores, top_k):
    return torch.ops.svb200.cohort_stats_scores(scores, int(top_k))


def score_trials(E, T, ei, ti, stats_e=None, stats_t=None):
    return torch.ops.svb200.score_trials(E, T, ei, ti, stats_e, stats_t)


def asnorm_sim(sim, stats_c, stats_v):
    return torch.ops.svb200.asnorm_sim(sim, stats_c, stats_v)


# ------------------------------------------------------------------------------------------ d-vector ops
def _dvector_windows(S: torch.Tensor, win_start: torch.Tensor, win: int) -> torch.Tensor:
    nmels, W = int(S.shape[0]), int(win_start.numel())
    if S.stride(1) != 1:
        S = S.contiguous()
    out = torch.empty(W, win, nmels, dtype=torch.float32, device=S.device)
    with torch.cuda.device(S.device):
        check(_lib.lib().svb_dvector_windows(ptr(S), _i64(S.stride(0)), nmels, ptr(win_start), W, int(win), ptr(out),
                                             stream_ptr(S.device)), "svb_dvector_windows")
    return out


_op("dvector_windows(Tensor S, Tensor win_start, int win) -> Tensor", _dvector_windows,
    lambda S, ws, win: S.new_empty(ws.numel(), win, S.shape[0]))


def _segment_mean(emb: torch.Tensor, seg_offsets: torch.Tensor) -> torch.Tensor:
    P, D = int(seg_offsets.numel()) - 1, int(emb.shape[1])
    emb = emb.contiguous()
    out = torch.empty(P, D, dtype=torch.float64, device=emb.device)
    with torch.cuda.device(emb.device):
        check(_lib.lib().svb_segment_mean(ptr(emb), D, ptr(seg_offsets), P, ptr(out), stream_ptr(emb.device)),
              "svb_segment_mean")
    return out


_op("segment_mean(Tensor emb, Tensor seg_offsets) -> Tensor", _segment_mean,
    lambda emb, so: emb.new_empty(so.numel() - 1, emb.shape[1], dtype=torch.float64))


def dvector_windows(S, win_start, win):
    """S (nmels, Ttot) float32 CUDA, win_start int32 CUDA (W,) -> (W, win, nmels)."""
    return torch.ops.svb200.dvector_windows(S, win_start, int(win))


def segment_mean(emb, seg_offsets):
    return torch.ops.svb200.segment_mean(emb, seg_offsets)


# ------------------------------------------------------------------------------------------ optimizer tail + front end
def _clip_sgd(params: List[torch.Tensor], grads: List[torch.Tensor], group: List[int], max_norm: List[float], lr: float,
              write_clipped_grads: bool, workspace: torch.Tensor) -> torch.Tensor:
    n, ng = len(params), len(max_norm)
    dev = params[0].device
    norms = torch.empty(4, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().svb_clip_sgd(_ptr_array(params), _ptr_array(grads), (ctypes.c_int64 * n)(*[p.numel() for p in params]),
                                      (ctypes.c_int32 * n)(*group), n, (ctypes.c_float * ng)(*max_norm), ng,
                                      ctypes.c_float(lr), int(write_clipped_grads), ptr(norms), ptr(workspace),
                                      _sz(workspace.numel()), stream_ptr(dev)), "svb_clip_sgd")
    return norms[:ng]


_op("clip_sgd(Tensor(a!)[] params, Tensor(b!)[] grads, int[] group, float[] max_norm, float lr, "
    "bool write_clipped_grads, Tensor(c!) workspace) -> Tensor", _clip_sgd,
    lambda params, grads, group, max_norm, lr, wcg, ws: params[0].new_empty(len(max_norm)))


def _logmel(y: torch.Tensor, window: torch.Tensor, twiddle: torch.Tensor, mel_w: torch.Tensor, hop: int, w0: int,
            w1: int) -> torch.Tensor:
    n, nmels = int(y.numel()), int(mel_w.shape[0])
    n_frames = 1 + n // hop
    out = torch.empty(nmels, n_frames, dtype=torch.float32, device=y.device)
    with torch.cuda.device(y.device):
        check(_lib.lib().svb_logmel(ptr(y.contiguous()), _i64(n), int(hop), ptr(window), int(w0), int(w1), ptr(twiddle),
                                    ptr(mel_w), nmels, ptr(out), n_frames, stream_ptr(y.device)), "svb_logmel")
    return out


_op("logmel(Tensor y, Tensor window, Tensor twiddle, Tensor mel_w, int hop, int w0, int w1) -> Tensor", _logmel,
    lambda y, window, twiddle, mel_w, hop, w0, w1: y.new_empty(mel_w.shape[0], 1 + y.numel() // hop))


# ------------------------------------------------------------------------------------------ TI-SV preprocessing
# split_nonsilent out (2 * n_slots + n_signals int64): the interval pairs of every signal's slot range, then the
# per-signal counts (-1: a non-finite sample), so that one host read fetches both (include/svb200.h)
def _split_nonsilent(y: torch.Tensor, offsets: torch.Tensor, slot_offsets: torch.Tensor, n_slots: int, top_db: float,
                     min_len: int) -> torch.Tensor:
    if y.dtype != torch.float32 or y.dim() != 1 or offsets.dtype != torch.int64 or slot_offsets.dtype != torch.int64:
        raise ValueError("split_nonsilent expects float32 samples (total,) and int64 offsets")
    if offsets.dim() != 1 or offsets.numel() < 1 or slot_offsets.shape != (offsets.numel() - 1,):
        raise ValueError("split_nonsilent expects offsets (n_signals + 1,) and slot_offsets (n_signals,)")
    _same_device("split_nonsilent", y, offsets, slot_offsets)
    ns, total = int(offsets.numel()) - 1, int(y.numel())
    out = torch.empty(2 * int(n_slots) + ns, dtype=torch.int64, device=y.device)
    if ns == 0:
        return out
    with torch.cuda.device(y.device):
        nbytes = _sz(0)
        check(_lib.lib().svb_split_workspace_bytes(_i64(total), ns, ctypes.byref(nbytes)), "svb_split_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=y.device)
        yc = y.contiguous() if total else y.new_zeros(1)
        check(_lib.lib().svb_split_nonsilent(ptr(yc), ptr(offsets.contiguous()), ns, _i64(total),
                                             ctypes.c_double(top_db), _i64(min_len), ptr(slot_offsets.contiguous()),
                                             ptr(ws), _sz(nbytes.value), ptr(out), ptr(out[2 * int(n_slots):]),
                                             stream_ptr(y.device)), "svb_split_nonsilent")
    return out


def _logmel_frames(y: torch.Tensor, rows: torch.Tensor, window: torch.Tensor, twiddle: torch.Tensor,
                   mel_w: torch.Tensor, frames: int, hop: int, w0: int, w1: int) -> torch.Tensor:
    if y.dtype != torch.float32 or rows.dtype != torch.int64 or rows.dim() != 2 or rows.shape[1] != 3:
        raise ValueError("logmel_frames expects float32 samples and int64 rows (P, 3)")
    _same_device("logmel_frames", y, rows, window, twiddle, mel_w)
    P, nmels = int(rows.shape[0]), int(mel_w.shape[0])
    out = torch.empty(P, nmels, int(frames), dtype=torch.float32, device=y.device)
    with torch.cuda.device(y.device):
        check(_lib.lib().svb_logmel_frames(ptr(y.contiguous()), ptr(rows.contiguous()), _i64(P), int(frames), int(hop),
                                           ptr(window), int(w0), int(w1), ptr(twiddle), ptr(mel_w), nmels, ptr(out),
                                           stream_ptr(y.device)), "svb_logmel_frames")
    return out


_op("split_nonsilent(Tensor y, Tensor offsets, Tensor slot_offsets, int n_slots, float top_db, int min_len) -> Tensor",
    _split_nonsilent, lambda y, offsets, slot_offsets, n_slots, top_db, min_len:
    y.new_empty(2 * n_slots + offsets.shape[0] - 1, dtype=torch.int64))
_op("logmel_frames(Tensor y, Tensor rows, Tensor window, Tensor twiddle, Tensor mel_w, int frames, int hop, int w0, "
    "int w1) -> Tensor", _logmel_frames,
    lambda y, rows, window, twiddle, mel_w, frames, hop, w0, w1: y.new_empty(rows.shape[0], mel_w.shape[0], frames))

OP_NAMES = ["pack_weights", "embedder_fwd", "embedder_bwd", "ge2e_loss", "ge2e_rows", "scale3", "centroids", "centroids_bwd",
            "utterance_centroids", "cossim", "cossim_bwd", "calc_loss", "calc_loss_bwd", "eer_counts", "eer_sweep", "peer_gather", "peer_reduce",
            "eer_finish", "verif_metrics", "verif_metrics_sim", "cohort_stats", "cohort_stats_scores", "score_trials",
            "asnorm_sim", "calib_metrics", "calib_train", "dvector_windows", "segment_mean", "clip_sgd", "logmel",
            "split_nonsilent", "logmel_frames"]
