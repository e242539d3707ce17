"""Multi-GPU GE2E: one process per GPU, speakers sharded across ranks (SURVEY.md section 8e).

The LSTM / projection / L2 norm are independent per utterance (pure data parallel, no exchange).  GE2E couples
speakers only through the centroids: by default (design "A") the ranks all-gather their (N_local, D) centroids, score
their own rows against all of them and all-reduce the centroid gradients; design "B" (mode="gather") all-gathers the
(N_local*M, D) d-vectors and lets every rank evaluate the whole global batch.  Either way w.grad/b.grad are identical on
every rank.  Parameter gradients are
all-reduced with SUM -- not mean -- because the reference loss is a sum over rows (utils.py:131).

The reference has no distributed code at all; this module is new functionality behind the same GE2ELoss object.
"""
import functools

import torch
import torch.distributed as dist

from . import ops


def speaker_shard(n_speakers, rank, world):
    """Contiguous speaker range [lo, hi) owned by ``rank``; requires n_speakers % world == 0."""
    if n_speakers % world:
        raise ValueError(f"{n_speakers} speakers do not shard evenly over {world} ranks")
    per = n_speakers // world
    return rank * per, (rank + 1) * per


def _fused_loss_and_grads(E, w, b, loss=0):
    return torch.ops.svb200.ge2e_loss(E, w, b, 1, True, int(loss))


def _rows_loss_and_grads(E_local, C_all, w, b, col0, loss=0):
    """-> (reduction buffer [dC (N*D) | loss, dw, db] of this rank's rows, dE of the rows without the centroid path)"""
    return torch.ops.svb200.ge2e_rows(E_local, C_all, w, b, int(col0), int(loss))


def _native_rows(compute_rows):
    """True for the library's row-shard arithmetic (with or without a bound loss method)."""
    return compute_rows is _rows_loss_and_grads or getattr(compute_rows, "func", None) is _rows_loss_and_grads


class _GlobalGE2EFn(torch.autograd.Function):
    """Design "B": all-gather of the d-vectors, every rank evaluates the whole global batch and keeps its slice."""

    @staticmethod
    def forward(ctx, local_emb, w, b, group, compute):
        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        Nl, M, D = local_emb.shape
        E_all = torch.empty(world * Nl, M, D, dtype=local_emb.dtype, device=local_emb.device)
        dist.all_gather_into_tensor(E_all, local_emb.contiguous(), group=group)
        loss, dE, dw, db = compute(E_all, w.detach(), b.detach())
        ctx.save_for_backward(dE[rank * Nl:(rank + 1) * Nl], dw, db)
        return loss

    @staticmethod
    def backward(ctx, g):
        dE, dw, db = ctx.saved_tensors
        if dE.device.type == "cuda":
            dE, dw, db = torch.ops.svb200.scale3(dE, dw, db, g)
        else:                       # host-logic tests (gloo, injected compute)
            dE, dw, db = dE * g, dw * g, db * g
        return dE, dw, db, None, None


class _ShardedGE2EFn(torch.autograd.Function):
    """Design "A" (SURVEY.md section 8e): the speakers of other ranks enter a rank's rows only through their centroids,
    so the forward exchange is an all-gather of the (N_local, D) centroids (65 KB per rank at 64 x 256 instead of the
    655 KB of d-vectors), every rank scores ITS rows against all N centroids (1/world of the work instead of all of
    it), and one SUM all-reduce of [dC (N, D) | loss, dw, db] (524 KB at N = 512) returns the centroid gradients, which
    each rank spreads over its own utterances (dC_j / M)."""

    @staticmethod
    def forward(ctx, local_emb, w, b, group, compute_rows):
        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        Nl, M, D = local_emb.shape
        E = local_emb.contiguous()
        C_local = torch.ops.svb200.centroids(E) if _native_rows(compute_rows) else E.mean(dim=1)
        C_all = torch.empty(world * Nl, D, dtype=E.dtype, device=E.device)
        dist.all_gather_into_tensor(C_all, C_local.contiguous(), group=group)
        red, dE = compute_rows(E, C_all, w.detach(), b.detach(), rank * Nl)
        dist.all_reduce(red, op=dist.ReduceOp.SUM, group=group)
        N = world * Nl
        dC_own = red[:N * D].view(N, D)[rank * Nl:(rank + 1) * Nl]
        if dE.device.type == "cuda":
            dE = dE + torch.ops.svb200.centroids_bwd(dC_own.contiguous(), M)
        else:
            dE = dE + (dC_own / M).unsqueeze(1)
        ctx.save_for_backward(dE, red[N * D + 1].clone(), red[N * D + 2].clone())
        return red[N * D].clone()

    backward = _GlobalGE2EFn.backward


class PeerExchange:
    """Symmetric buffers of one process group for the GE2E exchange over NVLink peer memory
    (torch.distributed._symmetric_memory): every rank writes its centroids / its centroid-gradient partials into ITS
    buffer and reads the peers' buffers with plain loads (svb_peer_gather / svb_peer_reduce), two device-side barriers
    per step instead of two NCCL collectives.  Layout per rank (floats): [own centroids N_local*D (padded to 4) |
    dC partial Nc*D | loss, dw, db]."""

    def __init__(self, group, n_local, D, device):
        import torch.distributed._symmetric_memory as symm
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.n_local, self.D = int(n_local), int(D)
        self.nc = self.world * self.n_local
        self.off_c = 0
        self.len_c = (self.n_local * self.D + 3) // 4 * 4
        self.off_red = self.len_c
        self.len_red = self.nc * self.D + 3
        self.buf = symm.empty(self.len_c + (self.len_red + 3) // 4 * 4, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.ptrs = int(self.handle.buffer_ptrs_dev)
        torch.cuda.synchronize(device)
        self.handle.barrier(channel=0)

    def matches(self, n_local, D, device):
        return self.n_local == int(n_local) and self.D == int(D) and self.buf.device == device


class _PeerGE2EFn(torch.autograd.Function):
    """Design "A" with the exchange over peer memory: same arithmetic as _ShardedGE2EFn, no NCCL call on the GE2E path."""

    @staticmethod
    def forward(ctx, local_emb, w, b, px, loss=0):
        Nl, M, D = local_emb.shape
        E = local_emb.contiguous()
        N = px.nc
        px.buf[:Nl * D].view(Nl, D).copy_(torch.ops.svb200.centroids(E))
        px.handle.barrier(channel=0)                       # every rank's centroids are in its buffer
        C_all = torch.ops.svb200.peer_gather(px.buf, px.ptrs, px.world, px.off_c, px.len_c)[:, :Nl * D].reshape(N, D)
        red, dE = torch.ops.svb200.ge2e_rows(E, C_all.contiguous(), w.detach(), b.detach(), px.rank * Nl, int(loss))
        px.buf[px.off_red:px.off_red + px.len_red].copy_(red)
        px.handle.barrier(channel=1)                       # every rank's partials are in its buffer
        dC_own, tail = torch.ops.svb200.peer_reduce(px.buf, px.ptrs, px.world, px.off_red, px.rank * Nl * D, Nl * D,
                                                    N * D, 3)
        dE = dE + torch.ops.svb200.centroids_bwd(dC_own.view(Nl, D), M)
        ctx.save_for_backward(dE, tail[1].clone(), tail[2].clone())
        return tail[0].clone()

    @staticmethod
    def backward(ctx, g):
        dE, dw, db = ctx.saved_tensors
        dE, dw, db = torch.ops.svb200.scale3(dE, dw, db, g)
        return dE, dw, db, None, None




class GlobalGE2ELoss(torch.nn.Module):
    """Wraps a GE2ELoss so that ``forward(local_embeddings (N_local, M, D))`` returns the loss of the GLOBAL batch
    (the same number on every rank) and back-propagates this rank's slice of dL/dE.

    ``mode="rows"`` (default): centroid all-gather + this rank's rows against all centroids + one all-reduce of the
    centroid gradients (design A); ``mode="peer"``: the same with both exchange steps over NVLink peer memory
    (symmetric buffers, svb_peer_gather / svb_peer_reduce, no NCCL call on the GE2E path; falls back to "rows" where
    symmetric memory is unavailable); ``mode="gather"``: d-vector all-gather, every rank evaluates the global batch
    (design B, round 1).  ``compute`` injects the arithmetic (host-logic tests on CPU / gloo).  Without it, the loss
    method is the criterion's ``loss_method`` ("softmax" or "contrast"), read at every call."""

    def __init__(self, criterion, group=None, compute=None, mode="rows"):
        super().__init__()
        if mode not in ("rows", "gather", "peer"):
            raise ValueError(mode)
        self.criterion = criterion
        self.group = group
        self.mode = mode
        self._default_compute = compute is None
        self.compute = compute or (_fused_loss_and_grads if mode == "gather" else _rows_loss_and_grads)
        self._px = None

    def _loss_code(self):
        return ops.loss_code(getattr(self.criterion, "loss_method", "softmax"))

    def _compute(self):
        """The arithmetic of this call: an injected ``compute`` as given, else the library's with the criterion's loss
        method bound (the softmax default is the plain function)."""
        code = self._loss_code()
        if not self._default_compute or code == 0:
            return self.compute
        return functools.partial(self.compute, loss=code)

    def _peer(self, E):
        """The symmetric buffers of this (group, shape), or None when peer memory is not available (-> NCCL rows)."""
        if self._px is False:
            return None
        Nl, _, D = E.shape
        if self._px is None or not self._px.matches(Nl, D, E.device):
            try:
                if (Nl * D) % 4:
                    raise RuntimeError("N_local * D must be a multiple of 4")
                self._px = PeerExchange(self.group, Nl, D, E.device)
            except Exception as exc:                    # no symmetric memory on this system / build
                import warnings
                warnings.warn(f"GlobalGE2ELoss(mode='peer'): falling back to the NCCL exchange ({exc!r})")
                self._px = False
                return None
        return self._px

    def forward(self, local_embeddings):
        if self.mode == "peer" and local_embeddings.is_cuda:
            px = self._peer(local_embeddings)
            if px is not None:
                return _PeerGE2EFn.apply(local_embeddings, self.criterion.w, self.criterion.b, px, self._loss_code())
        fn = _GlobalGE2EFn if self.mode == "gather" else _ShardedGE2EFn
        return fn.apply(local_embeddings, self.criterion.w, self.criterion.b, self.group, self._compute())


class PeerAllReduce:
    """Two-shot SUM all-reduce of a flat float32 tensor over NVLink peer memory (symmetric buffer of ``numel`` floats per
    rank, csrc/peer.cu): reduce-scatter by plain loads from all peers, in place and in rank order, then an all-gather
    by plain loads.  48.5 MB of gradients at 8 GPUs: every rank pulls 2 x 42 MB over NVLink."""

    def __init__(self, group, numel, device):
        import torch.distributed._symmetric_memory as symm
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.numel = int(numel)
        sl = (self.numel + 4 * self.world - 1) // (4 * self.world) * 4
        self.buf = symm.empty(sl * self.world, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.ptrs = int(self.handle.buffer_ptrs_dev)
        torch.cuda.synchronize(device)
        self.handle.barrier(channel=0)

    def __call__(self, flat):
        if flat.numel() != self.numel or flat.dtype != torch.float32 or not flat.is_contiguous():
            raise ValueError("PeerAllReduce: tensor does not match the buffer")
        return ops.peer_allreduce_(flat, self.buf, self.ptrs, self.world, self.rank,
                                   lambda ch: self.handle.barrier(channel=ch))


_PEER_ALLREDUCE = {}


def _peer_allreduce_for(group, flat):
    """The PeerAllReduce of (group, size, device), or None when symmetric memory is unavailable."""
    key = (id(group), flat.numel(), str(flat.device))
    if key not in _PEER_ALLREDUCE:
        try:
            _PEER_ALLREDUCE[key] = PeerAllReduce(group, flat.numel(), flat.device)
        except Exception as exc:
            import warnings
            warnings.warn(f"allreduce_gradients(peer=True): falling back to NCCL ({exc!r})")
            _PEER_ALLREDUCE[key] = None
    return _PEER_ALLREDUCE[key]


def _flat_view(grads):
    """One contiguous 1-D tensor over the storage the gradients share, if they are contiguous slices of ONE allocation
    that tile it without gaps (what svb200::embedder_bwd returns; the slices come out of a custom op, so they carry no
    autograd ``_base``), else None."""
    g0 = grads[0]
    try:
        st = g0.untyped_storage()
        if any(not g.is_contiguous() or g.dtype != g0.dtype or g.device != g0.device or
               g.untyped_storage().data_ptr() != st.data_ptr() for g in grads):
            return None
    except Exception:
        return None
    spans = sorted((g.storage_offset(), g.numel()) for g in grads)
    pos = spans[0][0]
    for off, n in spans:
        if off != pos:
            return None
        pos += n
    total = pos - spans[0][0]
    return torch.as_strided(g0, (total,), (1,), spans[0][0])


def allreduce_gradients(params, group=None, peer=False):
    """SUM all-reduce of the parameter gradients (one call when the grads are views of one flat buffer, as
    EmbedderFn.backward produces them).  ``peer=True``: two-shot all-reduce over NVLink peer memory (PeerAllReduce)
    instead of NCCL for the flat buffer."""
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    base = _flat_view(grads)
    if base is not None:
        if peer and base.is_cuda and base.dtype == torch.float32 and base.is_contiguous():
            ar = _peer_allreduce_for(group, base)
            if ar is not None:
                ar(base)
                return
        dist.all_reduce(base, op=dist.ReduceOp.SUM, group=group)
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


class OverlappedGradReducer:
    """SUM all-reduce of the embedder's gradients in four buckets (projection, then the LSTM layers from the top),
    each started the moment its kernels are enqueued (svb_set_grad_ready_callback), so that the NCCL transfers run
    beside the remaining weight-gradient GEMMs instead of after the whole backward::

        reducer = OverlappedGradReducer()
        with reducer:
            loss.backward()

    Every rank issues the same buckets in the same order (the order is fixed by the library).

    The buckets are slices of the flat buffer the backward op returns its gradients in.  Before the op hands that
    buffer to autograd, ``finish()`` makes the compute stream wait for the all-reduces (called by the op itself, see
    ops.set_grad_bucket_hook), so whatever autograd then does with the gradients -- adopt the views as ``p.grad``
    (``zero_grad(set_to_none=True)``), add them to an existing ``p.grad`` (``set_to_none=False``, gradient
    accumulation over micro-batches), run parameter hooks -- happens on REDUCED values.  The transfers still overlap
    every kernel of the backward that follows their bucket; only the last bucket (layer 0) has nothing after it."""

    def __init__(self, group=None, all_reduce=None):
        self.group = group
        self.works = []
        self.buckets = 0
        self._all_reduce = all_reduce or (lambda t: dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group,
                                                                    async_op=True))

    def _hook(self, bucket):
        self.buckets += 1
        self.works.append(self._all_reduce(bucket))

    def __enter__(self):
        ops.set_grad_bucket_hook(self._hook, self.finish)
        return self

    def __exit__(self, *exc):
        ops.set_grad_bucket_hook(None)
        self.finish()
        return False

    def finish(self):
        """The current stream waits for every all-reduce started so far (idempotent)."""
        works, self.works = self.works, []
        for w in works:
            if w is not None:
                w.wait()
