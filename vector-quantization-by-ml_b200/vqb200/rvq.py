"""``ResidualVQ`` / ``GroupedResidualVQ``: drop-ins for reference vector_quantization/residual_vq.py.

The per-level loop (reference :212-243) has two implementations with identical results:
  * generic: each level is a ``VectorQuantize`` call and the residual arithmetic is autograd-visible;
  * fused (no autograd needed): one kernel per level does gather + straight-through + commitment loss
    + ``residual -= q`` + ``quantized_out += q`` and emits the next level's scaled fp16 search operand, so the
    residual is read once per level (``vqb_rvq_level``).
"""
from __future__ import annotations

import random
from functools import partial
from math import ceil

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import nn

from . import _lib, ops
from .vq import VectorQuantize


def _round_up_multiple(num, mult):
    return ceil(num / mult) * mult


class ResidualVQ(nn.Module):
    def __init__(self, *, dim, num_quantizers, codebook_dim=None, shared_codebook=False, heads=1,
                 quantize_dropout=False, quantize_dropout_cutoff_index=0, quantize_dropout_multiple_of=1,
                 rotation_trick=False, **kwargs):
        super().__init__()
        assert heads == 1, "residual vq is not compatible with multi-headed codes"
        codebook_dim = codebook_dim if codebook_dim is not None else dim
        requires_projection = codebook_dim * heads != dim
        self.project_in = nn.Linear(dim, codebook_dim) if requires_projection else nn.Identity()
        self.project_out = nn.Linear(codebook_dim, dim) if requires_projection else nn.Identity()
        self.has_projections = requires_projection
        self.num_quantizers = num_quantizers
        self.layers = nn.ModuleList([VectorQuantize(dim=codebook_dim, codebook_dim=codebook_dim, **kwargs)
                                     for _ in range(num_quantizers)])
        assert all(not vq.has_projections for vq in self.layers)
        for vq in self.layers:                  # the rotation-trick gradient (VectorQuantize.rotation_trick) on every level
            vq.rotation_trick = bool(rotation_trick)
        self.quantize_dropout = quantize_dropout and num_quantizers > 1
        assert quantize_dropout_cutoff_index >= 0
        self.quantize_dropout_cutoff_index = quantize_dropout_cutoff_index
        self.quantize_dropout_multiple_of = quantize_dropout_multiple_of
        self.use_fused_levels = True
        if shared_codebook:
            first = self.layers[0]._codebook
            for vq in self.layers[1:]:
                vq._codebook = first

    @property
    def codebooks(self):
        # full (K,d) codebooks: a sharded codebook is all-gathered (a collective when a shard changed since the last call)
        return torch.stack([layer._codebook.full_codebook()[0] if layer._codebook.sharded
                            else layer._codebook.embeddings[0] for layer in self.layers], dim=0)

    def get_codes_from_indices(self, indices):
        q_dim = indices.shape[-1]
        lead = tuple(indices.shape[:-1])
        flat = indices.reshape(indices.shape[0], -1, q_dim)
        if q_dim < self.num_quantizers:
            assert self.quantize_dropout > 0.0, "quantize dropout must be greater than 0 if you wish to " \
                                                "reconstruct from a signal with less fine quantizations"
            flat = F.pad(flat, (0, self.num_quantizers - q_dim), value=-1)
        dropped = flat == -1
        flat = flat.masked_fill(dropped, 0)
        books = self.codebooks
        codes = torch.stack([books[i][flat[..., i]] for i in range(self.num_quantizers)], dim=0)   # q b n d
        codes = codes.masked_fill(dropped.permute(2, 0, 1)[..., None], 0.0)
        return codes.reshape(self.num_quantizers, *lead, codes.shape[-1])

    def get_output_from_indices(self, indices):
        return self.project_out(self.get_codes_from_indices(indices).sum(dim=0))

    # ------------------------------------------------------------------ fused level loop
    def _can_fuse(self, x, dropout_active) -> bool:
        if not self.use_fused_levels or dropout_active or not x.is_cuda or x.ndim != 3:
            return False
        if any(l._codebook.sharded for l in self.layers):
            return False        # the level kernels search and update one whole codebook; shards need `Codebook._run`
        if torch.is_grad_enabled() and x.requires_grad and not self._can_fuse_autograd(x):
            return False
        l0 = self.layers[0]
        if self.training and (l0.commitment_use_cross_entropy_loss or l0.has_codebook_diversity_loss):
            return False        # losses on the dense similarities: the generic per-level loop computes them
        if l0.in_place_codebook_optimizer is not None:
            return False        # the optimizer step inside forward (reference vector_quantize_pytorch.py:233-256)
        if any(l._codebook._variants_active() or l.has_codebook_orthogonal_loss for l in self.layers):
            return False        # gumbel sampling / affine / orthogonal loss: the generic per-level loop
        if l0._codebook.learnable_codebook and self.training and torch.is_grad_enabled() and \
                any(l._codebook.embeddings.requires_grad for l in self.layers):
            # the commitment loss must reach the codebook Parameters (reference :263-269) even when the input carries
            # no gradient (frozen encoder): the fused loop runs under no_grad
            return False
        return l0.channel_last and not l0._codebook.input_l2norm and l0.heads == 1

    def _can_fuse_autograd(self, x) -> bool:
        """The fused loop under autograd (`_FusedRVQ`): training mode, EMA codebooks (the gradient to the input is all
        there is), at least two levels, a width the replay kernels take and one gradient estimator for all levels."""
        d = x.shape[-1]
        return bool(self.training and all(l.training for l in self.layers)
                    and not any(l._codebook.learnable_codebook for l in self.layers)
                    and len({l.rotation_trick for l in self.layers}) == 1
                    and len(self.layers) >= 2 and ops.rvq_replay_out_supported(d, len(self.layers)))

    def _forward_fused(self, x, mask, freeze_codebook):
        if torch.is_grad_enabled() and x.requires_grad:
            out, idx, losses = _FusedRVQ.apply(x, self, mask, freeze_codebook)
            Q = idx.shape[0]
            return out, [idx[i] for i in range(Q)], [losses[i:i + 1] for i in range(Q)]
        with torch.no_grad():
            out, all_idx, all_loss, late = self._fused_levels(x, mask, freeze_codebook)
            self._fused_expiry(late, mask)
        return out, all_idx, all_loss

    @torch.no_grad()
    def _fused_levels(self, x, mask, freeze_codebook, for_backward=False):
        """Everything of the fused level loop that needs no host round trip (capturable in a CUDA graph).
        `for_backward`: the codebooks each level gathered from are kept as copies for `_FusedRVQ.backward`, which may
        run after they moved (a later training forward of the same module refreshes them in place)."""
        B, n, d = x.shape
        N = B * n
        dev = x.device
        # level 0 reads the input itself (never written: every level writes its residual to another buffer)
        x0 = _lib.aligned(x.reshape(N, d).float())
        bufs = [torch.empty((N, d), dtype=torch.float32, device=dev) for _ in range(min(2, len(self.layers)))]
        all_idx, all_loss, loss_bufs = [], [], []
        Q = len(self.layers)
        # `quantized_out` (residual_vq.py:233) is not accumulated level by level -- that is a read-modify-write of an
        # (N,d) buffer in every level pass -- but replayed once at the end from x and the indices with the same IEEE
        # operations (vqb_rvq_replay_out): bit-identical, 2 x 4d bytes per row and level less HBM traffic
        replay = Q >= 2 and ops.rvq_replay_out_supported(d, Q)
        out = None if replay else torch.empty((N, d), dtype=torch.float32, device=dev)
        prepared = False
        # Dead-code check (reference codebooks.py:245-252) costs one host sync per level (0.75 ms of an 8.8 ms C4 step).
        # A level's codebook is not read again in this forward unless it is shared, so the checks of all levels are
        # answered by ONE sync after the loop; in the rare case that a code did die, that level's input is
        # reconstructed bit-exactly from the indices (same IEEE operations as the level kernel) and the draws happen
        # in level order, i.e. in the reference's RNG order.  Not possible while a later level still has to run its
        # kmeans init (that draws too) or when the codebook is shared.
        books = [l._codebook for l in self.layers]
        defer = len({id(b) for b in books}) == Q and all(b.is_initialized for b in books)
        pending, pre_emb, late_apply = [], [], []
        overlap = defer and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        for li, layer in enumerate(self.layers):
            cb = layer._codebook
            cur = x0 if li == 0 else bufs[(li - 1) % len(bufs)]
            nxt = bufs[li % len(bufs)]
            flat = cur[None]
            mask_u8 = cb._expand_mask(mask, N)
            if not cb.is_initialized:
                cb._kmeans_init(flat, mask_u8)
                cb.is_initialized = True
                prepared = False
            emb = cb.embeddings.detach()
            idx, _, ws = ops.search(flat, emb, cb._codebook_cache(), cb.use_cosine_sim, latents_prepared=prepared)
            training = self.training and layer.training
            do_ema = training and cb.ema_update and not freeze_codebook
            if defer or replay:   # the codebook the gather uses (the EMA refresh below overwrites it in place)
                pre_emb.append((emb.clone() if do_ema or for_backward else emb, training))
            # the next level's operands are prepared in the same pass when its codebook cache is already final:
            # a different codebook object (not shared) that is initialised
            next_cache = None
            if li + 1 < Q:
                ncb = self.layers[li + 1]._codebook
                if ncb is not cb and ncb.is_initialized:
                    next_cache = ncb._codebook_cache()
            if do_ema and mask_u8 is None and cb.fused_quantize_ema and ops.rvq_level_ema_supported(d):
                # un-masked training level: level step and EMA sums share one pass over the residual
                loss_buf, stats = ops.rvq_level_ema(cur, nxt, emb[0], idx[0], training, li == 0, out, next_cache,
                                                    bound_ws=ws)
            else:
                stats = ops.ema_reduce(flat, idx, mask_u8, cb.codebook_size, bound_ws=ws) if do_ema else None
                loss_buf = ops.rvq_level(cur, nxt, emb[0], idx[0], mask_u8, training, li == 0, out, next_cache)
            prepared = next_cache is not None
            if do_ema and overlap and cb.use_ddp:
                # data parallel, distinct codebooks: nothing later in this forward reads codebook `li` (the gather's
                # copy was taken above), so the statistics all_reduce of this level runs beside the next levels'
                # searches and its refresh is applied after the loop (reference residual_vq.py:212-243 with
                # codebooks.py:410,415 per level: same values, other order of independent operations)
                late_apply.append((dist.all_reduce(stats, async_op=True), stats, cb, li))
            elif do_ema:
                cb._all_reduce(stats)
                cb._apply_ema(stats)
                if not defer:
                    cb.expire_codes_(flat)
                elif cb.threshold_ema_dead_code != 0:
                    pending.append((li, cb, (cb.cluster_size < cb.threshold_ema_dead_code).sum()))
            loss = torch.zeros(1, device=dev)
            loss_bufs.append((loss_buf, layer.commitment_weight if (training and layer.has_commitment_loss) else 0.0))
            if training and layer.has_commitment_loss:
                loss = loss + loss_buf[0] * layer.commitment_weight
            all_idx.append(idx.reshape(B, n))
            all_loss.append(loss)
        if replay:
            out = ops.rvq_replay_out(x0, [e[0] for e, _ in pre_emb], [i.reshape(-1) for i in all_idx],
                                     [tr for _, tr in pre_emb], books[0]._expand_mask(mask, N))
        for work, stats, cb, li in late_apply:
            work.wait()
            cb._apply_ema(stats)
            if cb.threshold_ema_dead_code != 0:
                pending.append((li, cb, (cb.cluster_size < cb.threshold_ema_dead_code).sum()))
        dead_counts = torch.stack([p[2] for p in pending]) if pending else None
        late = (pending, dead_counts, x0, pre_emb, all_idx, loss_bufs)
        return out.reshape(B, n, d), all_idx, all_loss, late

    @torch.no_grad()
    def _fused_expiry(self, late, mask):
        """The deferred dead-code checks of all levels: ONE host sync, then (rarely) the replay described above."""
        pending, dead_counts, x0, pre_emb, all_idx = late[:5]
        if not pending:
            return
        dead = dead_counts.tolist()                                      # the one host sync
        if not any(dead):
            return
        N = x0.shape[0]
        live = None if mask is None else pending[0][1]._expand_mask(mask, N).bool()[:, None]
        r, at = x0, 0
        for (li, cb, _), m in zip(pending, dead):
            if not m:
                continue
            while at < li:                                               # replay levels at .. li-1 on the residual
                e, tr = pre_emb[at]
                cq = e[0][all_idx[at].reshape(-1)]
                q = r + (cq - r) if tr else cq
                if live is not None:
                    q = torch.where(live, q, r)
                r = r - q
                at += 1
            cb.expire_codes_(r[None])

    # ------------------------------------------------------------------ CUDA graph of the fused level loop (opt-in)
    def enable_cuda_graph(self, flag: bool = True, max_graphs: int = 4, data_parallel: bool = False) -> "ResidualVQ":
        """Replay the fused level loop (~25 launches per level) as ONE CUDA graph per (input address, shape, mode).
        Opt-in because graph outputs are STATIC buffers: the tensors returned by a forward are overwritten by the next
        forward on the same input address (clone what must survive).  The first forward on a new input address runs
        eagerly, the second captures, later ones replay; the dead-code check stays outside the graph (one host sync
        per forward, as in eager mode).  Not used while a codebook still needs its kmeans init, with a mask, with
        quantize-dropout, a shared codebook, or while `ops.TIME_SEARCH_KERNEL` brackets kernels with events.
        Under data parallelism the graph holds the per-level statistics all_reduce (NCCL collectives are capturable);
        that needs `data_parallel=True` as a promise that EVERY rank enables the graph and calls forward with the same
        sequence of (shape, mode) keys -- a rank that replays while another captures or runs eagerly would dead-lock
        in the collective.  Call `enable_cuda_graph(False)` before `destroy_process_group()`: a live graph keeps
        kernels of the communicator."""
        self._graph_on = bool(flag)
        self._graph_ddp = bool(data_parallel)
        self._graph_max = int(max_graphs)
        self._graphs = {}
        return self

    def _graph_usable(self, x, mask) -> bool:
        if not getattr(self, "_graph_on", False) or mask is not None or ops.TIME_SEARCH_KERNEL:
            return False
        if torch.is_grad_enabled() and x.requires_grad:
            return False        # the autograd form of the fused loop (`_FusedRVQ`) runs eagerly
        books = [l._codebook for l in self.layers]
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and any(b.use_ddp for b in books) \
                and not getattr(self, "_graph_ddp", False):
            return False        # the statistics all_reduce of every level has to be captured on all ranks at once
        return len({id(b) for b in books}) == len(books) and all(b.is_initialized and not b.sharded for b in books)

    def _forward_graphed(self, x, freeze_codebook):
        # under data parallelism the ranks' input addresses differ, their SEQUENCE of keys must not: the k-th distinct
        # address of a rank stands for the k-th of every other rank
        key = (x.data_ptr(), tuple(x.shape), x.dtype, bool(freeze_codebook), self.training, x.device.index)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= self._graph_max:
                return self._forward_fused(x, None, freeze_codebook)
            self._graphs[key] = "warm"                      # this forward is the eager warm-up of the key
            return self._forward_fused(x, None, freeze_codebook)
        if ent == "warm":
            g = torch.cuda.CUDAGraph()
            for layer in self.layers:       # the graph must ALWAYS rebuild the search operands of the codebooks: what
                layer._codebook._dirty = True   # python decides during capture is what every replay does
            torch.cuda.synchronize(x.device)
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                res = self._fused_levels(x, None, freeze_codebook)
            ent = self._graphs[key] = (g, res, x)           # `x` kept alive: its address is baked into the graph
        g, (out, all_idx, all_loss, late), _ = ent
        g.replay()
        for layer in self.layers:                           # the replayed EMA refresh changed `embeddings` in place
            layer._codebook._dirty = True
        self._fused_expiry(late, None)
        return out, all_idx, all_loss

    # ------------------------------------------------------------------ forward (reference :134-269)
    def forward(self, x, mask=None, indices=None, return_all_codes=False, freeze_codebook=False,
                rand_quantize_dropout_fixed_seed=None):
        assert indices is None, "the indices / cross-entropy path is disabled in the reference as well (:152)"
        num_quant, mult = self.num_quantizers, self.quantize_dropout_multiple_of
        device = x.device
        x = self.project_in(x)

        should_dropout = self.training and self.quantize_dropout
        if should_dropout:
            if rand_quantize_dropout_fixed_seed is not None:
                rand = random.Random(rand_quantize_dropout_fixed_seed)
            elif dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                # the reference's seed sync is broken (residual_vq.py:183-185); broadcast rank 0's seed instead
                t = torch.tensor([random.randrange(10_000)], device=device)
                dist.broadcast(t, src=0)
                rand = random.Random(int(t.item()))
            else:
                rand = random
            dropout_index = rand.randrange(self.quantize_dropout_cutoff_index, num_quant)
            if mult != 1:
                dropout_index = _round_up_multiple(dropout_index + 1, mult) - 1
            null_shape = (x.shape[0], *x.shape[-2:]) if x.ndim >= 4 else tuple(x.shape[:2])
            null_indices = torch.full(null_shape, -1, device=device, dtype=torch.long)
            null_loss = torch.full((1,), 0.0, device=device, dtype=x.dtype)

        if self._can_fuse(x, should_dropout):
            if self._graph_usable(x, mask):
                quantized_out, all_indices, all_losses = self._forward_graphed(x, freeze_codebook)
            else:
                quantized_out, all_indices, all_losses = self._forward_fused(x, mask, freeze_codebook)
        else:
            quantized_out = 0.0
            residual = x
            all_losses, all_indices = [], []
            for qi, layer in enumerate(self.layers):
                if should_dropout and qi > dropout_index:
                    all_indices.append(null_indices)
                    all_losses.append(null_loss)
                    continue
                quantized, idx, loss = layer(residual, mask=mask, freeze_codebook=freeze_codebook)
                residual = residual - quantized.detach()
                quantized_out = quantized_out + quantized
                all_indices.append(idx)
                all_losses.append(loss)

        quantized_out = self.project_out(quantized_out)
        all_losses, all_indices = map(partial(torch.stack, dim=-1), (all_losses, all_indices))
        ret = (quantized_out, all_indices, all_losses)
        if return_all_codes:
            ret = (*ret, self.get_codes_from_indices(all_indices))
        return ret


class _FusedRVQ(torch.autograd.Function):
    """The fused level loop with a gradient to the input.  Reference autograd through residual_vq.py:212-243: every
    level returns r_l + (q_l - r_l).detach() and the next residual subtracts a detached quantity, so d out / d x = Q I;
    the commitment loss of level l, mse(c_l.detach(), r_l), adds w_l 2 (r_l - c_l) / (rows d).  Backward is ONE pass
    that replays the residuals from x and the indices (vqb_rvq_backward) against the codebooks as they were before each
    level's EMA step -- the generic per-level loop instead keeps Q (N,d) residuals alive for autograd.  With
    `rotation_trick` on every level, each level's output gradient is transported by that level's rotation instead of
    passed through (vqb_rvq_backward_rot); the forward is the same."""

    @staticmethod
    def forward(ctx, x, rvq, mask, freeze_codebook):
        with torch.no_grad():
            out, all_idx, all_loss, late = rvq._fused_levels(x.detach(), mask, freeze_codebook, for_backward=True)
            rvq._fused_expiry(late, mask)
        _, _, x0, pre_emb, _, loss_bufs = late
        ctx.x0, ctx.pre_emb, ctx.loss_bufs = x0, pre_emb, loss_bufs
        ctx.idx = [i.reshape(-1) for i in all_idx]
        ctx.mask_u8 = rvq.layers[0]._codebook._expand_mask(mask, x0.shape[0])
        ctx.shape, ctx.dtype = x.shape, x.dtype
        ctx.rotation = rvq.layers[0].rotation_trick
        idx = torch.stack(all_idx, 0)
        ctx.mark_non_differentiable(idx)
        return out, idx, torch.cat(all_loss, 0)

    @staticmethod
    def backward(ctx, g_out, _g_idx, g_losses):
        N, d = ctx.x0.shape
        if g_losses is None:
            coef = torch.zeros(len(ctx.idx), device=ctx.x0.device)
        else:
            # grad of level l's loss * commitment weight * 2 / (rows used * d), all on the device
            coef = torch.stack([g_losses[l].float() * (w * 2.0 / d) / lb[1] for l, (lb, w) in enumerate(ctx.loss_bufs)])
        g = g_out.reshape(N, d) if g_out is not None else None
        backward = ops.rvq_backward_rot if ctx.rotation else ops.rvq_backward
        gx = backward(ctx.x0, [e[0] for e, _ in ctx.pre_emb], ctx.idx, [tr for _, tr in ctx.pre_emb], coef, g,
                      ctx.mask_u8)
        return gx.reshape(ctx.shape).to(ctx.dtype), None, None, None


class GroupedResidualVQ(nn.Module):
    """reference residual_vq.py:275-357: split the feature dim into groups, one ResidualVQ each."""

    def __init__(self, *, dim, groups=1, channel_last=True, **kwargs):
        super().__init__()
        self.dim = dim
        self.groups = groups
        assert dim % groups == 0
        self.channel_last = channel_last
        self.rvqs = nn.ModuleList([ResidualVQ(dim=dim // groups, **kwargs) for _ in range(groups)])

    @property
    def split_dim(self):
        return -1 if self.channel_last else 1

    @property
    def codebooks(self):
        return torch.stack(tuple(rvq.codebooks for rvq in self.rvqs))

    def get_codes_from_indices(self, indices):
        return torch.stack(tuple(rvq.get_codes_from_indices(i) for rvq, i in zip(self.rvqs, indices)))

    def get_output_from_indices(self, indices):
        outs = tuple(rvq.get_output_from_indices(i) for rvq, i in zip(self.rvqs, indices))
        return torch.cat(outs, dim=self.split_dim)

    def forward(self, x, indices=None, return_all_codes=False, freeze_codebook=False, mask=None):
        assert indices is None or len(indices) == 0, "the indices / cross-entropy path is not supported"
        assert x.shape[self.split_dim] == self.dim
        chunks = x.chunk(self.groups, dim=self.split_dim)
        seed = random.randint(0, int(1e7))
        out = tuple(rvq(c.contiguous(), return_all_codes=return_all_codes, mask=mask, freeze_codebook=freeze_codebook,
                        rand_quantize_dropout_fixed_seed=seed) for rvq, c in zip(self.rvqs, chunks))
        quantized, all_indices, commit_losses, *maybe_codes = tuple(zip(*out))
        ret = (torch.cat(quantized, dim=self.split_dim), torch.stack(all_indices), torch.stack(commit_losses))
        if maybe_codes:
            ret = (*ret, torch.stack(maybe_codes[0]))
        return ret
