"""``SimVQ`` / ``ResidualSimVQ``: upstream vector-quantize-pytorch's modules of the same names (arXiv:2411.02038).

The codebook is not stored.  It is C' = T(F): a frozen random buffer F (K, d_f) mapped by a learned linear layer T, so
every step moves all K codes through T and no EMA refresh or dead-code expiry is needed.  Each forward computes C' once
in fp32 and runs the library's kernels on it: the tensor-core search, then the one-pass gather + loss + per-code sums
(`vqb_quantize_ema`) whose sums (S_k, n_k) give the codebook gradient, and the straight-through or rotation-trick
backward.  The loss weighs its two gradients differently: weight 1 to the codebook, beta to the input,

    loss = cw * (mse(x.detach(), q) + beta * mse(x, q.detach()))
    d loss / d x     = cw * beta * 2 (x - q) / (N d)
    d loss / d C'[k] = cw * 2 (n_k C'[k] - S_k) / (N d)

and torch autograd carries the codebook gradient on from C' to T.  The returned `quantized` is the straight-through
value fl(x + fl(q - x)) with either gradient estimator, in training and in eval (upstream returns it in both).
"""
from __future__ import annotations

import torch
from torch import nn

from . import _lib, ops


def _identity(t):
    return t


def _codebook_grad(grad_loss, cw, rows, stats, codes):
    """cw * 2 (n_k C'[k] - S_k) / (rows d) * grad_loss, from the per-code sums stats (1,K,d+1) of `ops.ema_reduce`."""
    d = codes.shape[-1]
    return (grad_loss.float() * (2.0 * cw / d) / rows) * (stats[0, :, d:] * codes[0] - stats[0, :, :d])


class _SimVQQuantize(torch.autograd.Function):
    """Training forward of one SimVQ level on x (1,N,d) against the codebook C' (K,d): returns the straight-through
    value q (1,N,d) fp32 and the loss.  `codes` is C' detached as a (1,K,d) fp32 buffer, `idx` (1,N) the search's
    indices and `bound_ws` the workspace that search returned (it sizes the fixed-point sums of the fused pass)."""

    @staticmethod
    def forward(ctx, x, codebook, codes, idx, bound_ws, beta, cw, rotation):
        d = x.shape[-1]
        fused = ops.quantize_ema_supported(d)
        if fused:
            q, loss, stats = ops.quantize_ema(x, codes, idx, True, True, bound_ws)
        else:
            (q, loss), stats = ops.gather_st_loss(x, codes, idx, None, True, True), None
        ctx.save_for_backward(x, codes, idx, loss, stats if stats is not None else torch.empty(0))
        ctx.fused, ctx.beta, ctx.cw, ctx.rotation = fused, float(beta), float(cw), bool(rotation)
        return q, loss[0] * (ctx.cw * (1.0 + ctx.beta))

    @staticmethod
    def backward(ctx, grad_q, grad_loss):
        x, codes, idx, loss, stats = ctx.saved_tensors
        _, N, d = x.shape
        # no rows: the loss is the mean of an empty selection and reaches nothing (max(rows, 1) keeps 0 * inf away)
        rows = loss[1].clamp_min(1.0)
        gx = gc = None
        if ctx.needs_input_grad[1] and grad_loss is not None:
            if not ctx.fused:
                stats = ops.ema_reduce(x, idx, None, codes.shape[1])
            gc = _codebook_grad(grad_loss, ctx.cw, rows, stats, codes)
        if ctx.needs_input_grad[0]:
            grad_q = torch.zeros_like(x, dtype=torch.float32) if grad_q is None else grad_q.contiguous().float()
            if grad_loss is None and not ctx.rotation:
                gx = grad_q
            else:
                g = (grad_loss.float() * (2.0 * ctx.cw * ctx.beta / d) / rows).reshape(1).contiguous() \
                    if grad_loss is not None else torch.zeros(1, dtype=torch.float32, device=x.device)
                gx = (ops.rot_commit_backward if ctx.rotation else ops.st_commit_backward)(grad_q, g, x, codes, idx,
                                                                                             None)
            gx = gx.to(x.dtype)
        return gx, gc, None, None, None, None, None, None


class SimVQ(nn.Module):
    """SimVQ (arXiv:2411.02038): the codebook is `code_transform(frozen_codebook)`, searched by Euclidean distance.

    `frozen_codebook` (K, d_f) is `init_fn(randn(K, d_f) * d_f ** -0.5)`, drawn on the CPU generator so that
    data-parallel ranks seeded alike agree; `code_transform` defaults to `nn.Linear(d_f, dim, bias=False)`.
    `forward(x)` takes (b, n, dim), or (b, dim, ...) with `channel_first`, in fp32, bf16 or fp16, and returns
    (quantized fp32, indices, loss); see the module docstring for the loss and its gradients.  In eval mode, or when
    nothing needs a gradient, the forward is the search and one gather pass."""

    def __init__(self, dim, codebook_size, codebook_transform=None, init_fn=_identity, channel_first=False,
                 rotation_trick=True, input_to_quantize_commit_loss_weight=0.25, commitment_weight=1.0,
                 frozen_codebook_dim=None):
        super().__init__()
        self.dim = dim
        self.codebook_size = codebook_size
        self.channel_first = channel_first
        self.rotation_trick = rotation_trick
        self.input_to_quantize_commit_loss_weight = input_to_quantize_commit_loss_weight
        self.commitment_weight = commitment_weight
        d_f = frozen_codebook_dim or dim
        codes = torch.randn(codebook_size, d_f, device="cpu") * d_f ** -0.5
        self.register_buffer("frozen_codebook", init_fn(codes))
        self.code_transform = codebook_transform if codebook_transform is not None else nn.Linear(d_f, dim, bias=False)

    @property
    def codebook(self):
        """C' = code_transform(frozen_codebook), (K, dim) fp32, differentiable with respect to the transform."""
        return self.code_transform(self.frozen_codebook).float()

    def _rows(self, x):
        """x -> (1, N, dim) rows and the leading shape to restore."""
        if self.channel_first:
            x = x.movedim(1, -1)
        if x.shape[-1] != self.dim:
            raise ValueError(f"vqb200.SimVQ: input has {x.shape[-1]} features, expected dim={self.dim}")
        return _lib.aligned(x.reshape(1, -1, self.dim)), tuple(x.shape[:-1])

    def _unrows(self, t, lead):
        t = t.reshape(*lead, t.shape[-1])
        return t.movedim(-1, 1) if self.channel_first else t

    def indices_to_codes(self, indices):
        codes = self.codebook[indices]
        return codes.movedim(-1, 1) if self.channel_first else codes

    def get_output_from_indices(self, indices):
        return self.indices_to_codes(indices)

    @torch.amp.autocast(device_type="cuda", enabled=False)
    def forward(self, x):
        flat, lead = self._rows(x)
        codebook = self.codebook
        codes = codebook.detach().contiguous()[None]
        cache = ops.prepare_codebook(codes, False)
        idx, _, ws = ops.search(flat, codes, cache, False)
        cw, beta = self.commitment_weight, self.input_to_quantize_commit_loss_weight
        if self.training and torch.is_grad_enabled() and (flat.requires_grad or codebook.requires_grad):
            q, loss = _SimVQQuantize.apply(flat, codebook, codes, idx, ws, beta, cw, self.rotation_trick)
        else:
            with torch.no_grad():
                q, loss_buf = ops.gather_st_loss(flat, codes, idx, None, True, True)
                loss = loss_buf[0] * (float(cw) * (1.0 + float(beta)))
        return self._unrows(q, lead), idx.reshape(lead), loss


class ResidualSimVQ(nn.Module):
    """`num_quantizers` SimVQ levels, each with its own frozen codebook and transform, in the residual loop of
    ResidualVQ: r_{l+1} = r_l - quantized_l.detach(), output = sum of the levels' outputs.  Returns
    (quantized_out, indices (b, n, Q), losses (1, Q)).

    Two implementations with the same forward values: the fused loop (CUDA input, at least two levels, a width the
    level kernels take) builds every C'_l and its search cache first, so each level pass also prepares the next level's
    search operand (`vqb_rvq_level_ema`), replays the output once (`vqb_rvq_replay_out`), and backward is one pass
    over the input (`vqb_rvq_backward[_rot]`) plus the codebook gradients from the saved per-code sums; the generic
    loop calls the SimVQ levels one after the other."""

    def __init__(self, dim, num_quantizers, codebook_size, rotation_trick=True, **simvq_kwargs):
        super().__init__()
        self.dim = dim
        self.num_quantizers = num_quantizers
        self.channel_first = simvq_kwargs.pop("channel_first", False)
        self.layers = nn.ModuleList([SimVQ(dim, codebook_size, rotation_trick=rotation_trick, **simvq_kwargs)
                                     for _ in range(num_quantizers)])
        self.use_fused_levels = True

    @property
    def codebooks(self):
        return torch.stack([layer.codebook for layer in self.layers], dim=0)

    def get_codes_from_indices(self, indices):
        """indices (..., Q) -> codes (Q, ..., dim) in the channel-last layout."""
        return torch.stack([layer.codebook[indices[..., l]] for l, layer in enumerate(self.layers)], dim=0)

    def get_output_from_indices(self, indices):
        out = self.get_codes_from_indices(indices).sum(dim=0)
        return out.movedim(-1, 1) if self.channel_first else out

    def _can_fuse(self, x) -> bool:
        Q, d = len(self.layers), self.dim
        return bool(self.use_fused_levels and x.is_cuda and Q >= 2 and ops.rvq_level_ema_supported(d)
                    and ops.rvq_replay_out_supported(d, Q) and len({l.rotation_trick for l in self.layers}) == 1)

    @torch.amp.autocast(device_type="cuda", enabled=False)
    def forward(self, x):
        if self.channel_first:
            x = x.movedim(1, -1)
        if x.shape[-1] != self.dim:
            raise ValueError(f"vqb200.ResidualSimVQ: input has {x.shape[-1]} features, expected dim={self.dim}")
        lead = tuple(x.shape[:-1])
        if self._can_fuse(x):
            books = [layer.codebook for layer in self.layers]
            flat = x.reshape(-1, self.dim)
            train = self.training and torch.is_grad_enabled() and (flat.requires_grad or
                                                                    any(b.requires_grad for b in books))
            if train:
                out, idx, losses = _FusedResidualSimVQ.apply(flat, self, *books)
            else:
                with torch.no_grad():
                    out, idx, losses, _ = _fused_levels(self.layers, flat, books, False)
            out = out.reshape(*lead, self.dim)
            indices = idx.t().reshape(*lead, len(self.layers))
            losses = losses.reshape(1, -1)
        else:
            out, residual, all_idx, all_loss = 0.0, x, [], []
            for layer in self.layers:
                quantized, idx, loss = layer(residual)
                residual = residual - quantized.detach()
                out = out + quantized
                all_idx.append(idx)
                all_loss.append(loss.reshape(1))
            indices = torch.stack(all_idx, dim=-1)
            losses = torch.stack(all_loss, dim=-1)
        if self.channel_first:
            out = out.movedim(-1, 1)
        return out, indices, losses


@torch.no_grad()
def _fused_levels(layers, x, books, keep_sums):
    """The fused level loop on x (N,d): returns (output (N,d) fp32, indices (Q,N), losses (Q,) and, with `keep_sums`,
    each level's (codebook (1,K,d), per-code sums (1,K,d+1), loss buffer) for backward)."""
    N, d = x.shape
    x0 = _lib.aligned(x.float())            # level 0 reads the input itself: every level writes another buffer
    codes = [b.detach().contiguous()[None] for b in books]
    # all caches first: the pass of level l prepares level l+1's search operand against its cache
    caches = [ops.prepare_codebook(c, False) for c in codes]
    bufs = [torch.empty((N, d), dtype=torch.float32, device=x.device) for _ in range(2)]
    Q = len(layers)
    idxs, losses, saved = [], [], []
    prepared = False
    for l, layer in enumerate(layers):
        cur = x0 if l == 0 else bufs[(l - 1) % 2]
        nxt = bufs[l % 2]
        idx, _, ws = ops.search(cur[None], codes[l], caches[l], False, latents_prepared=prepared)
        next_cache = caches[l + 1] if l + 1 < Q else None
        if keep_sums:
            loss_buf, stats = ops.rvq_level_ema(cur, nxt, codes[l][0], idx[0], True, l == 0, None, next_cache,
                                                bound_ws=ws)
            saved.append((codes[l], stats, loss_buf))
        else:
            loss_buf = ops.rvq_level(cur, nxt, codes[l][0], idx[0], None, True, l == 0, None, next_cache)
        prepared = next_cache is not None
        cw, beta = float(layer.commitment_weight), float(layer.input_to_quantize_commit_loss_weight)
        idxs.append(idx[0])
        losses.append(loss_buf[0] * (cw * (1.0 + beta)))
    out = ops.rvq_replay_out(x0, [c[0] for c in codes], idxs, [True] * Q, None)
    return out, torch.stack(idxs, 0), torch.stack(losses, 0), (x0, saved)


class _FusedResidualSimVQ(torch.autograd.Function):
    """The fused level loop with gradients.  d out / d x = Q I under straight-through (every level's output is
    r_l + (q_l - r_l).detach() and the residual subtracts a detached quantity), sum_l T_l under the rotation trick, and
    level l's loss adds g_l cw_l beta_l 2 (r_l - c_l) / (N d): one replay pass (`vqb_rvq_backward[_rot]`) with
    coef_l = g_l cw_l beta_l 2 / (N d).  C'_l gets g_l cw_l 2 (n_k C'_l[k] - S_k) / (N d) from the sums of its pass.
    The C'_l are fresh tensors of this forward, so nothing is copied for backward."""

    @staticmethod
    def forward(ctx, x, rsim, *books):
        out, idx, losses, (x0, saved) = _fused_levels(rsim.layers, x, books, True)
        ctx.x0, ctx.saved, ctx.idx, ctx.dtype = x0, saved, idx, x.dtype
        ctx.rotation = bool(rsim.layers[0].rotation_trick)
        ctx.weights = [(float(l.commitment_weight), float(l.input_to_quantize_commit_loss_weight)) for l in rsim.layers]
        ctx.mark_non_differentiable(idx)
        return out, idx, losses

    @staticmethod
    def backward(ctx, g_out, _g_idx, g_losses):
        x0, saved = ctx.x0, ctx.saved
        d = x0.shape[1]
        Q = len(saved)
        rows = [lb[1].clamp_min(1.0) for _, _, lb in saved]
        gx = None
        if ctx.needs_input_grad[0]:
            if g_losses is None:
                coef = torch.zeros(Q, dtype=torch.float32, device=x0.device)
            else:
                coef = torch.stack([g_losses[l].float() * (2.0 * cw * beta / d) / rows[l]
                                    for l, (cw, beta) in enumerate(ctx.weights)])
            backward = ops.rvq_backward_rot if ctx.rotation else ops.rvq_backward
            gx = backward(x0, [c[0] for c, _, _ in saved], list(ctx.idx), [True] * Q, coef, g_out, None)
            gx = gx.to(ctx.dtype)
        gbooks = [None] * Q
        if g_losses is not None:
            for l, ((codes, stats, _), (cw, _)) in enumerate(zip(saved, ctx.weights)):
                if ctx.needs_input_grad[2 + l]:
                    gbooks[l] = _codebook_grad(g_losses[l], cw, rows[l], stats, codes)
        return (gx, None, *gbooks)
