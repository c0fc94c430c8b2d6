"""``VectorQuantize``: drop-in for reference vector_quantization/vector_quantize_pytorch.py:38-430.

Same constructor arguments and ``forward`` returns.  The layout glue (channel-first, images/video,
multi-head, projections, masks) is host code; search, gather + straight-through + commitment loss
and the EMA update are CUDA kernels behind ``Codebook``.  The consumers of the dense N x K similarity
matrix -- cross-entropy to given indices (reference :284-299), the cross-entropy commitment loss (:338-346)
and the codebook diversity loss (:324-333) -- run as fp32 online-softmax passes that never write the
matrix (csrc/dense.cu), forward, input gradient and -- with a learnable codebook -- codebook gradient.
A learnable codebook (`learnable_codebook=True, ema_update=False`, optionally `sync_update_v` and
`in_place_codebook_optimizer`) is supported, and so is the orthogonal regularisation of the codebook (reference
:366-390, utils/losses.py:22-27; the reference reads the non-existent `_codebook.embed` there and raises
AttributeError -- implemented on `embeddings`, as SURVEY 8(b) prescribes).
"""
from __future__ import annotations

from collections import namedtuple
from dataclasses import asdict, replace

import torch
import torch.distributed as dist
from torch import nn

from . import ops
from .codebook import Codebook
from .params import CodebookParams

LossBreakdown = namedtuple("LossBreakdown", ["commitment", "codebook_diversity", "orthogonal_reg", "inplace_optimize"])


def _is_distributed() -> bool:
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


class VectorQuantize(nn.Module):
    def __init__(self, dim, codebook_params: CodebookParams, codebook_dim=None, heads=1,
                 separate_codebook_per_head=False, layernorm_after_project_in=False, channel_last=True,
                 commitment_weight=1.0, commitment_use_cross_entropy_loss=False, orthogonal_reg_weight=0.0,
                 orthogonal_reg_active_codes_only=False, orthogonal_reg_max_codes=None,
                 codebook_diversity_loss_weight=0.0, codebook_diversity_temperature=100.0, sync_codebook=None,
                 in_place_codebook_optimizer=None, sync_update_v=0.0):
        super().__init__()
        self.dim = dim
        self.heads = heads
        self.separate_codebook_per_head = separate_codebook_per_head
        codebook_dim = codebook_dim if codebook_dim is not None else dim
        codebook_input_dim = codebook_dim * heads
        requires_projection = codebook_input_dim != dim

        if requires_projection and layernorm_after_project_in:
            self.project_in = nn.Sequential(nn.Linear(dim, codebook_input_dim), nn.LayerNorm(codebook_input_dim))
        elif requires_projection:
            self.project_in = nn.Linear(dim, codebook_input_dim)
        else:
            self.project_in = nn.Identity()
        self.project_out = nn.Linear(codebook_input_dim, dim) if requires_projection else nn.Identity()
        self.has_projections = requires_projection

        self.has_commitment_loss = commitment_weight > 0.0
        self.commitment_weight = commitment_weight

        self.commitment_use_cross_entropy_loss = commitment_use_cross_entropy_loss
        self.codebook_diversity_loss_weight = codebook_diversity_loss_weight
        self.codebook_diversity_temperature = codebook_diversity_temperature
        self.has_codebook_diversity_loss = codebook_diversity_loss_weight > 0.0

        has_codebook_orthogonal_loss = orthogonal_reg_weight > 0.0
        self.has_codebook_orthogonal_loss = has_codebook_orthogonal_loss
        self.orthogonal_reg_weight = orthogonal_reg_weight
        self.orthogonal_reg_active_codes_only = orthogonal_reg_active_codes_only
        self.orthogonal_reg_max_codes = orthogonal_reg_max_codes

        if sync_codebook is None:
            sync_codebook = _is_distributed()

        # reference :95-102: the orthogonal loss needs a gradient to the codebook, so it turns the codebook into a
        # Parameter even when `learnable_codebook` is off (the EMA update then still runs, through `.data`)
        self.codebook_params = replace(codebook_params, dim=codebook_dim,
                                       num_codebooks=heads if separate_codebook_per_head else 1,
                                       learnable_codebook=has_codebook_orthogonal_loss
                                       or codebook_params.learnable_codebook,
                                       use_ddp=sync_codebook)
        self.learnable_codebook = codebook_params.learnable_codebook
        assert not (codebook_params.ema_update and codebook_params.learnable_codebook), \
            "learnable codebook not compatible with EMA update"
        assert 0 <= sync_update_v <= 1.0
        assert not (sync_update_v > 0.0 and not codebook_params.learnable_codebook), "learnable codebook must be turned on"
        self.sync_update_v = sync_update_v
        # upstream vector-quantize-pytorch's `rotation_trick` option (arXiv:2410.06424): when set, the gradient reaches the
        # input through the rotation of x onto its code instead of the straight-through identity; the forward values do
        # not change.  An attribute, not a constructor argument, so that the constructor keeps the reference's
        # parameters exactly; `ResidualVQ(rotation_trick=...)` sets it on every level.
        self.rotation_trick = False
        kw = asdict(self.codebook_params)
        self._codebook = Codebook(**kw)
        # commit_quantize is detached unless VectorQuantize's OWN learnable_codebook is set (reference :262-268)
        self._codebook.commit_grad_to_codebook = bool(self.learnable_codebook)
        # reference :132-136: an optimizer factory over the codebook's parameters (needs a learnable codebook)
        self.in_place_codebook_optimizer = in_place_codebook_optimizer(self._codebook.parameters()) \
            if in_place_codebook_optimizer is not None else None
        self.channel_last = channel_last
        self.register_buffer("zero", torch.tensor(0.0), persistent=False)

    # reference :140-176 reads `_codebook.embed`, which does not exist there; implemented on `embeddings`
    # A sharded codebook (Codebook.sharded) reads and writes the full (K, d) codebook here: the getter all-gathers the
    # shards (a collective every rank must join when a shard changed since the last call), the setter keeps this
    # rank's rows of what it is given.
    @property
    def codebook(self):
        cb = self._codebook.full_codebook() if self._codebook.sharded else self._codebook.embeddings
        return cb if self.separate_codebook_per_head else cb[0]

    @codebook.setter
    def codebook(self, codes):
        if not self.separate_codebook_per_head:
            codes = codes[None]
        cb = self._codebook
        if cb.sharded:
            codes = codes[:, cb.shard_offset:cb.shard_offset + cb.shard_size]
        with torch.no_grad():
            cb.embeddings.copy_(codes)
        cb.invalidate_cache()

    def get_codes_from_indices(self, indices):
        cb = self.codebook
        if cb.ndim == 2:
            codes = cb[indices]
        else:
            b = indices.shape[0]
            h = indices.shape[-1]
            flat = indices.reshape(b, -1, h)                                   # b n h
            gathered = torch.stack([cb[i][flat[..., i]] for i in range(h)], dim=2)   # b n h d
            codes = gathered.reshape(b, flat.shape[1], -1).reshape(*indices.shape[:-1], -1)
        if not self.channel_last:
            codes = codes.movedim(-1, 1)
        return codes

    def get_output_from_indices(self, indices):
        return self.project_out(self.get_codes_from_indices(indices))

    @staticmethod
    def _draw_perm(n: int, device) -> torch.Tensor:
        # reference :384: torch.randperm(num_codes, device=device) on the global generator
        return torch.randperm(n, device=device)

    def _rows_of(self, t, B, multi):
        """(b, n[, h]) per-position integers -> the (H, N) row layout of the codebook's latents (reference
        vector_quantize_pytorch.py:217-219: "h b n d" / "1 (b h) n d")."""
        if not multi:
            return t.reshape(1, -1)
        t = t.reshape(B, -1, self.heads)
        if self.separate_codebook_per_head:
            return t.permute(2, 0, 1).reshape(self.heads, -1)
        return t.permute(0, 2, 1).reshape(1, -1)

    def _inplace_optimize(self, cb_in, mask, multi):
        """reference :233-256: one optimizer step on mse(codes, x.detach()) inside forward, before the pass whose
        results are returned.  Search and gather are the usual kernels; the codebook gradient is the segmented sum
        of `ops._GatherCodes`; the N x d mse on top is torch glue."""
        cb = self._codebook
        with torch.enable_grad():
            target = cb.transform_input(cb_in.detach())
            quant, _, _ = cb._run(target, mask, False, fuse_st=False, want_commit=False)
            if mask is not None:
                per = torch.nn.functional.mse_loss(quant, target.float(), reduction="none")
                m = mask
                if multi:      # "b n -> c (b h) n"
                    m = mask[None, :, None, :].expand(per.shape[0], mask.shape[0], per.shape[1] // mask.shape[0],
                                                      mask.shape[1]).reshape(per.shape[0], per.shape[1], mask.shape[1])
                else:
                    m = mask[None]
                loss = per[m].mean()
            else:
                loss = torch.nn.functional.mse_loss(quant, target.float())
            loss.backward()
        self.in_place_codebook_optimizer.step()
        self.in_place_codebook_optimizer.zero_grad()
        cb.invalidate_cache()
        return loss.detach()

    def forward(self, x, indices=None, mask=None, freeze_codebook=False, return_loss_breakdown=False):
        return_loss = indices is not None
        orig_input = x
        only_one = x.ndim == 2
        if only_one:
            assert mask is None
            x = x[:, None, :]
        heads, multi = self.heads, self.heads > 1
        B = x.shape[0]
        device = x.device

        if not self.channel_last:
            x = x.movedim(1, -1)
        spatial = None
        if x.ndim >= 4:
            spatial = tuple(x.shape[1:-1])
            x = x.reshape(B, -1, x.shape[-1])
        x = self.project_in(x)
        if multi:
            n, dh = x.shape[1], x.shape[-1] // heads
            xh = x.reshape(B, n, heads, dh)
            x = xh.permute(2, 0, 1, 3) if self.separate_codebook_per_head else \
                xh.permute(0, 2, 1, 3).reshape(1, B * heads, n, dh)
        cb_in = x if x.ndim == 4 else x[None]
        training = self.training
        ce_commit = training and self.has_commitment_loss and self.commitment_use_cross_entropy_loss
        want_commit = training and self.has_commitment_loss and not ce_commit
        diversity = training and self.has_codebook_diversity_loss
        keep_dense = return_loss or ce_commit or diversity
        inplace_loss = self.zero
        if self.in_place_codebook_optimizer is not None and training and not freeze_codebook:
            inplace_loss = self._inplace_optimize(cb_in, mask, multi)
        # transform_input (reference :221) happens inside _run, fused with the search's operand preparation
        # `rotation` is passed only when set, so a `_run` override without that keyword keeps working by default
        rot = {"rotation": True} if self.rotation_trick else {}
        quantize, embed_ind, commit = self._codebook._run(cb_in, mask, freeze_codebook, fuse_st=True,
                                                          want_commit=want_commit,
                                                          normalize_input=self._codebook.input_l2norm,
                                                          keep_dense=keep_dense, **rot)
        dense = self._codebook.dense_ctx
        self._codebook.dense_ctx = None
        # learnable codebook: the similarities stay attached to `embeddings` (reference codebooks.py:375-377, whatever
        # freeze_codebook says), so the dense losses also send a gradient to the codebook
        emb_param = self._codebook.embeddings if (self._codebook.learnable_codebook and torch.is_grad_enabled()
                                                  and self._codebook.embeddings.requires_grad) else None
        rows_idx = embed_ind.reshape(embed_ind.shape[0], -1)          # (H, N): the row layout of the dense passes
        if x.ndim < 4:
            quantize, embed_ind = quantize[0], embed_ind[0]
        if training and self.sync_update_v > 0.0:
            # reference :275-279: value unchanged, the gradient to the input is scaled by (1 + v)
            quantize = quantize + self.sync_update_v * (quantize - quantize.detach())

        if return_loss:
            # reference :284-299: F.cross_entropy(similarities, indices, ignore_index=-1); returns the codebook-side
            # quantize (before head merge / projection) and the loss only
            target = self._rows_of(indices.to(device=device, dtype=torch.int64), B, multi)
            return quantize, ops.dense_cross_entropy(dense, target, emb_param)

        commit_loss = diversity_loss = orthogonal_reg_loss = self.zero
        if multi:
            if self.separate_codebook_per_head:
                embed_ind = embed_ind.permute(1, 2, 0)
            else:
                embed_ind = embed_ind.reshape(B, heads, -1).permute(0, 2, 1)
        if spatial is not None:
            embed_ind = embed_ind.reshape(B, *spatial, *embed_ind.shape[2:])
        if only_one:
            embed_ind = embed_ind[:, 0]

        loss = torch.tensor([0.0], device=device, requires_grad=training)
        if diversity:
            # reference :324-333: softmax(-similarities * T) averaged over heads and batch ("... n l -> n l"),
            # then the negative entropy per position; the (n, K) entropy is torch glue on the kernel's output
            n_pos = cb_in.shape[-2]
            avg_prob = ops.dense_avg_prob(dense, n_pos, self.codebook_diversity_temperature, emb_param)
            diversity_loss = -((-avg_prob * avg_prob.clamp(min=1e-5).log()).sum(dim=-1)).mean()
            loss = loss + diversity_loss * self.codebook_diversity_loss_weight
        if ce_commit:
            # reference :338-346: cross-entropy of the similarities against the chosen codes; masked positions are
            # ignored AND the returned indices carry -1 there (masked_fill_ in place at :344)
            target = rows_idx
            if mask is not None:
                keep = self._codebook._expand_mask(mask, rows_idx.shape[1]).bool()
                target = torch.where(keep[None], rows_idx, torch.full_like(rows_idx, -1))
                m = mask.reshape(embed_ind.shape[:-1] if multi else embed_ind.shape)
                embed_ind = embed_ind.masked_fill(~(m[..., None] if multi else m), -1)
            commit_loss = ops.dense_cross_entropy(dense, target, emb_param)
            loss = loss + commit_loss * self.commitment_weight
        elif want_commit:
            commit_loss = commit
            loss = loss + commit_loss * self.commitment_weight
        if training and self.has_codebook_orthogonal_loss:
            # reference :366-390 on `embeddings` (K- or d-sized torch glue on the codebook, no latents involved)
            codebook = self._codebook.embeddings
            if self.orthogonal_reg_active_codes_only:
                assert not (multi and self.separate_codebook_per_head), \
                    "orthogonal regularization for only active codes not compatible with multi-headed with " \
                    "separate codebooks yet"
                codebook = codebook[:, torch.unique(embed_ind)]
            num_codes = codebook.shape[-2]
            if self.orthogonal_reg_max_codes is not None and num_codes > self.orthogonal_reg_max_codes:
                codebook = codebook[:, self._draw_perm(num_codes, device)[:self.orthogonal_reg_max_codes]]
            orthogonal_reg_loss = ops.orthogonal_loss(codebook)
            loss = loss + orthogonal_reg_loss * self.orthogonal_reg_weight

        if multi:
            if self.separate_codebook_per_head:
                quantize = quantize.permute(1, 2, 0, 3).reshape(B, quantize.shape[2], -1)
            else:
                n = quantize.shape[2]
                quantize = quantize.reshape(B, heads, n, -1).permute(0, 2, 1, 3).reshape(B, n, -1)
        quantize = self.project_out(quantize)
        if spatial is not None:
            quantize = quantize.reshape(B, *spatial, quantize.shape[-1])
        if not self.channel_last:
            quantize = quantize.movedim(-1, 1)
        if only_one:
            quantize = quantize[:, 0]
        if mask is not None:
            quantize = torch.where(mask[..., None], quantize, orig_input)

        if not return_loss_breakdown:
            return quantize, embed_ind, loss
        return quantize, embed_ind, loss, LossBreakdown(commit_loss, diversity_loss, orthogonal_reg_loss, inplace_loss)
