"""``Codebook``: drop-in for reference vector_quantization/codebooks.py:81-435 on the EMA path.

Same constructor, same persistent buffers (``embeddings`` (H,K,d), ``embed_avg`` (H,K,d),
``cluster_size`` (H,K), fp32) and the same ``forward(x, mask, freeze_codebook)`` contract;
the numeric work (search, gather, EMA statistics, refresh, expiry scatter) runs in
libvqb200.so.  ``learnable_codebook=True`` makes ``embeddings`` a Parameter that receives the gradient
of the commitment loss / of the gathered codes (a segmented sum over the rows of each code).

Variants off the named hot path run through the same `_run` with the fused passes off:
  * gumbel sampling (reference utils/general.py:107-151, codebooks.py:388): `stochastic` = argmax of
    similarities / temperature + gumbel noise as an epilogue of the tiled fp32 score pass (vqb_dense_gumbel_sample;
    the noise is generated in the kernel from torch's Philox stream, no N x K tensor exists);
    `straight_through` / `reinmax` change only the GRADIENT through the one-hot (their forward value is the hard
    one-hot to 2^-24), which the reference drops unless the codebook is learnable or `Codebook.forward` is used
    directly under autograd -- that corner runs the reference's formulas as row-chunked torch ops (library code, not
    kernels of this package);
  * affine re-parametrisation (codebooks.py:274-348,373-384,400-403): batch moments from one fp64 pass over the latents
    (vqb_column_moments), search / gather on the transformed codebook, EMA sums transformed per code instead of per row.
"""
from __future__ import annotations

from dataclasses import asdict, is_dataclass
from typing import Optional

import torch
import torch.distributed as dist
from torch import nn

from . import _lib, ops
from .params import GumbelParams, KmeansParameters


def _uniform_init(*shape):
    # reference utils/general.py:101-104
    t = torch.empty(shape)
    nn.init.kaiming_uniform_(t)
    return t


def _l2norm_cpu_or_cuda(t: torch.Tensor) -> torch.Tensor:
    # construction-time only (tiny, may be on CPU); the forward path uses the CUDA kernel
    return torch.nn.functional.normalize(t, p=2, dim=-1)


class Codebook(nn.Module):
    def __init__(self, dim, codebook_size, num_codebooks=1, initialization_by_kmeans: bool = False,
                 kmeans_params: KmeansParameters = None, decay: float = 0.8, eps_for_smoothing: float = 1e-5,
                 threshold_ema_dead_code: int = 2, reset_cluster_size: int = None, use_ddp: bool = False,
                 distributed_replace_codes: bool = True, learnable_codebook: bool = False,
                 gumbel_params: GumbelParams = GumbelParams(), ema_update: bool = True, use_affine: bool = False,
                 affine_params=None, transform_input: str = "identity", use_cosine_sim: bool = False,
                 weights_regularization: str = "identity"):
        super().__init__()
        for name, val in (("transform_input", transform_input), ("weights_regularization", weights_regularization)):
            if val not in ("identity", "l2norm"):
                # the reference does `raise f"..."` here (a TypeError); keep the intent, not the bug
                raise ValueError(f"The option {val} for {name} is not implemented")
        gp = asdict(gumbel_params) if is_dataclass(gumbel_params) else dict(gumbel_params)
        # reference codebooks.py:154-158: `sample_fn_training` (the only one forward() calls) = gumbel_sample(**params)
        self.gumbel = {"temperature": 1.0, "stochastic": False, "reinmax": False, "straight_through": False, "dim": -1,
                       "training": True, **gp}
        self._uniform_queue: list = []       # tests: the (H,N,K) draws a fixture was recorded with, in call order

        self.input_l2norm = transform_input == "l2norm"
        self.weights_l2norm = weights_regularization == "l2norm"
        self.use_cosine_sim = use_cosine_sim
        self.decay = decay
        self.ema_update = ema_update
        self.codebook_size = codebook_size
        self.num_codebooks = num_codebooks
        self.dim = dim
        self.kmeans_params = asdict(kmeans_params) if is_dataclass(kmeans_params) else kmeans_params
        self.eps_for_smoothing = eps_for_smoothing
        self.threshold_ema_dead_code = threshold_ema_dead_code
        self.reset_cluster_size = reset_cluster_size if reset_cluster_size is not None else threshold_ema_dead_code
        assert not (use_ddp and num_codebooks > 1 and initialization_by_kmeans), \
            "kmeans init is not compatible with multiple codebooks in distributed environment for now"
        self.use_ddp = use_ddp
        # the reference indexes kmeans_params["sync"] unconditionally and crashes when it is None
        # (codebooks.py:164-166); treat a missing KmeansParameters as its defaults instead
        self._kmeans_sync = bool((self.kmeans_params or {"sync": True})["sync"])
        self.distributed_replace_codes = distributed_replace_codes
        self.learnable_codebook = bool(learnable_codebook)
        # VectorQuantize clears this when ITS learnable_codebook is off while the codebook is a Parameter only because of
        # the orthogonal regularisation (reference vector_quantize_pytorch.py:99-104,262-268: commit_quantize is detached)
        self.commit_grad_to_codebook = True
        self.return_similarities = False       # opt in to the dense (H, ..., K) third return value of forward()
        self._sim: Optional[torch.Tensor] = None
        self.use_affine = bool(use_affine)
        if self.use_affine:
            if affine_params is None:
                raise ValueError("vqb200.Codebook: use_affine=True needs affine_params")
            self.affine_params = asdict(affine_params) if is_dataclass(affine_params) else dict(affine_params)

        init = torch.zeros(num_codebooks, codebook_size, dim) if initialization_by_kmeans else \
            _uniform_init(num_codebooks, codebook_size, dim)
        if self.weights_l2norm:
            init = _l2norm_cpu_or_cuda(init)

        # Sharded codebook (north star config 5; no reference counterpart): with >= SHARD_MIN_CODES codes, a process
        # group up and `use_ddp` set, rank r owns rows [r K/W, (r+1) K/W) of the three buffers.  Every rank draws the
        # same full initialisation (the ranks share the module seed, as replicated data parallel requires too) and
        # keeps its rows; `state_dict()` gathers the full (H,K,d) tensors under the reference's keys and
        # `load_state_dict()` takes this rank's rows of them (both collective-free on load, one all_gather on save).
        from . import distributed as D
        self.sharded = bool(use_ddp and D.is_distributed() and codebook_size >= D.SHARD_MIN_CODES
                            and codebook_size % D.world_size() == 0)
        self.shard_world = D.world_size() if self.sharded else 1
        self.shard_rank = D.rank() if self.sharded else 0
        self.shard_size = codebook_size // self.shard_world
        # "replicated": every rank passes the SAME latents (BASELINE config 5); "all_gather": every rank passes its own
        # batch and the ranks' batches are concatenated before the search (data parallel over a sharded codebook)
        self.sharded_input = "all_gather"
        self._replica: Optional[torch.Tensor] = None
        self._replica_dirty = True
        if self.sharded:
            if learnable_codebook or self.use_affine or any(self._variant_sampling()):
                raise NotImplementedError("vqb200: a sharded codebook (>= %d codes under a process group) is EMA-only "
                                          "with deterministic sampling and no affine re-parametrisation"
                                          % D.SHARD_MIN_CODES)
            lo = self.shard_rank * self.shard_size
            init = init[:, lo:lo + self.shard_size].contiguous()
            self._register_state_dict_hook(Codebook._gather_state_hook)
            self._register_load_state_dict_pre_hook(self._slice_state_pre_hook)
        self.is_initialized = not initialization_by_kmeans
        self.register_buffer("cluster_size", torch.zeros(num_codebooks, self.shard_size))
        self.register_buffer("embed_avg", init.clone())
        if self.learnable_codebook:          # reference codebooks.py:186-190: a Parameter, trained by the user's optimizer
            self.embeddings = nn.Parameter(init)
        else:
            self.register_buffer("embeddings", init)

        if self.use_affine:                    # reference codebooks.py:194-206, same buffer names
            self.register_buffer("batch_mean", None)
            self.register_buffer("batch_variance", None)
            self.register_buffer("codebook_mean_needs_init", torch.Tensor([True]))
            self.register_buffer("codebook_mean", torch.empty(num_codebooks, 1, dim))
            self.register_buffer("codebook_variance_needs_init", torch.Tensor([True]))
            self.register_buffer("codebook_variance", torch.empty(num_codebooks, 1, dim))

        # derived, non-persistent: scaled fp16 copy + norms for the tensor-core search
        self._cache: Optional[torch.Tensor] = None
        self._cache_key = None
        self._dirty = True
        self.dense_ctx = None
        self.last_search_ws: Optional[torch.Tensor] = None
        self.fused_quantize_ema = True     # False: separate gather and EMA-reduce passes (same results)

    # ------------------------------------------------------------------ transforms
    def transform_input(self, x: torch.Tensor) -> torch.Tensor:
        """reference: identity | l2norm (utils/losses.py:19), applied by VectorQuantize before the codebook."""
        if not self.input_l2norm:
            return x
        return ops.l2norm_rows(x.contiguous())

    # ------------------------------------------------------------------ cache
    def _codebook_cache(self) -> torch.Tensor:
        e = self.embeddings
        key = (e.data_ptr(), e._version, tuple(e.shape), self.use_cosine_sim)
        if self._dirty or self._cache is None or key != self._cache_key:
            self._cache = ops.prepare_codebook(e, self.use_cosine_sim, self._cache)
            self._cache_key = key
            self._dirty = False
        return self._cache

    def invalidate_cache(self) -> None:
        """Call after an in-place edit of `embeddings`: the search operands and, on a sharded codebook, the all-gathered
        replica the gather reads are rebuilt on next use."""
        self._dirty = self._replica_dirty = True

    # ------------------------------------------------------------------ helpers
    def _all_reduce(self, t: torch.Tensor) -> None:
        if self.use_ddp and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(t)

    @staticmethod
    def _draw_rows(num_rows: int, m: int, device) -> torch.Tensor:
        # reference utils/general.py:62-66 -- same calls on the same (global) generator
        if num_rows >= m:
            return torch.randperm(num_rows, device=device)[:m]
        return torch.randint(0, num_rows, (m,), device=device)

    def _flatten(self, x: torch.Tensor):
        """(H, ..., d) -> contiguous (H, N, d) in a kernel dtype; also returns the leading shape."""
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        H, d = x.shape[0], x.shape[-1]
        lead = tuple(x.shape[1:-1])
        return _lib.aligned(x.reshape(H, -1, d)), lead

    def _expand_mask(self, mask: Optional[torch.Tensor], n_rows: int) -> Optional[torch.Tensor]:
        # reference codebooks.py:361-367: repeat(mask, "b n -> c (b h n)")
        if mask is None:
            return None
        b, n = mask.shape
        rep = n_rows // (b * n)
        m = mask[:, None, :].expand(b, rep, n).reshape(-1)
        return m.to(torch.uint8).contiguous()

    # ------------------------------------------------------------------ kmeans init (reference utils/kmeans.py)
    @torch.no_grad()
    def _kmeans_init(self, flat: torch.Tensor, mask_u8: Optional[torch.Tensor]) -> None:
        """reference utils/kmeans.py:38-120.  On a sharded codebook rank 0's draw picks the K start rows (all ranks hold
        the same latents) and every iteration is a sharded search + segment means on the owned rows."""
        from . import distributed as D
        H, N, d = flat.shape
        K = self.codebook_size
        data = flat.float()
        if mask_u8 is not None:
            data = data[:, mask_u8.bool()].contiguous()
            N = data.shape[1]
        iters = int((self.kmeans_params or {"iter": 10})["iter"])
        sync = self.use_ddp and self._kmeans_sync and not self.sharded
        if self.sharded:
            lo, Ks = self.shard_offset, self.shard_size
            cents = [data[h][D.broadcast_from_rank0(self._draw_rows(N, K, data.device).to(torch.long))[lo:lo + Ks]]
                     for h in range(H)]
        elif sync and D.is_distributed():    # reference codebooks.py:164-168: identical centroids on every rank
            cents = [D.sample_vectors_distributed(data[h], K, self._draw_rows) for h in range(H)]
        else:
            cents = [data[h][self._draw_rows(N, K, data.device)] for h in range(H)]
        cents = torch.stack(cents, 0).contiguous()
        counts = torch.zeros(H, self.shard_size, device=data.device)
        for _ in range(iters):
            cache = ops.prepare_codebook(cents, self.use_cosine_sim)
            if self.sharded:
                stats = self._shard_stats(data, self._shard_search(data, cents, cache), None)
            else:
                idx, _, ws = ops.search(data, cents, cache, self.use_cosine_sim)
                stats = ops.ema_reduce(data, idx, None, K, bound_ws=ws)
            counts = stats[..., d].clone()
            if sync:
                self._all_reduce(counts)
            empty = counts == 0
            means = stats[..., :d] / counts.masked_fill(empty, 1.0)[..., None]
            if sync:
                means = means.contiguous()
                self._all_reduce(means)
            if self.use_cosine_sim:
                means = ops.l2norm_rows(means.contiguous())
            cents = torch.where(empty[..., None], cents, means).contiguous()
        self.embeddings.data.copy_(cents)
        self.embed_avg.data.copy_(cents * counts[..., None])
        self.cluster_size.data.copy_(counts)
        self._dirty = self._replica_dirty = True

    # ------------------------------------------------------------------ EMA refresh
    def _apply_ema(self, stats: torch.Tensor) -> None:
        """Refresh the buffers from one step's statistics (H, K, d+1), already all-reduced under data parallel; on a
        shard, the statistics of this rank's codes.  No host sync: ResidualVQ's fused level loop calls this inside a
        CUDA graph."""
        if self.sharded:
            from . import distributed as D
            ops.ema_apply_sharded(stats, self.cluster_size.data, self.embed_avg.data, self.embeddings.data,
                                  1 - self.decay, self.eps_for_smoothing, self.weights_l2norm, self.codebook_size,
                                  D.all_reduce_sum)
            self._replica_dirty = True
        else:
            ops.ema_apply(stats, self.cluster_size.data, self.embed_avg.data, self.embeddings.data, 1 - self.decay,
                          self.eps_for_smoothing, self.weights_l2norm)
        self._dirty = True

    # ------------------------------------------------------------------ expiry (reference codebooks.py:230-255)
    @torch.no_grad()
    def expire_codes_(self, flat: torch.Tensor) -> None:
        if self.threshold_ema_dead_code == 0:
            return
        dead = self.cluster_size < self.threshold_ema_dead_code
        # ONE host sync: the per-codebook counts (the reference syncs twice: torch.any at :251, .item() at :234)
        counts = dead.sum(dim=-1).tolist()
        if not any(counts):
            return
        H, N, d = flat.shape
        from . import distributed as D
        synced = self.use_ddp and self._kmeans_sync and self.distributed_replace_codes and D.is_distributed()
        for h in range(H):
            m = int(counts[h])
            if synced:
                # reference codebooks.py:171-175: sample_vectors_distributed -> identical replacements on every rank
                src = D.sample_vectors_distributed(flat[h], m, self._draw_rows)
                rows = torch.arange(m, device=flat.device)
            elif not self.distributed_replace_codes and D.is_distributed():
                # reference codebooks.py:231-239: every rank samples locally (after weights_regularization) and the
                # replacements are the mean over the ranks (not re-normalised)
                src = flat[h][self._draw_rows(N, m, flat.device)].float().contiguous()
                if self.weights_l2norm:
                    src = ops.l2norm_rows(src)
                src = D.maybe_distributed_mean(src)
                ops.expire_scatter(src, torch.arange(m, device=flat.device), float(self.threshold_ema_dead_code),
                                   float(self.reset_cluster_size), False, self.cluster_size.data[h],
                                   self.embed_avg.data[h], self.embeddings.data[h])
                continue
            else:
                src, rows = flat[h], self._draw_rows(N, m, flat.device)
            ops.expire_scatter(src, rows, float(self.threshold_ema_dead_code), float(self.reset_cluster_size),
                               self.weights_l2norm, self.cluster_size.data[h], self.embed_avg.data[h],
                               self.embeddings.data[h])
        self._dirty = True

    # ------------------------------------------------------------------ sharded codebook (config 5)
    @property
    def shard_offset(self) -> int:
        return self.shard_rank * self.shard_size

    @staticmethod
    def _gather_state_hook(module, state_dict, prefix, local_metadata):
        from . import distributed as D
        for name in ("embeddings", "embed_avg", "cluster_size"):
            state_dict[prefix + name] = D.all_gather_codes(getattr(module, name).detach(), dim=1)

    def _slice_state_pre_hook(self, state_dict, prefix, *args):
        lo = self.shard_offset
        for name in ("embeddings", "embed_avg", "cluster_size"):
            t = state_dict.get(prefix + name)
            if t is not None and t.shape[1] == self.codebook_size:
                state_dict[prefix + name] = t[:, lo:lo + self.shard_size]
        self._dirty = self._replica_dirty = True

    def load_full_codebook(self, full: torch.Tensor, cluster_size: float = 1.0) -> None:
        """(H,K,d) or (K,d) codebook -> this rank's rows (or all of them when not sharded); embed_avg = embeddings."""
        full = full if full.ndim == 3 else full[None]
        lo = self.shard_offset
        rows = full[:, lo:lo + self.shard_size].to(self.embeddings.device, torch.float32)
        with torch.no_grad():
            self.embeddings.copy_(rows); self.embed_avg.copy_(rows); self.cluster_size.fill_(cluster_size)
        self._dirty = self._replica_dirty = True

    def full_codebook(self) -> torch.Tensor:
        """(H,K,d) replica of the sharded `embeddings` (one all_gather when a shard changed since the last call)."""
        if not self.sharded:
            return self.embeddings.detach()
        if self._replica_dirty or self._replica is None:
            from . import distributed as D
            self._replica = D.all_gather_codes(self.embeddings.detach(), dim=1, out=self._replica)
            self._replica_dirty = False
        return self._replica

    def _shard_search(self, flat: torch.Tensor, emb: torch.Tensor, cache) -> torch.Tensor:
        """Global nearest code of every row: local shard search -> (fp32 score of the reference recipe, global index)
        packed into int64 keys -> all_reduce(MIN): smallest score, lowest index on ties = torch.argmax on the
        un-sharded similarities.  Every rank evaluates the score with the same fp64-accumulated recipe, so the
        cross-shard comparison is consistent."""
        from . import distributed as D
        H, N, _ = flat.shape
        idx, score, ws = ops.search(flat, emb, cache, self.use_cosine_sim, idx_offset=self.shard_offset,
                                    want_score=True)
        self.last_search_ws = ws
        keys = ops.minkey_pack(score.reshape(-1), idx.reshape(-1))
        D.merge_min_keys(keys)
        gidx, _ = ops.minkey_unpack(keys)
        return gidx.reshape(H, N)

    def _shard_stats(self, rows: torch.Tensor, gidx: torch.Tensor, mask_u8: Optional[torch.Tensor]) -> torch.Tensor:
        """EMA statistics (H, K/W, d+1) of this rank's codes: the sums over the rows whose global code id is one of
        them."""
        lo, Ks = self.shard_offset, self.shard_size
        mine = (gidx >= lo) & (gidx < lo + Ks)
        if mask_u8 is not None:
            mine = mine & mask_u8.bool()[None]
        return torch.stack([ops.ema_reduce(rows[h:h + 1], (gidx[h:h + 1] - lo).clamp_(0, Ks - 1),
                                           mine[h].to(torch.uint8), Ks)[0] for h in range(rows.shape[0])], 0)

    @torch.no_grad()
    def _expire_codes_sharded(self, flat: torch.Tensor) -> None:
        """reference codebooks.py:230-255 on shards: the dead codes of all shards, in ascending GLOBAL code order, take
        the rows rank 0 draws with the reference's calls (utils/general.py:62-66) -- exactly what one process does on
        the un-sharded codebook with rank 0's generator.  One all_gather of the per-shard dead counts (the host sync
        the reference has too) and one broadcast of the drawn row ids."""
        if self.threshold_ema_dead_code == 0:
            return
        from . import distributed as D
        H, N, d = flat.shape
        dead = self.cluster_size < self.threshold_ema_dead_code
        counts = D.all_gather_small(dead.sum(dim=-1))                  # (W, H) on the host
        if int(counts.sum()) == 0:
            return
        for h in range(H):
            m_total = int(counts[:, h].sum())
            if m_total == 0:
                continue
            rows = D.broadcast_from_rank0(self._draw_rows(N, m_total, flat.device).to(torch.long))
            first = int(counts[:self.shard_rank, h].sum())
            m = int(counts[self.shard_rank, h])
            if m:
                ops.expire_scatter(flat[h], rows[first:first + m], float(self.threshold_ema_dead_code),
                                   float(self.reset_cluster_size), self.weights_l2norm, self.cluster_size.data[h],
                                   self.embed_avg.data[h], self.embeddings.data[h])
        self._dirty = self._replica_dirty = True

    # ------------------------------------------------------------------ variants: gumbel sampling, affine
    def _variant_sampling(self):
        """(stochastic, straight_through) as reference gumbel_sample applies them (utils/general.py:121-137)."""
        g = self.gumbel
        active = bool(g["training"]) and g["temperature"] > 0
        return (active and bool(g["stochastic"])), (active and bool(g["straight_through"]))

    def _variants_active(self) -> bool:
        stochastic, st = self._variant_sampling()
        return self.use_affine or stochastic or st

    def _update_with_decay(self, name: str, new_value: torch.Tensor, decay: float) -> None:
        # reference codebooks.py:258-272
        old = getattr(self, name)
        needs_init = getattr(self, name + "_needs_init", None)
        first = needs_init is not None and bool(needs_init.item())
        if first:
            needs_init.fill_(0.0)
        if old is None or first:
            setattr(self, name, new_value.detach().clone())
            return
        setattr(self, name, old * decay + new_value.detach() * (1 - decay))

    @torch.no_grad()
    def _update_affine(self, flat: torch.Tensor, mask_u8: Optional[torch.Tensor]) -> None:
        """reference codebooks.py:274-348.  The batch moments come from ONE fp64 pass over the latents; with
        `affine_params.sync` the per-rank sums are all-reduced (mean and variance of the union of the batches, as the
        reference's three all_reduce calls compute)."""
        ap = self.affine_params
        emb = self.embeddings.detach()
        if self.training:
            self._update_with_decay("codebook_mean", emb.mean(dim=1, keepdim=True), ap["codebook_decay"])
            self._update_with_decay("codebook_variance", emb.var(dim=1, unbiased=False, keepdim=True),
                                    ap["codebook_decay"])
        sums, rows = ops.column_moments(flat.detach(), mask_u8)
        if ap["sync"]:
            from . import distributed as D
            packed = torch.cat([sums.reshape(-1), rows.double()])
            D.all_reduce_sum(packed)
            sums, rows = packed[:sums.numel()].reshape(sums.shape), packed[sums.numel():]
        n = rows.double()[:, None]
        mean = sums[..., 0] / n
        var = (sums[..., 1] / n - mean * mean).clamp_min(0.0)
        self._update_with_decay("batch_mean", mean.float()[:, None, :], ap["batch_decay"])
        self._update_with_decay("batch_variance", var.float()[:, None, :], ap["batch_decay"])

    def _gumbel_st_quantize(self, flat: torch.Tensor, emb_g: torch.Tensor, idx: torch.Tensor,
                            mask_u8: Optional[torch.Tensor], fuse_st: bool, want_commit: bool, rotation: bool):
        """quantize = one_hot' @ embeddings with the straight-through / reinmax one-hot of reference
        utils/general.py:139-149, as torch ops under autograd (library code): only the gradient through the one-hot
        differs from a gather.  Row-chunked (bounds the size of each temporary, not the total the graph keeps);
        `reinmax` cannot be chunked because the reference normalises `prob1` over dim=1 -- the ROW axis of (h, n, c) --
        which couples all rows.  No recomputation in backward: with an EMA codebook `emb_g` aliases the live buffer,
        which this forward's EMA step overwrites in place before backward runs -- the reference's graph has exactly that
        aliasing (its saved `embeddings.detach()` shares the buffer's storage, codebooks.py:375-377,425), so the same
        torch ops on the same alias reproduce its gradient: pre-update distances and probabilities, post-update code
        vectors.  Returns (quantize, commit | None); with `fuse_st`, VectorQuantize's straight-through output."""
        import torch.nn.functional as F
        g = self.gumbel
        tau, K, cos = float(g["temperature"]), emb_g.shape[1], self.use_cosine_sim

        def log_eps(t):
            return t.clamp(min=1e-5).log()

        def piece(xc, e, ic):
            xc = xc.float()
            logits = torch.einsum("hnd,hcd->hnc", xc, e) if cos else -torch.cdist(xc, e)
            one_hot = F.one_hot(ic, K).type(logits.dtype)
            if g["reinmax"]:
                prob0 = logits.softmax(dim=-1)
                prob1 = (one_hot + (logits / tau).softmax(dim=-1)) / 2
                prob1 = ((log_eps(prob1) - logits).detach() + logits).softmax(dim=1)
                prob2 = 2 * prob1 - 0.5 * prob0
                one_hot = prob2 - prob2.detach() + one_hot
            else:
                prob1 = (logits / tau).softmax(dim=-1)
                one_hot = one_hot + prob1 - prob1.detach()
            return torch.einsum("hnc,hcd->hnd", one_hot, e)

        H, N = idx.shape
        rows = N if g["reinmax"] else max(1, (1 << 24) // max(K, 1))
        if rows >= N:
            q_graph = piece(flat, emb_g, idx)
        else:
            q_graph = torch.cat([piece(flat[:, lo:lo + rows], emb_g, idx[:, lo:lo + rows]) for lo in range(0, N, rows)],
                                dim=1)
        if not fuse_st:
            return q_graph, None
        # reference vector_quantize_pytorch.py:262-273,335-362 with commit_quantize attached
        xf = flat.float()
        commit = None
        if want_commit:
            per = (q_graph - xf) ** 2
            commit = per[:, mask_u8.bool()].mean() if mask_u8 is not None else per.mean()
        if not rotation:
            return xf + (q_graph - xf).detach(), commit
        # the rotation-trick gradient towards c = q_graph (a detached (H,N,d) "codebook" gathered row by row): same
        # forward value fl(x + fl(c - x)), same op as the gather path of `_run`
        c = q_graph.detach().contiguous()
        rows = torch.arange(N, device=c.device).expand(H, N).contiguous()
        quant, _, _ = ops.quantize_training(xf, c, rows, mask_u8, False, rotation=True)
        return quant, commit

    # ------------------------------------------------------------------ core
    def _run(self, x: torch.Tensor, mask: Optional[torch.Tensor], freeze_codebook: bool, fuse_st: bool,
             want_commit: bool, normalize_input: bool = False, keep_dense: bool = False, rotation: bool = False):
        """Shared by forward() and VectorQuantize.  x: (H, ..., d).  Returns (quantize (H,...,d), idx (H,...),
        commit scalar | None).  `keep_dense`: leave in `self.dense_ctx` what the consumers of the dense similarities
        (cross-entropy to indices, CE commitment, diversity loss) need: the (H,N,d) latents the search saw and the
        codebook as it was BEFORE this forward's EMA step (reference codebooks.py:386 runs before :425).
        `rotation`: where `fuse_st` applies the straight-through estimator, use the rotation-trick gradient instead
        (`VectorQuantize.rotation_trick`; the returned values do not change).

        One sequence for every configuration; the variants (gumbel sampling, affine; see the module docstring) and the
        sharded codebook differ from the plain EMA path only where noted.  A shard ends up with the quantised vectors /
        indices of ITS latents (all of them when the input is replicated) and updates ITS rows of the EMA buffers from
        the rows they won -- no statistics all_reduce; its exchanges are the min-key all_reduce of the search, one
        scalar all_reduce in the refresh and the all_gather of the codebook replica the gather reads."""
        if self.sharded and keep_dense:
            raise NotImplementedError("vqb200: the dense-similarity losses are not available on a sharded codebook")
        g = self.gumbel
        variants = not self.sharded and self._variants_active()
        stochastic, st = self._variant_sampling() if variants else (False, False)
        assert not (variants and g["reinmax"] and not g["straight_through"]), \
            "reinmax can only be turned on if using straight through gumbel softmax"
        _lib.require_device(x)        # raises for a CPU tensor: there is no CPU implementation
        flat, lead = self._flatten(x)
        H, n, d = flat.shape
        if H != self.num_codebooks or d != self.embeddings.shape[-1]:
            raise ValueError(f"vqb200.Codebook: input {tuple(x.shape)} does not match codebook "
                             f"(H={self.num_codebooks}, d={self.embeddings.shape[-1]})")
        mask_u8 = self._expand_mask(mask, n)
        grad_on = torch.is_grad_enabled()

        prepared = False
        if normalize_input:
            # transform_input="l2norm" (reference vector_quantize_pytorch.py:221)
            if grad_on and flat.requires_grad:
                # the encoder's gradient passes through the normalisation: same kernel forward (so the values do not
                # depend on whether a gradient is wanted), F.normalize's Jacobian on the way back
                flat = ops.l2norm_rows_autograd(flat)
            elif not (self.sharded or variants) and self.is_initialized and ops.l2norm_prepare_supported(d):
                # normalisation and the search's operand preparation share one pass over x when the codebook cache is
                # already final
                flat = ops.l2norm_prepare(flat, self.codebook_size, self._codebook_cache())
                prepared = True
            else:
                flat = ops.l2norm_rows(flat)
        wants_x = grad_on and flat.requires_grad

        # the latents the search, the EMA statistics and the expiry read: on a shard with "all_gather" input, the
        # batches of all ranks
        rows, rows_mask = flat, mask_u8
        gathered = self.sharded and self.sharded_input == "all_gather"
        if self.sharded:
            from . import distributed as D
            rows = flat.detach()
            if gathered:
                rows = D.all_gather_rows(rows, dim=1)
                if mask_u8 is not None:
                    rows_mask = D.all_gather_rows(mask_u8, dim=0)
        if not self.is_initialized:
            self._kmeans_init(rows, rows_mask)
            self.is_initialized = True

        # the codebook of this forward
        training = self.training
        update = training and self.ema_update and not freeze_codebook
        # learnable codebook (reference codebooks.py:375-377, vector_quantize_pytorch.py:262-268): the commitment loss
        # and the gathered codes are differentiable with respect to `embeddings`
        emb_param = self.embeddings if (self.learnable_codebook and self.commit_grad_to_codebook and training
                                        and not freeze_codebook and grad_on and self.embeddings.requires_grad) else None
        live = self.full_codebook() if self.sharded else self.embeddings.detach()
        emb_eff = live if emb_param is None else emb_param          # the codes as autograd sees them
        if self.use_affine:
            self._update_affine(flat, mask_u8)
            codebook_std = self.codebook_variance.clamp(min=1e-5).sqrt()
            batch_std = self.batch_variance.clamp(min=1e-5).sqrt()
            cm, bm, inv_scale = self.codebook_mean, self.batch_mean, codebook_std / batch_std
            emb_eff = ((emb_eff - cm) * (batch_std / codebook_std) + bm).contiguous()          # reference :381-384
            codes = emb_eff.detach()
        elif keep_dense or wants_x:
            # the EMA step of this forward, or of a later training forward before backward runs (gradient
            # accumulation; this one may be frozen), overwrites `embeddings` (on a shard: the replica) in place; the
            # reference's commitment loss holds the gathered codes of THIS forward (vector_quantize_pytorch.py:262-268,
            # a tensor materialised at codebooks.py:395 before :425), so everything saved for backward reads a snapshot
            codes = live.clone()
        else:
            codes = live
        if keep_dense:
            self.dense_ctx = ops._DenseCtx(flat, codes, codes if self.use_affine else self.embeddings,
                                           self.use_cosine_sim)

        # index assignment
        if self.sharded:
            idx_rows = self._shard_search(rows, self.embeddings.detach(), self._codebook_cache())
            ws = self.last_search_ws
            lo_r = self.shard_rank * n                              # this rank's batch among the gathered rows
            idx = idx_rows[:, lo_r:lo_r + n].contiguous() if gathered else idx_rows
        else:
            if stochastic:
                u = self._uniform_queue.pop(0) if self._uniform_queue else None
                idx = ops.dense_gumbel_sample(rows, codes, self.use_cosine_sim, float(g["temperature"]), uniforms=u)
                ws = None
            else:
                cache = ops.prepare_codebook(codes, self.use_cosine_sim) if self.use_affine else self._codebook_cache()
                idx, _, ws = ops.search(rows, codes, cache, self.use_cosine_sim, latents_prepared=prepared)
            self.last_search_ws = ws
            idx_rows = idx
            if self.return_similarities and not fuse_st:
                self._sim = ops.dense_scores(flat.detach(), codes, self.use_cosine_sim)   # before the EMA step, as :386

        # quantize.  Un-masked EMA training step: gather/ST/loss and the EMA sums share ONE pass over the latents (on a
        # shard with replicated input: the sums of all codes, of which this rank keeps its own)
        fused = update and mask_u8 is None and not (variants or gathered) and self.fused_quantize_ema \
            and ops.quantize_ema_supported(d) and emb_param is None
        commit = stats = None
        if st and training and grad_on and (emb_param is not None or (wants_x and not fuse_st)):
            quant, commit = self._gumbel_st_quantize(flat, emb_eff, idx, mask_u8, fuse_st, want_commit, rotation)
        elif fused and fuse_st:
            quant, commit, stats = ops.quantize_training(flat, codes, idx, None, want_commit, ema=True, bound_ws=ws,
                                                         rotation=rotation)
        elif fused:
            with torch.no_grad():
                quant, _, stats = ops.quantize_ema(flat, codes, idx, False, False, bound_ws=ws)
        elif fuse_st and training:
            quant, commit, _ = ops.quantize_training(flat, codes if emb_param is None else emb_eff, idx, mask_u8,
                                                     want_commit, rotation=rotation)
        elif emb_param is not None:
            quant = ops.gather_codes(emb_eff, idx)
        else:
            with torch.no_grad():
                quant, _ = ops.gather_st_loss(flat, codes, idx, None, False, False)

        if update:
            with torch.no_grad():
                if self.sharded:
                    lo, Ks = self.shard_offset, self.shard_size
                    stats = stats[:, lo:lo + Ks].contiguous() if stats is not None \
                        else self._shard_stats(rows, idx_rows, rows_mask)
                else:
                    if stats is None:
                        # the variants take no search bound (it picks the fixed-point scale of the sums)
                        stats = ops.ema_reduce(rows, idx, mask_u8, self.codebook_size,
                                               bound_ws=None if variants else ws)
                    if self.use_affine:
                        # reference :400-403 transforms every latent, (x - batch_mean) * (codebook_std / batch_std) +
                        # codebook_mean, before the sums; the map is affine, so the per-code sums transform the same way
                        cnt = stats[..., d:]
                        stats[..., :d] = (stats[..., :d] - cnt * bm) * inv_scale + cnt * cm
                    self._all_reduce(stats)                   # one packed (H,K,d+1) allreduce (reference: two)
                self._apply_ema(stats)
                if self.sharded:
                    self._expire_codes_sharded(rows)
                else:
                    self.expire_codes_(rows)
        return quant.reshape(H, *lead, d), idx.reshape(H, *lead), commit

    @torch.amp.autocast(device_type="cuda", enabled=False)
    def forward(self, x, mask=None, freeze_codebook=False):
        """reference codebooks.py:350-435.  Returns (quantize, embed_ind, similarities).  `similarities` is None unless
        `self.return_similarities` is set: the (H, ..., K) matrix is not needed by anything on this path and is only
        materialised on request (one extra fp32 score pass, vqb_dense_scores); like the reference's it keeps the leading
        codebook axis even when the input had none (:431-433)."""
        needs_codebook_dim = x.ndim < 4
        if needs_codebook_dim:
            x = x[None]
        self._sim = None
        quant, ind, _ = self._run(x, mask, freeze_codebook, fuse_st=False, want_commit=False)
        sim, self._sim = self._sim, None
        if sim is not None:
            sim = sim.reshape(*ind.shape, sim.shape[-1])
        if needs_codebook_dim:
            quant, ind = quant[0], ind[0]
        return quant, ind, sim


class EuclideanCodebook(Codebook):
    """Upstream name for ``Codebook(use_cosine_sim=False)`` (reference Changelog.md:11-12)."""

    def __init__(self, dim, codebook_size, **kw):
        kw.setdefault("use_cosine_sim", False)
        super().__init__(dim, codebook_size, **kw)


class CosineSimCodebook(Codebook):
    """Upstream name for the cosine codebook: dot similarity on l2-normalised inputs and codes."""

    def __init__(self, dim, codebook_size, **kw):
        kw.setdefault("use_cosine_sim", True)
        kw.setdefault("transform_input", "l2norm")
        kw.setdefault("weights_regularization", "l2norm")
        super().__init__(dim, codebook_size, **kw)
