"""Tensor-level wrappers over the C ABI (include/vqb.h).  PyTorch is plumbing here: it owns
device memory and the stream; every numeric step of the hot path runs in libvqb200.so.

Shapes: latents (H,N,d) contiguous, codebook (H,K,d) fp32 contiguous, indices (H,N) int64.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import _lib as L


def _on_device(fn):
    """Run `fn` with the CUDA device of its first tensor argument current.  The library launches on the stream it is
    given and creates TMA descriptors / queries attributes on the CURRENT device, so a module living on cuda:1 while
    the process's current device is cuda:0 must switch for the duration of the call (torch ops do the same)."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        for a in args:
            if isinstance(a, torch.Tensor):
                if a.is_cuda and a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kwargs)
                break
        return fn(*args, **kwargs)
    return wrapper

# ---------------------------------------------------------------------------------------------
# workspaces: caller-owned scratch, one growing buffer per (kind, device, stream)
# ---------------------------------------------------------------------------------------------
_WS: Dict[Tuple[str, int, int], torch.Tensor] = {}


def workspace(kind: str, nbytes: int, device: torch.device) -> torch.Tensor:
    key = (kind, device.index if device.index is not None else torch.cuda.current_device(),
           L.stream_ptr(device))
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


TIME_SEARCH_KERNEL = False   # bench.py: bracket the tensor-core kernel with CUDA events on its stream


def search_kernel_times_ms():
    """Durations (ms) of the tensor-core kernel of the searches made since the last call (needs TIME_SEARCH_KERNEL)."""
    import ctypes as C
    buf = (C.c_float * 64)()
    n = L.lib().vqb_search_timing(C.cast(buf, C.c_void_p), 64)
    if n < 0:
        L.check(n, "vqb_search_timing")
    return [float(buf[i]) for i in range(min(n, 64))]


def launch_count() -> int:
    return int(L.lib().vqb_launch_count())


def release_workspaces() -> None:
    _WS.clear()


def _metric(use_cosine_sim: bool) -> int:
    return L.VQB_DOT if use_cosine_sim else L.VQB_EUCLID


def _mask_u8(mask: Optional[torch.Tensor], n: int) -> Optional[torch.Tensor]:
    if mask is None:
        return None
    m = mask.reshape(-1).to(torch.uint8).contiguous()
    if m.numel() != n:
        raise ValueError(f"vqb200: mask has {m.numel()} rows, expected {n}")
    return m


# ---------------------------------------------------------------------------------------------
# codebook cache + search
# ---------------------------------------------------------------------------------------------
@_on_device
def prepare_codebook(embeddings: torch.Tensor, use_cosine_sim: bool,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Scaled fp16 copy + norms + rounding bounds of `embeddings` for the tensor-core search."""
    L.require_cuda(embeddings, "embeddings")
    assert embeddings.dtype == torch.float32 and embeddings.ndim == 3
    H, K, d = embeddings.shape
    nbytes = L.lib().vqb_codebook_cache_bytes(H, K, d)
    if out is None or out.numel() < nbytes or out.device != embeddings.device:
        out = torch.empty(nbytes, dtype=torch.uint8, device=embeddings.device)
    L.check(L.lib().vqb_prepare_codebook(L.ptr(embeddings), H, K, d, _metric(use_cosine_sim), L.ptr(out),
                                         out.numel(), L.stream_ptr(embeddings.device)), "vqb_prepare_codebook")
    return out


@_on_device
def search(x: torch.Tensor, embeddings: torch.Tensor, cache: Optional[torch.Tensor], use_cosine_sim: bool, *,
           idx_offset: int = 0, want_score: bool = False, latents_prepared: bool = False,
           force_exact: bool = False, fused_prep: bool = False) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor]:
    """Nearest code of every row.  Returns (idx (H,N) int64, score (H,N) fp32 | None, search workspace).
    `fused_prep` (opt-in, include/vqb.h VQB_SEARCH_FUSED_PREP): 16-bit latents are converted inside the search kernel."""
    L.require_cuda(x, "x")
    L.require_cuda(embeddings, "embeddings")
    H, N, d = x.shape
    Hc, K, dc = embeddings.shape
    if (Hc, dc) != (H, d):
        raise ValueError(f"vqb200: latents {tuple(x.shape)} do not match codebook {tuple(embeddings.shape)}")
    dev = x.device
    idx = torch.empty((H, N), dtype=torch.int64, device=dev)
    score = torch.empty((H, N), dtype=torch.float32, device=dev) if want_score else None
    ws = workspace("search", L.lib().vqb_search_workspace_bytes(H, N, K, d), dev)
    flags = (L.SEARCH_LATENTS_PREPARED if latents_prepared else 0) | (L.SEARCH_FORCE_EXACT if force_exact else 0) \
        | (L.SEARCH_TIMING if TIME_SEARCH_KERNEL else 0) | (L.SEARCH_FUSED_PREP if fused_prep else 0)
    L.check(L.lib().vqb_search(L.ptr(x), L.dtype_code(x), L.ptr(embeddings), L.ptr(cache), _metric(use_cosine_sim),
                               H, N, K, d, int(idx_offset), L.ptr(idx), L.ptr(score), flags, L.ptr(ws), ws.numel(),
                               L.stream_ptr(dev)), "vqb_search")
    return idx, score, ws


@_on_device
def search_stats(ws: torch.Tensor) -> Dict[str, int]:
    import ctypes as C
    out = (C.c_int64 * 3)()
    L.check(L.lib().vqb_search_stats(L.ptr(ws), C.cast(out, C.c_void_p), L.stream_ptr(ws.device)), "vqb_search_stats")
    return {"reranked_rows": int(out[0]), "rescanned_rows": int(out[1]), "tensor_core_pass": int(out[2])}


@_on_device
def l2norm_rows(x: torch.Tensor) -> torch.Tensor:
    L.require_cuda(x, "x")
    x = L.aligned(x)     # the kernel reads 4 elements at a time (16-byte loads for fp32)
    d = x.shape[-1]
    out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    rows = x.numel() // d if d else 0
    L.check(L.lib().vqb_l2norm_rows(L.ptr(x), L.dtype_code(x), L.ptr(out), rows, d, L.stream_ptr(x.device)),
            "vqb_l2norm_rows")
    return out


class _L2NormRows(torch.autograd.Function):
    """x / max(|x|, 1e-12) by the kernel (bit-identical with or without autograd), Jacobian of F.normalize on the way
    back (reference utils/losses.py:19 under autograd)."""

    @staticmethod
    def forward(ctx, x):
        y = l2norm_rows(x.contiguous())
        ctx.save_for_backward(x, y)
        return y

    @staticmethod
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        norm = x.float().norm(dim=-1, keepdim=True)
        denom = norm.clamp_min(1e-12)
        # y = x / denom;  d denom / dx = x / norm where norm > eps, else 0
        proj = (g * y).sum(dim=-1, keepdim=True) * torch.where(norm > 1e-12, denom / norm.clamp_min(1e-38),
                                                               torch.zeros_like(norm))
        return ((g - y * proj) / denom).to(x.dtype)


def l2norm_rows_autograd(x: torch.Tensor) -> torch.Tensor:
    return _L2NormRows.apply(x)


def l2norm_prepare_supported(d: int) -> bool:
    return bool(L.lib().vqb_l2norm_prepare_supported(int(d)))


@_on_device
def l2norm_prepare(x: torch.Tensor, K: int, cache: torch.Tensor) -> torch.Tensor:
    """x (H,N,d) -> x / |x| (fp32) and, in the shared search workspace, everything the next
    `search(out, ..., latents_prepared=True)` with this codebook cache needs."""
    L.require_cuda(x, "x")
    x = L.aligned(x)
    H, N, d = x.shape
    out = torch.empty((H, N, d), dtype=torch.float32, device=x.device)
    ws = workspace("search", L.lib().vqb_search_workspace_bytes(H, N, K, d), x.device)
    L.check(L.lib().vqb_l2norm_prepare(L.ptr(x), L.dtype_code(x), L.ptr(out), H, N, int(K), d, L.ptr(cache), L.ptr(ws),
                                       ws.numel(), L.stream_ptr(x.device)), "vqb_l2norm_prepare")
    return out


# ---------------------------------------------------------------------------------------------
# gather + straight-through + commitment loss (autograd-aware)
# ---------------------------------------------------------------------------------------------
@_on_device
def gather_st_loss(x: torch.Tensor, embeddings: torch.Tensor, idx: torch.Tensor, mask_u8: Optional[torch.Tensor],
                   training: bool, want_loss: bool) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """q (H,N,d) fp32 and loss_buf = [mean((c-x)^2), rows_used] (device) or None."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    K = embeddings.shape[1]
    dev = x.device
    q = torch.empty((H, N, d), dtype=torch.float32, device=dev)
    loss = torch.empty(2, dtype=torch.float32, device=dev) if want_loss else None
    ws = workspace("gather", L.lib().vqb_gather_workspace_bytes(H, N, d), dev)
    L.check(L.lib().vqb_gather_st_loss(L.ptr(x), L.dtype_code(x), L.ptr(embeddings), L.ptr(idx), L.ptr(mask_u8),
                                       int(training), int(want_loss), L.ptr(q), L.ptr(loss), H, N, K, d,
                                       L.ptr(ws), ws.numel(), L.stream_ptr(dev)), "vqb_gather_st_loss")
    return q, loss


def quantize_ema_supported(d: int) -> bool:
    return bool(L.lib().vqb_quantize_ema_supported(int(d)))


@_on_device
def quantize_ema(x: torch.Tensor, embeddings: torch.Tensor, idx: torch.Tensor, training: bool, want_loss: bool,
                 bound_ws: Optional[torch.Tensor] = None):
    """Fused gather/ST/loss + EMA sums (no mask): returns (q (H,N,d) fp32, loss_buf | None, stats (H,K,d+1)).
    `bound_ws`: the workspace `search` returned for this same `x`, with no other search in between (its first 8 bytes
    bound max|x_j|, which sizes the fixed-point sums; a stale or foreign bound can make them wrap around); None: one
    extra pass over x computes the bound."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    K = embeddings.shape[1]
    dev = x.device
    q = torch.empty((H, N, d), dtype=torch.float32, device=dev)
    loss = torch.empty(2, dtype=torch.float32, device=dev) if want_loss else None
    stats = torch.empty((H, K, d + 1), dtype=torch.float32, device=dev)
    ws = workspace("ema", L.lib().vqb_quantize_ema_workspace_bytes(H, N, K, d), dev)
    L.check(L.lib().vqb_quantize_ema(L.ptr(x), L.dtype_code(x), L.ptr(embeddings), L.ptr(idx), L.ptr(bound_ws),
                                     int(training), int(want_loss), L.ptr(q), L.ptr(loss), L.ptr(stats), H, N, K, d,
                                     L.ptr(ws), ws.numel(), L.stream_ptr(dev)), "vqb_quantize_ema")
    return q, loss, stats


@_on_device
def st_commit_backward(grad_q: torch.Tensor, g: torch.Tensor, x: torch.Tensor, embeddings: torch.Tensor,
                       idx: torch.Tensor, mask_u8: Optional[torch.Tensor]) -> torch.Tensor:
    """grad_x (H,N,d) fp32 = grad_q + g[0] * (x - C[idx]) on the rows with mask != 0, grad_q on the others."""
    H, N, d = x.shape
    K = embeddings.shape[1]
    gx = torch.empty((H, N, d), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_st_commit_backward(L.ptr(grad_q), L.ptr(g), L.ptr(x), L.dtype_code(x), L.ptr(embeddings),
                                           L.ptr(idx), L.ptr(mask_u8), 1.0, L.ptr(gx), H, N, K, d,
                                           L.stream_ptr(x.device)), "vqb_st_commit_backward")
    return gx


@_on_device
def rot_commit_backward(grad_q: torch.Tensor, g: torch.Tensor, x: torch.Tensor, embeddings: torch.Tensor,
                        idx: torch.Tensor, mask_u8: Optional[torch.Tensor]) -> torch.Tensor:
    """grad_x (H,N,d) fp32 = T(grad_q) + g[0] * (x - C[idx]) on the rows with mask != 0, grad_q on the others, where T
    is the rotation-trick transport of each row (vqb_rot_commit_backward)."""
    H, N, d = x.shape
    K = embeddings.shape[1]
    grad_q, x, embeddings = L.aligned(grad_q.float()), L.aligned(x), L.aligned(embeddings)
    gx = torch.empty((H, N, d), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_rot_commit_backward(L.ptr(grad_q), L.ptr(g), L.ptr(x), L.dtype_code(x), L.ptr(embeddings),
                                            L.ptr(idx), L.ptr(mask_u8), 1.0, L.ptr(gx), H, N, K, d,
                                            L.stream_ptr(x.device)), "vqb_rot_commit_backward")
    return gx


class _QuantizeST(torch.autograd.Function):
    """Training-mode quantize: returns (x + (c - x).detach(), mse(c.detach(), x), stats | None).

    With `ema` set (no mask) the forward is the fused pass that also produces the EMA statistics.
    Backward (SURVEY K16; reference autograd through vector_quantize_pytorch.py:273,362):
      grad_x = grad_q + grad_commit * 2 (x - c) / (rows_used * d);  the codebook gets no gradient.
    With `rotation` the gradient of `q` is the rotation trick's (upstream `rotate_to`, arXiv:2410.06424) instead:
      grad_x = T(grad_q) + grad_commit * 2 (x - c) / (rows_used * d)   on the rows with mask != 0 (vqb_rot_commit_backward);
    the forward value stays the straight-through one, fl(x + fl(c - x)), bit for bit.
    """

    @staticmethod
    def forward(ctx, x, embeddings, idx, mask_u8, want_loss, ema, bound_ws, rotation=False):
        stats = None
        if ema:
            q, loss, stats = quantize_ema(x, embeddings, idx, True, want_loss, bound_ws)
        else:
            q, loss = gather_st_loss(x, embeddings, idx, mask_u8, True, want_loss)
        ctx.save_for_backward(x, embeddings, idx, mask_u8 if mask_u8 is not None else torch.empty(0), loss
                              if loss is not None else torch.empty(0))
        ctx.has_mask = mask_u8 is not None
        ctx.want_loss = want_loss
        ctx.rotation = bool(rotation)
        commit = loss[0] if want_loss else torch.zeros((), device=x.device)
        if stats is None:
            stats = torch.empty(0, device=x.device)
        ctx.mark_non_differentiable(stats)
        return q, commit, stats

    @staticmethod
    def backward(ctx, grad_q, grad_commit, _grad_stats):
        x, embeddings, idx, mask_u8, loss = ctx.saved_tensors
        H, N, d = x.shape
        K = embeddings.shape[1]
        if grad_q is None:
            grad_q = torch.zeros((H, N, d), dtype=torch.float32, device=x.device)
        grad_q = grad_q.contiguous().float()
        g_emb = None
        # with no live rows (all masked, or N = 0) the loss is the mean of an empty selection: its gradient reaches no
        # row and no code, so dividing by max(rows, 1) sends zeros where rows = 0 would make 0 * inf = NaN
        rows = loss[1].clamp_min(1.0) if ctx.want_loss else None
        if ctx.needs_input_grad[1] and ctx.want_loss and grad_commit is not None:
            # learnable codebook: d mse(C[idx], x) / d C[k] = 2 (n_k C[k] - sum of the rows assigned to k) / (rows * d),
            # from the same deterministic segmented sums as the EMA statistics
            if H * N == 0:
                g_emb = torch.zeros_like(embeddings)
            else:
                st = ema_reduce(x, idx, mask_u8 if ctx.has_mask else None, K)
                g_emb = (grad_commit.float() * (2.0 / d) / rows) * (st[..., d:] * embeddings.detach() - st[..., :d])
        none = (g_emb,) + (None,) * 6
        has_commit = ctx.want_loss and grad_commit is not None
        if not has_commit and not ctx.rotation:
            return (grad_q.to(x.dtype),) + none
        # device scalar: grad_commit * 2 / (rows_used * d)   (no host sync)
        g = (grad_commit.float() * (2.0 / d) / rows).reshape(1).contiguous() if has_commit \
            else torch.zeros(1, dtype=torch.float32, device=x.device)
        mask = mask_u8 if ctx.has_mask else None
        gx = (rot_commit_backward if ctx.rotation else st_commit_backward)(grad_q, g, x, embeddings, idx, mask)
        return (gx.to(x.dtype),) + none


class _GatherCodes(torch.autograd.Function):
    """Codebook.forward with a learnable codebook: quantize = C[idx], d/dC[k] = sum of the incoming rows assigned to k."""

    @staticmethod
    def forward(ctx, embeddings, idx):
        H, K, d = embeddings.shape
        e = embeddings.detach()
        q = torch.stack([e[h][idx[h]] for h in range(H)], 0)      # plain gather; the backward is the kernel work
        ctx.save_for_backward(idx)
        ctx.K = K
        return q

    @staticmethod
    def backward(ctx, grad_q):
        (idx,) = ctx.saved_tensors
        st = ema_reduce(grad_q.contiguous().float(), idx, None, ctx.K)
        return st[..., :-1].contiguous(), None


def gather_codes(embeddings: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    return _GatherCodes.apply(embeddings, idx)


def quantize_training(x, embeddings, idx, mask_u8, want_loss, ema: bool = False, bound_ws=None, rotation: bool = False):
    """(q, commit, stats | None); `ema=True` (mask must be None) uses the fused gather+EMA pass; `rotation`: the
    rotation-trick gradient instead of the straight-through one (same forward values)."""
    assert not (ema and mask_u8 is not None)
    q, commit, stats = _QuantizeST.apply(x, embeddings, idx, mask_u8, want_loss, ema, bound_ws, rotation)
    return q, commit, (stats if ema else None)


# ---------------------------------------------------------------------------------------------
# EMA statistics / refresh / expiry
# ---------------------------------------------------------------------------------------------
@_on_device
def ema_reduce(x: torch.Tensor, idx: torch.Tensor, mask_u8: Optional[torch.Tensor], K: int,
               bound_ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """stats (H,K,d+1): per-code sums of assigned rows and counts.  Bitwise reproducible.
    `bound_ws`: the workspace `search` returned for this same `x`, with no other search in between (its first 8 bytes
    bound max|x_j|, which sizes the fixed-point sums; a stale or foreign bound can make them wrap around); None: one
    extra pass over x computes the bound."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    dev = x.device
    stats = torch.empty((H, K, d + 1), dtype=torch.float32, device=dev)
    ws = workspace("ema", L.lib().vqb_ema_workspace_bytes(H, N, K, d), dev)
    L.check(L.lib().vqb_ema_reduce(L.ptr(x), L.dtype_code(x), L.ptr(idx), L.ptr(mask_u8), L.ptr(bound_ws), H, N, K, d,
                                   L.ptr(stats), L.ptr(ws), ws.numel(), L.stream_ptr(dev)), "vqb_ema_reduce")
    return stats


@_on_device
def ema_apply(stats: torch.Tensor, cluster_size: torch.Tensor, embed_avg: torch.Tensor, embeddings: torch.Tensor,
              weight: float, eps: float, weights_l2norm: bool) -> None:
    H, K, d1 = stats.shape
    d = d1 - 1
    for t, n in ((stats, "stats"), (cluster_size, "cluster_size"), (embed_avg, "embed_avg"), (embeddings, "embeddings")):
        L.require_cuda(t, n)
    dev = stats.device
    ws = workspace("ema", max(256, 4 * H), dev)
    L.check(L.lib().vqb_ema_apply(L.ptr(stats), L.ptr(cluster_size), L.ptr(embed_avg), L.ptr(embeddings),
                                  float(weight), float(eps), int(weights_l2norm), H, K, d, L.ptr(ws), ws.numel(),
                                  L.stream_ptr(dev)), "vqb_ema_apply")


@_on_device
def ema_apply_sharded(stats: torch.Tensor, cluster_size: torch.Tensor, embed_avg: torch.Tensor,
                      embeddings: torch.Tensor, weight: float, eps: float, weights_l2norm: bool, k_total: int,
                      all_reduce) -> None:
    """vqb_ema_apply for a row-sharded codebook: `all_reduce(totals)` sums sum(cluster_size) over the shards."""
    H, K, d1 = stats.shape
    d = d1 - 1
    dev = stats.device
    totals = torch.empty(H, dtype=torch.float32, device=dev)
    st = L.stream_ptr(dev)
    L.check(L.lib().vqb_ema_apply_counts(L.ptr(stats), L.ptr(cluster_size), float(weight), H, K, d, L.ptr(totals), st),
            "vqb_ema_apply_counts")
    all_reduce(totals)
    L.check(L.lib().vqb_ema_apply_rows(L.ptr(stats), L.ptr(cluster_size), L.ptr(embed_avg), L.ptr(embeddings),
                                       float(weight), float(eps), int(k_total), int(weights_l2norm), H, K, d,
                                       L.ptr(totals), st), "vqb_ema_apply_rows")


@_on_device
def expire_scatter(x_rows: torch.Tensor, sample_rows: torch.Tensor, threshold: float, reset: float,
                   weights_l2norm: bool, cluster_size: torch.Tensor, embed_avg: torch.Tensor,
                   embeddings: torch.Tensor) -> None:
    """One codebook: x_rows (N,d); cluster_size (K,), embed_avg/embeddings (K,d) views of codebook h."""
    L.require_cuda(x_rows, "x")
    N, d = x_rows.shape
    K = cluster_size.shape[0]
    for t, n in ((cluster_size, "cluster_size"), (embed_avg, "embed_avg"), (embeddings, "embeddings")):
        L.require_cuda(t, n)
    sample_rows = sample_rows.to(device=x_rows.device, dtype=torch.int64).contiguous()
    L.check(L.lib().vqb_expire_scatter(L.ptr(x_rows), L.dtype_code(x_rows), L.ptr(sample_rows), sample_rows.numel(),
                                       float(threshold), float(reset), int(weights_l2norm), L.ptr(cluster_size),
                                       L.ptr(embed_avg), L.ptr(embeddings), N, K, d, L.stream_ptr(x_rows.device)),
            "vqb_expire_scatter")


# ---------------------------------------------------------------------------------------------
# ResidualVQ level step and sharded-codebook keys
# ---------------------------------------------------------------------------------------------
@_on_device
def rvq_level(residual: torch.Tensor, residual_next: torch.Tensor, embeddings: torch.Tensor, idx: torch.Tensor,
              mask_u8: Optional[torch.Tensor], training: bool, first_level: bool, quantized_out: torch.Tensor,
              next_cache: Optional[torch.Tensor], q_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Reads `residual` (N,d fp32), writes `residual_next` and updates `quantized_out` in place;
    returns loss_buf [mean sq err, rows used].  `next_cache`: codebook cache of the level that searches
    `residual_next` next (its operands are prepared in the same pass; same number of codes as `embeddings`), or None."""
    prepare_next = next_cache is not None
    L.require_cuda(residual, "residual")
    L.require_cuda(residual_next, "residual_next")
    assert residual.dtype == torch.float32 and residual.ndim == 2 and residual_next.shape == residual.shape
    residual, embeddings = L.aligned(residual), L.aligned(embeddings)
    for t, n in ((residual_next, "residual_next"), (quantized_out, "quantized_out"), (q_out, "q_out")):
        L.require_aligned(t, n)
    N, d = residual.shape
    K = embeddings.shape[-2]
    dev = residual.device
    loss = torch.empty(2, dtype=torch.float32, device=dev)
    gws = workspace("gather", L.lib().vqb_gather_workspace_bytes(1, N, d), dev)
    nws = workspace("search", L.lib().vqb_search_workspace_bytes(1, N, K, d), dev) if prepare_next else None
    L.check(L.lib().vqb_rvq_level(L.ptr(residual), L.ptr(residual_next), L.ptr(embeddings), L.ptr(idx), L.ptr(mask_u8), int(training),
                                  int(first_level), L.ptr(quantized_out), L.ptr(q_out), L.ptr(loss), N, K, d,
                                  L.ptr(gws), gws.numel(), L.ptr(nws), nws.numel() if nws is not None else 0,
                                  L.ptr(next_cache), L.stream_ptr(dev)), "vqb_rvq_level")
    return loss


def rvq_replay_out_supported(d: int, num_levels: int) -> bool:
    return bool(L.lib().vqb_rvq_replay_out_supported(int(d), int(num_levels)))


@_on_device
def rvq_replay_out(x: torch.Tensor, codebooks, idxs, training, mask_u8: Optional[torch.Tensor],
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Sum of the levels' outputs of a ResidualVQ forward (what `quantized_out` accumulates level by level), replayed
    bit-exactly from the level-0 input x (N,d) fp32, the (K,d) codebook each level gathered from and its (N,) indices."""
    import ctypes as C
    L.require_cuda(x, "x")
    assert x.dtype == torch.float32 and x.ndim == 2
    x = L.aligned(x)
    N, d = x.shape
    Q = len(codebooks)
    keep = [L.aligned(c) for c in codebooks] + [i.contiguous() for i in idxs]
    cbp = (C.c_void_p * Q)(*[L.ptr(c) for c in keep[:Q]])
    ixp = (C.c_void_p * Q)(*[L.ptr(i) for i in keep[Q:]])
    trp = (C.c_int * Q)(*[int(bool(t)) for t in training])
    if out is None:
        out = torch.empty((N, d), dtype=torch.float32, device=x.device)
    L.require_aligned(out, "out")
    L.check(L.lib().vqb_rvq_replay_out(L.ptr(x), C.cast(cbp, C.c_void_p), C.cast(ixp, C.c_void_p),
                                       C.cast(trp, C.c_void_p), Q, L.ptr(mask_u8), L.ptr(out), N, d,
                                       L.stream_ptr(x.device)), "vqb_rvq_replay_out")
    return out


def _rvq_backward(entry: str, x, codebooks, idxs, training, coef, g_out, mask_u8) -> torch.Tensor:
    import ctypes as C
    L.require_cuda(x, "x")
    x = L.aligned(x)
    N, d = x.shape
    Q = len(codebooks)
    keep = [L.aligned(c) for c in codebooks] + [i.contiguous() for i in idxs]
    cbp = (C.c_void_p * Q)(*[L.ptr(c) for c in keep[:Q]])
    ixp = (C.c_void_p * Q)(*[L.ptr(i) for i in keep[Q:]])
    trp = (C.c_int * Q)(*[int(bool(t)) for t in training])
    coef = coef.to(device=x.device, dtype=torch.float32).contiguous()
    # a contiguous fp32 gradient can still start at any element (a view into a larger buffer): the kernel reads it
    # with 128-bit loads
    g = L.aligned(g_out.float()) if g_out is not None else None
    gx = torch.empty((N, d), dtype=torch.float32, device=x.device)
    L.check(getattr(L.lib(), entry)(L.ptr(x), C.cast(cbp, C.c_void_p), C.cast(ixp, C.c_void_p),
                                    C.cast(trp, C.c_void_p), Q, L.ptr(coef), L.ptr(g), L.ptr(mask_u8), L.ptr(gx), N, d,
                                    L.stream_ptr(x.device)), entry)
    return gx


@_on_device
def rvq_backward(x: torch.Tensor, codebooks, idxs, training, coef: torch.Tensor, g_out: Optional[torch.Tensor],
                 mask_u8: Optional[torch.Tensor]) -> torch.Tensor:
    """Input gradient (N,d) of a ResidualVQ training forward: Q * g_out + sum_l coef[l] * (r_l - C_l[idx_l]) on the
    rows with mask != 0 (vqb_rvq_backward); the residuals are replayed from x and the indices."""
    return _rvq_backward("vqb_rvq_backward", x, codebooks, idxs, training, coef, g_out, mask_u8)


@_on_device
def rvq_backward_rot(x: torch.Tensor, codebooks, idxs, training, coef: torch.Tensor, g_out: Optional[torch.Tensor],
                     mask_u8: Optional[torch.Tensor]) -> torch.Tensor:
    """`rvq_backward` for levels with the rotation-trick gradient: sum_l T_l(g_out) + sum_l coef[l] * (r_l - c_l) on
    the rows with mask != 0, T_l the rotation transport of level l (identity on masked rows; vqb_rvq_backward_rot)."""
    return _rvq_backward("vqb_rvq_backward_rot", x, codebooks, idxs, training, coef, g_out, mask_u8)


def rvq_level_ema_supported(d: int) -> bool:
    return bool(L.lib().vqb_rvq_level_ema_supported(int(d)))


@_on_device
def rvq_level_ema(residual: torch.Tensor, residual_next: torch.Tensor, embeddings: torch.Tensor, idx: torch.Tensor,
                  training: bool, first_level: bool, quantized_out: torch.Tensor, next_cache: Optional[torch.Tensor],
                  bound_ws: Optional[torch.Tensor] = None, q_out: Optional[torch.Tensor] = None):
    """rvq_level + ema_reduce of an un-masked level in one pass: returns (loss_buf, stats (1,K,d+1)).
    `bound_ws` as in `ema_reduce`: the workspace of the search on this `residual`."""
    L.require_cuda(residual, "residual")
    L.require_cuda(residual_next, "residual_next")
    assert residual.dtype == torch.float32 and residual.ndim == 2 and residual_next.shape == residual.shape
    residual, embeddings = L.aligned(residual), L.aligned(embeddings)
    for t, n in ((residual_next, "residual_next"), (quantized_out, "quantized_out"), (q_out, "q_out")):
        L.require_aligned(t, n)
    N, d = residual.shape
    K = embeddings.shape[-2]
    dev = residual.device
    loss = torch.empty(2, dtype=torch.float32, device=dev)
    stats = torch.empty((1, K, d + 1), dtype=torch.float32, device=dev)
    ws = workspace("ema", L.lib().vqb_quantize_ema_workspace_bytes(1, N, K, d), dev)
    nws = workspace("search", L.lib().vqb_search_workspace_bytes(1, N, K, d), dev) if next_cache is not None else None
    L.check(L.lib().vqb_rvq_level_ema(L.ptr(residual), L.ptr(residual_next), L.ptr(embeddings), L.ptr(idx),
                                      L.ptr(bound_ws), int(training), int(first_level), L.ptr(quantized_out),
                                      L.ptr(q_out), L.ptr(loss), L.ptr(stats), N, K, d, L.ptr(ws), ws.numel(),
                                      L.ptr(nws), nws.numel() if nws is not None else 0, L.ptr(next_cache),
                                      L.stream_ptr(dev)), "vqb_rvq_level_ema")
    return loss, stats


@_on_device
def minkey_pack(score: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    L.require_cuda(score, "score")
    keys = torch.empty(score.numel(), dtype=torch.int64, device=score.device)
    L.check(L.lib().vqb_minkey_pack(L.ptr(score), L.ptr(idx), score.numel(), L.ptr(keys), L.stream_ptr(score.device)),
            "vqb_minkey_pack")
    return keys


@_on_device
def minkey_unpack(keys: torch.Tensor, want_score: bool = False):
    L.require_cuda(keys, "keys")
    idx = torch.empty(keys.numel(), dtype=torch.int64, device=keys.device)
    score = torch.empty(keys.numel(), dtype=torch.float32, device=keys.device) if want_score else None
    L.check(L.lib().vqb_minkey_unpack(L.ptr(keys), keys.numel(), L.ptr(idx), L.ptr(score), L.stream_ptr(keys.device)),
            "vqb_minkey_unpack")
    return idx, score


# ---------------------------------------------------------------------------------------------
# consumers of the dense N x K similarities (cross-entropy to indices, CE commitment, diversity loss):
# fp32 CUDA-core passes with an online softmax, nothing of size N x K is written (csrc/dense.cu)
# ---------------------------------------------------------------------------------------------
@_on_device
def dense_row_norms(t: torch.Tensor) -> torch.Tensor:
    """|row|^2 of a (..., d) tensor -> (...,) fp32."""
    L.require_cuda(t, "t")
    d = t.shape[-1]
    out = torch.empty(t.shape[:-1], dtype=torch.float32, device=t.device)
    L.check(L.lib().vqb_dense_row_norms(L.ptr(t), L.dtype_code(t), t.numel() // d if d else 0, d, L.ptr(out),
                                        L.stream_ptr(t.device)), "vqb_dense_row_norms")
    return out


@_on_device
def dense_rowstats(x, xn2, emb, cn2, use_cosine_sim: bool, alpha: float, target: Optional[torch.Tensor]):
    """lse (H,N) = log sum_k exp(alpha s_k) and, with `target` (H,N) int64 (-1 = ignore), the score of the target."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    K = emb.shape[1]
    lse = torch.empty((H, N), dtype=torch.float32, device=x.device)
    st = torch.zeros((H, N), dtype=torch.float32, device=x.device) if target is not None else None
    L.check(L.lib().vqb_dense_rowstats(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                       _metric(use_cosine_sim), float(alpha), L.ptr(target), L.ptr(lse), L.ptr(st),
                                       H, N, K, d, L.stream_ptr(x.device)), "vqb_dense_rowstats")
    return lse, st


@_on_device
def dense_avgprob(x, xn2, emb, cn2, use_cosine_sim: bool, alpha: float, lse, n_pos: int) -> torch.Tensor:
    """(n_pos, K): softmax(alpha s) averaged over the codebooks and the N / n_pos batch entries of each position."""
    H, N, d = x.shape
    K = emb.shape[1]
    avg = torch.empty((n_pos, K), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_dense_avgprob(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                      _metric(use_cosine_sim), float(alpha), L.ptr(lse), L.ptr(avg), int(n_pos),
                                      H, N, K, d, L.stream_ptr(x.device)), "vqb_dense_avgprob")
    return avg


@_on_device
def dense_rowdot(x, xn2, emb, cn2, use_cosine_sim: bool, alpha: float, lse, table, n_pos: int) -> torch.Tensor:
    """(H,N): sum_k softmax(alpha s)_k * table[row % n_pos, k]."""
    H, N, d = x.shape
    K = emb.shape[1]
    out = torch.empty((H, N), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_dense_rowdot(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                     _metric(use_cosine_sim), float(alpha), L.ptr(lse), L.ptr(table), int(n_pos),
                                     L.ptr(out), H, N, K, d, L.stream_ptr(x.device)), "vqb_dense_rowdot")
    return out


@_on_device
def dense_backward(x, xn2, emb_dist, cn2, emb_comb, use_cosine_sim: bool, alpha: float, lse, coef, target=None,
                   table=None, rdot=None, n_pos: int = 1) -> torch.Tensor:
    """Input gradient (H,N,d) fp32 of a loss on the similarities (see include/vqb.h: vqb_dense_backward)."""
    H, N, d = x.shape
    K = emb_dist.shape[1]
    gx = torch.empty((H, N, d), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_dense_backward(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb_dist), L.ptr(cn2),
                                       L.ptr(emb_comb), _metric(use_cosine_sim), float(alpha), L.ptr(lse), L.ptr(coef),
                                       L.ptr(target), L.ptr(table), L.ptr(rdot), int(n_pos), L.ptr(gx), H, N, K, d,
                                       L.stream_ptr(x.device)), "vqb_dense_backward")
    return gx


@_on_device
def dense_backward_codes(x, xn2, emb, cn2, use_cosine_sim: bool, alpha: float, lse, coef, target=None, table=None,
                         rdot=None, n_pos: int = 1) -> torch.Tensor:
    """Codebook gradient (H,K,d) fp32 of a loss on the similarities (learnable codebook): the transposed contraction
    of `dense_backward`; partial sums over latent tiles are added in a fixed order."""
    H, N, d = x.shape
    K = emb.shape[1]
    splits = int(L.lib().vqb_dense_backward_codes_splits(H, N, K, d))
    part = torch.empty((splits, H, K, d), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_dense_backward_codes(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                             _metric(use_cosine_sim), float(alpha), L.ptr(lse), L.ptr(coef),
                                             L.ptr(target), L.ptr(table), L.ptr(rdot), int(n_pos), L.ptr(part),
                                             splits, H, N, K, d, L.stream_ptr(x.device)), "vqb_dense_backward_codes")
    return part[0] if splits == 1 else part.sum(dim=0)


class _DenseCtx:
    """What the dense consumers of one forward share: latents (H,N,d), the codebook the similarities are defined on
    (`emb_dist`: a private copy when the EMA step overwrites `embeddings` in this forward) and the live buffer
    (`emb_live`) whose rows the reference's backward combines (see csrc/dense.cu header), plus the row norms."""

    def __init__(self, x, emb_dist, emb_live, use_cosine_sim):
        self.x, self.emb_dist, self.emb_live, self.cos = x, emb_dist, emb_live, bool(use_cosine_sim)
        self.xn2 = None if self.cos else dense_row_norms(x.detach())
        self.cn2 = None if self.cos else dense_row_norms(emb_dist)


class _DenseCE(torch.autograd.Function):
    """mean over rows with target >= 0 of (logsumexp_k s_k - s_target): F.cross_entropy(similarities, codes,
    ignore_index=-1) of reference vector_quantize_pytorch.py:284-296 on the (H,N) row layout.  `emb` is the learnable
    codebook Parameter (it then receives the gradient through the similarities, codebooks.py:375-377) or None."""

    @staticmethod
    def forward(ctx, x, emb, dc, target):
        lse, st = dense_rowstats(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, 1.0, target)
        valid = target >= 0
        n_valid = valid.sum()
        loss = (((lse.double() - st.double()) * valid).sum() / n_valid).float()
        ctx.dc, ctx.lse, ctx.target, ctx.valid, ctx.n_valid = dc, lse, target, valid, n_valid
        ctx.save_for_backward(x)
        return loss

    @staticmethod
    def backward(ctx, g):
        dc, (x,) = ctx.dc, ctx.saved_tensors
        coef = ((g.float() / ctx.n_valid) * ctx.valid).contiguous()
        gx = ge = None
        if ctx.needs_input_grad[0]:
            gx = dense_backward(x, dc.xn2, dc.emb_dist, dc.cn2, dc.emb_live.detach(), dc.cos, 1.0, ctx.lse, coef,
                                target=ctx.target).to(x.dtype)
        if ctx.needs_input_grad[1]:
            ge = dense_backward_codes(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, 1.0, ctx.lse, coef, target=ctx.target)
        return gx, ge, None, None


def dense_cross_entropy(dc: "_DenseCtx", target: torch.Tensor, emb_param=None) -> torch.Tensor:
    """`target` (H,N) int64 in the row layout of dc.x, -1 = ignored."""
    return _DenseCE.apply(dc.x, emb_param, dc, target.contiguous())


class _DenseAvgProb(torch.autograd.Function):
    """avg_prob (n_pos, K) of reference vector_quantize_pytorch.py:324-328: softmax(-similarities * temperature)
    averaged over heads and batch; the entropy on top of it is K-sized torch glue."""

    @staticmethod
    def forward(ctx, x, emb, dc, n_pos, alpha):
        lse, _ = dense_rowstats(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, alpha, None)
        avg = dense_avgprob(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, alpha, lse, n_pos)
        ctx.dc, ctx.lse, ctx.n_pos, ctx.alpha = dc, lse, n_pos, alpha
        ctx.save_for_backward(x)
        return avg

    @staticmethod
    def backward(ctx, g_avg):
        dc, (x,), n_pos, alpha = ctx.dc, ctx.saved_tensors, ctx.n_pos, ctx.alpha
        H, N, _ = x.shape
        table = g_avg.contiguous().float()
        rdot = dense_rowdot(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, alpha, ctx.lse, table, n_pos)
        coef = torch.full((H, N), alpha / (H * (N // n_pos)), dtype=torch.float32, device=x.device)
        gx = ge = None
        if ctx.needs_input_grad[0]:
            gx = dense_backward(x, dc.xn2, dc.emb_dist, dc.cn2, dc.emb_live.detach(), dc.cos, alpha, ctx.lse, coef,
                                table=table, rdot=rdot, n_pos=n_pos).to(x.dtype)
        if ctx.needs_input_grad[1]:
            ge = dense_backward_codes(x, dc.xn2, dc.emb_dist, dc.cn2, dc.cos, alpha, ctx.lse, coef, table=table,
                                      rdot=rdot, n_pos=n_pos)
        return gx, ge, None, None, None


def dense_avg_prob(dc: "_DenseCtx", n_pos: int, temperature: float, emb_param=None) -> torch.Tensor:
    return _DenseAvgProb.apply(dc.x, emb_param, dc, int(n_pos), -float(temperature))


# ---------------------------------------------------------------------------------------------
# f4 variants: gumbel sampling, materialised similarities, column moments (affine)
# ---------------------------------------------------------------------------------------------
def _aten_uniform_launch(numel: int, device: torch.device):
    """(threads, counter_offset) of ATen's CUDA `uniform_` on `numel` elements (DistributionTemplates.h,
    calc_execution_policy: block 256, unroll 4, grid = min(SMs * maxThreadsPerSM / 256, ceil(numel / 256)))."""
    props = torch.cuda.get_device_properties(device)
    block, unroll = 256, 4
    grid = (numel + block - 1) // block
    grid = min(props.multi_processor_count * (props.max_threads_per_multi_processor // block), grid)
    grid = max(grid, 1)
    counter_offset = ((numel - 1) // (block * grid * unroll) + 1) * 4
    return block * grid, counter_offset


@_on_device
def dense_gumbel_sample(x: torch.Tensor, emb: torch.Tensor, use_cosine_sim: bool, temperature: float,
                        uniforms: Optional[torch.Tensor] = None, generator: Optional[torch.Generator] = None):
    """idx (H,N) = argmax_k(s_k / temperature - log(-log(u_k))) (reference utils/general.py:107-129).  `uniforms`
    (H,N,K) fp32 injects the draw; otherwise the kernel generates, in place, the numbers that
    `torch.zeros(H,N,K, device=...).uniform_(0, 1)` would draw from `generator` (default: the device's default
    generator) and advances that generator by the same amount (bitwise the same stream while H*N*K < 2^31, where ATen
    uses one launch)."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    K = emb.shape[1]
    dev = x.device
    xn2 = None if use_cosine_sim else dense_row_norms(x)
    cn2 = None if use_cosine_sim else dense_row_norms(emb)
    idx = torch.empty((H, N), dtype=torch.int64, device=dev)
    seed = offset = threads = 0
    if uniforms is not None:
        uniforms = uniforms.to(device=dev, dtype=torch.float32).contiguous()
        assert uniforms.numel() == H * N * K, "uniforms must be (H,N,K)"
    elif H * N * K > 0:
        gen = generator if generator is not None else torch.cuda.default_generators[dev.index]
        threads, counter = _aten_uniform_launch(H * N * K, dev)
        seed, offset = int(gen.initial_seed()), int(gen.get_offset())
        gen.set_offset(offset + counter)
    L.check(L.lib().vqb_dense_gumbel_sample(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                            _metric(use_cosine_sim), float(temperature), L.ptr(uniforms),
                                            seed & 0xFFFFFFFFFFFFFFFF, offset, threads, L.ptr(idx), H, N, K, d,
                                            L.stream_ptr(dev)), "vqb_dense_gumbel_sample")
    return idx


@_on_device
def dense_scores(x: torch.Tensor, emb: torch.Tensor, use_cosine_sim: bool) -> torch.Tensor:
    """The reference's `similarities` (H,N,K) fp32, materialised (opt-in third return value of Codebook.forward)."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    K = emb.shape[1]
    xn2 = None if use_cosine_sim else dense_row_norms(x)
    cn2 = None if use_cosine_sim else dense_row_norms(emb)
    out = torch.empty((H, N, K), dtype=torch.float32, device=x.device)
    L.check(L.lib().vqb_dense_scores(L.ptr(x), L.dtype_code(x), L.ptr(xn2), L.ptr(emb), L.ptr(cn2),
                                     _metric(use_cosine_sim), L.ptr(out), H, N, K, d, L.stream_ptr(x.device)),
            "vqb_dense_scores")
    return out


@_on_device
def column_moments(x: torch.Tensor, mask_u8: Optional[torch.Tensor]):
    """x (H,N,d): per codebook and column (sum, sum of squares) fp64 (H,d,2) over the rows with mask != 0, and the
    number of rows counted (H,) int64 -- one pass (vqb_column_moments)."""
    L.require_cuda(x, "x")
    H, N, d = x.shape
    sums = torch.empty((H, d, 2), dtype=torch.float64, device=x.device)
    rows = torch.empty((H,), dtype=torch.int64, device=x.device)
    L.check(L.lib().vqb_column_moments(L.ptr(x), L.dtype_code(x), L.ptr(mask_u8), H, N, d, L.ptr(sums), L.ptr(rows),
                                       L.stream_ptr(x.device)), "vqb_column_moments")
    return sums, rows


def orthogonal_loss(t: torch.Tensor) -> torch.Tensor:
    """reference utils/losses.py:22-27 (eq. 2 of arXiv:2112.00384): mean squared cosine similarity between the codes of
    each codebook, minus 1/n.  sum_ij (n_i . n_j)^2 = |N^T N|_F^2 = |N N^T|_F^2: the smaller of the (d,d) and (n,n) Gram
    matrices is formed (a K = 65536 codebook never allocates K x K).  Plain library GEMM on codebook-sized operands."""
    h, n = t.shape[:2]
    normed = torch.nn.functional.normalize(t, p=2, dim=-1)
    if t.shape[-1] < n:
        gram = torch.einsum("hnd,hne->hde", normed, normed)
    else:
        gram = torch.einsum("hid,hjd->hij", normed, normed)
    return (gram ** 2).sum() / (h * n ** 2) - (1 / n)
