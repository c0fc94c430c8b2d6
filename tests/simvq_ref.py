"""fp64 statement of the SimVQ / ResidualSimVQ contract (vqb200/simvq.py, upstream vector-quantize-pytorch's SimVQ) by
torch autograd, with the indices given: the search is checked on its own, this states everything after it.

One level on rows x (N,d) with codebook C' (K,d) and indices idx (N,):
    q = C'[idx],  loss = cw (mse(x.detach(), q) + beta mse(x, q.detach())),
    out = x + (q - x).detach()  or, with the rotation trick, upstream `rotate_to(x, q)` (rotation and norm ratio detached).
A residual stack runs r_{l+1} = r_l - out_l.detach() and returns sum_l out_l."""
import torch
import torch.nn.functional as F


def rotate_to(x, c):
    """Upstream `rotate_to(src=x, tgt=c)` on (R, d) rows: the gradient flows through e = x only."""
    e = x
    x, c = x.detach(), c.detach()
    nx, nc = x.norm(dim=-1, keepdim=True), c.norm(dim=-1, keepdim=True)
    u, q = x / nx.clamp_min(1e-6), c / nc.clamp_min(1e-6)
    w = F.normalize(u + q, dim=-1, eps=1e-12)
    lam = nc / nx.clamp_min(1e-6)
    return lam * (e - 2 * (e * w).sum(-1, keepdim=True) * w + 2 * (e * u).sum(-1, keepdim=True) * q)


def level(x, codebook, idx, beta, cw, rotation):
    """(out, loss) of one level."""
    q = codebook[idx]
    loss = cw * (F.mse_loss(x.detach(), q) + beta * F.mse_loss(x, q.detach()))
    out = rotate_to(x, q) if rotation else x + (q - x).detach()
    return out, loss


def stack(x, codebooks, idxs, beta, cw, rotation):
    """(sum of the levels' outputs, [loss_l]) of a residual stack."""
    r, out, losses = x, 0.0, []
    for cb, idx in zip(codebooks, idxs):
        o, loss = level(r, cb, idx, beta, cw, rotation)
        r = r - o.detach()
        out = out + o
        losses.append(loss)
    return out, losses


def grads(x, params, codebooks_of, idxs, beta, cw, rotation, w, g_losses):
    """fp64 gradients of (out * w).sum() + sum_l g_losses[l] * loss_l with respect to x (N,d) and `params`.
    `codebooks_of(params)` -> the list of C'_l in fp64."""
    x = x.detach().double().requires_grad_(True)
    ps = [p.detach().double().requires_grad_(True) for p in params]
    out, losses = stack(x, codebooks_of(ps), idxs, beta, cw, rotation)
    obj = (out * w.double()).sum() + sum(g * l for g, l in zip(g_losses, losses))
    gs = torch.autograd.grad(obj, [x] + ps)
    return out.detach(), torch.stack([l.detach() for l in losses]), gs[0], list(gs[1:])


def fp64_argmin_and_gap(x, codebook):
    """Nearest code by the fp64 Euclidean distance and the relative top-2 distance gap of every row (N,)."""
    dist = torch.cdist(x.double(), codebook.double())
    top = dist.topk(min(2, dist.shape[1]), dim=-1, largest=False)
    if dist.shape[1] < 2:
        return top.indices[:, 0], torch.full((x.shape[0],), float("inf"), dtype=torch.float64, device=x.device)
    gap = (top.values[:, 1] - top.values[:, 0]) / top.values[:, 0].clamp_min(1e-30)
    return top.indices[:, 0], gap
