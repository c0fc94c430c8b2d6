"""The rotation-trick gradient (`VectorQuantize.rotation_trick = True`, Fifty et al., arXiv:2410.06424) against an fp64
restatement of upstream vector-quantize-pytorch's `rotate_to`.

For one row with input x and code c (the input after projection, head split and cosine normalisation; for a
ResidualVQ level its residual), with sx = max(|x|, 1e-6), sc = max(|c|, 1e-6), u = x / sx, q = c / sc,
w = F.normalize(u + q) and lambda = |c| / sx, upstream returns lambda (e - 2 (e.w) w + 2 (e.u) q) with e = x and
everything but e detached.  The returned value here stays the straight-through one, fl(x + fl(c - x)); the input
gradient is autograd through the fp64 statement below plus the commitment MSE.

Bar, per row: |got - ref|_2 <= 1e-5 f (lambda |g|_2 + |coef| |x - c|_2), f = max(1, 1 / |u + q|) (f = 1 where u + q
is exactly 0).  Rows outside the loss get grad_q bit for bit.

Part A: `vqb_rot_commit_backward`; part B: `vqb_rvq_backward_rot`; part C: the modules."""
import random

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5


def _cpu_draw(num_rows, m, device):
    if num_rows >= m:
        return torch.randperm(num_rows)[:m].to(device)
    return torch.randint(0, num_rows, (m,)).to(device)


@pytest.fixture(autouse=True)
def _patch_draw(monkeypatch):
    from vqb200 import codebook
    monkeypatch.setattr(codebook.Codebook, "_draw_rows", staticmethod(_cpu_draw))


# ----------------------------------------------------------------------------------------------------- reference
def rotate_to(x, c):
    """Upstream `rotate_to(src=x, tgt=c)` in fp64 on (R, d) rows: the gradient flows through e = x only."""
    e = x
    x, c = x.detach(), c.detach()
    nx, nc = x.norm(dim=-1, keepdim=True), c.norm(dim=-1, keepdim=True)
    u, q = x / nx.clamp_min(1e-6), c / nc.clamp_min(1e-6)
    w = F.normalize(u + q, dim=-1, eps=1e-12)
    lam = nc / nx.clamp_min(1e-6)
    return lam * (e - 2 * (e * w).sum(-1, keepdim=True) * w + 2 * (e * u).sum(-1, keepdim=True) * q)


def ref_grad(x, c, g, coef, live):
    """fp64 input gradient of sum(g * where(live, rotate_to(x, c), x)) + coef / 2 * sum_live |x - c|^2, and the bar."""
    x, c, g = x.double(), c.double(), g.double()
    live = torch.ones(x.shape[0], dtype=torch.bool, device=x.device) if live is None else live.bool()
    e = x.clone().requires_grad_(True)
    out = torch.where(live[:, None], rotate_to(e, c), e)
    obj = (out * g).sum() + 0.5 * coef * (((e - c) ** 2).sum(-1) * live).sum()
    (gx,) = torch.autograd.grad(obj, e)
    return gx, row_bar(x, c, g, coef) * live


def row_bar(x, c, g, coef):
    x, c, g = x.double(), c.double(), g.double()
    nx, nc = x.norm(dim=-1), c.norm(dim=-1)
    upq = (x / nx.clamp_min(1e-6)[:, None] + c / nc.clamp_min(1e-6)[:, None]).norm(dim=-1)
    f = torch.where(upq > 0, (1 / upq).clamp_min(1.0), torch.ones_like(upq))
    lam = nc / nx.clamp_min(1e-6)
    return TOL * f * (lam * g.norm(dim=-1) + abs(float(coef)) * (x - c).norm(dim=-1))


def assert_rows(got, ref, bar, what):
    err = (got.double() - ref).norm(dim=-1)
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite gradient"
    bad = err > bar
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} rows over the bar, worst err/bar " \
                                f"{float((err / bar.clamp_min(1e-300))[bad].max()):.3g}"


# ------------------------------------------------------------------------------------------------------------- A
PLANTS = ("x0", "c0", "tiny_x", "x_eq_c", "antiparallel", "mag_1e-20", "mag_1e6")


def _vq_case(H, N, d, dtype, seed):
    """x (H,N,d) in `dtype`, codebook (H,K,d) fp32 and indices with the planted rows 0..6 on codes 0..6 of each head."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    K = 16
    x = torch.randn(H, N, d, generator=g, device=DEV).to(dtype)
    cb = torch.randn(H, K, d, generator=g, device=DEV)
    idx = torch.randint(len(PLANTS), K, (H, N), generator=g, device=DEV)
    idx[:, :len(PLANTS)] = torch.arange(len(PLANTS), device=DEV)
    for h in range(H):
        x[h, 0] = 0                                          # x = 0
        cb[h, 1] = 0                                         # c = 0
        x[h, 2] = (torch.randn(d, generator=g, device=DEV) * (1e-7 / d ** 0.5)).to(dtype)   # 0 < |x| < 1e-6
        cb[h, 3] = x[h, 3].float()                           # x == c
        cb[h, 4] = -2 * x[h, 4].float()                      # u + q == 0 exactly
        if dtype == torch.float32:
            x[h, 5] *= 1e-20
            x[h, 6] *= 1e6
        cb[h, 5] *= 1e-20
        cb[h, 6] *= 1e6
    return x, cb, idx


def _mask(kind, N, seed):
    if kind == "none":
        return None
    if kind == "all_off":
        return torch.zeros(N, dtype=torch.uint8, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.rand(N, generator=g, device=DEV) >= 0.3).to(torch.uint8)


def _check_vq_kernel(x, cb, idx, gq, s, mask, what):
    from vqb200 import ops
    H, N, d = x.shape
    gl = torch.full((1,), s, device=DEV)
    got = ops.rot_commit_backward(gq, gl, x, cb, idx, mask)
    again = ops.rot_commit_backward(gq, gl, x, cb, idx, mask)
    assert torch.equal(got, again), f"{what}: two launches differ"
    live = None if mask is None else mask.bool()
    for h in range(H):
        c = cb[h][idx[h]]
        ref, bar = ref_grad(x[h].float(), c, gq[h], s, live)
        rows = torch.ones(N, dtype=torch.bool, device=DEV) if live is None else live
        assert_rows(got[h][rows], ref[rows], bar[rows], f"{what} h={h}")
        assert torch.equal(got[h][~rows], gq[h][~rows].float()), f"{what} h={h}: masked rows are not grad_q"
        if live is None or bool(live[4]):
            # the antiparallel plant: u + q is exactly 0 in fp64, so w = 0 there
            xr, cr = x[h, 4].double(), c[4].double()
            assert float((xr / xr.norm() + cr / cr.norm()).abs().max()) == 0.0
    return got


@pytest.mark.parametrize("mask_kind", ["none", "30pct_off", "all_off"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("d", [1, 3, 64, 100, 256, 512, 640, 1024])
@pytest.mark.parametrize("H", [1, 3])
def test_rot_commit_backward_matches_fp64(H, d, dtype, mask_kind):
    N = 37
    x, cb, idx = _vq_case(H, N, d, dtype, seed=d * 7 + H)
    gq = torch.randn(H, N, d, generator=torch.Generator(device=DEV).manual_seed(d), device=DEV)
    _check_vq_kernel(x, cb, idx, gq, 2.0 / (N * d) * 3.0, _mask(mask_kind, N, d), f"H={H} d={d} {dtype} {mask_kind}")


@pytest.mark.parametrize("d", [3, 256, 640])
def test_rot_commit_backward_without_loss_or_output_gradient(d):
    """want_loss off (coefficient 0), no gradient of the output (zeros), and a gradient view one float off alignment."""
    H, N = 3, 41
    x, cb, idx = _vq_case(H, N, d, torch.float32, seed=d)
    gq = torch.randn(H, N, d, generator=torch.Generator(device=DEV).manual_seed(d + 1), device=DEV)
    m = _mask("30pct_off", N, d)
    _check_vq_kernel(x, cb, idx, gq, 0.0, m, f"d={d} no loss")
    got = _check_vq_kernel(x, cb, idx, torch.zeros_like(gq), 3.0 / (N * d), m, f"d={d} no grad_q")
    live = m.bool()
    st = (3.0 / (N * d)) * (x - torch.stack([cb[h][idx[h]] for h in range(H)]))
    assert torch.allclose(got[:, live], st[:, live], rtol=1e-6, atol=0), "g = 0 must leave the commitment term alone"
    buf = torch.randn(H * N * d + 1, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
    odd = buf[1:].view(H, N, d)
    assert odd.data_ptr() % 16 == 4
    _check_vq_kernel(x, cb, idx, odd, 1.0 / (N * d), m, f"d={d} misaligned grad_q")


# ------------------------------------------------------------------------------------------------------------- B
def _rvq_replay(x, books, idxs, live):
    """fp32 residuals r_l and codes c_l exactly as the level kernels form them (training levels)."""
    r, rs, cs = x, [], []
    for cb, ix in zip(books, idxs):
        c = cb[ix]
        q = torch.where(live[:, None], r + (c - r), r)
        rs.append(r)
        cs.append(c)
        r = r - q
    return rs, cs


def rvq_ref(x, books, idxs, g, coefs, live):
    """fp64 sum over the levels of the rotation transport and commitment term, and the summed per-level bar."""
    rs, cs = _rvq_replay(x, books, idxs, live)
    tot = torch.zeros(x.shape, dtype=torch.float64, device=DEV)
    bar = torch.zeros(x.shape[0], dtype=torch.float64, device=DEV)
    for r, c, s in zip(rs, cs, coefs):
        gr, b = ref_grad(r, c, g, s, live)
        tot += gr
        bar += torch.where(live, b, torch.zeros_like(b))
    return tot, bar


@pytest.mark.parametrize("mask_kind", ["none", "30pct_off"])
@pytest.mark.parametrize("d", [4, 128, 132, 256, 260, 512])
@pytest.mark.parametrize("Q", [2, 8, 32])
def test_rvq_backward_rot_matches_fp64(Q, d, mask_kind):
    from vqb200 import ops
    N, K = 300, 32
    gen = torch.Generator(device=DEV).manual_seed(Q * 1000 + d)
    x = torch.randn(N, d, generator=gen, device=DEV)
    books = [torch.randn(K, d, generator=gen, device=DEV) * (0.7 / 1.3 ** l) for l in range(Q)]
    idxs = [torch.randint(0, K, (N,), generator=gen, device=DEV) for _ in range(Q)]
    g = torch.randn(N, d, generator=gen, device=DEV)
    coefs = [(l + 1) * 2.0 / (N * d) for l in range(Q)]
    mask = _mask(mask_kind, N, d)
    live = torch.ones(N, dtype=torch.bool, device=DEV) if mask is None else mask.bool()
    coef = torch.tensor(coefs, device=DEV)
    for g_out in (g, None):
        got = ops.rvq_backward_rot(x, books, idxs, [True] * Q, coef, g_out, mask)
        assert torch.equal(got, ops.rvq_backward_rot(x, books, idxs, [True] * Q, coef, g_out, mask)), "repeatability"
        ref, bar = rvq_ref(x, books, idxs, g if g_out is not None else torch.zeros_like(g), coefs, live)
        assert_rows(got[live], ref[live], bar[live], f"Q={Q} d={d} {mask_kind} g_out={g_out is not None}")
        if not bool(live.all()):
            gm = g[~live] * Q if g_out is not None else torch.zeros_like(g[~live])
            assert torch.allclose(got[~live], gm, rtol=1e-6, atol=0), "masked rows: every level is the identity"


# ------------------------------------------------------------------------------------------------------------- C
def _vq(rotation, seed=0, **kw):
    from vqb200 import CodebookParams, VectorQuantize
    torch.manual_seed(seed)
    dim = kw.pop("dim", 64)
    cp = dict(dim=dim, codebook_size=kw.pop("codebook_size", 128), threshold_ema_dead_code=kw.pop("threshold", 0))
    cp.update(kw.pop("cp", {}))
    vq = VectorQuantize(dim=dim, codebook_params=CodebookParams(**cp), **kw).to(DEV)
    vq.rotation_trick = rotation
    return vq


VQ_CONFIGS = {
    "euclid": dict(),
    "cosine": dict(cp=dict(use_cosine_sim=True, transform_input="l2norm", weights_regularization="l2norm")),
    "heads_shared": dict(dim=96, heads=3, codebook_dim=32),
    "heads_separate": dict(dim=96, heads=3, codebook_dim=32, separate_codebook_per_head=True),
    "masked": dict(),
    "image_channel_first": dict(channel_last=False),
    "expiry": dict(threshold=2),
}


def _vq_inputs(name, seed):
    gen = torch.Generator().manual_seed(seed)
    if name == "image_channel_first":
        x = torch.randn(2, 64, 6, 7, generator=gen)
        mask = None
    else:
        dim = VQ_CONFIGS[name].get("dim", 64)
        x = torch.randn(3, 50, dim, generator=gen)
        mask = (torch.rand(3, 50, generator=gen) >= 0.3).to(DEV) if name == "masked" else None
    return x.to(DEV), torch.randn(x.shape, generator=gen).to(DEV), mask


def _vq_steps(rotation, name, steps=2):
    vq = _vq(rotation, **dict(VQ_CONFIGS[name])).train()
    outs = []
    for s in range(steps):
        x, w, mask = _vq_inputs(name, 100 + s)
        x.requires_grad_(True)
        torch.manual_seed(7 + s)
        q, ind, loss = vq(x, mask=mask)
        ((q * w).sum() + loss.sum() * 3.0).backward()
        outs.append((q.detach(), ind, loss.detach(), x.grad))
    cb = vq._codebook
    return outs, (cb.embeddings.detach().clone(), cb.embed_avg.clone(), cb.cluster_size.clone())


@pytest.mark.parametrize("name", list(VQ_CONFIGS))
def test_vq_forward_is_bitwise_the_straight_through_forward(name):
    a, ba = _vq_steps(True, name)
    b, bb = _vq_steps(False, name)
    for s, (oa, ob) in enumerate(zip(a, b)):
        for what, u, v in zip(("quantize", "indices", "loss"), oa[:3], ob[:3]):
            assert torch.equal(u, v), f"{name} step {s}: {what} differs"
    for what, u, v in zip(("embeddings", "embed_avg", "cluster_size"), ba, bb):
        assert torch.equal(u, v), f"{name}: {what} differs after 2 steps"
    assert not torch.equal(a[0][3], b[0][3]), f"{name}: the input gradient did not change"


def _rows_and_back(vq, x):
    """x (B, n, dim) -> the codebook-side rows (H, N, dh), and the inverse map for a gradient of that shape."""
    B, n, dim = x.shape
    H = vq.heads
    dh = dim // H
    if H == 1:
        return x.reshape(1, B * n, dim), lambda t: t.reshape(B, n, dim)
    xh = x.reshape(B, n, H, dh)
    if vq.separate_codebook_per_head:
        return xh.permute(2, 0, 1, 3).reshape(H, B * n, dh), \
            lambda t: t.reshape(H, B, n, dh).permute(1, 2, 0, 3).reshape(B, n, dim)
    return xh.permute(0, 2, 1, 3).reshape(1, B * H * n, dh), \
        lambda t: t.reshape(B, H, n, dh).permute(0, 2, 1, 3).reshape(B, n, dim)


def _index_rows(vq, ind):
    if vq.heads == 1:
        return ind.reshape(1, -1)
    B, n, H = ind.shape
    return ind.permute(2, 0, 1).reshape(H, -1) if vq.separate_codebook_per_head else ind.permute(0, 2, 1).reshape(1, -1)


@pytest.mark.parametrize("name", ["euclid", "masked", "heads_shared", "heads_separate"])
def test_vq_input_gradient_matches_fp64(name):
    """Driven by the module's own indices and the codebook it gathered from (a copy taken before the EMA step)."""
    vq = _vq(True, **dict(VQ_CONFIGS[name])).train()
    x, w, mask = _vq_inputs(name, 3)
    pre = vq._codebook.embeddings.detach().clone()
    x.requires_grad_(True)
    q, ind, loss = vq(x, mask=mask)
    ((q * w).sum() + loss.sum() * 3.0).backward()
    rows, back = _rows_and_back(vq, x.detach())
    grow, _ = _rows_and_back(vq, w)
    irow = _index_rows(vq, ind)
    H, N, dh = rows.shape
    live = None
    if mask is not None:
        live = vq._codebook._expand_mask(mask, N).bool()
    used = H * (N if live is None else int(live.sum()))         # the commitment MSE averages over all heads' rows
    s = 3.0 * vq.commitment_weight * 2.0 / (used * dh)
    ref, got_rows = [], _rows_and_back(vq, x.grad)[0]
    for h in range(H):
        c = pre[h][irow[h]]
        r, bar = ref_grad(rows[h], c, grow[h], s, live)
        keep = torch.ones(N, dtype=torch.bool, device=DEV) if live is None else live
        assert_rows(got_rows[h][keep], r[keep], bar[keep], f"{name} h={h}")
        ref.append(r)
    if mask is not None:
        # masked positions return the input itself (reference vector_quantize_pytorch.py:415-418): gradient w
        assert torch.equal(x.grad[~mask], w[~mask])


def test_vq_cosine_input_gradient_matches_fp64():
    """Cosine codebook: the rows the rotation sees are l2-normalised; the reference differentiates through F.normalize."""
    vq = _vq(True, **dict(VQ_CONFIGS["cosine"])).train()
    x, w, _ = _vq_inputs("cosine", 4)
    pre = vq._codebook.embeddings.detach().clone()
    x.requires_grad_(True)
    q, ind, loss = vq(x)
    ((q * w).sum() + loss.sum() * 3.0).backward()
    xd = x.detach().reshape(-1, x.shape[-1]).double().requires_grad_(True)
    e = F.normalize(xd, dim=-1, eps=1e-12)
    c = pre[0][ind.reshape(-1)].double()
    N, d = e.shape
    obj = (rotate_to(e, c) * w.reshape(N, d).double()).sum() + 3.0 * ((e - c) ** 2).mean()
    (ref,) = torch.autograd.grad(obj, xd)
    err = (x.grad.reshape(N, d).double() - ref).abs().max() / ref.abs().max()
    assert float(err) <= 1e-5, float(err)


def test_learnable_codebook_gets_the_straight_through_codebook_gradient():
    res = {}
    for rot in (True, False):
        vq = _vq(rot, cp=dict(learnable_codebook=True, ema_update=False)).train()
        x, w, mask = _vq_inputs("masked", 5)
        x.requires_grad_(True)
        q, ind, loss = vq(x, mask=mask)
        ((q * w).sum() + loss.sum() * 3.0).backward()
        res[rot] = (vq._codebook.embeddings.grad.clone(), x.grad.clone(), q.detach(), ind)
    assert torch.equal(res[True][0], res[False][0]), "codebook gradient changed"
    assert torch.equal(res[True][2], res[False][2]) and torch.equal(res[True][3], res[False][3])
    assert not torch.equal(res[True][1], res[False][1])


def test_sync_update_v_scales_the_rotated_gradient():
    from vqb200 import CodebookParams, VectorQuantize
    grads = {}
    for v in (0.0, 0.5):
        torch.manual_seed(0)
        vq = VectorQuantize(dim=64, codebook_params=CodebookParams(dim=64, codebook_size=128, learnable_codebook=True,
                                                                   ema_update=False, threshold_ema_dead_code=0),
                            commitment_weight=0.0, sync_update_v=v).to(DEV).train()
        vq.rotation_trick = True
        x, w, _ = _vq_inputs("euclid", 6)
        x.requires_grad_(True)
        q, _, _ = vq(x)
        (q * w).sum().backward()
        grads[v] = x.grad
    assert torch.allclose(grads[0.5], grads[0.0] * 1.5, rtol=1e-6, atol=1e-7)


# ------------------------------------------------------------------------------------------------ ResidualVQ
def _rvq(d, Q, rotation, fused, seed=0, **kw):
    from vqb200 import CodebookParams, ResidualVQ
    torch.manual_seed(0)
    K = 64
    rvq = ResidualVQ(dim=d, num_quantizers=Q, rotation_trick=rotation,
                     codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0), **kw).to(DEV)
    gen = torch.Generator().manual_seed(seed)
    for li, layer in enumerate(rvq.layers):
        c = torch.randn(1, K, d, generator=gen) * (0.6 / 1.3 ** li)
        cb = layer._codebook
        with torch.no_grad():
            cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0)
        cb.invalidate_cache()
    rvq.use_fused_levels = fused
    return rvq


def _rvq_inputs(d, seed, B=2, n=150):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, n, d, generator=gen)
    w = torch.randn(B, n, d, generator=gen)
    mask = torch.rand(B, n, generator=gen) >= 0.3
    return x.to(DEV), w.to(DEV), mask.to(DEV)


@pytest.fixture
def calls(monkeypatch):
    from vqb200 import ops
    seen = {"rvq_backward_rot": 0, "rvq_backward": 0, "rot_commit_backward": 0}
    for name in seen:
        real = getattr(ops, name)

        def wrap(*a, _real=real, _name=name, **k):
            seen[_name] += 1
            return _real(*a, **k)
        monkeypatch.setattr(ops, name, wrap)
    return seen


def _rvq_step(rvq, x0, w, mask, freeze=False, seed=None):
    x = x0.clone().requires_grad_(True)
    torch.manual_seed(7)
    kw = {} if seed is None else {"rand_quantize_dropout_fixed_seed": seed}
    q, ind, losses = rvq(x, mask=mask, freeze_codebook=freeze, **kw)
    Q = losses.shape[-1]
    ((q * w).sum() + (losses * torch.arange(1, Q + 1, device=DEV)).sum() * 3.0).backward()
    return q.detach(), ind, losses.detach(), x.grad


def _rvq_check(rvq, x, w, mask, books, got, what, levels=None):
    """got (B,n,d) against the fp64 sum over the levels driven by the module's indices and pre-update codebooks."""
    q, ind, losses, grad = got
    d = x.shape[-1]
    N = x.shape[0] * x.shape[1]
    Q = len(books) if levels is None else levels
    live = torch.ones(N, dtype=torch.bool, device=DEV) if mask is None else mask.reshape(-1)
    used = int(live.sum())
    coefs = [3.0 * (l + 1) * 2.0 / (used * d) for l in range(Q)]
    ref, bar = rvq_ref(x.reshape(N, d), [b[0] for b in books[:Q]], [ind.reshape(N, -1)[:, l] for l in range(Q)],
                       w.reshape(N, d), coefs, live)
    assert_rows(grad.reshape(N, d)[live], ref[live], bar[live], what)


@pytest.mark.parametrize("mask", [False, True])
@pytest.mark.parametrize("Q", [8, 33])
@pytest.mark.parametrize("d", [64, 132, 512])
def test_fused_rvq_rotation_equals_generic_loop(d, Q, mask, calls):
    x, w, m = _rvq_inputs(d, d + Q)
    m = m if mask else None
    res = {}
    for fused in (True, False):
        rvq = _rvq(d, Q, True, fused, seed=d).train()
        books = [l._codebook.embeddings.detach().clone() for l in rvq.layers]
        before = calls["rvq_backward_rot"]
        res[fused] = _rvq_step(rvq, x, w, m)
        ran = calls["rvq_backward_rot"] - before
        assert ran == (1 if fused and Q <= 32 else 0), f"rvq_backward_rot ran {ran} times (fused={fused}, Q={Q})"
        _rvq_check(rvq, x, w, m, books, res[fused], f"d={d} Q={Q} mask={mask} fused={fused}")
    assert torch.equal(res[True][0], res[False][0]) and torch.equal(res[True][1], res[False][1])
    # the two loops reduce the commitment loss in different orders (as with straight-through)
    la, lb = res[True][2].double(), res[False][2].double()
    assert float((la - lb).abs().max() / lb.abs().max()) <= 1e-6, (la, lb)
    assert calls["rvq_backward"] == 0


def test_fused_rvq_rotation_with_frozen_codebook(calls):
    d, Q = 132, 8
    x, w, m = _rvq_inputs(d, 9)
    for fused in (True, False):
        rvq = _rvq(d, Q, True, fused, seed=3).train()
        books = [l._codebook.embeddings.detach().clone() for l in rvq.layers]
        got = _rvq_step(rvq, x, w, m, freeze=True)
        _rvq_check(rvq, x, w, m, books, got, f"freeze fused={fused}")
        for l, b in zip(rvq.layers, books):
            assert torch.equal(l._codebook.embeddings, b)
    assert calls["rvq_backward_rot"] == 1


def test_rvq_forward_is_bitwise_the_straight_through_forward():
    d, Q = 132, 4
    res = {}
    for rot in (True, False):
        rvq = _rvq(d, Q, rot, True, seed=1).train()
        outs = []
        for s in range(2):
            x, w, m = _rvq_inputs(d, 40 + s)
            outs.append(_rvq_step(rvq, x, w, m if s else None))
        res[rot] = (outs, [(l._codebook.embeddings.clone(), l._codebook.embed_avg.clone(),
                            l._codebook.cluster_size.clone()) for l in rvq.layers])
    for (oa, ob) in zip(res[True][0], res[False][0]):
        for a, b in zip(oa[:3], ob[:3]):
            assert torch.equal(a, b)
        assert not torch.equal(oa[3], ob[3])
    for la, lb in zip(res[True][1], res[False][1]):
        for a, b in zip(la, lb):
            assert torch.equal(a, b)


def test_mixed_flags_take_the_generic_loop(calls):
    d, Q = 64, 3
    rvq = _rvq(d, Q, True, True, seed=2).train()
    rvq.layers[1].rotation_trick = False
    x, w, _ = _rvq_inputs(d, 5)
    _rvq_step(rvq, x, w, None)
    assert calls["rvq_backward_rot"] == 0 and calls["rvq_backward"] == 0
    assert calls["rot_commit_backward"] == 2


def test_quantize_dropout_runs_the_generic_loop(calls):
    d, Q, seed = 64, 6, 1234
    rvq = _rvq(d, Q, True, True, seed=4, quantize_dropout=True).train()
    books = [l._codebook.embeddings.detach().clone() for l in rvq.layers]
    x, w, _ = _rvq_inputs(d, 6)
    got = _rvq_step(rvq, x, w, None, seed=seed)
    kept = random.Random(seed).randrange(0, Q) + 1
    assert calls["rvq_backward_rot"] == 0 and calls["rot_commit_backward"] == kept
    q, ind, losses, grad = got
    _rvq_check(rvq, x, w, None, books, (q, ind[..., :kept], losses, grad), "quantize dropout", levels=kept)


def test_grouped_rvq_rotation_fused_equals_generic(calls):
    from vqb200 import CodebookParams, GroupedResidualVQ
    d, G, Q = 128, 2, 4
    x, w, _ = _rvq_inputs(d, 8)
    res = {}
    for fused in (True, False):
        torch.manual_seed(0)
        g = GroupedResidualVQ(dim=d, groups=G, num_quantizers=Q, rotation_trick=True,
                              codebook_params=CodebookParams(dim=d // G, codebook_size=64,
                                                             threshold_ema_dead_code=0)).to(DEV).train()
        for r in g.rvqs:
            r.use_fused_levels = fused
        xx = x.clone().requires_grad_(True)
        torch.manual_seed(7)
        q, ind, losses = g(xx)
        ((q * w).sum() + losses.sum() * 3.0).backward()
        res[fused] = (q.detach(), ind, losses.detach(), xx.grad)
    assert torch.equal(res[True][0], res[False][0]) and torch.equal(res[True][1], res[False][1])
    err = (res[True][3] - res[False][3]).abs().max() / res[False][3].abs().max()
    assert float(err) <= 1e-5, float(err)
    assert calls["rvq_backward_rot"] == G and calls["rot_commit_backward"] == G * Q
