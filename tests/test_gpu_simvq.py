"""`SimVQ` / `ResidualSimVQ` on the GPU against the fp64 autograd statement of the contract (tests/simvq_ref.py), with
the indices fixed to the library's search.

Per forward: the indices equal `ops.search` on the same C' and the fp64 nearest code outside a 1e-6 relative top-2
distance gap; `quantized` is the straight-through value fl(x + fl(C'[idx] - x)) bit for bit; the loss is within 1e-5
relative.  Input gradient, per row: |got - ref|_2 <= 1e-5 f (lambda |g|_2 + |coef| |x - c|_2) as in
tests/test_gpu_rotation_trick.py (lambda = f = 1 for straight-through; summed over the levels of a stack), plus one
rounding of the reference for a 16-bit input, whose gradient is returned in its own dtype.  Transform gradients: the
largest error within 1e-5 of the largest reference entry."""
import pytest
import torch

import simvq_ref

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5
BETA, CW, G_LOSS = 0.3, 1.5, 3.0


def row_bar(x, c, g, coef, rotation):
    x, c, g = x.double(), c.double(), g.double()
    if not rotation:
        return TOL * (g.norm(dim=-1) + abs(coef) * (x - c).norm(dim=-1))
    nx, nc = x.norm(dim=-1), c.norm(dim=-1)
    upq = (x / nx.clamp_min(1e-6)[:, None] + c / nc.clamp_min(1e-6)[:, None]).norm(dim=-1)
    f = torch.where(upq > 0, (1 / upq).clamp_min(1.0), torch.ones_like(upq))
    lam = nc / nx.clamp_min(1e-6)
    return TOL * f * (lam * g.norm(dim=-1) + abs(coef) * (x - c).norm(dim=-1))


def assert_rows(got, ref, bar, what):
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite gradient"
    if got.dtype != torch.float32:
        bar = bar + 2.0 ** -8 * ref.norm(dim=-1)          # the gradient is rounded to the input's 16-bit dtype
    err = (got.double() - ref).norm(dim=-1)
    bad = err > bar
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} rows over the bar, worst err/bar " \
                                f"{float((err / bar.clamp_min(1e-300))[bad].max()):.3g}"


def assert_close(got, ref, what):
    err = float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))
    assert err <= TOL, f"{what}: relative error {err:.3g}"


def _simvq(d, K, d_f=None, rotation=True, seed=0, **kw):
    from vqb200 import SimVQ
    torch.manual_seed(seed)
    return SimVQ(d, K, rotation_trick=rotation, frozen_codebook_dim=d_f, commitment_weight=CW,
                 input_to_quantize_commit_loss_weight=BETA, **kw).to(DEV).train()


def _inputs(shape, scale, dtype, seed):
    """Latents on the scale of the codes (entries of C' have variance 1 / (3 d_f) at the default init), and the
    output gradient."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = (torch.randn(shape, generator=g, device=DEV) * scale).to(dtype)
    return x, torch.randn(shape, generator=g, device=DEV)


def _linear_books(mods):
    return lambda ps: [torch.nn.functional.linear(m.frozen_codebook.double(), p) for m, p in zip(mods, ps)]


def _check_indices(rows, codebook, ind, what):
    from vqb200 import ops
    cb = codebook[None].contiguous()
    idx, _, _ = ops.search(rows[None].contiguous(), cb, ops.prepare_codebook(cb, False), False)
    assert torch.equal(ind, idx[0]), f"{what}: indices differ from ops.search on the same codebook"
    best, gap = simvq_ref.fp64_argmin_and_gap(rows.float(), codebook)
    bad = (ind != best) & (gap >= 1e-6)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} rows off the fp64 nearest code outside the tie window"


def _step(vq, x, w):
    xg = x.clone().requires_grad_(True)
    q, ind, loss = vq(xg)
    ((q * w).sum() + G_LOSS * loss).backward()
    return q.detach(), ind, loss.detach(), xg.grad


def _check_simvq(vq, x, w, params, books, what):
    d = vq.dim
    q, ind, loss, gx = _step(vq, x, w)
    rows, ind_r = x.reshape(-1, d), ind.reshape(-1)
    cb = vq.codebook.detach()
    _check_indices(rows, cb, ind_r, what)
    xf = rows.float()
    assert torch.equal(q.reshape(-1, d), xf + (cb[ind_r] - xf)), f"{what}: not the straight-through value"
    _, losses, gref, pref = simvq_ref.grads(rows, params, books, [ind_r], BETA, CW, vq.rotation_trick,
                                            w.reshape(-1, d), [G_LOSS])
    assert abs(float(loss) - float(losses[0])) <= TOL * abs(float(losses[0])), (what, float(loss), float(losses[0]))
    N = rows.shape[0]
    coef = G_LOSS * CW * BETA * 2.0 / (N * d)
    assert gx.dtype == x.dtype
    assert_rows(gx.reshape(-1, d), gref, row_bar(xf, cb[ind_r], w.reshape(-1, d), coef, vq.rotation_trick), what)
    for p, r in zip(params, pref):
        assert_close(p.grad, r, f"{what}: transform gradient")
    return q, ind, loss


# (d, d_f, K, B, n): every width of the fused gather + sums pass and beside it, d_f != d, K 512 / 8192, N = 1 and
# ragged N
CASES = [(64, None, 512, 3, 347), (64, 32, 8192, 1, 1), (96, None, 512, 2, 301), (96, 128, 512, 1, 1),
         (256, None, 8192, 4, 257), (256, 64, 512, 3, 347), (512, None, 512, 2, 333), (640, None, 512, 1, 1),
         (640, 256, 8192, 2, 129)]


@pytest.mark.parametrize("rotation", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "d{}_df{}_K{}_N{}".format(c[0], c[1], c[2], c[3] * c[4]))
def test_simvq_matches_fp64(case, dtype, rotation):
    d, d_f, K, B, n = case
    vq = _simvq(d, K, d_f, rotation, seed=d + K)
    x, w = _inputs((B, n, d), (3 * (d_f or d)) ** -0.5, dtype, seed=d * 3 + n)
    _check_simvq(vq, x, w, [vq.code_transform.weight], _linear_books([vq]), f"d={d} d_f={d_f} K={K} N={B * n}")


def test_simvq_custom_transform():
    mlp = torch.nn.Sequential(torch.nn.Linear(48, 128), torch.nn.SiLU(), torch.nn.Linear(128, 256)).to(DEV)
    vq = _simvq(256, 1024, 48, True, codebook_transform=mlp)
    assert vq.code_transform is mlp
    x, w = _inputs((2, 300, 256), 0.05, torch.float32, seed=5)
    ps = list(mlp.parameters())

    def books(p):
        h = torch.nn.functional.silu(torch.nn.functional.linear(vq.frozen_codebook.double(), p[0], p[1]))
        return [torch.nn.functional.linear(h, p[2], p[3])]
    _check_simvq(vq, x, w, ps, books, "custom transform")


@pytest.mark.parametrize("d", [64, 96])
def test_simvq_channel_first_eval_and_no_grad(d):
    vq = _simvq(d, 512, rotation=True, channel_first=True)
    x, w = _inputs((2, d, 9, 11), (3 * d) ** -0.5, torch.float32, seed=d)
    q, ind, loss = vq(x)
    assert q.shape == x.shape and ind.shape == (2, 9, 11)
    rows = x.movedim(1, -1).reshape(-1, d)
    cb = vq.codebook.detach()
    _check_indices(rows, cb, ind.reshape(-1), "channel_first")
    assert torch.equal(q, (rows + (cb[ind.reshape(-1)] - rows)).reshape(2, 9, 11, d).movedim(-1, 1))
    assert torch.equal(vq.get_output_from_indices(ind), cb[ind].movedim(-1, 1))
    # the same values with no gradient: eval mode, and a training-mode forward under no_grad
    for mode in ("eval", "no_grad"):
        vq.train(mode != "eval")
        with torch.set_grad_enabled(mode != "no_grad"):
            q2, ind2, loss2 = vq(x.clone().requires_grad_(True))
        assert not q2.requires_grad and not loss2.requires_grad
        assert torch.equal(q2, q) and torch.equal(ind2, ind), mode
        assert abs(float(loss2) - float(loss)) <= 1e-6 * abs(float(loss)), mode
    # the channel-first gradient is the channel-last one moved back
    vq.train()
    xc = x.clone().requires_grad_(True)
    qc, _, lc = vq(xc)
    ((qc * w).sum() + G_LOSS * lc).backward()
    vq_last = _simvq(d, 512, rotation=True)
    xl = x.movedim(1, -1).contiguous().requires_grad_(True)
    ql, _, ll = vq_last(xl)
    ((ql * w.movedim(1, -1)).sum() + G_LOSS * ll).backward()
    assert torch.equal(xc.grad, xl.grad.movedim(-1, 1))
    assert torch.equal(vq.code_transform.weight.grad, vq_last.code_transform.weight.grad)


# ----------------------------------------------------------------------------------------------- ResidualSimVQ
def _rsim(d, Q, rotation, fused, K=512):
    from vqb200 import ResidualSimVQ
    torch.manual_seed(0)
    r = ResidualSimVQ(d, Q, K, rotation_trick=rotation, commitment_weight=CW,
                      input_to_quantize_commit_loss_weight=BETA).to(DEV).train()
    r.use_fused_levels = fused
    return r


@pytest.fixture
def calls(monkeypatch):
    from vqb200 import ops
    seen = {"rvq_level_ema": 0, "rvq_backward_rot": 0, "rvq_backward": 0}
    for name in seen:
        real = getattr(ops, name)

        def wrap(*a, _real=real, _name=name, **k):
            seen[_name] += 1
            return _real(*a, **k)
        monkeypatch.setattr(ops, name, wrap)
    return seen


def _rsim_step(rsim, x, w):
    xg = x.clone().requires_grad_(True)
    q, ind, losses = rsim(xg)
    Q = losses.shape[-1]
    ((q * w).sum() + (losses * torch.arange(1, Q + 1, device=DEV)).sum() * G_LOSS).backward()
    return q.detach(), ind, losses.detach(), xg.grad, [l.code_transform.weight.grad.clone() for l in rsim.layers]


def _check_rsim_fp64(rsim, x, w, got, what):
    q, ind, losses, gx, gws = got
    d, Q = rsim.dim, len(rsim.layers)
    rows, wr = x.reshape(-1, d), w.reshape(-1, d)
    N = rows.shape[0]
    idxs = [ind.reshape(N, Q)[:, l] for l in range(Q)]
    g_losses = [G_LOSS * (l + 1) for l in range(Q)]
    _, lref, gref, wref = simvq_ref.grads(rows, [l.code_transform.weight for l in rsim.layers],
                                          _linear_books(rsim.layers), idxs, BETA, CW, rsim.layers[0].rotation_trick,
                                          wr, g_losses)
    assert_close(losses[0], lref, f"{what}: losses")
    r, bar = rows.float(), torch.zeros(N, dtype=torch.float64, device=DEV)
    for l, layer in enumerate(rsim.layers):
        cb = layer.codebook.detach()
        c = cb[idxs[l]]
        _check_indices(r, cb, idxs[l], f"{what} level {l}")
        bar += row_bar(r, c, wr, g_losses[l] * CW * BETA * 2.0 / (N * d), layer.rotation_trick)
        r = r - (r + (c - r))
    assert_rows(gx.reshape(N, d), gref, bar, f"{what}: input gradient")
    for l, (a, b) in enumerate(zip(gws, wref)):
        assert_close(a, b, f"{what}: transform gradient of level {l}")


@pytest.mark.parametrize("rotation", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Q", [2, 4, 8])
@pytest.mark.parametrize("d", [64, 512])
def test_residual_simvq_fused_equals_generic(d, Q, dtype, rotation, calls):
    x, w = _inputs((3, 211, d), (3 * d) ** -0.5, dtype, seed=d + Q)
    res = {}
    for fused in (True, False):
        rsim = _rsim(d, Q, rotation, fused)
        before = dict(calls)
        res[fused] = _rsim_step(rsim, x, w)
        name = "rvq_backward_rot" if rotation else "rvq_backward"
        assert calls[name] - before[name] == int(fused) and calls["rvq_level_ema"] - before["rvq_level_ema"] == \
            Q * int(fused), calls
        _check_rsim_fp64(rsim, x, w, res[fused], f"d={d} Q={Q} {dtype} fused={fused}")
    a, b = res[True], res[False]
    assert a[0].shape == x.shape and a[1].shape == (3, 211, Q) and a[2].shape == (1, Q)
    for what, u, v in zip(("quantized", "indices", "losses"), a[:3], b[:3]):
        assert torch.equal(u, v), f"{what}: fused and generic loops differ"
    ga, gb = a[3].double(), b[3].double()
    if dtype == torch.float32:
        assert_close(ga, gb, "input gradient, fused against generic")
    else:
        # the fused gradient is rounded to bf16 once; autograd through the generic loop rounds each level's share and
        # adds them in bf16, up to Q + 1 roundings of a row's size (both loops are held to fp64 above)
        err, size = (ga - gb).reshape(-1, d).norm(dim=-1), gb.reshape(-1, d).norm(dim=-1)
        bad = err > (Q + 1) * 2.0 ** -8 * size
        assert not bool(bad.any()), f"input gradient, fused against generic: {int(bad.sum())} rows apart"
    for u, v in zip(a[4], b[4]):
        assert_close(u, v.double(), "transform gradient, fused against generic")


def test_residual_simvq_eval_no_grad_and_fallbacks(calls):
    d = 256
    x, w = _inputs((2, 150, d), (3 * d) ** -0.5, torch.float32, seed=11)
    outs = {}
    for fused in (True, False):
        rsim = _rsim(d, 4, True, fused)
        train_q, train_ind, train_losses, _, _ = _rsim_step(rsim, x, w)
        for mode in ("eval", "no_grad"):
            rsim.train(mode != "eval")
            with torch.set_grad_enabled(mode != "no_grad"):
                q, ind, losses = rsim(x.clone().requires_grad_(True))
            assert not q.requires_grad
            # the fused loop without the sums: the loss is reduced in another order than the training pass's
            assert torch.equal(q, train_q) and torch.equal(ind, train_ind), mode
            assert_close(losses, train_losses.double(), mode)
            outs[(fused, mode)] = (q, ind)
        codes = rsim.get_codes_from_indices(train_ind)
        assert codes.shape == (4, 2, 150, d)
        assert torch.equal(rsim.get_output_from_indices(train_ind), codes.sum(0))
    before = calls["rvq_level_ema"]
    # widths the level kernels do not take, and a single level: the generic loop
    for d, Q in ((96, 3), (256, 1)):
        rsim = _rsim(d, Q, True, True)
        x, w = _inputs((2, 150, d), (3 * d) ** -0.5, torch.float32, seed=d)
        _check_rsim_fp64(rsim, x, w, _rsim_step(rsim, x, w), f"fallback d={d} Q={Q}")
    assert calls["rvq_level_ema"] == before and calls["rvq_backward_rot"] == 1


def test_residual_simvq_channel_first():
    d = 64
    x, w = _inputs((2, d, 8, 8), (3 * d) ** -0.5, torch.float32, seed=3)
    from vqb200 import ResidualSimVQ
    torch.manual_seed(0)
    rsim = ResidualSimVQ(d, 3, 512, channel_first=True).to(DEV).train()
    q, ind, losses = rsim(x)
    assert q.shape == x.shape and ind.shape == (2, 8, 8, 3) and losses.shape == (1, 3)
    assert torch.equal(rsim.get_output_from_indices(ind), rsim.get_codes_from_indices(ind).sum(0).movedim(-1, 1))
    torch.manual_seed(0)
    last = ResidualSimVQ(d, 3, 512).to(DEV).train()
    q2, ind2, losses2 = last(x.movedim(1, -1).contiguous())
    assert torch.equal(q, q2.movedim(-1, 1)) and torch.equal(ind, ind2) and torch.equal(losses, losses2)


@pytest.mark.parametrize("rotation", [True, False])
def test_residual_simvq_sgd_steps_agree(rotation):
    d, Q = 256, 4
    weights = {}
    for fused in (True, False):
        rsim = _rsim(d, Q, rotation, fused)
        start = [l.code_transform.weight.detach().clone() for l in rsim.layers]
        opt = torch.optim.SGD(rsim.parameters(), lr=0.5)
        for s in range(3):
            x, w = _inputs((4, 256, d), (3 * d) ** -0.5, torch.bfloat16, seed=100 + s)
            opt.zero_grad()
            q, _, losses = rsim(x.requires_grad_(True))
            ((q * w).sum() * 1e-3 + losses.sum()).backward()
            opt.step()
        weights[fused] = [l.code_transform.weight.detach().clone() for l in rsim.layers]
        assert all(not torch.equal(a, b) for a, b in zip(weights[fused], start)), "the transforms did not move"
    for a, b in zip(weights[True], weights[False]):
        assert_close(a, b.double(), "transform after three SGD steps")
