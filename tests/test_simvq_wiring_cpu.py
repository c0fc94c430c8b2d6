"""Host logic of `SimVQ` / `ResidualSimVQ` (CPU, no library): which kernels each forward and backward calls and with
which coefficients, checked against the fp64 autograd statement of tests/simvq_ref.py.

The tensor-level wrappers of `vqb200.ops` are replaced by the plain-torch statements of tests/cpu_kernels.py plus the
ones below (the fused gather + sums pass and the rotation-trick backward ops), all counting their calls.  The kernels
themselves are tested on the GPU (tests/test_gpu_simvq.py)."""
import pytest
import torch

import cpu_kernels
import simvq_ref

CALLS = {}


def _count(name, fn):
    def wrapped(*a, **k):
        CALLS[name] = CALLS.get(name, 0) + 1
        return fn(*a, **k)
    return wrapped


def quantize_ema(x, embeddings, idx, training, want_loss, bound_ws=None):
    """vqb_quantize_ema: vqb_gather_st_loss (no mask) and vqb_ema_reduce in one pass."""
    q, loss = cpu_kernels.gather_st_loss(x, embeddings, idx, None, training, want_loss)
    return q, loss, cpu_kernels.ema_reduce(x, idx, None, embeddings.shape[1])


def rot_commit_backward(grad_q, g, x, embeddings, idx, mask_u8):
    """vqb_rot_commit_backward (no mask): T(grad_q) + g[0] (x - c)."""
    xf = x.detach().float()
    c = torch.stack([embeddings[h][idx[h]] for h in range(x.shape[0])], 0)
    return _transport(grad_q.float(), xf, c) + g[0] * (xf - c)


def rvq_backward_rot(x, codebooks, idxs, training, coef, g_out, mask_u8):
    """vqb_rvq_backward_rot (no mask): sum_l T_l(g_out) + coef[l] (r_l - c_l), residuals replayed from x."""
    g = g_out.float() if g_out is not None else torch.zeros_like(x)
    r, acc = x, torch.zeros_like(x)
    for l, (c, i) in enumerate(zip(codebooks, idxs)):
        cq = c[i]
        acc = acc + _transport(g, r, cq) + coef[l] * (r - cq)
        r = r - (r + (cq - r))
    return acc


def _transport(g, x, c):
    """The rotation-trick Jacobian applied to g: autograd of simvq_ref.rotate_to in the dtype given."""
    with torch.enable_grad():
        e = x.clone().requires_grad_(True)
        (out,) = torch.autograd.grad(simvq_ref.rotate_to(e, c), e, g)
    return out


@pytest.fixture()
def wired(monkeypatch):
    from vqb200 import _lib, ops, simvq
    extra = {"quantize_ema": quantize_ema, "rot_commit_backward": rot_commit_backward,
             "rvq_backward_rot": rvq_backward_rot}
    for n in cpu_kernels.REPLACED + tuple(extra):
        monkeypatch.setattr(ops, n, getattr(ops, n))
    monkeypatch.setattr(_lib, "require_device", _lib.require_device)
    cpu_kernels.install(ops, _lib)
    for n, fn in extra.items():
        setattr(ops, n, fn)
    for n in ("search", "prepare_codebook", "quantize_ema", "gather_st_loss", "ema_reduce", "st_commit_backward",
              "rot_commit_backward", "rvq_level", "rvq_level_ema", "rvq_replay_out", "rvq_backward",
              "rvq_backward_rot"):
        setattr(ops, n, _count(n, getattr(ops, n)))
    # the fused level loop needs a CUDA input; here every other condition decides
    real = simvq.ResidualSimVQ._can_fuse

    class _OnDevice:
        is_cuda = True
    monkeypatch.setattr(simvq.ResidualSimVQ, "_can_fuse", lambda self, x: real(self, _OnDevice()))
    CALLS.clear()
    return ops


def _simvq(**kw):
    from vqb200 import SimVQ
    torch.manual_seed(0)
    kw.setdefault("dim", 16)
    kw.setdefault("codebook_size", 32)
    return SimVQ(**kw).train()


def _inputs(shape, seed=1):
    gen = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=gen) * 0.3, torch.randn(shape, generator=gen)


def _linear_books(mods):
    return lambda ps: [torch.nn.functional.linear(m.frozen_codebook.double(), p) for m, p in zip(mods, ps)]


@pytest.mark.parametrize("fused_pass", [True, False])
@pytest.mark.parametrize("rotation", [True, False])
def test_simvq_step_matches_fp64(wired, rotation, fused_pass):
    ops = wired
    ops.quantize_ema_supported = lambda d: fused_pass
    vq = _simvq(rotation_trick=rotation, commitment_weight=1.5, input_to_quantize_commit_loss_weight=0.4)
    x0, w = _inputs((3, 20, 16))
    x = x0.clone().requires_grad_(True)
    q, ind, loss = vq(x)
    (q * w).sum().add(loss * 2.0).backward()
    assert q.shape == x.shape and ind.shape == (3, 20) and loss.shape == ()
    cb = vq.codebook.detach()
    assert torch.equal(ind.reshape(-1), torch.cdist(x0.reshape(-1, 16), cb).argmin(-1))
    assert torch.equal(q, x0 + (cb[ind] - x0)), "the straight-through value"
    out, losses, gx, (gw,) = simvq_ref.grads(x0.reshape(-1, 16), [vq.code_transform.weight], _linear_books([vq]),
                                             [ind.reshape(-1)], 0.4, 1.5, rotation, w.reshape(-1, 16), [2.0])
    assert torch.allclose(loss.double(), losses[0], rtol=1e-6)
    assert torch.allclose(x.grad.reshape(-1, 16).double(), gx, rtol=1e-5, atol=1e-7)
    assert torch.allclose(vq.code_transform.weight.grad.double(), gw, rtol=1e-5, atol=1e-7)
    # one gather pass; the codebook gradient reads the sums of the fused pass, or makes one sums pass in backward
    assert CALLS.get("quantize_ema", 0) == int(fused_pass) and CALLS.get("gather_st_loss", 0) == int(not fused_pass)
    assert CALLS.get("ema_reduce", 0) == int(not fused_pass)
    assert CALLS.get("rot_commit_backward", 0) == int(rotation)
    assert CALLS.get("st_commit_backward", 0) == int(not rotation)


def test_simvq_eval_no_grad_and_frozen_input(wired):
    vq = _simvq(channel_first=True, dim=8)
    x0, w = _inputs((2, 8, 5, 3))
    cb = vq.codebook.detach()
    rows = x0.movedim(1, -1).reshape(-1, 8)
    ref_ind = torch.cdist(rows, cb).argmin(-1)
    ref_q = (rows + (cb[ref_ind] - rows)).reshape(2, 5, 3, 8).movedim(-1, 1)
    for mode in ("eval", "no_grad"):
        vq.train(mode != "eval")
        with torch.set_grad_enabled(mode != "no_grad"):
            q, ind, loss = vq(x0.clone().requires_grad_(True))
        assert not q.requires_grad and not loss.requires_grad
        assert torch.equal(q, ref_q) and torch.equal(ind, ref_ind.reshape(2, 5, 3))
        assert torch.allclose(loss, 1.25 * ((cb[ref_ind] - rows) ** 2).mean())
    assert torch.equal(vq.get_output_from_indices(ind), cb[ind].movedim(-1, 1))
    assert CALLS.get("quantize_ema", 0) == 0 and CALLS["gather_st_loss"] == 2
    # a frozen encoder: the input carries no gradient, the transform still learns
    vq.train()
    q, ind, loss = vq(x0)
    loss.backward()
    assert vq.code_transform.weight.grad is not None
    assert CALLS.get("st_commit_backward", 0) == 0 and CALLS.get("rot_commit_backward", 0) == 0


def test_simvq_custom_transform_and_frozen_dim(wired):
    from vqb200 import SimVQ
    torch.manual_seed(0)
    mlp = torch.nn.Sequential(torch.nn.Linear(6, 12), torch.nn.Tanh(), torch.nn.Linear(12, 16))
    vq = SimVQ(16, 32, codebook_transform=mlp, frozen_codebook_dim=6, init_fn=lambda t: t * 2.0).train()
    assert vq.frozen_codebook.shape == (32, 6) and vq.code_transform is mlp
    x0, w = _inputs((2, 30, 16))
    x = x0.clone().requires_grad_(True)
    q, ind, loss = vq(x)
    ((q * w).sum() + loss).backward()
    ps = list(mlp.parameters())

    def books(p):
        h = torch.tanh(torch.nn.functional.linear(vq.frozen_codebook.double(), p[0], p[1]))
        return [torch.nn.functional.linear(h, p[2], p[3])]
    _, _, gx, gps = simvq_ref.grads(x0.reshape(-1, 16), ps, books, [ind.reshape(-1)], 0.25, 1.0, True,
                                    w.reshape(-1, 16), [1.0])
    assert torch.allclose(x.grad.reshape(-1, 16).double(), gx, rtol=1e-5, atol=1e-7)
    for p, g in zip(ps, gps):
        assert torch.allclose(p.grad.double(), g, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("rotation", [True, False])
def test_residual_simvq_fused_equals_generic_and_fp64(wired, rotation):
    from vqb200 import ResidualSimVQ
    ops = wired
    ops.rvq_level_ema_supported = ops.quantize_ema_supported = lambda d: True
    x0, w = _inputs((2, 25, 16), seed=4)
    res = {}
    for fused in (True, False):
        torch.manual_seed(0)
        rsim = ResidualSimVQ(dim=16, num_quantizers=3, codebook_size=32, rotation_trick=rotation,
                             commitment_weight=0.7).train()
        rsim.use_fused_levels = fused
        CALLS.clear()
        x = x0.clone().requires_grad_(True)
        q, ind, losses = rsim(x)
        ((q * w).sum() + (losses * torch.tensor([1.0, 2.0, 3.0])).sum()).backward()
        assert q.shape == x.shape and ind.shape == (2, 25, 3) and losses.shape == (1, 3)
        res[fused] = (q.detach(), ind, losses.detach(), x.grad, [l.code_transform.weight.grad for l in rsim.layers])
        backward = "rvq_backward_rot" if rotation else "rvq_backward"
        assert CALLS.get(backward, 0) == int(fused) and CALLS.get("rvq_level_ema", 0) == 3 * int(fused)
        assert CALLS.get("rvq_replay_out", 0) == int(fused) and CALLS.get("ema_reduce", 0) == 0
        assert CALLS.get("quantize_ema", 0) == 3 * int(not fused)
        out, ls, gx, gws = simvq_ref.grads(x0.reshape(-1, 16), [l.code_transform.weight for l in rsim.layers],
                                           _linear_books(rsim.layers), [ind.reshape(-1, 3)[:, l] for l in range(3)],
                                           0.25, 0.7, rotation, w.reshape(-1, 16), [1.0, 2.0, 3.0])
        assert torch.allclose(losses[0].double(), ls, rtol=1e-6)
        assert torch.allclose(x.grad.reshape(-1, 16).double(), gx, rtol=1e-5, atol=1e-7)
        for got, ref in zip(res[fused][4], gws):
            assert torch.allclose(got.double(), ref, rtol=1e-5, atol=1e-7)
    for a, b in zip(res[True][:3], res[False][:3]):
        assert torch.equal(a, b)


def test_residual_simvq_fallbacks(wired):
    from vqb200 import ResidualSimVQ
    ops = wired
    x0, _ = _inputs((2, 10, 16))
    for Q, supported in ((1, True), (3, False)):
        ops.rvq_level_ema_supported = lambda d, s=supported: s
        CALLS.clear()
        rsim = ResidualSimVQ(dim=16, num_quantizers=Q, codebook_size=32).train()
        q, ind, losses = rsim(x0.clone().requires_grad_(True))
        losses.sum().backward()
        assert CALLS.get("rvq_level_ema", 0) == 0 and CALLS.get("rvq_backward_rot", 0) == 0
        assert CALLS["rot_commit_backward"] == Q
    # eval: the fused loop without the sums or anything saved for backward
    ops.rvq_level_ema_supported = lambda d: True
    CALLS.clear()
    rsim.eval()
    q, ind, losses = rsim(x0.clone().requires_grad_(True))
    assert not q.requires_grad and CALLS["rvq_level"] == 3 and CALLS.get("rvq_level_ema", 0) == 0
    codes = rsim.get_codes_from_indices(ind)
    assert codes.shape == (3, 2, 10, 16)
    assert torch.equal(rsim.get_output_from_indices(ind), codes.sum(0))
