"""Where `VectorQuantize.rotation_trick` / `ResidualVQ(rotation_trick=True)` reaches the backward (CPU, no library).

The tensor-level wrappers of `vqb200.ops` are replaced by plain-torch statements of their C entry points
(tests/cpu_kernels.py), and the two rotation-trick backward ops by the statements below, which also count their calls.
The checks: the flag reaches `_QuantizeST.backward` from `Codebook._run` on the plain path, with the variants (gumbel
straight-through, affine) and on a sharded codebook (two Gloo ranks), and `_FusedRVQ.backward` / the generic level
loop of ResidualVQ; with the flag off neither op is called.  The kernels themselves are tested on the GPU
(tests/test_gpu_rotation_trick.py)."""
import datetime
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

import cpu_kernels

CALLS = {"rot_commit_backward": 0, "rvq_backward_rot": 0}


def transport(g, x, c):
    """Rotation-trick transport of g for rows x -> c (upstream `rotate_to`'s Jacobian)."""
    nx, nc = x.norm(dim=-1, keepdim=True), c.norm(dim=-1, keepdim=True)
    u, q = x / nx.clamp_min(1e-6), c / nc.clamp_min(1e-6)
    w = F.normalize(u + q, dim=-1, eps=1e-12)
    lam = nc / nx.clamp_min(1e-6)
    return lam * (g - 2 * (g * w).sum(-1, keepdim=True) * w + 2 * (g * q).sum(-1, keepdim=True) * u)


def rot_commit_backward(grad_q, g, x, embeddings, idx, mask_u8):
    """vqb_rot_commit_backward: T(grad_q) + g[0] (x - c) on the rows with mask != 0, grad_q on the others."""
    CALLS["rot_commit_backward"] += 1
    H = x.shape[0]
    xf, gq = x.detach().float(), grad_q.float()
    c = torch.stack([embeddings.detach()[h][idx[h]] for h in range(H)], 0).float()
    out = transport(gq, xf, c) + g[0] * (xf - c)
    if mask_u8 is None:
        return out
    return torch.where(mask_u8.bool()[None, :, None], out, gq)


def rvq_backward_rot(x, codebooks, idxs, training, coef, g_out, mask_u8):
    """vqb_rvq_backward_rot: sum_l T_l(g_out) + live coef[l] (r_l - c_l), residuals replayed from x."""
    CALLS["rvq_backward_rot"] += 1
    keep = torch.ones(x.shape[0], dtype=torch.bool) if mask_u8 is None else mask_u8.bool()
    g = g_out.float() if g_out is not None else torch.zeros_like(x)
    r, acc = x, torch.zeros_like(x)
    for l, (c, i, tr) in enumerate(zip(codebooks, idxs, training)):
        cq = c[i]
        acc = acc + torch.where(keep[:, None], transport(g, r, cq) + coef[l] * (r - cq), g)
        q = r + (cq - r) if tr else cq
        r = r - torch.where(keep[:, None], q, r)
    return acc


def _install(ops, lib, RVQ):
    cpu_kernels.install(ops, lib)
    ops.rot_commit_backward = rot_commit_backward
    ops.rvq_backward_rot = rvq_backward_rot
    CALLS.update({k: 0 for k in CALLS})
    # the fused level loop is eligible on the GPU only: let `_can_fuse` see a device tensor
    real = RVQ.ResidualVQ._can_fuse

    class _OnDevice:
        def __init__(self, t):
            self.is_cuda, self.ndim, self.requires_grad, self.shape = True, t.ndim, t.requires_grad, t.shape

    return real, lambda self, x, dropout_active: real(self, _OnDevice(x), dropout_active)


@pytest.fixture()
def wired(monkeypatch):
    from vqb200 import _lib, codebook, ops, rvq as RVQ
    for n in cpu_kernels.REPLACED + ("rot_commit_backward", "rvq_backward_rot"):
        monkeypatch.setattr(ops, n, getattr(ops, n))
    monkeypatch.setattr(_lib, "require_device", _lib.require_device)
    monkeypatch.setattr(RVQ.ResidualVQ, "_can_fuse", RVQ.ResidualVQ._can_fuse)
    monkeypatch.setattr(codebook.Codebook, "_draw_rows",
                        staticmethod(lambda n, m, device: torch.randperm(n)[:m] if n >= m else torch.randint(0, n, (m,))))
    _, can_fuse = _install(ops, _lib, RVQ)
    RVQ.ResidualVQ._can_fuse = can_fuse
    counted = {"st_commit_backward": 0, "rvq_backward": 0}
    for n in counted:
        real = getattr(ops, n)

        def wrap(*a, _real=real, _n=n):
            counted[_n] += 1
            return _real(*a)
        setattr(ops, n, wrap)
    return CALLS, counted


def _vq(rotation, **cp):
    from vqb200 import CodebookParams, VectorQuantize
    torch.manual_seed(0)
    cp.setdefault("threshold_ema_dead_code", 0)
    vq = VectorQuantize(dim=16, codebook_params=CodebookParams(dim=16, codebook_size=32, **cp)).train()
    vq.rotation_trick = rotation
    return vq


def _step(mod, x, mask=None):
    x = x.clone().requires_grad_(True)
    w = torch.randn(x.shape, generator=torch.Generator().manual_seed(3))
    q, ind, loss = mod(x, mask=mask)
    ((q * w).sum() + loss.sum() * 2.0).backward()
    return q.detach(), ind, x.grad, w


def _x(shape=(2, 40, 16), seed=1):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))


def test_run_passes_the_flag_and_the_gradient_is_the_rotation(wired):
    calls, counted = wired
    mask = torch.rand(2, 40, generator=torch.Generator().manual_seed(2)) >= 0.3
    for m in (None, mask):
        vq = _vq(True)
        pre = vq._codebook.embeddings.detach().clone()
        q, ind, grad, w = _step(vq, _x(), m)
        c = pre[0][ind.reshape(-1)]
        xf = _x().reshape(-1, 16)
        live = torch.ones(80, dtype=torch.bool) if m is None else m.reshape(-1)
        s = 2.0 * 2.0 / (int(live.sum()) * 16)
        ref = torch.where(live[:, None], transport(w.reshape(-1, 16), xf, c) + s * (xf - c), w.reshape(-1, 16))
        assert torch.allclose(grad.reshape(-1, 16), ref, rtol=1e-5, atol=1e-6)
    assert calls["rot_commit_backward"] == 2 and counted["st_commit_backward"] == 0


def test_flag_off_never_calls_the_rotation_ops(wired):
    from vqb200 import AffineParameters, CodebookParams, GumbelParams, ResidualVQ
    calls, counted = wired
    _step(_vq(False), _x())
    _step(_vq(False, use_affine=True, affine_params=AffineParameters(sync=False)), _x())
    _step(_vq(False, learnable_codebook=True, ema_update=False,
              gumbel_params=GumbelParams(straight_through=True)), _x())
    for fused in (True, False):
        torch.manual_seed(0)
        rvq = ResidualVQ(dim=16, num_quantizers=3, codebook_params=CodebookParams(dim=16, codebook_size=32,
                                                                                  threshold_ema_dead_code=0)).train()
        rvq.use_fused_levels = fused
        _step(rvq, _x())
    assert calls == {"rot_commit_backward": 0, "rvq_backward_rot": 0}
    assert counted["st_commit_backward"] == 5 and counted["rvq_backward"] == 1


def test_run_variants_gumbel_straight_through_and_affine(wired):
    from vqb200 import AffineParameters, GumbelParams
    calls, counted = wired
    vq = _vq(True, learnable_codebook=True, ema_update=False, gumbel_params=GumbelParams(straight_through=True))
    ref = _vq(False, learnable_codebook=True, ema_update=False, gumbel_params=GumbelParams(straight_through=True))
    a, b = _step(vq, _x()), _step(ref, _x())
    assert calls["rot_commit_backward"] == 1
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), "the forward value must not change"
    assert not torch.allclose(a[2], b[2])
    assert torch.equal(vq._codebook.embeddings.grad, ref._codebook.embeddings.grad), "codebook gradient changed"
    _step(_vq(True, use_affine=True, affine_params=AffineParameters(sync=False)), _x())
    assert calls["rot_commit_backward"] == 2


@pytest.mark.parametrize("fused", [True, False])
def test_residual_vq_loops(wired, fused):
    from vqb200 import CodebookParams, ResidualVQ
    calls, counted = wired
    mask = torch.rand(2, 40, generator=torch.Generator().manual_seed(2)) >= 0.3
    res = {}
    for use in (True, False):
        torch.manual_seed(0)
        rvq = ResidualVQ(dim=16, num_quantizers=3, rotation_trick=True,
                         codebook_params=CodebookParams(dim=16, codebook_size=32, threshold_ema_dead_code=0)).train()
        rvq.use_fused_levels = use and fused
        res[use] = _step(rvq, _x(), mask)
    assert torch.equal(res[True][0], res[False][0])
    assert torch.allclose(res[True][2], res[False][2], rtol=1e-5, atol=1e-6)
    assert calls["rvq_backward_rot"] == (1 if fused else 0)
    assert calls["rot_commit_backward"] == (3 if fused else 6)
    assert counted == {"st_commit_backward": 0, "rvq_backward": 0}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    from vqb200 import CodebookParams, VectorQuantize, _lib, distributed as D, ops, rvq as RVQ
    _install(ops, _lib, RVQ)
    D.SHARD_MIN_CODES = 32
    res = {}
    for rot in (True, False):
        torch.manual_seed(0)
        vq = VectorQuantize(dim=8, codebook_params=CodebookParams(dim=8, codebook_size=64, threshold_ema_dead_code=0),
                            sync_codebook=True).train()
        vq.rotation_trick = rot
        assert vq._codebook.sharded
        x = torch.randn(2, 30, 8, generator=torch.Generator().manual_seed(rank)).requires_grad_(True)
        q, ind, loss = vq(x)
        ((q * x.detach()).sum() + loss.sum()).backward()
        res[rot] = (q.detach(), ind, x.grad, CALLS["rot_commit_backward"])
    ok = torch.equal(res[True][0], res[False][0]) and torch.equal(res[True][1], res[False][1])
    out_res = {"calls": res[False][3], "same_forward": ok, "grad_differs": not torch.equal(res[True][2], res[False][2])}
    if rank == 0:
        torch.save(out_res, out)
    dist.destroy_process_group()


def test_two_rank_gloo_sharded_codebook_passes_the_flag(tmp_path):
    out = str(tmp_path / "rot_sharded.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    res = torch.load(out)
    assert res == {"calls": 1, "same_forward": True, "grad_differs": True}, res
