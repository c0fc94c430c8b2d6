"""The product's orchestration -- `Codebook._run` (branch selection, EMA step order, pre-update snapshot), dead-code
expiry, kmeans init, the VectorQuantize / ResidualVQ glue around them -- on CPU, with the tensor-level wrappers of
vqb200/ops.py replaced by plain-torch statements of what each C entry point computes (tests/cpu_kernels.py), against
the fixtures recorded from the live reference.  The kernels behind those wrappers are tested on the GPU."""
import pytest
import torch

import cpu_kernels
import golden_util as gu


def _cpu_draw(num_rows, m, device):
    if num_rows >= m:
        return torch.randperm(num_rows)[:m]
    return torch.randint(0, num_rows, (m,))


@pytest.fixture()
def cpu_ops(monkeypatch):
    from vqb200 import _lib, codebook, ops
    # the real entry points are recorded with the test's own monkeypatch before anything replaces them, so they are
    # what is restored last: a test that patches one of them again (tests/f4_util.py) cannot leave a plain-torch
    # statement in place of a kernel for the tests that follow
    for n in cpu_kernels.REPLACED:
        monkeypatch.setattr(ops, n, getattr(ops, n))
    monkeypatch.setattr(_lib, "require_device", _lib.require_device)
    cpu_kernels.install(ops, _lib)
    monkeypatch.setattr(codebook.Codebook, "_draw_rows", staticmethod(_cpu_draw))


@pytest.fixture()
def cpu_dense_ops(cpu_ops, monkeypatch):
    """... plus the dense-similarity entry points as their plain-torch statements (tests/dense_ref.py)."""
    import dense_ref as R
    from vqb200 import ops
    f = lambda t: t.detach().float()  # noqa: E731
    monkeypatch.setattr(ops, "dense_row_norms", lambda t: (f(t) * f(t)).sum(-1))
    monkeypatch.setattr(ops, "dense_rowstats", lambda x, xn2, e, cn2, cos, a, t: R.rowstats(f(x), e, cos, a, t))
    monkeypatch.setattr(ops, "dense_avgprob", lambda x, xn2, e, cn2, cos, a, lse, n: R.avgprob(f(x), e, cos, a, lse, n))
    monkeypatch.setattr(ops, "dense_rowdot",
                        lambda x, xn2, e, cn2, cos, a, lse, tab, n: R.rowdot(f(x), e, cos, a, lse, tab, n))
    monkeypatch.setattr(ops, "dense_backward",
                        lambda x, xn2, ed, cn2, ec, cos, a, lse, coef, target=None, table=None, rdot=None, n_pos=1:
                        R.backward(f(x), ed, ec, cos, a, lse, coef, target, table, rdot, n_pos))
    monkeypatch.setattr(ops, "dense_backward_codes",
                        lambda x, xn2, e, cn2, cos, a, lse, coef, target=None, table=None, rdot=None, n_pos=1:
                        R.backward_codes(f(x), e.detach(), cos, a, lse, coef, target, table, rdot, n_pos))


@pytest.mark.parametrize("name", gu.grad_fixture_names())
def test_orchestration_input_gradient_matches_reference_fixture(name, cpu_ops):
    """The autograd wiring of the real `_run` (`_QuantizeST`, the pre-update codebook snapshot, `_L2NormRows`, the
    ResidualVQ loop) against the gradients recorded from the live reference on the EMA path."""
    from test_gpu_parity import build_module, load_state
    fx = gu.load_grad(name)
    cfg = fx["cfg"]
    mod, books = build_module(cfg)
    with torch.no_grad():
        load_state(books, fx)
    mod.train()
    x = fx["x"].clone().requires_grad_(True)
    q, ind, loss = mod(x, mask=fx["mask"])
    ((q * fx["w"]).sum() + loss.sum() * 1.7).backward()
    assert torch.equal(ind, fx["indices"])
    assert gu.rel_err(q.detach(), fx["quantize"]) <= 1e-6
    assert torch.allclose(loss.detach(), fx["loss"], rtol=1e-5)
    assert gu.rel_err(x.grad - fx["w"], fx["grad_x"] - fx["w"]) <= 1e-3
    assert gu.rel_err(x.grad, fx["grad_x"]) <= 1e-6
    for cb, after in zip(books, fx["after"]):
        assert torch.equal(cb.cluster_size, after["cluster_size"])
        assert gu.rel_err(cb.embeddings, after["embeddings"]) <= 1e-5


@pytest.mark.parametrize("name", gu.dense_fixture_names())
def test_orchestration_dense_losses_match_reference_fixture(name, cpu_dense_ops):
    """The dense-similarity losses through the REAL `_run` (keep_dense context, pre-update snapshot shared with the
    commitment term) -- tests/test_dense_host_cpu.py covers vq.py with `_run` replaced."""
    from test_dense_host_cpu import build_module, load_state
    fx = gu.load_dense(name)
    cfg = fx["cfg"]
    vq = build_module(cfg)
    vq.train(cfg["training"])
    load_state(vq, fx)
    x = fx["x"].clone().requires_grad_(True)
    if cfg["kind"] == "indices":
        q, ce = vq(x, indices=fx["targets"])
        (q.sum() * 0.01 + ce * 1.3 if cfg["training"] else ce * 1.3).backward()
        assert torch.allclose(ce.detach(), fx["ce"], rtol=1e-6)
    else:
        q, ind, loss, bd = vq(x, mask=fx["mask"], return_loss_breakdown=True)
        ((q * fx["w"]).sum() + loss.sum() * 1.7).backward()
        assert torch.equal(ind, fx["indices"])
        assert torch.allclose(loss.detach(), fx["loss"], rtol=1e-6, atol=1e-7)
        assert torch.allclose(bd.commitment.detach(), fx["commitment"], rtol=1e-6)
        assert torch.allclose(bd.codebook_diversity.detach(), fx["codebook_diversity"], rtol=1e-6)
    assert gu.rel_err(q.detach(), fx["quantize"]) <= 1e-6
    assert gu.rel_err(x.grad, fx["grad_x"]) <= 2e-6
    assert torch.equal(vq._codebook.cluster_size, fx["after"]["cluster_size"])
    assert gu.rel_err(vq._codebook.embeddings, fx["after"]["embeddings"]) <= 1e-6


LEARNABLE = ["learnable_plain", "learnable_masked_v", "inplace_sgd", "inplace_sgd_masked", "learnable_ce_commit",
             "learnable_ce_commit_dot", "learnable_diversity", "learnable_ce_indices"]


@pytest.mark.parametrize("name", LEARNABLE)
def test_orchestration_learnable_codebook_matches_reference_fixture(name, cpu_dense_ops):
    """Learnable codebook through the real `_run`: codebook gradients of the commitment loss (segmented sums), of the
    dense losses, sync_update_v, the in-place optimizer step."""
    import os
    from vqb200 import CodebookParams, VectorQuantize
    fx = torch.load(os.path.join(gu.GOLDEN_DIR, "learnable", name + ".pt"), weights_only=False)
    cfg = fx["cfg"]
    cp = CodebookParams(dim=cfg["dim"], codebook_size=cfg["K"], learnable_codebook=True, ema_update=False,
                        threshold_ema_dead_code=0, use_cosine_sim=cfg.get("cosine", False))
    extra = {}
    if cfg.get("ce"):
        extra["commitment_use_cross_entropy_loss"] = True
    if cfg.get("dw"):
        extra.update(codebook_diversity_loss_weight=cfg["dw"], codebook_diversity_temperature=cfg["temp"])
    if "lr" in cfg:
        extra["in_place_codebook_optimizer"] = lambda p: torch.optim.SGD(p, lr=cfg["lr"])
    vq = VectorQuantize(dim=cfg["dim"], codebook_params=cp, commitment_weight=cfg["cw"], sync_update_v=cfg["v"],
                        sync_codebook=False, **extra).train()
    with torch.no_grad():
        vq._codebook.embeddings.copy_(fx["init_embeddings"])
    x = fx["x"].clone().requires_grad_(True)
    if cfg.get("indices"):
        q, ce = vq(x, indices=fx["targets"])
        (q.sum() * 0.01 + ce * 1.3).backward()
        assert torch.allclose(ce.detach(), fx["ce"], rtol=1e-6)
    else:
        q, ind, loss, bd = vq(x, mask=fx["mask"], return_loss_breakdown=True)
        (q * fx["w"]).sum().add(loss.sum() * 1.7).backward()
        assert torch.equal(ind, fx["indices"])
        assert torch.allclose(loss.detach(), fx["loss"], rtol=1e-6)
        if "lr" in cfg:
            assert torch.allclose(bd.inplace_optimize, fx["inplace_optimize"], rtol=1e-6)
            assert gu.rel_err(vq._codebook.embeddings.detach(), fx["after_embeddings"]) <= 1e-6
    assert gu.rel_err(q.detach(), fx["quantize"]) <= 1e-6
    assert gu.rel_err(x.grad, fx["grad_x"]) <= 2e-6
    assert gu.rel_err(vq._codebook.embeddings.grad, fx["grad_embeddings"]) <= 2e-6


@pytest.mark.parametrize("name", gu.fixture_names())
def test_orchestration_matches_reference_fixture(name, cpu_ops):
    from test_gpu_parity import build_module, load_state
    fx = gu.load(name)
    cfg = fx["cfg"]
    mod, books = build_module(cfg)
    with torch.no_grad():
        load_state(books, fx)
    mod.train(cfg.get("training", True))
    for s, step in enumerate(fx["steps"]):
        torch.manual_seed(fx["rng_seed"] + s)
        with torch.no_grad():
            q, ind, loss = mod(fx["x"] + 0.01 * s, mask=fx["mask"])
        assert torch.equal(ind, step["indices"]), f"{name} step {s}: indices"
        assert ind.dtype == torch.int64 and q.dtype == torch.float32 and loss.shape == step["loss"].shape
        assert gu.rel_err(q, step["quantize"]) <= 1e-6
        assert torch.allclose(loss, step["loss"], rtol=1e-5, atol=1e-12)
        for cb, after in zip(books, step["after"]):
            assert torch.equal(cb.cluster_size, after["cluster_size"])
            assert gu.rel_err(cb.embed_avg, after["embed_avg"]) <= 1e-5
            assert gu.rel_err(cb.embeddings, after["embeddings"]) <= 1e-5


def test_device_guard_is_back_after_the_stand_ins():
    from vqb200 import CodebookParams, VectorQuantize
    vq = VectorQuantize(dim=8, codebook_params=CodebookParams(dim=8, codebook_size=4))
    with pytest.raises(RuntimeError, match="CUDA"):
        vq(torch.randn(1, 3, 8))


@pytest.mark.parametrize("seed", list(range(40)))
def test_orchestration_equals_restatement_on_random_options(seed, cpu_dense_ops):
    """The seeded random option combinations of tests/test_random_configs_cpu.py through the REAL `_run`."""
    import test_random_configs_cpu as T
    from vqb200 import CodebookParams, VectorQuantize
    cfg = T.make_case(seed)
    T.compare(T.run_module(cfg, VectorQuantize, CodebookParams), T.run_oracle(cfg), exact=False, cfg=cfg)


@pytest.mark.parametrize("fused_ema", [False, True])
@pytest.mark.parametrize("name", [n for n in gu.fixture_names() if n.startswith("rvq")])
def test_fused_rvq_level_loop_matches_reference_fixture(name, fused_ema, cpu_ops, monkeypatch):
    """`ResidualVQ._forward_fused` (one pass per level, operands of the next level prepared on the way, the dead-code
    checks of all levels answered by one sync and replayed in level order) against the reference fixtures, both with
    the level step and the EMA sums in one call (`rvq_level_ema`) and as separate calls."""
    from test_gpu_parity import build_module, load_state
    from vqb200 import ops, rvq
    monkeypatch.setattr(ops, "rvq_level_ema_supported", lambda d: fused_ema)
    real_can_fuse = rvq.ResidualVQ._can_fuse
    calls = {"fused": 0}

    class _OnDevice:          # what `_can_fuse` asks of its input, answered as for a CUDA tensor
        def __init__(self, t):
            self.is_cuda, self.ndim, self.requires_grad = True, t.ndim, t.requires_grad

    def can_fuse(self, x, dropout_active):
        ok = real_can_fuse(self, _OnDevice(x), dropout_active)
        calls["fused"] += int(ok)
        return ok

    monkeypatch.setattr(rvq.ResidualVQ, "_can_fuse", can_fuse)
    fx = gu.load(name)
    cfg = fx["cfg"]
    mod, books = build_module(cfg)
    with torch.no_grad():
        load_state(books, fx)
    mod.train(cfg.get("training", True))
    for s, step in enumerate(fx["steps"]):
        torch.manual_seed(fx["rng_seed"] + s)
        with torch.no_grad():
            q, ind, loss = mod(fx["x"] + 0.01 * s, mask=fx["mask"])
        assert torch.equal(ind, step["indices"]), f"{name} step {s}: indices"
        assert gu.rel_err(q, step["quantize"]) <= 1e-6
        assert torch.allclose(loss, step["loss"], rtol=1e-5, atol=1e-12)
        for cb, after in zip(books, step["after"]):
            assert torch.equal(cb.cluster_size, after["cluster_size"])
            assert gu.rel_err(cb.embeddings, after["embeddings"]) <= 1e-5
    assert calls["fused"] == len(fx["steps"])          # the fused loop is what ran


@pytest.mark.parametrize("name", gu.rvq_learnable_fixture_names())
def test_orchestration_rvq_learnable_codebooks_get_their_gradient(name, cpu_ops):
    """ResidualVQ over learnable codebooks: the fused (no_grad) level loop must NOT be taken while a codebook Parameter
    wants a gradient, even if the input carries none (reference vector_quantize_pytorch.py:263-269)."""
    gu.check_rvq_learnable(name, torch.device("cpu"))


@pytest.mark.parametrize("name", [n for n in gu.grad_fixture_names() if "rvq" in n])
def test_fused_rvq_loop_under_autograd_matches_reference_gradient(name, cpu_ops, monkeypatch):
    """`_FusedRVQ`: the fused level loop with a gradient to the input (one replay pass backward, `rvq_backward`) against
    the input gradients recorded from the live reference (3 levels; shared codebook + mask)."""
    from test_gpu_parity import build_module, load_state
    from vqb200 import rvq
    real_can_fuse = rvq.ResidualVQ._can_fuse
    calls = {"fused": 0}

    class _OnDevice:
        def __init__(self, t):
            self.is_cuda, self.ndim, self.requires_grad, self.shape = True, t.ndim, t.requires_grad, t.shape

    def can_fuse(self, x, dropout_active):
        ok = real_can_fuse(self, _OnDevice(x), dropout_active)
        calls["fused"] += int(ok)
        return ok

    monkeypatch.setattr(rvq.ResidualVQ, "_can_fuse", can_fuse)
    fx = gu.load_grad(name)
    mod, books = build_module(fx["cfg"])
    with torch.no_grad():
        load_state(books, fx)
    mod.train()
    x = fx["x"].clone().requires_grad_(True)
    q, ind, loss = mod(x, mask=fx["mask"])
    assert calls["fused"] == 1 and q.grad_fn is not None
    ((q * fx["w"]).sum() + loss.sum() * 1.7).backward()
    assert torch.equal(ind, fx["indices"])
    assert gu.rel_err(q.detach(), fx["quantize"]) <= 1e-6
    assert torch.allclose(loss.detach(), fx["loss"], rtol=1e-5)
    assert gu.rel_err(x.grad, fx["grad_x"]) <= 1e-6
    for cb, after in zip(books, fx["after"]):
        assert torch.equal(cb.cluster_size, after["cluster_size"])
        assert gu.rel_err(cb.embeddings, after["embeddings"]) <= 1e-5
