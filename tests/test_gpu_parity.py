"""GPU parity tests: the CUDA path (through the C ABI, via the vqb200 modules) against
(a) the golden fixtures recorded from the live reference and (b) the CPU oracle on seeded inputs.

Bars (BASELINE.json north_star): indices identical except rows whose REFERENCE fp32 top-2 gap is
< 1e-6 relative; quantize bit-exact given the indices; loss and EMA buffers within 1e-5 relative
(relative to the buffer's max magnitude); cluster_size exact.
"""
import pytest
import torch

import golden_util as gu

pytestmark = pytest.mark.gpu

REL = 1e-5


def _dev():
    return torch.device("cuda:0")


def _cpu_draw(num_rows, m, device):
    """Draw replacement/kmeans rows from the CPU generator exactly like the oracle/reference-on-CPU did."""
    if num_rows >= m:
        return torch.randperm(num_rows)[:m].to(device)
    return torch.randint(0, num_rows, (m,)).to(device)


@pytest.fixture(autouse=True)
def _patch_draw(monkeypatch):
    from vqb200 import codebook
    monkeypatch.setattr(codebook.Codebook, "_draw_rows", staticmethod(_cpu_draw))


def build_module(cfg):
    from vqb200 import CodebookParams, KmeansParameters, ResidualVQ, VectorQuantize
    cb_dim = cfg.get("cb_dim", cfg["dim"])
    cp = CodebookParams(dim=cb_dim, codebook_size=cfg["K"], threshold_ema_dead_code=cfg["thr"],
                        use_cosine_sim=cfg.get("cosine", False),
                        transform_input="l2norm" if cfg.get("l2in") else "identity",
                        weights_regularization="l2norm" if cfg.get("l2w") else "identity",
                        initialization_by_kmeans=cfg.get("kmeans", False),
                        kmeans_params=KmeansParameters() if cfg.get("kmeans") else None)
    if cfg["kind"] == "vq":
        mod = VectorQuantize(dim=cfg["dim"], codebook_params=cp, codebook_dim=cfg.get("cb_dim"),
                             heads=cfg.get("heads", 1), separate_codebook_per_head=cfg.get("separate", False),
                             channel_last=cfg.get("channel_last", True), sync_codebook=False)
        books = [mod._codebook]
    else:
        mod = ResidualVQ(dim=cfg["dim"], num_quantizers=cfg["Q"], codebook_params=cp,
                         shared_codebook=cfg.get("shared", False), sync_codebook=False)
        books = [l._codebook for l in mod.layers]
    return mod, books


def load_state(books, fx):
    seen = set()
    for cb, init in zip(books, fx["init"]):
        if id(cb) in seen:
            continue
        seen.add(id(cb))
        cb.embeddings.copy_(init["embeddings"])
        cb.embed_avg.copy_(init["embed_avg"])
        cb.cluster_size.copy_(init["cluster_size"])
        cb.invalidate_cache()


def run_fixture(name, fused):
    fx = gu.load(name)
    cfg = fx["cfg"]
    mod, books = build_module(cfg)
    mod = mod.to(_dev())
    load_state(books, fx)
    training = cfg.get("training", True)
    mod.train(training)
    if cfg["kind"] == "rvq":
        mod.use_fused_levels = fused
    l2 = bool(cfg.get("l2in"))
    mask = fx["mask"].to(_dev()) if fx["mask"] is not None else None
    for s, step in enumerate(fx["steps"]):
        x = (fx["x"] + 0.01 * s).to(_dev())
        torch.manual_seed(fx["rng_seed"] + s)
        with torch.no_grad():
            q, ind, loss = mod(x, mask=mask)
        torch.cuda.synchronize()
        q, ind, loss = q.cpu(), ind.cpu(), loss.cpu()
        ref_ind = step["indices"]
        assert ind.shape == ref_ind.shape and ind.dtype == torch.int64
        assert q.shape == step["quantize"].shape and q.dtype == torch.float32
        assert loss.shape == step["loss"].shape
        diff = ind != ref_ind
        if bool(diff.any()):
            # only rows inside the reference's own fp32 tie zone may differ
            gaps = step["top2_rel_gap"]
            if cfg["kind"] == "vq" and len(gaps) == 1 and gaps[0].numel() == ind.numel() and cfg.get("heads", 1) == 1:
                g = gaps[0].reshape(ind.shape)
                assert bool((g[diff] < 1e-6).all()), f"{name} step {s}: index mismatch outside the tie exemption"
                pytest.skip(f"{name}: {int(diff.sum())} exempt tie rows changed the trajectory; later values not comparable")
            raise AssertionError(f"{name} step {s}: {int(diff.sum())} index mismatches")
        # bit-exact given the indices AND identical codebooks: true on the first step (buffers loaded from the
        # fixture, every level's codebook untouched); after an EMA refresh (later steps, or later levels of a
        # shared codebook) the codebooks agree to 1e-5, and so does quantize.
        if s == 0 and not l2 and not cfg.get("kmeans") and not cfg.get("shared"):
            assert torch.equal(q, step["quantize"]), f"{name} step {s}: quantize not bit-exact"
        else:
            assert gu.rel_err(q, step["quantize"]) <= REL, f"{name} step {s}: quantize"
        ref_loss = step["loss"]
        assert torch.allclose(loss, ref_loss, rtol=REL, atol=1e-12), f"{name} step {s}: loss {loss} vs {ref_loss}"
        for lvl, after in enumerate(step["after"]):
            cb = books[lvl]
            assert torch.equal(cb.cluster_size.cpu(), after["cluster_size"]), f"{name} step {s} lvl {lvl}: cluster_size"
            assert gu.rel_err(cb.embed_avg.cpu(), after["embed_avg"]) <= REL, f"{name} step {s} lvl {lvl}: embed_avg"
            assert gu.rel_err(cb.embeddings.cpu(), after["embeddings"]) <= REL, f"{name} step {s} lvl {lvl}: embeddings"


@pytest.mark.parametrize("name", gu.fixture_names())
def test_module_matches_reference_fixture(name):
    run_fixture(name, fused=True)


@pytest.mark.parametrize("name", [n for n in gu.fixture_names() if n.startswith("rvq")])
def test_rvq_generic_loop_matches_reference_fixture(name):
    run_fixture(name, fused=False)


# ------------------------------------------------------------------------------------------------
# op level: search (tensor-core path) vs exact scan vs oracle, many shapes incl. ragged / padded
# ------------------------------------------------------------------------------------------------
SEARCH_SHAPES = [
    # H, N, K, d, cosine, codebook scale (None = reference default kaiming-uniform scale)
    (1, 1, 1, 1, False, 0.5),
    (1, 7, 3, 5, False, 0.5),
    (1, 128, 256, 64, False, 0.5),
    (1, 1024, 512, 256, False, 0.5),
    (1, 1024, 512, 256, False, None),
    (1, 1000, 300, 100, False, 0.5),
    (3, 333, 260, 72, False, 0.5),
    (2, 777, 520, 96, True, 0.5),
    (1, 2048, 1024, 512, False, 0.5),
    (1, 2048, 1024, 512, True, 0.5),
    (1, 513, 2050, 64, False, 0.5),
    (1, 300, 64, 640, False, 0.5),       # d_pad > 512: exact-scan path
]


@pytest.mark.parametrize("H,N,K,d,cos,scale", SEARCH_SHAPES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_search_matches_oracle(H, N, K, d, cos, scale, dtype):
    from oracle import vq_oracle as O
    from vqb200 import ops
    g = torch.Generator().manual_seed(1000 * N + K + d)
    x = torch.randn(H, N, d, generator=g).to(dtype)
    if scale is None:
        c = (torch.rand(H, K, d, generator=g) * 2 - 1) * (6.0 / (K * d)) ** 0.5
    else:
        c = torch.randn(H, K, d, generator=g) * scale
    xd, cd = x.to(_dev()), c.to(_dev())
    cache = ops.prepare_codebook(cd, cos)
    idx, score, ws = ops.search(xd, cd, cache, cos, want_score=True)
    stats = ops.search_stats(ws)          # before the next search reuses (and zeroes) the workspace
    idx_ex, score_ex, _ = ops.search(xd, cd, cache, cos, force_exact=True, want_score=True)
    torch.cuda.synchronize()
    if ((d + 63) // 64) * 64 <= 512:
        assert stats["tensor_core_pass"] == 1
    # the two CUDA paths use the same fp64-accumulated score: they must agree exactly
    assert torch.equal(idx, idx_ex), f"tc vs exact: {int((idx != idx_ex).sum())} mismatches, stats {stats}"
    assert torch.equal(score, score_ex)
    sim = O.similarities(x.float(), c, cos)
    ref = sim.argmax(-1)
    if K > 1:
        top2 = sim.topk(2, -1).values
        gap = (top2[..., 0] - top2[..., 1]).abs() / top2[..., 0].abs().clamp_min(1e-30)
    else:
        gap = torch.full(ref.shape, float("inf"))
    bad = (idx.cpu() != ref) & (gap >= 1e-6)
    if bool(bad.any()):
        # strict: only rows inside the reference's own fp32 1e-6 window may differ (tools/oracle_noise.py: the oracle's
        # rounding noise never reaches outside it); print what is needed to diagnose
        hh, nn = bad.nonzero(as_tuple=True)
        detail = []
        for h_, n_ in list(zip(hh.tolist(), nn.tolist()))[:8]:
            x64, c64 = x[h_, n_].double(), c[h_].double()
            s64 = c64 @ x64 if cos else -(c64 - x64).pow(2).sum(-1).sqrt()
            t2 = s64.topk(2).values
            g64 = float((t2[0] - t2[1]).abs() / t2[0].abs().clamp_min(1e-30))
            detail.append((h_, n_, int(idx[h_, n_]), int(ref[h_, n_]), int(s64.argmax()), float(gap[h_, n_]), g64))
        raise AssertionError(f"{int(bad.sum())} rows differ from the oracle outside its 1e-6 window; (h, row, got, "
                             f"oracle, fp64 argmin, oracle gap, fp64 gap): {detail}; stats {stats}")
    # score: distance (euclid) or -similarity (dot) of the winner
    ref_score = -sim.gather(-1, idx.cpu()[..., None])[..., 0]
    assert torch.allclose(score.cpu(), ref_score, rtol=2e-5, atol=2e-5 * float(ref_score.abs().max()) + 1e-7)


def test_search_duplicate_codes_and_ties():
    """Exact duplicates in the codebook (expiry copies batch rows): the lowest index must win, as torch.argmax."""
    from vqb200 import ops
    g = torch.Generator().manual_seed(5)
    c = torch.randn(1, 512, 64, generator=g)
    c[0, 100] = c[0, 7]
    c[0, 300] = c[0, 7]
    c[0, 301] = c[0, 7]
    c[0, 411] = c[0, 7]
    x = torch.randn(1, 256, 64, generator=g)
    x[0, :64] = c[0, 7] + 1e-3 * torch.randn(64, 64, generator=g)
    xd, cd = x.to(_dev()), c.to(_dev())
    idx, _, ws = ops.search(xd, cd, ops.prepare_codebook(cd, False), False)
    ref = (-torch.cdist(x, c)).argmax(-1)
    assert torch.equal(idx.cpu()[0, :64], torch.full((64,), 7))
    assert torch.equal(idx.cpu(), ref)


def test_gather_st_loss_and_backward_match_torch():
    from vqb200 import ops
    g = torch.Generator().manual_seed(3)
    H, N, K, d = 2, 300, 50, 40
    x = torch.randn(H, N, d, generator=g)
    c = torch.randn(H, K, d, generator=g)
    idx = torch.randint(0, K, (H, N), generator=g)
    mask = torch.rand(N, generator=g) > 0.3
    xd = x.to(_dev()).requires_grad_(True)
    q, commit, _ = ops.quantize_training(xd, c.to(_dev()), idx.to(_dev()), mask.to(torch.uint8).to(_dev()), True)
    gq = torch.randn(H, N, d, generator=g)
    (q * gq.to(_dev())).sum().add(commit * 0.7).backward()
    xr = x.clone().requires_grad_(True)
    cq = torch.stack([c[h][idx[h]] for h in range(H)])
    qr = xr + (cq - xr).detach()
    lr = torch.nn.functional.mse_loss(cq, xr, reduction="none")[:, mask].mean()
    (qr * gq).sum().add(lr * 0.7).backward()
    assert torch.equal(q.detach().cpu(), qr.detach())
    assert torch.allclose(commit.detach().cpu(), lr.detach(), rtol=1e-6)
    assert torch.allclose(xd.grad.cpu(), xr.grad, rtol=1e-5, atol=1e-7)


def test_ema_reduce_is_deterministic_and_exact():
    from vqb200 import ops
    g = torch.Generator().manual_seed(11)
    H, N, K, d = 2, 5000, 97, 72
    x = torch.randn(H, N, d, generator=g)
    idx = torch.randint(0, K, (H, N), generator=g)
    idx[:, :2000] = 3                      # one very long segment
    mask = torch.rand(N, generator=g) > 0.2
    xd, idd, md = x.to(_dev()), idx.to(_dev()), mask.to(torch.uint8).to(_dev())
    a = ops.ema_reduce(xd, idd, md, K).cpu()
    b = ops.ema_reduce(xd, idd, md, K).cpu()
    assert torch.equal(a, b), "EMA statistics must be bitwise reproducible"
    onehot = torch.nn.functional.one_hot(idx, K).double()
    onehot[:, ~mask] = 0
    ref_cnt = onehot.sum(1)
    ref_sum = torch.einsum("hnd,hnc->hcd", x.double(), onehot)
    assert torch.equal(a[..., d].double(), ref_cnt)
    assert float((a[..., :d].double() - ref_sum).abs().max()) <= 1e-6 * float(ref_sum.abs().max())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("H,N,K,d", [(1, 5000, 97, 64), (2, 3000, 50, 256), (1, 2500, 31, 512), (3, 700, 9, 8),
                                      (1, 4097, 300, 128), (1, 1, 4, 32)])
def test_fused_quantize_ema_matches_separate_passes(H, N, K, d, dtype):
    """vqb_quantize_ema == vqb_gather_st_loss + vqb_ema_reduce (q bit-exact, counts exact, sums vs fp64), and is
    bitwise reproducible although its row placement uses atomics."""
    from vqb200 import ops
    assert ops.quantize_ema_supported(d)
    g = torch.Generator().manual_seed(5 + d)
    x = (torch.randn(H, N, d, generator=g) * 3).to(dtype)
    c = torch.randn(H, K, d, generator=g)
    idx = torch.randint(0, K, (H, N), generator=g)
    idx[:, : N // 3] = K - 1                # one long segment, spanning several 64-row chunks
    xd, cd, idd = x.to(_dev()), c.to(_dev()), idx.to(_dev())
    for training in (True, False):
        q, loss, stats = ops.quantize_ema(xd, cd, idd, training, True)
        q2, loss2, stats2 = ops.quantize_ema(xd, cd, idd, training, True)
        assert torch.equal(q, q2) and torch.equal(loss, loss2) and torch.equal(stats, stats2)
        qs, ls = ops.gather_st_loss(xd, cd, idd, None, training, True)
        assert torch.equal(q, qs), "fused q must be bit-identical to the gather kernel"
        assert torch.allclose(loss.cpu(), ls.cpu(), rtol=1e-6)
        xf = x.double()
        onehot = torch.nn.functional.one_hot(idx, K).double()
        ref_sum = torch.einsum("hnd,hnc->hcd", xf, onehot)
        st = stats.cpu()
        assert torch.equal(st[..., d].double(), onehot.sum(1))
        assert float((st[..., :d].double() - ref_sum).abs().max()) <= 1e-6 * max(float(ref_sum.abs().max()), 1e-30)
        sep = ops.ema_reduce(xd, idd, None, K).cpu()
        assert float((st - sep).abs().max()) <= 2e-6 * max(float(sep.abs().max()), 1e-30)
        cq = torch.stack([c[h][idx[h]] for h in range(H)])
        ref_loss = ((cq.double() - xf) ** 2).mean()
        assert abs(float(loss[0]) - float(ref_loss)) <= 1e-6 * float(ref_loss)
        assert float(loss[1]) == H * N


def test_fused_quantize_ema_extreme_scales_and_module_switch():
    """Tiny / huge magnitudes go through the fixed-point scale; the module gives the same buffers with the fused pass
    on and off."""
    from vqb200 import CodebookParams, VectorQuantize, ops
    g = torch.Generator().manual_seed(9)
    for scale in (1e-20, 1e15):
        x = torch.randn(1, 1000, 64, generator=g) * scale
        c = torch.randn(1, 16, 64, generator=g) * scale
        idx = torch.randint(0, 16, (1, 1000), generator=g)
        _, _, st = ops.quantize_ema(x.to(_dev()), c.to(_dev()), idx.to(_dev()), True, False)
        ref = torch.einsum("hnd,hnc->hcd", x.double(), torch.nn.functional.one_hot(idx, 16).double())
        assert float((st[..., :64].cpu().double() - ref).abs().max()) <= 1e-6 * float(ref.abs().max())
    outs = []
    for fused in (True, False):
        torch.manual_seed(0)
        vq = VectorQuantize(dim=64, codebook_params=CodebookParams(dim=64, codebook_size=128,
                                                                  threshold_ema_dead_code=0)).to(_dev()).train()
        vq._codebook.fused_quantize_ema = fused
        xx = torch.randn(4, 500, 64, generator=torch.Generator().manual_seed(1)).to(_dev()).requires_grad_(True)
        q, ind, loss = vq(xx)
        (q.sum() + loss.sum()).backward()
        outs.append((q.detach(), ind, loss.detach(), xx.grad, vq._codebook.embeddings.clone(),
                     vq._codebook.cluster_size.clone()))
    a, b = outs
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[5], b[5])
    assert torch.allclose(a[2], b[2], rtol=1e-6) and torch.allclose(a[3], b[3], rtol=1e-5, atol=1e-8)
    assert torch.allclose(a[4], b[4], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("d,K", [(512, 64), (256, 37), (64, 100), (128, 8)])
def test_rvq_level_ema_matches_separate_kernels(d, K):
    """vqb_rvq_level_ema == vqb_rvq_level + vqb_ema_reduce on every output, including the next level's operands
    (checked through the search they feed)."""
    from vqb200 import ops
    g = torch.Generator().manual_seed(d + K)
    N = 3000
    res = (torch.randn(N, d, generator=g) * 2).to(_dev())
    c = torch.randn(1, K, d, generator=g).to(_dev())
    c2 = (torch.randn(1, K, d, generator=g) * 0.5).to(_dev())
    idx = torch.randint(0, K, (1, N), generator=g).to(_dev())
    idx[:, :700] = K - 1
    cache2 = ops.prepare_codebook(c2, False)
    for first in (True, False):
        outs = []
        for fused in (True, False):
            out = torch.full((N, d), 0.25, device=_dev())
            nxt = torch.empty_like(res)
            if fused:
                loss, stats = ops.rvq_level_ema(res, nxt, c[0], idx[0], True, first, out, cache2)
            else:
                stats = ops.ema_reduce(res[None], idx, None, K)
                loss = ops.rvq_level(res, nxt, c[0], idx[0], None, True, first, out, cache2)
            nidx, _, _ = ops.search(nxt[None], c2, cache2, False, latents_prepared=True)
            outs.append((out.clone(), nxt.clone(), loss.clone(), stats.clone(), nidx.clone()))
        a, b = outs
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[4], b[4])
        assert torch.allclose(a[2], b[2], rtol=1e-6)
        assert torch.equal(a[3][..., d], b[3][..., d])
        assert float((a[3] - b[3]).abs().max()) <= 2e-6 * float(b[3].abs().max())
        ref_idx, _, _ = ops.search(a[1][None], c2, cache2, False)
        assert torch.equal(a[4], ref_idx)


def test_search_is_repeatable_through_a_shared_workspace():
    """Searches of different shapes alternate through one workspace; every repetition must reproduce the first result
    of its shape bit for bit (indices and scores): nothing may depend on timing (shared running minima, atomic
    pair-list order) or on what the previous search left behind."""
    from vqb200 import ops
    g = torch.Generator(device=_dev()).manual_seed(3)
    cases = []
    for (N, K, d, dt) in [(40000, 1000, 72, torch.float32), (150000, 2048, 256, torch.bfloat16),
                          (9000, 512, 64, torch.float32), (70000, 700, 512, torch.float32)]:
        x = torch.randn(1, N, d, generator=g, device=_dev()).to(dt).contiguous()
        c = torch.randn(1, K, d, generator=g, device=_dev()) * 0.5
        cache = ops.prepare_codebook(c, False)
        ref, rs, _ = ops.search(x, c, cache, False, want_score=True)
        cases.append((x, c, cache, ref.clone(), rs.clone()))
    for r in range(6):
        for ci, (x, c, cache, ref, rs) in enumerate(cases):
            want = (r + ci) % 2 == 0
            idx, sc, _ = ops.search(x, c, cache, False, want_score=want)
            assert torch.equal(idx, ref), f"repetition {r} of case {ci}: {int((idx != ref).sum())} indices changed"
            if want:
                assert torch.equal(sc, rs)


@pytest.mark.parametrize("name", ["learnable_plain", "learnable_masked_v"])
def test_learnable_codebook_matches_reference_fixture(name):
    """learnable_codebook=True, ema_update=False (+ sync_update_v): outputs and the gradients with respect to the input
    and the codebook against the live reference (tests/golden/make_golden_learnable.py)."""
    import os
    from vqb200 import CodebookParams, VectorQuantize
    fx = torch.load(os.path.join(gu.GOLDEN_DIR, "learnable", name + ".pt"), weights_only=False)
    cfg = fx["cfg"]
    cp = CodebookParams(dim=cfg["dim"], codebook_size=cfg["K"], learnable_codebook=True, ema_update=False,
                        threshold_ema_dead_code=0)
    vq = VectorQuantize(dim=cfg["dim"], codebook_params=cp, commitment_weight=cfg["cw"], sync_update_v=cfg["v"],
                        sync_codebook=False).to(_dev()).train()
    assert isinstance(vq._codebook.embeddings, torch.nn.Parameter)
    with torch.no_grad():
        vq._codebook.embeddings.copy_(fx["init_embeddings"])
    vq._codebook.invalidate_cache()
    x = fx["x"].to(_dev()).requires_grad_(True)
    mask = fx["mask"].to(_dev()) if fx["mask"] is not None else None
    q, ind, loss = vq(x, mask=mask)
    (q * fx["w"].to(_dev())).sum().add(loss.sum() * 1.7).backward()
    assert torch.equal(ind.cpu(), fx["indices"])
    assert torch.equal(q.detach().cpu(), fx["quantize"])
    assert torch.allclose(loss.detach().cpu(), fx["loss"], rtol=1e-6)
    assert torch.allclose(x.grad.cpu(), fx["grad_x"], rtol=1e-5, atol=1e-7)
    ge = vq._codebook.embeddings.grad.cpu()
    assert gu.rel_err(ge, fx["grad_embeddings"]) <= 1e-5
    # the codebook did not move (no EMA) and an optimizer step invalidates the search cache through the version counter
    assert torch.equal(vq._codebook.embeddings.detach().cpu(), fx["init_embeddings"])
    torch.optim.SGD(vq.parameters(), lr=0.5).step()
    q2, ind2, _ = vq(fx["x"].to(_dev()), mask=mask)
    from vqb200 import ops
    ex, _, _ = ops.search(fx["x"].to(_dev()).reshape(1, -1, cfg["dim"]).contiguous(), vq._codebook.embeddings.detach(),
                          None, False, force_exact=True)
    assert torch.equal(ind2.reshape(-1), ex.reshape(-1))


@pytest.mark.parametrize("name", gu.grad_fixture_names())
def test_input_gradient_on_the_ema_path_matches_reference_fixture(name):
    """One training forward under autograd, the EMA step moving the codebook inside it, then backward: outputs,
    buffers and the input gradient of the live reference (tests/golden/make_golden_grads.py).  The commitment term
    must read the PRE-update codes; one / shared / separate heads, masks, cosine, channel-first images, 2-D input,
    ResidualVQ (generic level loop: the fused loop is forward-only)."""
    fx = gu.load_grad(name)
    cfg = fx["cfg"]
    mod, books = build_module(cfg)
    mod = mod.to(_dev()).train()
    with torch.no_grad():
        load_state(books, fx)
    x = fx["x"].to(_dev()).requires_grad_(True)
    mask = fx["mask"].to(_dev()) if fx["mask"] is not None else None
    q, ind, loss = mod(x, mask=mask)
    ((q * fx["w"].to(_dev())).sum() + loss.sum() * 1.7).backward()
    assert torch.equal(ind.cpu(), fx["indices"])
    if cfg.get("l2in") or cfg["kind"] == "rvq":
        assert gu.rel_err(q.detach().cpu(), fx["quantize"]) <= 1e-6
    else:
        assert torch.equal(q.detach().cpu(), fx["quantize"])
    assert torch.allclose(loss.detach().cpu(), fx["loss"], rtol=REL)
    # the straight-through term alone would already give grad = w: compare what is left of it as well
    got, ref, w = x.grad.cpu(), fx["grad_x"], fx["w"]
    assert gu.rel_err(got, ref) <= REL
    assert gu.rel_err(got - w, ref - w) <= 1e-3, gu.rel_err(got - w, ref - w)
    for cb, after in zip(books, fx["after"]):
        assert torch.equal(cb.cluster_size.cpu(), after["cluster_size"])
        assert gu.rel_err(cb.embeddings.cpu(), after["embeddings"]) <= REL


@pytest.mark.parametrize("name", ["inplace_sgd", "inplace_sgd_masked"])
def test_in_place_codebook_optimizer_matches_reference_fixture(name):
    """in_place_codebook_optimizer (reference vector_quantize_pytorch.py:233-256): an SGD step on the learnable codebook
    inside forward (search + gather kernels, codebook gradient = segmented sum), then the pass whose results are
    returned -- outputs, the stepped codebook and both gradients against the live reference."""
    import os
    from vqb200 import CodebookParams, VectorQuantize
    fx = torch.load(os.path.join(gu.GOLDEN_DIR, "learnable", name + ".pt"), weights_only=False)
    cfg = fx["cfg"]
    cp = CodebookParams(dim=cfg["dim"], codebook_size=cfg["K"], learnable_codebook=True, ema_update=False,
                        threshold_ema_dead_code=0)
    vq = VectorQuantize(dim=cfg["dim"], codebook_params=cp, commitment_weight=cfg["cw"], sync_update_v=cfg["v"],
                        sync_codebook=False,
                        in_place_codebook_optimizer=lambda p: torch.optim.SGD(p, lr=cfg["lr"])).to(_dev()).train()
    with torch.no_grad():
        vq._codebook.embeddings.copy_(fx["init_embeddings"])
    vq._codebook.invalidate_cache()
    x = fx["x"].to(_dev()).requires_grad_(True)
    mask = fx["mask"].to(_dev()) if fx["mask"] is not None else None
    q, ind, loss, bd = vq(x, mask=mask, return_loss_breakdown=True)
    (q * fx["w"].to(_dev())).sum().add(loss.sum() * 1.7).backward()
    assert torch.allclose(bd.inplace_optimize.cpu(), fx["inplace_optimize"], rtol=1e-6)
    assert gu.rel_err(vq._codebook.embeddings.detach().cpu(), fx["after_embeddings"]) <= 1e-6
    assert torch.equal(ind.cpu(), fx["indices"])
    assert gu.rel_err(q.detach().cpu(), fx["quantize"]) <= 1e-6      # gathered from the stepped codebook
    assert torch.allclose(loss.detach().cpu(), fx["loss"], rtol=1e-5)
    assert torch.allclose(x.grad.cpu(), fx["grad_x"], rtol=1e-5, atol=1e-7)
    assert gu.rel_err(vq._codebook.embeddings.grad.cpu(), fx["grad_embeddings"]) <= 1e-5
    # eval / freeze_codebook: no step
    before = vq._codebook.embeddings.detach().clone()
    vq(fx["x"].to(_dev()), mask=mask, freeze_codebook=True)
    vq.eval()
    vq(fx["x"].to(_dev()), mask=mask)
    assert torch.equal(vq._codebook.embeddings.detach(), before)


@pytest.mark.parametrize("cos", [False, True])
@pytest.mark.parametrize("case", ["mixed_row_scales", "zero_codebook", "huge_codes_tiny_rows", "huge_rows_tiny_codes",
                                  "padded_codes", "constant_rows"])
@pytest.mark.parametrize("N", [3000, 100])
def test_search_scale_extremes_match_exact_scan(N, case, cos):
    """The bias k-step folds s_row 2^-q and s_c 2^q |c|^2/2 into fp16 operands: rows / codebooks at the edges of those
    ranges (zero rows, 10 orders of magnitude between rows, all-zero codebook, bias far larger or smaller than the dot
    products, padded code columns) must still give the exact scan's answer, index and score, bit for bit.  N = 100 is
    one row tile: that search adds the bias in the epilogue of the single-CTA kernel instead."""
    from vqb200 import ops
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    K, d = 1024, 128
    x = torch.randn(1, N, d, generator=g)
    c = torch.randn(1, K, d, generator=g) * 0.5
    if case == "mixed_row_scales":
        scale = 10.0 ** torch.randint(-6, 5, (N, 1), generator=g).float()
        x = x * scale
        x[0, :50] = 0.0
        x[0, 50:60] = 1e-30
    elif case == "zero_codebook":
        c = torch.zeros(1, K, d)
        c[0, 5] = 1e-3
    elif case == "huge_codes_tiny_rows":
        c, x = c * 1e3, x * 1e-4
    elif case == "huge_rows_tiny_codes":
        c, x = c * 1e-3, x * 1e4
    elif case == "padded_codes":
        K = 1000
        c = c[:, :K].contiguous()
    elif case == "constant_rows":
        x = torch.ones(1, N, d) * torch.linspace(-3, 3, N)[None, :, None]
    if cos:
        c = torch.nn.functional.normalize(c, dim=-1) if case != "zero_codebook" else c
    xd, cd = x.to(_dev()).contiguous(), c.to(_dev()).contiguous()
    cache = ops.prepare_codebook(cd, cos)
    idx, score, ws = ops.search(xd, cd, cache, cos, want_score=True)
    st = ops.search_stats(ws)
    ex, es, _ = ops.search(xd, cd, None, cos, force_exact=True, want_score=True)
    assert st["tensor_core_pass"] == 1
    assert torch.equal(idx, ex), f"{case}: {int((idx != ex).sum())} rows differ from the exact scan; stats {st}"
    assert torch.equal(score, es)


def test_cosine_input_gradient_passes_through_the_normalisation():
    """transform_input="l2norm": d loss / d x must include the Jacobian of x -> x / |x| (reference: F.normalize under
    autograd), and the no-grad path (normalisation fused with the search's operand preparation) must give the same
    forward results as the differentiable one."""
    from vqb200 import CodebookParams, VectorQuantize
    torch.manual_seed(0)
    cp = CodebookParams(dim=64, codebook_size=96, use_cosine_sim=True, transform_input="l2norm",
                        weights_regularization="l2norm", threshold_ema_dead_code=0)
    vq = VectorQuantize(dim=64, codebook_params=cp, sync_codebook=False).to(_dev()).train()
    g = torch.Generator().manual_seed(4)
    x = (torch.randn(3, 200, 64, generator=g) * 2.5)
    w = torch.randn(3, 200, 64, generator=g)
    emb0 = vq._codebook.embeddings.clone()
    xd = x.to(_dev()).requires_grad_(True)
    q, ind, loss = vq(xd)
    (q * w.to(_dev())).sum().add(loss.sum() * 0.9).backward()
    # torch restatement with the indices the module chose
    xr = x.clone().requires_grad_(True)
    xn = torch.nn.functional.normalize(xr, p=2, dim=-1)
    cq = emb0[0].cpu()[ind.cpu()]
    qr = xn + (cq - xn).detach()
    lr = torch.nn.functional.mse_loss(cq, xn)
    (qr * w).sum().add(lr * 0.9).backward()
    # (torch's CUDA and CPU normalisations reduce in different orders: last-bit differences in x^ are expected here)
    assert torch.allclose(q.detach().cpu(), qr.detach(), rtol=1e-6, atol=1e-7)
    assert torch.allclose(loss.detach().cpu(), lr.detach().reshape(1), rtol=1e-5)
    assert torch.allclose(xd.grad.cpu(), xr.grad, rtol=1e-4, atol=1e-6)
    # same forward through the fused no-grad path (fresh module with the same initial codebook)
    vq2 = VectorQuantize(dim=64, codebook_params=cp, sync_codebook=False).to(_dev()).train()
    vq2._codebook.embeddings.copy_(emb0); vq2._codebook.embed_avg.copy_(emb0); vq2._codebook.invalidate_cache()
    with torch.no_grad():
        q2, ind2, loss2 = vq2(x.to(_dev()))
    assert float((ind2 == ind).float().mean()) > 0.999
    same = (ind2 == ind)[..., None].expand_as(q2)
    assert torch.allclose(q2[same], q.detach()[same], rtol=1e-6, atol=1e-7) and torch.allclose(loss2, loss.detach(), rtol=1e-5)
    assert torch.allclose(vq2._codebook.embeddings, vq._codebook.embeddings, rtol=1e-4, atol=1e-6)


def test_minkey_roundtrip_and_order():
    from vqb200 import ops
    g = torch.Generator().manual_seed(2)
    score = torch.randn(1000, generator=g) * 10
    score[:10] = 0.0
    score[10:20] = -0.0
    idx = torch.randint(0, 1 << 20, (1000,), generator=g)
    keys = ops.minkey_pack(score.to(_dev()), idx.to(_dev()))
    i2, s2 = ops.minkey_unpack(keys, want_score=True)
    assert torch.equal(i2.cpu(), idx)
    assert torch.equal(s2.cpu().abs(), score.abs()) and torch.equal(s2.cpu()[20:], score[20:])
    k = keys.cpu()
    order = torch.argsort(k, stable=True)
    s_sorted = score[order]
    assert bool((s_sorted[1:] >= s_sorted[:-1]).all())


def test_state_dict_roundtrip_and_cache_invalidation():
    from vqb200 import CodebookParams, VectorQuantize
    vq = VectorQuantize(dim=32, codebook_params=CodebookParams(dim=32, codebook_size=64, threshold_ema_dead_code=0)).to(_dev())
    x = torch.randn(2, 50, 32, device=_dev())
    vq.eval()
    _, i0, _ = vq(x)
    sd = {k: v.clone() for k, v in vq.state_dict().items()}
    assert set(sd) == {"_codebook.cluster_size", "_codebook.embed_avg", "_codebook.embeddings"}
    new = torch.randn(1, 64, 32, device=_dev())
    sd["_codebook.embeddings"] = new
    vq.load_state_dict(sd)
    _, i1, _ = vq(x)
    ref = (-torch.cdist(x.reshape(1, -1, 32).cpu(), new.cpu())).argmax(-1).reshape(2, 50)
    assert torch.equal(i1.cpu(), ref), "search must see embeddings written through load_state_dict"


@pytest.mark.parametrize("H,N,K,d,cos", [(1, 700, 300, 72, False), (2, 1500, 520, 256, True),
                                         (1, 40000, 2048, 128, False), (1, 257, 4096, 512, False)])
def test_default_search_kernels_match_exact_scan(H, N, K, d, cos):
    """The tensor-core search must give the exact scan's indices: several heads, both metrics, many row tiles, d = 512."""
    from vqb200 import ops
    g = torch.Generator().manual_seed(N)
    x = torch.randn(H, N, d, generator=g).to(_dev())
    c = (torch.randn(H, K, d, generator=g) * 0.5).to(_dev())
    cache = ops.prepare_codebook(c, cos)
    a, _, ws = ops.search(x, c, cache, cos)
    st = ops.search_stats(ws)
    b, _, _ = ops.search(x, c, cache, cos, force_exact=True)
    assert st["tensor_core_pass"] == 1
    assert torch.equal(a, b), (H, N, K, d, int((a != b).sum()))


@pytest.mark.parametrize("name", gu.rvq_learnable_fixture_names())
def test_rvq_learnable_codebooks_get_their_gradient(name):
    gu.check_rvq_learnable(name, _dev())
