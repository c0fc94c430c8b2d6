"""The fused ResidualVQ kernels against plain statements of what they compute.

`ResidualVQ` runs its level loop on four kernels whenever the input is on the GPU: `vqb_rvq_level` (gather, straight
through, commitment loss, `residual -= q`, `quantized_out += q` and the next level's fp16 search operands),
`vqb_rvq_replay_out` (the sum of the level outputs replayed from x and the indices), `vqb_rvq_backward` (the one-pass
input gradient of `_FusedRVQ`) and `vqb_rvq_level_ema`.  The references here are written in torch in this file:

* fp32 on the device for what the kernels promise bit for bit, with the IEEE operations the kernels state:
  q = live ? (training ? fl(r + fl(c - r)) : c) : r,  out = fl(0 + q) at level 0 and fl(out + q) after,  r' = fl(r - q);
* fp64 for the commitment loss and the input gradient.

Part A tests `rvq_level` alone, at widths on both sides of every loop bound of the kernel (the scalar path for d % 4 != 0,
the 2048-column span of the vector path), masks and row counts that make the persistent grid loop.  Part B checks the
next level's search operands through the search they feed: the tensor-core search on them must equal the exact scan.
Part C tests the replay and the backward at both sides of each `VEC` width and up to the 32-level limit.  Part D runs
the module with the fused loop against the generic per-level loop and, with dead-code expiry at deep levels, against
the oracle."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _cpu_draw(num_rows, m, device):
    # expiry draws on the host generator, so the oracle (CPU) and the module (GPU) replace the same codes by the same rows
    if num_rows >= m:
        return torch.randperm(num_rows)[:m].to(device)
    return torch.randint(0, num_rows, (m,)).to(device)


@pytest.fixture(autouse=True)
def _patch_draw(monkeypatch):
    from vqb200 import codebook
    monkeypatch.setattr(codebook.Codebook, "_draw_rows", staticmethod(_cpu_draw))


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _indices(N, K, g):
    """Random codes with a long run of one code and the last code K - 1 at both ends of the rows."""
    idx = torch.randint(0, K, (N,), generator=g, device=DEV)
    idx[: N // 3] = K // 2
    idx[N // 3: N // 3 + N // 5] = K - 1
    idx[-1] = K - 1
    return idx


def _mask(kind, N, g):
    if kind == "none":
        return None
    if kind == "all_on":
        return torch.ones(N, dtype=torch.uint8, device=DEV)
    if kind == "all_off":
        return torch.zeros(N, dtype=torch.uint8, device=DEV)
    m = (torch.rand(N, generator=g, device=DEV) >= 0.3).to(torch.uint8)
    m[0] = 0
    return m


def ref_level(r, c, idx, live, training):
    """One level in fp32, operation for operation: (q, new residual)."""
    cq = c[idx]
    q = r + (cq - r) if training else cq
    if live is not None:
        q = torch.where(live[:, None] != 0, q, r)
    return q, r - q


def ref_loss(r, c, idx, live):
    """Commitment loss in fp64: mean over the live rows of (c - r)^2, and the number of live rows."""
    err = (c[idx].double() - r.double()) ** 2
    if live is not None:
        err = err[live != 0]
    n = err.shape[0]
    return (float(err.sum()) / (n * r.shape[1]) if n else float("nan")), n


# ------------------------------------------------------------------------------------------------------------- A
LEVEL_D = [1, 3, 4, 5, 37, 64, 102, 132, 256, 260, 510, 512, 516, 2048, 2052, 2560, 4096]
N_BIG = 148 * 8 * 8 * 2 + 77      # more rows than one sweep of the persistent grid (148 SMs x 8 blocks x 8 warps)


@pytest.mark.parametrize("d", LEVEL_D)
def test_rvq_level_matches_fp32_reference(d):
    from vqb200 import ops
    K = 333
    g = _gen(d)
    c = torch.randn(K, d, generator=g, device=DEV) * 0.5
    for N in (1, 7, 5003, N_BIG):
        r = torch.randn(N, d, generator=g, device=DEV)
        idx = _indices(N, K, g)
        prev = torch.randn(N, d, generator=g, device=DEV)
        for mk in ("none", "some_off", "all_off", "all_on"):
            live = _mask(mk, N, g)
            want_loss, want_n = ref_loss(r, c, idx, live)
            for training in (True, False):
                q_ref, rn_ref = ref_level(r, c, idx, live, training)
                for first in (True, False):
                    what = f"d={d} N={N} mask={mk} training={training} first={first}"
                    # unwritten columns must show: NaN where the kernel writes, random values where it accumulates
                    nxt = torch.full((N, d), float("nan"), device=DEV)
                    out = torch.full((N, d), float("nan"), device=DEV) if first else prev.clone()
                    q = torch.full((N, d), float("nan"), device=DEV)
                    loss = ops.rvq_level(r, nxt, c, idx, live, training, first, out, None, q_out=q).cpu()
                    out_ref = (torch.zeros_like(q_ref) if first else prev) + q_ref
                    assert torch.equal(nxt, rn_ref), f"{what}: residual_next, {int((nxt != rn_ref).sum())} values differ"
                    assert torch.equal(q, q_ref), f"{what}: q_out"
                    assert torch.equal(out, out_ref), f"{what}: quantized_out, {int((out != out_ref).sum())} values differ"
                    assert float(loss[1]) == want_n, f"{what}: rows used {float(loss[1])} != {want_n}"
                    if want_n:
                        assert abs(float(loss[0]) - want_loss) <= 1e-6 * want_loss, (what, float(loss[0]), want_loss)
                    else:
                        assert torch.isnan(loss[0]), f"{what}: loss of no rows must be NaN, got {float(loss[0])}"


# ------------------------------------------------------------------------------------------------------------- B
NEXT_D = [d for d in LEVEL_D if (d + 63) // 64 * 64 <= 512]


def _search_pair(nxt, c2, cache2, what):
    """The search on the operands `rvq_level` prepared must be the exact scan, bit for bit, and must have run on the
    tensor cores."""
    from vqb200 import ops
    idx, score, ws = ops.search(nxt[None], c2, cache2, False, latents_prepared=True, want_score=True)
    stats = ops.search_stats(ws)
    idx, score = idx.clone(), score.clone()
    ex_idx, ex_score, _ = ops.search(nxt[None], c2, cache2, False, force_exact=True, want_score=True)
    assert stats["tensor_core_pass"] == 1, f"{what}: {stats}"
    assert torch.equal(idx, ex_idx), f"{what}: {int((idx != ex_idx).sum())} indices differ from the exact scan"
    assert torch.equal(score, ex_score), f"{what}: {int((score != ex_score).sum())} scores differ from the exact scan"


@pytest.mark.parametrize("d", NEXT_D)
def test_rvq_level_next_operands_search_exactly(d):
    from vqb200 import ops
    K, N = 300, 3001           # the next level has as many codes as this one (the workspace layout assumes it)
    g = _gen(100 + d)
    c = torch.randn(K, d, generator=g, device=DEV) * 0.5
    c2 = torch.randn(1, K, d, generator=g, device=DEV) * 0.3
    c2[0, 40:48] = c2[0, 7]                        # planted duplicates: the lowest index must win
    c2[0, K - 1] = c2[0, 11]
    idx = _indices(N, K, g)
    base = torch.randn(N, d, generator=g, device=DEV)
    cases = [
        ("plain", base, c, c2, None),
        ("masked", base, c, c2, _mask("some_off", N, g)),      # masked rows leave an all-zero next residual
        ("scale 1e-20", base * 1e-20, c * 1e-20, c2 * 1e-20, None),
        ("scale 1e6", base * 1e6, c * 1e6, c2 * 1e6, None),
        ("zero residual", c[idx].clone(), c, c2, None),          # r = c exactly: every new residual is 0
        ("all masked", base, c, c2, _mask("all_off", N, g)),
    ]
    for name, r, cc, cc2, live in cases:
        cache2 = ops.prepare_codebook(cc2, False)
        for training in (True, False):
            nxt = torch.empty_like(r)
            ops.rvq_level(r, nxt, cc, idx, live, training, True, None, cache2)
            _, rn_ref = ref_level(r, cc, idx, live, training)
            what = f"d={d} {name} training={training}"
            assert torch.equal(nxt, rn_ref), f"{what}: residual_next"
            if name == "zero residual" and training:
                assert not bool(nxt.any())
            _search_pair(nxt, cc2, cache2, what)
    # stale cache: the next codebook is rebuilt with another 2^q after its operands were prepared; the search must
    # notice (the scale recorded with the operands) and still return the exact result
    cache2 = ops.prepare_codebook(c2, False)
    nxt = torch.empty_like(base)
    ops.rvq_level(base, nxt, c, idx, None, True, True, None, cache2)
    c2s = c2 * 1024.0
    ops.prepare_codebook(c2s, False, out=cache2)
    _search_pair(nxt, c2s, cache2, f"d={d} stale cache")


# ------------------------------------------------------------------------------------------------------------- C
def _levels(Q, K, d, N, g):
    cbs = [torch.randn(K, d, generator=g, device=DEV) * (0.6 / 1.3 ** l) for l in range(Q)]
    idx = [_indices(N, K, g) for _ in range(Q)]
    for l in range(Q):
        idx[l][(l * 37) % N::max(1, N // 7)] = l % K
    training = [l % 3 != 1 for l in range(Q)]
    return cbs, idx, training


def ref_replay(x, cbs, idx, training, live):
    """(sum of the level outputs in fp32, the residual each level saw)"""
    r, out, seen = x, None, []
    for c, i, tr in zip(cbs, idx, training):
        seen.append(r)
        q, r = ref_level(r, c, i, live, tr)
        out = (torch.zeros_like(q) if out is None else out) + q
    return out, seen


@pytest.mark.parametrize("d", [4, 8, 124, 128, 132, 252, 256, 260, 508, 512])
@pytest.mark.parametrize("Q", [1, 2, 3, 31, 32])
def test_rvq_replay_out_and_backward_match_references(d, Q):
    from vqb200 import ops
    K, N = 97, 1203
    g = _gen(1000 * Q + d)
    cbs, idx, training = _levels(Q, K, d, N, g)
    x = torch.randn(N, d, generator=g, device=DEV)
    g_out = torch.randn(N, d, generator=g, device=DEV)
    coef = torch.randn(Q, generator=g, device=DEV) * 0.3
    coef[::2] = 0.0
    for mk in ("none", "some_off", "all_off"):
        live = _mask(mk, N, g)
        out = ops.rvq_replay_out(x, cbs, idx, training, live)
        out_ref, seen = ref_replay(x, cbs, idx, training, live)
        assert torch.equal(out, out_ref), f"d={d} Q={Q} mask={mk}: replay, {int((out != out_ref).sum())} values differ"
        cf = coef.clone()
        if mk == "all_off":       # no live rows: the module's coefficient is a division by zero and must not leak
            cf[0], cf[-1] = float("inf"), float("nan")
        for go in (g_out, None):
            gx = ops.rvq_backward(x, cbs, idx, training, cf, go, live)
            if mk == "all_off":
                want = torch.zeros(N, d, device=DEV) if go is None else float(Q) * go     # fp32, as the kernel
                assert torch.equal(gx, want), f"d={d} Q={Q} g_out={go is not None}: rows without loss must get Q g_out"
                continue
            want = torch.zeros(N, d, dtype=torch.float64, device=DEV) if go is None else Q * go.double()
            scale = want.abs()
            lv = torch.ones(N, 1, dtype=torch.float64, device=DEV) if live is None else live[:, None].double()
            for l in range(Q):
                term = float(cf[l]) * lv * (seen[l].double() - cbs[l][idx[l]].double())
                want = want + term
                scale = scale + term.abs()
            what = f"d={d} Q={Q} mask={mk} g_out={'none' if go is None else 'given'}"
            err = ((gx.double() - want).abs().amax(1) / scale.amax(1).clamp_min(1e-30)).max()
            assert float(err) <= 1e-6, f"{what}: gradient error {float(err):.3g} of the row scale"


def test_rvq_replay_out_supported_limits():
    from vqb200 import ops
    assert ops.rvq_replay_out_supported(512, 32)
    assert not ops.rvq_replay_out_supported(516, 8)
    assert not ops.rvq_replay_out_supported(64, 33)
    assert not ops.rvq_replay_out_supported(250, 4)


# ------------------------------------------------------------------------------------------------------------- D
def _rvq(d, Q, K, threshold, seed, fused):
    from vqb200 import CodebookParams, ResidualVQ
    torch.manual_seed(0)
    rvq = ResidualVQ(dim=d, num_quantizers=Q,
                     codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=threshold)).to(DEV)
    gen = torch.Generator().manual_seed(seed)
    for li, layer in enumerate(rvq.layers):
        c = torch.randn(1, K, d, generator=gen) * (0.6 / 1.3 ** li)
        c[0, K - 4:] = c[0, 1]                  # duplicates: they lose every row and die when expiry is on
        cb = layer._codebook
        with torch.no_grad():
            cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0)
        cb.invalidate_cache()
    rvq.use_fused_levels = fused
    return rvq


def _inputs(B, n, d, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, n, d, generator=gen)
    w = torch.randn(B, n, d, generator=gen)
    mask = torch.rand(B, n, generator=gen) >= 0.3
    return x.to(DEV), w.to(DEV), mask.to(DEV)


def _buffers(rvq):
    return [(l._codebook.embeddings.detach().clone(), l._codebook.embed_avg.clone(), l._codebook.cluster_size.clone())
            for l in rvq.layers]


def _compare(a, b, what, grads=False):
    (qa, ia, la, ba), (qb, ib, lb, bb) = a[:4], b[:4]
    assert torch.equal(ia, ib), f"{what}: {int((ia != ib).sum())} indices differ"
    assert torch.equal(qa, qb), f"{what}: quantized_out differs"
    assert _rel(la, lb) <= 1e-6, (what, la, lb)
    for li, (x, y) in enumerate(zip(ba, bb)):
        for name, s, t in zip(("embeddings", "embed_avg", "cluster_size"), x, y):
            assert _rel(s, t) <= 1e-6, f"{what}: level {li} {name} {_rel(s, t)}"
    if grads:
        assert _rel(a[4], b[4]) <= 1e-6, f"{what}: input gradient {_rel(a[4], b[4])}"


def _forward(rvq, x, mask=None, train=True):
    rvq.train(train)
    torch.manual_seed(7)
    with torch.no_grad():
        q, ind, losses = rvq(x, mask=mask)
    return q, ind, losses, _buffers(rvq)


@pytest.mark.parametrize("d,Q,mask", [(132, 3, False), (250, 3, False), (2560, 2, False), (64, 33, False),
                                      (128, 4, True), (260, 3, True)])
def test_fused_loop_equals_generic_loop(d, Q, mask):
    """d = 132: replay with VEC = 2; d = 250: the scalar level path, no replay; d = 2560: rows wider than 2048;
    Q = 33: more levels than the replay takes; masks over distinct codebooks with EMA."""
    K = 64
    x, _, m = _inputs(2, 150, d, d + Q)
    res = {f: _forward(_rvq(d, Q, K, 0, d, f), x, m if mask else None) for f in (True, False)}
    _compare(res[True], res[False], f"d={d} Q={Q} mask={mask}")


def test_fused_loop_equals_generic_loop_in_eval_mode():
    d, Q, K = 132, 4, 64
    x, _, m = _inputs(2, 150, d, 3)
    for mask in (None, m):
        res = {f: _forward(_rvq(d, Q, K, 2, 5, f), x, mask, train=False) for f in (True, False)}
        _compare(res[True], res[False], f"eval mask={mask is not None}")


def test_fused_masked_expiry_at_deep_levels_matches_generic_loop_and_oracle():
    """Dead-code expiry at levels > 0 with a mask: the fused loop answers all levels' checks after the loop and replays
    the masked residual of each expiring level (`_fused_expiry`)."""
    from oracle import vq_oracle as O
    d, Q, K = 64, 4, 64
    x, _, m = _inputs(2, 300, d, 11)
    res = {}
    for f in (True, False):
        rvq = _rvq(d, Q, K, 2, 13, f)
        pre = [(l._codebook.embeddings.detach().cpu().clone()) for l in rvq.layers]
        res[f] = _forward(rvq, x, m)
    _compare(res[True], res[False], "masked expiry")
    # expiry fired at a level > 0: codes reset to cluster_size == threshold
    assert any(bool((b[2] == 2.0).any()) for b in res[True][3][1:]), "no code expired at a level > 0"
    sts = [O.CodebookState(e.clone(), e.clone(), torch.ones(1, K)) for e in pre]
    torch.manual_seed(7)
    qo, io, lo, extras = O.rvq_forward(sts, x.cpu(), O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=2)),
                                       training=True, mask=m.cpu(), want_gap=True)
    q, ind, losses, bufs = res[True]
    got, ref = ind.cpu().reshape(-1, Q), io.reshape(-1, Q)
    alive = torch.ones(got.shape[0], dtype=torch.bool)       # rows whose residual is still identical
    n_flips = 0
    for li in range(Q):
        diff = (got[:, li] != ref[:, li]) & alive
        gap = extras[li]["top2_rel_gap"].reshape(-1)
        assert bool((gap[diff] < 1e-6).all()), f"level {li}: index mismatches outside the 1e-6 window"
        n_flips += int(diff.sum())
        alive &= ~diff
    assert torch.equal(q.cpu().reshape(-1, d)[alive], qo.reshape(-1, d)[alive]), "quantized_out differs from the oracle"
    if n_flips == 0:
        assert torch.allclose(losses.cpu(), lo, rtol=1e-5), (losses, lo)
        for li, ((em, ea, cs), st) in enumerate(zip(bufs, sts)):
            assert torch.equal(cs.cpu(), st.cluster_size), f"level {li}: cluster_size"
            assert _rel(ea.cpu(), st.embed_avg) <= 1e-5 and _rel(em.cpu(), st.embeddings) <= 1e-5, f"level {li}"


def _train_step(rvq, x, w, mask, freeze=False):
    q, ind, losses = rvq(x, mask=mask, freeze_codebook=freeze)
    Q = losses.shape[-1]
    return q, ind, losses, (q * w).sum() + (losses * torch.arange(1, Q + 1, device=DEV)).sum() * 3.0


@pytest.mark.parametrize("d", [132, 260])
def test_fused_autograd_with_mask_equals_generic_loop(d):
    Q, K = 3, 64
    x0, w, m = _inputs(2, 200, d, d)
    res = {}
    for f in (True, False):
        rvq = _rvq(d, Q, K, 0, d, f).train()
        x = x0.clone().requires_grad_(True)
        torch.manual_seed(7)
        q, ind, losses, obj = _train_step(rvq, x, w, m)
        obj.backward()
        res[f] = (q.detach(), ind, losses.detach(), _buffers(rvq), x.grad.clone())
    _compare(res[True], res[False], f"autograd d={d}", grads=True)


def test_fused_autograd_keeps_the_frozen_codebook_of_its_forward():
    """Forward A with `freeze_codebook`, then forward B of the same module without it (its EMA step moves the codebooks
    in place), then one backward through both (gradient accumulation).  A's gradient must use the codebooks A gathered
    from: it must equal the gradient of A taken before B ran, in both loops, and the two loops must agree."""
    d, Q, K = 128, 3, 64
    xa0, wa, _ = _inputs(2, 200, d, 21)
    xb0, wb, _ = _inputs(2, 200, d, 22)
    res = {}
    for f in (True, False):
        grads = {}
        for late in (True, False):
            rvq = _rvq(d, Q, K, 0, 23, f).train()
            xa, xb = xa0.clone().requires_grad_(True), xb0.clone().requires_grad_(True)
            torch.manual_seed(7)
            qa, ia, la, oa = _train_step(rvq, xa, wa, None, freeze=True)
            if not late:
                oa.backward()
            qb, ib, lb, ob = _train_step(rvq, xb, wb, None)
            (oa + ob).backward() if late else ob.backward()
            grads[late] = (xa.grad.clone(), xb.grad.clone())
        assert _rel(grads[True][0], grads[False][0]) <= 1e-6, \
            f"fused={f}: the frozen forward's gradient changed when the codebooks moved before backward " \
            f"({_rel(grads[True][0], grads[False][0]):.3g})"
        assert torch.equal(grads[True][1], grads[False][1])
        res[f] = (torch.cat([qa, qb]).detach(), torch.cat([ia, ib]), torch.cat([la, lb]).detach(), _buffers(rvq),
                  torch.cat(grads[True]))
    _compare(res[True], res[False], "freeze_codebook then training forward", grads=True)


def test_fused_autograd_misaligned_output_gradient():
    """The gradient of `quantized_out` arrives as a view one float into a larger buffer (the second input of a cat)."""
    d, Q, K = 132, 3, 64
    x0, w, m = _inputs(2, 200, d, 31)
    res = {}
    for f in (True, False):
        rvq = _rvq(d, Q, K, 0, 32, f).train()
        x = x0.clone().requires_grad_(True)
        torch.manual_seed(7)
        q, ind, losses = rvq(x, mask=m)
        flat = torch.cat([torch.zeros(1, device=DEV), q.reshape(-1)])
        wf = torch.cat([torch.ones(1, device=DEV), w.reshape(-1)])
        ((flat * wf).sum() + losses.sum()).backward()
        res[f] = (q.detach(), ind, losses.detach(), _buffers(rvq), x.grad.clone())
    _compare(res[True], res[False], "misaligned output gradient", grads=True)
