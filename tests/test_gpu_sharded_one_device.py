"""The sharded codebook (Codebook.sharded: rank r owns codes [r K/W, (r+1) K/W)) with the real kernels on ONE device.

Part 1, op level, one process: the codebook is split into W contiguous shards on cuda:0 and each shard runs exactly
what rank r runs; each collective is replaced by its definition (all_reduce(MIN) of the packed (score, global index)
keys = torch.minimum over the W key tensors, all_reduce(SUM) of the per-shard EMA totals = their sum in rank order).
  a. search + min-key merge == the un-sharded search, bit for bit (index and score), and == the oracle's argmax outside
     its own fp32 1e-6 top-2 window; planted edges (cross-shard duplicates, rows equidistant from two shards, winning
     scores of exactly 0 in several shards, a shard that wins nothing, N not a multiple of the row tile);
  b. EMA refresh on shards (vqb_ema_apply_counts / vqb_ema_apply_rows with k_total = K) == vqb_ema_apply on the whole
     codebook, and both == an fp64 restatement of the reference refresh;
  c. expiry on shard views == one expire_scatter on the whole codebook == a torch restatement of the reference.
Part 2, module level: tools/mgpu_check.py in its single-device mode (2 ranks on cuda:0 over Gloo).

Signed zeros.  The packed keys order -0.0 before +0.0 while the un-sharded search compares floats, so the merge equals
the un-sharded search only if a zero score has ONE sign for every code of a row.  The kernels guarantee that: the dot
score is float(-dot) with dot an fma chain started at +0.0, and IEEE round-to-nearest never produces -0.0 from such a
chain (a sum of opposite zeros or of x and -x is +0.0), so a zero dot score is always -0.0; the euclidean score is
sqrtf(fmaxf(d2, 0)) with d2 = float(|x|^2 + |c|^2 - 2 x.c) = +0.0 when x == c, so a zero distance is +0.0.
`_check_zero_signs` checks this on every row where some shard scores exactly 0."""
import ctypes
import os
import signal
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24                 # unit roundoff of fp32


# ------------------------------------------------------------------------------------------------ a. search + merge
def _shard_search(x, c, W, cos):
    """What W ranks compute: per-shard search with the global index offset, packed keys, min over the shards."""
    from vqb200 import ops
    H, K, d = c.shape
    Ks = K // W
    keys, per_shard = None, []
    for r in range(W):
        sh = c[:, r * Ks:(r + 1) * Ks].contiguous()
        idx, score, ws = ops.search(x, sh, ops.prepare_codebook(sh, cos), cos, idx_offset=r * Ks, want_score=True)
        per_shard.append((idx, score, ops.search_stats(ws)))
        k = ops.minkey_pack(score.reshape(-1), idx.reshape(-1))
        keys = k if keys is None else torch.minimum(keys, k)
    gidx, gscore = ops.minkey_unpack(keys, want_score=True)
    return gidx.reshape(idx.shape), gscore.reshape(idx.shape), per_shard


def _bits(t):
    return t.contiguous().view(torch.int32)


def _check_zero_signs(per_shard, ref_score):
    """Every exact-zero score a shard emits for a row has the sign bit of the un-sharded search's zero (if any)."""
    for r, (_, score, _) in enumerate(per_shard):
        z = score == 0
        if bool(z.any()):
            signs = torch.signbit(score[z])
            assert bool((signs == signs[0]).all()), f"shard {r} emits both -0.0 and +0.0 scores"
            rz = (ref_score == 0) & z
            if bool(rz.any()):
                assert bool((torch.signbit(ref_score[rz]) == signs[0]).all()), f"shard {r}: zero sign differs"


def _merge_matches_unsharded(x, c, W, cos, sample=4096):
    from test_gpu_fullsize import _sample_check
    from vqb200 import ops
    ref_idx, ref_score, _ = ops.search(x, c, ops.prepare_codebook(c, cos), cos, want_score=True)
    gidx, gscore, per_shard = _shard_search(x, c, W, cos)
    n_bad = int((gidx != ref_idx).sum())
    assert n_bad == 0, f"W={W}: {n_bad} merged indices differ from the un-sharded search"
    assert torch.equal(_bits(gscore), _bits(ref_score)), f"W={W}: merged scores differ from the un-sharded search"
    _check_zero_signs(per_shard, ref_score)
    if sample:
        _sample_check(x, c, gidx, cos, n_sample=sample, seed=W)
    return gidx, per_shard


def _latents(N, d, cos, dtype, seed):
    from vqb200 import ops
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(1, N, d, generator=g, device=DEV)
    if cos:
        x = ops.l2norm_rows(x)
    return x.to(dtype).contiguous(), g


def _codebook(K, d, cos, g):
    c = torch.randn(1, K, d, generator=g, device=DEV) * 0.5
    return torch.nn.functional.normalize(c, dim=-1) if cos else c


def test_c5_full_size_merge_two_and_eight_shards():
    """BASELINE config C5: N = 2^22, K = 65536, d = 64, fp32, W = 2 and 8."""
    x, g = _latents(1 << 22, 64, False, torch.float32, 11)
    c = _codebook(65536, 64, False, g)
    for W in (2, 8):
        _, per_shard = _merge_matches_unsharded(x, c, W, False)
        assert all(st["tensor_core_pass"] == 1 for _, _, st in per_shard)


@pytest.mark.parametrize("name,N,K,d,W,cos,dtype", [
    ("bf16_cosine_d256", 1 << 18, 65536, 256, 4, True, torch.bfloat16),
    ("three_shards", (1 << 18) + 77, 98304, 64, 3, False, torch.float32),
])
def test_merge_equals_unsharded_search(name, N, K, d, W, cos, dtype):
    x, g = _latents(N, d, cos, dtype, 12)
    c = _codebook(K, d, cos, g)
    _merge_matches_unsharded(x, c, W, cos)


def test_merge_at_d640_takes_the_exact_scan_on_every_shard():
    """d = 640 has no tensor-core pass (d_pad > 512): every shard settles every row in the exact scan."""
    x, g = _latents(20000 + 77, 640, False, torch.float32, 13)
    c = _codebook(8192, 640, False, g)
    _, per_shard = _merge_matches_unsharded(x, c, 2, False)
    assert all(st["tensor_core_pass"] == 0 for _, _, st in per_shard)


def _planted(cos, K=8192, W=4, d=64, n_rand=30000 + 77):
    """Codebook and rows with the edges of a cross-shard merge; returns (x, c, {name: (rows, expected index)})."""
    g = torch.Generator().manual_seed(5)
    Ks = K // W
    c = torch.randn(K, d, generator=g) * 0.5
    rows, expect = [], {}

    def add(name, r, want):
        lo = sum(t.shape[0] for t in rows)
        rows.append(r)
        expect[name] = (torch.arange(lo, lo + r.shape[0]), want)

    if cos:
        c = torch.nn.functional.normalize(c, dim=-1)
        # dot score exactly 0 against EVERY code (in every shard): zero rows, and rows orthogonal to all codes
        c[:, :8] = 0.0
        c = torch.nn.functional.normalize(c, dim=-1)
        orth = torch.zeros(16, d)
        orth[:, :8] = torch.randn(16, 8, generator=g)
        add("zero_rows", torch.zeros(8, d), 0)
        add("orthogonal_rows", torch.nn.functional.normalize(orth, dim=-1), 0)
        # cross-shard duplicate: a row on the code itself; the copy in the last shard must lose
        c[(W - 1) * Ks + 5] = c[17]
        add("duplicate", c[17][None].repeat(8, 1), 17)
    else:
        # cross-shard duplicate; many copies of one code in two shards (more ties than the candidate slots of a row:
        # the tiled rescan settles these rows), rows exactly on them score 0 in both shards
        c[(W - 2) * Ks + 5] = c[17]
        c[Ks + 100:Ks + 140] = c[Ks + 99]
        c[2 * Ks + 200:2 * Ks + 240] = c[Ks + 99]
        add("duplicate", c[17][None] + 0.01 * torch.randn(8, d, generator=g), 17)
        add("zero_in_several_shards", c[Ks + 99][None].repeat(8, 1), Ks + 99)
        # rows equidistant from the last code of shard r and the first code of shard r+1: dyadic values, so every
        # product and sum of the fp64 score is exact and the two scores are EQUAL; the lower index wins
        for r in range(1, W - 1):
            p = torch.round(torch.randn(d, generator=g) * 16) / 16 + 8.0
            v = torch.zeros(d)
            v[r] = 0.5
            c[r * Ks - 1], c[r * Ks] = p + v, p - v
            add(f"equidistant_{r}", p[None].repeat(4, 1), r * Ks - 1)
        c[(W - 1) * Ks:] *= 100.0                  # far away: the last shard wins no row
    xr = torch.randn(n_rand, d, generator=g)
    if cos:
        xr = torch.nn.functional.normalize(xr, dim=-1)
    x = torch.cat(rows + [xr], 0)
    return x[None].to(DEV).contiguous(), c[None].to(DEV).contiguous(), expect, Ks


@pytest.mark.parametrize("cos", [False, True], ids=["euclid", "cosine"])
def test_merge_planted_edges(cos):
    W = 4
    x, c, expect, Ks = _planted(cos, W=W)
    assert x.shape[1] % 128 != 0 and x.shape[1] % 256 != 0
    gidx, per_shard = _merge_matches_unsharded(x, c, W, cos)
    for name, (rows, want) in expect.items():
        got = gidx[0, rows.to(DEV)]
        assert bool((got == want).all()), f"{name}: {got.tolist()} != {want}"
    if not cos:
        assert bool((gidx < (W - 1) * Ks).all()), "the far shard won a row"
        assert any(st["reranked_rows"] > 0 for _, _, st in per_shard), [st for _, _, st in per_shard]
        assert any(st["rescanned_rows"] > 0 for _, _, st in per_shard), [st for _, _, st in per_shard]
    else:
        # zero and orthogonal rows: every shard scores exactly -0.0 for them
        zr = torch.cat([expect["zero_rows"][0], expect["orthogonal_rows"][0]]).to(DEV)
        for _, score, _ in per_shard:
            assert bool((score[0, zr] == 0).all()) and bool(torch.signbit(score[0, zr]).all())


# ------------------------------------------------------------------------------------------------ b. EMA refresh
def _ema_apply_shards(stats, cs, ea, em, w, eps, l2, W):
    """What W ranks run in ops.ema_apply_sharded, with the all_reduce(SUM) of the totals as a sum in rank order."""
    from vqb200 import _lib as L
    H, K, d1 = stats.shape
    d, Ks = d1 - 1, K // W
    st = L.stream_ptr(stats.device)
    views, totals = [], []
    for r in range(W):
        sl = slice(r * Ks, (r + 1) * Ks)
        v = (stats[:, sl].contiguous(), cs[:, sl].contiguous(), ea[:, sl].contiguous(), em[:, sl].contiguous())
        t = torch.empty(H, dtype=torch.float32, device=stats.device)
        L.check(L.lib().vqb_ema_apply_counts(L.ptr(v[0]), L.ptr(v[1]), float(w), H, Ks, d, L.ptr(t), st),
                "vqb_ema_apply_counts")
        views.append(v)
        totals.append(t)
    total = totals[0].clone()
    for t in totals[1:]:
        total = total + t
    for v in views:
        L.check(L.lib().vqb_ema_apply_rows(L.ptr(v[0]), L.ptr(v[1]), L.ptr(v[2]), L.ptr(v[3]), float(w),
                                           ctypes.c_double(eps), K, int(l2), H, Ks, d, L.ptr(total), st),
                "vqb_ema_apply_rows")
    return tuple(torch.cat([v[i] for v in views], 1) for i in (1, 2, 3))


def _ema_fp64(stats, cs, ea, w, eps, l2):
    """reference codebooks.py:410-425 in fp64: lerp, Laplace smoothing with K eps, divide, optional l2norm."""
    s, cs, ea = stats.double(), cs.double(), ea.double()
    K = cs.shape[-1]
    cs = cs + w * (s[..., -1] - cs)
    ea = ea + w * (s[..., :-1] - ea)
    total = cs.sum(-1, keepdim=True)
    smoothed = (cs + eps) / (total + K * eps) * total
    em = ea / smoothed[..., None]
    if l2:
        em = em / em.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    return cs, ea, em


def _rowrel(a, ref):
    """max over rows of max|a - ref| / max|ref| (the row's own scale)."""
    a, ref = a.double(), ref.double()
    err = (a - ref).abs().amax(-1)
    return float((err / ref.abs().amax(-1).clamp_min(1e-300)).max())


def _ema_inputs(H, K, d, kind, seed):
    from vqb200 import ops
    g = torch.Generator(device=DEV).manual_seed(seed)
    N = 1 if kind == "tiny" else 4 * K
    x = torch.randn(H, N, d, generator=g, device=DEV)
    c = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    idx, _, ws = ops.search(x, c, ops.prepare_codebook(c, False), False)
    if ops.quantize_ema_supported(d):
        _, _, stats = ops.quantize_ema(x, c, idx, False, False, bound_ws=ws)
    else:
        stats = ops.ema_reduce(x, idx, None, K)
    cs = torch.rand(H, K, generator=g, device=DEV) * 3.0
    ea = torch.randn(H, K, d, generator=g, device=DEV)
    if kind == "tiny":
        cs.fill_(1e-7)
    return stats.contiguous(), cs, ea, c.clone()


@pytest.mark.parametrize("H,K,d,W,l2,kind,eps", [
    (1, 65536, 64, 8, False, "plain", 1e-5),
    (1, 65536, 64, 8, True, "plain", 1e-5),
    (2, 6144, 64, 3, False, "zero_shard", 1e-5),
    (3, 12288, 32, 4, True, "tiny", 1e-3),
    (3, 12288, 48, 4, False, "plain", 1e-5),
], ids=["C5_l2off", "C5_l2on", "zero_shard_H2", "tiny_counts_H3_l2on", "H3"])
def test_ema_refresh_on_shards(H, K, d, W, l2, kind, eps):
    from vqb200 import ops
    w = 1 - 0.8
    stats, cs0, ea0, em0 = _ema_inputs(H, K, d, kind, 7)
    if kind == "zero_shard":                   # shard 1: no rows won, and every count in it was already 0
        Ks = K // W
        stats[:, Ks:2 * Ks] = 0.0
        cs0[:, Ks:2 * Ks] = 0.0
    if kind == "tiny":                          # eps dominates the Laplace smoothing: K eps >> total
        assert float(cs0.sum(-1).max()) * (1 - w) + w < 0.1 * K * eps
    cs_w, ea_w, em_w = cs0.clone(), ea0.clone(), em0.clone()
    ops.ema_apply(stats, cs_w, ea_w, em_w, w, eps, l2)
    cs_s, ea_s, em_s = _ema_apply_shards(stats, cs0.clone(), ea0.clone(), em0.clone(), w, eps, l2, W)
    assert torch.equal(cs_s, cs_w), "cluster_size: sharded refresh differs from the whole-codebook refresh"
    assert torch.equal(ea_s, ea_w), "embed_avg: sharded refresh differs from the whole-codebook refresh"
    # The only difference is the total: whole = fl(T), sharded = W fp32 shard totals fl(T_r) added in W-1 fp32
    # additions, so |t_s - t_w| <= (W + 1) u t (all terms >= 0).  The Laplace factor t / (t + K eps) passes a
    # relative change of t through with a gain <= 1; then each side rounds its own add, divide, multiply (smoothed)
    # and divide (embeddings): 4 more u per side.  With l2norm the common factor cancels, and what is left is the
    # rounding of each side's norm: its fp32 sum of d squares (<= (d/32 + 5) u with 32 lanes and a 5-step shuffle
    # tree), halved by the square root, and two divisions per side.
    bound = ((W + 1) + 8 + ((d / 32 + 5) + 4 if l2 else 0)) * U
    rel = (em_s.double() - em_w.double()).abs() / em_w.double().abs().clamp_min(1e-30)
    rel = torch.where(em_w == 0, (em_s != 0).double(), rel)
    assert float(rel.max()) <= bound, f"embeddings: sharded vs whole {float(rel.max()):.3e} > {bound:.3e}"
    cs64, ea64, em64 = _ema_fp64(stats, cs0, ea0, w, eps, l2)
    for name, (a, ref) in {"cluster_size": (cs_w, cs64), "embed_avg": (ea_w, ea64), "embeddings": (em_w, em64),
                           "sharded embeddings": (em_s, em64)}.items():
        r = _rowrel(a, ref) if a.ndim == 3 else float((a.double() - ref).abs().max() / ref.abs().max())
        assert r <= 1e-6, f"{name} vs fp64 reference: {r:.3e}"


def test_ema_apply_odd_K_matches_fp64():
    from vqb200 import ops
    H, K, d, w, eps = 3, 12345, 64, 0.2, 1e-5
    stats, cs0, ea0, em0 = _ema_inputs(H, K, d, "plain", 9)
    for l2 in (False, True):
        cs, ea, em = cs0.clone(), ea0.clone(), em0.clone()
        ops.ema_apply(stats, cs, ea, em, w, eps, l2)
        cs64, ea64, em64 = _ema_fp64(stats, cs0, ea0, w, eps, l2)
        assert float((cs.double() - cs64).abs().max() / cs64.abs().max()) <= 1e-6
        assert _rowrel(ea, ea64) <= 1e-6 and _rowrel(em, em64) <= 1e-6, (l2, _rowrel(ea, ea64), _rowrel(em, em64))


# ------------------------------------------------------------------------------------------------ c. expiry
def _expire_shards(x_rows, rows, thr, reset, l2, cs, ea, em, W):
    """Codebook._expire_codes_sharded with the collectives written out: the dead codes of all shards, in ascending
    global order, take `rows` in order, so shard r takes the slice after the dead codes of the shards before it."""
    from vqb200 import ops
    K = cs.shape[0]
    Ks = K // W
    counts = [int((cs[r * Ks:(r + 1) * Ks] < thr).sum()) for r in range(W)]
    first = 0
    for r in range(W):
        sl = slice(r * Ks, (r + 1) * Ks)
        m = counts[r]
        if m:
            ops.expire_scatter(x_rows, rows[first:first + m], thr, reset, l2, cs[sl], ea[sl], em[sl])
        first += m


@pytest.mark.parametrize("dtype,l2", [(torch.float32, False), (torch.bfloat16, False), (torch.float32, True)],
                         ids=["fp32", "bf16", "fp32_l2norm"])
def test_expiry_on_shards(dtype, l2):
    from vqb200 import ops
    K, d, N, W, thr, reset = 12288, 64, 5000, 4, 2.0, 2.0
    Ks = K // W
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(N, d, generator=g, device=DEV).to(dtype)
    cs0 = 2.0 + torch.rand(K, generator=g, device=DEV)
    # dead codes on the 1024-code chunk boundaries of the kernel's scan and on the shard boundaries, plus random ones
    edges = [k for b in range(0, K + 1, 1024) for k in (b - 1, b) if 0 <= k < K]
    edges += [k for b in range(0, K + 1, Ks) for k in (b - 1, b) if 0 <= k < K]
    dead = torch.tensor(sorted(set(edges)), device=DEV)
    cs0[dead] = 0.5
    cs0[torch.randperm(K, generator=g, device=DEV)[:300]] = 1.0
    ea0 = torch.randn(K, d, generator=g, device=DEV)
    em0 = torch.randn(K, d, generator=g, device=DEV)
    is_dead = cs0 < thr
    m_total = int(is_dead.sum())
    rows = torch.randperm(N, generator=g, device=DEV)[:m_total]
    whole = [cs0.clone(), ea0.clone(), em0.clone()]
    ops.expire_scatter(x, rows, thr, reset, l2, *whole)
    shards = [cs0.clone(), ea0.clone(), em0.clone()]
    _expire_shards(x, rows, thr, reset, l2, *shards, W)
    for name, a, b in zip(("cluster_size", "embed_avg", "embeddings"), shards, whole):
        assert torch.equal(a, b), f"{name}: expiry on shards differs from expiry on the whole codebook"
    # reference codebooks.py:230-255: the j-th dead code (ascending) takes sampled row j
    picked = x[rows].float()
    if l2:
        picked = picked / picked.double().norm(dim=-1, keepdim=True).clamp_min(1e-12).float()
    cs_ref, ea_ref, em_ref = cs0.clone(), ea0.clone(), em0.clone()
    em_ref[is_dead] = picked
    ea_ref[is_dead] = picked * reset
    cs_ref[is_dead] = reset
    assert torch.equal(whole[0], cs_ref)
    assert torch.equal(whole[1][~is_dead], ea0[~is_dead]) and torch.equal(whole[2][~is_dead], em0[~is_dead])
    if l2:
        assert _rowrel(whole[2], em_ref) <= 1e-6 and _rowrel(whole[1], ea_ref) <= 1e-6
    else:
        assert torch.equal(whole[2], em_ref) and torch.equal(whole[1], ea_ref)


# ------------------------------------------------------------------------------------------------ part 2: module level
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_module_level_two_ranks_on_one_gpu():
    """tools/mgpu_check.py with VQB_MGPU_SINGLE_DEVICE=1: 2 ranks over Gloo, both on cuda:0 (the CUDA-graph section
    needs NCCL and is skipped)."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "mgpu_check.py")]
    env = dict(os.environ, VQB_MGPU_SINGLE_DEVICE="1")
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env,
                         start_new_session=True)
    try:
        out, err = p.communicate(timeout=600)
    finally:
        if p.poll() is None or p.returncode != 0:
            try:
                os.killpg(p.pid, signal.SIGKILL)
            except ProcessLookupError:
                pass
            p.wait()
    assert p.returncode == 0 and "MGPU OK" in out, out[-3000:] + err[-5000:]
    print(out[-3000:])
