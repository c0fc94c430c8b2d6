"""The EMA sums against fp64, under the bound each search route leaves in its workspace.

The EMA statistics (per-code sums of the assigned rows and counts) are accumulated in 64-bit fixed point whose scale
comes from a bound a + b >= max|x_j| (ema.cu).  The modules do not compute that bound: they pass the search workspace,
whose first 8 bytes hold it after `vqb_search` on the same x (include/vqb.h, above vqb_ema_reduce).  A bound that is too
small makes the integer sums wrap around without an error.

(a) the contract itself, after every search route: the single row tile kernel, the aug kernel (Euclidean and dot), the
    exact route (by width, by `force_exact`, without a cache), the in-kernel conversion with rows far above its sampled
    bound, and operands prepared by `rvq_level` / `rvq_level_ema`; each right after a search of a much larger and of a
    much smaller batch through the same shared workspace.
(b) the sums `ema_reduce`, `quantize_ema` and `rvq_level_ema` compute under that bound, against fp64 one-hot sums of the
    same inputs, per code and per column, with a bar of count x the quantum the kernel states (ema_scale_kernel,
    fused_scale_kernel) plus half an fp32 ulp of the result -- never a bar relative to the batch maximum.
(c) one training step of VectorQuantize and ResidualVQ, and a kmeans init, against an fp64 restatement of the refresh.
"""
import math
import zlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# ------------------------------------------------------------------------------------------------------ bound and bars
def _bound_pair(ws):
    a, b = ws[:8].view(torch.float32).tolist()
    return a, b


def _bound_exponent(ws):
    """e with b < 2^e for the bound the EMA kernels form from the workspace: fp32 a + b, 1 when not positive/finite."""
    a, b = _bound_pair(ws)
    s = float(np.float32(a) + np.float32(b))
    if not (s > 0.0) or not math.isfinite(s):
        s = 1.0
    return math.frexp(s)[1]


def _log2_rows(rows):
    lr = 0
    while (1 << lr) < rows + 1:
        lr += 1
    return lr


def quantum_ema_reduce(ws, rows):
    """2^-s, s = 61 - (e + lr) clamped to [-60, 100] (ema_scale_kernel)."""
    s = min(100, max(-60, 61 - (_bound_exponent(ws) + _log2_rows(rows))))
    return 2.0 ** -s


def quantum_fused(ws, rows, two_terms):
    """2^(e - P), e = exponent + 1 clamped to [-100, 100], P = 22 or min(62 - lr, 44) (fused_scale_kernel)."""
    e = min(100, max(-100, _bound_exponent(ws) + 1))
    P = min(62 - _log2_rows(rows), 44) if two_terms else 22
    return 2.0 ** (e - P)


def check_contract(ws, x, what):
    """a + b >= max|x_j| over the whole batch (all heads, masked rows included), in fp64."""
    a, b = _bound_pair(ws)
    mx = float(x.double().abs().max()) if x.numel() else 0.0
    assert a + b >= mx, f"{what}: bound a + b = {a} + {b} < max|x_j| = {mx}"


def ref_stats(x, idx, mask, K):
    """fp64 one-hot sums (H,K,d) and counts (H,K) over the rows with mask != 0."""
    H, N, d = x.shape
    xs = x.double()
    sums = torch.zeros(H, K, d, dtype=torch.float64, device=DEV)
    cnt = torch.zeros(H, K, dtype=torch.float64, device=DEV)
    keep = torch.ones(N, dtype=torch.bool, device=DEV) if mask is None else mask.bool()
    for h in range(H):
        sums[h].index_add_(0, idx[h][keep], xs[h][keep])
        cnt[h].index_add_(0, idx[h][keep], torch.ones(int(keep.sum()), dtype=torch.float64, device=DEV))
    return sums, cnt


def check_stats(stats, ref_sums, ref_cnt, q, what):
    d = ref_sums.shape[-1]
    got_cnt = stats[..., d].double()
    assert torch.equal(got_cnt, ref_cnt), f"{what}: counts differ at {int((got_cnt != ref_cnt).sum())} codes"
    got = stats[..., :d]
    mag = torch.maximum(got.abs(), ref_sums.abs().float())
    half_ulp = (torch.nextafter(mag, torch.full_like(mag, math.inf)) - mag).double() * 0.5
    bar = ref_cnt[..., None] * q + half_ulp
    err = (got.double() - ref_sums).abs()
    bad = ~(err <= bar)
    if bool(bad.any()):
        i = int(torch.argmax((err - bar).flatten()))
        raise AssertionError(f"{what}: {int(bad.sum())} sums outside count x {q:.3g} + half an ulp; worst got "
                             f"{float(got.flatten()[i])} want {float(ref_sums.flatten()[i])} "
                             f"(count {float(ref_cnt.flatten()[i // d])})")


# ------------------------------------------------------------------------------------------------------------- routes
EXACT_ROUTES = [f"exact_d{d}_{n}_h{H}" for d in (513, 520, 640, 1024) for n in ("f32", "bf16", "f16") for H in (1, 3)]
ROUTES = (["single_tile", "aug_euclid_f32", "aug_euclid_bf16", "aug_dot"] + EXACT_ROUTES
          + ["force_exact_d64", "no_cache_d64", "fused_prep_bf16", "fused_prep_f16"]
          + [f"prepared_{p}_d{d}" for p in ("level", "level_ema") for d in (64, 256, 512)])
MAGS = ["unit", "plus20", "plus100", "x1e3", "row1e6", "x1e-20", "zero"]
_DT = {"f32": F32, "bf16": BF16, "f16": F16}


def _spec(route):
    """(dtype, H, N, K, d, cosine)"""
    if route == "single_tile":
        return F32, 1, 100, 256, 64, False
    if route == "aug_euclid_f32":
        return F32, 1, 4000, 512, 128, False
    if route == "aug_euclid_bf16":
        return BF16, 1, 4000, 512, 256, False
    if route == "aug_dot":
        return F32, 1, 4000, 512, 128, True
    if route.startswith("exact_"):
        _, d, n, H = route.split("_")
        return _DT[n], int(H[1:]), 2000, 64, int(d[1:]), False
    if route == "force_exact_d64":
        return F32, 1, 2000, 256, 64, False
    if route == "no_cache_d64":
        return BF16, 1, 2000, 256, 64, False
    if route.startswith("fused_prep_"):
        return _DT[route.split("_")[-1]], 1, 40000, 8192, 256, False
    return F32, 1, 3001, 300, int(route.split("_d")[-1]), False


def _latents(shape, dtype, mag, g):
    x = torch.randn(*shape, generator=g, device=DEV)
    if mag == "plus20":
        x += 20.0
    elif mag == "plus100":
        x += 100.0
    elif mag == "x1e3":
        x *= 1e3
    elif mag == "row1e6":
        big = 6e4 if dtype == F16 else 1e6          # the largest fp16 is 65504
        x.view(-1, shape[-1])[shape[-2] // 3] = x.view(-1, shape[-1])[shape[-2] // 3].clamp(-4, 4) * (big / 4)
    elif mag == "x1e-20":
        x *= 1e-20
    elif mag == "zero":
        x.zero_()
    return x.to(dtype)


def _plant_outliers(x, big):
    """Rows far above the sampled bound of the in-kernel conversion, off the sample's stride (as test_gpu_fused_prep)."""
    H, N, d = x.shape
    stride = max((H * N) // 16384, 1)
    flat = x.view(-1, d)
    bad = torch.arange(1, H * N, 997, device=DEV)
    bad = bad[(bad % stride) != 0][:50]
    flat[bad] = (flat[bad].float() * big).to(x.dtype)
    return x


def run_route(route, mag, pre, seed):
    """The route's search on a batch of magnitude `mag`, right after a search of a `pre` x larger batch through the same
    shared workspace.  Returns (x (H,N,d), fp32 codebook (H,K,d), idx (H,N), ws)."""
    from vqb200 import ops
    dtype, H, N, K, d, cos = _spec(route)
    g = _gen(seed)
    c = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    if cos:
        c = torch.nn.functional.normalize(c, dim=-1)
    if route.startswith("prepared_"):
        # operands of the next level, written by rvq_level / rvq_level_ema into the shared search workspace
        c2 = torch.randn(1, K, d, generator=g, device=DEV) * 0.3
        cache2 = ops.prepare_codebook(c2, False)
        idx0 = torch.randint(0, K, (N,), generator=g, device=DEV)
        r = c[0][idx0].clone() if mag == "zero" else _latents((N, d), F32, mag, g)
        stale = torch.randn(1, N, d, generator=g, device=DEV) * pre
        ops.search(stale, c2, cache2, False)
        nxt = torch.empty_like(r)
        if "level_ema" in route:
            cache = ops.prepare_codebook(c, False)
            i0, _, ws0 = ops.search(r[None], c, cache, False)
            ops.rvq_level_ema(r, nxt, c[0], i0[0], True, True, torch.empty_like(r), cache2, bound_ws=ws0)
        else:
            ops.rvq_level(r, nxt, c[0], idx0, None, True, True, None, cache2)
        idx, _, ws = ops.search(nxt[None], c2, cache2, False, latents_prepared=True)
        return nxt[None], c2, idx, ws
    x = _latents((H, N, d), dtype, mag, g)
    kw = {}
    if route.startswith("fused_prep_"):
        x = _plant_outliers(x, 1e4 if dtype == F16 or mag != "unit" else 1e6)
        kw["fused_prep"] = True
    if route == "force_exact_d64":
        kw["force_exact"] = True
    cache = None if route == "no_cache_d64" else ops.prepare_codebook(c, cos)
    ops.search((torch.randn(H, N, d, generator=g, device=DEV) * pre).to(dtype), c, cache, cos, **kw)
    idx, _, ws = ops.search(x, c, cache, cos, **kw)
    return x, c, idx, ws


def _mags(route):
    dtype = _spec(route)[0]
    if route.startswith("fused_prep_"):
        return ["unit", "plus20"] if dtype == BF16 else ["unit"]      # fp16 holds no plus20 row x 1e4
    return MAGS


@pytest.mark.parametrize("route", ROUTES)
def test_search_leaves_bound_on_max_abs(route):
    """(a) After every route of vqb_search, a + b in the workspace bounds max|x_j| of this batch, and it is this batch's
    bound: the same bits whether a 300x larger or a 1e-3x smaller batch went through the shared workspace before.  The
    exact scan leaves max|x_j| itself.  (The tensor-core routes' bound is a bound of the row norms, and for 16-bit
    latents it includes an analytical bound of the fp16 rounding residual with an absolute floor set by the row-scale
    clamp, so it is not compared with max|x_j| from above.)"""
    for mag in _mags(route):
        seed = zlib.crc32(f"{route} {mag}".encode()) % 10000
        bounds = []
        for pre in (300.0, 1e-3):
            x, _, _, ws = run_route(route, mag, pre, seed=seed)
            check_contract(ws, x, f"{route} {mag} after x{pre:g}")
            bounds.append(ws[:8].clone())
        assert torch.equal(bounds[0], bounds[1]), \
            f"{route} {mag}: the bound depends on the batch searched before: {bounds[0].view(torch.float32).tolist()} " \
            f"after x300, {bounds[1].view(torch.float32).tolist()} after x1e-3"
        if route.startswith(("exact_", "force_exact", "no_cache")):
            a, b = _bound_pair(ws)
            assert (a, b) == (float(x.double().abs().max()), 0.0), f"{route} {mag}: exact scan left {(a, b)}"


def _idx_kinds(idx, K, g):
    H, N = idx.shape
    one = torch.full_like(idx, K // 2)
    seg = idx.clone()
    lo = N // 5
    seg[:, lo:lo + (3 * N) // 5] = K - 1
    return [("search", idx), ("one code", one), ("60% segment", seg)]


def _masks(N, g):
    some = (torch.rand(N, generator=g, device=DEV) >= 0.3).to(torch.uint8)
    return [("no mask", None), ("30% off", some), ("all off", torch.zeros(N, dtype=torch.uint8, device=DEV))]


def _cases_b():
    for route in ROUTES:
        for mag in _mags(route):
            yield pytest.param(route, mag, id=f"{route}-{mag}")


@pytest.mark.parametrize("route,mag", list(_cases_b()))
def test_ema_sums_under_search_bound_match_fp64(route, mag):
    """(b) ema_reduce, quantize_ema and rvq_level_ema with the route's workspace as the bound, against fp64 per code and
    per column; counts exact.  The bar follows from the bound as read back, so a bound too small to hold the sums shows
    here only where they wrap around ((a) checks the bound itself)."""
    from vqb200 import ops
    x, c, idx, ws = run_route(route, mag, 1e-3, seed=zlib.crc32(f"{route} {mag} b".encode()) % 10000)
    H, N, d = x.shape
    K = c.shape[1]
    g = _gen(7)
    q_red = quantum_ema_reduce(ws, N)
    fused = ops.quantize_ema_supported(d)
    rvq = H == 1 and x.dtype == F32 and ops.rvq_level_ema_supported(d)
    for iname, ix in _idx_kinds(idx, K, g):
        ix = ix.contiguous()
        for mname, m in _masks(N, g):
            what = f"{route} {mag} idx={iname} {mname}"
            ref_s, ref_c = ref_stats(x, ix, m, K)
            check_stats(ops.ema_reduce(x, ix, m, K, bound_ws=ws), ref_s, ref_c, q_red, f"{what} ema_reduce")
            if m is not None:
                continue
            if fused:
                q_f = quantum_fused(ws, N, x.dtype == F32)
                _, _, st = ops.quantize_ema(x, c, ix, True, False, bound_ws=ws)
                check_stats(st, ref_s, ref_c, q_f, f"{what} quantize_ema")
            if rvq:
                q_f = quantum_fused(ws, N, True)
                r = x[0]
                _, st = ops.rvq_level_ema(r, torch.empty_like(r), c[0], ix[0], True, True, torch.empty_like(r), None,
                                          bound_ws=ws)
                check_stats(st, ref_s, ref_c, q_f, f"{what} rvq_level_ema")


# ------------------------------------------------------------------------------------------------------------ modules
def _cpu_draw(num_rows, m, device):
    if num_rows >= m:
        return torch.randperm(num_rows)[:m].to(device)
    return torch.randint(0, num_rows, (m,)).to(device)


@pytest.fixture
def _patch_draw(monkeypatch):
    from vqb200 import codebook
    monkeypatch.setattr(codebook.Codebook, "_draw_rows", staticmethod(_cpu_draw))


def _init_codebook(cb, c):
    with torch.no_grad():
        cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0)
    cb.invalidate_cache()


def ref_refresh(cs, ea, sums, cnt, decay, eps):
    """codebooks.py:410-425 in fp64: lerp of cluster_size and embed_avg, Laplace smoothing, divide."""
    w = 1.0 - decay
    cs, ea = cs.double(), ea.double()
    cs_new = cs + w * (cnt - cs)
    ea_new = ea + w * (sums - ea)
    tot = cs_new.sum(-1, keepdim=True)
    K = cs.shape[-1]
    smoothed = (cs_new + eps) / (tot + K * eps) * tot
    return cs_new, ea_new, ea_new / smoothed[..., None], smoothed


def quantum_upper(rows, fused16=False):
    """An upper limit of the quantum of the EMA sums under the bound a search leaves for `rows` of the magnitudes used
    here (at most a row-norm bound, 2.5 sqrt(d) max|x_j|): ema_reduce's, or with `fused16` that of the fused 16-bit
    sums."""
    N, d = rows.shape[-2], rows.shape[-1]
    b = 2.5 * math.sqrt(d) * float(rows.double().abs().max())
    e = math.frexp(b if b > 0 else 1.0)[1]
    if fused16:
        return 2.0 ** (min(100, e + 1) - 22)
    return 2.0 ** -min(100, max(-60, 61 - (e + _log2_rows(N))))


def check_refresh(cb, pre, rows, idx, mask, what, fused16=False):
    """cb's buffers after one step against the fp64 refresh from the pre-step buffers `pre` and the step's indices.
    Bars per code and column: 1e-6 of the magnitudes that enter (never of the batch maximum), plus count x the
    quantum of the EMA sums."""
    cs0, ea0 = pre
    H, N, d = rows.shape
    K = cs0.shape[-1]
    sums, cnt = ref_stats(rows, idx, mask, K)
    abs_sums, _ = ref_stats(rows.abs(), idx, mask, K)
    cs, ea, emb, smoothed = ref_refresh(cs0, ea0, sums, cnt, cb.decay, cb.eps_for_smoothing)
    w = 1.0 - cb.decay
    scale = ea0.double().abs() + w * abs_sums + ea.abs() + 1e6 * w * cnt[..., None] * quantum_upper(rows, fused16)
    assert float(((cb.cluster_size.double() - cs).abs() / cs.abs().clamp_min(1e-30)).max()) <= 1e-6, \
        f"{what}: cluster_size"
    err = (cb.embed_avg.double() - ea).abs()
    assert bool((err <= 1e-6 * scale + 1e-30).all()), f"{what}: embed_avg, worst {float((err - 1e-6 * scale).max())}"
    err = (cb.embeddings.detach().double() - emb).abs()
    bar = 2e-6 * scale / smoothed[..., None] + 1e-30
    assert bool((err <= bar).all()), f"{what}: embeddings, worst {float((err - bar).max())}"


@pytest.mark.parametrize("dim,dtype,mask", [(640, F32, False), (640, F32, True), (1024, F32, False),
                                            (1024, F32, True), (256, BF16, False)])
def test_vector_quantize_step_matches_fp64_refresh(dim, dtype, mask):
    """(c) One training step: d = 640 and 1024 search on the exact route, d = 256 bf16 runs the fused quantize_ema."""
    from vqb200 import CodebookParams, VectorQuantize
    K, B, n = 256, 2, 4000
    torch.manual_seed(0)
    vq = VectorQuantize(dim=dim, codebook_params=CodebookParams(dim=dim, codebook_size=K,
                                                                threshold_ema_dead_code=0)).to(DEV)
    gen = torch.Generator().manual_seed(dim)
    cb = vq._codebook
    _init_codebook(cb, torch.randn(1, K, dim, generator=gen))
    x = (torch.randn(B, n, dim, generator=gen) + 20.0).to(DEV).to(dtype)
    m = (torch.rand(B, n, generator=gen) >= 0.3).to(DEV) if mask else None
    pre = (cb.cluster_size.clone(), cb.embed_avg.clone())
    vq.train()
    with torch.no_grad():
        _, ind, _ = vq(x, mask=m)
    rows = x.reshape(1, B * n, dim)
    check_refresh(cb, pre, rows, ind.reshape(1, -1), None if m is None else m.reshape(-1).to(torch.uint8),
                  f"VectorQuantize d={dim} {dtype} mask={mask}", fused16=dtype != F32)


@pytest.mark.parametrize("fused", [True, False])
def test_residual_vq_step_matches_fp64_refresh(fused):
    """(c) ResidualVQ(dim=640, 3 levels): every level's refresh from the residual it saw, restated in fp32 with the IEEE
    operations of the level kernel (q = r + (c - r), r' = r - q)."""
    from vqb200 import CodebookParams, ResidualVQ
    d, Q, K, B, n = 640, 3, 256, 2, 4000
    torch.manual_seed(0)
    rvq = ResidualVQ(dim=d, num_quantizers=Q,
                     codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0)).to(DEV)
    gen = torch.Generator().manual_seed(5)
    for li, layer in enumerate(rvq.layers):
        _init_codebook(layer._codebook, torch.randn(1, K, d, generator=gen) * (0.6 / 1.3 ** li))
    rvq.use_fused_levels = fused
    x = (torch.randn(B, n, d, generator=gen) + 20.0).to(DEV)
    pre = [(l._codebook.embeddings.detach().clone(), l._codebook.cluster_size.clone(), l._codebook.embed_avg.clone())
           for l in rvq.layers]
    rvq.train()
    with torch.no_grad():
        _, ind, _ = rvq(x)
    r = x.reshape(-1, d)
    for li, layer in enumerate(rvq.layers):
        emb0, cs0, ea0 = pre[li]
        idx = ind[..., li].reshape(-1)
        check_refresh(layer._codebook, (cs0, ea0), r[None], idx[None], None, f"ResidualVQ fused={fused} level {li}")
        cq = emb0[0][idx]
        r = r - (r + (cq - r))


def test_kmeans_init_matches_fp64_means(_patch_draw):
    """(c) Kmeans init at d = 640 (exact route), one iteration: the initial codebook is the fp64 mean of the rows each
    drawn centroid won (the centroid itself where it won none)."""
    from vqb200 import CodebookParams, KmeansParameters, VectorQuantize, ops
    d, K, B, n = 640, 256, 2, 4000
    torch.manual_seed(0)
    vq = VectorQuantize(dim=d, codebook_params=CodebookParams(
        dim=d, codebook_size=K, threshold_ema_dead_code=0, initialization_by_kmeans=True,
        kmeans_params=KmeansParameters(iter=1))).to(DEV)
    gen = torch.Generator().manual_seed(11)
    x = torch.randn(B, n, d, generator=gen) + 20.0
    x[1, 17] *= 1e4                                   # one outlier row
    x = x.to(DEV)
    vq.eval()
    torch.manual_seed(3)
    with torch.no_grad():
        vq(x)
    data = x.reshape(1, -1, d)
    torch.manual_seed(3)
    cents = data[0][_cpu_draw(B * n, K, DEV)][None].contiguous()
    idx, _, _ = ops.search(data, cents, None, False, force_exact=True)
    sums, cnt = ref_stats(data, idx, None, K)
    abs_sums, _ = ref_stats(data.abs(), idx, None, K)
    want = torch.where(cnt[..., None] > 0, sums / cnt.clamp_min(1)[..., None], cents.double())
    got = vq._codebook.embeddings.detach().double()
    assert torch.equal(vq._codebook.cluster_size.double(), cnt), "kmeans init: counts"
    bar = (1e-6 * abs_sums / cnt.clamp_min(1)[..., None] + quantum_upper(data)) * (cnt[..., None] > 0) + 1e-30
    err = (got - want).abs()
    assert bool((err <= bar).all()), f"kmeans init: means, worst {float((err - bar).max())}"
