"""The tensor-core search against an fp64 statement of its contract, on every resolve route, with the inputs of its
exactness proof (codebook cache, per-search bounds, candidate keys) checked on their own.

Contract (include/vqb.h, csrc/search_resolve.cu).  For a row x and a code c of a codebook (H, K, d):
  dot = sum_j x_j c_j, |x|^2 = sum_j x_j^2, |c|^2 = sum_j c_j^2, each accumulated in fp64 in the order j = 0 .. d-1;
  euclid score = sqrtf(max(float((|x|^2 + |c|^2) - 2 dot), 0)),   dot score = float(-dot);
  idx = the lowest index among the codes of smallest fp32 score (+ idx_offset), score = that fp32 score.
`restate` below evaluates exactly this in torch, one `acc = acc + a * c` per j with fp64 tensors.  A product of two fp32,
bf16 or fp16 values is exact in fp64, so that step rounds once, like the kernels' `fma(a, c, acc)`, and the chains of
`exact_score`, `exact_score_norm`, `exact_scan_kernel` and the SCORE path of `resolve_classify_kernel` all walk j in
order: the restatement is bit-identical to every exact route.  (No fp64 bmm / cdist: another summation order can move
the fp32 rounding at the very ties built below.)  sqrt(float(d2)) in fp64 rounded to fp32 is the correctly rounded
sqrtf: fp64 has more than 2 * 24 + 2 bits.  Every search case asserts idx and score bit for bit, and runs again without
`want_score` (the `resolve_classify_kernel<float, false>` instance and the finalisers that write no score): same idx.

Why the search may skip codes (the header of search_resolve.cu).  e_k = |c_k|^2/2 - x.c_k (euclid) or -x.c_k (dot)
ranks the codes like the score.  With x~ = fp16(x s_row) / s_row and c~ = fp16(c s_c) / s_c (the operands of the
tensor-core pass) Cauchy-Schwarz gives
    |x.c - x~.c~| <= |x~| |c - c~| + |x - x~| |c| <= X |c - c~| + DX |c|,      X = scal[0] >= max |x~|, DX = scal[1] >= max |x - x~|,
so E_k = X dcn_k + DX cn_k + (fp32 accumulation slack) bounds the error of the key, given cn_k >= |c_k| and
dcn_k >= |c_k - c~_k| from the codebook cache (section (b)) and the batch bounds X, DX (section (c)).  The key L_k written
by the kernel is lowered by E_k (bias_k = cn2h_k - E_k, in the epilogue of the single-tile kernel, aug mode 0, or as the
extra MMA k-step of aug mode 1), so L_k <= e_k <= L_k + 2 E_k; with no bias (aug mode 2: dot metric, K % 256 == 0) or
when the bias operand would leave fp16 (scal[8] = 1, "unlowered") the key is centred: |e_k - L_k| <= E_k <= Emax.
Six mantissa bits of every key carry the code's column id (2^-17 relative), and the key itself is one fp32 rounding, so
the bounds hold to s = (|L| + E) kPackSlack (6.2e-5).  The epilogue stores the keys in TRUE units in both kernels: the
single-tile kernel forms bias + acc / (s_row s_c) with one FFMA, the pair kernel multiplies its scaled minima by
|xinv| / s_c when it writes them.  Section (d) checks these windows on every valid candidate of every row with xinv > 0.
Resolve then keeps every code with L <= thr = L_min + 2 E (+ packing slack + kTieSlack |x|^2, the codes that the fp32
rounding of the distance can make EQUAL to the winner), and accepts, re-ranks from (row, code) pairs, rescans the
64-column group of two entries from one group (hazard ii) or rescans the row (hazard i, a third entry of a class inside
the window; also rows that do not fit `pair_cap`).  Flagged rows are scored as pairs when n K <= 2^17, else by the
tiled K-split scan.  Section (e) builds inputs for each route and proves from the workspace counters that it ran:
scal[2] rows rescanned, scal[3] rows queued for re-rank, scal[8] unlowered, scal[9] pairs, cnt[H..2H) rows left to the
tiled scan, cnt[2H..3H) the pair plan; the aug mode shows in the caug block of a workspace filled with 0xFF before the
search (only aug mode 1 writes it).

(b) Codebook cache (`vqb_prepare_codebook`, prepare.cu), per codebook: s_c = hdr[0] a power of two, hdr[0] hdr[1] = 1,
    hdr[2] = max |c| exactly, max |c| s_c < 2^14 (>= 2^13 inside the +-100 binade clamp of pow2_scale), hdr[3] =
    max cn2h (0 for dot), hdr[4] hdr[5] = 1 and s_c hdr[4] hdr[3] in [2^12, 2^13) unless hdr[3] = 0 or q is clamped;
    per code: the fp16 block is -fp16(c s_c) bit for bit and zero beyond d, cn >= |c|, dcn >= |c - c~| in fp64, cn2h
    within one fp32 ulp of |c|^2/2 (0 for dot); padded codes: cn2h = 3e38, cn = dcn = 0, zero rows.
(c) Per search (`make_bias_kernel`, `make_bias_operand_kernel`): err_k >= X |c_k - c~_k| + DX |c_k| in fp64 (with the
    in-kernel conversion, whose DX is derived, against the measured max |x~| and max |x - x~| of the rows it keeps);
    X, DX bound max |x~|, max |x - x~|; bias_k = cn2h_k - err_k in fp32; scal[6] = max_k err_k; the three fp16 pieces of
    caug sum, in fp64, to b = float((cn2h - err) s_c 2^q) (cn2h s_c 2^q when unlowered) within 2^-33 |b| + 2^-25 (fp16
    keeps 11 bits per piece; 2^-25 is half its smallest subnormal), i.e. 2^-37 of the largest bias (>= 2^12); padded
    codes +inf, bias 3e38, err 0; on aug mode 1 scal[8] = 1 exactly when some head has (hdr[3] + Emax) s_c 2^q >= 60000,
    on every other search 0.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
EUCLID, DOT = 0, 1
PACK_SLACK = float(np.float32(6.2e-5))
PAD_BIAS = float(np.float32(3.0e38))
FLAG_PAIR_BUDGET = 1 << 17


def _al(n):
    return (n + 255) // 256 * 256


def _kp(K):
    return (K + 255) // 256 * 256


def _dp(d):
    return (d + 63) // 64 * 64


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# ---- layouts (common.cuh: cache_layout, search_layout) ------------------------------------------------------------
def cache_dec(cache, H, K, d):
    Kp, dp = _kp(K), _dp(d)
    o = 0
    out = {}
    out["hdr"] = cache[o:o + H * 32].view(F32).reshape(H, 8)
    o += _al(H * 32)
    out["cb"] = cache[o:o + H * Kp * dp * 2].view(F16).reshape(H, Kp, dp)
    o += _al(H * Kp * dp * 2)
    for name in ("cn2h", "cn", "dcn"):
        out[name] = cache[o:o + H * Kp * 4].view(F32).reshape(H, Kp)
        o += _al(H * Kp * 4)
    return out


def ws_dec(ws, H, N, K, d):
    """a copy of everything the checks read from a search workspace"""
    Kp, dp, R = _kp(K), _dp(d), H * N
    w = {"scal": ws[:256].view(torch.int32).clone(), "cnt": ws[256:256 + H * 12].view(torch.int32).clone()}
    o = 256 + _al(H * 12)
    w["xb"] = ws[o:o + R * dp * 2].view(F16).reshape(H, N, dp).clone()
    o += _al(R * dp * 2)
    w["xinv"] = ws[o:o + R * 4].view(F32).reshape(H, N).clone()
    o += _al(R * 4)
    w["xn2"] = ws[o:o + R * 4].view(F32).reshape(H, N).clone()
    o += _al(R * 4)
    o += _al(R * 16)                                  # xaug
    o += _al(R * 8)                                   # keys
    w["cand"] = ws[o:o + R * 24 * 8].view(torch.int32).reshape(H, N, 24, 2).clone()
    o += _al(R * 24 * 8)
    o += 2 * _al(R * 4)                               # flag list, re-rank list
    w["bias"] = ws[o:o + H * Kp * 4].view(F32).reshape(H, Kp).clone()
    o += _al(H * Kp * 4)
    w["err"] = ws[o:o + H * Kp * 4].view(F32).reshape(H, Kp).clone()
    o += _al(H * Kp * 4)
    w["caug"] = ws[o:o + H * Kp * 16].view(F16).reshape(H, Kp, 8).clone()
    w["pair_cap"] = R * 4 + 4096
    return w


def sc(w, i):
    """scal[i] as an unsigned int"""
    return int(w["scal"][i]) & 0xFFFFFFFF


def scf(w, i):
    return float(w["scal"][i:i + 1].view(F32))


def aug_mode(N, K, metric):
    if (N + 127) // 128 < 2:
        return 0
    return 2 if (metric == DOT and K % 256 == 0) else 1


# ---- (a) the fp64 restatement ---------------------------------------------------------------------------------------
def restate(x, C, metric):
    """(idx (H,N) int64, score (H,N) fp32) of the contract, every sum in fp64 in the order j = 0 .. d-1"""
    H, N, d = x.shape
    K = C.shape[1]
    xd = x.float().double()
    cd = C.double()
    cn2 = torch.zeros(H, K, dtype=torch.float64, device=DEV)
    for j in range(d):
        cn2 = cn2 + cd[:, :, j] * cd[:, :, j]
    idx = torch.empty(H, N, dtype=torch.int64, device=DEV)
    score = torch.empty(H, N, dtype=F32, device=DEV)
    rows = max(1, (1 << 26) // K)
    ar = torch.arange(K, device=DEV)
    for h in range(H):
        cT = cd[h].t().contiguous()
        for r0 in range(0, N, rows):
            xs = xd[h, r0:r0 + rows]
            acc = torch.zeros(xs.shape[0], K, dtype=torch.float64, device=DEV)
            n2 = torch.zeros(xs.shape[0], dtype=torch.float64, device=DEV)
            for j in range(d):
                xj = xs[:, j]
                acc.add_(xj[:, None] * cT[j][None, :])
                n2 = n2 + xj * xj
            if metric == EUCLID:
                d2 = ((n2[:, None] + cn2[h][None, :]) - 2.0 * acc).float()
                s = torch.sqrt(d2.clamp_min(0.0).double()).float()
            else:
                s = (-acc).float()
            del acc
            m = s.min(dim=1).values
            idx[h, r0:r0 + rows] = torch.where(s == m[:, None], ar, K).min(dim=1).values
            score[h, r0:r0 + rows] = m
    return idx, score


def run_search(x, C, metric, cache, *, offset=0, poison=True, **kw):
    """search with and without the score; both against the restatement.  Returns the decoded workspace of the first."""
    from vqb200 import _lib as L
    from vqb200 import ops
    H, N, d = x.shape
    K = C.shape[1]
    if poison:
        nb = L.lib().vqb_search_workspace_bytes(H, N, K, d)
        ops.workspace("search", nb, x.device)[:nb].fill_(255)
    idx, score, ws = ops.search(x, C, cache, metric == DOT, idx_offset=offset, want_score=True, **kw)
    w = ws_dec(ws, H, N, K, d)
    w["raw"] = ws[:256 + _al(H * 12) + _al(H * N * _dp(d) * 2) + 2 * _al(H * N * 4) + _al(H * N * 16)].clone()
    w["poisoned"] = poison
    idx2, _, _ = ops.search(x, C, cache, metric == DOT, idx_offset=offset, want_score=False, **kw)
    want_idx, want_score = restate(x, C, metric)
    bad = (idx != want_idx + offset) | (score.view(torch.int32) != want_score.view(torch.int32))
    if bool(bad.any()):
        r = bad.nonzero()[:4].tolist()
        got = [(int(idx[h, n]) - offset, float(score[h, n]), int(want_idx[h, n]), float(want_score[h, n])) for h, n in r]
        pytest.fail(f"{int(bad.sum())} rows differ from the fp64 restatement; (row, (idx, score, want idx, want score)): "
                    f"{list(zip(r, got))}")
    assert torch.equal(idx2, idx), f"{int((idx2 != idx).sum())} rows differ between want_score and no score"
    w["want_idx"] = want_idx
    return w


# ---- (b) codebook cache -----------------------------------------------------------------------------------------
def _pow2(t):
    m, _ = torch.frexp(t)
    return bool((m == 0.5).all())


def _ulp32(t):
    t = t.float().abs()
    return (torch.nextafter(t, torch.full_like(t, math.inf)) - t).double()


def decoded_codes(D, K, d):
    """c~ = fp16 block / -s_c in fp64, (H, K, d)"""
    return D["cb"][:, :K, :d].double() * (-D["hdr"][:, 1].double())[:, None, None]


def check_cache(C, metric, cache, what):
    H, K, d = C.shape
    Kp = _kp(K)
    D = cache_dec(cache, H, K, d)
    hdr = D["hdr"]
    h64 = hdr.double()
    s = h64[:, 0]
    assert _pow2(s), f"{what}: s_c not a power of two"
    assert bool((h64[:, 0] * h64[:, 1] == 1).all()), f"{what}: hdr[0] hdr[1] != 1"
    amax = C.abs().amax(dim=(1, 2))
    assert torch.equal(hdr[:, 2], amax), f"{what}: hdr[2] {hdr[:, 2].tolist()} != max|c| {amax.tolist()}"
    assert bool((amax.double() * s < 2.0 ** 14).all()), f"{what}: max|c| s_c >= 2^14"
    inside = (amax > 0) & (s < 2.0 ** 100) & (s > 2.0 ** -100)
    assert bool((amax.double() * s >= 2.0 ** 13)[inside].all()), f"{what}: max|c| s_c < 2^13 inside the clamp"
    cn2h = D["cn2h"]
    want3 = cn2h[:, :K].amax(dim=1) if metric == EUCLID else torch.zeros(H, device=DEV)
    assert torch.equal(hdr[:, 3], want3), f"{what}: hdr[3] {hdr[:, 3].tolist()} != max cn2h {want3.tolist()}"
    assert _pow2(h64[:, 4]) and bool((h64[:, 4] * h64[:, 5] == 1).all()), f"{what}: hdr[4], hdr[5]"
    t = s * h64[:, 4] * h64[:, 3]
    free = (h64[:, 3] > 0) & (h64[:, 4] < 2.0 ** 100) & (h64[:, 4] > 2.0 ** -100)
    assert bool(((t >= 2.0 ** 12) & (t < 2.0 ** 13))[free].all()), f"{what}: s_c 2^q hdr[3] = {t.tolist()}"
    want_cb = -(C * hdr[:, 0][:, None, None]).half()
    assert torch.equal(D["cb"][:, :K, :d].view(torch.int16), want_cb.view(torch.int16)), f"{what}: fp16 block"
    assert bool((D["cb"][:, :, d:] == 0).all()), f"{what}: fp16 block not zero beyond d"
    assert bool((D["cb"][:, K:] == 0).all()), f"{what}: padded codes not zero"
    cd = C.double()
    norm = cd.norm(dim=2)
    resid = (cd - decoded_codes(D, K, d)).norm(dim=2)
    assert bool((D["cn"][:, :K].double() >= norm).all()), f"{what}: cn < |c|"
    assert bool((D["dcn"][:, :K].double() >= resid).all()), f"{what}: dcn < |c - c~|"
    if metric == EUCLID:
        half = (cd * cd).sum(dim=2) / 2
        dev = (cn2h[:, :K].double() - half).abs()
        assert bool((dev <= _ulp32(half)).all()), f"{what}: cn2h off |c|^2/2 by {float((dev / _ulp32(half)).max())} ulp"
    else:
        assert bool((cn2h[:, :K] == 0).all()), f"{what}: cn2h != 0 for the dot metric"
    if Kp > K:
        assert bool((cn2h[:, K:] == PAD_BIAS).all()), f"{what}: padded cn2h"
        assert bool((D["cn"][:, K:] == 0).all()) and bool((D["dcn"][:, K:] == 0).all()), f"{what}: padded cn / dcn"
    return D


def _cache_codebook(kind, seed):
    g = _gen(seed)
    if kind == "ragged_K":
        return torch.randn(1, 1000, 64, generator=g, device=DEV)
    if kind.startswith("d"):
        d = int(kind[1:])
        return torch.randn(2, 300, d, generator=g, device=DEV) * 0.3
    if kind == "head_scales":
        C = torch.randn(3, 700, 72, generator=g, device=DEV)
        return C * torch.tensor([1e-6, 1.0, 1e4], device=DEV)[:, None, None]
    if kind == "zero_and_mixed":
        C = torch.zeros(2, 300, 100, device=DEV)
        C[1] = torch.where(torch.rand(300, 100, generator=g, device=DEV) < 0.5, 1e-30, 1e3)
        C[1] *= torch.randn(300, 100, generator=g, device=DEV).sign()
        return C
    if kind == "subnormal":
        C = torch.randn(2, 256, 64, generator=g, device=DEV)
        C[0] *= 1e-39                                                       # every entry an fp32 subnormal
        C[1] = torch.where(torch.rand(256, 64, generator=g, device=DEV) < 0.25, C[1] * 1e-40, C[1])
        return C
    raise ValueError(kind)


CACHE_KINDS = ["ragged_K", "d30", "d72", "d100", "head_scales", "zero_and_mixed", "subnormal"]


@pytest.mark.parametrize("metric", [EUCLID, DOT], ids=["euclid", "dot"])
@pytest.mark.parametrize("kind", CACHE_KINDS)
def test_codebook_cache(kind, metric):
    from vqb200 import ops
    C = _cache_codebook(kind, 11)
    check_cache(C, metric, ops.prepare_codebook(C, metric == DOT), f"cache {kind}")


# ---- (c) per-search bounds and bias operand ------------------------------------------------------------------------
def check_bounds(w, D, C, x, aug, conv=False):
    """section (c); returns whether the search ran unlowered"""
    from test_gpu_operand_format import decode
    H, K, d = C.shape
    N = x.shape[1]
    err, bias = w["err"], w["bias"]
    cd = C.double()
    resid = (cd - decoded_codes(D, K, d)).norm(dim=2)
    norm = cd.norm(dim=2)
    X, DX = scf(w, 0), scf(w, 1)
    xb, xinv, _, _, _ = decode(w["raw"], H, N, d)
    keep = xinv > 0
    xt = xb[:, :d] * xinv.abs()[:, None]
    dx = (x.reshape(H * N, d).float().double() - xt).norm(dim=1)
    if not conv:
        assert float(xt.norm(dim=1).max()) <= X, f"max |x~| > scal[0] = {X}"
        assert float(dx.max()) <= DX, f"max |x - x~| > scal[1] = {DX}"
    else:      # the bound the in-kernel conversion derives must cover the rows it keeps
        X = float(xt.norm(dim=1)[keep].max())
        DX = float(dx[keep].max())
    need = X * resid + DX * norm
    short = err[:, :K].double() < need
    assert not bool(short.any()), f"err_k below X |c - c~| + DX |c| for {int(short.sum())} codes"
    assert torch.equal(bias[:, :K], D["cn2h"][:, :K] - err[:, :K]), "bias != cn2h - err"
    assert sc(w, 6) == int(err[:, :K].max().view(torch.int32)) & 0xFFFFFFFF, "scal[6] != max_k err_k"
    if _kp(K) > K:
        assert bool((bias[:, K:] == PAD_BIAS).all()) and bool((err[:, K:] == 0).all()), "padded bias / err"
    hdr = D["hdr"]
    emax = err[:, :K].max()
    scq = hdr[:, 0] * hdr[:, 4]
    unl = bool(((hdr[:, 3] + emax) * scq >= 60000.0).any()) if aug == 1 else False
    assert sc(w, 8) == int(unl), f"scal[8] = {sc(w, 8)}, expected {int(unl)} (aug mode {aug})"
    caug = w["caug"]
    if aug != 1:
        if w["poisoned"]:
            assert bool((caug.view(torch.int16) == -1).all()), f"aug mode {aug} wrote the bias operand"
        return unl
    b = ((D["cn2h"][:, :K] if unl else D["cn2h"][:, :K] - err[:, :K]) * scq[:, None]).double()
    got = caug[:, :K, :3].double().sum(dim=2)
    off = (got - b).abs()
    lim = 2.0 ** -33 * b.abs() + 2.0 ** -25
    assert not bool((off > lim).any()), f"caug pieces off by up to {float((off / lim).max())} of the bound"
    assert bool((caug[:, :K, 3:] == 0).all()), "caug beyond the three pieces"
    if _kp(K) > K:
        assert bool((caug[:, K:, 0] == math.inf).all()) and bool((caug[:, K:, 1:] == 0).all()), "padded caug"
    return unl


# ---- (d) candidate keys against the exact e_k ----------------------------------------------------------------------
def check_keys(w, C, x, metric, aug, unl):
    H, K, d = C.shape
    N = x.shape[1]
    key = w["cand"][..., 0].contiguous().view(F32).double()
    code = w["cand"][..., 1].long()
    valid = (code >= 0) & (code < K) & (w["xinv"] > 0)[:, :, None]
    assert bool(valid.any()), "no candidate to check"
    centred = aug == 2 or unl
    cd = C.double()
    half = (cd * cd).sum(dim=2) / 2 if metric == EUCLID else torch.zeros(H, K, dtype=torch.float64, device=DEV)
    err = w["err"][:, :K].double()
    emax = float(w["err"][:, :K].max())
    rows = max(1, (1 << 24) // (24 * d))
    bad = 0
    for h in range(H):
        for r0 in range(0, N, rows):
            v = valid[h, r0:r0 + rows]
            cc = code[h, r0:r0 + rows].clamp(0, K - 1)
            xs = x[h, r0:r0 + rows].float().double()
            e = half[h][cc] - torch.einsum("nd,ncd->nc", xs, cd[h][cc])
            L = key[h, r0:r0 + rows]
            E = torch.full_like(L, emax) if centred else err[h][cc]
            s = (L.abs() + E) * PACK_SLACK
            if centred:
                ok = (e - L).abs() <= E + s
            else:
                ok = (L - s <= e) & (e <= L + 2 * E + s)
            bad += int((v & ~ok).sum())
    assert bad == 0, f"{bad} candidate keys outside their window ({'centred' if centred else 'lowered'}, aug {aug})"


def full_check(x, C, metric, *, offset=0, cache=None, conv=False, poison=True, **kw):
    """search + restatement, cache, bounds and keys; returns (workspace, aug mode)"""
    from vqb200 import ops
    H, N, d = x.shape
    K = C.shape[1]
    if cache is None:
        cache = ops.prepare_codebook(C, metric == DOT)
    w = run_search(x, C, metric, cache, offset=offset, poison=poison, **kw)
    assert sc(w, 4) == 1, "the tensor-core pass did not run"
    D = check_cache(C, metric, cache, "cache")
    aug = aug_mode(N, K, metric)
    unl = check_bounds(w, D, C, x, aug, conv=conv)
    check_keys(w, C, x, metric, aug, unl)
    return w, aug


# ---- (e) inputs per route --------------------------------------------------------------------------------------------
def near_dup_case(H, N, K, d, dtype, codes, hot, seed, sigma=1.0):
    """randn codebook in which `codes` are c* + delta u (delta far below the fp16 rounding of c*); the first `hot` rows of
    each head lie near c*, the others are randn rows"""
    g = _gen(seed)
    C = torch.randn(H, K, d, generator=g, device=DEV) * sigma
    base = C[:, codes[0]].clone()
    for k in codes:
        C[:, k] = base + sigma * 2.0 ** -16 * torch.randn(H, d, generator=g, device=DEV)
    x = torch.randn(H, N, d, generator=g, device=DEV) * sigma
    x[:, :hot] = base[:, None, :] + 0.1 * sigma * torch.randn(H, hot, d, generator=g, device=DEV)
    return x.to(dtype), C


def counts(w, H):
    c = w["cnt"].long() & 0xFFFFFFFF
    return c[:H], c[H:2 * H], c[2 * H:3 * H]


RANDN_CASES = [
    # (name, H, N, K, d, dtype, metric, offset): aug mode 0 (one row tile), 1 (bias k-step), 2 (dot, K % 256 == 0)
    ("tile_euclid", 3, 100, 1000, 72, F32, EUCLID, 0),
    ("tile_dot", 1, 128, 512, 64, BF16, DOT, 7),
    ("tile_euclid_d30", 2, 77, 300, 30, F16, EUCLID, 0),
    ("aug1_euclid", 2, 300, 1000, 64, F16, EUCLID, 1000),
    ("aug1_euclid_d512", 1, 300, 512, 512, F32, EUCLID, 0),
    ("aug1_dot", 2, 300, 1000, 72, BF16, DOT, 0),
    ("aug2_dot", 2, 300, 1024, 256, F32, DOT, 5),
]


@pytest.mark.parametrize("name,H,N,K,d,dtype,metric,offset", RANDN_CASES, ids=[c[0] for c in RANDN_CASES])
def test_route_randn(name, H, N, K, d, dtype, metric, offset):
    """control: randn rows, most of them accepted on their single candidate; the aug mode shows in caug"""
    g = _gen(21)
    C = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    x = torch.randn(H, N, d, generator=g, device=DEV).to(dtype)
    w, aug = full_check(x, C, metric, offset=offset)
    assert aug == {"tile": 0, "aug1": 1, "aug2": 2}[name.split("_")[0]]
    flagged, _, _ = counts(w, H)
    accepted = H * N - sc(w, 3) - int(flagged.sum())
    assert accepted >= H * N // 2, f"only {accepted} of {H * N} rows accepted on one candidate"


@pytest.mark.parametrize("N,dtype,metric", [(100, F32, EUCLID), (300, BF16, EUCLID), (300, F16, DOT)])
def test_route_rerank(N, dtype, metric):
    """near-duplicates one per class (quarter x parity): every hot row queued, re-ranked from a few pairs each"""
    H, K, d = 1, 1024, 64
    x, C = near_dup_case(H, N, K, d, dtype, [0, 1, 64, 65, 130, 195], N, 31)
    w, _ = full_check(x, C, metric, offset=3)
    assert sc(w, 3) >= 0.9 * N, f"{sc(w, 3)} rows re-ranked"
    assert sc(w, 2) == 0, f"{sc(w, 2)} rows rescanned"
    assert sc(w, 9) <= 24 * sc(w, 3), f"{sc(w, 9)} pairs: a group rescan ran"


@pytest.mark.parametrize("N,hot,metric,codes", [
    (60, 60, EUCLID, [4, 6]), (300, 50, EUCLID, [4, 6]), (300, 50, DOT, [4, 6]),
    (60, 60, EUCLID, [4, 6, 8]), (300, 50, EUCLID, [4, 6, 8]),    # a third code hidden in the group: only the rescan sees it
])
def test_route_group_rescan(N, hot, metric, codes):
    """near-duplicates in one 64-column group (codes 4, 6 and maybe 8): hazard (ii), the 64 columns are scored as pairs"""
    H, K, d = 1, 1000, 64
    x, C = near_dup_case(H, N, K, d, F32, codes, hot, 41)
    w, _ = full_check(x, C, metric)
    assert sc(w, 3) >= 0.9 * hot, f"{sc(w, 3)} rows re-ranked"
    assert sc(w, 9) >= 64 * 0.9 * hot, f"{sc(w, 9)} pairs: no group rescan"
    assert sc(w, 9) <= w["pair_cap"] and sc(w, 2) == 0, "rows left the pair route"
    if len(codes) == 3:
        won = torch.bincount(w["want_idx"][0, :hot], minlength=K)[codes]
        assert int(won[2]) > 0, f"the hidden code never wins: {won.tolist()}"


@pytest.mark.parametrize("N,hot,K,d,dtype,tiled", [
    (4000, 6, 1600, 64, F32, False),       # few flagged rows, n K <= 2^17 and inside pair_cap: pairs over every code
    (100, 100, 1600, 256, BF16, True),     # single-tile kernel, n K > 2^17: tiled K-split rescan
    (300, 300, 1600, 64, F16, True),
    (200, 40, 70000, 64, F32, True),       # K > 65536: the widest code split of the rescan
])
def test_route_full_rescan(N, hot, K, d, dtype, tiled):
    """four near-duplicates in one class from four 512-code blocks: hazard (i), the row is rescanned (the class keeps
    three entries: the fourth code is seen by the rescan only)"""
    H = 1
    x, C = near_dup_case(H, N, K, d, dtype, [0, 512, 1024, 1536], hot, 51)
    w, _ = full_check(x, C, EUCLID, offset=11)
    flagged, scan, plan = counts(w, H)
    assert int(flagged[0]) >= 0.9 * hot and sc(w, 2) >= int(flagged[0]), (flagged.tolist(), sc(w, 2))
    assert int(flagged[0]) * K > FLAG_PAIR_BUDGET if tiled else int(flagged[0]) * K <= FLAG_PAIR_BUDGET
    if tiled:
        assert int(scan[0]) == int(flagged[0]) and int(plan[0]) == 0xFFFFFFFF, (scan.tolist(), plan.tolist())
    else:
        assert int(scan[0]) == 0 and int(plan[0]) != 0xFFFFFFFF, (scan.tolist(), plan.tolist())


def test_route_pair_cap_overflow():
    """a hazard-(ii) pair for every row: 66 pairs per row overflow 4 N + 4096, the rows left over go to the rescan"""
    H, N, K, d = 1, 2000, 1024, 64
    x, C = near_dup_case(H, N, K, d, F32, [4, 6], N, 61)
    w, _ = full_check(x, C, EUCLID)
    flagged, scan, _ = counts(w, H)
    assert sc(w, 9) > w["pair_cap"], f"{sc(w, 9)} pairs reserved, cap {w['pair_cap']}"
    assert int(flagged[0]) > 0 and int(scan[0]) == int(flagged[0]), (flagged.tolist(), scan.tolist())
    assert sc(w, 3) >= 0.9 * N


@pytest.mark.parametrize("metric", [EUCLID, DOT])
def test_route_multihead_mixed(metric):
    """three heads, each with its own route: re-rank, group rescan, full rescan"""
    H, N, K, d = 3, 300, 1100, 64
    g = _gen(71)
    C = torch.randn(H, K, d, generator=g, device=DEV)
    x = torch.randn(H, N, d, generator=g, device=DEV)
    for h, codes in enumerate([[0, 1, 64], [4, 6], [0, 512, 1024]]):
        xh, Ch = near_dup_case(1, N, K, d, F32, codes, 40, 72 + h)
        C[h], x[h] = Ch[0], xh[0]
    w, _ = full_check(x.to(BF16), C, metric, offset=2)
    flagged, _, _ = counts(w, H)
    assert int(flagged[2]) >= 36 and sc(w, 9) >= 64 * 36 and sc(w, 3) >= 2 * 36, (flagged.tolist(), sc(w, 9), sc(w, 3))


def test_route_unlowered():
    """rows ~1e5 above codes ~1e-3: E_k far above max |c|^2/2, the bias operand is left unlowered (scal[8] = 1)"""
    H, N, K, d = 1, 300, 1000, 64
    g = _gen(81)
    C = torch.randn(H, K, d, generator=g, device=DEV) * 1e-3
    x = torch.randn(H, N, d, generator=g, device=DEV) * 100.0
    w, aug = full_check(x, C, EUCLID)
    assert aug == 1 and sc(w, 8) == 1


@pytest.mark.parametrize("N,dtype", [(300, F32), (300, BF16), (100, F32)])
def test_route_negative_xinv(N, dtype):
    """one row 2^45 above the codebook: its bias operand is below fp16's range (xinv < 0), the row is rescanned"""
    H, K, d = 1, 512, 64
    g = _gen(91)
    C = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    x = torch.randn(H, N, d, generator=g, device=DEV)
    x[:, 2] *= 2.0 ** 45
    w, aug = full_check(x.to(dtype), C, EUCLID)
    assert float(w["xinv"][0, 2]) < 0 and bool((w["xinv"][0, 3:] > 0).all())
    if aug:
        assert sc(w, 2) >= 1


def test_route_prepared_l2norm():
    from vqb200 import ops
    H, N, K, d = 1, 300, 1000, 64
    g = _gen(101)
    C = torch.nn.functional.normalize(torch.randn(H, K, d, generator=g, device=DEV), dim=-1)
    cache = ops.prepare_codebook(C, True)
    xn = ops.l2norm_prepare(torch.randn(H, N, d, generator=g, device=DEV).to(BF16), K, cache)
    w, _ = full_check(xn, C, DOT, cache=cache, poison=False, latents_prepared=True)
    assert sc(w, 7) == int(cache[16:20].view(torch.int32)) & 0xFFFFFFFF, "scal[7] is not the cache's 2^q"


@pytest.mark.parametrize("ema,d", [(False, 100), (False, 64), (True, 64)])
def test_route_prepared_rvq(ema, d):
    from vqb200 import ops
    N, K = 1001, 512
    g = _gen(111)
    c = torch.randn(K, d, generator=g, device=DEV) * 0.5
    c2 = torch.randn(1, K, d, generator=g, device=DEV) * 0.2
    cache2 = ops.prepare_codebook(c2, False)
    r = torch.randn(N, d, generator=g, device=DEV)
    idx = torch.randint(0, K, (N,), generator=g, device=DEV)
    nxt = torch.empty_like(r)
    if ema:
        ops.rvq_level_ema(r, nxt, c, idx, True, False, torch.zeros_like(r), cache2)
    else:
        ops.rvq_level(r, nxt, c, idx, None, True, False, torch.zeros_like(r), cache2)
    w, _ = full_check(nxt[None], c2, EUCLID, cache=cache2, poison=False, latents_prepared=True)
    assert sc(w, 7) == int(cache2[16:20].view(torch.int32)) & 0xFFFFFFFF, "scal[7] is not the cache's 2^q"


@pytest.mark.parametrize("dtype", [BF16, F16])
def test_route_fused_prep(dtype):
    """in-kernel conversion (fused_prep) with outlier rows outside the sampled bound: they get xinv < 0 and are
    rescanned, and scal[1] carries their norm bound"""
    H, N, K, d = 2, 8200, 6144, 256
    g = _gen(121)
    C = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    x = torch.randn(H, N, d, generator=g, device=DEV)
    x[1, -8:] *= 50.0                                  # rows 16392.. of the batch: beyond the 16384 sampled ones
    w, aug = full_check(x.to(dtype), C, EUCLID, conv=True, fused_prep=True)
    assert aug == 1
    assert bool((w["xinv"][1, -8:] < 0).all()), "outlier rows kept their tensor-core candidates"
    assert sc(w, 2) >= 8
    assert scf(w, 1) >= 0.99 * float(x[1, -8:].float().norm(dim=1).max()), "scal[1] is not the outliers' norm bound"


@pytest.mark.parametrize("how,d,dtype", [("force_exact", 64, F32), ("no_cache", 30, BF16), ("wide", 640, F16)])
def test_route_exact(how, d, dtype):
    """the exact scan the rest of the suite compares with, against the restatement (scal[4] = 0: no tensor-core pass)"""
    from vqb200 import ops
    H, N, K = 2, 300, 1000
    g = _gen(131)
    C = torch.randn(H, K, d, generator=g, device=DEV) * 0.5
    x = torch.randn(H, N, d, generator=g, device=DEV)
    x[0, :64] = C[0, 900:964] + 1e-6 * x[0, :64]                       # near-ties with codes of high index
    C[0, 100:164] = C[0, 900:964]                                      # ... and exact duplicates at a lower one
    x = x.to(dtype)
    for metric in (EUCLID, DOT):
        cache = None if how == "no_cache" else ops.prepare_codebook(C, metric == DOT)
        w = run_search(x, C, metric, cache, offset=9, force_exact=how == "force_exact")
        assert sc(w, 4) == 0, "the tensor-core pass ran"
        if metric == EUCLID:
            assert bool((w["want_idx"][0, :64] < 900).all()), "duplicate codes: the lower index must win"


# ---- the tie edge ----------------------------------------------------------------------------------------------------
def _np_scores(x, cs, metric):
    """fp64 value before the fp32 cast, the fp32 d2 (euclid) and the fp32 score of row x against codes cs, as restate"""
    xd, cd = x.astype(np.float64), cs.astype(np.float64)
    dot = np.zeros(cs.shape[0])
    cn2 = np.zeros(cs.shape[0])
    n2 = 0.0
    for j in range(x.shape[0]):
        dot = dot + xd[j] * cd[:, j]
        cn2 = cn2 + cd[:, j] * cd[:, j]
        n2 = n2 + xd[j] * xd[j]
    if metric == EUCLID:
        pre = (n2 + cn2) - 2.0 * dot
        d2 = pre.astype(np.float32)
        return pre, d2, np.sqrt(np.maximum(d2, 0).astype(np.float64)).astype(np.float32)
    pre = -dot
    return pre, pre.astype(np.float32), pre.astype(np.float32)


def _partner(x, a, metric, kind):
    """b = a with one coordinate moved toward x so that b is nearer in fp64 and
    kind 'd2': fp32 d2 equal; 'sqrt': fp32 d2 differ, sqrtf equal; 'dot': fp32 -x.c equal; 'ulp': b's fp32 score one ulp
    below a's.  None if the ladder of step sizes finds no such b."""
    pre_a, d2_a, s_a = (v[0] for v in _np_scores(x, a[None], metric))
    if metric == EUCLID:
        diff = x.astype(np.float64) - a
        j = int(np.argmax(np.abs(diff)))
        unit = float(np.spacing(np.float32(d2_a))) / (2 * abs(diff[j]))
        sign = np.sign(diff[j])
    else:
        j = int(np.argmax(np.abs(x)))
        unit = float(np.spacing(np.float32(abs(s_a)))) / abs(float(x[j]))
        sign = np.sign(x[j])
    fs = np.linspace(0.01, 4.0, 800)
    bs = np.repeat(a[None], fs.size, axis=0)
    bs[:, j] = (a[j] + sign * fs * unit).astype(np.float32)
    pre, d2, s = _np_scores(x, bs, metric)
    ok = pre < pre_a
    if kind == "d2":
        ok &= d2 == d2_a
    elif kind == "sqrt":
        ok &= (d2 != d2_a) & (s == s_a)
    elif kind == "dot":
        ok &= s == s_a
    else:
        ok &= s == np.nextafter(s_a, np.float32(-np.inf))
    hit = np.nonzero(ok)[0]
    return bs[hit[len(hit) // 2]] if hit.size else None


def tie_case(regime, kinds, H, N, K, d, ia, ib, seed):
    """one tie pair (a at ia < ib) per head, N copies of the head's row; the other codes are clearly farther.
    far: |x| = 2^12, |c| = 2^-4 (kTieSlack alone covers the tie: 2 E_k ~ 2^-3 < ulp(d2) / 2 = 1);
    opposite: |x - c|^2 ~ 4 |x|^2 (codes opposite the row);  dot: x.a ~ 1, the other codes ~ 0.1"""
    rng = np.random.default_rng(seed)
    metric = DOT if regime == "dot" else EUCLID
    C = np.zeros((H, K, d), np.float32)
    X = np.zeros((H, d), np.float32)
    want = []
    for h in range(H):
        kind = kinds[h % len(kinds)]
        for _ in range(20):
            u = rng.standard_normal(d)
            u /= np.linalg.norm(u)
            if regime == "far":
                x = (u * 2.0 ** 12).astype(np.float32)
                a = (2.0 ** -4 * (u + 0.05 * rng.standard_normal(d) / math.sqrt(d))).astype(np.float32)
                fill = 2.0 ** -4 * rng.standard_normal((K, d)) / math.sqrt(d)
            elif regime == "opposite":
                x = u.astype(np.float32)
                a = (-u + 0.01 * rng.standard_normal(d) / math.sqrt(d)).astype(np.float32)
                fill = -1.6 * u + 0.3 * rng.standard_normal((K, d)) / math.sqrt(d)
            else:
                x = u.astype(np.float32)
                a = (u + 0.1 * rng.standard_normal(d) / math.sqrt(d)).astype(np.float32)
                fill = 0.1 * rng.standard_normal((K, d)) / math.sqrt(d)
            b = _partner(x, a, metric, kind)
            if b is not None:
                break
        assert b is not None, f"no {kind} partner found"
        C[h] = fill.astype(np.float32)
        C[h, ia], C[h, ib] = a, b
        X[h] = x
        want.append(ib if kind == "ulp" else ia)
    x = torch.from_numpy(np.repeat(X[:, None], N, axis=1)).to(DEV)
    return x, torch.from_numpy(C).to(DEV), metric, torch.tensor(want, device=DEV)


TIE_CASES = [
    # (regime, kinds, H, N, K): N = 1: single-tile kernel, N = 200: pair kernel (aug 1, or aug 2 for dot at K = 768)
    ("far", ("d2", "sqrt", "ulp"), 48, 1, 700),
    ("far", ("d2", "sqrt", "ulp"), 12, 200, 700),
    ("opposite", ("d2", "sqrt", "ulp"), 48, 1, 700),
    ("opposite", ("d2", "sqrt", "ulp"), 12, 200, 700),
    ("dot", ("dot", "ulp"), 48, 1, 700),
    ("dot", ("dot", "ulp"), 12, 200, 700),
    ("dot", ("dot", "ulp"), 12, 200, 768),
]


@pytest.mark.parametrize("regime,kinds,H,N,K", TIE_CASES,
                         ids=[f"{c[0]}-H{c[2]}-N{c[3]}-K{c[4]}" for c in TIE_CASES])
def test_tie_edge(regime, kinds, H, N, K):
    """a < b whose fp64 scores differ (b nearer: the tensor-core key ranks it first) but whose fp32 scores are equal:
    the search returns a; and the mirror, fp32 scores one ulp apart with b lower: not a tie, the search returns b"""
    d, ia, ib = 64, 5, 5 + 512 + 64 + 1
    x, C, metric, want = tie_case(regime, kinds, H, N, K, d, ia, ib, 141 + N + K)
    w, _ = full_check(x, C, metric, offset=100)
    got = w["want_idx"]
    assert torch.equal(got, want[:, None].expand(H, N)), "tie construction: the restatement's winner is not the intended code"
