"""The single-codebook gather, commitment backward and row normalisation kernels against fp64, on every dispatch branch.

(a) `gather_st_loss` (csrc/gather.cu): the narrow form (d a power of two from 8 to 128, several rows per warp), the
    8-wide form (d % 8 == 0), the float4 form (d % 8 == 4) and the scalar form (d % 4 != 0), in fp32, bf16 and fp16, with
    no mask, a partial mask, all ones and all zeros, training and eval, with and without the loss, empty batches and
    grids large enough for the persistent grid to stride and for `loss_finalize_kernel` to fold more than 256 partials.
(b) `st_commit_backward` and `quantize_training` under autograd, a learnable codebook included.
(c) `l2norm_rows`, `l2norm_prepare` (bit-identical outputs) and the normalisation's backward.
(d) one `VectorQuantize` training or eval step per path, against an fp64 restatement driven by the module's indices.
(e) the normalisation path hands the kernel a 16-byte aligned input.

Bounds.  u = 2^-24.  The depth m of a kernel is the number of fp32 terms one lane accumulates for one row:
  gather_st_loss: narrow 8, 8-wide 8 ceil(d/256), float4 4 ceil(d/128), scalar ceil(d/32);
  quantize_ema (the fused pass of an un-masked EMA step): 8 ceil(d/256) terms, then a butterfly over the log2(d/8)
    lanes of a row (d <= 256 here);
  l2norm_rows: float4 4 ceil(d/128) for d % 4 == 0, else scalar ceil(d/32).
* loss[0] = mean over the live rows of (c - x)^2.  Every lane squares fl(c - x) = (c - x)(1 + e), |e| <= u, so each term
  carries (1 + e)^2 (2u), the chain of m fmas of non-negative terms adds gamma_m ~ m u, the per-row partials are folded
  in fp64 (relative error below 2^-45 for the batches here) and the fp64 mean is cast to fp32 (u):
      |loss[0] - ref| <= 1.01 (m + 3) u ref
  (1.01 covers gamma_m - m u and the fp64 folding).  loss[1] is the live row count over all heads, exactly; with no
  live row loss[0] is NaN and loss[1] is 0, as torch's mean of an empty tensor gives.
* q: training fl(x + fl(c - x)), eval c, bit for bit (two correctly rounded fp32 operations, no contraction).
* st_commit_backward: fmaf(s, fl(x - c), g) with s = fl(coef g_loss) in fp32.  The subtraction adds u |s (x - c)|, the
  fma one rounding of the result:
      |got - (g + s (x - c))| <= u (|g + s (x - c)| + |s (x - c)|) (1 + 2u);   rows outside the mask: g bit for bit.
* quantize_training backward: s = fl(fl(w fl(2/d)) / rows) is within 3u of 2w/(rows d), so the bound above becomes
  u |ref| + 4.01 u |s (x - c)| in fp32; a 16-bit x receives the gradient rounded to its type, adding
  u16 (|ref| + bound32) (u16 = 2^-8 bf16, 2^-11 fp16) plus half the fp16 subnormal spacing.
  Codebook gradient s (n_k C_k - S_k), S_k the fixed-point segmented sum of the assigned rows (ema.cu: error at most
  n_k times the quantum 2^(e + lr - 61) <= max|x| (N + 1) 2^-59, plus half an fp32 ulp): fl(n_k C_k) (u n_k |C_k|), the
  subtraction (u |D|), s (3u) and the product (u) give
      |got - s D| <= 1.01 |s| (u (n_k |C_k| + |S_k|) + 5 u |D| + n_k max|x| (N + 1) 2^-59).
* l2norm_rows: x / max(|x|, 1e-12) with eps the fp32 1e-12 that F.normalize uses.  The squared norm has m fma roundings
  and 5 of the warp butterfly (gamma_(m+5) on non-negative terms), sqrtf halves that and adds u, __fdiv_rn adds u:
      |got - ref| <= ((m + 5)/2 + 2) u |ref|   per element.
  Rows whose fp32 |x|^2 leaves the normal range follow fp32 F.normalize on the device (test_l2norm_rows_extreme_scales).
* normalisation backward (torch fp32 glue in `_L2NormRows.backward`): g.y and |x| are fp32 reductions in torch's order
  (gamma_d for any order), y carries the bound above, the rest is 4 roundings:
      |got - ref| <= (d + 10) u ((|g_i| + 2 |y_i| |g|_2) / max(|x|, eps) + |ref_i|).
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
DTYPES = (F32, BF16, F16)
U16 = {F32: 0.0, BF16: 2.0 ** -8, F16: 2.0 ** -11}
ABS16 = {F32: 0.0, BF16: 0.0, F16: 2.0 ** -25}       # half the fp16 subnormal spacing
EPS32 = float(torch.tensor(1e-12, dtype=F32))
DN = {F32: "f32", BF16: "bf16", F16: "f16"}


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(shape, seed, dtype=F32, scale=1.0):
    return (torch.randn(shape, generator=_gen(seed), device=DEV) * scale).to(dtype)


def depth_gather(d):
    if 8 <= d <= 128 and d & (d - 1) == 0:
        return 8
    if d % 8 == 0:
        return 8 * math.ceil(d / 256)
    if d % 4 == 0:
        return 4 * math.ceil(d / 128)
    return math.ceil(d / 32)


def depth_fused(d):
    assert d % 8 == 0 and d <= 256
    return 8 + int(math.log2(d // 8))


def depth_l2(d):
    return 4 * math.ceil(d / 128) if d % 4 == 0 else math.ceil(d / 32)


def _mask(kind, N, seed):
    """(bool live (N,), uint8 mask for the kernels or None)."""
    if kind == "none":
        return torch.ones(N, dtype=torch.bool, device=DEV), None
    if kind == "partial":
        live = torch.rand(N, generator=_gen(seed), device=DEV) > 0.4
    elif kind == "ones":
        live = torch.ones(N, dtype=torch.bool, device=DEV)
    else:
        live = torch.zeros(N, dtype=torch.bool, device=DEV)
    return live, live.to(torch.uint8)


def _inputs(H, N, d, dtype, seed, K=37):
    x = _randn((H, N, d), seed, dtype)
    cb = _randn((H, K, d), seed + 1)
    idx = torch.randint(0, K, (H, N), generator=_gen(seed + 2), device=DEV)
    return x, cb, idx


def _gathered(cb, idx):
    H, N = idx.shape
    d = cb.shape[-1]
    return torch.gather(cb, 1, idx[..., None].expand(H, N, d))


def _bits(t):
    return t.contiguous().view(torch.int32)


def check_loss(loss, x, c, live, m, what):
    """loss = [mean over live rows of (c - x)^2, live rows over all heads] against fp64 (bound in the module doc)."""
    H = x.shape[0]
    n_live = H * int(live.sum())
    got0, got1 = float(loss[0]), float(loss[1])
    assert got1 == float(n_live), f"{what}: rows used {got1} != {n_live}"
    if n_live == 0:
        assert math.isnan(got0), f"{what}: loss of no live row is {got0}, not NaN"
        return
    per = ((c.double() - x.double()) ** 2).sum(-1)
    ref = float(per[:, live].sum()) / (n_live * x.shape[-1])
    err = abs(got0 - ref)
    bar = 1.01 * (m + 3) * U * ref
    assert err <= bar, f"{what}: loss {got0} vs fp64 {ref}: |err| {err:.3e} > {bar:.3e} (m = {m})"


# --------------------------------------------------------------------------------------------------- (a) gather
FORMS = {"narrow": (8, 16, 32, 64, 128), "wide8": (136, 256, 384, 1024, 2048), "float4": (4, 12, 100, 260),
         "scalar": (1, 3, 30, 129, 641)}
NS = (0, 1, 7, 1000, 4097)
MASKS = ("none", "partial", "ones", "zeros")
FLAGS = ((True, True), (True, False), (False, True), (False, False))      # (training, want_loss)


def _gather_cases():
    """Per form: every dtype x mask x (training, want_loss); the widths, N and H cycle under that product."""
    out = []
    for form, ds in FORMS.items():
        i = 0
        for dt in DTYPES:
            for mk in MASKS:
                for tr, wl in FLAGS:
                    d, N, H = ds[i % len(ds)], NS[(i // len(ds)) % len(NS)], (1, 3)[(i // 2) % 2]
                    out.append(pytest.param(d, dt, H, N, mk, tr, wl,
                                            id=f"{form}-d{d}-{DN[dt]}-H{H}-N{N}-{mk}-{'train' if tr else 'eval'}"
                                               f"{'-loss' if wl else ''}"))
                    i += 1
    return out


def _check_gather(d, dtype, H, N, mask_kind, training, want_loss, seed):
    from vqb200 import ops
    x, cb, idx = _inputs(H, N, d, dtype, seed)
    live, m8 = _mask(mask_kind, N, seed + 3)
    what = f"gather d={d} {dtype} H={H} N={N} {mask_kind} training={training}"
    q, loss = ops.gather_st_loss(x, cb, idx, m8, training, want_loss)
    c = _gathered(cb, idx)
    if training:
        xf = x.float()
        ref = xf + (c - xf)
    else:
        ref = c
    assert torch.equal(_bits(q), _bits(ref)), f"{what}: q differs from {'fl(x + fl(c - x))' if training else 'C[idx]'}"
    if want_loss:
        check_loss(loss, x, c, live, depth_gather(d), what)
    else:
        assert loss is None


@pytest.mark.parametrize("d,dtype,H,N,mask_kind,training,want_loss", _gather_cases())
def test_gather_st_loss_matches_fp64(d, dtype, H, N, mask_kind, training, want_loss):
    _check_gather(d, dtype, H, N, mask_kind, training, want_loss, seed=d * 7 + N)


@pytest.mark.parametrize("d,dtype,H,N", [
    pytest.param(8, F32, 1, 1 << 20, id="narrow-d8-32rows_per_warp"),
    pytest.param(64, BF16, 2, 1 << 19, id="narrow-d64"),
    pytest.param(1024, F16, 1, 100_000, id="wide8-d1024"),
])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_gather_st_loss_strided_grid(d, dtype, H, N, training):
    """H N rows far above the persistent grid (148 SMs x 8 blocks x 8 warps): every warp strides, the finalize folds
    1184 partials (its strided loop and its tree)."""
    _check_gather(d, dtype, H, N, "partial", training, True, seed=5)


# ------------------------------------------------------------------------------------------ (b) commitment backward
def _backward_cases():
    out = []
    svals = (0.37, -1.9e-3, 0.0, 3.5)
    for form, ds in FORMS.items():
        i = 0
        for dt in DTYPES:
            for mk in MASKS:
                d, N, H = ds[i % len(ds)], NS[1 + i % 4], (1, 3)[i % 2]
                s, gzero = svals[i % 4], (i // 4) % 3 == 1
                out.append(pytest.param(d, dt, H, N, mk, s, gzero,
                                        id=f"{form}-d{d}-{DN[dt]}-H{H}-N{N}-{mk}-s{s}{'-g0' if gzero else ''}"))
                i += 1
    return out


@pytest.mark.parametrize("d,dtype,H,N,mask_kind,s,g_zero", _backward_cases())
def test_st_commit_backward_matches_fp64(d, dtype, H, N, mask_kind, s, g_zero):
    from vqb200 import ops
    x, cb, idx = _inputs(H, N, d, dtype, seed=d + 11 * N)
    live, m8 = _mask(mask_kind, N, seed=d)
    gq = torch.zeros(H, N, d, device=DEV) if g_zero else _randn((H, N, d), seed=d + 1)
    gl = torch.tensor([s], dtype=F32, device=DEV)
    gx = ops.st_commit_backward(gq, gl, x, cb, idx, m8)
    sd = float(gl[0])                                    # fl(1.0 * g_loss) = g_loss
    sdiff = sd * (x.double() - _gathered(cb, idx).double())
    ref = gq.double() + sdiff
    bar = U * (ref.abs() + sdiff.abs()) * (1 + 2 * U)
    err = (gx.double() - ref).abs()
    rows = live[None, :].expand(H, N)
    bad = (err > bar) & rows[..., None]
    assert not bool(bad.any()), f"{int(bad.sum())} elements beyond the bound, worst {float((err - bar).max()):.3e}"
    assert torch.equal(_bits(gx[~rows]), _bits(gq[~rows])), "rows outside the mask must return grad_q bit for bit"


def _codebook_grad_bar(x, cb, idx, live, s):
    """(|s| (u (n_k |C_k| + |S_k|) + 5 u |D| + n_k max|x| (N + 1) 2^-59) 1.01, D = n_k C - S) per code (module doc)."""
    H, N, d = x.shape
    K = cb.shape[1]
    xs = x.double() * live[None, :, None]
    S = torch.zeros(H, K, d, dtype=torch.float64, device=DEV).scatter_add_(1, idx[..., None].expand(H, N, d), xs)
    n = torch.zeros(H, K, dtype=torch.float64, device=DEV).scatter_add_(
        1, idx, live[None, :].expand(H, N).double())[..., None]
    D = n * cb.double() - S
    mx = float(x.double().abs().max()) if x.numel() else 0.0
    return 1.01 * abs(s) * (U * (n * cb.double().abs() + S.abs()) + 5 * U * D.abs() + n * mx * (N + 1) * 2.0 ** -59)


def _autograd_case(d, dtype, H, N, mask_kind, grads, learnable, seed):
    """x.grad and, for a learnable codebook, embeddings.grad of quantize_training against fp64 autograd of
    x + (c - x).detach() and w mean_live((c - x)^2) with the same indices."""
    from vqb200 import ops
    W = 0.75
    x0, cb0, idx = _inputs(H, N, d, dtype, seed)
    live, m8 = _mask(mask_kind, N, seed + 3)
    gq = _randn((H, N, d), seed + 4)
    x = x0.clone().requires_grad_(True)
    emb = cb0.clone().requires_grad_(learnable)
    q, commit, _ = ops.quantize_training(x, emb, idx, m8, True)
    obj = 0
    if grads in ("q", "both"):
        obj = obj + (q * gq).sum()
    if grads in ("loss", "both"):
        obj = obj + commit * W
    obj.backward()

    xr = x0.double().requires_grad_(True)
    cr = cb0.double().requires_grad_(learnable)
    c = _gathered(cr, idx)
    qr = xr + (c - xr).detach()
    objr = 0
    if grads in ("q", "both"):
        objr = objr + (qr * gq.double()).sum()
    if grads in ("loss", "both"):
        objr = objr + ((c - xr) ** 2)[:, live].mean() * W
    objr.backward()

    rows = H * int(live.sum())
    s = 2.0 * W / (rows * d) if (rows and grads != "q") else 0.0
    what = f"d={d} {dtype} H={H} N={N} {mask_kind} grads={grads} learnable={learnable}"
    assert x.grad.dtype == dtype
    ref = xr.grad
    sdiff = (s * (x0.double() - c.detach())).abs() * live[None, :, None]
    b32 = U * ref.abs() + 4.01 * U * sdiff
    bar = b32 + U16[dtype] * (ref.abs() + b32) + ABS16[dtype]
    err = (x.grad.double() - ref).abs()
    assert bool((err <= bar).all()), f"{what}: x.grad off by {float((err - bar).max()):.3e} beyond the bound"
    if learnable:
        g = emb.grad
        assert g is not None and bool(torch.isfinite(g).all()), f"{what}: codebook gradient not finite"
        bar_c = _codebook_grad_bar(x0, cb0, idx, live, s)
        ref_c = cr.grad if cr.grad is not None else torch.zeros_like(cr)      # c enters q only detached
        err_c = (g.double() - ref_c).abs()
        assert bool((err_c <= bar_c).all()), \
            f"{what}: embeddings.grad off by {float((err_c - bar_c).max()):.3e} beyond the bound"
    else:
        assert emb.grad is None


@pytest.mark.parametrize("learnable", [False, True], ids=["frozen", "learnable"])
@pytest.mark.parametrize("grads", ["loss", "q", "both"])
@pytest.mark.parametrize("dtype,d", [(F32, 64), (BF16, 100), (F16, 30)], ids=["f32-d64", "bf16-d100", "f16-d30"])
@pytest.mark.parametrize("mask_kind", ["none", "partial", "zeros"])
def test_quantize_training_autograd_matches_fp64(mask_kind, dtype, d, grads, learnable):
    _autograd_case(d, dtype, 2, 777, mask_kind, grads, learnable, seed=d)


@pytest.mark.parametrize("grads", ["loss", "both"])
@pytest.mark.parametrize("N,mask_kind", [(0, "none"), (0, "partial"), (300, "zeros")], ids=["N0", "N0-mask", "all-masked"])
def test_quantize_training_no_live_rows_sends_no_codebook_gradient(N, mask_kind, grads):
    """The mean over an empty selection: loss NaN, and a zero gradient to the codebook (the reference indexes an empty
    selection) rather than 0 * inf."""
    _autograd_case(64, F32, 1, N, mask_kind, grads, True, seed=9)


# ------------------------------------------------------------------------------------------------ (c) normalisation
def _l2_rows(R, d, dtype, seed):
    """Rows at scales 1e-3 .. 1e3, two zero rows and (outside fp16) two rows with |x| < 1e-12."""
    x = _randn((R, d), seed) * torch.logspace(-3, 3, R, device=DEV)[:, None]
    x[3] = 0
    x[R - 2] = 0
    if dtype != F16:
        x[5] *= 1e-14 / float(x[5].norm())
        x[7] = _randn((d,), seed + 1) * 1e-16
    return x.to(dtype)


def _l2_ref(x):
    xd = x.double()
    return xd / xd.norm(dim=-1, keepdim=True).clamp_min(EPS32)


@pytest.mark.parametrize("dtype", DTYPES, ids=[DN[t] for t in DTYPES])
@pytest.mark.parametrize("d", [1, 3, 30, 129, 641, 2047, 4, 12, 64, 100, 260, 512, 2048])
def test_l2norm_rows_matches_fp64(d, dtype):
    from vqb200 import ops
    x = _l2_rows(40, d, dtype, seed=d)
    y = ops.l2norm_rows(x)
    ref = _l2_ref(x)
    bar = ((depth_l2(d) + 5) / 2 + 2) * U * ref.abs()
    err = (y.double() - ref).abs()
    assert bool((err <= bar).all()), f"d={d}: worst excess {float((err - bar).max()):.3e}"
    assert bool((y[3] == 0).all()) and bool((y[-2] == 0).all()), "zero rows must give zeros"
    if dtype != F16:
        tiny = x[[5, 7]].float()
        assert torch.equal(_bits(y[[5, 7]]), _bits(tiny / torch.tensor(EPS32, device=DEV))), \
            "rows with |x| < 1e-12 must give x / 1e-12"


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["f32", "bf16"])
@pytest.mark.parametrize("d", [3, 64, 641, 2048])
def test_l2norm_rows_extreme_scales(d, dtype):
    """fp32 |x|^2 subnormal (1e-22) or overflowing (1e19, 1e20).  Both this kernel and fp32 F.normalize on the device
    return x / 1e-12 for the first (|x| < 1e-12 whatever the squares round to) and zeros for the others (|x|^2 = inf,
    x / inf = 0): the contract is F.normalize's, bit for bit."""
    from vqb200 import ops
    base = _randn((6, d), seed=d)
    scales = torch.tensor([1e-22, 1e-22, 1e19, 1e19, 1e20, 1e20], device=DEV)[:, None]
    x = (base * scales).to(dtype)
    y = ops.l2norm_rows(x)
    ref = F.normalize(x.float(), dim=-1)
    assert torch.equal(_bits(y), _bits(ref)), "differs from fp32 F.normalize"
    assert torch.equal(_bits(y[:2]), _bits(x[:2].float() / torch.tensor(EPS32, device=DEV)))
    big = y[2:] if d > 3 else y[4:]          # d = 3 at 1e19: |x|^2 stays finite
    assert bool((big == 0).all())


@pytest.mark.parametrize("dtype", DTYPES, ids=[DN[t] for t in DTYPES])
def test_l2norm_prepare_out_is_l2norm_rows_bit_for_bit(dtype):
    from vqb200 import ops
    for d in range(4, 513, 4):
        assert ops.l2norm_prepare_supported(d), d
        for H in (1, 2):
            x = _l2_rows(40, d, dtype, seed=d + H).reshape(H, 40 // H, d)
            cache = ops.prepare_codebook(_randn((H, 33, d), seed=d), True)
            got = ops.l2norm_prepare(x, 33, cache)
            ref = ops.l2norm_rows(x)
            assert torch.equal(_bits(got), _bits(ref)), f"d={d} H={H}: l2norm_prepare out != l2norm_rows"


@pytest.mark.parametrize("dtype", DTYPES, ids=[DN[t] for t in DTYPES])
@pytest.mark.parametrize("d", [3, 64, 100, 641])
def test_l2norm_rows_autograd_matches_fp64(d, dtype):
    from vqb200 import ops
    x0 = _l2_rows(40, d, dtype, seed=d)
    if dtype == F16:
        x0[3] = x0[-2] = x0[0]      # g / 1e-12 overflows fp16: zero rows are checked in fp32 and bf16
    g = _randn((40, d), seed=d + 5)
    x = x0.clone().requires_grad_(True)
    (ops.l2norm_rows_autograd(x) * g).sum().backward()
    xr = x0.double().requires_grad_(True)
    (F.normalize(xr, dim=-1, eps=EPS32) * g.double()).sum().backward()
    ref = xr.grad
    denom = x0.double().norm(dim=-1, keepdim=True).clamp_min(EPS32)
    y = _l2_ref(x0)
    b32 = (d + 10) * U * ((g.double().abs() + 2 * y.abs() * g.double().norm(dim=-1, keepdim=True)) / denom + ref.abs())
    bar = b32 + U16[dtype] * (ref.abs() + b32) + ABS16[dtype]
    err = (x.grad.double() - ref).abs()
    assert x.grad.dtype == dtype
    assert bool((err <= bar).all()), f"d={d}: worst excess {float((err - bar).max()):.3e}"


# ---------------------------------------------------------------------------------------- (d) one module step per path
def _vq(**kw):
    from vqb200 import CodebookParams, VectorQuantize
    torch.manual_seed(0)
    dim = kw.pop("dim", 64)
    cp = dict(dim=dim, codebook_size=128, threshold_ema_dead_code=0)
    cp.update(kw.pop("cp", {}))
    return VectorQuantize(dim=dim, codebook_params=CodebookParams(**cp), **kw).to(DEV)


STEPS = {
    "fused-f32": dict(),
    "fused-bf16": dict(dtype=BF16),
    "masked-f32": dict(mask=True),
    "masked-bf16": dict(mask=True, dtype=BF16),
    "heads3-separate": dict(vq=dict(dim=96, heads=3, codebook_dim=32, separate_codebook_per_head=True)),
    "heads3-separate-masked": dict(mask=True, vq=dict(dim=96, heads=3, codebook_dim=32, separate_codebook_per_head=True)),
    "learnable-masked": dict(mask=True, vq=dict(cp=dict(learnable_codebook=True, ema_update=False))),
    "learnable-bf16": dict(dtype=BF16, vq=dict(cp=dict(learnable_codebook=True, ema_update=False))),
    "cosine-l2norm": dict(vq=dict(cp=dict(use_cosine_sim=True, transform_input="l2norm",
                                          weights_regularization="l2norm"))),
    "eval": dict(eval=True),
    "eval-masked-bf16": dict(eval=True, mask=True, dtype=BF16),
}


def _split_rows(vq, t):
    """(B, n, dim) -> the codebook's (H, B n, dh) row layout, and its inverse."""
    B, n, dim = t.shape
    H = vq.heads
    if H == 1:
        return t.reshape(1, B * n, dim), lambda r: r.reshape(B, n, dim)
    dh = dim // H
    return t.reshape(B, n, H, dh).permute(2, 0, 1, 3).reshape(H, B * n, dh), \
        lambda r: r.reshape(H, B, n, dh).permute(1, 2, 0, 3).reshape(B, n, dim)


@pytest.mark.parametrize("name", list(STEPS))
def test_vq_step_matches_fp64(name):
    cfg = STEPS[name]
    dtype = cfg.get("dtype", F32)
    vq = _vq(**dict(cfg.get("vq", {})))
    vq.eval() if cfg.get("eval") else vq.train()
    dim = vq.dim
    B, n = 3, 170
    x0 = _randn((B, n, dim), seed=1, dtype=dtype)
    w = _randn((B, n, dim), seed=2)
    mask = (torch.rand(B, n, generator=_gen(3), device=DEV) > 0.3) if cfg.get("mask") else None
    cb = vq._codebook
    pre = cb.embeddings.detach().clone()
    learnable = cb.embeddings.requires_grad
    training = not cfg.get("eval")
    x = x0.clone().requires_grad_(training)
    q, ind, loss = vq(x, mask=mask)
    rows, back = _split_rows(vq, x0)
    H, N, dh = rows.shape
    irow = ind.permute(2, 0, 1).reshape(H, N) if H > 1 else ind.reshape(1, N)
    live = cb._expand_mask(mask, N).bool() if mask is not None else torch.ones(N, dtype=torch.bool, device=DEV)
    keep = live[None, :, None]

    # the rows the codebook saw
    xr = rows.double().requires_grad_(training)
    e = F.normalize(xr, dim=-1, eps=EPS32) if cb.input_l2norm else xr
    cr = pre.double().requires_grad_(learnable and training)
    c = _gathered(cr, irow)
    q_rows = _split_rows(vq, q.detach())[0]
    if not training:
        got = torch.where(keep, q_rows, rows.float())
        ref = torch.where(keep, c.detach().float(), rows.float())
        assert torch.equal(_bits(got), _bits(ref)), f"{name}: eval quantize is not C[idx]"
        return
    ef = cb.transform_input(rows.detach()) if cb.input_l2norm else rows.float()
    ref_q = torch.where(keep, ef + (c.detach().float() - ef), rows.float())
    assert torch.equal(_bits(q_rows), _bits(ref_q)), f"{name}: quantize is not fl(x + fl(c - x))"

    fused = mask is None and not learnable and cb.fused_quantize_ema
    m = depth_fused(dh) if fused else depth_gather(dh)
    # a cosine codebook: against the fp64 loss of the kernel's own normalised rows (their bound is checked in (c))
    check_loss(torch.stack([loss.detach().reshape(()), torch.tensor(float(H * int(live.sum())), device=DEV)]),
               ef, c.detach(), live, m, name)

    ((q * w).sum() + loss.sum() * 3.0).backward()
    wr = _split_rows(vq, w)[0].double()
    qr = e + (c - e).detach()
    per = ((c - e) ** 2)[:, live].mean()
    ((torch.where(keep, qr, xr) * wr).sum() + per * 3.0).backward()
    s = 2.0 * 3.0 / (H * int(live.sum()) * dh)
    ref = back(xr.grad)
    if cb.input_l2norm:
        # grad through F.normalize: (d + 10) u relative to (|g| + 2 |y| |g|_2) / |x| on top of the commitment bound
        gi = (wr + s * (e - c) * keep).detach()
        denom = xr.detach().norm(dim=-1, keepdim=True).clamp_min(EPS32)
        b32 = back((dh + 10) * U * ((gi.abs() + 2 * e.detach().abs() * gi.norm(dim=-1, keepdim=True)) / denom
                                     + xr.grad.abs()))
    else:
        sdiff = back((s * (xr - c).detach()).abs() * keep)
        b32 = U * ref.abs() + 4.01 * U * sdiff
    bar = b32 + U16[dtype] * (ref.abs() + b32) + ABS16[dtype]
    err = (x.grad.double() - ref).abs()
    assert bool((err <= bar).all()), f"{name}: x.grad worst excess {float((err - bar).max()):.3e}"
    if learnable:
        bar_c = _codebook_grad_bar(rows, pre, irow, live, s)
        err_c = (cb.embeddings.grad.double() - cr.grad).abs()
        assert bool((err_c <= bar_c).all()), f"{name}: embeddings.grad worst excess {float((err_c - bar_c).max()):.3e}"


# -------------------------------------------------------------------------------------- (e) alignment of the input
def _unaligned(shape, dtype):
    """A contiguous tensor whose data starts 4 bytes past a 16-byte boundary."""
    numel = math.prod(shape)
    step = 4 // torch.tensor([], dtype=dtype).element_size()
    buf = _randn((numel + 16,), seed=numel, dtype=dtype)
    t = buf[step:step + numel].view(shape)
    assert t.is_contiguous() and t.data_ptr() % 16 == 4
    return t


def test_l2norm_wrappers_hand_the_kernel_an_aligned_input(monkeypatch):
    """With the library entry stubbed (no kernel runs), every route to vqb_l2norm_rows passes a 16-byte aligned x."""
    from vqb200 import _lib, ops
    from vqb200.codebook import Codebook
    seen = []
    real = _lib.lib()

    class Stub:
        def __getattr__(self, name):
            return getattr(real, name)

        @staticmethod
        def vqb_l2norm_rows(x, dtype, out, rows, d, stream):
            seen.append(x)
            return 0

    cb = Codebook(dim=64, codebook_size=16, transform_input="l2norm").to(DEV)
    monkeypatch.setattr(_lib, "lib", lambda: Stub())
    for dtype in DTYPES:
        x = _unaligned((5, 64), dtype)
        ops.l2norm_rows(x)
        cb.transform_input(x)                  # VectorQuantize._inplace_optimize normalises its input this way
        ops.l2norm_rows_autograd(x)
    assert len(seen) == 9
    assert all(p % 16 == 0 for p in seen), [p % 16 for p in seen]


@pytest.mark.parametrize("dtype", DTYPES, ids=[DN[t] for t in DTYPES])
def test_l2norm_rows_unaligned_input_real_kernel(dtype):
    """An input 4 bytes past a 16-byte boundary gives the same rows as an aligned copy."""
    from vqb200 import ops
    x = _unaligned((33, 128), dtype)
    assert torch.equal(_bits(ops.l2norm_rows(x)), _bits(ops.l2norm_rows(x.clone())))
