"""The latent operand of the tensor-core search, decoded from the search workspace and checked against fp64.

make_bias and resolve build their proof on these values (search_resolve.cu), the EMA kernels on scal[0] + scal[1]
(vqb.h).  Every writer is run: the generic prepare (lane-strided and 8-wide rows, several heads with N % 8 != 0),
prepare_latents4 (three dtypes, one and two heads), the narrow form (d_pad = 64 and 128), l2norm_prepare, the
ResidualVQ level (with and without a mask, training and eval, first and later level, lane-strided and float4 rows)
and the fused ResidualVQ level + EMA pass.  Per row:
  * |xinv| is a power of two, and xinv < 0 exactly when the bias operand a = 2^-q / |xinv| falls below 2^-24;
  * xaug = fp16({a, a, a, 0, 0, 0, 0, 0}), a = 0 for those rows;
  * xb is zero beyond d, and xn2 >= |x|^2;
and per batch: max |x~| <= scal[0] and max |x - x~| <= scal[1] with x~ = xb |xinv|, and scal[7] is the 2^q of the
cache for the writers outside the search (rvq_level, rvq_level_ema, l2norm_prepare with one head), else 0.
The offsets mirror search_layout (common.cuh).
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


def _align(n):
    return (n + 255) // 256 * 256


def decode(ws, H, N, d):
    """(xb (H*N, dp), xinv, xn2, xaug (H*N, 8), scal u32[10]) as fp64 / int tensors on the device"""
    dp = (d + 63) // 64 * 64
    rows = H * N
    o = 256 + _align(H * 12)
    xb = ws[o:o + rows * dp * 2].view(torch.float16).reshape(rows, dp).double()
    o += _align(rows * dp * 2)
    xinv = ws[o:o + rows * 4].view(torch.float32).double()
    o += _align(rows * 4)
    xn2 = ws[o:o + rows * 4].view(torch.float32).double()
    o += _align(rows * 4)
    xaug = ws[o:o + rows * 16].view(torch.float16).reshape(rows, 8)
    scal = ws[:40].view(torch.int32)
    return xb, xinv, xn2, xaug, scal


def check_operand(ws, x, cache, H, N, d, stamped, what):
    """x: the rows the operand was built from (H*N, d); cache: the codebook cache the operand is built for"""
    xb, xinv, xn2, xaug, scal = decode(ws, H, N, d)
    x = x.reshape(H * N, d).double()
    hdr = cache[:H * 32].view(torch.float32).reshape(H, 8)
    two_mq = hdr[:, 5].double().repeat_interleave(N)
    ainv = xinv.abs()
    mant, _ = torch.frexp(ainv)
    assert bool((mant == 0.5).all()), f"{what}: |xinv| not a power of two"
    a = two_mq / ainv
    a = torch.where(a >= 2.0 ** -24, a, torch.zeros_like(a))
    assert torch.equal(xinv < 0, a == 0), f"{what}: sign of xinv does not match the bias operand"
    want = torch.zeros(H * N, 8, dtype=torch.float16, device=DEV)
    want[:, :3] = a.to(torch.float16)[:, None]
    assert torch.equal(xaug.view(torch.int16), want.view(torch.int16)), f"{what}: xaug"
    assert bool((xb[:, d:] == 0).all()), f"{what}: xb not zero beyond d"
    n2 = (x * x).sum(1)
    bad = xn2 < n2
    assert not bool(bad.any()), f"{what}: xn2 < |x|^2 in {int(bad.sum())} rows"
    xt = xb[:, :d] * ainv[:, None]
    b0, b1 = scal[:2].view(torch.float32).double().tolist()
    assert float(xt.norm(dim=1).max()) <= b0, f"{what}: max |x~| > scal[0] = {b0}"
    assert float((x - xt).norm(dim=1).max()) <= b1, f"{what}: max |x - x~| > scal[1] = {b1}"
    s7 = int(scal[7])
    want7 = int(hdr[0, 4:5].view(torch.int32)) if stamped else 0
    assert s7 == want7, f"{what}: scal[7] = {s7:#x}, expected {want7:#x}"


def _codebook(H, K, d, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(H, K, d, generator=g, device=DEV) * 0.5


def _latents(H, N, d, dtype, seed):
    """rows of mixed scale, one zero row and, where the dtype has the range, one row far above the codebook (its bias
    operand falls below fp16's smallest subnormal: a negative xinv)"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(H, N, d, generator=g, device=DEV)
    x = x * torch.exp2(torch.randint(-6, 7, (H, N, 1), generator=g, device=DEV).float())
    x[:, 1] = 0.0
    if dtype != F16:
        x[:, 2] *= 2.0 ** 45
    return x.to(dtype)


# (d, H, N, dtype): generic prepare, prepare_latents4, narrow
SEARCH_CASES = [
    (100, 1, 1000, F32), (100, 2, 777, BF16),          # generic, lane-strided (d % 8 != 0)
    (384, 1, 1000, F32), (384, 1, 999, F16),           # generic, 8-wide
    (256, 2, 1001, F32), (256, 2, 1001, BF16),         # generic: two heads, N % 8 != 0
    (256, 1, 1003, F32), (256, 1, 1003, BF16), (256, 1, 1003, F16),    # prepare_latents4, one head
    (256, 2, 1000, F32), (256, 2, 1000, BF16), (256, 2, 1000, F16),    # prepare_latents4, two heads
    (64, 1, 1001, F32), (64, 2, 1000, BF16), (72, 1, 1001, F16), (72, 2, 999, F32),   # narrow
]


@pytest.mark.parametrize("d,H,N,dtype", SEARCH_CASES)
def test_prepare_latents(d, H, N, dtype):
    from vqb200 import ops
    c = _codebook(H, 512, d, 1)
    cache = ops.prepare_codebook(c, False)
    x = _latents(H, N, d, dtype, 2)
    _, _, ws = ops.search(x, c, cache, False)
    check_operand(ws, x, cache, H, N, d, False, f"prepare d={d} H={H} N={N} {dtype}")


@pytest.mark.parametrize("d,H,dtype", [(100, 1, F32), (100, 2, BF16), (512, 1, F16), (512, 2, F32)])
def test_l2norm_prepare(d, H, dtype):
    from vqb200 import _lib as L
    from vqb200 import ops
    N, K = 1001, 512
    c = _codebook(H, K, d, 3)
    cache = ops.prepare_codebook(c, True)
    x = _latents(H, N, d, dtype, 4)
    xn = ops.l2norm_prepare(x, K, cache)
    ws = ops.workspace("search", L.lib().vqb_search_workspace_bytes(H, N, K, d), x.device)
    check_operand(ws, xn, cache, H, N, d, H == 1, f"l2norm_prepare d={d} H={H} {dtype}")


@pytest.mark.parametrize("d,masked,training,first", [
    (30, False, True, True), (30, True, False, False),
    (100, True, True, False), (100, False, False, True),
    (512, False, True, False), (512, True, True, True), (512, False, False, False),
])
def test_rvq_level(d, masked, training, first):
    from vqb200 import _lib as L
    from vqb200 import ops
    N, K = 1001, 512
    g = torch.Generator(device=DEV).manual_seed(5)
    c = _codebook(1, K, d, 6)[0]
    cache2 = ops.prepare_codebook(_codebook(1, K, d, 7), False)
    r = _latents(1, N, d, F32, 8)[0]
    idx = torch.randint(0, K, (N,), generator=g, device=DEV)
    mask = (torch.rand(N, generator=g, device=DEV) < 0.7).to(torch.uint8) if masked else None
    out = torch.randn(N, d, generator=g, device=DEV)
    nxt = torch.empty_like(r)
    ops.rvq_level(r, nxt, c, idx, mask, training, first, out, cache2)
    ws = ops.workspace("search", L.lib().vqb_search_workspace_bytes(1, N, K, d), r.device)
    check_operand(ws, nxt, cache2, 1, N, d, True, f"rvq_level d={d} mask={masked} train={training} first={first}")


@pytest.mark.parametrize("d", [64, 512])
def test_rvq_level_ema(d):
    from vqb200 import _lib as L
    from vqb200 import ops
    N, K = 1001, 512
    g = torch.Generator(device=DEV).manual_seed(9)
    c = _codebook(1, K, d, 10)[0]
    cache2 = ops.prepare_codebook(_codebook(1, K, d, 11), False)
    r = _latents(1, N, d, F32, 12)[0]
    idx = torch.randint(0, K, (N,), generator=g, device=DEV)
    nxt = torch.empty_like(r)
    ops.rvq_level_ema(r, nxt, c, idx, True, False, torch.zeros_like(r), cache2)
    ws = ops.workspace("search", L.lib().vqb_search_workspace_bytes(1, N, K, d), r.device)
    check_operand(ws, nxt, cache2, 1, N, d, True, f"rvq_level_ema d={d}")
