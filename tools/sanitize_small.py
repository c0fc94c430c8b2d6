"""Small end-to-end run for compute-sanitizer (one tool per run): search, gather, EMA reduce/apply, expiry scatter,
RVQ level, on small ragged shapes."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vector-quantization-by-ml_b200"))
import torch

from vqb200 import CodebookParams, ResidualVQ, VectorQuantize, ops

dev = torch.device("cuda:0")
torch.manual_seed(0)
for (H, N, K, d, cos) in [(1, 300, 520, 72, False), (2, 257, 300, 256, True), (1, 1000, 1100, 512, False)]:
    x = torch.randn(H, N, d, device=dev)
    c = torch.randn(H, K, d, device=dev) * 0.5
    cache = ops.prepare_codebook(c, cos)
    a, _, ws = ops.search(x, c, cache, cos, want_score=True)
    b, _, _ = ops.search(x, c, cache, cos, force_exact=True)
    assert torch.equal(a, b)
    q, loss = ops.gather_st_loss(x, c, a, None, True, True)
    st = ops.ema_reduce(x, a, None, K, bound_ws=ws)
vq = VectorQuantize(dim=40, codebook_params=CodebookParams(dim=40, codebook_size=70)).to(dev).train()
xx = torch.randn(3, 50, 40, device=dev, requires_grad=True)
q, i, l = vq(xx)
(q.sum() + l.sum()).backward()
rvq = ResidualVQ(dim=24, num_quantizers=3, codebook_params=CodebookParams(dim=24, codebook_size=40)).to(dev).train()
with torch.no_grad():
    rvq(torch.randn(2, 64, 24, device=dev))
torch.cuda.synchronize()
print("SANITIZE RUN OK")
