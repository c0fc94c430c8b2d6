"""What a SimVQ training step costs on the GPU.

(a) `SimVQ` forward + backward + Adam step on the transform at the C2 shape (2^20 bf16 rows, d = 256) with K = 8192 and
    K = 65536 codes, rotation trick on (the default), against the same module written in plain torch (nearest code by
    `torch.cdist` on row chunks, upstream's loss and `rotate_to` by autograd) on the same GPU, and against the EMA
    `VectorQuantize` forward + backward at the same shape (no optimizer: its codebook is refreshed inside forward).
(b) `ResidualSimVQ` at the C4 shape (8 levels, K = 1024, d = 512, 64 x 4096 fp32 rows) forward + backward + Adam step,
    fused level loop against the generic per-level loop.

The inputs of every arm are two rotating buffers larger than the 126 MB L2.  Timing: CUDA events around `--iters`
steps after a warm-up, `--rounds` alternated rounds, median reported.  The card's name and power limit are read in
the same run.  One JSON line per measurement, appended to `--out`.

    python tools/bench_simvq.py --out profiles/bench_simvq.jsonl
"""
import argparse
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_rotation import ROOT, alternate, card, emit, rotate_to  # noqa: E402

DEV = "cuda:0"


class TorchSimVQ(torch.nn.Module):
    """Upstream SimVQ in plain torch: the same buffers and transform as a `vqb200.SimVQ`."""

    def __init__(self, ref, chunk):
        super().__init__()
        self.register_buffer("frozen_codebook", ref.frozen_codebook.clone())
        self.code_transform = torch.nn.Linear(ref.frozen_codebook.shape[1], ref.dim, bias=False).to(DEV)
        self.code_transform.load_state_dict(ref.code_transform.state_dict())
        self.beta, self.chunk = ref.input_to_quantize_commit_loss_weight, chunk

    def forward(self, x):
        x = x.reshape(-1, x.shape[-1]).float()
        codebook = self.code_transform(self.frozen_codebook)
        with torch.no_grad():
            cb = codebook.detach()
            idx = torch.cat([torch.cdist(x[i:i + self.chunk], cb).argmin(-1) for i in range(0, x.shape[0], self.chunk)])
        q = codebook[idx]
        loss = F.mse_loss(x.detach(), q) + self.beta * F.mse_loss(x, q.detach())
        return rotate_to(x, q), idx, loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_simvq.jsonl"))
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parts", default="a,b")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_simvq.py needs a CUDA device")
    from vqb200 import CodebookParams, ResidualSimVQ, SimVQ, VectorQuantize
    meta = card()
    parts = set(args.parts.split(","))
    gen = torch.Generator(device=DEV).manual_seed(0)

    def train_step(mod, xs, opt, out_grad):
        def f(i):
            x = xs[i % 2]
            x.grad = None
            q, _, loss = mod(x)
            torch.autograd.backward([q.reshape(out_grad.shape), loss.sum()], [out_grad, None])
            if opt is not None:
                opt.step()
                opt.zero_grad(set_to_none=True)
        return f

    if "a" in parts:
        N, d = 1 << 20, 256
        xs = [(torch.randn(1, N, d, generator=gen, device=DEV) * 0.04).to(torch.bfloat16).requires_grad_(True)
              for _ in range(2)]
        gq = torch.randn(1, N, d, generator=gen, device=DEV) * 1e-6
        for K in (8192, 65536):
            torch.manual_seed(0)
            vq = SimVQ(d, K).to(DEV).train()
            ref = TorchSimVQ(vq, chunk=16384 if K > 8192 else 65536).train()
            arms = {"vqb200_simvq": train_step(vq, xs, torch.optim.Adam(vq.parameters(), lr=1e-4), gq),
                    "torch_simvq": train_step(ref, xs, torch.optim.Adam(ref.parameters(), lr=1e-4), gq.reshape(N, d))}
            if K == 8192:
                torch.manual_seed(0)
                ema = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K,
                                                                           threshold_ema_dead_code=0)).to(DEV).train()
                ema.rotation_trick = True
                arms["vqb200_ema_vector_quantize"] = train_step(ema, xs, None, gq)
            res = alternate(arms, args.iters, args.rounds)
            for k, v in res.items():
                emit(args.out, {"part": "a", "workload": f"C2 shape: bf16 x (1, 2^20, 256), K={K}, rotation trick, "
                                "forward + backward" + (" + Adam step" if "simvq" in k else ""), "arm": k,
                                "ms_per_step": v["ms"], "ms_all": v["ms_all"]}, meta)
            emit(args.out, {"part": "a", "K": K, "speedup_over_torch": res["torch_simvq"]["ms"]
                            / res["vqb200_simvq"]["ms"]}, meta)
            del vq, ref, arms
            torch.cuda.empty_cache()
        del xs, gq
        torch.cuda.empty_cache()

    if "b" in parts:
        Q, K, d = 8, 1024, 512
        xs = [(torch.randn(64, 4096, d, generator=gen, device=DEV) * 0.03).requires_grad_(True) for _ in range(2)]
        g = torch.randn(64, 4096, d, generator=gen, device=DEV) * 1e-6
        arms = {}
        for fused in (True, False):
            torch.manual_seed(0)
            rsim = ResidualSimVQ(d, Q, K).to(DEV).train()
            rsim.use_fused_levels = fused
            arms["fused" if fused else "generic"] = train_step(rsim, xs, torch.optim.Adam(rsim.parameters(), lr=1e-4), g)
        res = alternate(arms, args.iters, args.rounds)
        for k, v in res.items():
            emit(args.out, {"part": "b", "workload": "C4 shape: ResidualSimVQ 8 x K=1024 x d=512, fp32 x (64, 4096, 512), "
                            "rotation trick, forward + backward + Adam step", "arm": k, "ms_per_step": v["ms"],
                            "ms_all": v["ms_all"]}, meta)
        emit(args.out, {"part": "b", "ratio_generic_over_fused": res["generic"]["ms"] / res["fused"]["ms"]}, meta)


if __name__ == "__main__":
    main()
