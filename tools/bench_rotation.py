"""What the rotation-trick gradient (`VectorQuantize.rotation_trick`) costs on the GPU, against straight-through.

(a) `vqb_rot_commit_backward` against `vqb_st_commit_backward` at the C2 shape (N = 2^20 rows, d = 256, K = 8192 codes,
    fp32 and bf16 x; every input is larger than the 126 MB L2), launched alternately.  GB/s is on the algorithmic bytes
    of a row: x (sz d), grad_q (4 d), the index (8) and grad_x (4 d).  The code rows are not counted: the 8 MiB codebook
    is L2-resident.
(b) The C2 `VectorQuantize` forward + backward step (fp32 latents with requires_grad), straight-through vs rotation.
(c) The C4 `ResidualVQ` (8 levels, K = 1024, d = 512, 64 x 4096 latents) forward + backward step: fused loop with
    rotation, fused with straight-through, and the generic per-level loop with rotation.
(d) Upstream's `rotate_to` written in torch (autograd forward + backward) at the C2 shape, for context.

Timing: CUDA events around `--iters` calls after a warm-up, `--rounds` alternated rounds, median reported.  The card's
name and power limit are read in the same run.  One JSON line per measurement, appended to `--out`.

    python tools/bench_rotation.py --out profiles/bench_rotation.jsonl
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vector-quantization-by-ml_b200")]

DEV = "cuda:0"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(arms, iters, rounds, warmup=2):
    """{name: fn}: every arm warmed up, then `rounds` rounds of one timed window per arm; median ms per call."""
    for fn in arms.values():
        for i in range(warmup):
            fn(i)
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn, iters))
    return {k: {"ms": statistics.median(v), "ms_all": v} for k, v in times.items()}


def emit(out, rec, meta):
    rec = {**rec, **meta}
    print(json.dumps(rec), flush=True)
    with open(out, "a") as f:
        f.write(json.dumps(rec) + "\n")


def rotate_to(x, c):
    """Upstream vector-quantize-pytorch `rotate_to(src=x, tgt=c)` in torch."""
    nx, nc = x.norm(dim=-1, keepdim=True), c.norm(dim=-1, keepdim=True)
    u, q = x / nx.clamp(min=1e-6), c / nc.clamp(min=1e-6)
    w = F.normalize(u + q, dim=-1).detach()
    e = x[:, None, :]
    rot = (e - 2 * (e @ w[:, :, None] @ w[:, None, :])
           + 2 * (e @ u[:, :, None].detach() @ q[:, None, :].detach())).squeeze(1)
    return rot * (nc / nx.clamp(min=1e-6)).detach()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_rotation.jsonl"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--parts", default="a,b,c,d")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rotation.py needs a CUDA device")
    from vqb200 import CodebookParams, ResidualVQ, VectorQuantize, ops
    meta = card()
    parts = set(args.parts.split(","))
    N, d, K = 1 << 20, 256, 8192
    gen = torch.Generator(device=DEV).manual_seed(0)

    if "a" in parts:
        cb = torch.randn(1, K, d, generator=gen, device=DEV) * 0.5
        idx = torch.randint(0, K, (1, N), generator=gen, device=DEV)
        gl = torch.full((1,), 2.0 / (N * d), device=DEV)
        for dt in (torch.float32, torch.bfloat16):
            xs = [torch.randn(1, N, d, generator=gen, device=DEV).to(dt) for _ in range(2)]
            gqs = [torch.randn(1, N, d, generator=gen, device=DEV) for _ in range(2)]
            arms = {"st_commit_backward": lambda i: ops.st_commit_backward(gqs[i % 2], gl, xs[i % 2], cb, idx, None),
                    "rot_commit_backward": lambda i: ops.rot_commit_backward(gqs[i % 2], gl, xs[i % 2], cb, idx, None)}
            res = alternate(arms, args.iters * 2, args.rounds)
            nbytes = N * (xs[0].element_size() * d + 4 * d + 8 + 4 * d)
            for k, v in res.items():
                emit(args.out, {"part": "a", "kernel": k, "x_dtype": str(dt).split(".")[-1], "N": N, "d": d, "K": K,
                                "ms": v["ms"], "ms_all": v["ms_all"], "algorithmic_bytes": nbytes,
                                "gbs": nbytes / (v["ms"] / 1e3) / 1e9, "code_rows_counted": False,
                                "inputs": "2 rotating buffers of x and grad_q, each larger than L2"}, meta)
            emit(args.out, {"part": "a", "ratio_rot_over_st": res["rot_commit_backward"]["ms"]
                            / res["st_commit_backward"]["ms"], "x_dtype": str(dt).split(".")[-1]}, meta)
            del xs, gqs
        del cb, idx
        torch.cuda.empty_cache()

    if "b" in parts:
        mods = {}
        for rot in (False, True):
            torch.manual_seed(0)
            vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K,
                                                                      threshold_ema_dead_code=0)).to(DEV).train()
            vq.rotation_trick = rot
            c = torch.randn(1, K, d, generator=torch.Generator().manual_seed(0)) * 0.5
            cbk = vq._codebook
            cbk.embeddings.copy_(c); cbk.embed_avg.copy_(c); cbk.cluster_size.fill_(1.0); cbk.invalidate_cache()
            mods[rot] = vq
        x = torch.randn(1, N, d, generator=gen, device=DEV).requires_grad_(True)
        gq = torch.randn(1, N, d, generator=gen, device=DEV)

        def step(vq):
            def f(i):
                x.grad = None
                q, _, loss = vq(x)
                torch.autograd.backward([q, loss], [gq, torch.ones_like(loss)])
            return f
        res = alternate({"straight_through": step(mods[False]), "rotation": step(mods[True])}, args.iters, args.rounds)
        for k, v in res.items():
            emit(args.out, {"part": "b", "workload": "C2 VectorQuantize forward + backward, fp32 x (1, 2^20, 256), "
                            "K=8192", "estimator": k, "ms_per_step": v["ms"], "ms_all": v["ms_all"]}, meta)
        emit(args.out, {"part": "b", "ratio_rot_over_st": res["rotation"]["ms"] / res["straight_through"]["ms"]}, meta)
        del mods, x, gq
        torch.cuda.empty_cache()

    if "c" in parts:
        Q, Kr, dr = 8, 1024, 512
        xs = [torch.randn(64, 4096, dr, generator=gen, device=DEV).requires_grad_(True) for _ in range(2)]

        def make(rot, fused):
            torch.manual_seed(0)
            rvq = ResidualVQ(dim=dr, num_quantizers=Q, rotation_trick=rot,
                             codebook_params=CodebookParams(dim=dr, codebook_size=Kr)).to(DEV).train()
            g = torch.Generator().manual_seed(0)
            for li, layer in enumerate(rvq.layers):
                c = (torch.randn(1, Kr, dr, generator=g) * (0.5 / 1.4 ** li)).to(DEV)
                cbk = layer._codebook
                cbk.embeddings.copy_(c); cbk.embed_avg.copy_(c); cbk.cluster_size.fill_(8.0); cbk.invalidate_cache()
            rvq.use_fused_levels = fused

            def f(i):
                x = xs[i % 2]
                x.grad = None
                q, _, loss = rvq(x)
                (q.sum() * 1e-6 + loss.sum()).backward()
            return f
        arms = {"fused_rotation": make(True, True), "fused_straight_through": make(False, True),
                "generic_rotation": make(True, False)}
        res = alternate(arms, max(2, args.iters // 2), args.rounds)
        for k, v in res.items():
            emit(args.out, {"part": "c", "workload": "C4 ResidualVQ 8 x K=1024 x d=512, 64 x 4096 fp32 latents, "
                            "forward + backward", "arm": k, "ms_per_step": v["ms"], "ms_all": v["ms_all"]}, meta)
        emit(args.out, {"part": "c", "ratio_fused_rot_over_fused_st": res["fused_rotation"]["ms"]
                        / res["fused_straight_through"]["ms"]}, meta)
        del arms, xs
        torch.cuda.empty_cache()

    if "d" in parts:
        cb = torch.randn(K, d, generator=gen, device=DEV) * 0.5
        idx = torch.randint(0, K, (N,), generator=gen, device=DEV)
        x = torch.randn(N, d, generator=gen, device=DEV).requires_grad_(True)
        gq = torch.randn(N, d, generator=gen, device=DEV)
        c = cb[idx]

        def torch_rot(i):
            x.grad = None
            rotate_to(x, c).backward(gq)
        res = alternate({"torch_rotate_to": torch_rot}, args.iters, args.rounds)
        emit(args.out, {"part": "d", "what": "upstream rotate_to in torch, autograd forward + backward, fp32 "
                        "(2^20, 256), codes gathered beforehand", "ms": res["torch_rotate_to"]["ms"],
                        "ms_all": res["torch_rotate_to"]["ms_all"]}, meta)


if __name__ == "__main__":
    main()
