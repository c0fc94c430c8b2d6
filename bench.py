#!/usr/bin/env python
"""bench.py -- VQ lookups/s on BASELINE.json's headline workload, plus the other named shapes.

A "step" is one pass of the codebook hot path over one batch of synthetic latents: the training-mode
`VectorQuantize.forward` = nearest-code search + gather/straight-through/commitment loss + EMA statistics,
codebook refresh and dead-code check.  Headline workload (configs[1] of BASELINE.json, "C2"): 1,048,576 latents x
d=256, codebook K=8192, bf16 latents, Euclidean, EMA decay 0.8; config 2 is "search+EMA" (dead-code expiry belongs to
config 3), so threshold_ema_dead_code=0 there -- stated in the JSON line -- in both arms.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs C3,C4,C5|none]
                    [--dump-outputs DIR]

N>1 is launched by the driver through torch.distributed.run (one rank per GPU, NCCL): data parallel, every rank
quantises its own 1M latents ("weak" scaling) and the EMA statistics are summed with one packed all_reduce.
The same JSON line carries a `configs` block with the other named shapes at the same N (north star: "throughput on
synthetic latents of each named shape is reported at 1, 2, 4 and 8 GPUs"):
  C3  cosine codebook, 512K x d=512, K=16384, EMA + dead-code expiry, data parallel (weak)
  C4  ResidualVQ 8 x K=1024 x d=512 on 64 x 4096 latents, data-parallel EMA all_reduce per level: weak (64 sequences
      per rank) and strong (the 64 sequences split over the ranks)
  C5  K=65536 x d=64, 4M latents replicated on every rank, codebook rows sharded over the N ranks with the cross-GPU
      (score, index) min-reduction (N=1: the whole codebook on one GPU)
`--impl reference` times the UNMODIFIED reference (baseline/_ref, installed by baseline/install_ref.sh) on the host
CPU on a bounded sample of the headline workload, on rank 0 only; if baseline/_ref is missing it falls back to the
oracle port (oracle/ restates the reference op for op) and says so in `cpu_baseline.kind`.
`--dump-outputs DIR` writes what the last timed step of the headline computed (rank 0) as .npy files, so that two
builds can be compared output for output on identical seeded inputs: see dump_outputs().
Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vector-quantization-by-ml_b200"))

import torch  # noqa: E402

N_ROWS, K_CODES, DIM = 1 << 20, 8192, 256
SHAPE = (1024, 1024, DIM)               # (batch, tokens, d) -> N = 2^20 latents
CPU_SAMPLE_ROWS = 16384                 # bounded sample for the CPU legs (N x K fp32 must fit the host)
WORKLOAD = "C2: EuclideanCodebook search+EMA, N=1048576 latents x d=256, K=8192, bf16 latents"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
DUMP_QUANTIZE_ROWS = 16384              # --dump-outputs: seeded sample of the 2^20 quantize rows (16 MiB of 1 GiB)


def dump_outputs(path, out, cb):
    """Writes one headline step's results to `path` as .npy: quantize (a fixed seeded sample of its rows, fp32),
    indices and loss (fp64, exact), and the codebook state the step's EMA update left (embeddings, embed_avg,
    cluster_size, fp32).  About 40 MB in all."""
    import numpy as np
    q, ind, loss = out
    rows = torch.randperm(N_ROWS, generator=torch.Generator().manual_seed(0))[:DUMP_QUANTIZE_ROWS].sort().values
    arrays = {"quantize": q.reshape(N_ROWS, DIM)[rows.to(q.device)].float(), "indices": ind.double(),
              "loss": loss.double(), "embeddings": cb.embeddings.float(), "embed_avg": cb.embed_avg.float(),
              "cluster_size": cb.cluster_size.float()}
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().cpu().numpy())


def ncu_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum of one search-kernel launch, from the committed ncu --set full
    capture of this same command (profiles/rNN_ncu_summary.json); None if there is no capture."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_summary.json")))
    if not files:
        return None
    try:
        for k in json.load(open(files[-1]))["ncu_full"]:
            if "search_aug_kernel" in k["kernel"] or "search_tc_kernel" in k["kernel"]:
                return (k["dram_rd_MB"] + k["dram_wr_MB"]) * 1e6
    except Exception:
        return None
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"tflops": float(p["bf16_tflops"]), "tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "hbm_gbs": float(p["hbm_gbs"]), "source": "measured"}
    return {"tflops": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe's clocks line)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        import datetime
        for line in self.proc.stdout:
            line = line.strip()
            t = time.time()
            try:    # nvidia-smi's own timestamp (local time, ms): immune to pipe buffering
                t = datetime.datetime.strptime(line.split(",")[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                pass
            self.rows.append((t, line))

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples taken in [t_begin, t_end] (host clock around the timed region, which ends with a
        device sync).  nvidia-smi needs ~0.2 s to deliver its first line, so the sampler is started before the
        warm-up; if the window is shorter than the sampling period the samples nearest to it (all under the same
        load: the warm-up runs the same step) are used."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        rows = self.rows
        if t_begin is not None:
            inside = [r for (t, r) in rows if t_begin <= t <= t_end + 0.03]
            if len(inside) < 3:
                mid = 0.5 * (t_begin + t_end)
                inside = [r for (_, r) in sorted(rows, key=lambda tr: abs(tr[0] - mid))[:5]]
        else:
            inside = [r for (_, r) in rows]
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU legs: the live reference (baseline/_ref) or, without it, the oracle port
# ------------------------------------------------------------------------------------------------------------------
def reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "vector_quantization"))


def cpu_reference_step(rows, threads):
    """One training forward of the UNMODIFIED reference's VectorQuantize on `rows` latents of the headline workload
    (its own public API and stock code path; `einx`, absent from the image, is only imported by residual_vq.py and
    never called on this path: baseline/einx_standin)."""
    for p in (os.path.join(ROOT, "baseline", "einx_standin"), REF_DIR):
        if p not in sys.path:
            sys.path.insert(0, p)
    from vector_quantization import VectorQuantize as RefVQ
    from vector_quantization.codebooks import CodebookParams as RefParams
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    c = torch.randn(1, K_CODES, DIM, generator=g) * 0.5
    vq = RefVQ(dim=DIM, codebook_params=RefParams(dim=DIM, codebook_size=K_CODES, threshold_ema_dead_code=0),
               sync_codebook=False).train()
    with torch.no_grad():
        vq._codebook.embeddings.copy_(c); vq._codebook.embed_avg.copy_(c); vq._codebook.cluster_size.fill_(1.0)
    x = torch.randn(1, rows, DIM, generator=g).bfloat16()

    def step():
        with torch.no_grad():
            vq(x)
    return step


def cpu_port_step(rows, threads):
    """One training forward of the reference path (oracle port) on `rows` latents of the workload, on the CPU."""
    from oracle import vq_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    c = torch.randn(1, K_CODES, DIM, generator=g) * 0.5
    st = O.CodebookState(c.clone(), c.clone(), torch.ones(1, K_CODES))
    x = torch.randn(1, rows, DIM, generator=g).bfloat16()
    opts = O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=0))

    def step():
        O.vq_forward(st, x, opts, training=True)
    return step


def cpu_step(rows, threads):
    if reference_available():
        return cpu_reference_step(rows, threads), "reference"
    return cpu_port_step(rows, threads), "port"


def time_cpu_leg(budget_s, threads, rows=CPU_SAMPLE_ROWS, warmup=1, max_steps=None):
    step, kind = cpu_step(rows, threads)
    for _ in range(warmup):
        step()
    times = []
    t_end = time.time() + budget_s
    while (time.time() < t_end and (max_steps is None or len(times) < max_steps)) or not times:
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    return rows / (sum(times) / len(times)), len(times), kind


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rows = CPU_SAMPLE_ROWS
    step, kind = cpu_step(rows, threads)
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = rows / dt
    what = ("the unmodified reference VectorQuantize (baseline/_ref) on CPU tensors" if kind == "reference"
            else "the oracle port (baseline/_ref not installed)")
    sample = (f"{what}: {rows} of {N_ROWS} latents per step (the reference materialises N x K fp32/int64: the full "
              f"batch needs >=160 GiB), K={K_CODES}, d={DIM}, all host threads")
    out = {"impl": "reference", "metric": "vq_lookups_per_sec", "value": val, "unit": "lookups/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": WORKLOAD, "sample": sample},
           "cpu_baseline": {"value": val, "unit": "lookups/s", "cores": threads, "kind": kind, "sample": sample},
           "e2e": {"value": val, "unit": "lookups/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# helpers of the GPU arm
# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(local_rank):
    """Pin this process (and therefore its pinned host buffers, first touch) to the NUMA node of its GPU: eight ranks
    copying 0.5-1 GiB per step through one socket's memory controllers is what flattened `e2e` at 4 GPUs in round 1.
    Best effort (containers often hide the topology); returns what was done and the original affinity."""
    info = {"numa_node": None, "bound": False, "orig_affinity": None}
    try:
        info["orig_affinity"] = os.sched_getaffinity(0)
        bdf = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        ids = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= info["orig_affinity"]
        if ids:
            os.sched_setaffinity(0, ids)
            info["bound"], info["cpus"] = True, len(ids)
    except Exception as e:
        info["why"] = str(e)[:80]
    return info


class Ctx:
    def __init__(self, rank, local_rank, world, dev):
        self.rank, self.local_rank, self.world, self.dev = rank, local_rank, world, dev

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        t = torch.tensor(vals, device=self.dev, dtype=torch.float64)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]


def timed_loop(ctx, step, steps, warmup, time_kernels=True):
    """W untimed steps, then exactly `steps` steps between barrier + synchronize, CUDA events; max over ranks.
    Returns (ms_total, launches, search_kernel_ms list)."""
    from vqb200 import ops
    for i in range(warmup):
        step(i)
    ctx.barrier()
    ops.TIME_SEARCH_KERNEL = bool(time_kernels)
    ops.search_kernel_times_ms()
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_count() - l0
    tc = ops.search_kernel_times_ms()
    ops.TIME_SEARCH_KERNEL = False
    (ms,) = ctx.max_over_ranks([ms])
    return ms, launches, tc


def free_all():
    from vqb200 import ops
    import gc
    gc.collect()
    ops.release_workspaces()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------
# the other named shapes (the `configs` block)
# ------------------------------------------------------------------------------------------------------------------
def bench_c3(ctx, steps, warmup, pk):
    from vqb200 import CodebookParams, VectorQuantize
    K, d, shape = 16384, 512, (512, 1024, 512)
    N = shape[0] * shape[1]
    torch.manual_seed(0)
    vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=2,
                                                              use_cosine_sim=True, transform_input="l2norm",
                                                              weights_regularization="l2norm"),
                        sync_codebook=ctx.world > 1).to(ctx.dev).train()
    g = torch.Generator().manual_seed(0)
    c = torch.nn.functional.normalize(torch.randn(1, K, d, generator=g), dim=-1).to(ctx.dev)
    cb = vq._codebook
    cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0); cb.invalidate_cache()
    gx = torch.Generator(device=ctx.dev).manual_seed(1234 + ctx.rank)
    xs = [torch.randn(shape, generator=gx, device=ctx.dev) for _ in range(2)]       # 1 GiB each

    def step(i):
        with torch.no_grad():
            return vq(xs[i % 2])
    ms, launches, tc = timed_loop(ctx, step, steps, warmup)
    tc_avg = sum(tc) / max(len(tc), 1)
    flops = 2.0 * N * K * d
    out = {"workload": "C3: cosine codebook (l2norm in / weights), 524288 x d=512 fp32, K=16384, EMA + dead-code expiry "
                       "(threshold 2), data parallel", "scaling": "weak", "rows_per_gpu": N,
           "ms_per_step": ms / steps, "lookups_per_s": N * ctx.world * steps / (ms / 1e3), "steps": steps,
           "search_kernel_ms": tc_avg, "search_tflops": flops / (tc_avg / 1e3) / 1e12 if tc_avg else None,
           "search_frac_of_tensor_peak": flops / (tc_avg / 1e3) / 1e12 / pk["tflops"] if tc_avg else None,
           "gpu_launches_per_step": launches / steps}
    del vq, xs
    free_all()
    return out


def bench_c4(ctx, steps, warmup, pk, strong):
    from vqb200 import CodebookParams, ResidualVQ
    Q, K, d = 8, 1024, 512
    seqs = 64 // ctx.world if strong else 64
    if seqs == 0:
        return None
    shape = (seqs, 4096, d)
    N = seqs * 4096
    torch.manual_seed(0)
    rvq = ResidualVQ(dim=d, num_quantizers=Q, codebook_params=CodebookParams(dim=d, codebook_size=K),
                     sync_codebook=ctx.world > 1).to(ctx.dev).train()
    g = torch.Generator().manual_seed(0)
    for li, layer in enumerate(rvq.layers):
        c = (torch.randn(1, K, d, generator=g) * (0.5 / 1.4 ** li)).to(ctx.dev)
        cb = layer._codebook
        cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(8.0); cb.invalidate_cache()
    gx = torch.Generator(device=ctx.dev).manual_seed(1234 + ctx.rank)
    xs = [torch.randn(shape, generator=gx, device=ctx.dev) for _ in range(2)]

    def step(i):
        with torch.no_grad():
            return rvq(xs[i % 2])
    # eager loop first: per-level search-kernel time (event brackets cannot be captured) and the launch count
    ms_eager, launches, tc = timed_loop(ctx, step, max(2, min(steps, 4)), 2)
    eager_steps = max(2, min(steps, 4))
    # the timed number: the 8-level loop replayed as one CUDA graph per input buffer (ResidualVQ.enable_cuda_graph);
    # warm-up covers the eager pass and the capture of both rotating buffers
    rvq.enable_cuda_graph(data_parallel=True)   # every rank runs this same sequence of forwards
    ms, _, _ = timed_loop(ctx, step, steps, max(warmup, 4) + 2, time_kernels=False)
    launches = launches * steps / eager_steps
    per_level = sum(tc) / max(len(tc), 1)
    # the same step with a gradient to the input (an encoder trained through the quantiser): fused loop forward + ONE
    # replay pass backward (vqb_rvq_backward)
    xg = [t.clone().requires_grad_(True) for t in xs]

    def grad_step(i):
        x = xg[i % 2]
        x.grad = None
        q, _, loss = rvq(x)
        (q.sum() * 1e-6 + loss.sum()).backward()
    ms_grad, _, _ = timed_loop(ctx, grad_step, max(2, min(steps, 5)), 2, time_kernels=False)
    grad_steps = max(2, min(steps, 5))
    del xg
    flops = 2.0 * N * K * d
    total_rows = N * ctx.world
    out = {"workload": f"C4: ResidualVQ 8 x K=1024 x d=512, {'64 sequences split over the ranks' if strong else '64 sequences per rank'}"
                       " x 4096 latents fp32, EMA (default threshold 2) with one packed statistics all_reduce per level",
           "scaling": "strong" if strong else "weak", "rows_per_gpu": N, "ms_per_step": ms / steps,
           "tokens_per_s": total_rows * steps / (ms / 1e3), "lookups_per_s": total_rows * Q * steps / (ms / 1e3),
           "steps": steps, "search_kernel_ms_per_level": per_level,
           "search_frac_of_tensor_peak": flops / (per_level / 1e3) / 1e12 / pk["tflops"] if per_level else None,
           "search_kernels_share_of_step": per_level * Q / (ms / steps) if per_level else None,
           "gpu_launches_per_step": launches / steps, "cuda_graph": True,
           "eager_ms_per_step": ms_eager / eager_steps, "autograd_ms_per_step": ms_grad / grad_steps,
           "note": "ms_per_step: no-grad forward replayed as one CUDA graph (under data parallelism the graph holds the "
                   "per-level statistics all_reduce, launched beside the next level's search); "
                   "autograd_ms_per_step: forward with requires_grad + backward"}
    del rvq, xs
    free_all()
    return out


def bench_c5(ctx, steps, warmup, pk):
    from vqb200 import CodebookParams, VectorQuantize
    K, d, shape = 65536, 64, (4096, 1024, 64)
    N = shape[0] * shape[1]
    torch.manual_seed(0)
    vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0),
                        sync_codebook=ctx.world > 1).to(ctx.dev).train()
    cb = vq._codebook
    g = torch.Generator().manual_seed(0)
    full = torch.randn(1, K, d, generator=g) * 0.5
    cb.load_full_codebook(full)
    cb.sharded_input = "replicated"
    gx = torch.Generator(device=ctx.dev).manual_seed(4321)                   # the SAME latents on every rank
    xs = [torch.randn(shape, generator=gx, device=ctx.dev) for _ in range(2)]

    def step(i):
        with torch.no_grad():
            return vq(xs[i % 2])
    ms, launches, tc = timed_loop(ctx, step, steps, warmup)
    tc_avg = sum(tc) / max(len(tc), 1)
    flops = 2.0 * N * (K // (ctx.world if cb.sharded else 1)) * d
    out = {"workload": "C5: K=65536 x d=64, 4194304 latents fp32 replicated on every rank, codebook rows sharded over "
                       "the ranks, cross-GPU (score, index) min-reduction, EMA on the owned rows",
           "scaling": "strong", "sharded": bool(cb.sharded), "codes_per_gpu": K // (ctx.world if cb.sharded else 1),
           "ms_per_step": ms / steps, "lookups_per_s": N * steps / (ms / 1e3), "steps": steps,
           "search_kernel_ms": tc_avg,
           "search_frac_of_tensor_peak": flops / (tc_avg / 1e3) / 1e12 / pk["tflops"] if tc_avg else None,
           "search_kernel_share_of_step": tc_avg / (ms / steps) if tc_avg else None,
           "gpu_launches_per_step": launches / steps}
    del vq, xs
    free_all()
    return out


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--configs", default="C3,C4,C5", help="other named shapes to time after the headline ('none' to skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed headline step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from vqb200 import CodebookParams, VectorQuantize, ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU implementation")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx = Ctx(rank, local_rank, world, dev)
    pk = peaks()
    warmup = max(args.warmup, 3)

    # ---- module + synthetic data (seeds: module 0 on every rank, latents 1234 + rank) ----
    torch.manual_seed(0)
    vq = VectorQuantize(dim=DIM, codebook_params=CodebookParams(dim=DIM, codebook_size=K_CODES,
                                                                threshold_ema_dead_code=0),
                        sync_codebook=world > 1).to(dev)
    g = torch.Generator().manual_seed(0)
    c = (torch.randn(1, K_CODES, DIM, generator=g) * 0.5).to(dev)      # trained-like codebook (SURVEY 8d)
    cb = vq._codebook
    cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0)
    cb.invalidate_cache()
    vq.train()
    gx = torch.Generator(device=dev).manual_seed(1234 + rank)
    n_bufs = 2                                                          # 512 MiB each, > 126 MB L2: never L2-hot
    xs = [torch.randn(SHAPE, generator=gx, device=dev, dtype=torch.float32).bfloat16() for _ in range(n_bufs)]
    keep_last = args.dump_outputs is not None and rank == 0
    last = []                             # --dump-outputs: the outputs of the latest step

    def step(i):
        last.clear()                      # the previous outputs are freed before the next step, as without the flag
        with torch.no_grad():
            out = vq(xs[i % n_bufs])
        if keep_last:
            last.append(out)
        return out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                   # nvidia-smi is streaming by the time the warm-up starts
    t_warm = time.time()                  # the warm-up runs the same step: its samples are under the same load
    # ---- timed region: device-resident inputs ----
    ms, launches, tc_ms = timed_loop(ctx, step, args.steps, warmup)
    t_end = time.time()
    clocks = sampler.stop(t_warm, t_end) if rank == 0 else None
    stats = ops.search_stats(cb.last_search_ws)
    if keep_last:
        dump_outputs(args.dump_outputs, last[0], cb)
        last.clear()

    # ---- the bandwidth-bound part of the step on its own: gather + straight-through + loss + EMA sums in one pass over
    #      the latents (counting sort included), against its ALGORITHMIC bytes (DESIGN 4.2: sz(x) d + 12 read,
    #      4 d + 4 write per row) and the measured HBM copy peak ----
    with torch.no_grad():
        flat = xs[0].reshape(1, -1, DIM)
        idx_b, _, ws_b = ops.search(flat, cb.embeddings, cb._codebook_cache(), False)
        for _ in range(3):
            ops.quantize_ema(flat, cb.embeddings, idx_b, True, True, bound_ws=ws_b)
        eb0, eb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        eb0.record()
        for i in range(10):
            ops.quantize_ema(xs[i % n_bufs].reshape(1, -1, DIM), cb.embeddings, idx_b, True, True, bound_ws=ws_b)
        eb1.record()
        torch.cuda.synchronize()
    gather_ms = eb0.elapsed_time(eb1) / 10
    gather_bytes = N_ROWS * (2 * DIM + 12 + 4 * DIM + 4)
    hbm = {"kernel": "vqb_quantize_ema: counting sort + quantize_ema_kernel + finalize (gather, straight-through, "
                     "commitment loss and EMA sums in one pass)",
           "ms": gather_ms, "algorithmic_bytes": gather_bytes, "achieved_gbs": gather_bytes / (gather_ms / 1e3) / 1e9,
           "peak_gbs": pk["hbm_gbs"], "frac": gather_bytes / (gather_ms / 1e3) / 1e9 / pk["hbm_gbs"]}
    del idx_b, flat

    # ---- the step a training loop takes: input requires grad, forward + backward (codebook snapshot, _QuantizeST,
    #      vqb_st_commit_backward); fp32 latents (the reference's own backward rejects bf16 inputs) ----
    x_grad = xs[0].float().requires_grad_(True)
    gq = torch.randn(SHAPE, device=dev, dtype=torch.float32)

    def autograd_step(i):
        x_grad.grad = None
        q, _, loss = vq(x_grad)
        torch.autograd.backward([q, loss], [gq, torch.ones_like(loss)])
    ag_steps = max(3, min(args.steps, 10))
    ag_ms, ag_launches, _ = timed_loop(ctx, autograd_step, ag_steps, 3)
    del x_grad, gq
    torch.cuda.empty_cache()

    # ---- e2e: host buffers in, EVERY output (quantize fp32, indices, loss) back to host, copies inside the timed
    # region.  H2D, kernels and D2H run on three streams, double buffered, so the copy of step i+1's latents and the
    # read-back of step i-1's outputs overlap step i's kernels (PCIe is full duplex); nothing is cached between steps.
    x_host = torch.empty(SHAPE, dtype=torch.bfloat16).pin_memory()
    x_host.copy_(xs[0])
    q_host = [torch.empty(SHAPE, dtype=torch.float32).pin_memory() for _ in range(2)]
    idx_host = [torch.empty(SHAPE[:2], dtype=torch.int64).pin_memory() for _ in range(2)]
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    h2d_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)
    dbuf = [torch.empty(SHAPE, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    drained = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        with torch.cuda.stream(h2d_stream):
            h2d_stream.wait_event(consumed[i % 2])
            dbuf[i % 2].copy_(x_host, non_blocking=True)
            ready[i % 2].record(h2d_stream)

    def e2e_loop(n, with_quantize):
        outs = [None, None]
        for b in range(2):
            consumed[b].record(main_stream)
            drained[b].record(d2h_stream)
        prefetch(0)
        for i in range(n):
            if i + 1 < n:
                prefetch(i + 1)
            main_stream.wait_event(ready[i % 2])
            main_stream.wait_event(drained[i % 2])         # the outputs of step i-2 have left the device
            with torch.no_grad():
                q, ind, loss = vq(dbuf[i % 2])
            consumed[i % 2].record(main_stream)
            done = torch.cuda.Event()
            done.record(main_stream)
            outs[i % 2] = (q, ind, loss)                   # keep the tensors alive until their copy has run
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                if with_quantize:
                    q_host[i % 2].copy_(q, non_blocking=True)
                idx_host[i % 2].copy_(ind, non_blocking=True)
                loss_host[i % 2].copy_(loss, non_blocking=True)
                drained[i % 2].record(d2h_stream)
        main_stream.wait_stream(d2h_stream)

    e2e_steps = max(3, min(args.steps, 10))

    def time_e2e(with_quantize):
        e2e_loop(2, with_quantize)
        ctx.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        e2e_loop(e2e_steps, with_quantize)
        f1.record()
        ctx.barrier()
        return f0.elapsed_time(f1)
    e2e_ms = time_e2e(True)
    e2e_idx_ms = time_e2e(False)

    # bare copies, all ranks at once: what the host side can deliver to / take from this many GPUs
    def bare(fn, reps):
        fn()
        ctx.barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(reps):
            fn()
        b1.record()
        ctx.barrier()
        return b0.elapsed_time(b1) / reps
    q_dev = torch.empty(SHAPE, dtype=torch.float32, device=dev)
    h2d_ms = bare(lambda: dbuf[0].copy_(x_host, non_blocking=True), 5)
    d2h_ms = bare(lambda: q_host[0].copy_(q_dev, non_blocking=True), 3)
    del q_dev
    ag_ms_, e2e_ms, e2e_idx_ms, h2d_ms, d2h_ms = ctx.max_over_ranks([ag_ms, e2e_ms, e2e_idx_ms, h2d_ms, d2h_ms])
    del xs, dbuf, q_host, idx_host
    free_all()

    # ---- the other named shapes, same N ----
    configs = {}
    want = [] if args.configs.lower() == "none" else [s.strip().upper() for s in args.configs.split(",") if s.strip()]
    cfg_steps = max(3, min(args.steps, 10))
    if "C3" in want:
        configs["C3"] = bench_c3(ctx, cfg_steps, 3, pk)
    if "C4" in want:
        configs["C4_weak"] = bench_c4(ctx, cfg_steps, 3, pk, strong=False)
        if world > 1:
            configs["C4_strong"] = bench_c4(ctx, cfg_steps, 3, pk, strong=True)
    if "C5" in want:
        configs["C5"] = bench_c5(ctx, max(3, min(args.steps, 5)), 2, pk)

    if rank == 0:
        total_rows = N_ROWS * world
        value = total_rows * args.steps / (ms / 1e3)
        e2e_val = total_rows * e2e_steps / (e2e_ms / 1e3)
        flops = 2.0 * N_ROWS * K_CODES * DIM                     # algorithmic flops per launch of the search kernel
        tc_avg = sum(tc_ms) / len(tc_ms) if tc_ms else float("nan")
        achieved = flops / (tc_avg / 1e3) / 1e12
        roofline = {"kernel": "search_aug_kernel (tcgen05 GEMM, bias as an extra MMA k-step, fused packed top-k epilogue)", "bound": "tensor",
                    "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"],
                    "peak_source": pk["source"] + " bf16 burst (cuBLAS 8192^3); sustained %.1f" % pk["tflops_sustained"],
                    "frac_of_sustained": achieved / pk["tflops_sustained"],
                    "kernel_ms": tc_avg, "kernel_share_of_step": tc_avg / (ms / args.steps),
                    "algorithmic_flops_per_launch": flops, "traffic": ncu_traffic_bytes(),
                    "traffic_unit": "bytes of DRAM read+write per launch (ncu --set full, profiles/)"}
        if numa.get("orig_affinity"):
            try:
                os.sched_setaffinity(0, numa["orig_affinity"])          # the CPU leg may use every host core again
            except Exception:
                pass
        threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        cpu_val, cpu_n, cpu_kind = time_cpu_leg(args.cpu_seconds, threads)
        sample = (f"{CPU_SAMPLE_ROWS} of {N_ROWS} latents per step x {cpu_n} steps (the reference materialises N x K: "
                  f"the full batch needs >=160 GiB), K={K_CODES}, d={DIM}; "
                  + ("the unmodified reference (baseline/_ref)" if cpu_kind == "reference" else "oracle port"))
        h2d_b, d2h_b = x_host.numel() * 2, SHAPE[0] * SHAPE[1] * (DIM * 4 + 8) + 4
        out = {"metric": "vq_lookups_per_sec", "value": value, "unit": "lookups/s", "n_gpus": world,
               "steps": args.steps, "warmup": warmup, "ms_per_step": ms / args.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
               "data": "synthetic",
               "config": {"workload": WORKLOAD, "step": "VectorQuantize training forward: search + gather/ST/commit loss "
                          "+ EMA reduce/refresh (config 2 = search+EMA: threshold_ema_dead_code=0; expiry is measured "
                          "with config 3 in the `configs` block)", "rows_per_gpu": N_ROWS, "codebook_size": K_CODES,
                          "dim": DIM, "latent_dtype": "bf16", "parallelism": f"dp{world}",
                          "l2": "inputs (512 MiB per batch, 2 rotating buffers) exceed the 126 MB L2; no flush",
                          "search": stats,
                          "numa": {k: v for k, v in numa.items() if k != "orig_affinity"}},
               "roofline": roofline,
               "cpu_baseline": {"value": cpu_val, "unit": "lookups/s", "cores": threads, "kind": cpu_kind, "sample": sample},
               "e2e": {"value": e2e_val, "unit": "lookups/s", "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                       "h2d_bytes_per_step": h2d_b * world, "d2h_bytes_per_step": d2h_b * world,
                       "outputs": "quantize fp32 (1 GiB) + indices int64 + loss, all to pinned host memory",
                       "indices_only_value": total_rows * e2e_steps / (e2e_idx_ms / 1e3),
                       "indices_only_note": "same loop with quantize left on the device (round-1 definition)",
                       "bare_h2d_gbs_per_rank": h2d_b / (h2d_ms / 1e3) / 1e9,
                       "bare_d2h_gbs_per_rank": SHAPE[0] * SHAPE[1] * DIM * 4 / (d2h_ms / 1e3) / 1e9,
                       "host_bound_ms_per_step": max(h2d_ms, d2h_ms * d2h_b / (SHAPE[0] * SHAPE[1] * DIM * 4)),
                       "note": "pinned host latents -> device, forward, every output -> pinned host; three streams, "
                               "double buffered; bare_* = the same copies alone, all ranks at once (the host-side limit)"},
               "autograd_step": {"ms_per_step": ag_ms_ / ag_steps, "lookups_per_s": total_rows * ag_steps / (ag_ms_ / 1e3),
                                 "what": "fp32 latents with requires_grad: forward (search, codebook snapshot, fused "
                                         "gather/ST/loss+EMA) + backward (vqb_st_commit_backward)",
                                 "gpu_launches_per_step": ag_launches / ag_steps},
               "roofline_hbm": hbm,
               "configs": configs,
               "gpu_launches": int(launches), "clocks": clocks}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
