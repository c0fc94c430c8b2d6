"""Multi-GPU parity check, launched as: torchrun --nproc-per-node W --master-addr 127.0.0.1 tools/mgpu_check.py
 1. data parallel: W ranks, each quantising its slice, end up with the codebook a single process gets on the
    concatenated batch (cluster_size exact, embeddings/embed_avg 1e-6), identical on every rank, incl. expiry.
 1c. the same data-parallel step against the CPU ORACLE on the rank-concatenated batch.
 2. sharded codebook through the module API (Codebook.sharded; replicated and all_gather inputs) against the CPU
    ORACLE on the un-sharded codebook: indices, bit-exact quantize, every shard's EMA + dead-code expiry result equals
    the matching rows of the reference update, state_dict holds the full tensors.
 3. sharded codebook at the real threshold (K = 65536, SHARD_MIN_CODES unchanged), masked bf16 input with expiry,
    against the ORACLE; the input gradient of a training step equals an un-sharded VectorQuantize's.
 4. ResidualVQ over sharded codebooks (generic level loop) against the ORACLE's rvq_forward, return_all_codes and
    get_output_from_indices; the input gradient equals an un-sharded ResidualVQ's.
 5. accessors of a sharded codebook: full (K, d) codebooks, the setter keeps this rank's rows, an in-place edit plus
    invalidate_cache() reaches the next eval forward.
Prints 'MGPU OK' from rank 0 on success.

VQB_MGPU_SINGLE_DEVICE=1 runs every rank on cuda:0 over Gloo (a machine with one GPU).  Section 1d is skipped there:
it captures NCCL collectives in a CUDA graph.  In that mode every collective is staged through host memory by this
script (the wrappers below), so the check does not depend on which collectives Gloo accepts for CUDA tensors; the
product code is unchanged and issues the same collectives."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "vector-quantization-by-ml_b200"))
import torch
import torch.distributed as dist

from oracle import vq_oracle as O  # noqa: E402  (test tool: the oracle is the checker)
from vqb200 import CodebookParams, KmeansParameters, VectorQuantize, distributed as D, ops

import datetime  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
SINGLE = os.environ.get("VQB_MGPU_SINGLE_DEVICE", "0") == "1"
if SINGLE:
    local = 0
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if SINGLE:
    dist.init_process_group("gloo", timeout=datetime.timedelta(seconds=180))

    class _Done:
        def wait(self):
            return True

    _real = {n: getattr(dist, n) for n in ("all_reduce", "broadcast", "all_gather_into_tensor", "all_gather")}

    def _all_reduce(t, op=dist.ReduceOp.SUM, group=None, async_op=False):
        h = t.cpu()
        _real["all_reduce"](h, op=op, group=group)
        t.copy_(h)
        return _Done() if async_op else None

    def _broadcast(t, src, group=None, async_op=False):
        h = t.cpu()
        _real["broadcast"](h, src=src, group=group)
        t.copy_(h)
        return _Done() if async_op else None

    def _all_gather_into_tensor(out, inp, group=None, async_op=False):
        h = out.cpu()
        _real["all_gather_into_tensor"](h, inp.contiguous().cpu(), group=group)
        out.copy_(h)
        return _Done() if async_op else None

    def _all_gather(outs, inp, group=None, async_op=False):
        hs = [o.cpu() for o in outs]
        _real["all_gather"](hs, inp.contiguous().cpu(), group=group)
        for o, h in zip(outs, hs):
            o.copy_(h)
        return _Done() if async_op else None

    dist.all_reduce, dist.broadcast = _all_reduce, _broadcast
    dist.all_gather_into_tensor, dist.all_gather = _all_gather_into_tensor, _all_gather
else:
    dist.init_process_group("nccl", device_id=dev)
SHARD_REAL = D.SHARD_MIN_CODES


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def check(cond, msg):
    t = torch.tensor([0 if cond else 1], device=dev)
    dist.all_reduce(t)
    if int(t.item()):
        raise SystemExit(f"[rank {rank}] FAILED: {msg}")


def untouched(cb, flips):
    """((K/W,) mask of this rank's codes that no exempt tie touched on ANY rank, whether no code was touched at all --
    the same on every rank); `flips` lists (got, oracle, differ) index tensors: a flipped row moves its statistics
    between its two codes."""
    t = torch.zeros(cb.codebook_size, dtype=torch.int32, device=dev)
    for got, ref, differ in flips:
        t[got[differ].to(dev)] = 1
        t[ref[differ].to(dev)] = 1
    dist.all_reduce(t)
    return (t == 0)[cb.shard_offset:cb.shard_offset + cb.shard_size].cpu(), not bool(t.any())


def compare_shard_buffers(cb, st, keep, what):
    """This rank's rows of the oracle's buffers: cluster_size exact, embed_avg / embeddings 1e-5, on the kept codes."""
    sl = slice(cb.shard_offset, cb.shard_offset + cb.shard_size)
    check(torch.equal(cb.cluster_size[0].cpu()[keep], st.cluster_size[0, sl][keep]), f"{what}: cluster_size")
    check(rel(cb.embed_avg[0].cpu()[keep], st.embed_avg[0, sl][keep]) < 1e-5
          and rel(cb.embeddings[0].detach().cpu()[keep], st.embeddings[0, sl][keep]) < 1e-5, f"{what}: EMA buffers / expiry")


# ---------------- 1. data parallel ----------------
K, d, n_per = 512, 64, 4096
g = torch.Generator().manual_seed(3)
x_all = torch.randn(world, n_per, d, generator=g)
c0 = torch.randn(1, K, d, generator=g) * 0.5
for thr in (0, 2):
    torch.manual_seed(0)
    dp = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=thr,
                                                              kmeans_params=KmeansParameters()), sync_codebook=True).to(dev)
    single = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0),
                            sync_codebook=False).to(dev)
    for m in (dp, single):
        cb = m._codebook
        cb.embeddings.copy_(c0); cb.embed_avg.copy_(c0); cb.cluster_size.fill_(1.0 if thr == 0 else 0.5); cb.invalidate_cache()
        m.train()
    assert dp._codebook.use_ddp
    with torch.no_grad():
        q, ind, loss = dp(x_all[rank][None].to(dev))
        qs, inds, _ = single(x_all.reshape(1, -1, d).to(dev))
    check(torch.equal(ind[0], inds[0, rank * n_per:(rank + 1) * n_per]), "DP indices differ from single-process")
    if thr == 0:
        check(torch.equal(dp._codebook.cluster_size, single._codebook.cluster_size), "DP cluster_size")
        check(rel(dp._codebook.embed_avg, single._codebook.embed_avg) < 1e-6, "DP embed_avg")
        check(rel(dp._codebook.embeddings, single._codebook.embeddings) < 1e-6, "DP embeddings")
    # replicas identical on every rank (also after dead-code replacement)
    for name in ("embeddings", "embed_avg", "cluster_size"):
        mine = getattr(dp._codebook, name).contiguous()
        ref = mine.clone()
        dist.broadcast(ref, src=0)
        check(torch.equal(mine, ref), f"replicas diverged: {name} (thr={thr})")

# ---------------- 1b. distributed_replace_codes=False (reference codebooks.py:238-239) ----------------
# every rank samples its own replacement rows and the replacements are their mean over the ranks: replicas must stay
# identical, and the replaced codes must differ from any single rank's rows (they are means of W rows)
torch.manual_seed(1 + rank)            # different local draws on every rank
dpm = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=2,
                                                           kmeans_params=KmeansParameters(),
                                                           distributed_replace_codes=False), sync_codebook=True).to(dev)
cbm = dpm._codebook
cbm.embeddings.copy_(c0); cbm.embed_avg.copy_(c0); cbm.cluster_size.fill_(0.5); cbm.invalidate_cache()
dpm.train()
with torch.no_grad():
    dpm(x_all[rank][None].to(dev))
for name in ("embeddings", "embed_avg", "cluster_size"):
    mine = getattr(cbm, name).contiguous()
    ref = mine.clone()
    dist.broadcast(ref, src=0)
    check(torch.equal(mine, ref), f"replicas diverged with distributed_replace_codes=False: {name}")

# ---------------- 1c. data parallel against the ORACLE (single process on the rank-concatenated batch) ----------------
torch.manual_seed(0)
dpo = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0),
                     sync_codebook=True).to(dev).train()
cbo = dpo._codebook
cbo.embeddings.copy_(c0); cbo.embed_avg.copy_(c0); cbo.cluster_size.fill_(1.0); cbo.invalidate_cache()
with torch.no_grad():
    qd, indd, _ = dpo(x_all[rank][None].to(dev))
sto = O.CodebookState(c0.clone(), c0.clone(), torch.ones(1, K))
qo, io, lo, exo = O.vq_forward(sto, x_all.reshape(1, -1, d), O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=0)),
                               want_gap=True)
rows = slice(rank * n_per, (rank + 1) * n_per)
diff = indd[0].cpu() != io[0, rows]
check(bool((exo["top2_rel_gap"][0, rows][diff] < 1e-6).all()), "DP indices differ from the ORACLE outside its 1e-6 window")
if not bool(diff.any()):
    check(torch.equal(qd[0].cpu(), qo[0, rows]), "DP quantize vs oracle")
    check(torch.equal(cbo.cluster_size.cpu(), sto.cluster_size), "DP cluster_size vs oracle")
    check(rel(cbo.embeddings.cpu(), sto.embeddings) < 1e-5, "DP embeddings vs oracle")

# ---------------- 1d. ResidualVQ data parallel: CUDA graph (with the captured statistics all_reduce) == eager ----------------
from vqb200 import ResidualVQ  # noqa: E402


def _make_rvq(thr):
    torch.manual_seed(0)
    m = ResidualVQ(dim=64, num_quantizers=4, codebook_params=CodebookParams(dim=64, codebook_size=96,
                                                                            threshold_ema_dead_code=thr),
                   sync_codebook=True).to(dev).train()
    gg = torch.Generator().manual_seed(3)
    for li, layer in enumerate(m.layers):
        c = (torch.randn(1, 96, 64, generator=gg) * (0.6 / 1.5 ** li)).to(dev)
        cb = layer._codebook
        cb.embeddings.copy_(c); cb.embed_avg.copy_(c); cb.cluster_size.fill_(1.0); cb.invalidate_cache()
    return m


for thr in (() if SINGLE else (0, 2)):
    eager, graphed = _make_rvq(thr), _make_rvq(thr)
    graphed.enable_cuda_graph(data_parallel=True)
    gg = torch.Generator().manual_seed(11 + rank)
    x_e = torch.empty(3, 700, 64, device=dev)
    x_g = torch.empty(3, 700, 64, device=dev)
    for step in range(5):
        xx = torch.randn(3, 700, 64, generator=gg)
        x_e.copy_(xx); x_g.copy_(xx)
        torch.manual_seed(100 + step)
        with torch.no_grad():
            qe, ie, le = eager(x_e)
        torch.manual_seed(100 + step)
        with torch.no_grad():
            qg, ig, lg = graphed(x_g)
        check(torch.equal(qe, qg) and torch.equal(ie, ig) and torch.equal(le, lg), f"RVQ DP graph step {step} thr {thr}: outputs")
        for le_, lg_ in zip(eager.layers, graphed.layers):
            for name in ("embeddings", "embed_avg", "cluster_size"):
                check(torch.equal(getattr(le_._codebook, name), getattr(lg_._codebook, name)),
                      f"RVQ DP graph step {step} thr {thr}: {name}")
    check(any(isinstance(v, tuple) for v in graphed._graphs.values()), "RVQ DP graph was never captured")
    # a captured graph holds NCCL kernels of this communicator: release it before the process group goes away
    # (destroy_process_group with such a graph alive never returned on two B200s)
    graphed.enable_cuda_graph(False)
    del eager, graphed
import gc  # noqa: E402
gc.collect()
torch.cuda.synchronize()
if rank == 0:
    print("1d. ResidualVQ data-parallel CUDA graph == eager: " + ("skipped (Gloo)" if SINGLE else "ok"), flush=True)

# ---------------- 2. sharded codebook, through the module API, against the ORACLE (un-sharded reference path) -------
# codebooks.py:350-435 on the whole codebook is the oracle; the sharded path must give its indices (outside the
# reference's own 1e-6 ties), bit-exact quantize, and on every rank the matching rows of its EMA + expiry result
D.SHARD_MIN_CODES = 4096
K, d, N = 4096, 64, 20000
g = torch.Generator().manual_seed(9)
x = torch.randn(N, d, generator=g)
full = torch.randn(K, d, generator=g) * 0.5
full[3000] = full[11]                 # duplicate in another shard: the lowest index must win every row
full[100:104] *= 30.0                 # never chosen -> die -> replaced by the rows rank 0 draws
for mode in ("replicated", "all_gather"):
    torch.manual_seed(0)
    vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=2),
                        sync_codebook=True).to(dev).train()
    cb = vq._codebook
    check(cb.sharded and cb.embeddings.shape[1] == K // world, "Codebook did not shard")
    cb.sharded_input = mode
    cb.load_full_codebook(full)
    n_loc = N // world
    x_in = x if mode == "replicated" else x[rank * n_loc:(rank + 1) * n_loc]
    x_ref = x if mode == "replicated" else x[:n_loc * world]
    from vqb200.codebook import Codebook
    Codebook._draw_rows = staticmethod(lambda n, m, device: (torch.randperm(n)[:m] if n >= m else torch.randint(0, n, (m,))).to(device))
    torch.manual_seed(21)
    with torch.no_grad():
        q, gidx, loss = vq(x_in[None].to(dev))
    st = O.CodebookState(full[None].clone(), full[None].clone(), torch.ones(1, K))
    torch.manual_seed(21)
    qo, io, lo, ex = O.vq_forward(st, x_ref[None], O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=2)), want_gap=True)
    rows = slice(0, N) if mode == "replicated" else slice(rank * n_loc, (rank + 1) * n_loc)
    diff = gidx[0].cpu() != io[0, rows]
    check(bool((ex["top2_rel_gap"][0, rows][diff] < 1e-6).all()),
          f"sharded ({mode}) indices differ from the oracle outside its 1e-6 window: {int(diff.sum())}")
    check(bool((gidx != 3000).all()), "duplicate code: the higher index won")
    same = ~diff
    check(torch.equal(q[0].cpu()[same], qo[0, rows][same]), f"sharded ({mode}) quantize not bit-exact")
    keep, none_touched = untouched(cb, [(gidx[0].cpu(), io[0, rows], diff)])
    if none_touched and mode == "replicated":
        check(abs(float(loss) - float(lo)) <= 1e-5 * float(lo), "sharded loss")
    compare_shard_buffers(cb, st, keep, f"sharded ({mode})")
    check(int((st.cluster_size[0] == 2.0).sum()) >= 4, "expiry did not fire in the sharded scenario")
    sd = vq.state_dict()
    check(tuple(sd["_codebook.embeddings"].shape) == (1, K, d), "state_dict must hold the full codebook")
if rank == 0:
    print("2. sharded codebook (K = 4096) vs oracle: ok", flush=True)

# ---------------- 3. sharded at the real threshold: masked bf16 input, expiry, input gradient ----------------
D.SHARD_MIN_CODES = SHARD_REAL
K, d, B, n = 65536, 64, 8, 2048
g = torch.Generator().manual_seed(13)
full = torch.randn(K, d, generator=g) * 0.5
full[40000] = full[11]                # duplicate in another shard
full[200:208] *= 30.0                 # never chosen -> die -> replaced
x = torch.randn(B, n, d, generator=g).to(torch.bfloat16)
mask = torch.rand(B, n, generator=g) > 0.2
bl = B // world
for mode in ("replicated", "all_gather"):
    torch.manual_seed(0)
    vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=2),
                        sync_codebook=True).to(dev).train()
    cb = vq._codebook
    check(cb.sharded and cb.embeddings.shape[1] == K // world, "K = 65536 did not shard at the real threshold")
    cb.sharded_input = mode
    cb.load_full_codebook(full)
    b_rows = slice(0, B) if mode == "replicated" else slice(rank * bl, (rank + 1) * bl)
    x_ref, m_ref = (x, mask) if mode == "replicated" else (x[:bl * world], mask[:bl * world])
    torch.manual_seed(21)
    with torch.no_grad():
        q, gidx, loss = vq(x[b_rows].to(dev), mask=mask[b_rows].to(dev))
    st = O.CodebookState(full[None].clone(), full[None].clone(), torch.ones(1, K))
    torch.manual_seed(21)
    qo, io, lo, ex = O.vq_forward(st, x_ref, O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=2)), mask=m_ref,
                                  want_gap=True, row_chunk=2048)
    got, ref = gidx.cpu(), io[b_rows]
    diff = got != ref
    gap = ex["top2_rel_gap"][0].reshape(x_ref.shape[:2])[b_rows]
    check(bool((gap[diff] < 1e-6).all()), f"K=65536 ({mode}) indices differ from the oracle outside its 1e-6 window")
    check(bool((gidx != 40000).all()), "K=65536: duplicate code, the higher index won")
    check(torch.equal(q.float().cpu()[~diff], qo[b_rows].float()[~diff]), f"K=65536 ({mode}) quantize not bit-exact")
    keep, none_touched = untouched(cb, [(got.reshape(-1), ref.reshape(-1), (diff & mask[b_rows]).reshape(-1))])
    if none_touched and mode == "replicated":
        check(abs(float(loss) - float(lo)) <= 1e-5 * float(lo), "K=65536 loss")
    compare_shard_buffers(cb, st, keep, f"K=65536 ({mode})")
    check(int((st.cluster_size[0] == 2.0).sum()) >= 8, "K=65536: expiry did not fire")
# input gradient of one training step: sharded == un-sharded VectorQuantize on the same (replicated) batch
mods = []
for sync in (True, False):
    torch.manual_seed(0)
    m = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0),
                       sync_codebook=sync).to(dev).train()
    m._codebook.sharded_input = "replicated"
    m._codebook.load_full_codebook(full)
    mods.append(m)
check(mods[0]._codebook.sharded and not mods[1]._codebook.sharded, "gradient check: sharding flags")
grads, inds = [], []
for m in mods:
    xg = x.to(dev).float().requires_grad_()
    q, ind, loss = m(xg, mask=mask.to(dev))
    (q.square().sum() * 1e-3 + loss.sum()).backward()
    grads.append(xg.grad)
    inds.append(ind)
same = inds[0] == inds[1]
check(bool(same.float().mean() > 0.999), "gradient check: too many index differences")
check(torch.equal(grads[0][same], grads[1][same]), "sharded input gradient differs from the un-sharded one")
if rank == 0:
    print("3. sharded K = 65536 (masked bf16, expiry, input gradient): ok", flush=True)

# ---------------- 4. ResidualVQ over sharded codebooks ----------------
Q, B, n = 2, 4, 2048
g = torch.Generator().manual_seed(17)
books = [torch.randn(K, d, generator=g) * (0.5 / 1.5 ** li) for li in range(Q)]
books[0][300:304] *= 30.0
xr = torch.randn(B, n, d, generator=g)


def _rvq(sync, thr):
    torch.manual_seed(0)
    m = ResidualVQ(dim=d, num_quantizers=Q, codebook_params=CodebookParams(dim=d, codebook_size=K,
                                                                           threshold_ema_dead_code=thr),
                   sync_codebook=sync).to(dev).train()
    for layer, c in zip(m.layers, books):
        layer._codebook.sharded_input = "replicated"
        layer._codebook.load_full_codebook(c)
    return m


rvq = _rvq(True, 2)
check(all(l._codebook.sharded for l in rvq.layers), "ResidualVQ codebooks did not shard")
sts = [O.CodebookState(c[None].clone(), c[None].clone(), torch.ones(1, K)) for c in books]
torch.manual_seed(23)
with torch.no_grad():
    q, ind, losses, codes = rvq(xr.to(dev), return_all_codes=True)
torch.manual_seed(23)
qo, io, lo, exs = O.rvq_forward(sts, xr, O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=2)), want_gap=True,
                                row_chunk=2048)
ind_c = ind.cpu()
row_diff = (ind_c != io).any(-1)
gap0 = exs[0]["top2_rel_gap"][0].reshape(B, n)
first_diff = ind_c[..., 0] != io[..., 0]
check(bool((gap0[first_diff] < 1e-6).all()), "RVQ level 0 differs from the oracle outside its 1e-6 window")
gap1 = exs[1]["top2_rel_gap"][0].reshape(B, n)
check(bool((gap1[row_diff & ~first_diff] < 1e-6).all()), "RVQ level 1 differs from the oracle outside its 1e-6 window")
check(torch.equal(q.cpu()[~row_diff], qo[~row_diff]), "RVQ quantized_out not bit-exact")
if not bool(row_diff.any()):
    check(bool(torch.allclose(losses.cpu(), lo, rtol=1e-5)), "RVQ losses")
for li, (layer, stl) in enumerate(zip(rvq.layers, sts)):
    keep, _ = untouched(layer._codebook, [(ind_c[..., li].reshape(-1), io[..., li].reshape(-1), row_diff.reshape(-1))])
    compare_shard_buffers(layer._codebook, stl, keep, f"RVQ level {li}")
check(int((sts[0].cluster_size[0] == 2.0).sum()) >= 4, "RVQ: expiry did not fire")
books_now = rvq.codebooks
check(tuple(books_now.shape) == (Q, K, d), "ResidualVQ.codebooks must be (Q, K, d)")
want = torch.stack([books_now[li][ind[..., li]] for li in range(Q)], 0)
check(torch.equal(codes, want), "return_all_codes")
check(torch.equal(rvq.get_output_from_indices(ind), want.sum(0)), "get_output_from_indices")
for li in range(Q):
    sl = slice(rvq.layers[li]._codebook.shard_offset, rvq.layers[li]._codebook.shard_offset + K // world)
    check(torch.equal(books_now[li][sl], rvq.layers[li]._codebook.embeddings[0]), "ResidualVQ.codebooks rows")
# input gradient: sharded (generic loop) == un-sharded (fused loop under autograd)
grads, inds = [], []
for sync in (True, False):
    m = _rvq(sync, 0)
    xg = xr.to(dev).requires_grad_()
    qq, ii, ll = m(xg)
    (qq.square().sum() * 1e-3 + ll.sum()).backward()
    grads.append(xg.grad)
    inds.append(ii)
same = (inds[0] == inds[1]).all(-1)
check(bool(same.float().mean() > 0.999), "RVQ gradient check: too many index differences")
check(bool(torch.allclose(grads[0][same], grads[1][same], rtol=1e-5, atol=1e-8)), "RVQ sharded input gradient")
if rank == 0:
    print("4. ResidualVQ over sharded codebooks: ok", flush=True)

# ---------------- 5. accessors ----------------
vq = VectorQuantize(dim=d, codebook_params=CodebookParams(dim=d, codebook_size=K, threshold_ema_dead_code=0),
                    sync_codebook=True).to(dev)
cb = vq._codebook
cb.load_full_codebook(full)
lo_, hi_ = cb.shard_offset, cb.shard_offset + cb.shard_size
check(torch.equal(vq.codebook.cpu(), full), "vq.codebook must be the full (K, d) codebook")
idx_probe = torch.randint(0, K, (3, 50), generator=g)
check(torch.equal(vq.get_codes_from_indices(idx_probe.to(dev)).cpu(), full[idx_probe]), "get_codes_from_indices")
new = torch.randn(K, d, generator=torch.Generator().manual_seed(77))
vq.codebook = new.to(dev)
check(torch.equal(cb.embeddings[0].cpu(), new[lo_:hi_]), "setter must keep this rank's rows")
check(torch.equal(vq.codebook.cpu(), new), "getter after setter")
with torch.no_grad():
    cb.embeddings.mul_(-2.0)
cb.invalidate_cache()
edited = (new * -2.0).to(dev)
vq.eval()
xe = torch.randn(1, 4096, d, generator=g).to(dev)
with torch.no_grad():
    qe, ie, _ = vq(xe)
ex_idx, _, _ = ops.search(xe, edited[None].contiguous(), None, False, force_exact=True)
check(torch.equal(ie, ex_idx), "after an in-place edit the eval forward must search the edited codebook")
check(torch.equal(qe, edited[ie]), "after an in-place edit the eval forward must gather the edited codebook")
if rank == 0:
    print("5. sharded accessors: ok", flush=True)
if rank == 0:
    print("MGPU OK", flush=True)
torch.cuda.synchronize()
dist.barrier()
dist.destroy_process_group()
