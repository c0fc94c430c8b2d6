"""world_size-2 Gloo tests (CPU) of a ResidualVQ over SHARDED codebooks and of the codebook accessors on shards, through
the product's orchestration with the tensor-level wrappers replaced by plain-torch statements (tests/cpu_kernels.py).

A sharded level must take the generic per-level loop (`VectorQuantize` -> `Codebook._run` on shards): the fused level
kernels search and update one whole codebook.  The accessors (`VectorQuantize.codebook`, `get_codes_from_indices`,
`ResidualVQ.codebooks`) speak in global code ids, so they read the full codebook, and the `codebook` setter takes the
full codebook and keeps this rank's rows."""
import datetime
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_full(t):
    """(1, K/W, ...) shards of every rank -> (K, ...) in rank order, with the test's own collective."""
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t.detach().contiguous())
    return torch.cat(parts, dim=1)[0]


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "tests"), os.path.join(root, "vector-quantization-by-ml_b200")):
        sys.path.insert(0, p)
    import cpu_kernels
    from oracle import vq_oracle as O
    from vqb200 import CodebookParams, ResidualVQ, _lib, distributed as D, ops, rvq as RVQ
    cpu_kernels.install(ops, _lib)
    D.SHARD_MIN_CODES = 32

    # On the GPU the fused level loop would be eligible for these inputs: let `_can_fuse` see a device tensor, so that
    # only the codebooks being sharded can send the levels to the generic loop
    real_can_fuse = RVQ.ResidualVQ._can_fuse

    class _OnDevice:
        def __init__(self, t):
            self.is_cuda, self.ndim, self.requires_grad, self.shape = True, t.ndim, t.requires_grad, t.shape

    fused = []

    def can_fuse(self, x, dropout_active):
        ok = real_can_fuse(self, _OnDevice(x), dropout_active)
        fused.append(ok)
        return ok
    RVQ.ResidualVQ._can_fuse = can_fuse

    res = {}
    Q, K, d, b, n = 2, 64, 8, 2, 90
    g = torch.Generator().manual_seed(4)
    x_all = torch.randn(world * b, n, d, generator=g)
    books = [torch.randn(K, d, generator=g) * (0.6 / 1.5 ** li) for li in range(Q)]
    books[0][40] = books[0][7]                   # a duplicate in the other shard: the lowest index must win
    books[0][50:53] *= 30.0                      # never chosen: these die and are replaced (expiry on a shard)

    for mode in ("replicated", "all_gather"):
        torch.manual_seed(0)
        m = ResidualVQ(dim=d, num_quantizers=Q, codebook_params=CodebookParams(dim=d, codebook_size=K,
                                                                               threshold_ema_dead_code=2),
                       sync_codebook=True).train()
        sts = []
        for layer, c in zip(m.layers, books):
            cb = layer._codebook
            assert cb.sharded and cb.embeddings.shape == (1, K // world, d)
            cb.sharded_input = mode
            cb.load_full_codebook(c)
            sts.append(O.CodebookState(c[None].clone(), c[None].clone(), torch.ones(1, K)))
        x_in = x_all if mode == "replicated" else x_all[rank * b:(rank + 1) * b]
        rows = slice(0, world * b) if mode == "replicated" else slice(rank * b, (rank + 1) * b)
        torch.manual_seed(21)
        with torch.no_grad():
            q, ind, loss, codes = m(x_in, return_all_codes=True)
        torch.manual_seed(21)
        qo, io, lo, _ = O.rvq_forward(sts, x_all, O.VQOpts(codebook=O.CodebookOpts(threshold_ema_dead_code=2)))
        res[f"idx_{mode}"] = torch.equal(ind, io[rows]) and bool((ind[..., 0] != 40).all())
        res[f"q_{mode}"] = torch.equal(q, qo[rows])
        if mode == "replicated":
            res["loss"] = bool(torch.allclose(loss, lo, rtol=1e-6))
        bufs = True
        for layer, st in zip(m.layers, sts):
            cb = layer._codebook
            sl = slice(cb.shard_offset, cb.shard_offset + cb.shard_size)
            bufs &= torch.equal(cb.cluster_size[0], st.cluster_size[0, sl])
            bufs &= float((cb.embeddings[0] - st.embeddings[0, sl]).abs().max()) < 1e-5
            bufs &= float((cb.embed_avg[0] - st.embed_avg[0, sl]).abs().max()) < 1e-5
        res[f"bufs_{mode}"] = bufs
        res[f"expired_{mode}"] = int((sts[0].cluster_size[0] == 2.0).sum())
        # the codes returned with the output and the accessors read the full (post-update) codebooks
        full = [_gather_full(layer._codebook.embeddings) for layer in m.layers]
        want = torch.stack([full[li][ind[..., li]] for li in range(Q)], 0)
        res[f"all_codes_{mode}"] = torch.equal(codes, want)
        res[f"from_indices_{mode}"] = torch.equal(m.get_output_from_indices(ind), want.sum(0))
        res[f"codebooks_{mode}"] = torch.equal(m.codebooks, torch.stack(full, 0))
        vq0 = m.layers[0]
        res[f"vq_codebook_{mode}"] = torch.equal(vq0.codebook, full[0])
        res[f"vq_codes_{mode}"] = torch.equal(vq0.get_codes_from_indices(ind[..., 0]), full[0][ind[..., 0]])

    # setter: takes the full codebook, keeps this rank's rows
    cb0 = vq0._codebook
    new = torch.randn(K, d, generator=torch.Generator().manual_seed(77))
    vq0.codebook = new
    res["setter_rows"] = torch.equal(cb0.embeddings[0], new[cb0.shard_offset:cb0.shard_offset + cb0.shard_size])
    res["setter_full"] = torch.equal(vq0.codebook, new)
    # an in-place edit of the shard + invalidate_cache(): the next eval forward searches AND gathers the edited codebook
    with torch.no_grad():
        cb0.embeddings.mul_(-2.0)
    cb0.invalidate_cache()
    edited = new * -2.0
    vq0.eval()
    xe = x_all[rank * b:(rank + 1) * b]
    with torch.no_grad():
        qe, ie, _ = vq0(xe)
    ref_i = O.similarities(x_all.reshape(1, -1, d), edited[None], False).argmax(-1)[0].reshape(world * b, n)
    res["edit_idx"] = torch.equal(ie, ref_i[rank * b:(rank + 1) * b])
    res["edit_q"] = torch.equal(qe, edited[ie])
    res["never_fused"] = len(fused) == 2 and not any(fused)
    if rank == 0:
        torch.save(res, out)
    dist.destroy_process_group()


def test_two_rank_gloo_residual_vq_over_sharded_codebooks_and_accessors(tmp_path):
    out = str(tmp_path / "rvq_sharded.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    res = torch.load(out)
    for mode in ("replicated", "all_gather"):
        assert res[f"expired_{mode}"] >= 3, res
    assert all(v for k, v in res.items() if not k.startswith("expired_")), res
