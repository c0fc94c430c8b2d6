"""The ResidualVQ level entry points of `vqb200.ops` hand the library only 16-byte aligned tensors (CPU, no library).

`rvq_level`, `rvq_level_ema`, `rvq_replay_out` and `rvq_backward` read their rows with 128-bit loads.  A contiguous fp32
tensor can still start at any element: a view into a larger buffer, e.g. the gradient of the second input of a
`torch.cat`.  Such an input must be copied to an aligned buffer before the call; a buffer the kernel writes in place
cannot be copied and is refused instead.

The library is replaced by a recorder, so every pointer a wrapper would pass is visible without a GPU."""
import ctypes as C

import pytest
import torch

N, D, K, Q = 6, 8, 5, 3


class _Recorder:
    """Stands in for the loaded library: returns 0 (success, or 0 workspace bytes) and records every call."""

    def __init__(self):
        self.calls, self.kept = [], []

    def __getattr__(self, name):
        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn

    def last(self, name):
        hits = [a for n, a in self.calls if n == name]
        assert len(hits) == 1, f"{name} called {len(hits)} times"
        return hits[0]


@pytest.fixture
def rec(monkeypatch):
    from vqb200 import _lib, ops
    r = _Recorder()
    monkeypatch.setattr(ops, "workspace", lambda kind, nbytes, device: torch.empty(max(int(nbytes), 256),
                                                                                   dtype=torch.uint8))
    monkeypatch.setattr(_lib, "require_cuda", lambda t, name: None)
    monkeypatch.setattr(_lib, "stream_ptr", lambda device: 0)
    monkeypatch.setattr(_lib, "lib", lambda: r)
    real_aligned = _lib.aligned

    def aligned(t):       # keeps the copies alive, so the test can read what a pointer points to after the call
        out = real_aligned(t)
        r.kept.append(out)
        return out
    monkeypatch.setattr(_lib, "aligned", aligned)
    return r


def _odd(*shape, dtype=torch.float32):
    """A contiguous tensor whose data starts one element past a 16-byte boundary."""
    n = 1
    for s in shape:
        n *= s
    buf = torch.randn(n + 1, generator=torch.Generator().manual_seed(n)).to(dtype)
    t = buf[1:].view(*shape)
    assert t.is_contiguous() and t.data_ptr() % 16 == t.element_size()
    return t


def _value(a):
    return a.value if isinstance(a, C.c_void_p) else a


def _array(a, n):
    """The n pointers of a `(c_void_p * n)` array passed by address."""
    return [p or 0 for p in (C.c_void_p * n).from_address(_value(a))]


def _floats(p, n):
    return torch.tensor(list((C.c_float * n).from_address(p)))


def _assert_aligned(name, args, ptr_pos, array_pos=(), n=0):
    ptrs = {f"arg{i}": _value(args[i]) or 0 for i in ptr_pos}
    for i in array_pos:
        for l, p in enumerate(_array(args[i], n)):
            ptrs[f"arg{i}[{l}]"] = p
    bad = {k: hex(v) for k, v in ptrs.items() if v % 16}
    assert not bad, f"{name}: pointers off a 16-byte boundary: {bad}"


def _levels():
    g = torch.Generator().manual_seed(3)
    cbs = [_odd(K, D) for _ in range(Q)]
    idx = [torch.randint(0, K, (N,), generator=g) for _ in range(Q)]
    return cbs, idx


def test_rvq_backward_aligns_a_gradient_view(rec):
    from vqb200 import ops
    cbs, idx = _levels()
    x = _odd(N, D)
    g_out = _odd(N, D)
    mask = torch.tensor([1, 0, 1, 1, 0, 1], dtype=torch.uint8)
    ops.rvq_backward(x, cbs, idx, [True, False, True], torch.ones(Q), g_out, mask)
    a = rec.last("vqb_rvq_backward")
    # x, codebooks, indices, training, Q, coef, g_out, mask, grad_x, N, d, stream
    _assert_aligned("vqb_rvq_backward", a, (0, 5, 6, 7, 8), (1, 2), Q)
    assert torch.equal(_floats(_value(a[6]), N * D), g_out.reshape(-1)), "the aligned g_out lost its values"
    assert torch.equal(_floats(_value(a[0]), N * D), x.reshape(-1))
    for p, c in zip(_array(a[1], Q), cbs):
        assert torch.equal(_floats(p, K * D), c.reshape(-1))


def test_rvq_backward_aligns_a_low_precision_gradient(rec):
    from vqb200 import ops
    cbs, idx = _levels()
    g_out = _odd(N, D, dtype=torch.bfloat16)
    ops.rvq_backward(torch.randn(N, D), cbs, idx, [True] * Q, torch.ones(Q), g_out, None)
    a = rec.last("vqb_rvq_backward")
    _assert_aligned("vqb_rvq_backward", a, (0, 5, 6, 7, 8), (1, 2), Q)
    assert torch.equal(_floats(_value(a[6]), N * D), g_out.float().reshape(-1))


def test_rvq_replay_out_aligns_its_inputs(rec):
    from vqb200 import ops
    cbs, idx = _levels()
    x = _odd(N, D)
    ops.rvq_replay_out(x, cbs, idx, [True, True, False], None)
    a = rec.last("vqb_rvq_replay_out")
    # x, codebooks, indices, training, Q, mask, out, N, d, stream
    _assert_aligned("vqb_rvq_replay_out", a, (0, 5, 6), (1, 2), Q)
    assert torch.equal(_floats(_value(a[0]), N * D), x.reshape(-1))
    with pytest.raises(ValueError, match="out"):
        ops.rvq_replay_out(torch.randn(N, D), cbs, idx, [True] * Q, None, out=_odd(N, D))


@pytest.mark.parametrize("ema", [False, True])
def test_rvq_level_aligns_its_inputs_and_refuses_unaligned_outputs(rec, ema):
    from vqb200 import ops
    residual, emb = _odd(N, D), _odd(K, D)
    idx = torch.randint(0, K, (N,), generator=torch.Generator().manual_seed(5))
    nxt, out, q = torch.empty(N, D), torch.zeros(N, D), torch.empty(N, D)
    if ema:
        ops.rvq_level_ema(residual, nxt, emb, idx, True, False, out, None, q_out=q)
        name = "vqb_rvq_level_ema"
        # residual, residual_next, embeddings, idx, bound_ws, training, first, out, q_out, loss, stats, N, K, d, ws,
        # ws_bytes, next_ws, next_ws_bytes, next_cache, stream
        pos = (0, 1, 2, 3, 4, 7, 8, 9, 10, 14, 16, 18)
    else:
        ops.rvq_level(residual, nxt, emb, idx, None, True, False, out, None, q_out=q)
        name = "vqb_rvq_level"
        # residual, residual_next, embeddings, idx, mask, training, first, out, q_out, loss, N, K, d, gather_ws,
        # gather_ws_bytes, next_ws, next_ws_bytes, next_cache, stream
        pos = (0, 1, 2, 3, 4, 7, 8, 9, 13, 15, 17)
    a = rec.last(name)
    _assert_aligned(name, a, pos)
    assert torch.equal(_floats(_value(a[0]), N * D), residual.reshape(-1))
    assert torch.equal(_floats(_value(a[2]), K * D), emb.reshape(-1))
    assert (_value(a[1]), _value(a[7]), _value(a[8])) == (nxt.data_ptr(), out.data_ptr(), q.data_ptr()), \
        "buffers written in place must reach the kernel as they are"
    call = ops.rvq_level_ema if ema else ops.rvq_level
    for which in ("residual_next", "quantized_out", "q_out"):
        bufs = {"residual_next": torch.empty(N, D), "quantized_out": torch.zeros(N, D), "q_out": torch.empty(N, D)}
        bufs[which] = _odd(N, D)
        with pytest.raises(ValueError, match=which):
            if ema:
                call(torch.randn(N, D), bufs["residual_next"], torch.randn(K, D), idx, True, False,
                     bufs["quantized_out"], None, q_out=bufs["q_out"])
            else:
                call(torch.randn(N, D), bufs["residual_next"], torch.randn(K, D), idx, None, True, False,
                     bufs["quantized_out"], None, q_out=bufs["q_out"])
