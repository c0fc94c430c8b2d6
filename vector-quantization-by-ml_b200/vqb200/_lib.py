"""ctypes binding of libvqb200.so (include/vqb.h).

There is no CPU implementation and no alternative backend: if the shared library
is missing or a tensor is not on a CUDA device the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvqb200.so")

VQB_F32, VQB_BF16, VQB_F16 = 0, 1, 2
VQB_EUCLID, VQB_DOT = 0, 1
SEARCH_LATENTS_PREPARED = 1
SEARCH_FORCE_EXACT = 2
SEARCH_TIMING = 4
SEARCH_FUSED_PREP = 8

_DTYPES = {torch.float32: VQB_F32, torch.bfloat16: VQB_BF16, torch.float16: VQB_F16}

_p, _i64, _i32, _sz, _f32, _f64 = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_float, C.c_double

# name -> (restype, argtypes); must list every symbol declared in include/vqb.h
SIGNATURES = {
    "vqb_version": (_i32, []),
    "vqb_last_error": (C.c_char_p, []),
    "vqb_launch_count": (_i64, []),
    "vqb_search_timing": (_i32, [_p, _i32]),
    "vqb_codebook_cache_bytes": (_sz, [_i64, _i32, _i32]),
    "vqb_prepare_codebook": (_i32, [_p, _i64, _i32, _i32, _i32, _p, _sz, _p]),
    "vqb_search_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "vqb_search": (_i32, [_p, _i32, _p, _p, _i32, _i64, _i64, _i32, _i32, _i64, _p, _p, _i32, _p, _sz, _p]),
    "vqb_search_stats": (_i32, [_p, _p, _p]),
    "vqb_l2norm_rows": (_i32, [_p, _i32, _p, _i64, _i32, _p]),
    "vqb_l2norm_prepare_supported": (_i32, [_i32]),
    "vqb_l2norm_prepare": (_i32, [_p, _i32, _p, _i64, _i64, _i32, _i32, _p, _p, _sz, _p]),
    "vqb_gather_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "vqb_gather_st_loss": (_i32, [_p, _i32, _p, _p, _p, _i32, _i32, _p, _p, _i64, _i64, _i32, _i32, _p, _sz, _p]),
    "vqb_st_commit_backward": (_i32, [_p, _p, _p, _i32, _p, _p, _p, _f32, _p, _i64, _i64, _i32, _i32, _p]),
    "vqb_rot_commit_backward": (_i32, [_p, _p, _p, _i32, _p, _p, _p, _f32, _p, _i64, _i64, _i32, _i32, _p]),
    "vqb_ema_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "vqb_ema_reduce": (_i32, [_p, _i32, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _sz, _p]),
    "vqb_ema_apply": (_i32, [_p, _p, _p, _p, _f32, _f64, _i32, _i64, _i32, _i32, _p, _sz, _p]),
    "vqb_ema_apply_counts": (_i32, [_p, _p, _f32, _i64, _i32, _i32, _p, _p]),
    "vqb_ema_apply_rows": (_i32, [_p, _p, _p, _p, _f32, _f64, _i64, _i32, _i64, _i32, _i32, _p, _p]),
    "vqb_quantize_ema_supported": (_i32, [_i32]),
    "vqb_quantize_ema_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "vqb_quantize_ema": (_i32, [_p, _i32, _p, _p, _p, _i32, _i32, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _sz, _p]),
    "vqb_expire_scatter": (_i32, [_p, _i32, _p, _i64, _f32, _f32, _i32, _p, _p, _p, _i64, _i32, _i32, _p]),
    "vqb_rvq_level": (_i32, [_p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _i64, _i32, _i32, _p, _sz, _p, _sz, _p, _p]),
    "vqb_column_moments": (_i32, [_p, _i32, _p, _i64, _i64, _i32, _p, _p, _p]),
    "vqb_dense_gumbel_sample": (_i32, [_p, _i32, _p, _p, _p, _i32, _f32, _p, C.c_uint64, C.c_uint64, C.c_uint32, _p,
                                       _i64, _i64, _i32, _i32, _p]),
    "vqb_dense_scores": (_i32, [_p, _i32, _p, _p, _p, _i32, _p, _i64, _i64, _i32, _i32, _p]),
    "vqb_rvq_backward": (_i32, [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _i64, _i32, _p]),
    "vqb_rvq_backward_rot": (_i32, [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _i64, _i32, _p]),
    "vqb_rvq_replay_out_supported": (_i32, [_i32, _i32]),
    "vqb_rvq_replay_out": (_i32, [_p, _p, _p, _p, _i32, _p, _p, _i64, _i32, _p]),
    "vqb_rvq_level_ema_supported": (_i32, [_i32]),
    "vqb_rvq_level_ema": (_i32, [_p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p, _p, _i64, _i32, _i32, _p, _sz, _p, _sz,
                                  _p, _p]),
    "vqb_minkey_pack": (_i32, [_p, _p, _i64, _p, _p]),
    "vqb_minkey_unpack": (_i32, [_p, _i64, _p, _p, _p]),
    "vqb_dense_row_norms": (_i32, [_p, _i32, _i64, _i32, _p, _p]),
    "vqb_dense_rowstats": (_i32, [_p, _i32, _p, _p, _p, _i32, _f32, _p, _p, _p, _i64, _i64, _i32, _i32, _p]),
    "vqb_dense_rowdot": (_i32, [_p, _i32, _p, _p, _p, _i32, _f32, _p, _p, _i64, _p, _i64, _i64, _i32, _i32, _p]),
    "vqb_dense_avgprob": (_i32, [_p, _i32, _p, _p, _p, _i32, _f32, _p, _p, _i64, _i64, _i64, _i32, _i32, _p]),
    "vqb_dense_backward": (_i32, [_p, _i32, _p, _p, _p, _p, _i32, _f32, _p, _p, _p, _p, _p, _i64, _p, _i64, _i64, _i32,
                                  _i32, _p]),
    "vqb_dense_backward_codes_splits": (_i32, [_i64, _i64, _i32, _i32]),
    "vqb_dense_backward_codes": (_i32, [_p, _i32, _p, _p, _p, _i32, _f32, _p, _p, _p, _p, _p, _i64, _p, _i32, _i64, _i64,
                                        _i32, _i32, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"vqb200: CUDA library not found at {LIB_PATH}. Build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C vector-quantization-by-ml_b200/csrc`). "
                "There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = lib().vqb_last_error().decode("utf-8", "replace")
    exc = {-1: ValueError, -4: NotImplementedError}.get(rc, RuntimeError)
    raise exc(f"{what} failed (code {rc}): {msg}")


def dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"vqb200: unsupported latent dtype {t.dtype} (float32, bfloat16, float16 only)") from None


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"vqb200: `{name}` must live on a CUDA device (got {t.device}); there is no CPU path")
    if not t.is_contiguous():
        raise RuntimeError(f"vqb200: `{name}` must be contiguous")


def require_device(x: torch.Tensor) -> None:
    if not x.is_cuda:
        raise RuntimeError(f"vqb200.Codebook: input must be on a CUDA device (got {x.device}); "
                           "there is no CPU implementation")


def aligned(t: torch.Tensor) -> torch.Tensor:
    """Contiguous and 16-byte aligned (the kernels use 128-bit loads); copies only when needed."""
    if not t.is_contiguous() or t.data_ptr() % 16:
        t = t.contiguous()
        if t.data_ptr() % 16:
            t = t.clone(memory_format=torch.contiguous_format)
    return t


def require_aligned(t, name: str) -> None:
    """A buffer the kernels write in place cannot be swapped for an aligned copy: it must be 16-byte aligned already."""
    if t is not None and t.data_ptr() % 16:
        raise ValueError(f"vqb200: `{name}` must be 16-byte aligned (the kernels use 128-bit stores)")


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream
