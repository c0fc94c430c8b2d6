"""Times only the tensor-core search kernel (CUDA events from the library) under the env set by the caller:
VQB_FUSED_PREP, and VQB_LIB_OVERRIDE for another build of the library (e.g. with a patch from profiles/ applied)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "vector-quantization-by-ml_b200"))
import torch
from vqb200 import ops, _lib as _L
if os.environ.get("VQB_LIB_OVERRIDE"):
    _L.LIB_PATH = os.path.join(ROOT, os.environ["VQB_LIB_OVERRIDE"])
dev = torch.device("cuda:0")
N, K, d = (int(a) for a in sys.argv[1:4]) if len(sys.argv) > 3 else (1 << 20, 8192, 256)
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn(1, N, d, generator=g, device=dev)
if not (len(sys.argv) > 4 and sys.argv[4] == "f32"):
    x = x.bfloat16()
c = torch.randn(1, K, d, generator=g, device=dev) * 0.5
cache = ops.prepare_codebook(c, False)
ops.TIME_SEARCH_KERNEL = True
for _ in range(3):
    ops.search(x, c, cache, False)
torch.cuda.synchronize(); ops.search_kernel_times_ms()
for _ in range(5):
    ops.search(x, c, cache, False)
torch.cuda.synchronize()
t = ops.search_kernel_times_ms()
ms = sum(t) / len(t)
print(os.environ.get('VQB_LIB_OVERRIDE','shipped'), end=' ')
print(f"N={N} K={K} d={d}: "
      f"tc kernel {ms:.3f} ms  {2*N*K*d/ms/1e9:.0f} TFLOP/s", flush=True)
