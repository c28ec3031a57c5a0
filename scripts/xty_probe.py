"""Timing / profiling driver for the X^T Y weight-gradient kernel at the stencil-backward shape."""
import os, sys, torch
sys.path.insert(0, os.getcwd())
from tensoflow_b200 import _lib
from tensoflow_b200._lib import check, ptr, stream_ptr
dev = torch.device('cuda:0')
lib = _lib.load()
rows, M, N = int(sys.argv[1]) if len(sys.argv) > 1 else 2340000, 256, 112
X = torch.randn(rows, M, device=dev); Y = torch.randn(rows, N, device=dev)
out = torch.zeros(M, N, device=dev)
for _ in range(2):
    check(lib.tf_xty_accumulate(ptr(X), ptr(Y), rows, M, N, ptr(out), stream_ptr()), "xty")
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(5):
    check(lib.tf_xty_accumulate(ptr(X), ptr(Y), rows, M, N, ptr(out), stream_ptr()), "xty")
b.record(); torch.cuda.synchronize()
ms = a.elapsed_time(b) / 5
print(f"rows={rows} {ms:.3f} ms  {rows * (M + N) * 4 / ms / 1e6:.1f} GB/s")
