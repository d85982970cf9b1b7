"""tcgen05 wgrad at the C2 / full-fine-tune shapes (timed alone, CUDA events)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adapter4rec_b200 import ops
M = 161280
def r(*s): return (torch.randn(*s, device="cuda") * 0.05).to(torch.bfloat16)
def t(fn, it=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(it): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / it * 1e3
for (N, K) in [(2304, 64), (64, 768), (768, 768), (3072, 768), (768, 3072), (768, 64), (64, 64)]:
    a, b = r(M, N), r(M, K)
    us = t(lambda: ops.wgrad(a, b))
    fl = 2.0 * M * N * K
    by = M * (N + K) * 2
    print("N=%5d K=%5d  %8.1f us (%7.1f TFLOP/s, %6.0f GB/s)" % (N, K, us, fl / us / 1e6, by / us / 1e3), flush=True)
