"""ncu target: the remaining kernels of one C2 pass that had no capture — the short-sequence (text) attention forward /
backward with dropout, and the tcgen05 weight-gradient kernel at the LoRA and the full-fine-tuning shapes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adapter4rec_b200 import ops
N, L, heads, dh = 5376, 30, 12, 64
H = heads * dh
M = N * L
qkv = torch.randn(M, 3 * H, device="cuda").to(torch.bfloat16)
dctx = torch.randn(M, H, device="cuda").to(torch.bfloat16)
mask = (torch.rand(N, L, device="cuda") < 0.7).float()
mask[:, 0] = 1
x = torch.randn(M, H, device="cuda").to(torch.bfloat16)
t1 = torch.randn(M, 64, device="cuda").to(torch.bfloat16)
du = torch.randn(M, 4 * H, device="cuda").to(torch.bfloat16)
for it in range(2):
    ctx = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, dropout=(0.1, 1234, 0))
    dq = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, dropout=(0.1, 1234, 0))
    g1 = ops.wgrad(qkv, t1)             # d(B_ext) = dqkv^T [T | 1]   (2304 x 64)
    g2 = ops.wgrad(t1, x)               # d(A_cat) = dT^T x           (64 x 768)
    g3 = ops.wgrad(du, x)               # full fine-tuning: d(W_1)    (3072 x 768)
torch.cuda.synchronize()
print("done")
