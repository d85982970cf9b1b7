"""Race stress of the K5 kernel: the same launch repeated `trials` times at a benchmarked row count, every result
compared with ONE torch fp32 reference.  A data race between the epilogue's shared-memory reads and the TMA refill of the residual
ring (fixed in round 2: adapter_rows_sm100.cu `loads_returned`) showed up in 1-3 % of such launches as a few rows of one warp
carrying the NEXT ring box's bytes; tools/k5_debug.py explains such mismatches by brute-force search over the operands."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adapter4rec_b200 import ops

H, r = 768, 64
M = int(sys.argv[1]) if len(sys.argv) > 1 else 161280
trials = int(sys.argv[2]) if len(sys.argv) > 2 else 300


def rnd(*s, sc=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)


wd, wu = rnd(r, H, sc=0.05, seed=3), rnd(H, r, sc=0.05, seed=4)
gen = torch.Generator(device="cuda").manual_seed(9)
bd, bu = torch.randn(r, device="cuda", generator=gen) * 0.1, torch.randn(H, device="cuda", generator=gen) * 0.1
g, b = torch.rand(H, device="cuda", generator=gen) + 0.5, torch.randn(H, device="cuda", generator=gen) * 0.1
h, inp = rnd(M, H, seed=M + 1), rnd(M, H, seed=M + 2)
U = torch.relu(h.float() @ wd.float().t() + bd).to(torch.bfloat16).float() @ wu.float().t() + bu + h.float()
bad = 0
for tail in (1, 0, 2):
    z = U + (inp.float() if tail != 2 else 0)
    ref = torch.nn.functional.layer_norm(z.to(torch.bfloat16).float(), (H,), g, b, 1e-12) if tail == 0 else z
    first = None
    for t in range(trials):
        out = ops.adapter_ln_fwd(h, inp if tail != 2 else None, wd, bd, wu, bu, g if tail == 0 else None, b if tail == 0 else None,
                                 1e-12, act="relu", tail=tail, save=(t % 2 == 1))[0]
        n = int(((out.float() - ref).abs() > 0.08).sum())
        if first is None:
            first = out.clone()
        elif not torch.equal(out, first):          # the kernel is deterministic: every launch must give the same bits
            n += 1
        if n:
            bad += 1
            print("BAD  tail=%d trial %d: %d elements off" % (tail, t, n))
print("ALL OK" if bad == 0 else "FAILED (%d launches)" % bad)
