"""Debug helper: stress one K5 configuration and explain every mismatching 8-column piece by testing where a stale / foreign
operand would have come from (residual h / input of another chunk, up-projection U of another chunk)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adapter4rec_b200 import ops
H, r = 768, 64
def rnd(*s, sc=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)
wd, wu = rnd(r, H, sc=0.05, seed=3), rnd(H, r, sc=0.05, seed=4)
gen = torch.Generator(device="cuda").manual_seed(9)
bd, bu = torch.randn(r, device="cuda", generator=gen) * 0.1, torch.randn(H, device="cuda", generator=gen) * 0.1
M = int(sys.argv[1]) if len(sys.argv) > 1 else 161280
trials = int(sys.argv[2]) if len(sys.argv) > 2 else 40
tail = int(sys.argv[3]) if len(sys.argv) > 3 else 1
dbg = int(sys.argv[4]) if len(sys.argv) > 4 else 0
h, inp = rnd(M, H, seed=M + 1), rnd(M, H, seed=M + 2)
pre = h.float() @ wd.float().t() + bd
sr = torch.relu(pre).to(torch.bfloat16)
U = sr.float() @ wu.float().t()
ref = h.float() + U + bu + (inp.float() if tail == 1 else 0)
nbad_total = 0
for t in range(trials):
    out = ops.adapter_ln_fwd(h, inp if tail == 1 else None, wd, bd, wu, bu, None, None, 1e-12, act="relu", tail=tail, save=(t % 2 == 1))[0]
    torch.cuda.synchronize()
    e = (out.float() - ref).abs()
    piece = e.view(M, H // 8, 8).max(2).values > 0.08           # [M, 96] 8-column pieces
    idx = piece.nonzero()
    if idx.numel() == 0:
        continue
    nbad_total += idx.shape[0]
    tiles = sorted(set((idx[:, 0] // 128).tolist()))
    pcs = sorted(set(idx[:, 1].tolist()))
    print("trial %d: %d bad pieces; tiles %s (tile %% 148 = %s, tile // 148 = %s); pieces %s (chunk %s, piece-in-chunk %s)" % (
        t, idx.shape[0], tiles[:8], [x % 148 for x in tiles[:8]], [x // 148 for x in tiles[:8]], pcs[:8], [x // 4 for x in pcs[:8]], [x % 4 for x in pcs[:8]]))
    rows_in_tile = sorted(set((idx[:, 0] % 128).tolist()))
    print("   rows in tile:", rows_in_tile[:40], "n=%d" % len(rows_in_tile))
    # brute-force explanation of the first bad pieces: which operand piece ANYWHERE in the tensors reproduces the result?
    s_bf = sr.float()
    for row, pc in idx[:6].tolist():
        c0 = pc * 8
        got = out[row, c0:c0 + 8].float()
        hh, ii, uu, bb = h[row, c0:c0 + 8].float(), (inp[row, c0:c0 + 8].float() if tail == 1 else 0), U[row, c0:c0 + 8], bu[c0:c0 + 8]
        res = []
        def search(name, target, pool):
            err = (pool.view(-1, 8).float() - target[None, :]).abs().max(1).values
            j = int(err.argmin())
            res.append((round(float(err[j]), 4), name, j // 96, j % 96))
        search("h stale", got - uu - bb - ii, h)
        if tail == 1:
            search("i stale", got - uu - bb - hh, inp)
            search("h+i stale (same place)", got - uu - bb, (h.float() + inp.float()).to(torch.bfloat16))
        search("U foreign", got - hh - ii - bb, U)
        search("z foreign", got, ref.to(torch.bfloat16))
        # partial up-projection: subsets of the four 16-wide k-slices
        parts = torch.stack([s_bf[row, 16 * k:16 * k + 16] @ wu[c0:c0 + 8, 16 * k:16 * k + 16].float().t() for k in range(4)])
        for mask in range(16):
            pu = sum(parts[k] for k in range(4) if mask >> k & 1) if mask else torch.zeros(8, device="cuda")
            res.append((round(float((pu + bb + hh + ii - got).abs().max()), 4), "partial U k-mask %d" % mask, row, pc))
        res.sort()
        print("   row %d (tile %d row %d) piece %d: %s" % (row, row // 128, row % 128, pc, res[:3]))
print("total bad pieces over %d trials: %d" % (trials, nbad_total))
