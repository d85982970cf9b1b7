"""Correctness of K5 (a4r_adapter_ln_fwd) against torch: all tails, relu / gelu, save on / off, ragged M; `--big` adds the
benchmarked row counts (M = 161,280 = 8.5 tiles per persistent CTA and M = 645,120 = 34 tiles per CTA: the multi-tile ring /
phase path), checked on EVERY row in row blocks."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
if "--lib" in sys.argv:      # A/B against a variant build of the library (tools/variants/*.so)
    import adapter4rec_b200.lib as _lib
    _i = sys.argv.index("--lib")
    _lib.LIB_PATH = os.path.abspath(sys.argv[_i + 1])
    del sys.argv[_i:_i + 2]
from adapter4rec_b200 import ops

H, r = 768, 64


def rnd(*s, sc=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)


def check(M, wd, wu, bd, bu, g, b, tails=(0, 1, 2), acts=("relu", "gelu"), saves=(False, True), blk=32768):
    ok = True
    h, inp = rnd(M, H, seed=M + 1), rnd(M, H, seed=M + 2)
    for tail in tails:
        for act in acts:
            for save in saves:
                gg, bb = (g, b) if tail == 0 else (None, None)
                out, z, mean, rstd, s, u = ops.adapter_ln_fwd(h, inp if tail != 2 else None, wd, bd, wu, bu, gg, bb, 1e-12, act=act,
                                                              tail=tail, save=save)
                torch.cuda.synchronize()
                e = es = ez = em = 0.0
                ones_ok = True
                detail = []
                for i in range(0, M, blk):          # torch fp32 reference in row blocks (every row is checked)
                    j = min(M, i + blk)
                    pre = h[i:j].float() @ wd.float().t() + bd
                    sr = torch.relu(pre) if act == "relu" else torch.nn.functional.gelu(pre)
                    zr = h[i:j].float() + sr.to(torch.bfloat16).float() @ wu.float().t() + bu + (inp[i:j].float() if tail != 2 else 0)
                    ref = torch.nn.functional.layer_norm(zr.to(torch.bfloat16).float(), (H,), g, b, 1e-12) if tail == 0 else zr
                    err = (out[i:j].float() - ref).abs()
                    e = max(e, float(err.max()))
                    if float(err.max()) >= 0.08 and len(detail) < 12:      # where: (row, tile, first / last bad column, count)
                        for rr in (err.max(1).values >= 0.08).nonzero().flatten()[:6].tolist():
                            cols = (err[rr] >= 0.08).nonzero().flatten()
                            detail.append((i + rr, (i + rr) // 128, int(cols.min()), int(cols.max()), int(cols.numel())))
                    if save:
                        es = max(es, float((s[i:j].float() - sr).abs().max()))
                        if tail == 0:
                            ez = max(ez, float((z[i:j].float() - zr).abs().max()))
                            em = max(em, float((mean[i:j] - zr.to(torch.bfloat16).float().mean(1)).abs().max()))
                        ones_ok &= bool((ops.s_ext(s)[i:j, r] == 1).all())
                # |z| <= ~6: final bf16 rounding 2^-8 * 6 = 0.023 (+ the bf16 rounding of z before the LayerNorm)
                good = e < 0.08 and es < 0.03 and ez < 0.05 and em < 1e-3 and ones_ok
                if not good:
                    ok = False
                    print("BAD  M=%d tail=%d %s save=%d out err %.4f s %.4f z %.4f mean %.5f ones %s %s" % (M, tail, act, save, e, es, ez, em, ones_ok, detail))
    return ok


def main():
    big = "--big" in sys.argv
    wd, wu = rnd(r, H, sc=0.05, seed=3), rnd(H, r, sc=0.05, seed=4)
    gen = torch.Generator(device="cuda").manual_seed(9)
    bd, bu = torch.randn(r, device="cuda", generator=gen) * 0.1, torch.randn(H, device="cuda", generator=gen) * 0.1
    g, b = torch.rand(H, device="cuda", generator=gen) + 0.5, torch.randn(H, device="cuda", generator=gen) * 0.1
    ok = True
    if big:
        ok &= check(161280, wd, wu, bd, bu, g, b)
        ok &= check(645120, wd, wu, bd, bu, g, b, acts=("relu",))
        ok &= check(645120 + 77, wd, wu, bd, bu, g, b, tails=(0,), acts=("gelu",), saves=(True,))
    else:
        for M in (128, 1000, 20000):
            ok &= check(M, wd, wu, bd, bu, g, b)
    print("ALL OK" if ok else "FAILED")


if __name__ == "__main__":
    main()
