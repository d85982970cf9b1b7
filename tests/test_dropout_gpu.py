"""-m gpu: counter-based dropout (train-mode semantics of nn.Dropout in the reference's BERT / SASRec blocks).
The RNG is restated on the host (tests/dropout_rng.py) so the kernels can be checked against torch with the SAME mask."""
import os
import sys

import pytest
import torch

import dropout_rng as R

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def keep_mask(seed, offset, n, p):
    """f32 mask of n consecutive elements starting at counter `offset` (4 elements per counter), and the kept scale"""
    return R.element_keep(seed, offset, p, torch.zeros(1, dtype=torch.int64), n)[0].float(), R.keep_scale(p)


def test_dropout_kernel_matches_host_rng_and_is_unbiased():
    from adapter4rec_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn((4096, 768), generator=g, device="cuda").to(BF16)
    res = torch.randn((4096, 768), generator=g, device="cuda").to(BF16)
    p, seed, off = 0.1, 12345, 777
    out = ops.dropout(x, res, p, seed, off)
    mask, scale = keep_mask(seed, off, x.numel(), p)
    ref = (x.float().cpu().flatten() * mask * scale + res.float().cpu().flatten()).view_as(x)
    assert float((out.float().cpu() - ref).abs().max()) <= 2 ** -7 * float(ref.abs().max())
    keep = float(mask.mean())
    assert abs(keep - 0.9) < 2e-3, keep
    assert torch.equal(ops.dropout(x, res, p, seed, off), out)                 # deterministic
    assert not torch.equal(ops.dropout(x, res, p, seed, off + 1), out)         # a different counter range
    assert torch.equal(ops.dropout(x, None, 0.0, seed, off), x)                # p = 0 is the identity


def test_dropout_add_function_backward_reuses_the_mask():
    from adapter4rec_b200 import functional as Fn
    Fn.DropoutState.manual_seed(99)
    x = torch.randn((512, 64), device="cuda").to(BF16).requires_grad_(True)
    r = torch.randn((512, 64), device="cuda").to(BF16).requires_grad_(True)
    out = Fn.dropout_add(x, r, 0.25)
    mask, scale = keep_mask(99, 0, x.numel(), 0.25)
    dy = torch.randn_like(out)
    out.backward(dy)
    ref_dx = (dy.float().cpu().flatten() * mask * scale).view_as(x)
    assert float((x.grad.float().cpu() - ref_dx).abs().max()) <= 2 ** -7 * float(ref_dx.abs().max())
    assert torch.equal(r.grad, dy)


@pytest.mark.parametrize("N,L,heads,dh,causal", [(6, 30, 12, 64, False), (9, 20, 2, 32, True)])
def test_attention_probability_dropout(N, L, heads, dh, causal):
    """probability dropout of the short-sequence kernel, without and with a key mask (BERT: the int64 [ids | mask] right
    half, right-padded; SASRec: f32, left-padded; both with a fully masked row)"""
    from adapter4rec_b200 import ops
    H = heads * dh
    g = torch.Generator(device="cuda").manual_seed(3)
    qkv = torch.randn((N * L, 3 * H), generator=g, device="cuda").to(BF16)
    dctx = torch.randn((N * L, H), generator=g, device="cuda").to(BF16)
    p, seed, off = 0.1, 4242, 1000
    keep = R.prob_keep(seed, off, p, torch.arange(N, device="cuda"), heads, L).float()
    lens = torch.randint(1, L + 1, (N,), generator=g, device="cuda")
    lens[1] = 0
    ok = torch.arange(L, device="cuda")[None, :] < lens[:, None]
    if causal:
        ok = ok.flip(1)
        masks = [(None, None), (ok, ok.float())]
    else:
        both = torch.zeros((N, 2 * L), dtype=torch.int64, device="cuda")
        both[:, L:] = ok.long()
        masks = [(None, None), (ok, both[:, L:])]
    mask_neg = -1e9
    for key_ok, mask in masks:
        qf = qkv.float().requires_grad_(True)
        q, k, v = [t.view(N, L, heads, dh).transpose(1, 2) for t in qf.view(N * L, 3, H).unbind(1)]
        s = (q @ k.transpose(-1, -2)) * dh ** -0.5
        allowed = torch.ones(N, 1, L, L, dtype=torch.bool, device="cuda")
        if key_ok is not None:
            allowed = allowed & key_ok.view(N, 1, 1, L)
        if causal:
            allowed = allowed & torch.tril(torch.ones(L, L, dtype=torch.bool, device="cuda"))
        s = s + torch.where(allowed, 0.0, mask_neg)
        ref = ((torch.softmax(s, -1) * keep * R.keep_scale(p)) @ v).transpose(1, 2).reshape(N * L, H)
        got = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=(p, seed, off))
        err = (got.float() - ref.detach()).abs()
        assert bool((err <= 2e-2 + 2 ** -6 * ref.detach().abs()).all()), (mask is not None, float(err.max()))
        ref.backward(dctx.float())
        dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg,
                                  dropout=(p, seed, off))
        for j, nm in enumerate(("dq", "dk", "dv")):
            a, b = dqkv[:, j * H:(j + 1) * H].float(), qf.grad[:, j * H:(j + 1) * H]
            rel = float((a - b).norm() / b.norm())
            assert rel <= 2e-2, "%s relative L2 error %.4f (key mask: %s)" % (nm, rel, mask is not None)


def test_train_mode_step_is_deterministic_given_the_seed_and_close_to_eval():
    import cases
    from adapter4rec_b200 import functional as Fn
    from test_model_gpu import build_gpu_model
    c = cases.tiny_case("houlsby")
    sd = cases.build_state_dict(c)
    model, _ = build_gpu_model(c, sd)
    items = cases.build_item_content(c)
    sample_items, log_mask, _ = cases.build_batch(c, items)
    rows, lm = sample_items.view(-1, 2 * c.L).cuda(), log_mask.cuda()
    model.eval()
    base = float(model(rows, lm, 0))
    model.train()
    losses, grads = [], []
    for _ in range(2):
        Fn.DropoutState.manual_seed(7)
        model.zero_grad(set_to_none=True)
        loss = model(rows, lm, 0)
        loss.backward()
        losses.append(float(loss))
        grads.append(torch.cat([p.grad.flatten() for p in model.parameters() if p.grad is not None]))
    assert losses[0] == losses[1] and torch.equal(grads[0], grads[1])        # same seed -> bit-identical step
    assert losses[0] != base and abs(losses[0] - base) < 0.5 * abs(base)      # dropout changes the loss, moderately
    assert torch.isfinite(grads[0]).all() and float(grads[0].norm()) > 0
    Fn.DropoutState.manual_seed(8)
    assert float(model(rows, lm, 0)) != losses[0]                             # another seed, another mask


@pytest.mark.parametrize("after", [False, True])
@pytest.mark.parametrize("block_n", [0, 64, 128, 256, 512])
@pytest.mark.parametrize("M,N,K", [(1000, 768, 64), (333, 72, 40)])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("res2", [False, True])
def test_gemm_epilogue_dropout_before_and_after_the_residual(after, block_n, M, N, K, bias, res2):
    """a4r_gemm_bf16_tn LINEAR epilogue: dropout(acc + bias) + residual(s) (forward of dense -> dropout -> + input) and
    dropout(acc + bias + residual(s)) (dropout_after_residual: the gradient through a dropout whose input gradient is a
    sum), against torch with the host-restated mask, on every tile width (0 = the automatic choice) and a ragged shape
    (partial row and column tiles), counter offsets below and past 2^32."""
    from adapter4rec_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    p = 0.1
    a = (torch.randn((M, K), generator=g, device="cuda") * 0.5).to(BF16)
    w = (torch.randn((N, K), generator=g, device="cuda") * 0.2).to(BF16)
    res = torch.randn((M, N), generator=g, device="cuda").to(BF16)
    r2 = torch.randn((M, N), generator=g, device="cuda").to(BF16) if res2 else None
    b = torch.randn((N,), generator=g, device="cuda") if bias else None
    seed, off = 0x1234567, 4096 if bias else (1 << 32) + 12345
    out = ops.gemm(a, w, bias=b, residual=res, residual2=r2, block_n=block_n, dropout=(p, seed, off), dropout_after=after)
    mask = R.element_keep(seed, off, p, torch.arange(M, device="cuda"), N).float()
    scale = R.keep_scale(p)
    acc = a.float() @ w.float().t() + (b if bias else 0.0)
    rsum = res.float() + (r2.float() if res2 else 0.0)
    ref = (acc + rsum) * mask * scale if after else acc * mask * scale + rsum
    err = (out.float() - ref).abs()
    assert bool((err <= 1e-2 + 8e-3 * ref.abs()).all()), float(err.max())
    if after:   # dropped elements of the SUM are exactly zero
        assert bool((out[mask == 0] == 0).all())


def test_fused_houlsby_block_matches_the_composed_path_in_train_mode():
    """HoulsbyPostLNBlockFunction (dense + dropout + adapter + LayerNorm in one node, dropout in GEMM epilogues both ways)
    against dense -> a4r_dropout -> fused adapter block: both draw the same counters in the same order, so under one
    seed the masks are identical and the results differ by bf16 rounding only."""
    import cases
    from adapter4rec_b200 import functional as Fn
    from adapter4rec_b200.model import model as M
    from test_model_gpu import build_gpu_model
    c = cases.tiny_case("houlsby")
    sd = cases.build_state_dict(c)
    model, _ = build_gpu_model(c, sd)
    items = cases.build_item_content(c)
    sample_items, log_mask, _ = cases.build_batch(c, items)
    rows, lm = sample_items.view(-1, 2 * c.L).cuda(), log_mask.cuda()
    model.train()
    results = []
    fused_forward_block = M.BertAdaptedSelfOutput.forward_block
    calls = [0]

    def counting(self, *a, **k):
        r = fused_forward_block(self, *a, **k)
        calls[0] += r is not None
        return r
    try:
        for variant in (counting, lambda self, *a, **k: None):
            M.BertAdaptedSelfOutput.forward_block = variant
            Fn.DropoutState.manual_seed(11)
            model.zero_grad(set_to_none=True)
            loss = model(rows, lm, 0)
            loss.backward()
            results.append((float(loss), {n: p.grad.float().clone() for n, p in model.named_parameters() if p.grad is not None}))
    finally:
        M.BertAdaptedSelfOutput.forward_block = fused_forward_block
    assert calls[0] >= 2 * c.layers - 1, "the fused node must be the path that runs (%d calls)" % calls[0]
    (l0, g0), (l1, g1) = results
    assert abs(l0 - l1) <= 5e-3 * abs(l1), (l0, l1)
    assert g0.keys() == g1.keys()
    a0, a1 = torch.cat([g0[k].flatten() for k in g0]), torch.cat([g1[k].flatten() for k in g0])
    assert float((a0 - a1).norm() / a1.norm()) <= 3e-2
