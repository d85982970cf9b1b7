"""-m gpu: each sm_100a kernel, called through the C ABI (adapter4rec_b200.ops -> ctypes -> .so), against a plain
PyTorch fp32 reference of the same op on the same seeded inputs.  Tolerances are stated per test: inputs are
bf16-exact, accumulation is fp32, so the only error is the final bf16 rounding (2^-8 relative) unless noted."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


def _ops():
    from adapter4rec_b200 import ops
    return ops


def _rand(shape, scale=1.0, seed=0, dtype=BF16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda", dtype=torch.float32) * scale).to(dtype)


def _close(got, ref, rtol, atol, what):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = err > tol
    assert not bad.any(), "%s: %d/%d mismatches, max abs err %.4g (ref max %.4g)" % (
        what, int(bad.sum()), bad.numel(), float(err.max()), float(ref.abs().max()))


GEMM_SHAPES = [
    # M, N, K, block_n
    (128, 256, 64, 0), (128, 64, 64, 0), (128, 128, 128, 0),
    (256, 768, 768, 0), (1000, 2304, 768, 0), (300, 3072, 768, 0), (515, 768, 3072, 0),
    (77, 64, 768, 0), (4096, 768, 768, 128), (2048, 256, 64, 64), (130, 72, 40, 0),
    (10240, 64, 256, 0), (148 * 128 * 2 + 5, 768, 768, 0),
    # block_n = 512: the 256-wide tile on a CTA pair (tcgen05 cta_group::2, 256 x 256 per cluster)
    (256, 256, 64, 512), (512, 768, 768, 512), (1000, 2304, 768, 512), (300, 3072, 768, 512), (515, 768, 3072, 512),
    (77, 256, 128, 512), (148 * 256 + 133, 768, 768, 512),
]


@pytest.mark.parametrize("M,N,K,bn", GEMM_SHAPES)
def test_gemm_linear(M, N, K, bn):
    ops = _ops()
    a, b = _rand((M, K), 1.0, 1), _rand((N, K), K ** -0.5, 2)
    bias = _rand((N,), 1.0, 3, torch.float32)
    ref = a.float() @ b.float().t() + bias
    got = ops.gemm(a, b, bias=bias, block_n=bn)
    _close(got, ref, 2 ** -7, 1e-2, "gemm bf16 out")
    got32 = ops.gemm(a, b, bias=bias, block_n=bn, out_dtype=torch.float32)
    _close(got32, ref, 1e-4, 1e-3, "gemm f32 out")


@pytest.mark.parametrize("bn", [0, 512])
def test_gemm_epilogues(bn):
    ops = _ops()
    M, N, K = 700, 768, 256
    a, b = _rand((M, K), 1.0, 1), _rand((N, K), K ** -0.5, 2)
    bias = _rand((N,), 0.5, 3, torch.float32)
    r1, r2 = _rand((M, N), 1.0, 4), _rand((M, N), 1.0, 5)
    v = a.float() @ b.float().t() + bias
    _close(ops.gemm(a, b, bias=bias, residual=r1, residual2=r2, block_n=bn), v + r1.float() + r2.float(), 2 ** -7, 2e-2, "linear+res")
    aux = torch.empty((M, N), dtype=BF16, device="cuda")
    got = ops.gemm(a, b, bias=bias, epilogue=ops.EPI_GELU, aux=aux, block_n=bn)
    _close(aux, v, 2 ** -7, 1e-2, "gelu aux (pre-activation)")
    _close(got, torch.nn.functional.gelu(v), 2 ** -7, 1e-2, "gelu")
    _close(ops.gemm(a, b, bias=bias, epilogue=ops.EPI_RELU, block_n=bn), torch.relu(v), 2 ** -7, 1e-2, "relu")
    u = _rand((M, N), 1.5, 6)
    uf = u.float().requires_grad_(True)
    torch.nn.functional.gelu(uf).sum().backward()
    _close(ops.gemm(a, b, epilogue=ops.EPI_DGELU, aux=u, block_n=bn), (v - bias) * uf.grad, 2 ** -6, 2e-2, "dgelu")
    _close(ops.gemm(a, b, epilogue=ops.EPI_DRELU, aux=u, block_n=bn), (v - bias) * (u.float() > 0), 2 ** -7, 1e-2, "drelu")
    _close(ops.gemm(a, b, alpha=0.125, block_n=bn), (v - bias) * 0.125, 2 ** -7, 1e-2, "alpha")


def test_gemm_k_extension_and_strided_a():
    ops = _ops()
    M, N, K, K2 = 900, 2304, 768, 64
    a, b = _rand((M, K), 1.0, 1), _rand((N, K), K ** -0.5, 2)
    a2, b2 = _rand((M, K2), 1.0, 3), _rand((N, K2), 0.1, 4)
    ref = a.float() @ b.float().t() + a2.float() @ b2.float().t()
    _close(ops.gemm(a, b, a2=a2, b2=b2), ref, 2 ** -7, 2e-2, "k-extension")
    # strided A: the CLS rows (row 0 of every 30-token item) of a [N_items*30, 768] activation
    items, L = 333, 30
    h = _rand((items * L, K), 1.0, 5)
    w = _rand((64, K), K ** -0.5, 6)
    cls = h.view(items, L, K)[:, 0]
    assert cls.stride(0) == L * K
    _close(ops.gemm(cls, w), cls.float() @ w.float().t(), 2 ** -7, 1e-2, "strided A")
    # strided C: write into column block of a wider buffer
    wide = torch.zeros((M, 1024), dtype=BF16, device="cuda")
    ops.gemm(a, b[:256], out=wide[:, 512:768])
    _close(wide[:, 512:768], a.float() @ b[:256].float().t(), 2 ** -7, 1e-2, "strided C")
    assert float(wide[:, :512].abs().max()) == 0.0 and float(wide[:, 768:].abs().max()) == 0.0


def test_gemm_rejects_bad_args():
    ops = _ops()
    a, b = _rand((64, 60), 1, 1), _rand((64, 60), 1, 2)  # K % 8 != 0
    with pytest.raises(RuntimeError, match="multiples of 8"):
        ops.gemm(a, b)


def _attn_ref(qkv, N, L, heads, dh, mask, causal, mask_neg):
    H = heads * dh
    q, k, v = [t.view(N, L, heads, dh).transpose(1, 2) for t in qkv.float().view(N * L, 3, H).unbind(1)]
    s = (q @ k.transpose(-1, -2)) * dh ** -0.5
    ok = torch.ones(N, 1, L, L, dtype=torch.bool, device=qkv.device)
    if mask is not None:
        ok = ok & (mask[:, :L] != 0).view(N, 1, 1, L)
    if causal:
        ok = ok & torch.tril(torch.ones(L, L, dtype=torch.bool, device=qkv.device))
    s = s + torch.where(ok, 0.0, mask_neg)
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(N * L, H)


@pytest.mark.parametrize("N,L,heads,dh,mask_kind,causal", [
    (37, 30, 12, 64, "int64", False), (5, 30, 12, 64, None, False), (64, 20, 2, 32, "f32", True),
    (9, 10, 2, 32, "f32", True), (3, 32, 4, 64, "int64", True), (2, 1, 2, 32, None, False),
    # mid-length kernel (ViT): L = 197 / 207 (+prompt) / 37 / 256, 64-wide heads, no causal mask
    (7, 197, 12, 64, None, False), (3, 207, 12, 64, None, False), (5, 37, 12, 64, "int64", False),
    (2, 256, 2, 64, None, False), (2, 64, 3, 64, "f32", False), (1, 33, 1, 64, None, False),
])
def test_attention_small_fwd_bwd(N, L, heads, dh, mask_kind, causal):
    ops = _ops()
    H = heads * dh
    qkv = _rand((N * L, 3 * H), 1.0, 7)
    mask = None
    if mask_kind is not None:
        g = torch.Generator(device="cuda").manual_seed(11)
        lens = torch.randint(0, L + 1, (N,), generator=g, device="cuda")  # includes fully masked rows (len 0)
        m = (torch.arange(L, device="cuda")[None, :] < lens[:, None])
        if causal:  # SASRec: left padding
            m = m.flip(1)
        mask = m.to(torch.int64 if mask_kind == "int64" else torch.float32)
        if mask_kind == "int64":  # the reference's [ids | mask] rows: pass the strided right half
            both = torch.zeros((N, 2 * L), dtype=torch.int64, device="cuda")
            both[:, L:] = mask
            mask = both[:, L:]
    mask_neg = -1e9 if causal else ops.F32_MIN
    qf = qkv.float().requires_grad_(True)
    ref = _attn_ref(qf, N, L, heads, dh, mask, causal, mask_neg)
    got, lse = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, want_lse=True)
    _close(got, ref.detach(), 2 ** -6, 2e-2, "attention fwd")
    dctx = _rand((N * L, H), 1.0, 8)
    ref.backward(dctx.float())
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, lse=lse, ctx=got)
    # probabilities and dS are rounded to bf16 before the second contraction: 2^-6 relative + small absolute
    _close(dqkv, qf.grad, 2 ** -5, 6e-2, "attention bwd")
    # aggregate accuracy per block (dq | dk | dv) and of their column sums (what bias gradients are made of)
    for j, nm in enumerate(("dq", "dk", "dv")):
        got, ref_g = dqkv[:, j * H:(j + 1) * H].float(), qf.grad[:, j * H:(j + 1) * H]
        rel = float((got - ref_g).norm() / (ref_g.norm() + 1e-20))
        assert rel <= 2e-2, "%s relative L2 error %.4f" % (nm, rel)
        if nm != "dk":   # the column sum of dk over a sequence is identically 0 (softmax shift invariance)
            cs, cr = got.sum(0), ref_g.sum(0)
            relc = float((cs - cr).norm() / (cr.norm() + 1e-20))
            assert relc <= 5e-2, "%s column-sum relative L2 error %.4f" % (nm, relc)


@pytest.mark.parametrize("M,H", [(1000, 768), (515, 64), (33, 256), (7, 128), (4099, 1024), (64, 512)])
def test_layernorm_fwd_bwd(M, H):
    ops = _ops()
    x, res = _rand((M, H), 1.0, 1), _rand((M, H), 1.0, 2)
    gamma, beta = 1 + 0.1 * _rand((H,), 1, 3, torch.float32), 0.1 * _rand((H,), 1, 4, torch.float32)
    y, z, mean, rstd = ops.layernorm_fwd(x, gamma, beta, 1e-12, res=res, want_z=True)
    zr = (x.float() + res.float())
    _close(z, zr, 2 ** -8, 1e-6, "z")
    zf = z.float().requires_grad_(True)
    gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(zf, (H,), gf, bf, 1e-12)
    _close(y, ref.detach(), 2 ** -7, 1e-2, "ln fwd")
    dy = _rand((M, H), 1.0, 5)
    ref.backward(dy.float())
    dg, db = torch.empty(H, device="cuda"), torch.empty(H, device="cuda")
    dz = ops.layernorm_bwd(dy, z, mean, rstd, gamma, dgamma=dg, dbeta=db)
    _close(dz, zf.grad, 2 ** -6, 2e-2, "ln bwd dz")
    _close(dg, gf.grad, 1e-3, 1e-2 * math.sqrt(M), "ln bwd dgamma")
    _close(db, bf.grad, 1e-3, 1e-2 * math.sqrt(M), "ln bwd dbeta")
    # broadcast residual (SASRec position embedding): res_rows = S
    S = 5 if M % 5 == 0 else 1
    pos = _rand((S, H), 1.0, 6)
    y2, _, _, _ = ops.layernorm_fwd(x, gamma, beta, 1e-6, res=pos)
    ref2 = torch.nn.functional.layer_norm(x.float() + pos.float().repeat(M // S, 1), (H,), gamma, beta, 1e-6)
    _close(y2, ref2, 2 ** -7, 1e-2, "ln fwd broadcast residual")


@pytest.mark.parametrize("roberta,prompt", [(False, 0), (True, 0), (False, 10), (True, 7)])
def test_embed_ln(roberta, prompt):
    ops = _ops()
    N, L, H, V, P = 50, 30, 768, 1000, 64
    g = torch.Generator(device="cuda").manual_seed(3)
    pad = 1 if roberta else 0
    ids = torch.randint(3, V, (N, L), generator=g, device="cuda")
    lens = torch.randint(2, L + 1, (N,), generator=g, device="cuda")
    ids = torch.where(torch.arange(L, device="cuda")[None] < lens[:, None], ids, torch.full_like(ids, pad))
    rows = torch.cat([ids, (ids != pad).long()], 1)  # the reference's [ids | mask] layout
    word, pos, typ = _rand((V, H), 0.02, 1), _rand((P, H), 0.02, 2), _rand((1, H), 0.02, 3)
    gamma, beta = 1 + 0.1 * _rand((H,), 1, 4, torch.float32), 0.1 * _rand((H,), 1, 5, torch.float32)
    pr = _rand((prompt, H), 0.02, 6) if prompt else None
    out, z, mean, rstd = ops.embed_ln_fwd(rows[:, :L], L, word, pos, typ[0], gamma, beta, 1e-5,
                                          roberta_pad_id=(1 if roberta else -1), prompt=pr, want_z=True)
    w = word.float()[ids]
    if prompt:
        w = torch.cat([pr.float()[None].expand(N, -1, -1), w[:, prompt:]], 1)
    if roberta:
        m = (ids != pad).long()
        pid = torch.cumsum(m, 1) * m + pad
    else:
        pid = torch.arange(L, device="cuda")[None].expand(N, -1)
    zr = w + pos.float()[pid] + typ.float()[0]
    ref = torch.nn.functional.layer_norm(zr, (H,), gamma, beta, 1e-5).view(N * L, H)
    _close(out, ref, 2 ** -6, 3e-2, "embed+ln")


def test_act_bwd_colsum():
    ops = _ops()
    dy, u = _rand((1000, 64), 1, 1), _rand((1000, 64), 1.5, 2)
    uf = u.float().requires_grad_(True)
    torch.nn.functional.gelu(uf).sum().backward()
    _close(ops.act_bwd(dy, u, "gelu"), dy.float() * uf.grad, 2 ** -6, 1e-2, "act_bwd gelu")
    _close(ops.act_bwd(dy, u, "relu"), dy.float() * (u.float() > 0), 2 ** -8, 1e-6, "act_bwd relu")
    x = _rand((5000, 2304), 1, 3)
    _close(ops.colsum(x), x.float().sum(0), 1e-4, 2e-2, "colsum")
    _close(ops.colsum(x[:, 768:1536]), x[:, 768:1536].float().sum(0), 1e-4, 2e-2, "colsum strided")
    for M, W in ((40960, 64), (4104, 16), (4097, 64)):      # narrow: rows folded 16 / 8 / 1 at a time
        xn = _rand((M, W), 1, 6)
        _close(ops.colsum(xn), xn.float().sum(0), 1e-4, 2e-2, "colsum narrow %dx%d" % (M, W))


@pytest.mark.parametrize("B,S,D,cpc", [(64, 20, 64, False), (7, 10, 256, False), (33, 20, 768, False), (16, 20, 64, True)])
def test_bce_loss(B, S, D, cpc):
    ops = _ops()
    prec = _rand((B, S, D), D ** -0.5, 1)
    emb = _rand((B, S + 1, 2, D), 1.0, 2)
    g = torch.Generator(device="cuda").manual_seed(5)
    lens = torch.randint(1, S + 1, (B,), generator=g, device="cuda")
    log_mask = (torch.arange(S, device="cuda")[None] >= (S - lens)[:, None]).float()
    pf, ef = prec.float().requires_grad_(True), emb.float().requires_grad_(True)
    pos, neg = ef[:, :, 0], ef[:, :, 1]
    ps, ns = (pf * pos[:, 1:]).sum(-1), (pf * neg[:, :-1]).sum(-1)
    bce = torch.nn.BCEWithLogitsLoss()
    if cpc:
        ref = bce(ps[:, -1], torch.ones(B, device="cuda")) + bce(ns[:, -1], torch.zeros(B, device="cuda"))
    else:
        idx = torch.where(log_mask != 0)
        ref = bce(ps[idx], torch.ones_like(ps[idx])) + bce(ns[idx], torch.zeros_like(ns[idx]))
    loss, count, p, n = ops.bce_loss_fwd(prec, emb.view(B, S + 1, 2, D), None if cpc else log_mask, cpc=cpc)
    assert abs(float(loss) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref))), (float(loss), float(ref))
    assert float(count) == (B if cpc else float(log_mask.sum()))
    ref.backward()
    go = torch.full((1,), 2.0, device="cuda")
    d_prec, d_emb = ops.bce_loss_bwd(prec, emb, None if cpc else log_mask, p, n, count, grad_out=go, cpc=cpc)
    _close(d_prec, 2 * pf.grad, 2 ** -7, 1e-6, "d_prec")
    _close(d_emb, 2 * ef.grad, 2 ** -7, 1e-6, "d_emb")


def test_adam_matches_torch():
    """torch.optim.Adam fed g · grad_scale, without and with weight decay (the reference's --l2_weight): the decay term is
    added to the SCALED gradient"""
    ops = _ops()
    n = 100003
    p0 = _rand((n,), 1, 1, torch.float32)
    for wd in (0.0, 0.01):
        p = p0.clone()
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        ref = torch.nn.Parameter(p0.clone())
        opt = torch.optim.Adam([ref], lr=1e-3, weight_decay=wd)
        for step in range(1, 4):
            g = _rand((n,), 1, 10 + step, torch.float32)
            ref.grad = g.clone()
            opt.step()
            ops.adam_step(p, g * 4, m, v, 1e-3, 0.9, 0.999, 1e-8, wd, step, grad_scale=0.25)
        _close(p, ref.detach(), 1e-6, 1e-6, "adam weight_decay=%g" % wd)


def test_adam_dev_is_bit_identical_to_adam_step():
    """a4r_adam_step_dev (bias corrections read from device memory: the form a CUDA-graph replay needs) against a4r_adam_step
    for the same step numbers: bit-identical parameters and moments."""
    ops = _ops()
    n = 70001
    p0 = _rand((n,), 1, 1, torch.float32)
    pa, pb = p0.clone(), p0.clone()
    ma, va, mb, vb = (torch.zeros_like(p0) for _ in range(4))
    bc = torch.zeros(2, dtype=torch.float32, device="cuda")
    for step in (1, 2, 3, 1000, 123456):
        g = _rand((n,), 1, 20 + step % 97, torch.float32)
        ops.adam_step(pa, g, ma, va, 1e-3, 0.9, 0.999, 1e-8, 0.01, step, grad_scale=0.5)
        bc.copy_(torch.tensor(ops.adam_bias_corrections(0.9, 0.999, step), dtype=torch.float32))
        ops.adam_step_dev(pb, g, mb, vb, 1e-3, 0.9, 0.999, 1e-8, 0.01, bc, grad_scale=0.5)
        assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), step


def test_trainer_resumes_from_a_reference_format_optimizer_checkpoint():
    """SURVEY.md 8f-4 "checkpoint I/O compatibility", the GPU half: moments + step written by torch.optim.Adam (the format
    data_utils/utils.py:109-115 stores) are loaded into FlatAdamTrainer, then both take two more steps on the same gradients:
    the flat fused Adam continues exactly where torch's left off (fp32 rounding: 1e-6)."""
    from adapter4rec_b200.trainer import FlatAdamTrainer
    torch.manual_seed(11)

    def make():
        torch.manual_seed(11)
        return torch.nn.ModuleDict({
            "bert_encoder": torch.nn.ModuleDict({"adapter": torch.nn.Linear(96, 64), "query": torch.nn.Linear(96, 128)}),
            "user_encoder": torch.nn.ModuleDict({"lora_x": torch.nn.Linear(64, 8, bias=False), "fc": torch.nn.Linear(128, 96)})
        }).cuda()

    ref, mine = make(), make()
    groups = {"bert": [], "recsys": [], "adapter_bert": [], "adapter_recsys": []}
    for name, p in ref.named_parameters():
        ad = "adapter" in name or "lora" in name
        groups[("adapter_bert" if ad else "bert") if 'bert_encoder' in name else ("adapter_recsys" if ad else "recsys")].append(p)
    opt = torch.optim.Adam([{'params': groups["bert"], 'lr': 2e-3}, {'params': groups["recsys"], 'lr': 1e-3},
                            {'params': groups["adapter_bert"], 'lr': 3e-3}, {'params': groups["adapter_recsys"], 'lr': 4e-3}])
    g = torch.Generator(device="cuda").manual_seed(3)

    def grads():
        return [torch.randn(p.shape, generator=g, device="cuda") for p in ref.parameters()]

    for _ in range(3):
        for p, gr in zip(ref.parameters(), grads()):
            p.grad = gr
        opt.step()
    mine.load_state_dict(ref.state_dict())
    tr = FlatAdamTrainer(mine, 1e-3, 2e-3, 3e-3, 4e-3)
    tr.load_state_dict(opt.state_dict())
    assert tr.step_count == 3
    for _ in range(2):
        gs = grads()
        for p, q, gr in zip(ref.parameters(), mine.parameters(), gs):
            p.grad = gr
            q.grad.copy_(gr)                       # .grad of a trainer parameter is a view of the flat gradient buffer
        opt.step()
        tr.optimizer_step()
    assert tr.step_count == 5
    for (n, a), b in zip(ref.named_parameters(), mine.parameters()):
        _close(b.detach(), a.detach(), 1e-6, 1e-6, n)
    back = tr.state_dict()
    for i, p in enumerate(q for grp in opt.param_groups for q in grp["params"]):
        _close(back["state"][i]["exp_avg"], opt.state[p]["exp_avg"], 1e-6, 1e-7, "exp_avg %d" % i)
        assert float(back["state"][i]["step"]) == 5.0


@pytest.mark.parametrize("M,H,r,act,tail", [
    (128, 768, 64, "relu", 0), (1000, 768, 64, "gelu", 0), (148 * 128 + 77, 768, 64, "relu", 0),
    (300, 128, 16, "relu", 0), (300, 128, 16, "gelu", 0), (515, 256, 8, "relu", 0), (70, 64, 16, "relu", 0),
    (1000, 768, 64, "relu", 1), (1000, 768, 64, "gelu", 2), (333, 384, 48, "relu", 0),
])
def test_adapter_ln_fused(M, H, r, act, tail):
    """K5: the fused Houlsby block against the fp32 statement of model.py:292-297 / modules.py:131-134 on bf16-exact
    inputs.  s and z are rounded to bf16 inside the kernel exactly where the composed GEMM -> GEMM -> LayerNorm path
    rounds them, so the reference rounds there too; what is left is fp32 summation order and the final bf16 rounding."""
    ops = _ops()
    h = _rand((M, H), 1.0, 1)
    inp = _rand((M, H), 1.0, 2)
    wd, wu = _rand((r, H), 0.05, 3), _rand((H, r), 0.05, 4)
    bd, bu = _rand((r,), 0.1, 5, torch.float32), _rand((H,), 0.1, 6, torch.float32)
    g, b = 1 + _rand((H,), 0.1, 7, torch.float32), _rand((H,), 0.1, 8, torch.float32)
    eps = 1e-12
    out, z, mean, rstd, s, u = ops.adapter_ln_fwd(h, None if tail == 2 else inp, wd, bd, wu, bu, g, b, eps, act=act, tail=tail,
                                                  save=True)
    pre = h.float() @ wd.float().t() + bd
    s_ref = (torch.nn.functional.gelu(pre) if act == "gelu" else torch.relu(pre)).to(BF16)
    z_ref = s_ref.float() @ wu.float().t() + bu + h.float() + (0 if tail == 2 else inp.float())
    _close(s, s_ref, 2 ** -7, 1e-3, "s")
    if act == "gelu":
        _close(u, pre, 2 ** -7, 1e-3, "u")
    if tail != 0:
        _close(out, z_ref, 2 ** -7, 2e-2, "out (no LayerNorm)")
        return
    _close(z, z_ref, 2 ** -7, 2e-2, "z")
    zf = z.float()                                   # LayerNorm of the tensor the kernel itself rounded
    mu, var = zf.mean(-1), zf.var(-1, unbiased=False)
    _close(mean, mu, 1e-4, 1e-4, "mean")
    _close(rstd, (var + eps).rsqrt(), 1e-4, 1e-4, "rstd")
    ref = (zf - mu[:, None]) * (var[:, None] + eps).rsqrt() * g + b
    _close(out, ref, 2 ** -7, 1e-2, "out")
    out2 = ops.adapter_ln_fwd(h, inp, wd, bd, wu, bu, g, b, eps, act=act, tail=0, save=False)[0]
    assert torch.equal(out, out2), "the inference variant (z staged in `out`) must give identical results"


@pytest.mark.parametrize("M,N,K", [(5000, 768, 8), (3001, 8, 768), (4096, 768, 64), (777, 64, 768), (10240, 64, 16),
                                   (100, 16, 64), (6400, 768, 768), (4100, 3072, 768), (2050, 768, 3072), (64, 128, 256),
                                   (63, 136, 264), (0, 64, 64), (20000, 2304, 64)])
def test_wgrad(M, N, K):
    """tcgen05 weight gradient (MN-major operands, split over tokens): dW = alpha * A^T B against fp32 torch on the same
    bf16-rounded operands; tolerance = fp32 accumulation-order noise, sqrt(M)-scaled."""
    ops = _ops()
    a, b = _rand((M, N), 1, 4), _rand((M, K), 1, 5)
    ref = a.float().t() @ b.float()
    got = ops.wgrad(a, b, alpha=0.5)
    _close(got, 0.5 * ref, 1e-3, 2e-3 * math.sqrt(max(M, 1)), "wgrad %dx%dx%d" % (M, N, K))
    got2 = ops.wgrad(a, b, alpha=0.5, out=got.clone(), accumulate=True)
    _close(got2, ref, 1e-3, 4e-3 * math.sqrt(max(M, 1)), "wgrad accumulate")
    assert torch.equal(ops.wgrad(a, b, alpha=0.5), got), "fixed-order reduction must be deterministic"


def test_wgrad_strided_operands():
    ops = _ops()
    t = _rand((3000, 64), 1, 6)
    dq = _rand((3000, 2304), 1, 7)
    _close(ops.wgrad(dq[:, :768], t, k=8), dq[:, :768].float().t() @ t[:, :8].float(), 1e-3, 0.2, "wgrad sliced")
    _close(ops.wgrad(dq[:, 768:1536], dq[:, 1536:], n=768, k=768), dq[:, 768:1536].float().t() @ dq[:, 1536:].float(),
           1e-3, 0.3, "wgrad two column slices")


def test_scatter_add_rows_matches_embedding_backward():
    """dst[idx[r]] += src[r] with nn.Embedding's padding_idx semantics (the row never receives a gradient), negative and
    out-of-range indices skipped; fp32 accumulation of bf16 rows against torch.index_add_ on the same values."""
    ops = _ops()
    g = torch.Generator().manual_seed(3)
    R, H, V, pad = 20000, 768, 300, 1
    src = _rand((R, H), 1.0, 8)
    idx = torch.randint(-1, V + 2, (R,), generator=g).cuda()          # includes -1 and V, V+1 (skipped)
    got = ops.scatter_add_rows(src, idx, V, skip_idx=pad)
    ok = (idx >= 0) & (idx < V) & (idx != pad)
    ref = torch.zeros((V, H), dtype=torch.float32, device="cuda").index_add_(0, idx[ok], src.float()[ok])
    _close(got, ref, 1e-5, 1e-3, "scatter_add_rows")
    assert float(got[pad].abs().max()) == 0.0
    # a strided source (column slice) and an empty call
    wide = _rand((64, 2 * H), 1.0, 9)
    i2 = torch.arange(64).cuda() % 7
    _close(ops.scatter_add_rows(wide[:, H:], i2, 7), torch.zeros((7, H), device="cuda").index_add_(0, i2, wide[:, H:].float()),
           1e-5, 1e-3, "scatter_add_rows strided")
    assert ops.scatter_add_rows(src[:0], idx[:0], V).abs().sum() == 0


@pytest.mark.parametrize("kind,fn", [("leaky_relu", torch.nn.functional.leaky_relu),
                                     ("gelu_new", lambda x: torch.nn.functional.gelu(x, approximate="tanh")),
                                     ("gelu", torch.nn.functional.gelu), ("relu", torch.relu)])
def test_act_fwd_bwd_kinds(kind, fn):
    """stand-alone activations of the Pfeiffer (LeakyReLU 0.01) and Compacter (tanh-GELU) bottlenecks"""
    ops = _ops()
    u = _rand((1000, 64), 1.5, 11)
    dy = _rand((1000, 64), 1.0, 12)
    uf = u.float().requires_grad_(True)
    y = fn(uf)
    y.sum().backward()
    out = ops.act_fwd(u, kind)
    _close(out, y.detach(), 2 ** -7, 1e-2, "act_fwd " + kind)
    saved = out if kind in ("relu", "leaky_relu") else u       # what the backward is given (output vs pre-activation)
    _close(ops.act_bwd(dy, saved, kind), dy.float() * uf.grad, 2 ** -6, 1e-2, "act_bwd " + kind)


def test_layernorm_bwd_add_fuses_the_skip_gradient():
    """a4r_layernorm_bwd_add == a4r_layernorm_bwd followed by `+ dskip` (fp32 sum, one bf16 rounding)."""
    from adapter4rec_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    for M, H in ((1000, 768), (333, 64), (77, 128)):
        x = torch.randn((M, H), generator=g, device="cuda").to(torch.bfloat16)
        dy = torch.randn((M, H), generator=g, device="cuda").to(torch.bfloat16)
        dskip = torch.randn((M, H), generator=g, device="cuda").to(torch.bfloat16)
        gamma = torch.rand(H, generator=g, device="cuda") + 0.5
        beta = torch.zeros(H, device="cuda")
        _, _, mean, rstd = ops.layernorm_fwd(x, gamma, beta, 1e-6, want_stats=True)
        fused = ops.layernorm_bwd_add(dy, x, mean, rstd, gamma, dskip)
        xr = x.float().requires_grad_(True)
        torch.nn.functional.layer_norm(xr, (H,), gamma, beta, 1e-6).backward(dy.float())
        ref = xr.grad + dskip.float()
        err = (fused.float() - ref).abs()
        assert bool((err <= 2e-2 + 8e-3 * ref.abs()).all()), (M, H, float(err.max()))


def _run_tool(*argv, timeout=600):
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", argv[0])] + list(argv[1:]), capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0 and r.stdout.strip().endswith("ALL OK"), (r.stdout[-1500:], r.stderr[-1500:])


def test_adapter_block_matches_torch():
    """K5 (a4r_adapter_ln_fwd, adapter_rows_sm100.cu): tools/k5_check.py runs every tail x activation x save combination at
    M = 128 / 1,000 / 20,000 (ragged last tile, several tiles per CTA) against torch."""
    _run_tool("k5_check.py")


def test_adapter_block_at_the_benchmarked_row_counts():
    """K5 at M = 161,280 (8.5 tiles per persistent CTA: C1 at 128 users per pass) and M = 645,120 (+ a ragged 645,197): the
    multi-tile ring / phase path the benchmark runs, every row against torch fp32, both ViT tails, both activations, save on
    and off."""
    _run_tool("k5_check.py", "--big", timeout=900)


def test_vit_attention_tcgen05_forward_and_backward():
    """attention_tc_sm100.cu / attention_tc_bwd_sm100.cu (a4r_attn_mid_fwd / _bwd, unmasked): L = 33 ... 256 incl. every tile
    boundary (112 / 113 / 128 / 129), 197 and 207 at several batch sizes, inputs 6x larger (scores of +-100 nats), and rows
    whose maximum sits 116 nats ahead in a LATER register block (the lazily raised softmax shift) — context, log-sum-exp and
    dq | dk | dv against fp64 torch."""
    _run_tool("attn_tc_check.py", "--bwd", timeout=600)


@pytest.mark.parametrize("rows,cols", [(768, 768), (3072, 768), (64, 768), (768, 64), (30522, 768), (37, 101), (1, 8)])
def test_cast_transpose_matches_torch(rows, cols):
    """a4r_cast_transpose_f32_bf16 (the weight caches): bf16 copy and bf16 transpose of an fp32 matrix, bit-equal to torch's
    round-to-nearest-even cast, incl. ragged tiles, a row-strided source and either output alone."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(rows * 7 + cols)
    base = torch.randn(rows, cols + 8, generator=g, device="cuda")
    for w in (base[:, :cols].contiguous(), base[:, :cols]):
        ref = w.to(torch.bfloat16)
        a, at = ops.cast_transpose(w, True, True)
        assert torch.equal(a, ref) and torch.equal(at, ref.t().contiguous())
        a2, none_t = ops.cast_transpose(w, True, False)
        none_a, at2 = ops.cast_transpose(w, False, True)
        assert none_t is None and none_a is None and torch.equal(a2, ref) and torch.equal(at2, ref.t().contiguous())


def test_vit_attention_tcgen05_repeated_launches_are_bit_identical():
    """The tcgen05 attention forward and backward use no atomics: ~1,000 launches over five shapes (197 / 207 / 256 / 129 / 64
    tokens) must each reproduce the first launch bit for bit — the check for hand-over races (per-warp TMA result boxes,
    tensor-memory column reuse, mbarrier phases, converged-warp issue) that a single launch cannot be relied on to show."""
    _run_tool("attn_stress.py", "60", timeout=600)


def test_adapter_block_repeated_launches_are_bit_identical_and_correct():
    """900 launches of the default K5 kernel at M = 161,280 (300 per tail), each compared element-wise with one torch fp32
    reference and bit-wise with the first launch: the epilogue / TMA-refill race fixed in round 2 corrupted a few rows in 1-3 % of
    such launches, which no single-launch test can be relied on to see."""
    _run_tool("k5_stress.py", "161280", "300", timeout=900)


@pytest.mark.parametrize("M,N,K,K2,epi", [(645120, 768, 3072, 0, "res"), (645120, 3072, 768, 0, "gelu"),
                                          (645120, 2304, 768, 64, "linear"), (645120, 768, 768, 0, "res"),
                                          (645120, 768, 3072, 0, "dgelu"), (161280 + 333, 3072, 768, 0, "dgelu")])
def test_gemm_at_the_benchmarked_row_counts(M, N, K, K2, epi):
    """The five GEMM shapes of the C2 step at the benchmarked M = 645,120 (one 512-user pass: 2,520 256-row tiles = 34 tiles per
    CTA pair, byte offsets past 2^31 in A and C), a strided sample of 4,099 rows (stride 157 + the first and last 256 rows)
    against torch fp32 on the same operands, plus an all-rows finiteness / magnitude check."""
    ops = _ops()
    a, b = _rand((M, K), 1.0, 1), _rand((N, K), K ** -0.5, 2)
    bias = _rand((N,), 0.5, 3, torch.float32)
    rows = torch.cat([torch.arange(0, 256), torch.arange(256, M - 256, 157), torch.arange(M - 256, M)]).cuda()
    kw, ref = {}, a[rows].float() @ b.float().t()
    if K2:
        a2, b2 = _rand((M, K2), 1.0, 4), _rand((N, K2), 0.1, 5)
        kw.update(a2=a2, b2=b2)
        ref = ref + a2[rows].float() @ b2.float().t()
    if epi in ("res", "linear", "gelu"):
        kw["bias"] = bias
        ref = ref + bias
    if epi == "res":
        res = _rand((M, N), 1.0, 6)
        kw["residual"] = res
        ref = ref + res[rows].float()
    aux = None
    if epi == "gelu":
        aux = torch.empty((M, N), dtype=BF16, device="cuda")
        kw.update(epilogue=ops.EPI_GELU, aux=aux)
    if epi == "dgelu":
        aux = _rand((M, N), 1.5, 7)
        kw.update(epilogue=ops.EPI_DGELU, aux=aux)
        uf = aux[rows].float().requires_grad_(True)
        torch.nn.functional.gelu(uf).sum().backward()
        ref = ref * uf.grad
    got = ops.gemm(a, b, **kw)
    if epi == "gelu":
        _close(aux[rows], ref, 2 ** -7, 1e-2, "pre-activation at M=%d" % M)
        ref = torch.nn.functional.gelu(ref)
    _close(got[rows], ref, 2 ** -6 if epi == "dgelu" else 2 ** -7, 2e-2, "gemm %s at M=%d N=%d K=%d" % (epi, M, N, K))
    assert bool(torch.isfinite(got).all())
    # every row block of 8,192 rows must carry the magnitude the sampled rows carry (a skipped or doubled tile would not)
    blocks = got.float().pow(2).view(-1, N)[: (M // 8192) * 8192].view(-1, 8192 * N).mean(1).sqrt()
    rms = float(ref.pow(2).mean().sqrt())
    assert float(blocks.min()) > 0.8 * rms and float(blocks.max()) < 1.25 * rms, (float(blocks.min()), float(blocks.max()), rms)
