"""-m gpu: the train-mode kernel paths at the sizes the C2 step runs them (BERT-base + LoRA, 512 users per pass: 21,504
item sequences of 30 tokens = 645,120 token rows; SASRec over 512 users x 20 positions; dropout 0.1 everywhere).

At these sizes every grid-stride / persistent loop runs many iterations (attention: 258,048 (sequence, head) pairs on at
most SMs x 8 blocks x 4 warps; LayerNorm backward: 645,120 rows on one wave of 4,736 / 14,208), and the dropout counters
pass 2^32.  Each kernel is compared, one at a time, with an fp32 (or fp64) torch statement of the same operation that
applies the mask the kernel must have drawn, rebuilt on the GPU by tests/dropout_rng.py.  Where dropping an element
changes the result by less than a bf16 tolerance, the mask is also read back exactly."""
import math

import pytest
import torch

import dropout_rng as R
from test_kernels_gpu import _close, _rand

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
P = 0.1
SEED = (1 << 47) | 0x5EEDA4D2            # DropoutState keeps seeds below 2^48
BIG_OFF = (1 << 32) + 12345              # where an eager C2 run's counter is from its second step on
C2_ITEMS, C2_TOKENS = 21504, 30          # item sequences and tokens per sequence of one 512-user pass
C2_ROWS = C2_ITEMS * C2_TOKENS           # 645,120


def _ops():
    from adapter4rec_b200 import ops
    return ops


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _lengths(N, L, seed, lo=1):
    """ragged sequence lengths with a zero-length (fully masked, padding-item) sequence every 97"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    lens = torch.randint(lo, L + 1, (N,), generator=g, device="cuda")
    lens[::97] = 0
    return lens


def _allowed(key_ok, causal, n, L, dev):
    """[n, 1, L, L] bool: key j may be attended by query i (before the fully-masked-row rule)"""
    ok = torch.ones(n, 1, L, L, dtype=torch.bool, device=dev)
    if key_ok is not None:
        ok = ok & key_ok.view(n, 1, 1, L)
    if causal:
        ok = ok & torch.tril(torch.ones(L, L, dtype=torch.bool, device=dev))
    return ok


def _attn_ref(qf, n, L, heads, dh, key_ok, causal, mask_neg, keep, scale):
    """fp32 attention of the short-sequence kernel with probability dropout: qf [n*L, 3*heads*dh], key_ok [n, L] bool or
    None, keep [n, heads, L, L] bool.  One additive mask_neg per excluded key, so a query with every key excluded is
    uniform over all L keys, as in the reference."""
    H = heads * dh
    q, k, v = [t.view(n, L, heads, dh).transpose(1, 2) for t in qf.view(n * L, 3, H).unbind(1)]
    s = (q @ k.transpose(-1, -2)) * scale + torch.where(_allowed(key_ok, causal, n, L, qf.device), 0.0, mask_neg)
    pr = torch.softmax(s, -1) * keep * R.keep_scale(P)
    return (pr @ v).transpose(1, 2).reshape(n * L, H)


def _valid_keys(key_ok, causal, mask_neg, n, L, dev):
    """[n, 1, L, L] bool: probability (i, j) is non-zero (the softmax of the additive mask alone)"""
    return torch.softmax(torch.where(_allowed(key_ok, causal, n, L, dev), 0.0, mask_neg), -1) > 0


class _RelL2:
    """relative L2 error of dq | dk | dv accumulated over chunks"""

    def __init__(self):
        self.err, self.ref = [0.0] * 3, [0.0] * 3

    def add(self, got, ref, H):
        for j in range(3):
            a, b = got[:, j * H:(j + 1) * H].float(), ref[:, j * H:(j + 1) * H]
            self.err[j] += float((a - b).pow(2).sum())
            self.ref[j] += float(b.pow(2).sum())

    def check(self, what):
        for j, nm in enumerate(("dq", "dk", "dv")):
            rel = math.sqrt(self.err[j] / self.ref[j])
            assert rel <= 2e-2, "%s: %s relative L2 error %.4f" % (what, nm, rel)


def _attention_against_fp32(qkv, dctx, N, L, heads, dh, mask, key_ok, causal, mask_neg, off, chunk, scale=None):
    """kernel forward and backward over all N sequences against _attn_ref, every row, `chunk` sequences at a time, with
    the tolerances of test_attention_small_fwd_bwd"""
    ops = _ops()
    H = heads * dh
    drop = (P, SEED, off)
    got = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop)
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop)
    rel = _RelL2()
    for n0 in range(0, N, chunk):
        n1 = min(N, n0 + chunk)
        r0, r1 = n0 * L, n1 * L
        keep = R.prob_keep(SEED, off, P, torch.arange(n0, n1, device="cuda"), heads, L)
        qf = qkv[r0:r1].float().requires_grad_(True)
        ref = _attn_ref(qf, n1 - n0, L, heads, dh, None if key_ok is None else key_ok[n0:n1], causal, mask_neg, keep,
                        dh ** -0.5 if scale is None else scale)
        _close(got[r0:r1], ref.detach(), 2 ** -6, 2e-2, "attention fwd, sequences %d..%d" % (n0, n1))
        ref.backward(dctx[r0:r1].float())
        _close(dqkv[r0:r1], qf.grad, 2 ** -5, 6e-2, "attention bwd, sequences %d..%d" % (n0, n1))
        rel.add(dqkv[r0:r1], qf.grad, H)
        del keep, qf, ref
    rel.check("attention bwd")


def _attention_mask_readback(N, L, heads, dh, mask, key_ok, causal, mask_neg, off, chunk):
    """The keep bits themselves.  With q = k = 0 the probabilities are uniform over the valid keys; v[token j] = e_j makes
    ctx[i, j] = P'(i, j) (dropped: exactly 0), and dctx[token i] = e_i makes dv[j, i] = P'(i, j) as the backward
    regenerated it.  A wrong keep bit moves ctx by only ~1/L of a value, inside a bf16 tolerance; here it cannot hide."""
    ops = _ops()
    assert dh >= L
    H = heads * dh
    eye = torch.eye(L, dh, dtype=BF16, device="cuda")[None, :, None, :]
    qkv = torch.zeros((N * L, 3 * H), dtype=BF16, device="cuda")
    qkv.view(N, L, 3, heads, dh)[:, :, 2] = eye
    dctx = torch.zeros((N * L, H), dtype=BF16, device="cuda")
    dctx.view(N, L, heads, dh)[:] = eye
    drop = (P, SEED, off)
    ctx = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop)
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop)
    fwd = ctx.view(N, L, heads, dh)[..., :L].permute(0, 2, 1, 3)                 # [n, h, i, j]
    bwd = dqkv.view(N, L, 3, heads, dh)[:, :, 2, :, :L].permute(0, 2, 3, 1)     # dv[n, j, h, i] -> [n, h, i, j]
    for n0 in range(0, N, chunk):
        n1 = min(N, n0 + chunk)
        keep = R.prob_keep(SEED, off, P, torch.arange(n0, n1, device="cuda"), heads, L)
        want = keep & _valid_keys(None if key_ok is None else key_ok[n0:n1], causal, mask_neg, n1 - n0, L, "cuda")
        for got, what in ((fwd[n0:n1] != 0, "forward (ctx)"), (bwd[n0:n1] != 0, "backward (dv)")):
            bad = got != want
            assert not bool(bad.any()), "%s keeps %d probabilities the restated mask does not, drops %d it keeps (sequences %d..%d)" % (
                what, int((bad & got).sum()), int((bad & want).sum()), n0, n1)
        del keep, want


def _bert_mask(lens, L):
    """the reference's int64 [ids | mask] rows: the mask is their strided right half (right-padded)"""
    key_ok = torch.arange(L, device="cuda")[None, :] < lens[:, None]
    both = torch.zeros((lens.numel(), 2 * L), dtype=torch.int64, device="cuda")
    both[:, L:] = key_ok.long()
    return key_ok, both[:, L:]


def test_attention_bert_shape_against_fp32():
    """BERT: 21,504 sequences x 30 tokens x 12 heads of 64 (~55 (sequence, head) pairs per warp), int64 strided key mask,
    ragged lengths incl. zero, p = 0.1, counters past 2^32"""
    N, L, heads, dh = C2_ITEMS, C2_TOKENS, 12, 64
    key_ok, mask = _bert_mask(_lengths(N, L, 11), L)
    qkv = _rand((N * L, 3 * heads * dh), 1.0, 7)
    dctx = _rand((N * L, heads * dh), 1.0, 8)
    _attention_against_fp32(qkv, dctx, N, L, heads, dh, mask, key_ok, False, _ops().F32_MIN, BIG_OFF, 3072)
    del qkv, dctx
    _free()


def test_attention_bert_shape_mask_readback():
    N, L, heads, dh = C2_ITEMS, C2_TOKENS, 12, 64
    key_ok, mask = _bert_mask(_lengths(N, L, 11), L)
    _attention_mask_readback(N, L, heads, dh, mask, key_ok, False, _ops().F32_MIN, BIG_OFF, 3072)
    _free()


def _sasrec_mask(N, L):
    """SASRec's f32 log_mask: left-padded"""
    key_ok = (torch.arange(L, device="cuda")[None, :] < _lengths(N, L, 13)[:, None]).flip(1)
    return key_ok, key_ok.float()


@pytest.mark.parametrize("off", [777, BIG_OFF])
def test_attention_sasrec_shape(off):
    """SASRec: 512 users x 20 positions x 2 heads of 32, causal, f32 left-padded mask, mask_neg = -1e9"""
    N, L, heads, dh = 512, 20, 2, 32
    key_ok, mask = _sasrec_mask(N, L)
    qkv = _rand((N * L, 3 * heads * dh), 1.0, 9)
    dctx = _rand((N * L, heads * dh), 1.0, 10)
    _attention_against_fp32(qkv, dctx, N, L, heads, dh, mask, key_ok, True, -1e9, off, N)
    _attention_mask_readback(N, L, heads, dh, mask, key_ok, True, -1e9, off, N)


def test_attention_narrow_heads_zero_padded_to_32():
    """8-wide heads (K-adapter inside SASRec) zero-padded into the kernel's 32-wide slots with the temperature of the true
    width (model/modules.py): equal to the 8-wide attention, and the padding columns of ctx and dq | dk | dv stay 0"""
    ops = _ops()
    N, L, heads, d, w = 512, 20, 2, 8, 32
    key_ok, mask = _sasrec_mask(N, L)
    qkv8 = _rand((N * L, 3 * heads * d), 1.0, 14)
    dctx8 = _rand((N * L, heads * d), 1.0, 15)
    qkv = torch.nn.functional.pad(qkv8.view(-1, 3 * heads, d), (0, w - d)).reshape(-1, 3 * heads * w)
    dctx = torch.nn.functional.pad(dctx8.view(-1, heads, d), (0, w - d)).reshape(-1, heads * w)
    drop = (P, SEED, BIG_OFF)
    got = ops.attn_small_fwd(qkv, N, L, heads, w, mask=mask, causal=True, mask_neg=-1e9, dropout=drop, scale=d ** -0.5)
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, w, mask=mask, causal=True, mask_neg=-1e9, dropout=drop,
                              scale=d ** -0.5)
    got, dqkv = got.view(-1, heads, w), dqkv.view(-1, 3 * heads, w)
    assert bool((got[..., d:] == 0).all()) and bool((dqkv[..., d:] == 0).all())
    keep = R.prob_keep(SEED, BIG_OFF, P, torch.arange(N, device="cuda"), heads, L)
    qf = qkv8.float().requires_grad_(True)
    ref = _attn_ref(qf, N, L, heads, d, key_ok, True, -1e9, keep, d ** -0.5)
    _close(got[..., :d].reshape(-1, heads * d), ref.detach(), 2 ** -6, 2e-2, "narrow-head attention fwd")
    ref.backward(dctx8.float())
    _close(dqkv[..., :d].reshape(-1, 3 * heads * d), qf.grad, 2 ** -5, 6e-2, "narrow-head attention bwd")
    rel = _RelL2()
    rel.add(dqkv[..., :d].reshape(-1, 3 * heads * d), qf.grad, heads * d)
    rel.check("narrow-head attention bwd")


def test_packed_attention_train_mode():
    """The unpadded token layout (PackedTokens, cu_seqlens) with dropout at the C2 size.  Its dropout counters are indexed
    by (sequence, head, query, key) as in the padded layout, and a masked key or padded query adds exact zeros there, so:
    forward bit-identical to the padded kernel at every kept token; backward bit-identical when the padded rows' dctx is
    zero; both against fp32."""
    from adapter4rec_b200.model.bert import PackedTokens
    ops = _ops()
    N, L, heads, dh = C2_ITEMS, C2_TOKENS, 12, 64
    H = heads * dh
    key_ok = torch.arange(L, device="cuda")[None, :] < _lengths(N, L, 16)[:, None]
    fmask = key_ok.float()
    pk = PackedTokens(fmask)
    rows = pk.token_rows
    assert pk.num_tokens < N * L
    qkv = _rand((N * L, 3 * H), 1.0, 17)
    kept = torch.zeros(N * L, dtype=torch.bool, device="cuda")
    kept[rows] = True
    dctx = torch.where(kept[:, None], _rand((N * L, H), 1.0, 18), torch.zeros((), dtype=BF16, device="cuda"))
    drop = (P, SEED, BIG_OFF)
    kw = dict(causal=False, mask_neg=ops.F32_MIN, dropout=drop)
    qkv_p, dctx_p = qkv[rows].contiguous(), dctx[rows].contiguous()
    ctx_pad = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=fmask, **kw)
    ctx_pk = ops.attn_small_fwd(qkv_p, N, L, heads, dh, mask=pk.token_mask, cu_seqlens=pk.cu_seqlens, **kw)
    assert torch.equal(ctx_pk, ctx_pad[rows]), "packed forward differs from the padded one at %d elements" % int(
        (ctx_pk != ctx_pad[rows]).sum())
    d_pad = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=fmask, **kw)
    d_pk = ops.attn_small_bwd(qkv_p, dctx_p, N, L, heads, dh, mask=pk.token_mask, cu_seqlens=pk.cu_seqlens, **kw)
    for j, nm in enumerate(("dq", "dk", "dv")):
        a, b = d_pk[:, j * H:(j + 1) * H], d_pad[rows, j * H:(j + 1) * H]
        assert torch.equal(a, b), "packed %s differs from the padded one at %d elements" % (nm, int((a != b).sum()))
    del ctx_pad, d_pad
    cu = pk.cu_seqlens.tolist()
    rel = _RelL2()
    chunk = 3072
    for n0 in range(0, N, chunk):
        n1 = min(N, n0 + chunk)
        r0, r1 = n0 * L, n1 * L
        keep = R.prob_keep(SEED, BIG_OFF, P, torch.arange(n0, n1, device="cuda"), heads, L)
        qf = qkv[r0:r1].float().requires_grad_(True)
        ref = _attn_ref(qf, n1 - n0, L, heads, dh, key_ok[n0:n1], False, ops.F32_MIN, keep, dh ** -0.5)
        ref.backward(dctx[r0:r1].float())
        sel = rows[cu[n0]:cu[n1]] - r0
        _close(ctx_pk[cu[n0]:cu[n1]], ref.detach()[sel], 2 ** -6, 2e-2, "packed attention fwd")
        _close(d_pk[cu[n0]:cu[n1]], qf.grad[sel], 2 ** -5, 6e-2, "packed attention bwd")
        rel.add(d_pk[cu[n0]:cu[n1]], qf.grad[sel], H)
        del keep, qf, ref
    rel.check("packed attention bwd")
    del qkv, dctx, qkv_p, dctx_p, ctx_pk, d_pk
    _free()


LN_SHAPES = [(C2_ROWS, 768)] + [(M, H) for M in (77, 1000, 4099) for H in (64, 128, 768, 1024)]


@pytest.mark.parametrize("wgrad", [True, False])
@pytest.mark.parametrize("M,H", LN_SHAPES)
def test_layernorm_bwd_dropout_mask(M, H, wgrad):
    """a4r_layernorm_bwd with masked = (p, seed, offset): dz against fp32 torch, dz_masked exactly 0 wherever the restated
    mask drops and dz * scale within one bf16 rounding of each where it keeps; dgamma / dbeta (the trainable-LayerNorm
    instantiation; without them the frozen one runs) against fp64 sums, accumulated onto non-zero values, and
    bit-identical from launch to launch."""
    ops = _ops()
    off = BIG_OFF if H != 64 else 5
    x, dy = _rand((M, H), 1.0, 1), _rand((M, H), 1.0, 5)
    gamma, beta = 1 + 0.1 * _rand((H,), 1, 3, torch.float32), 0.1 * _rand((H,), 1, 4, torch.float32)
    _, _, mean, rstd = ops.layernorm_fwd(x, gamma, beta, 1e-12)
    dg = db = None
    if wgrad:
        dg, db = torch.empty(H, device="cuda"), torch.empty(H, device="cuda")
    masked = (P, SEED, off)
    dz, dzm = ops.layernorm_bwd(dy, x, mean, rstd, gamma, dgamma=dg, dbeta=db, masked=masked)
    s = R.keep_scale(P)
    sdg = torch.zeros(H, dtype=torch.float64, device="cuda")
    sdb = torch.zeros(H, dtype=torch.float64, device="cuda")
    chunk = 65536
    for r0 in range(0, M, chunk):
        r1 = min(M, r0 + chunk)
        xf = x[r0:r1].float().requires_grad_(True)
        gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
        ref = torch.nn.functional.layer_norm(xf, (H,), gf, bf, 1e-12)
        ref.backward(dy[r0:r1].float())
        _close(dz[r0:r1], xf.grad, 2 ** -6, 2e-2, "ln bwd dz, rows %d..%d" % (r0, r1))
        sdg += gf.grad.double()
        sdb += bf.grad.double()
        keep = R.element_keep(SEED, off, P, torch.arange(r0, r1, device="cuda"), H)
        m = dzm[r0:r1].float()
        assert bool((m[~keep] == 0).all()), "dz_masked non-zero at %d dropped elements (rows %d..%d)" % (
            int((m[~keep] != 0).sum()), r0, r1)
        want = dz[r0:r1].float() * s
        err = (m - want).abs()[keep]
        tol = (2 ** -7 * 1.01 * want.abs())[keep]
        assert bool((err <= tol).all()), "dz_masked != dz * scale at %d kept elements (rows %d..%d)" % (
            int((err > tol).sum()), r0, r1)
        del xf, ref, keep, m, want, err, tol
    if not wgrad:
        return
    _close(dg, sdg.float(), 1e-3, 1e-2 * math.sqrt(M), "ln bwd dgamma")
    _close(db, sdb.float(), 1e-3, 1e-2 * math.sqrt(M), "ln bwd dbeta")
    start_g, start_b = _rand((H,), 1.0, 6, torch.float32), _rand((H,), 1.0, 7, torch.float32)
    dg2, db2 = start_g.clone(), start_b.clone()
    dz2, dzm2 = ops.layernorm_bwd(dy, x, mean, rstd, gamma, dgamma=dg2, dbeta=db2, accumulate=True, masked=masked)
    assert torch.equal(dg2, start_g + dg) and torch.equal(db2, start_b + db), "accumulate=True"
    assert torch.equal(dz2, dz) and torch.equal(dzm2, dzm)
    if M == C2_ROWS:
        dg3, db3 = torch.empty(H, device="cuda"), torch.empty(H, device="cuda")
        ops.layernorm_bwd(dy, x, mean, rstd, gamma, dgamma=dg3, dbeta=db3, masked=masked)
        assert torch.equal(dg3, dg) and torch.equal(db3, db), "dgamma / dbeta must be bit-identical from launch to launch"
    del x, dy, dz, dzm, dz2, dzm2
    _free()


def _sample_rows(M):
    """the first and last 256 rows and every 157th row between them"""
    return torch.cat([torch.arange(0, 256), torch.arange(256, M - 256, 157), torch.arange(M - 256, M)]).cuda()


@pytest.mark.parametrize("after", [False, True])
def test_gemm_dropout_epilogue_at_the_benchmarked_row_count(after):
    """BertSelfOutput.dense at M = 645,120: dropout(x Wᵀ + b) + residual (forward), and the DROPSUM form that masks
    (x Wᵀ + b + residual) (the Houlsby backward), counters past 2^32.  A row sample against fp32; over the WHOLE output,
    a dropped element is exactly the residual (forward) or exactly 0 (DROPSUM)."""
    ops = _ops()
    M, N, K = C2_ROWS, 768, 768
    a, w = _rand((M, K), 1.0, 1), _rand((N, K), K ** -0.5, 2)
    bias = _rand((N,), 0.5, 3, torch.float32)
    res = _rand((M, N), 1.0, 6)
    out = ops.gemm(a, w, bias=bias, residual=res, dropout=(P, SEED, BIG_OFF), dropout_after=after)
    s = R.keep_scale(P)
    rows = _sample_rows(M)
    keep = R.element_keep(SEED, BIG_OFF, P, rows, N)
    v = a[rows].float() @ w.float().t() + bias
    ref = (v + res[rows].float()) * keep * s if after else v * keep * s + res[rows].float()
    _close(out[rows], ref, 2 ** -7, 2e-2, "gemm dropout epilogue (after=%s) at M=%d" % (after, M))
    del v, ref, keep
    for r0 in range(0, M, 65536):
        r1 = min(M, r0 + 65536)
        drop = ~R.element_keep(SEED, BIG_OFF, P, torch.arange(r0, r1, device="cuda"), N)
        o = out[r0:r1][drop]
        want = torch.zeros_like(o) if after else res[r0:r1][drop]
        assert bool((o == want).all()), "%d dropped elements are not %s (rows %d..%d)" % (
            int((o != want).sum()), "0" if after else "the residual", r0, r1)
        del drop, o, want
    del a, res, out
    _free()


def test_dropout_kernel_whole_output_past_2_32():
    """a4r_dropout over 645,120 x 768 elements from counter 2^32 + 12,345: every element bit-equal to
    bf16(x * keep * scale), and the kept fraction within 2e-3 of 0.9"""
    ops = _ops()
    M, N = C2_ROWS, 768
    x = _rand((M, N), 1.0, 21)
    out = ops.dropout(x, None, P, SEED, BIG_OFF)
    s = R.keep_scale(P)
    kept = 0
    for r0 in range(0, M, 65536):
        r1 = min(M, r0 + 65536)
        keep = R.element_keep(SEED, BIG_OFF, P, torch.arange(r0, r1, device="cuda"), N)
        ref = (x[r0:r1].float() * keep * s).to(BF16)
        assert torch.equal(out[r0:r1], ref), "%d elements differ (rows %d..%d)" % (int((out[r0:r1] != ref).sum()), r0, r1)
        kept += int(keep.sum())
        del keep, ref
    frac = kept / (M * N)
    assert abs(frac - 0.9) < 2e-3, frac
    del x, out
    _free()


@pytest.mark.parametrize("cpc", [False, True])
@pytest.mark.parametrize("B", [512, 513])
def test_bce_loss_at_the_benchmarked_batch(B, cpc):
    """the BCE head at 512 users x 20 positions (10,240 rows: the forward's grid covers 2,368 per wave, the backward's 9,472)
    and at 513 users (B·S not a multiple of the warps per block): ragged left-padded log_mask incl. empty histories, and the
    CPC variant.  Loss and count against fp64 torch, gradients as in test_bce_loss, and two runs bit-identical."""
    ops = _ops()
    S, D = 20, 64
    prec = _rand((B, S, D), D ** -0.5, 1)
    emb = _rand((B, S + 1, 2, D), 1.0, 2)
    lens = _lengths(B, S, 5, lo=0)
    log_mask = (torch.arange(S, device="cuda")[None] >= (S - lens)[:, None]).float()
    pf, ef = prec.double().requires_grad_(True), emb.double().requires_grad_(True)
    ps, ns = (pf * ef[:, 1:, 0]).sum(-1), (pf * ef[:, :-1, 1]).sum(-1)
    valid = torch.zeros_like(log_mask, dtype=torch.bool)
    if cpc:
        valid[:, -1] = True
    else:
        valid = log_mask != 0
    bce = torch.nn.BCEWithLogitsLoss()
    ref = bce(ps[valid], torch.ones_like(ps[valid])) + bce(ns[valid], torch.zeros_like(ns[valid]))
    lm = None if cpc else log_mask
    loss, count, p, n = ops.bce_loss_fwd(prec, emb, lm, cpc=cpc)
    r = float(ref.detach())
    assert abs(float(loss) - r) <= 1e-5 * max(1.0, abs(r)), (float(loss), r)
    assert float(count) == float(valid.sum())
    _close(p, ps.detach(), 1e-5, 1e-4, "pos scores")
    _close(n, ns.detach(), 1e-5, 1e-4, "neg scores")
    ref.backward()
    go = torch.full((1,), 2.0, device="cuda")
    d_prec, d_emb = ops.bce_loss_bwd(prec, emb, lm, p, n, count, grad_out=go, cpc=cpc)
    _close(d_prec, 2 * pf.grad, 2 ** -7, 1e-6, "d_prec")
    _close(d_emb, 2 * ef.grad, 2 ** -7, 1e-6, "d_emb")
    loss2, count2, p2, n2 = ops.bce_loss_fwd(prec, emb, lm, cpc=cpc)
    assert torch.equal(loss2, loss) and torch.equal(count2, count) and torch.equal(p2, p) and torch.equal(n2, n)
    d_prec2, d_emb2 = ops.bce_loss_bwd(prec, emb, lm, p, n, count, grad_out=go, cpc=cpc)
    assert torch.equal(d_prec2, d_prec) and torch.equal(d_emb2, d_emb)
