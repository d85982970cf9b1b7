"""-m gpu: SASRec user encoders with heads up to 128 wide.  The short-sequence attention kernel at head_dim 128 against an
fp32 torch reference (every mask kind, causal, dropout with counters past 2^32, the packed layout) at a size where the
grid-stride loop runs many iterations; other widths up to 128 zero-padded to the next native width with the temperature of
the true width; whole train steps at D = 256 with 2 heads (and the padded D = 96 / 192) against the oracle; the evaluator at
d = 256; and the text entry scripts on their default flags (--embedding_dim 256, --num_attention_heads 2)."""
import logging
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
sys.path.insert(0, HERE)

import cases  # noqa: E402
import dropout_rng as R  # noqa: E402
import transrec_oracle as O  # noqa: E402
from test_id_tower_cpu import ID_KEY, id_args, id_batch, oracle_id_loss  # noqa: E402
from test_kernels_gpu import _close, _rand  # noqa: E402
from test_train_kernels_gpu import (BIG_OFF, SEED, _RelL2, _allowed, _attention_mask_readback, _bert_mask,  # noqa: E402
                                    _free, _lengths, _sasrec_mask)

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
P = 0.1
# 65,536 sequences x 2 heads = 131,072 (sequence, head) pairs: many times the warps the grid holds (SMs x resident CTAs x 2)
N_BIG = 65536


def _ops():
    from adapter4rec_b200 import ops
    return ops


def _ref(qf, n, L, heads, dh, key_ok, causal, mask_neg, keep, p, scale):
    """fp32 attention with probability dropout (keep None: no dropout); one additive mask_neg per excluded key"""
    H = heads * dh
    q, k, v = [t.view(n, L, heads, dh).transpose(1, 2) for t in qf.view(n * L, 3, H).unbind(1)]
    s = (q @ k.transpose(-1, -2)) * scale + torch.where(_allowed(key_ok, causal, n, L, qf.device), 0.0, mask_neg)
    pr = torch.softmax(s, -1)
    if keep is not None:
        pr = pr * keep * R.keep_scale(p)
    return (pr @ v).transpose(1, 2).reshape(n * L, H)


def _check(qkv, dctx, N, L, heads, dh, mask, key_ok, causal, mask_neg, drop, chunk=8192, scale=None):
    """kernel forward and dq | dk | dv against _ref over every row, with the tolerances of test_train_kernels_gpu.py"""
    ops = _ops()
    H = heads * dh
    got = ops.attn_small_fwd(qkv, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop, scale=scale)
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, mask=mask, causal=causal, mask_neg=mask_neg, dropout=drop,
                              scale=scale)
    rel = _RelL2()
    for n0 in range(0, N, chunk):
        n1 = min(N, n0 + chunk)
        r0, r1 = n0 * L, n1 * L
        keep = None if drop is None else R.prob_keep(SEED, drop[2], drop[0], torch.arange(n0, n1, device="cuda"), heads, L)
        qf = qkv[r0:r1].float().requires_grad_(True)
        ref = _ref(qf, n1 - n0, L, heads, dh, None if key_ok is None else key_ok[n0:n1], causal, mask_neg, keep,
                   0.0 if drop is None else drop[0], dh ** -0.5 if scale is None else scale)
        _close(got[r0:r1], ref.detach(), 2 ** -6, 2e-2, "attention fwd d=%d, sequences %d..%d" % (dh, n0, n1))
        ref.backward(dctx[r0:r1].float())
        _close(dqkv[r0:r1], qf.grad, 2 ** -5, 6e-2, "attention bwd d=%d, sequences %d..%d" % (dh, n0, n1))
        rel.add(dqkv[r0:r1], qf.grad, H)
        del keep, qf, ref
    rel.check("attention bwd d=%d" % dh)
    return got, dqkv


# ---- 1. the kernel at head_dim 128 ------------------------------------------------------------------------------------

@pytest.mark.parametrize("dropout", [False, True])
@pytest.mark.parametrize("L", [20, 32])
def test_d128_sasrec_shape(L, dropout):
    """SASRec: causal, f32 left-padded log_mask with all-padding rows (every 97th history), mask_neg = -1e9"""
    N, heads, dh = N_BIG, 2, 128
    key_ok, mask = _sasrec_mask(N, L)
    assert bool((~key_ok).all(1).any()), "the case must contain all-padding rows"
    qkv = _rand((N * L, 3 * heads * dh), 1.0, 31 + L)
    dctx = _rand((N * L, heads * dh), 1.0, 32 + L)
    _check(qkv, dctx, N, L, heads, dh, mask, key_ok, True, -1e9, (P, SEED, BIG_OFF) if dropout else None)
    del qkv, dctx
    _free()


@pytest.mark.parametrize("masked", [False, True])
def test_d128_non_causal(masked):
    """non-causal with the int64 strided [ids | mask] key mask (ragged lengths, empty rows), and with no mask; dropout with
    counters past 2^32"""
    ops = _ops()
    N, L, heads, dh = N_BIG, 30, 2, 128
    key_ok, mask = _bert_mask(_lengths(N, L, 33), L) if masked else (None, None)
    qkv = _rand((N * L, 3 * heads * dh), 1.0, 34)
    dctx = _rand((N * L, heads * dh), 1.0, 35)
    _check(qkv, dctx, N, L, heads, dh, mask, key_ok, False, ops.F32_MIN, (P, SEED, BIG_OFF))
    del qkv, dctx
    _free()


def test_d128_scale_override():
    """an explicit temperature replaces head_dim ** -0.5"""
    N, L, heads, dh = 4096, 20, 2, 128
    key_ok, mask = _sasrec_mask(N, L)
    qkv = _rand((N * L, 3 * heads * dh), 1.0, 36)
    dctx = _rand((N * L, heads * dh), 1.0, 37)
    _check(qkv, dctx, N, L, heads, dh, mask, key_ok, True, -1e9, (P, SEED, 5), scale=0.3)


@pytest.mark.parametrize("causal", [False, True])
def test_d128_keep_bits_read_back(causal):
    """the keep bits themselves, forward (ctx) and backward (dv), against tests/dropout_rng.py's attention layout: the 128
    kernels draw exactly the counters of the 32 / 64 ones"""
    N, L, heads, dh = N_BIG, 32, 2, 128
    key_ok, mask = _sasrec_mask(N, L)
    _attention_mask_readback(N, L, heads, dh, mask, key_ok, causal, -1e9, BIG_OFF, 8192)
    _free()


def test_d128_packed_layout():
    """the cu_seqlens layout: bit-identical to the padded kernel at every kept token (backward with zero dctx on the padded
    rows), and against fp32"""
    from adapter4rec_b200.model.bert import PackedTokens
    ops = _ops()
    N, L, heads, dh = N_BIG, 30, 2, 128
    H = heads * dh
    key_ok = torch.arange(L, device="cuda")[None, :] < _lengths(N, L, 38)[:, None]
    fmask = key_ok.float()
    pk = PackedTokens(fmask)
    rows = pk.token_rows
    qkv = _rand((N * L, 3 * H), 1.0, 39)
    kept = torch.zeros(N * L, dtype=torch.bool, device="cuda")
    kept[rows] = True
    dctx = torch.where(kept[:, None], _rand((N * L, H), 1.0, 40), torch.zeros((), dtype=BF16, device="cuda"))
    kw = dict(causal=False, mask_neg=ops.F32_MIN, dropout=(P, SEED, BIG_OFF))
    ctx_pad, d_pad = _check(qkv, dctx, N, L, heads, dh, fmask, key_ok, False, ops.F32_MIN, kw["dropout"])
    qkv_p, dctx_p = qkv[rows].contiguous(), dctx[rows].contiguous()
    ctx_pk = ops.attn_small_fwd(qkv_p, N, L, heads, dh, mask=pk.token_mask, cu_seqlens=pk.cu_seqlens, **kw)
    assert torch.equal(ctx_pk, ctx_pad[rows]), "packed forward differs at %d elements" % int((ctx_pk != ctx_pad[rows]).sum())
    d_pk = ops.attn_small_bwd(qkv_p, dctx_p, N, L, heads, dh, mask=pk.token_mask, cu_seqlens=pk.cu_seqlens, **kw)
    for j, nm in enumerate(("dq", "dk", "dv")):
        a, b = d_pk[:, j * H:(j + 1) * H], d_pad[rows, j * H:(j + 1) * H]
        assert torch.equal(a, b), "packed %s differs at %d elements" % (nm, int((a != b).sum()))
    del qkv, dctx, qkv_p, dctx_p, ctx_pad, d_pad, ctx_pk, d_pk
    _free()


def test_other_widths_are_refused_by_the_kernel():
    ops = _ops()
    qkv = torch.zeros((20, 3 * 2 * 96), dtype=BF16, device="cuda")
    with pytest.raises(Exception, match="head_dim must be 32, 64 or 128"):
        ops.attn_small_fwd(qkv, 1, 20, 2, 96)


# ---- 2. the padding rule ----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("d", [48, 96])
def test_heads_zero_padded_to_the_next_native_width(d):
    """d_k = 48 (D = 96, 2 heads) and 96 (D = 192, 2 heads): zero-padded to 64 / 128 as MultiHeadedAttention does, with the
    temperature of the true width; the padding columns stay 0 and the rest equals the d-wide fp32 attention"""
    from adapter4rec_b200.model.modules import MultiHeadedAttention
    ops = _ops()
    N, L, heads = 4096, 20, 2
    w = MultiHeadedAttention.kernel_width(d)
    assert w == {48: 64, 96: 128}[d]
    key_ok, mask = _sasrec_mask(N, L)
    qkv_d = _rand((N * L, 3 * heads * d), 1.0, 41)
    dctx_d = _rand((N * L, heads * d), 1.0, 42)
    qkv = torch.nn.functional.pad(qkv_d.view(-1, 3 * heads, d), (0, w - d)).reshape(-1, 3 * heads * w)
    dctx = torch.nn.functional.pad(dctx_d.view(-1, heads, d), (0, w - d)).reshape(-1, heads * w)
    drop = (P, SEED, BIG_OFF)
    got = ops.attn_small_fwd(qkv, N, L, heads, w, mask=mask, causal=True, mask_neg=-1e9, dropout=drop, scale=d ** -0.5)
    dqkv = ops.attn_small_bwd(qkv, dctx, N, L, heads, w, mask=mask, causal=True, mask_neg=-1e9, dropout=drop,
                              scale=d ** -0.5)
    got, dqkv = got.view(-1, heads, w), dqkv.view(-1, 3 * heads, w)
    assert bool((got[..., d:] == 0).all()) and bool((dqkv[..., d:] == 0).all())
    keep = R.prob_keep(SEED, BIG_OFF, P, torch.arange(N, device="cuda"), heads, L)
    qf = qkv_d.float().requires_grad_(True)
    ref = _ref(qf, N, L, heads, d, key_ok, True, -1e9, keep, P, d ** -0.5)
    _close(got[..., :d].reshape(-1, heads * d), ref.detach(), 2 ** -6, 2e-2, "padded attention fwd")
    ref.backward(dctx_d.float())
    _close(dqkv[..., :d].reshape(-1, 3 * heads * d), qf.grad, 2 ** -5, 6e-2, "padded attention bwd")
    rel = _RelL2()
    rel.add(dqkv[..., :d].reshape(-1, 3 * heads * d), qf.grad, heads * d)
    rel.check("padded attention bwd")


def test_kernel_width_rule():
    from adapter4rec_b200.model.modules import MultiHeadedAttention
    kw = MultiHeadedAttention.kernel_width
    assert [kw(d) for d in (8, 31, 32, 33, 48, 64, 65, 96, 128)] == [32, 32, 32, 64, 64, 64, 128, 128, 128]
    with pytest.raises(AssertionError, match="up to 128"):
        kw(129)


def test_heads_wider_than_128_fail_at_the_first_forward():
    from adapter4rec_b200.model.modules import MultiHeadedAttention
    m = MultiHeadedAttention(n_heads=1, d_model=256, dropout=0.0).cuda()
    m.eval()
    x = torch.randn(2, 5, 256, device="cuda")
    with pytest.raises(AssertionError, match="head width 256"):
        m(x, x, x, torch.ones(2, 5, device="cuda"))


# ---- 3. whole train steps against the oracle ---------------------------------------------------------------------------

def _grad_rel(named, osd, keys):
    got = torch.cat([named[k].grad.float().cpu().flatten() for k in keys])
    want = torch.cat([osd[k].grad.flatten() for k in keys])
    return float((got - want).norm() / want.norm())


def _user_encoder_widths(model):
    from adapter4rec_b200.model.modules import MultiHeadedAttention
    return {m.d_k for m in model.modules() if isinstance(m, MultiHeadedAttention)}


def _id_state_dict(seed, item_num, D, heads):
    """the tiny text case's user encoder at width D, plus a seeded table (row 0 = padding = zeros)"""
    c = cases.tiny_case("base")
    c.D, c.rec_heads = D, heads
    sd = {k: v for k, v in cases.build_state_dict(c).items() if k.startswith("user_encoder.")}
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(item_num + 1, D, generator=g) * 0.3
    table[0] = 0
    sd[ID_KEY] = table
    return sd


def _id_model(cpc, sd, S, D, heads):
    from adapter4rec_b200.model import Model, ModelCPC
    args = id_args(S=S, D=D)
    args.num_attention_heads = heads
    model = (ModelCPC if cpc else Model)(args, sd[ID_KEY].shape[0] - 1, False, None).cuda()
    model.load_state_dict(sd)
    return model


# The id tower's gradient at D >= 192 is further from the fp32 oracle than at D = 64 whatever the head width: on one B200
# the case below measured 7.3-7.7e-2 (D = 256) with 2 heads of 128 (this kernel), 7.7-8.1e-2 with 4 heads of 64 (the 64-wide
# kernel, unchanged) and 7.5-8.6e-2 at D = 192 with 4 heads of 48; 2.4-3.5e-2 at D = 64 and 96.  The bf16 activations of a
# wider user encoder set that resolution, not the attention kernel; the bound below covers it.  The kernel's own accuracy
# is checked above against fp32 at the tolerances of the 32 / 64 kernels, and the modality tower at D = 256 (next test)
# meets the 5e-2 of tests/test_model_gpu.py.
ID_GRAD_BOUND = {64: 5e-2, 96: 5e-2, 192: 1e-1, 256: 1e-1}


@pytest.mark.parametrize("D,heads", [(256, 2), (96, 2), (192, 4)])
@pytest.mark.parametrize("cpc", [False, True])
def test_id_tower_step_matches_the_oracle(D, heads, cpc):
    """the id tower's Model / ModelCPC (the case of tests/test_id_tower_gpu.py) at D = 256 with 2 heads (d_k = 128, native)
    and at D = 96 / 192 (d_k = 48, padded to 64): loss <= 2e-2 relative as in tests/test_model_gpu.py, concatenated
    gradient within ID_GRAD_BOUND relative L2"""
    S, I, B = 5, 40, 6
    sd = _id_state_dict(41, I, D, heads)
    ids, mask = id_batch(42, B, S, I)
    rec = O.RecConfig(max_seq_len=S, embedding_dim=D, heads=heads, blocks=2)
    osd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    rounded = dict(osd)
    rounded[ID_KEY] = osd[ID_KEY] + (osd[ID_KEY].to(BF16).float() - osd[ID_KEY]).detach()
    oloss = oracle_id_loss(ids, mask, rounded, rec, cpc)
    oloss.backward()
    model = _id_model(cpc, sd, S, D, heads)
    assert _user_encoder_widths(model) == {D // heads}
    model.eval()
    loss = model(ids.view(-1).cuda(), mask.cuda(), 0)
    loss.backward()
    lv, ov = float(loss.detach()), float(oloss.detach())
    assert abs(lv - ov) <= 2e-2 * abs(ov), (lv, ov)
    rel = _grad_rel(dict(model.named_parameters()), osd, sorted(sd))
    assert rel <= ID_GRAD_BOUND[D], rel


@pytest.mark.parametrize("kind", ["base", "houlsby", "lora"])
def test_modality_tower_step_at_d256_matches_the_oracle(kind):
    """a tiny BERT body + the projection to D = 256 + SASRec with 2 heads of 128: no adapter, Houlsby (SASRec-side adapter
    blocks at H = 256) and LoRA (on the 256-wide w_Q / w_V); loss <= 2e-2 relative, gradient <= 5e-2 relative L2"""
    from test_model_gpu import build_gpu_model, oracle_setup
    c = cases.tiny_case(kind)
    c.D, c.rec_heads = 256, 2
    sd = cases.build_state_dict(c)
    items = cases.build_item_content(c)
    sample_items, log_mask, _ = cases.build_batch(c, items)
    rows = sample_items.view(-1, 2 * c.L)
    cfg, rec = oracle_setup(c)
    assert rec.embedding_dim == 256 and rec.heads == 2
    train = cases.trainable_keys(c, sd)
    osd = {k: v.clone() for k, v in sd.items()}
    for k in train:
        osd[k].requires_grad_(True)
    oloss = O.model_forward(rows, log_mask, osd, cfg, rec, cpc=c.cpc)
    model, _ = build_gpu_model(c, sd)
    assert _user_encoder_widths(model) == {128}
    model.eval()
    loss = model(rows.cuda(), log_mask.cuda(), 0)
    lv, ov = float(loss.detach()), float(oloss.detach())
    assert abs(lv - ov) <= 2e-2 * abs(ov), (lv, ov)
    if kind == "lora":
        assert any("lora_A" in k for k in train) and any("user_encoder" in k and "lora_A" in k for k in train)
    if kind == "houlsby":
        assert any(k.startswith("user_encoder.") and "adapter" in k for k in train)
    if train:
        oloss.backward()
        loss.backward()
        rel = _grad_rel(dict(model.named_parameters()), osd, train)
        assert rel <= 5e-2, rel


# ---- 4. the evaluator at d = 256 ---------------------------------------------------------------------------------------

def _exact(n, d, g):
    """entries in {-2..2} / 8: every dot product is exact in fp32 whatever the accumulation order"""
    return torch.randint(-2, 3, (n, d), generator=g).float() * 0.125


def test_score_topk_at_d256_bit_exact_against_the_oracle():
    """a4r_score_topk + merge at d = 256 on exactly representable user and item vectors: top-10 ids, HR@10 and NDCG@10
    equal the oracle's (score desc, id asc) ranking user for user"""
    ops = _ops()
    U, I, d, hl = 200, 5000, 256, 20
    g = torch.Generator().manual_seed(81)
    users, items = _exact(U, d, g), _exact(I, d, g)
    hist = torch.randint(0, I, (U, hl), generator=g).int()
    tgt = torch.randint(1, I, (U,), generator=g).int()
    sc, ids = ops.score_topk(users.to(BF16).cuda(), items.to(BF16).cuda(), id_base=0, history=hist.cuda(), k=10)
    _, top, hit, ndcg = ops.topk_merge(sc, ids, target=tgt.cuda())
    scores = users.double() @ items.double().t()
    top, hit, ndcg = top.cpu(), hit.float().cpu(), ndcg.float().cpu()
    for u in range(U):
        assert top[u].tolist() == O.topk_ids(scores[u], hist[u].tolist()), "user %d" % u
        eh, en = O.rank_metrics(scores[u], hist[u].tolist(), int(tgt[u]))
        assert float(hit[u]) == eh and abs(float(ndcg[u]) - en) < 1e-6, "user %d" % u


def test_evaluator_with_a_d256_user_encoder():
    """eval_arrays with the D = 256 / 2-head user encoder of the id tower over an exactly representable item table: top-10
    ids, HR and NDCG bit-exact against the oracle's ranking of the evaluator's own user vectors, and the user vectors within
    bf16 distance of the oracle's user encoder"""
    from adapter4rec_b200.data_utils import metrics as M
    S, D, I, U = 5, 256, 3000, 200
    sd = _id_state_dict(82, I, D, 2)
    g = torch.Generator().manual_seed(83)
    sd[ID_KEY] = _exact(I + 1, D, g)
    sd[ID_KEY][0] = 0
    model = _id_model(False, sd, S, D, 2)
    model.eval()
    args = id_args(S=S, D=D)
    table = M.get_item_embeddings(model, None, 512, args, False, 0)
    tok = torch.randint(1, I + 1, (U, S), generator=g)
    tok[:, :2] = 0
    lm = (tok != 0).float()
    tgt = torch.randint(1, I + 1, (U,), generator=g).int()
    hist = tok.int()
    hit, ndcg, top = M.eval_arrays(model, tok, lm, tgt, hist, table, 64)
    with torch.no_grad():
        prec = model.user_encoder(table.gather(tok.cuda()), lm.cuda(), 0)[:, -1].float().cpu()
        oprec = O.user_encoder(sd[ID_KEY][tok], lm, sd, O.RecConfig(max_seq_len=S, embedding_dim=D, heads=2, blocks=2))[:, -1]
    assert float((prec - oprec).norm() / oprec.norm()) <= 2e-2
    # the user vectors are bf16 and the table {-2..2}/8: scores are sums of 256 products; rank in float64 and keep users
    # whose rank-10 boundary is clear of fp32 rounding
    scores = prec.double() @ sd[ID_KEY].double().t()
    top, hit, ndcg = top.cpu(), hit.float().cpu(), ndcg.float().cpu()
    n = 0
    for u in range(U):
        s = scores[u].clone()
        s[hist[u].long()] = -float("inf")
        s[0] = -float("inf")
        srt = torch.sort(s, descending=True).values
        if abs(float(srt[9] - srt[10])) <= 1e-4 * abs(float(srt[0])):
            continue
        n += 1
        assert top[u].tolist() == O.topk_ids(scores[u], hist[u].tolist()), "user %d" % u
        eh, en = O.rank_metrics(scores[u], hist[u].tolist(), int(tgt[u]))
        assert float(hit[u]) == eh and abs(float(ndcg[u]) - en) < 1e-6, "user %d" % u
    assert n > U // 2, n


# ---- 5. the text entry scripts on their default width ------------------------------------------------------------------

def _capture(name):
    log = logging.getLogger(name)
    records = []
    log.addHandler(type("H", (logging.Handler,), {"emit": lambda self, r: records.append(r.getMessage())})())
    log.setLevel(logging.INFO)
    return log, records


def _tiny_body():
    from adapter4rec_b200.model import TextConfigLite
    return TextConfigLite(vocab_size=500, hidden_size=128, num_hidden_layers=2, num_attention_heads=2,
                          intermediate_size=512, max_position_embeddings=32, hidden_dropout_prob=0.0,
                          attention_probs_dropout_prob=0.0)


def test_downstream_entry_trains_on_its_default_width(tmp_path):
    """adapter4rec_b200.run without --embedding_dim / --num_attention_heads: D = 256, 2 heads of 128, Houlsby adapters on
    both sides, dropout on; the loss goes down, validation runs, and the checkpoint loads in --mode test"""
    from adapter4rec_b200 import run
    from adapter4rec_b200.parameters import parse_args
    args = parse_args(["--batch_size", "32", "--epoch", "3", "--adapter_type", "houslby", "--adding_adapter_to", "all",
                       "--bert_model_load", "bert_tiny", "--word_embedding_dim", "128", "--bert_adapter_down_size", "16",
                       "--adapter_bert_lr", "5e-3", "--adapter_sasrec_lr", "5e-3", "--max_seq_len", "10",
                       "--num_words_title", "12", "--pretrained_model_name", "None"])
    assert (args.embedding_dim, args.num_attention_heads) == (256, 2)
    run.setup_seed(123456)
    data = run.synthetic_data(item_num=300, users=96, num_words=12, max_seq_len=10, vocab=500)
    cfg = _tiny_body()
    log, records = _capture("wide_heads_run")
    model, trainer, hit10 = run.train(args, True, 0, data, Log_file=log, bert_config=cfg, users_per_pass=16,
                                      model_dir=str(tmp_path))
    assert _user_encoder_widths(model) == {128}
    losses = [float(m.split(":")[-1]) for m in records if "mean batch loss" in m]
    assert len(losses) == 3 and losses[-1] < losses[0], losses
    assert 0.0 <= hit10 <= 1.0 and any("valid_results" in m for m in records)
    saved = sorted(f for f in os.listdir(tmp_path) if f.startswith("epoch-"))
    assert "epoch-3.pt" in saved
    args.load_ckpt_name = "epoch-3.pt"
    hr = run.test(args, True, 0, data, Log_file=log, bert_config=cfg, model_dir=str(tmp_path))
    assert 0.0 <= hr <= 1.0


def test_pretraining_entry_trains_on_its_default_width(tmp_path):
    """adapter4rec_b200.pretraining.text_run without --embedding_dim / --num_attention_heads (D = 256, 2 heads of 128)"""
    from adapter4rec_b200.pretraining import text_run as run
    from adapter4rec_b200.pretraining.text_parameters import parse_args
    args = parse_args(["--batch_size", "32", "--epoch", "3", "--bert_model_load", "bert_tiny", "--freeze_paras_before", "21",
                       "--lr", "2e-3", "--fine_tune_lr", "5e-4", "--max_seq_len", "10", "--num_words_title", "12"])
    assert (args.embedding_dim, args.num_attention_heads) == (256, 2)
    run.setup_seed(123456)
    data = run.synthetic_data(item_num=300, users=96, num_words=12, max_seq_len=10, vocab=500)
    cfg = _tiny_body()
    log, records = _capture("wide_heads_pretrain")
    model, trainer, hit10 = run.train(args, True, 0, data, Log_file=log, bert_config=cfg, users_per_pass=16,
                                      model_dir=str(tmp_path))
    assert _user_encoder_widths(model) == {128}
    losses = [float(m.split(":")[-1]) for m in records if "mean batch loss" in m]
    assert len(losses) == 3 and losses[-1] < losses[0], losses
    assert 0.0 <= hit10 <= 1.0 and sum("valid_results" in m for m in records) == 3
    assert sorted(os.listdir(tmp_path)) == ["epoch-1.pt", "epoch-2.pt", "epoch-3.pt"]
    args.load_ckpt_name = "epoch-3.pt"
    assert 0.0 <= run.test(args, True, 0, data, Log_file=log, bert_config=cfg, model_dir=str(tmp_path)) <= 1.0
    assert any("test_results" in m for m in records)
