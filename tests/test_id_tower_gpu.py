"""-m gpu: the ID-embedding item tower (--item_tower id) on the sm_100a kernels: the gather and the deterministic table
gradient bit for bit against host restatements, the ids-only sampler, the whole step of both trees against the oracle
(tests/test_id_tower_cpu.py composes its id branch), the recorded step, the evaluator and the entry scripts."""
import logging
import os
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
sys.path.insert(0, HERE)

import transrec_oracle as O  # noqa: E402
from test_id_tower_cpu import ID_KEY, host_id_embed_bwd, id_args, id_batch, id_state_dict, oracle_id_loss  # noqa: E402

pytestmark = pytest.mark.gpu
BF16 = torch.bfloat16


def _ids(B, S1, V, seed, mode="random"):
    g = torch.Generator().manual_seed(seed)
    if mode == "same":
        return torch.full((B, S1, 2), 7, dtype=torch.int64)
    ids = torch.randint(0, V, (B, S1, 2), generator=g)
    if mode == "padding":
        ids[:, : S1 // 2] = 0
    return ids


@pytest.mark.parametrize("D", [64, 256])
def test_gather_is_bit_equal_to_the_rne_cast(D):
    from adapter4rec_b200 import ops
    B, S1, V = 512, 21, 20375
    table = torch.randn(V, D, generator=torch.Generator().manual_seed(1)).cuda()
    ids = _ids(B, S1, V, 2).cuda()
    emb, hist = ops.id_embed_fwd(table, ids)
    ref = table[ids].to(BF16)
    assert torch.equal(emb, ref)
    assert torch.equal(hist, ref[:, :-1, 0].contiguous())


@pytest.mark.parametrize("D", [64, 256])
@pytest.mark.parametrize("mode", ["random", "same", "padding"])
@pytest.mark.parametrize("B,S1", [(3, 6), (512, 21)])
def test_backward_is_bit_equal_to_the_host_restatement(D, mode, B, S1):
    from adapter4rec_b200 import ops
    V = 20375 if mode == "random" else 50
    ids = _ids(B, S1, V, 3, mode)
    g = torch.Generator().manual_seed(4)
    d_emb = torch.randn(B, S1, 2, D, generator=g).to(BF16)
    d_hist = torch.randn(B, S1 - 1, D, generator=g).to(BF16)
    grad0 = torch.randn(V, D, generator=g)
    want = host_id_embed_bwd(ids.numpy(), d_emb.float().numpy(), d_hist.float().numpy(), grad0.numpy(), V)
    runs = []
    for _ in range(2):                                    # two launches: identical bits
        grad = grad0.cuda()
        ops.id_embed_bwd(ids.cuda(), d_emb.cuda(), d_hist.cuda(), grad, accumulate=True)
        runs.append(grad.cpu())
    assert torch.equal(runs[0], runs[1])
    assert np.array_equal(runs[0].numpy(), want)
    assert torch.equal(runs[0][0], grad0[0])             # padding row never written


def test_backward_accumulates_over_two_calls_and_overwrites_without_accumulate():
    from adapter4rec_b200 import ops
    B, S1, D, V = 64, 21, 64, 300
    g = torch.Generator().manual_seed(5)
    ids = [_ids(B, S1, V, 6), _ids(B, S1, V, 7)]
    de = [torch.randn(B, S1, 2, D, generator=g).to(BF16) for _ in range(2)]
    dh = [torch.randn(B, S1 - 1, D, generator=g).to(BF16) for _ in range(2)]
    want = np.zeros((V, D), np.float32)
    grad = torch.zeros(V, D).cuda()
    for k in range(2):
        want = host_id_embed_bwd(ids[k].numpy(), de[k].float().numpy(), dh[k].float().numpy(), want, V)
        ops.id_embed_bwd(ids[k].cuda(), de[k].cuda(), dh[k].cuda(), grad, accumulate=True)
    assert np.array_equal(grad.cpu().numpy(), want)
    start = torch.randn(V, D, generator=g)
    over = start.cuda()
    ops.id_embed_bwd(ids[0].cuda(), de[0].cuda(), None, over, accumulate=False)
    ref = host_id_embed_bwd(ids[0].numpy(), de[0].float().numpy(), None, start.numpy(), V, accumulate=False)
    assert np.array_equal(over.cpu().numpy(), ref)


def test_ids_only_sampler_returns_the_full_calls_negatives():
    from adapter4rec_b200 import ops
    B, S1, I = 256, 21, 500
    g = torch.Generator().manual_seed(8)
    seqs = torch.zeros(B, S1, dtype=torch.int64)
    for b in range(B):
        n = int(torch.randint(2, S1 + 1, (1,), generator=g))
        seqs[b, S1 - n:] = torch.randperm(I, generator=g)[:n] + 1
    content = torch.randint(0, 1000, (I + 1, 8), generator=g)
    full = ops.sample_train_batch(seqs.cuda(), content.cuda(), I, 99, 1 << 40)
    ids_only = ops.sample_train_batch(seqs.cuda(), None, I, 99, 1 << 40)
    assert ids_only[0] is None
    assert torch.equal(full[1], ids_only[1]) and torch.equal(full[2], ids_only[2])
    assert int(ids_only[3]) == 0
    from adapter4rec_b200.data_utils.dataset import BuildTrainDataset
    ds = BuildTrainDataset({u: seqs[u][seqs[u] != 0].tolist() for u in range(B)}, None, I, S1 - 1, use_modal=False)
    items, mask = ds.batch(list(range(B)))
    assert torch.equal(items, torch.stack([seqs.cuda(), ds.last_negatives], -1)) and torch.equal(mask, full[1])


def _gpu_model(tree, cpc, sd, S=5):
    if tree == "text":
        from adapter4rec_b200.model import Model, ModelCPC
    else:
        from adapter4rec_b200.cv.model import Model, ModelCPC
    model = (ModelCPC if cpc else Model)(id_args(S=S), sd[ID_KEY].shape[0] - 1, False, None).cuda()
    assert set(model.state_dict()) == set(sd)
    model.load_state_dict(sd)
    return model


@pytest.mark.parametrize("tree", ["text", "cv"])
@pytest.mark.parametrize("cpc", [False, True])
def test_train_step_matches_the_oracle(tree, cpc):
    """loss <= 2e-2 relative, concatenated gradient <= 5e-2 relative L2 (the bounds of tests/test_model_gpu.py).  The tower's
    forward is defined on the bf16-rounded rows (the gather is bit-equal to weight[ids].to(bfloat16), tested above), so the
    oracle reads the rounded table (its gradient still lands on the fp32 table): what remains is the bf16 arithmetic of the
    user encoder and the loss."""
    S, D, I, B = 5, 64, 40, 6
    sd = id_state_dict(41, I, S, D)
    ids, mask = id_batch(42, B, S, I)
    rec = O.RecConfig(max_seq_len=S, embedding_dim=D, heads=2, blocks=2)
    osd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    table = osd[ID_KEY]
    rounded = dict(osd)
    rounded[ID_KEY] = table + (table.to(BF16).float() - table).detach()
    oloss = oracle_id_loss(ids, mask, rounded, rec, cpc)
    oloss.backward()
    model = _gpu_model(tree, cpc, sd, S)
    model.eval()
    loss = model(ids.view(-1).cuda(), mask.cuda(), 0)
    loss.backward()
    lv, ov = float(loss.detach()), float(oloss.detach())
    assert abs(lv - ov) <= 2e-2 * abs(ov), (lv, ov)
    params = dict(model.named_parameters())
    got = torch.cat([params[k].grad.float().cpu().flatten() for k in sorted(sd)])
    want = torch.cat([osd[k].grad.flatten() for k in sorted(sd)])
    per = {k: round(float((params[k].grad.float().cpu() - osd[k].grad).norm() / want.norm()), 5) for k in sorted(sd)}
    assert float((got - want).norm()) <= 5e-2 * float(want.norm()), per
    assert float(params[ID_KEY].grad[0].abs().max()) == 0.0


def test_graphed_step_is_bit_identical_to_eager():
    """dropout on, two passes per step, several steps: parameters and losses bit-identical between the recorded and the eager
    step (the table gradient has no atomics; its sort is recorded with the rest)"""
    from adapter4rec_b200 import functional as Fn
    from adapter4rec_b200.trainer import FlatAdamTrainer
    S, D, I, B = 5, 64, 40, 6
    sd = id_state_dict(51, I, S, D)
    ids, mask = id_batch(52, B, S, I)
    pairs = []
    for _ in range(2):
        model = _gpu_model("text", False, sd, S)
        model.train()
        pairs.append((model, FlatAdamTrainer(model, 1e-3, 1e-4, 1e-3, 1e-3, users_per_pass=B // 2, overlap=False)))
    (_, tr_g), (_, tr_e) = pairs

    def batch(t):
        return torch.roll(ids, t, 0).reshape(B * (S + 1), 2).cuda(), torch.roll(mask, t, 0).cuda()

    Fn.DropoutState.manual_seed(77)
    l_g = tr_g.train_step_graphed(*batch(0)).clone()
    Fn.DropoutState.manual_seed(77)
    l_e = tr_e.train_step(*batch(0)).clone()
    assert torch.equal(l_g, l_e) and torch.equal(tr_g.flat_param, tr_e.flat_param)
    for t in range(1, 5):
        Fn.DropoutState.manual_seed(77)
        l_g = tr_g.train_step_graphed(*batch(t)).clone()
        Fn.DropoutState.seed, Fn.DropoutState.counter = tr_g.graph_seed(tr_g.step_count), tr_g.graph_counter0
        l_e = tr_e.train_step(*batch(t)).clone()
        assert torch.isfinite(l_g).all()
        assert torch.equal(l_g, l_e), "step %d: loss %r vs %r" % (t, float(l_g), float(l_e))
        assert torch.equal(tr_g.flat_param, tr_e.flat_param), "step %d: parameters differ" % t
        assert torch.equal(tr_g.exp_avg, tr_e.exp_avg)
    tr_g.release_graph()


def test_evaluator_uses_the_table_and_shards_exactly(monkeypatch):
    """the item table is the RNE bf16 cast of id_embedding.weight (the training gather's rounding); top-10 ids, HR and NDCG
    equal a torch restatement on exactly representable embeddings; three id shards merged == one table"""
    from adapter4rec_b200 import ops
    from adapter4rec_b200.data_utils import metrics as M
    S, D, I, U = 5, 64, 3000, 200
    sd = id_state_dict(61, I, S, D)
    g = torch.Generator().manual_seed(62)
    sd[ID_KEY] = torch.randint(-2, 3, (I + 1, D), generator=g).float() * 0.125
    sd[ID_KEY][0] = 0
    model = _gpu_model("text", False, sd, S)
    args = id_args(S=S)
    table = M.get_item_embeddings(model, None, 512, args, False, 0)
    assert torch.equal(table.shard, model.id_embedding.weight.detach().to(BF16))
    tok = torch.randint(1, I + 1, (U, S), generator=g)
    tok[:, :2] = 0
    lm = (tok != 0).float()
    tgt = torch.randint(1, I + 1, (U,), generator=g).int()
    hist = tok.int()
    hit, ndcg, top = M.eval_arrays(model, tok, lm, tgt, hist, table, 64)
    # the user vectors: the evaluator's gather of the bf16 table equals the training gather
    emb, _ = ops.id_embed_fwd(model.id_embedding.weight.detach(), torch.stack([tok, tok], -1).cuda())
    assert torch.equal(table.gather(tok.cuda()), emb[:, :, 0])
    with torch.no_grad():
        prec = model.user_encoder(table.gather(tok.cuda()), lm.cuda(), 0)[:, -1].float()
    sc = prec @ table.shard.float().t()
    sc[:, 0] = -float("inf")
    sc.scatter_(1, hist.long().cuda(), -float("inf"))
    ids = torch.arange(I + 1, device="cuda").expand(U, -1)             # ids ascending: a stable sort gives (score desc, id asc)
    ref = torch.gather(ids, 1, torch.sort(sc, dim=1, descending=True, stable=True).indices)[:, :10]
    margin = torch.sort(sc, dim=1, descending=True).values
    clear = (margin[:, 9] - margin[:, 10]).abs() > 1e-3 * margin[:, 0].abs()
    assert int(clear.sum()) > U // 2
    assert torch.equal(top.long()[clear], ref[clear]), "top-10 ids differ"
    rank = (ref == tgt.long().cuda()[:, None]).float()
    hit_ref = rank.sum(1)
    ndcg_ref = (rank / torch.log2(torch.arange(2, 12, device="cuda").float())).sum(1)
    assert torch.equal(hit[clear], hit_ref[clear]) and torch.allclose(ndcg[clear], ndcg_ref[clear], rtol=0, atol=1e-6)
    # sharded: three ranks' tables, per-shard partial lists merged == the one-table result
    sc1, id1 = ops.score_topk(prec.to(BF16), table.shard, id_base=0, history=hist.cuda())
    full = ops.topk_merge(sc1, id1, target=tgt.cuda())
    parts_s, parts_i = [], []
    for r in range(3):
        monkeypatch.setattr(M, "_dist_info", lambda r=r: (r, 3))
        t = M.get_item_embeddings(model, None, 512, args, False, 0)
        assert (t.id_base, t.rank, t.world) == (M.shard_range(I + 1, r, 3)[0], r, 3)
        s, i = ops.score_topk(prec.to(BF16), t.shard, id_base=t.id_base, history=hist.cuda())
        ms, mi, _, _ = ops.topk_merge(s, i)
        parts_s.append(ms)
        parts_i.append(mi)
    merged = ops.topk_merge(torch.stack(parts_s).contiguous(), torch.stack(parts_i).contiguous(), target=tgt.cuda())
    for a, b in zip(full, merged):
        assert torch.equal(a, b)


def test_entry_scripts_pretrain_then_downstream_then_test(tmp_path):
    """text pre-training with --item_tower id writes epoch-N.pt; the downstream script loads it through
    --pretrained_model_name, trains, and --mode test ranks the test users from its own checkpoint"""
    from adapter4rec_b200 import run
    from adapter4rec_b200.cv import run_adapter
    from adapter4rec_b200.pretraining import text_run
    log = logging.getLogger("id_tower_test")
    data = run.synthetic_data(item_num=300, users=96, max_seq_len=5)
    data.item_content = None
    args = id_args(S=5)
    for k, v in dict(batch_size=32, epoch=2, lr=1e-3, fine_tune_lr=1e-4, adapter_bert_lr=1e-3, adapter_sasrec_lr=1e-3,
                     adapter_cv_lr=1e-3, logging_num=1, load_ckpt_name="None", pretrained_model_dir=str(tmp_path / "pre"),
                     mode="train").items():
        setattr(args, k, v)
    run.setup_seed(123456)
    pre_model, _, _ = text_run.train(args, False, 0, data, log, model_dir=str(tmp_path / "pre"))
    assert os.path.exists(tmp_path / "pre" / "epoch-2.pt")
    args.pretrained_model_name = "epoch-2"
    model, trainer, hit = run.train(args, False, 0, data, log, model_dir=str(tmp_path / "down"))
    assert torch.isfinite(model.id_embedding.weight).all()
    ck = torch.load(tmp_path / "down" / "epoch-2.pt", weights_only=False)
    assert set(ck["model_state_dict"]) >= {ID_KEY}
    assert len(ck["optimizer"]["param_groups"]) == 4            # torch.optim.Adam's format: bert, recsys, adapter_bert, adapter_recsys
    args.load_ckpt_name = "epoch-2.pt"
    hr = run.test(args, False, 0, data, log, model_dir=str(tmp_path / "down"))
    assert 0.0 <= hr <= 1.0
    # the image tree with the id tower: train two epochs from host-sampled ids
    cv_data = types.SimpleNamespace(**{k: getattr(data, k) for k in vars(data)})
    cv_data.item_images = None
    args.load_ckpt_name = "None"
    cm, _, _ = run_adapter.train(args, False, 0, cv_data, log, model_dir=str(tmp_path / "cv"))
    assert os.path.exists(tmp_path / "cv" / "epoch-2.pt") and not cm.use_modal
