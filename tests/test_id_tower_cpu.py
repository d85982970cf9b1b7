"""CPU: the ID-embedding item tower (--item_tower id, use_modal = False).

The id branch of the oracle is composed here from pieces that are already pinned: the table lookup
`id_embedding.weight[ids]` feeds the oracle's golden-pinned user encoder and BCE (transrec_oracle.loss_from_embeddings).
It is checked against an independent assembly with torch.nn.Embedding(I+1, D, padding_idx=0).  The rest checks the host
side of the tower: state-dict keys, learning-rate groups, the optimizer-state format, the routing of every entry point, the
refusal of adapter insertion, and a host restatement of the backward kernel's summation order (the GPU tests compare the
kernel against it bit for bit)."""
import os
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))

import cases  # noqa: E402
import cases_cv  # noqa: E402
import transrec_oracle as O  # noqa: E402

ID_KEY = "id_embedding.weight"


def id_args(S=5, D=64, arch="sasrec"):
    return types.SimpleNamespace(max_seq_len=S, min_seq_len=2, l2_weight=0, embedding_dim=D, num_attention_heads=2,
                                 drop_rate=0.1, transformer_block=2, arch=arch, adding_adapter_to="None",
                                 fine_tune_to="all", finetune_layernorm="None", pretrained_model_name="None",
                                 pretrained_recsys_model="None", adapter_type="None", CV_model_load="vit-base-patch16-224",
                                 freeze_paras_before=0, item_tower="id")


def oracle_id_loss(ids, log_mask, sd, rec, cpc=False):
    """Model.forward / ModelCPC.forward of the id tower: the item embeddings are rows of id_embedding.weight."""
    return O.loss_from_embeddings(sd[ID_KEY][ids.reshape(-1)], log_mask, sd, rec, cpc)


def id_state_dict(seed, item_num, S, D, blocks=2):
    """the user-encoder weights of the tiny text case plus a seeded table (row 0 = padding = zeros)"""
    c = cases.tiny_case("base")
    sd = {k: v for k, v in cases.build_state_dict(c).items() if k.startswith("user_encoder.")}
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(item_num + 1, D, generator=g) * 0.3
    table[0] = 0
    sd[ID_KEY] = table
    return sd


def id_batch(seed, B, S, item_num):
    """ids [B, S+1, 2] and log_mask [B, S] with the layout BuildTrainDataset(use_modal=False) returns: left padding, one
    negative per real slot except the last"""
    rng = np.random.RandomState(seed)
    ids = np.zeros((B, S + 1, 2), dtype=np.int64)
    mask = np.zeros((B, S), dtype=np.float32)
    for b in range(B):
        n = rng.randint(2, S + 2)
        seq = rng.choice(np.arange(1, item_num + 1), n, replace=False)
        ids[b, S + 1 - n:, 0] = seq
        mask[b, S - (n - 1):] = 1
        for i in range(n - 1):
            neg = rng.randint(1, item_num + 1)
            while neg in seq:
                neg = rng.randint(1, item_num + 1)
            ids[b, S + 1 - n + i, 1] = neg
    return torch.from_numpy(ids), torch.from_numpy(mask)


@pytest.mark.parametrize("cpc", [False, True])
def test_oracle_id_branch_equals_torch_embedding_assembly(cpc):
    """loss and every gradient (table and user encoder): oracle id branch == nn.Embedding + the oracle's user encoder/BCE"""
    S, D, I = 5, 64, 40
    sd = id_state_dict(31, I, S, D)
    rec = O.RecConfig(max_seq_len=S, embedding_dim=D, heads=2, blocks=2)
    ids, mask = id_batch(32, 6, S, I)
    a = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    la = oracle_id_loss(ids, mask, a, rec, cpc)
    la.backward()
    emb = torch.nn.Embedding(I + 1, D, padding_idx=0)
    with torch.no_grad():
        emb.weight.copy_(sd[ID_KEY])
    b = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k != ID_KEY}
    S1 = S + 1
    e = emb(ids).view(-1, S1, 2, D)
    prec = O.user_encoder(e[:, :-1, 0], mask, b, rec)
    ps, ns = (prec * e[:, 1:, 0]).sum(-1), (prec * e[:, :-1, 1]).sum(-1)
    if cpc:
        lb = torch.nn.functional.binary_cross_entropy_with_logits(ps[:, -1], torch.ones(6)) + \
            torch.nn.functional.binary_cross_entropy_with_logits(ns[:, -1], torch.zeros(6))
    else:
        idx = torch.where(mask != 0)
        lb = torch.nn.functional.binary_cross_entropy_with_logits(ps[idx], torch.ones(len(idx[0]))) + \
            torch.nn.functional.binary_cross_entropy_with_logits(ns[idx], torch.zeros(len(idx[0])))
    lb.backward()
    assert abs(float(la) - float(lb)) <= 1e-6 * abs(float(lb))
    assert torch.allclose(a[ID_KEY].grad, emb.weight.grad, rtol=1e-5, atol=1e-7)
    assert float(emb.weight.grad[0].abs().max()) == 0.0          # padding_idx: no gradient
    for k in b:
        assert torch.allclose(a[k].grad, b[k].grad, rtol=1e-5, atol=1e-7), k


def _text_model(cpc=False, use_modal=False):
    from adapter4rec_b200.model import Model, ModelCPC
    return (ModelCPC if cpc else Model)(id_args(), 40, use_modal, None)


def _cv_model(cpc=False):
    from adapter4rec_b200.cv.model import Model, ModelCPC
    return (ModelCPC if cpc else Model)(id_args(S=4), 40, False, None)


@pytest.mark.parametrize("cpc", [False, True])
def test_state_dict_keys_are_the_table_plus_the_user_encoder(cpc):
    text_user = {k for k in cases.build_state_dict(cases.tiny_case("base")) if k.startswith("user_encoder.")}
    cv_user = {k for k in cases_cv.build_state_dict(cases_cv.tiny_cv_case("cv_base")) if k.startswith("user_encoder.")}
    m = _text_model(cpc)
    assert set(m.state_dict()) == {ID_KEY} | text_user
    assert tuple(m.state_dict()[ID_KEY].shape) == (41, 64) and m.state_dict()[ID_KEY].dtype == torch.float32
    assert float(m.state_dict()[ID_KEY][0].abs().max()) == 0.0
    assert set(_cv_model(cpc).state_dict()) == {ID_KEY} | cv_user


def test_id_embedding_lands_in_the_lr_group_of_every_grouping():
    from adapter4rec_b200.cv.run_adapter import group_parameters_cv
    from adapter4rec_b200.pretraining.text_run import group_parameters_pretrain
    from adapter4rec_b200.trainer import group_parameters
    for model in (_text_model(), _cv_model()):
        for rule in (group_parameters, group_parameters_pretrain, group_parameters_cv):
            g = rule(model)
            names = {k: [n for n, _ in v] for k, v in g.items()}
            assert ID_KEY in names["recsys"], (rule.__name__, names)


def test_optimizer_state_of_an_id_model_round_trips_through_torch_adam(tmp_path):
    """the trainer's optimizer entry is torch.optim.Adam's own format: torch loads it, and it loads torch's back"""
    from adapter4rec_b200.trainer import FlatAdamTrainer, group_parameters
    model = _text_model()
    tr = FlatAdamTrainer(model, 1e-3, 1e-4, 1e-3, 1e-3)
    g = torch.Generator().manual_seed(5)
    tr.exp_avg.copy_(torch.randn(tr.exp_avg.shape, generator=g))
    tr.exp_avg_sq.copy_(torch.rand(tr.exp_avg_sq.shape, generator=g))
    tr.step_count = 3
    torch.save({"optimizer": tr.state_dict()}, tmp_path / "o.pt")
    sd = torch.load(tmp_path / "o.pt", weights_only=False)["optimizer"]
    groups = group_parameters(model)
    opt = torch.optim.Adam([{"params": [p for _, p in groups[k]], "lr": lr}
                            for k, lr in (("bert", 1e-4), ("recsys", 1e-3), ("adapter_bert", 1e-3), ("adapter_recsys", 1e-3))])
    opt.load_state_dict(sd)
    table = model.id_embedding.weight
    st = opt.state[table]
    off = dict((n, o) for n, o, _ in tr.names)[ID_KEY]
    assert torch.equal(st["exp_avg"].reshape(-1), tr.exp_avg[off:off + table.numel()])
    assert int(st["step"]) == 3
    back = FlatAdamTrainer(_text_model(), 1e-3, 1e-4, 1e-3, 1e-3)
    back.load_state_dict(opt.state_dict())
    assert torch.equal(back.exp_avg, tr.exp_avg) and torch.equal(back.exp_avg_sq, tr.exp_avg_sq) and back.step_count == 3


def test_adapter_insertion_is_refused_for_the_id_tower():
    from adapter4rec_b200 import surgery
    args = id_args()
    args.adding_adapter_to, args.adapter_type = "all", "houslby"
    with pytest.raises(ValueError, match="no item-encoder body"):
        surgery.insert_adapters(_text_model(), args)
    with pytest.raises(ValueError, match="no item-encoder body"):
        surgery.insert_adapters_cv(_cv_model(), args)
    from adapter4rec_b200 import run
    with pytest.raises(ValueError, match="no item-encoder body"):
        run.build_model(args, 40, "cpu", use_modal=False)
    from adapter4rec_b200.cv import run_adapter
    with pytest.raises(ValueError, match="no item-encoder body"):
        run_adapter.build_model(args, 40, "cpu", use_modal=False)


def test_entry_point_builders_make_the_id_model_without_a_body():
    from adapter4rec_b200 import run
    from adapter4rec_b200.cv import run as cv_run_downstream
    from adapter4rec_b200.cv import run_adapter
    from adapter4rec_b200.pretraining import cv_run, text_run
    args = id_args()
    built = [run.build_model(args, 40, "cpu", use_modal=False), text_run.build_model(args, 40, "cpu", use_modal=False),
             run_adapter.build_model(args, 40, "cpu", use_modal=False),
             cv_run.build_model(args, 40, "cpu", use_modal=False),
             cv_run_downstream._impl.build_model(args, 40, "cpu", downstream=True, use_modal=False)]
    for m in built:
        assert not m.use_modal and hasattr(m, "id_embedding")
        assert not hasattr(m, "bert_encoder") and not hasattr(m, "cv_encoder")
        assert all(p.requires_grad for p in m.parameters())
    args.arch = "cpc"
    assert type(text_run.build_model(args, 40, "cpu", use_modal=False)).__name__ == "ModelCPC"


@pytest.mark.parametrize("module", ["adapter4rec_b200.run", "adapter4rec_b200.pretraining.text_run"])
def test_text_mains_route_item_tower_id(module, tmp_path, monkeypatch):
    """--item_tower id: no body or tokenizer is loaded, the catalogue is read by name, train receives use_modal = False"""
    import importlib
    import preprocess_fixture as F
    import adapter4rec_b200.run as run_mod
    mod = importlib.import_module(module)
    seen = {}

    def fake_train(args, use_modal, local_rank, data, *a, **k):
        seen.update(use_modal=use_modal, data=data)

    def no_body(*a, **k):
        raise AssertionError("the id tower must not load a body")

    monkeypatch.setattr(mod, "train", fake_train)
    monkeypatch.setattr(run_mod, "load_body", no_body)
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    monkeypatch.chdir(tmp_path)
    mod.main(["--item_tower", "id", "--root_data_dir", os.path.dirname(F.DIR), "--dataset", os.path.basename(F.DIR),
              "--news", os.path.basename(F.NEWS), "--behaviors", os.path.basename(F.BEHAVIORS),
              "--max_seq_len", str(F.MAX_SEQ_LEN), "--min_seq_len", str(F.MIN_SEQ_LEN)])
    assert seen["use_modal"] is False
    assert seen["data"].item_content is None and seen["data"].item_num > 0
    if module.endswith("text_run"):
        assert any(d.startswith("checkpoint_id_") for d in os.listdir(tmp_path))    # run.py:142: item_tower in the name


def test_train_dataset_validates_ids_on_the_host():
    from adapter4rec_b200.data_utils.dataset import BuildTrainDataset
    with pytest.raises(ValueError, match=r"\[1, item_num"):
        BuildTrainDataset({0: [1, 2, 41]}, None, 40, 5, use_modal=False, device="cpu")
    with pytest.raises(ValueError, match=r"\[1, item_num"):
        BuildTrainDataset({0: [1, 0, 3]}, None, 40, 5, use_modal=False, device="cpu")
    ds = BuildTrainDataset({0: [1, 2, 40], 1: [5, 6]}, None, 40, 5, use_modal=False, device="cpu")
    assert ds.item_content is None and ds.seqs.shape == (2, 6)


def host_id_embed_bwd(ids, d_emb, d_hist, grad, V, padding_idx=0, accumulate=True):
    """numpy float32 restatement of a4r_id_embed_bwd: per id, the sum over occurrences in ascending flat index r of the
    [B, S1, 2] layout, with d_hist[b, j] right after d_emb[r] at an occurrence (b, j, 0), j < S1-1; added to the existing
    row (accumulate) or written over it.  Padding and ids outside [0, V) are skipped."""
    B, S1, _ = ids.shape
    flat = ids.reshape(-1)
    D = d_emb.shape[-1]
    de = d_emb.reshape(-1, D).astype(np.float32)
    dh = None if d_hist is None else d_hist.reshape(B, S1 - 1, D).astype(np.float32)
    out = grad.copy()
    for i in np.unique(flat):
        if i == padding_idx or i < 0 or i >= V:
            continue
        acc = np.zeros(D, dtype=np.float32)
        for r in np.flatnonzero(flat == i):
            acc = acc + de[r]
            b, j, t = r // (2 * S1), (r // 2) % S1, r % 2
            if dh is not None and t == 0 and j < S1 - 1:
                acc = acc + dh[b, j]
        out[i] = (out[i] + acc) if accumulate else acc
    return out


def test_host_restatement_of_the_backward_order():
    """the restatement is the fp32 gradient of nn.Embedding (to rounding), and its order is the stated one: a sum whose
    terms cancel only in that order comes out exactly"""
    rng = np.random.RandomState(3)
    B, S1, D, V = 3, 4, 8, 10
    ids = rng.randint(0, V + 2, (B, S1, 2)).astype(np.int64)
    de = rng.randn(B, S1, 2, D).astype(np.float32)
    dh = rng.randn(B, S1 - 1, D).astype(np.float32)
    got = host_id_embed_bwd(ids, de, dh, np.zeros((V, D), np.float32), V)
    w = torch.zeros(V + 2, D, requires_grad=True)
    e = torch.nn.functional.embedding(torch.from_numpy(ids), w, padding_idx=0)
    (e * torch.from_numpy(de)).sum().backward(retain_graph=True)
    (e[:, :-1, 0] * torch.from_numpy(dh)).sum().backward()
    assert np.allclose(got, w.grad[:V].numpy(), rtol=1e-5, atol=1e-5)
    ids = np.full((1, 2, 2), 7, np.int64)
    de = np.zeros((1, 2, 2, 1), np.float32)
    de[0, 0, 0], de[0, 0, 1], de[0, 1, 0] = 1.0, 1e8, -1e8        # ascending order: (1 + 1e8) - 1e8 = 0 in fp32
    dh = np.zeros((1, 1, 1), np.float32)
    dh[0, 0] = 1.0                                                # ... but d_hist follows d_emb at (0, 0, 0): 2 + 1e8 - 1e8
    out = host_id_embed_bwd(ids, de, dh, np.zeros((8, 1), np.float32), 8)
    assert out[7, 0] == np.float32(np.float32(np.float32(2.0) + np.float32(1e8)) - np.float32(1e8))
