"""CPU: the mirrors of the reference's three full-fine-tuning entry scripts — Pretraining/Text/run.py, Pretraining/CV/run.py and
Downstream/CV/run.py — as far as they run without a GPU: command lines flag for flag (goldens dumped by the reference's own
parsers, tests/golden/make_pretrain_flags.py), the prefix freeze, the model class chosen by --arch and the two learning-rate
groups.  The training loops themselves run in tests/test_run_gpu.py."""
import json
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("tree", ["text", "cv"])
def test_pretraining_flags_equal_the_reference_parser(tree):
    from adapter4rec_b200.pretraining import cv_parameters, text_parameters
    mod = text_parameters if tree == "text" else cv_parameters
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "pretrain_%s_flags.json" % tree)))
    got = vars(mod.parse_args([]))
    assert got == ref
    assert all(type(got[k]) is type(ref[k]) for k in ref)
    with pytest.raises(SystemExit):
        mod.parse_args(["--adapter_type", "houslby"])           # the pre-training scripts have no adapter flags


def _text_cfg():
    from adapter4rec_b200.model import TextConfigLite
    return TextConfigLite(vocab_size=100, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256,
                          max_position_embeddings=32)


def test_text_pretraining_build_freeze_and_groups():
    """Pretraining/Text/run.py:150-170 (prefix + pooler freeze, width from the body's name), :213-216 (--arch), :238-251 (two
    groups by 'bert_model' in the name: the 768 -> D projection trains at --lr, unlike downstream)."""
    from adapter4rec_b200.model import Model, ModelCPC
    from adapter4rec_b200.pretraining import text_run
    from adapter4rec_b200.pretraining.text_parameters import parse_args
    base = ["--bert_model_load", "bert_tiny", "--embedding_dim", "64", "--max_seq_len", "5", "--num_words_title", "8",
            "--word_embedding_dim", "999"]
    args = parse_args(base + ["--freeze_paras_before", "21"])
    model = text_run.build_model(args, 50, "cpu", _text_cfg())
    assert type(model) is Model and args.word_embedding_dim == 128
    bert = model.bert_encoder.text_encoders.title.bert_model
    flags = [p.requires_grad for _, p in bert.named_parameters()]
    assert not any(flags[:21]) and not flags[37] and not flags[38]
    assert all(f for i, f in enumerate(flags) if i >= 21 and i not in (37, 38))
    g = text_run.group_parameters_pretrain(model)
    assert not g["adapter_bert"] and not g["adapter_recsys"]
    assert all("bert_model" in n for n, _ in g["bert"]) and len(g["bert"]) == sum(flags)
    rec = [n for n, _ in g["recsys"]]
    assert "bert_encoder.text_encoders.title.fc.weight" in rec and any(n.startswith("user_encoder.") for n in rec)
    assert len(g["bert"]) + len(rec) == sum(p.requires_grad for p in model.parameters())
    assert type(text_run.build_model(parse_args(base + ["--arch", "cpc"]), 50, "cpu", _text_cfg())) is ModelCPC
    with pytest.raises(ValueError):
        text_run.build_model(parse_args(["--bert_model_load", "bert-base-uncased"]), 50, "cpu", _text_cfg())
    with pytest.raises(NotImplementedError):
        text_run.build_model(parse_args(["--bert_model_load", "opt-125m"]), 50, "cpu", _text_cfg())
    # 'small' exists only in the pre-training script's table: 512 wide, pooler at the 4-layer indices
    a = parse_args(["--bert_model_load", "bert_small"])
    text_run.freeze_bert_prefix(torch.nn.Linear(2, 2), a)
    assert a.word_embedding_dim == 512


def _vit_cfg():
    from adapter4rec_b200.cv import ViTConfigLite
    return ViTConfigLite(hidden_size=768, num_hidden_layers=2, num_attention_heads=12, intermediate_size=256, image_size=48,
                         patch_size=16)


def test_cv_full_finetuning_build_freeze_and_groups(tmp_path):
    """Pretraining/CV/run.py:98-112,142-147,173-189 and Downstream/CV/run.py:153-164: fresh classifier, the first
    --freeze_paras_before ViT parameters frozen (no pooler rule), Model / ModelCPC by --arch (downstream: always Model),
    classifier in the --lr group."""
    from adapter4rec_b200.cv import model as cvm
    from adapter4rec_b200.cv import run as cv_downstream
    from adapter4rec_b200.cv.parameters import parse_args as downstream_args
    from adapter4rec_b200.pretraining import cv_run
    from adapter4rec_b200.pretraining.cv_parameters import parse_args
    base = ["--CV_model_load", "vit-base-patch16-224", "--CV_resize", "48", "--max_seq_len", "6", "--freeze_paras_before", "20"]
    model = cv_run.build_model(parse_args(base), 60, "cpu", _vit_cfg())
    assert type(model) is cvm.Model
    net = model.cv_encoder.image_net
    flags = [p.requires_grad for _, p in net.named_parameters()]
    assert not any(flags[:20]) and all(flags[20:])
    assert tuple(net.classifier.weight.shape) == (64, 768) and float(net.classifier.bias.detach().abs().sum()) == 0.0
    g = cv_run.group_parameters_cv(model)
    assert len(g["bert"]) == sum(flags) - 2 and all("image_net" in n and "classifier" not in n for n, _ in g["bert"])
    assert {"cv_encoder.image_net.classifier.weight", "cv_encoder.image_net.classifier.bias"} <= {n for n, _ in g["recsys"]}
    assert type(cv_run.build_model(parse_args(base + ["--arch", "cpc"]), 60, "cpu", _vit_cfg())) is cvm.ModelCPC
    with pytest.raises(NotImplementedError):
        cv_run.build_model(parse_args(["--CV_model_load", "resnet-50"]), 60, "cpu", _vit_cfg())
    # downstream full fine-tuning: run_adapter's flag set, always Model, a missing --pretrained_recsys_model is an error
    d = cv_downstream.build_model(downstream_args(base + ["--arch", "cpc"]), 60, "cpu", _vit_cfg())
    assert type(d) is cvm.Model
    with pytest.raises(FileNotFoundError):
        cv_downstream.build_model(downstream_args(base + ["--pretrained_recsys_model", "epoch-99.pt"]), 60, "cpu", _vit_cfg())
