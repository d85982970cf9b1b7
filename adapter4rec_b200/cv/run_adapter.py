"""Entry points of the image tree, mirroring Downstream/CV/run_adapter.py: `train(args, use_modal, local_rank, data)` builds the
model as run_adapter.py:283-489 does (ViT-B/16 body with a fresh xavier `classifier` -> Model / ModelCPC -> optional
--pretrained_recsys_model checkpoint -> freeze -> adapter surgery -> --load_ckpt_name -> LayerNorm unfreeze -> the image tree's
four learning-rate groups), trains with the step of :571-598 and evaluates with get_item_embeddings + eval_model.

The LMDB reader and the PIL transforms (data_utils/dataset.py) are host-side and out of scope (DESIGN.md §7): the caller hands
in what they produce — `item_images` [I+1, 3, R, R] float32 already normalised to (x - 0.5) / 0.5 (row 0 = the padding item),
`users_train` {uid: [item ids]} and the eval dictionaries — via `data`.  `synthetic_data` builds such arrays.

Precision: the reference runs fp16 autocast + GradScaler when --use_scale contains 'half' (:565-590); this package computes in
bf16 with fp32 accumulation and fp32 master weights either way, which needs no loss scaling, so the flag is accepted and has no
effect."""
import logging
import os
import random
import re
import types

import numpy as np
import torch
import torch.distributed as dist
from torch.nn.init import constant_, xavier_normal_

from .. import surgery
from ..data_utils.metrics import core_model, eval_model, get_item_embeddings
from ..model.layers import Linear
from ..run import _checkpoint_path, rank_shard, save_model, setup_seed  # noqa: F401  (same helpers as the text tree)
from ..trainer import FlatAdamTrainer
from .model import Model, ModelCPC
from .vit import ViTConfigLite, ViTForImageClassification


def group_parameters_cv(model):
    """run_adapter.py:487-510: ('image_net' in name) x (classifier-like: 'fc' / 'classifier' / 'decoder_pred') x ('adapter' in
    name).  Unlike the text tree the test is 'adapter' ONLY: LoRA factors inside the ViT land in the image_net group
    (fine_tune_lr), as they do in the reference."""
    groups = {"bert": [], "recsys": [], "adapter_bert": [], "adapter_recsys": []}     # trainer slot names; 'bert' = image_net
    for name, param in model.named_parameters():
        if not param.requires_grad:
            continue
        is_adapter = "adapter" in name
        if 'image_net' in name and not ('fc' in name or 'classifier' in name or 'decoder_pred' in name):
            groups["adapter_bert" if is_adapter else "bert"].append((name, param))
        else:
            groups["adapter_recsys" if is_adapter else "recsys"].append((name, param))
    return groups


def build_vit(args, vit_config=None, vit_state_dict=None):
    """run_adapter.py:283-297: the ViT-B/16 body with a fresh xavier `classifier` [768 -> embedding_dim].  Only the ViT image
    tower is on this package's path ('vit' in --CV_model_load); ResNet / MAE / CLIP towers are out of scope (DESIGN.md §7)
    and refused."""
    if 'vit' not in args.CV_model_load or 'mae' in args.CV_model_load:
        raise NotImplementedError("CV_model_load %r: only the ViT-B/16 tower is implemented" % args.CV_model_load)
    cv_model = ViTForImageClassification(vit_config if vit_config is not None else ViTConfigLite())
    if vit_state_dict is not None:
        cv_model.load_state_dict(vit_state_dict, strict=False)
    cv_model.classifier = Linear(cv_model.config.hidden_size, args.embedding_dim)        # :291-297
    xavier_normal_(cv_model.classifier.weight.data)
    constant_(cv_model.classifier.bias.data, 0)
    return cv_model


def build_model(args, item_num, local_rank, vit_config=None, vit_state_dict=None, model_dir=None, use_modal=True):
    """run_adapter.py:283-480 without the DDP wrap.  use_modal = False (--item_tower id): no image body, the item table is
    id_embedding (adapter insertion is refused: there is no body to insert into)."""
    cv_model = build_vit(args, vit_config, vit_state_dict) if use_modal else None
    model = (ModelCPC if "cpc" in args.arch else Model)(args, item_num, use_modal, cv_model).to(local_rank)
    if 'None' not in args.pretrained_recsys_model:                                     # :350-358
        ckpt = torch.load(_checkpoint_path("../pretrained_models/", args.pretrained_recsys_model), map_location="cpu",
                          weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    if 'None' in args.fine_tune_to:                                                    # :360-367
        surgery.freeze_all(model)
    elif 'all' not in args.fine_tune_to:
        raise AssertionError("fine_tune_to should be defined properly")
    model = surgery.insert_adapters_cv(model, args)
    if 'None' not in args.finetune_layernorm:                                          # :482-486 ('layernorm' too: ViT's names)
        for name, param in model.named_parameters():
            if "adapter" not in name and ("LayerNorm" in name or "layer_norm" in name or "layernorm" in name):
                param.requires_grad = True
    return model


class ImageBatches:
    """BuildTrainDataset / Build_Lmdb_Dataset.__getitem__ (Downstream/CV/data_utils/dataset.py:56-113) for a list of users:
    left-padded sequences, one uniform negative per position rejected against the user's own sequence, the images gathered
    from the resident table: sample_items [B*(S+1)*2, 3, R, R] float32, log_mask [B, S].  item_images None (the id tower):
    sample_items are the item ids [B*(S+1)*2] int64 themselves."""

    def __init__(self, u2seq, item_images, item_num, max_seq_len, device, seed):
        self.u2seq, self.item_num, self.S, self.dev = u2seq, item_num, max_seq_len, device
        self.images = None if item_images is None else torch.as_tensor(item_images, dtype=torch.float32).to(device)
        self.rng = random.Random(seed)

    def batch(self, users):
        S1 = self.S + 1
        ids = np.zeros((len(users), S1, 2), dtype=np.int64)
        log_mask = np.zeros((len(users), self.S), dtype=np.float32)
        for b, u in enumerate(users):
            seq = list(self.u2seq[u])
            n = len(seq)
            ids[b, S1 - n:, 0] = seq
            log_mask[b, self.S - (n - 1):] = 1.0
            taken = set(seq)
            for i in range(n - 1):
                neg = self.rng.randint(1, self.item_num)
                while neg in taken:
                    neg = self.rng.randint(1, self.item_num)
                ids[b, S1 - n + i, 1] = neg
        flat = torch.from_numpy(ids).view(-1).to(self.dev)
        return flat if self.images is None else self.images[flat], torch.from_numpy(log_mask).to(self.dev)


def synthetic_data(item_num=200, users=64, resize=224, max_seq_len=10, seed=0):
    rng = np.random.RandomState(seed)
    images = (rng.rand(item_num + 1, 3, resize, resize).astype(np.float32) * 2 - 1)
    images[0] = 0
    seqs = {u: (rng.permutation(item_num)[:rng.randint(5, max_seq_len + 4)] + 1).tolist() for u in range(users)}
    d = types.SimpleNamespace(item_images=images, item_num=item_num)
    d.users_train = {u: s[:-2][-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_valid = {u: s[:-1][-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_test = {u: s[-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_history_for_valid = {u: torch.LongTensor(s[:-2]) for u, s in seqs.items()}
    d.users_history_for_test = {u: torch.LongTensor(s[:-1]) for u, s in seqs.items()}
    return d


def train(args, use_modal, local_rank, data, Log_file=None, vit_config=None, users_per_pass=32, model_dir=None):
    Log_file = Log_file or logging.getLogger("adapter4rec_b200.cv")
    model = build_model(args, data.item_num, local_rank, vit_config, use_modal=use_modal)
    start_epoch = 0
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_cv_lr, args.adapter_sasrec_lr,
                              users_per_pass=users_per_pass, grouping=group_parameters_cv)
    if 'None' not in args.load_ckpt_name:                                              # :467-476: resume
        if model_dir is None:
            raise ValueError("--load_ckpt_name needs the model_dir the checkpoint lives in")
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
        trainer.load_state_dict(ckpt['optimizer'])
        start_epoch = int(re.split(r'[._-]', args.load_ckpt_name)[1])
        torch.set_rng_state(ckpt['rng_state'])
        if ckpt.get('cuda_rng_state') is not None and torch.cuda.is_available():
            torch.cuda.set_rng_state(ckpt['cuda_rng_state'])
    Log_file.info("##### trainable_num {} #####".format(trainer.num_trainable))
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    users = sorted(data.users_train.keys())
    dev = next(model.parameters()).device
    batches = ImageBatches(data.users_train, data.item_images if use_modal else None, data.item_num, args.max_seq_len, dev,
                           12345 + rank)                                               # :681 seed
    max_hit10 = 0.0
    for ep in range(args.epoch):
        now_epoch = start_epoch + ep + 1
        model.train()
        random.Random(now_epoch).shuffle(users)                                        # sampler.set_epoch(now_epoch), :578
        mine = rank_shard(users, rank, world)
        loss_sum, n_batches = 0.0, 0
        for b0 in range(0, len(mine), args.batch_size):
            sample_items, log_mask = batches.batch(mine[b0:b0 + args.batch_size])
            loss = trainer.train_step(sample_items, log_mask)
            loss_sum, n_batches = loss_sum + float(loss), n_batches + 1
            if loss != loss:                                                           # NaN guard, :593-595
                raise FloatingPointError("loss is NaN")
        Log_file.info('epoch {} mean batch loss: {:.5f}'.format(now_epoch, loss_sum / max(1, n_batches)))
        hit10 = run_eval(model, data, args, Log_file, "valid", local_rank, batch_size=256)           # :604-607
        run_eval(model, data, args, Log_file, "test", local_rank, batch_size=args.batch_size)        # :608-610
        if hit10 > max_hit10 or max_hit10 == 0 or ep % 10 == 0:                        # :612-616
            max_hit10 = max(max_hit10, hit10)
            if model_dir is not None and rank == 0:
                save_model(now_epoch, model, model_dir, trainer, Log_file)
    if model_dir is not None and rank == 0 and args.epoch > 0:                         # :629-630: the last state is always kept
        save_model(start_epoch + args.epoch, model, model_dir, trainer, Log_file)
    return model, trainer, max_hit10


def run_eval(model, data, args, Log_file, v_or_t, local_rank, batch_size=256):
    """run_adapter.py:632-660: the item table from the image tower (or the id tower's embedding table), then full-ranking
    HR@10 / NDCG@10."""
    use_modal = core_model(model).use_modal
    table = get_item_embeddings(model, data.item_images if use_modal else None, batch_size, args, use_modal, local_rank)
    hist, seqs = (data.users_history_for_valid, data.users_valid) if v_or_t == "valid" else \
        (data.users_history_for_test, data.users_test)
    return eval_model(model, hist, seqs, table, batch_size, args, data.item_num, Log_file, v_or_t, local_rank)
