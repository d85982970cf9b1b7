"""Entry points of the image tree's full fine-tuning scripts: Pretraining/CV/run.py (source-domain stage) and, through
adapter4rec_b200.cv.run, Downstream/CV/run.py (target-domain full fine-tuning, the baseline the adapters are compared with).
`train(args, use_modal, local_rank, data)` builds the model as Pretraining/CV/run.py:91-171 does (ViT-B/16 body with a fresh
xavier `classifier` -> the first --freeze_paras_before parameters frozen -> Model, or ModelCPC when --arch is not sasrec ->
optional --load_ckpt_name resume), optimises TWO learning-rate groups (:173-189: image_net parameters other than fc / classifier
/ decoder_pred -> --fine_tune_lr, everything else -> --lr), runs the step of :236-252 and after every epoch evaluates on the
validation users (batch 256) and writes epoch-{n}.pt (:258-268).

No adapters: every unfrozen tensor of the ViT trains (patch projection, cls token, position embeddings included; DESIGN.md
§4.4).  Precision: the reference's fp16 autocast + GradScaler (:229,245-250) has no counterpart — bf16 compute with fp32
accumulation and fp32 master weights needs no loss scaling.  ResNet / MAE towers are out of scope (DESIGN.md §7); --item_tower
id (use_modal = False) trains the ID-embedding table and the user encoder.  The LMDB reader is host-side: the caller hands in the arrays it produces, as for adapter4rec_b200.cv.run_adapter."""
import logging
import random
import re

import torch
import torch.distributed as dist

from ..cv.model import Model, ModelCPC
from ..cv.run_adapter import ImageBatches, build_vit, group_parameters_cv, run_eval, synthetic_data  # noqa: F401
from ..run import _checkpoint_path, rank_shard, save_model, setup_seed  # noqa: F401
from ..trainer import FlatAdamTrainer


def build_model(args, item_num, local_rank, vit_config=None, vit_state_dict=None, downstream=False, use_modal=True):
    """Pretraining/CV/run.py:91-147 (downstream=False) / Downstream/CV/run.py:98-164 (downstream=True: always Model, and
    --pretrained_recsys_model is loaded right after construction) without the DDP wrap.  use_modal = False (--item_tower
    id): no image body, the item table is id_embedding."""
    cv_model = None
    if use_modal:
        cv_model = build_vit(args, vit_config, vit_state_dict)
        for index, (_, param) in enumerate(cv_model.named_parameters()):
            if index < args.freeze_paras_before:
                param.requires_grad = False
    cls = Model if downstream or "sasrec" in args.arch else ModelCPC
    model = cls(args, item_num, use_modal, cv_model).to(local_rank)
    if downstream and 'None' not in args.pretrained_recsys_model:
        ckpt = torch.load(_checkpoint_path("../pretrained_models/", args.pretrained_recsys_model), map_location="cpu",
                          weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    return model


def train(args, use_modal, local_rank, data, Log_file=None, vit_config=None, users_per_pass=32, model_dir=None,
          downstream=False):
    Log_file = Log_file or logging.getLogger("adapter4rec_b200.pretraining.cv")
    model = build_model(args, data.item_num, local_rank, vit_config, downstream=downstream, use_modal=use_modal)
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.fine_tune_lr, args.lr, users_per_pass=users_per_pass,
                              grouping=group_parameters_cv)
    Log_file.info("##### trainable_num {} #####".format(trainer.num_trainable))
    start_epoch = 0
    if 'None' not in args.load_ckpt_name:
        if model_dir is None:
            raise ValueError("--load_ckpt_name needs the model_dir the checkpoint lives in")
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
        trainer.load_state_dict(ckpt['optimizer'])
        start_epoch = int(re.split(r'[._-]', args.load_ckpt_name)[1])
        torch.set_rng_state(ckpt['rng_state'])
        if ckpt.get('cuda_rng_state') is not None and torch.cuda.is_available():
            torch.cuda.set_rng_state(ckpt['cuda_rng_state'])
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    users = sorted(data.users_train.keys())
    dev = next(model.parameters()).device
    batches = ImageBatches(data.users_train, data.item_images if use_modal else None, data.item_num, args.max_seq_len, dev,
                           12345 + rank)
    max_hit10, max_epoch = 0.0, 0
    for ep in range(args.epoch):
        now_epoch = start_epoch + ep + 1
        model.train()
        random.Random(now_epoch).shuffle(users)                                        # sampler.set_epoch(now_epoch), :235
        mine = rank_shard(users, rank, world)
        loss_sum, n_batches = 0.0, 0
        for b0 in range(0, len(mine), args.batch_size):
            sample_items, log_mask = batches.batch(mine[b0:b0 + args.batch_size])
            loss = trainer.train_step(sample_items, log_mask)
            loss_sum, n_batches = loss_sum + float(loss), n_batches + 1
            if loss != loss:                                                           # NaN guard, :252-254
                raise FloatingPointError("loss is NaN")
        Log_file.info('epoch {} mean batch loss: {:.5f}'.format(now_epoch, loss_sum / max(1, n_batches)))
        hit10 = run_eval(model, data, args, Log_file, "valid", local_rank, batch_size=256)            # :260-264
        if downstream:                                                                 # Downstream/CV/run.py:282-284
            run_eval(model, data, args, Log_file, "test", local_rank, batch_size=args.batch_size)
        if hit10 > max_hit10:
            max_hit10, max_epoch = hit10, now_epoch
        if model_dir is not None and rank == 0:                                        # :266-268: every epoch
            save_model(now_epoch, model, model_dir, trainer, Log_file)
    Log_file.info(' max eval Hit10 {:0.5f}  in epoch {}'.format(max_hit10 * 100, max_epoch))
    return model, trainer, max_hit10


def test(args, use_modal, local_rank, data, Log_file=None, vit_config=None, model_dir=None, downstream=False):
    """Pretraining/CV/run.py:25-77: build, load --load_ckpt_name if given, rank the TEST users."""
    Log_file = Log_file or logging.getLogger("adapter4rec_b200.pretraining.cv")
    model = build_model(args, data.item_num, local_rank, vit_config, downstream=downstream, use_modal=use_modal)
    if 'None' not in args.load_ckpt_name:
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    return run_eval(model, data, args, Log_file, "test", local_rank, batch_size=args.batch_size)
