"""Entry points of the text pre-training script, mirroring Pretraining/Text/run.py: `train(args, use_modal, local_rank, data)`
builds the model as run.py:127-235 does (BERT / RoBERTa body -> prefix + pooler freeze -> Model, or ModelCPC when --arch is not
sasrec -> optional --load_ckpt_name resume), optimises TWO learning-rate groups (run.py:238-251: 'bert_model' in the parameter
name -> --fine_tune_lr, everything else — the 768 -> D projection and the user encoder — -> --lr), runs the step of
run.py:311-324 and after every epoch evaluates on the validation users and writes epoch-{n}.pt (run.py:337-352) — the file the
downstream script loads through --pretrained_model_name.

There are no adapters here: every unfrozen tensor of the body trains, so the backward is the full fine-tuning path (weight
gradients on the tcgen05 split-token kernel, embedding-table scatter-adds; DESIGN.md §4.4).  Precision: the reference wraps the
step in fp16 autocast + GradScaler (run.py:301,319-324); this package computes in bf16 with fp32 accumulation and fp32 master
weights, which needs no loss scaling.  The OPT bodies of run.py:135-140 are out of scope (DESIGN.md §7).  --item_tower id
trains the ID-embedding table (id_embedding.weight, in the --lr group) and the user encoder; no body is read.
The TSV readers / tokeniser are host-side: the caller hands in the arrays they produce, as for adapter4rec_b200.run."""
import logging
import random
import re

import torch
import torch.distributed as dist

from ..data_utils.dataset import BuildTrainDataset
from ..model import BertModel, Model, ModelCPC, RobertaModel, TextConfigLite
from ..run import _checkpoint_path, rank_shard, run_eval, save_model, setup_seed, synthetic_data  # noqa: F401
from ..trainer import FlatAdamTrainer

# run.py:150-167: hidden width and named_parameters() indices of the pooler by body size; the checks run in this order and the
# last match wins ('small' is the pre-training script's own addition and shares the 4-layer pooler indices)
_BODY_SIZES = (("tiny", 128, (37, 38)), ("mini", 256, (69, 70)), ("small", 512, (69, 70)), ("medium", 512, (133, 134)),
               ("base", 768, (197, 198)), ("large", 1024, (389, 390)))


def freeze_bert_prefix(bert_model, args):
    """run.py:150-170: args.word_embedding_dim from the body's name; parameters with index < --freeze_paras_before and the
    pooler do not train."""
    pooler_para = ()
    for tag, width, pooler in _BODY_SIZES:
        if tag in args.bert_model_load:
            pooler_para, args.word_embedding_dim = pooler, width
    for index, (_, param) in enumerate(bert_model.named_parameters()):
        if index < args.freeze_paras_before or index in pooler_para:
            param.requires_grad = False


def group_parameters_pretrain(model):
    """run.py:238-251.  The test is 'bert_model' (not 'bert_encoder' as downstream): the projection
    bert_encoder.text_encoders.title.fc trains at --lr together with the user encoder."""
    groups = {"bert": [], "recsys": [], "adapter_bert": [], "adapter_recsys": []}       # trainer slot names
    for name, param in model.named_parameters():
        if param.requires_grad:
            groups["bert" if 'bert_model' in name else "recsys"].append((name, param))
    return groups


def build_model(args, item_num, local_rank, bert_config=None, bert_state_dict=None, use_modal=True):
    """run.py:127-218 without the DDP wrap; use_modal = False (--item_tower id): no body, the item table is id_embedding."""
    if not use_modal:
        return (Model if 'sasrec' in args.arch else ModelCPC)(args, item_num, False, None).to(local_rank)
    if 'opt' in args.bert_model_load:
        raise NotImplementedError("bert_model_load %r: the OPT bodies are outside the hot path" % args.bert_model_load)
    cfg = bert_config if bert_config is not None else TextConfigLite()
    bert_model = (RobertaModel if 'roberta' in args.bert_model_load else BertModel)(cfg)
    if bert_state_dict is not None:
        bert_model.load_state_dict(bert_state_dict, strict=False)
    freeze_bert_prefix(bert_model, args)
    if args.word_embedding_dim != cfg.hidden_size:
        raise ValueError("bert_model_load %r implies hidden width %d, the body has %d"
                         % (args.bert_model_load, args.word_embedding_dim, cfg.hidden_size))
    return (Model if 'sasrec' in args.arch else ModelCPC)(args, item_num, True, bert_model).to(local_rank)


def train(args, use_modal, local_rank, data, Log_file=None, bert_config=None, users_per_pass=128, model_dir=None,
          bert_state_dict=None):
    Log_file = Log_file or logging.getLogger("adapter4rec_b200.pretraining")
    model = build_model(args, data.item_num, local_rank, bert_config, bert_state_dict, use_modal)
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.lr, args.lr, users_per_pass=users_per_pass,
                              grouping=group_parameters_pretrain)
    Log_file.info("##### trainable_num {} #####".format(trainer.num_trainable))
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    start_epoch = 0
    if 'None' not in args.load_ckpt_name:                                   # run.py:221-231, 287-289
        if model_dir is None:
            raise ValueError("--load_ckpt_name needs the model_dir the checkpoint lives in")
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
        trainer.load_state_dict(ckpt['optimizer'])
        start_epoch = int(re.split(r'[._-]', args.load_ckpt_name)[1])
        torch.set_rng_state(ckpt['rng_state'])
        if ckpt.get('cuda_rng_state') is not None and torch.cuda.is_available():
            torch.cuda.set_rng_state(ckpt['cuda_rng_state'])
    users = sorted(data.users_train.keys())
    train_ds = BuildTrainDataset(data.users_train, data.item_content, data.item_num, args.max_seq_len, use_modal,
                                 device=next(model.parameters()).device, seed=123456 + rank)    # run.py:398 seed
    max_hit10, max_epoch = 0.0, 0
    for ep in range(args.epoch):
        now_epoch = start_epoch + ep + 1
        model.train()
        random.Random(now_epoch).shuffle(users)                             # sampler.set_epoch(now_epoch), run.py:309
        mine = rank_shard(users, rank, world)
        loss_sum, batches = 0.0, 0
        for b0 in range(0, len(mine), args.batch_size):
            items, log_mask = train_ds.batch(mine[b0:b0 + args.batch_size])
            loss = trainer.train_step(items.view(-1, items.size(-1)), log_mask)
            loss_sum, batches = loss_sum + float(loss), batches + 1
            if loss != loss:                                                # NaN guard, run.py:326-328
                raise FloatingPointError("loss is NaN")
        Log_file.info('epoch {} mean batch loss: {:.5f}'.format(now_epoch, loss_sum / max(1, batches)))
        hit10 = run_eval(model, data, args, Log_file, "valid", local_rank)  # run.py:337-341
        if hit10 > max_hit10:                                               # run.py:368-371
            max_hit10, max_epoch = hit10, now_epoch
        if model_dir is not None and rank == 0:                             # run.py:343-352: every epoch
            save_model(now_epoch, model, model_dir, trainer, Log_file)
    Log_file.info(' max eval Hit10 {:0.5f}  in epoch {}'.format(max_hit10 * 100, max_epoch))
    return model, trainer, max_hit10


def test(args, use_modal, local_rank, data, Log_file=None, bert_config=None, model_dir=None, bert_state_dict=None):
    """run.py:32-118: build, load --load_ckpt_name, rank the TEST users."""
    Log_file = Log_file or logging.getLogger("adapter4rec_b200.pretraining")
    model = build_model(args, data.item_num, local_rank, bert_config, bert_state_dict, use_modal)
    if 'None' not in args.load_ckpt_name:
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    return run_eval(model, data, args, Log_file, "test", local_rank)


def main(argv=None, pretrained_root="../pretrained_models", users_per_pass=128):
    """`python -m adapter4rec_b200.pretraining.text_run <flags of Pretraining/Text/run.py>`: run.py:393-431 — device, process
    group, seed 123456, the reference's checkpoint directory name, then train or test from the TSV files."""
    import os
    from ..data_utils.preprocess import load_text_data
    from ..run import _file_logger, load_body
    from .text_parameters import parse_args
    args = parse_args(argv)
    use_modal = 'modal' in args.item_tower                              # run.py:405-408
    local_rank = int(os.environ.get("LOCAL_RANK", max(args.local_rank, 0)))
    torch.cuda.set_device(local_rank)
    if "RANK" in os.environ and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend='nccl', init_method="env://")
    setup_seed(123456)
    dir_label = str(args.item_tower) + f'_{args.bert_model_load}_freeze_{args.freeze_paras_before}'
    log_paras = (f'{args.arch}_{args.bert_model_load}_bs_{args.batch_size}_ed_{args.embedding_dim}_lr_{args.lr}'
                 f'_L2_{args.l2_weight}_dp_{args.drop_rate}_Flr_{args.fine_tune_lr}')
    model_dir = os.path.join('./checkpoint_' + dir_label, 'cpt_' + log_paras)
    rank = dist.get_rank() if dist.is_initialized() else 0
    Log_file = _file_logger("Log_file", './logs_' + dir_label + ('_test' if 'test' in args.mode else '_train'), rank)
    Log_file.info(args)
    os.makedirs(model_dir, exist_ok=True)
    tokenizer, cfg, state = load_body(args, pretrained_root) if use_modal else (None, None, None)
    data = load_text_data(args, tokenizer, Log_file, use_modal)
    if 'train' in args.mode:
        return train(args, use_modal, local_rank, data, Log_file, cfg, users_per_pass, model_dir, bert_state_dict=state)
    if 'test' in args.mode:
        return test(args, use_modal, local_rank, data, Log_file, cfg, model_dir, bert_state_dict=state)


if __name__ == "__main__":
    main()
