"""Entry points of the text tree, mirroring Downstream/Text/run.py: `train(args, use_modal, local_rank, data)` builds
the model exactly as run.py:286-529 does (BERT/RoBERTa body -> Model / ModelCPC -> freeze -> adapter surgery ->
LayerNorm unfreeze -> 4 learning-rate groups), trains for args.epoch epochs with the step of run.py:586-600 and
evaluates with get_item_embeddings + eval_model (run.py:649-670).

The reference's TSV readers / tokeniser (data_utils/preprocess.py) are host-side and out of scope (DESIGN.md §7): the
caller hands in the arrays they produce — `item_content` [I+1, 2L] int (ids | mask rows), `users_train` {uid: [item
ids]}, and the eval dictionaries — via `data`.  `synthetic_data` builds such arrays for smoke runs."""
import logging
import os
import random
import re
import types

import numpy as np
import torch
import torch.distributed as dist

from . import functional as Fn
from . import surgery
from .data_utils.dataset import BuildTrainDataset
from .data_utils.metrics import core_model, eval_model, get_item_embeddings
from .model import BertModel, Model, ModelCPC, RobertaModel, TextConfigLite
from .trainer import FlatAdamTrainer


def setup_seed(seed):      # run.py:673-678
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    np.random.seed(seed)
    random.seed(seed)
    Fn.DropoutState.manual_seed(seed)     # the counter-RNG behind every dropout kernel of this package


def build_train_batch(users, u2seq, item_content, item_num, max_seq_len):
    """BuildTrainDataset.__getitem__ (data_utils/dataset.py:24-49) for a list of users, stacked:
    sample_items [B, S+1, 2, 2L] int64, log_mask [B, S] float32 (left padded, one uniform negative per position)."""
    S1 = max_seq_len + 1
    ids = np.zeros((len(users), S1, 2), dtype=np.int64)
    log_mask = np.zeros((len(users), max_seq_len), dtype=np.float32)
    for b, u in enumerate(users):
        seq = list(u2seq[u])
        n = len(seq)
        ids[b, S1 - n:, 0] = seq
        log_mask[b, max_seq_len - (n - 1):] = 1.0
        taken = set(seq)
        for i in range(n - 1):
            neg = random.randint(1, item_num)
            while neg in taken:
                neg = random.randint(1, item_num)
            ids[b, S1 - n + i, 1] = neg
    content = torch.as_tensor(np.asarray(item_content)).long()
    return content[torch.from_numpy(ids)], torch.from_numpy(log_mask)


def synthetic_data(item_num=2000, users=256, num_words=30, max_seq_len=20, vocab=30522, seed=0):
    rng = np.random.RandomState(seed)
    item_content = np.zeros((item_num + 1, 2 * num_words), dtype=np.int64)
    for i in range(1, item_num + 1):
        n = rng.randint(8, num_words + 1)
        item_content[i, :n] = rng.randint(min(1000, vocab // 2), vocab, n)
        item_content[i, 0], item_content[i, n - 1] = min(101, vocab - 2), min(102, vocab - 1)
        item_content[i, num_words:num_words + n] = 1
    seqs = {u: (rng.permutation(item_num)[:rng.randint(5, max_seq_len + 4)] + 1).tolist() for u in range(users)}
    d = types.SimpleNamespace(item_content=item_content, item_num=item_num)
    d.users_train = {u: s[:-2][-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_valid = {u: s[:-1][-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_test = {u: s[-(max_seq_len + 1):] for u, s in seqs.items()}
    d.users_history_for_valid = {u: torch.LongTensor(s[:-2]) for u, s in seqs.items()}
    d.users_history_for_test = {u: torch.LongTensor(s[:-1]) for u, s in seqs.items()}
    return d


# run.py:302-317: hidden width and the named_parameters() indices of the pooler, by body size
_BODY_SIZES = (("tiny", 128, (37, 38)), ("mini", 256, (69, 70)), ("medium", 512, (133, 134)), ("base", 768, (197, 198)),
               ("large", 1024, (389, 390)))


def freeze_bert_prefix(bert_model, args):
    """run.py:302-320: sets args.word_embedding_dim from the body's name and freezes every BERT parameter whose
    named_parameters() index is below --freeze_paras_before (default 165: everything up to and including encoder layer 9
    of a base body), plus the pooler.  Runs BEFORE the Model is built, exactly as the reference does, so with
    --fine_tune_to all only the tail of the body (and everything outside it) trains."""
    pooler_para = ()
    for tag, width, pooler in _BODY_SIZES:
        if tag in args.bert_model_load:
            pooler_para, args.word_embedding_dim = pooler, width
    for index, (_, param) in enumerate(bert_model.named_parameters()):
        if index < getattr(args, "freeze_paras_before", 0) or index in pooler_para:
            param.requires_grad = False


def _checkpoint_path(directory, name):
    """data_utils/utils.py get_checkpoint: the file must exist"""
    path = os.path.join(directory, name)
    if not os.path.exists(path):
        raise FileNotFoundError("checkpoint %s not found" % path)
    return path


def build_model(args, item_num, local_rank, bert_config=None, bert_state_dict=None, use_modal=True):
    """run.py:286-503 without the DDP wrap (the trainer owns the gradient all-reduce): body -> prefix/pooler freeze ->
    Model / ModelCPC -> fine_tune_to freeze -> --pretrained_model_name checkpoint (BEFORE the surgery, run.py:374-381) ->
    adapter insertion -> LayerNorm unfreeze.  use_modal = False (--item_tower id): no body; the model's item table is
    id_embedding and there is nothing to insert adapters into (surgery refuses)."""
    bert_model = None
    if use_modal:
        cfg = bert_config if bert_config is not None else TextConfigLite()
        roberta = 'roberta' in args.bert_model_load
        bert_model = (RobertaModel if roberta else BertModel)(cfg)
        if bert_state_dict is not None:
            bert_model.load_state_dict(bert_state_dict, strict=False)
        freeze_bert_prefix(bert_model, args)
        if args.word_embedding_dim != cfg.hidden_size:
            raise ValueError("bert_model_load %r implies hidden width %d, the body has %d"
                             % (args.bert_model_load, args.word_embedding_dim, cfg.hidden_size))
    model = (ModelCPC if "cpc" in args.arch else Model)(args, item_num, use_modal, bert_model).to(local_rank)
    if 'None' in args.fine_tune_to:
        surgery.freeze_all(model)
    elif 'all' not in args.fine_tune_to:
        raise AssertionError("fine_tune_to should be defined properly")
    if 'None' not in getattr(args, "pretrained_model_name", "None"):
        ckpt = torch.load(_checkpoint_path(args.pretrained_model_dir, "%s.pt" % args.pretrained_model_name),
                          map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    model = surgery.insert_adapters(model, args)
    surgery.unfreeze_layernorm(model, args)
    return model


def rank_shard(users, rank, world):
    """torch.utils.data.DistributedSampler's split (run.py:347): the list is padded to a multiple of the world size by
    wrapping around, then dealt round-robin — every rank gets ceil(len / world) users and therefore takes the SAME number
    of optimizer steps (each step holds one all-reduce, so unequal step counts would hang or mis-pair collectives)."""
    per = (len(users) + world - 1) // world
    padded = list(users)
    while len(padded) < per * world:
        padded += users[:per * world - len(padded)]
    return padded[rank:per * world:world]


def save_model(now_epoch, model, model_dir, trainer, Log_file):
    """data_utils/utils.py:109-115: epoch-{n}.pt with the model state dict (reference key names), the optimizer state and
    the RNG states (torch, CUDA, and this package's dropout counter)."""
    os.makedirs(model_dir, exist_ok=True)
    ckpt_path = os.path.join(model_dir, 'epoch-%d.pt' % now_epoch)
    torch.save({'model_state_dict': model.state_dict(), 'optimizer': trainer.state_dict(),
                'rng_state': torch.get_rng_state(),
                'cuda_rng_state': torch.cuda.get_rng_state() if torch.cuda.is_available() else None}, ckpt_path)
    Log_file.info("Model saved to %s" % ckpt_path)
    return ckpt_path


def train(args, use_modal, local_rank, data, Log_file=None, bert_config=None, users_per_pass=128, model_dir=None,
          bert_state_dict=None, graphed=False):
    """graphed=True replays each step from a CUDA graph per rank (trainer.train_step_graphed: bit-identical arithmetic, one
    recording per batch shape); the default is the eager step."""
    Log_file = Log_file or logging.getLogger("adapter4rec_b200")
    model = build_model(args, data.item_num, local_rank, bert_config, bert_state_dict, use_modal)
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_bert_lr, args.adapter_sasrec_lr,
                              users_per_pass=users_per_pass)
    Log_file.info("##### trainable_num {} #####".format(trainer.num_trainable))
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    start_epoch = 0
    if 'None' not in getattr(args, "load_ckpt_name", "None"):          # run.py:481-493: resume
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
                                 device=next(model.parameters()).device, seed=123456 + rank)   # run.py:686 seed; per-rank stream
    max_hit10, max_eval, max_epoch, now_epoch = 0.0, 0.0, 0, start_epoch
    # utils.py:90-102 (para_and_log): --logging_num progress lines per epoch
    steps_per_epoch = -(-((len(users) + world - 1) // world) // args.batch_size)
    steps_for_log = max(1, int(steps_per_epoch / max(1, args.logging_num)))
    for ep in range(args.epoch):
        now_epoch = start_epoch + ep + 1
        model.train()
        random.Random(now_epoch - 1).shuffle(users)                 # sampler.set_epoch(now_epoch), run.py:576
        mine = rank_shard(users, rank, world)
        loss_sum, batches = 0.0, 0
        for b0 in range(0, len(mine), args.batch_size):
            # negatives + token-row gather on the device (only the user indices cross PCIe); the host restatement
            # build_train_batch above stays as the reference-order implementation for CPU-side tools
            items, log_mask = train_ds.batch(mine[b0:b0 + args.batch_size])
            loss = (trainer.train_step_graphed if graphed else trainer.train_step)(items.view(-1, items.size(-1)), log_mask)
            loss_sum, batches = loss_sum + float(loss), batches + 1
            if loss != loss:                                        # NaN guard of run.py:602-604
                raise FloatingPointError("loss is NaN")
            if batches % steps_for_log == 0:                        # run.py:606-608
                Log_file.info('cnt: {}, Ed: {}, batch loss: {:.5f}, sum loss: {:.5f}'.format(
                    batches, batches * args.batch_size, loss_sum / batches, loss_sum))
        Log_file.info('epoch {} mean batch loss: {:.5f}'.format(now_epoch, loss_sum / max(1, batches)))
        hit10 = run_eval(model, data, args, Log_file, "valid", local_rank)
        if hit10 > max_eval:                                        # run.py:660-663
            max_eval, max_epoch = hit10, now_epoch
        if max_eval > max_hit10 or max_hit10 == 0 or ep % 10 == 0:  # run.py:618-630: rank the TEST users and checkpoint on a
            max_hit10 = max(max_hit10, max_eval)                    # better validation HR@10, and every tenth epoch
            run_eval(model, data, args, Log_file, "test", local_rank)
            if model_dir is not None and rank == 0:
                save_model(now_epoch, model, model_dir, trainer, Log_file)
    if model_dir is not None and rank == 0 and args.epoch > 0:      # run.py:637-638: the last state is always kept
        save_model(now_epoch, model, model_dir, trainer, Log_file)
    Log_file.info(' max eval Hit10 {:0.5f}  in epoch {}'.format(max_eval * 100, max_epoch))
    if graphed:
        trainer.release_graph()
    return model, trainer, max_eval


def run_eval(model, data, args, Log_file, v_or_t, local_rank, batch_size=512):
    """run.py:649-670: item table (the item encoder's, or the id tower's embedding table), then full-ranking HR@10 /
    NDCG@10."""
    table = get_item_embeddings(model, data.item_content, batch_size, args, core_model(model).use_modal, local_rank)
    hist, seqs = (data.users_history_for_valid, data.users_valid) if v_or_t == "valid" else \
        (data.users_history_for_test, data.users_test)
    return eval_model(model, hist, seqs, table, batch_size, args, data.item_num, Log_file, v_or_t, local_rank)


def test(args, use_modal, local_rank, data, Log_file=None, bert_config=None, bert_state_dict=None, model_dir=None):
    """run.py:86-275 (--mode test): the model built as for training, --load_ckpt_name from model_dir (a missing file is an
    error), then the TEST users ranked."""
    Log_file = Log_file or logging.getLogger("adapter4rec_b200")
    model = build_model(args, data.item_num, local_rank, bert_config, bert_state_dict, use_modal)
    if 'None' not in args.load_ckpt_name:
        ckpt = torch.load(_checkpoint_path(model_dir, args.load_ckpt_name), map_location="cpu", weights_only=False)
        model.load_state_dict(ckpt['model_state_dict'])
    return run_eval(model, data, args, Log_file, "test", local_rank)


def load_body(args, pretrained_root="../pretrained_models"):
    """run.py:288-300: tokenizer, config and (when the file is there) weights of the body named by --bert_model_load, from
    the directory layout the reference uses.  Tokenisation is transformers' (host-side, as in the reference); the body itself
    is this package's BertModel / RobertaModel, which takes the checkpoint's tensors by name."""
    import json
    from transformers import BertTokenizer, RobertaTokenizer
    roberta = 'roberta' in args.bert_model_load
    path = os.path.join(pretrained_root, 'roberta' if roberta else 'bert', args.bert_model_load)
    tokenizer = (RobertaTokenizer if roberta else BertTokenizer).from_pretrained(path)
    cfg = TextConfigLite(**json.load(open(os.path.join(path, "config.json"))))
    weights = os.path.join(path, "pytorch_model.bin")
    state = None
    if os.path.exists(weights):
        state = torch.load(weights, map_location="cpu", weights_only=True)
        state = {re.sub(r'^(bert|roberta)\.', '', k): v for k, v in state.items()}
    return tokenizer, cfg, state


def _file_logger(name, directory, rank):
    log = logging.getLogger(name)
    log.setLevel(logging.INFO if rank in (-1, 0) else logging.ERROR)
    if rank in (-1, 0) and not log.handlers:
        os.makedirs(directory, exist_ok=True)
        for h in (logging.FileHandler(os.path.join(directory, "log.log"), encoding="utf-8"), logging.StreamHandler()):
            h.setFormatter(logging.Formatter("[%(levelname)s %(asctime)s] %(message)s"))
            log.addHandler(h)
    return log


def main(argv=None, pretrained_root="../pretrained_models", users_per_pass=128):
    """`python -m adapter4rec_b200.run <flags of Downstream/Text/run.py>` under torchrun (or alone on one GPU): run.py:681-711
    — device, process group, seed 123456, the reference's checkpoint directory name, then train or test from the TSV files
    named by --root_data_dir / --dataset / --news / --behaviors."""
    from .data_utils.preprocess import load_text_data
    from .parameters import parse_args
    args = parse_args(argv)
    local_rank = int(os.environ.get("LOCAL_RANK", max(args.local_rank, 0)))
    torch.cuda.set_device(local_rank)
    if "RANK" in os.environ and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend='nccl', init_method="env://")
    setup_seed(123456)
    dir_label = (f'{args.arch}_{args.bert_model_load}_freeze_{args.freeze_paras_before}_{args.pretrained_model_name}'
                 f'_add_adapter_to_{args.adding_adapter_to}_adapter_bert_lr_{args.adapter_bert_lr}'
                 f'_adapter_sasrec_lr_{args.adapter_sasrec_lr}_adapter_down_size_{args.adapter_down_size}'
                 f'_bert_adapter_down_size_{args.bert_adapter_down_size}__serial_{args.is_serial}'
                 f'_layernorm_{args.finetune_layernorm}_{args.adapter_type}_adam')
    log_paras = (f'{args.bert_model_load}_bs_{args.batch_size}_ed_{args.embedding_dim}_lr_{args.lr}_L2_{args.l2_weight}'
                 f'_dp_{args.drop_rate}_Flr_{args.fine_tune_lr}_SASAlr_{args.adapter_sasrec_lr}_BAlr_{args.adapter_bert_lr}')
    model_dir = os.path.join('./checkpoint_' + dir_label, 'cpt_' + log_paras + args.pretrained_model_name + args.behaviors)
    rank = dist.get_rank() if dist.is_initialized() else 0
    Log_file = _file_logger("Log_file", './logs_' + dir_label + ('_test' if 'test' in args.mode else '_train'), rank)
    Log_file.info(args)
    os.makedirs(model_dir, exist_ok=True)
    use_modal = 'modal' in args.item_tower                      # run.py:695-698
    tokenizer, cfg, state = load_body(args, pretrained_root) if use_modal else (None, None, None)
    data = load_text_data(args, tokenizer, Log_file, use_modal)
    if 'train' in args.mode:
        return train(args, use_modal, local_rank, data, Log_file, cfg, users_per_pass, model_dir, bert_state_dict=state)
    if 'test' in args.mode:
        return test(args, use_modal, local_rank, data, Log_file, cfg, state, model_dir)


if __name__ == "__main__":
    main()
