"""Full-ranking evaluator, mirroring Downstream/Text/data_utils/metrics.py (function names and argument lists) on the
sm_100a kernels.

Differences from the reference that are deliberate and documented (DESIGN.md):
  * the item table stays on the GPU in bf16 (the reference returns it on the CPU in fp32 and ships rows to DataLoader
    workers); under torch.distributed it is SHARDED BY ITEM ID across ranks and never gathered (SURVEY.md §8e);
  * the [users x items] score matrix, the per-user argsort and the float64 one-hot labels are never materialised:
    scores, history mask and top-k are one kernel (a4r_score_topk), ranks come from top-k membership;
  * every rank evaluates every user against its own item shard; the partial top-k lists are all-gathered and merged.
"""
import math

import numpy as np
import torch
import torch.distributed as dist

from .. import ops

BF16 = torch.bfloat16


class ItemTable:
    """One rank's shard of the item-embedding table: rows = item ids [id_base, id_base + n_local), plus a trailing
    all-zero row used as the gather target for ids owned by other ranks."""

    def __init__(self, rows, id_base, num_rows_total, rank=0, world=1):
        self.id_base, self.total, self.rank, self.world = int(id_base), int(num_rows_total), rank, world
        self.n_local = rows.shape[0]
        self.dim = rows.shape[1]
        self.table = torch.cat([rows.to(BF16), torch.zeros((1, rows.shape[1]), dtype=BF16, device=rows.device)], 0).contiguous()

    @property
    def shard(self):
        return self.table[:self.n_local]

    def local_index(self, ids):
        """global item ids -> row of self.table: the shard row if this rank owns the id, else the trailing zero row"""
        local = ids - self.id_base
        owned = (local >= 0) & (local < self.n_local)
        return torch.where(owned, local, torch.full_like(local, self.n_local))

    def gather(self, ids):
        """Embeddings of arbitrary item ids [.., ..] -> bf16 [.., .., D]; exact under sharding: the owner contributes the
        row, every other rank a zero row, and the sum all-reduce of bf16 values with a single non-zero term is exact."""
        out = ops.gather_rows(self.table, self.local_index(ids))
        if self.world > 1:
            dist.all_reduce(out, op=dist.ReduceOp.SUM)
        return out


def to_bf16_2d(x):
    return x.to(BF16).reshape(x.shape[0], -1)


def core_model(model):
    """The object that owns `bert_encoder` / `user_encoder`: strips DDP's `.module` and CompacterModel's `.model`
    (metrics.py:72-73,101-102 reach through `model.module.model` when 'compacter' is in args.adapter_type)."""
    m = model.module if hasattr(model, "module") else model
    if not hasattr(m, "user_encoder") and hasattr(m, "model"):
        m = m.model
    return m


def _dist_info():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(num_rows, rank, world):
    """Contiguous id ranges [lo, hi) of near-equal size (SURVEY.md §8e: item table sharded by contiguous id range)."""
    per = (num_rows + world - 1) // world
    lo = min(num_rows, rank * per)
    return lo, min(num_rows, lo + per)


def print_metrics(x, Log_file, v_or_t):
    Log_file.info(v_or_t + "_results   {}".format('\t'.join(["{:0.5f}".format(i * 100) for i in x])))


def get_item_embeddings(model, item_content, test_batch_size, args, use_modal, local_rank):
    """metrics.py:62-79.  item_content [I+1, 2L] (numpy int or torch int64; row 0 = padding item).  Each rank encodes
    ITS shard of item ids with the item encoder under no_grad and keeps it on the device (an ItemTable).
    use_modal = False (the id tower): the table is id_embedding.weight itself (item_content is not read); the rank's
    shard is cast once to bf16 with the rounding of the training gather (RNE)."""
    module = core_model(model)
    module.eval()
    rank, world = _dist_info()
    if not use_modal:
        weight = module.id_embedding.weight.detach()
        lo, hi = shard_range(weight.shape[0], rank, world)
        emb, _ = ops.cast_transpose(weight[lo:hi], True, False) if hi > lo else (weight[:0].to(BF16), None)
        return ItemTable(emb, lo, weight.shape[0], rank, world)
    rows = torch.as_tensor(np.asarray(item_content) if not torch.is_tensor(item_content) else item_content)
    image_tree = hasattr(module, "cv_encoder")       # Downstream/CV: item_content = images [I+1, 3, R, R] float32
    rows = rows.float() if image_tree else rows.long()
    encoder = module.cv_encoder if image_tree else module.bert_encoder
    lo, hi = shard_range(rows.shape[0], rank, world)
    dev = next(module.parameters()).device
    outs = []
    with torch.no_grad():
        for i in range(lo, hi, test_batch_size):
            ids = rows[i:min(hi, i + test_batch_size)].to(dev, non_blocking=True)
            outs.append(to_bf16_2d(encoder(ids)))
    emb = torch.cat(outs, 0) if outs else torch.zeros((0, args.embedding_dim), dtype=BF16, device=dev)
    return ItemTable(emb, lo, rows.shape[0], rank, world)


def build_eval_arrays(eval_seq, user_history, max_seq_len):
    """Host-side restatement of BuildEvalDataset.__getitem__ (dataset.py:65-78) for all users at once:
    pad_tokens [U,S] int64 (left padded with item 0), log_mask [U,S] f32, target [U] int32, history [U,Hmax] int32."""
    users = sorted(eval_seq.keys()) if isinstance(eval_seq, dict) else list(range(len(eval_seq)))
    U = len(users)
    tok = np.zeros((U, max_seq_len), dtype=np.int64)
    mask = np.zeros((U, max_seq_len), dtype=np.float32)
    tgt = np.zeros((U,), dtype=np.int32)
    hists = []
    for r, u in enumerate(users):
        seq = list(eval_seq[u])
        t = seq[:-1]
        tok[r, max_seq_len - len(t):] = t
        mask[r, max_seq_len - len(t):] = 1.0
        tgt[r] = seq[-1]
        h = user_history[u]
        hists.append(np.asarray(h.cpu() if torch.is_tensor(h) else h, dtype=np.int32).reshape(-1))
    hmax = max(1, max(len(h) for h in hists))
    hist = np.zeros((U, hmax), dtype=np.int32)
    for r, h in enumerate(hists):
        hist[r, :len(h)] = h
    return tok, mask, tgt, hist


def eval_arrays(model, tok, mask, tgt, hist, item_table, user_block, topk=10):
    """Core evaluator on pre-built arrays (torch tensors, host or device): returns per-user (hit, ndcg) on the device
    plus the merged top-k ids."""
    module = core_model(model)
    module.eval()
    dev = item_table.table.device
    rank, world = item_table.rank, item_table.world
    U = tok.shape[0]
    hits, ndcgs, top_ids = [], [], []
    with torch.no_grad():
        for b0 in range(0, U, user_block):
            b1 = min(U, b0 + user_block)
            tk = tok[b0:b1].to(dev, non_blocking=True)
            lm = mask[b0:b1].to(dev, non_blocking=True)
            tg = tgt[b0:b1].to(dev, non_blocking=True).contiguous()
            hs = hist[b0:b1].to(dev, non_blocking=True).contiguous()
            prec = _user_vectors(module, item_table, tk, lm, dev)                      # K10 + K8 (+ last position)
            sc, ids = ops.score_topk(prec, item_table.shard, id_base=item_table.id_base, history=hs, k=topk)  # K11+K12
            if world > 1:
                lsc, lid, _, _ = ops.topk_merge(sc, ids)                              # local merge of the item splits
                gsc = torch.empty((world,) + tuple(lsc.shape), dtype=lsc.dtype, device=dev)
                gid = torch.empty((world,) + tuple(lid.shape), dtype=lid.dtype, device=dev)
                dist.all_gather_into_tensor(gsc, lsc)
                dist.all_gather_into_tensor(gid, lid)
                sc, ids = gsc, gid
            _, mid, hit, ndcg = ops.topk_merge(sc.contiguous(), ids.contiguous(), target=tg)   # K13
            hits.append(hit)
            ndcgs.append(ndcg)
            top_ids.append(mid)
    return torch.cat(hits), torch.cat(ndcgs), torch.cat(top_ids)


def _user_vectors(module, item_table, tk, lm, dev):
    """Last-position user vectors [U, D] (bf16) of one block (metrics.py:104: user_encoder(...)[:, -1]).  One rank: gather +
    encode.  N ranks: the USERS of the block are split — rank r gathers (ownership-masked rows + one sum all-reduce over the
    ranks, exact: a single non-zero term) and encodes only its U / N users, then the [U, D] vectors are all-gathered (1.5 KB
    per user at D = 768) — instead of N redundant encoders over the whole block."""
    world, rank = item_table.world, item_table.rank
    if world == 1:
        return module.user_encoder(item_table.gather(tk), lm, dev)[:, -1].contiguous()
    U = tk.shape[0]
    per = (U + world - 1) // world
    input_embs = item_table.gather(tk)                       # every rank needs rows of every shard: masked gather + all-reduce
    lo, hi = min(U, rank * per), min(U, rank * per + per)
    mine = torch.zeros((per, input_embs.shape[-1]), dtype=input_embs.dtype, device=dev)
    if hi > lo:
        mine[:hi - lo] = module.user_encoder(input_embs[lo:hi].contiguous(), lm[lo:hi].contiguous(), dev)[:, -1]
    allv = torch.empty((world * per, mine.shape[1]), dtype=mine.dtype, device=dev)
    dist.all_gather_into_tensor(allv, mine)
    return allv[:U].contiguous()


def eval_model(model, user_history, eval_seq, item_embeddings, test_batch_size, args, item_num, Log_file, v_or_t,
               local_rank):
    """metrics.py:82-116: HR@10 / NDCG@10 of full ranking; logs both, returns mean Hit10."""
    topK = 10
    Log_file.info(v_or_t + "_methods   {}".format('\t'.join(['Hit{}'.format(topK), 'nDCG{}'.format(topK)])))
    if not isinstance(item_embeddings, ItemTable):
        rank, world = _dist_info()
        assert world == 1, "pass the ItemTable returned by get_item_embeddings when running distributed"
        dev = next(core_model(model).parameters()).device
        item_embeddings = ItemTable(item_embeddings.to(dev), 0, item_embeddings.shape[0])
    tok, mask, tgt, hist = build_eval_arrays(eval_seq, user_history, args.max_seq_len)
    hit, ndcg, _ = eval_arrays(model, torch.from_numpy(tok), torch.from_numpy(mask), torch.from_numpy(tgt),
                               torch.from_numpy(hist), item_embeddings, test_batch_size, topk=topK)
    mean_eval = [float(hit.mean()), float(ndcg.mean())]
    print_metrics(mean_eval, Log_file, v_or_t)
    return mean_eval[0]


def metrics_topK(y_score, y_true, item_rank, topK, local_rank):
    """metrics.py:51-59 for ONE user, kept for API compatibility (scores already masked, id 0 dropped):
    rank = 1 + #{j: s_j > s_t} with ties resolved (score desc, id asc).  Host-side; the evaluator itself uses the
    fused kernels."""
    t = int(torch.argmax(y_true))
    s = y_score.float()
    ahead = int(((s > s[t]) | ((s == s[t]) & (torch.arange(s.numel(), device=s.device) < t))).sum())
    rank = ahead + 1
    out = torch.zeros(2, device=y_score.device)
    if rank <= topK:
        out[0] = 1
        out[1] = 1 / math.log2(rank + 1)
    return out
