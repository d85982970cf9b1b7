"""Train-batch assembly on the device, the counterpart of Downstream/Text/data_utils/dataset.py:10-49
(BuildTrainDataset + the DataLoader around it, run.py:347-357,587-594).

The reference builds every sample in a DataLoader worker: a Python rejection loop per history position and a NumPy
fancy index of 2(S+1) token rows per user, then ships [B, S+1, 2, 2L] int64 (10 MB at B = 512, L = 30) to the GPU.
Here the item token table (I+1 rows of 2L int64: 38 MB for 80 k items) and all user sequences live in HBM; a step
sends only the user indices of the batch and one kernel (a4r_sample_train_batch) draws the negatives and gathers the
rows.  Same sample layout, same log_mask, same admissibility rule for negatives; the random STREAM differs (counter
based, reproducible from (seed, step)) — Python's Mersenne Twister is not reproduced."""
import numpy as np
import torch

from .. import ops

ATTEMPTS = 64   # counters reserved per slot (must equal kMaxAttempts in csrc/batch_sampler.cu)


class BuildTrainDataset:
    """Same constructor as the reference's Dataset (dataset.py:11-16).  `__getitem__` keeps the reference's per-user
    contract for code that indexes it; `batch(users)` is the device path a training loop should call."""

    def __init__(self, u2seq, item_content, item_num, max_seq_len, use_modal=True, device=None, seed=123456):
        """use_modal = False (the id item tower): item_content is not read (may be None) and a sample is the item ids
        [S+1, 2] themselves; every id of u2seq must lie in [1, item_num] (checked here, once, on the host: the id tower's
        table has exactly item_num + 1 rows)."""
        self.u2seq = u2seq
        self.item_num = item_num
        self.max_seq_len = max_seq_len + 1
        self.use_modal = use_modal
        self.device = torch.device(device if device is not None else "cuda")
        self.seed = int(seed)
        self.batches_drawn = 0
        if use_modal:
            content = torch.as_tensor(np.asarray(item_content) if not torch.is_tensor(item_content) else item_content)
            self.item_content = content.to(device=self.device, dtype=torch.int64).contiguous()
        else:
            self.item_content = None
        self.users = sorted(u2seq.keys())
        self._row = {u: i for i, u in enumerate(self.users)}
        S1 = self.max_seq_len
        seqs = np.zeros((len(self.users), S1), dtype=np.int64)
        for i, u in enumerate(self.users):
            s = list(u2seq[u])
            assert 2 <= len(s) <= S1, "sequence length must be in [2, max_seq_len + 1] (preprocess.py:51-59)"
            seqs[i, S1 - len(s):] = s                                  # left padding, dataset.py:34
        if not use_modal and len(self.users):
            real = seqs[seqs != 0]
            if real.size != sum(len(u2seq[u]) for u in self.users) or real.min() < 1 or real.max() > item_num:
                raise ValueError("item_tower id: every item id of the sequences must lie in [1, item_num = %d]" % item_num)
        self.seqs = torch.from_numpy(seqs).to(self.device)

    def __len__(self):
        return len(self.u2seq)

    def batch(self, users, neg_items=None, check=False):
        """users: iterable of user ids -> (sample_items [B, S+1, 2, 2L] int64, log_mask [B, S] f32) on the device; the
        id tower's sample_items are the ids [B, S+1, 2] (history | negative).
        neg_items (optional int64 [B, S+1]) replays given negatives instead of sampling."""
        rows = torch.as_tensor([self._row[u] for u in users], dtype=torch.int64).to(self.device, non_blocking=True)
        seqs = self.seqs.index_select(0, rows)
        offset = self.batches_drawn * (1 << 40)                        # disjoint counter ranges per batch
        self.batches_drawn += 1
        neg_in = None if neg_items is None else neg_items.to(self.device, torch.int64).contiguous()
        out, log_mask, neg, fail = ops.sample_train_batch(seqs, self.item_content, self.item_num, self.seed, offset, neg_in)
        self.last_negatives = neg
        if check and int(fail.item()):
            raise RuntimeError("negative sampling found no admissible item (item_num <= max_seq_len + 1?)")
        if out is None:
            out = torch.stack([seqs, neg], -1)
        return out, log_mask

    def __getitem__(self, user_id):
        items, log_mask = self.batch([user_id])
        return items[0], log_mask[0]
