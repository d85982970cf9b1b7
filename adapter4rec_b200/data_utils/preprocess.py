"""The text tree's readers — the data formats on the INPUT side of the hot path — mirroring
Downstream/Text/data_utils/preprocess.py (identical in Pretraining/Text): the news TSV (`doc_name \\t title`) becomes the
token matrix `item_content [I+1, 2L]` (ids | attention mask, row 0 = the padding item) that the item encoder and the device
batch sampler read, and the behaviours TSV (`user \\t space-separated doc names`) becomes the train / valid / test sequences
and the history tensors of the evaluator.  Same function names, arguments and return structures as the reference, so
`run.py`'s call sites (Downstream/Text/run.py:319-341) read the same; the results are pinned bit for bit against the unmodified
reference on a fixture with every edge case (tests/golden/make_golden_preprocess.py, tests/test_preprocess_cpu.py).

Host-side, once per run; nothing here touches the GPU.  The tokenizer is whatever the caller passes (the reference passes
transformers' BertTokenizer / RobertaTokenizer: any callable `tok(text, max_length=, padding='max_length', truncation=True)`
returning `{'input_ids': [...], 'attention_mask': [...]}` of exactly max_length entries works)."""
import types

import numpy as np
import torch


def _rows(path):
    with open(path, "r") as f:
        for line in f:
            yield line.strip('\n').split('\t')


def read_news(news_path):
    """preprocess.py:64-75 (the id tower's reader; kept for signature completeness): 1-based ids in file order."""
    item_id_to_dic, item_name_to_id = {}, {}
    for item_id, (doc_name, _) in enumerate(_rows(news_path), start=1):
        item_name_to_id[doc_name] = item_id
        item_id_to_dic[item_id] = doc_name
    return item_id_to_dic, item_name_to_id


def read_images(images_path):
    """Downstream/CV/data_utils/preprocess.py:71-83 (the image tree's catalogue reader): 1-based ids in file order, the LMDB key
    of an item is its name in ASCII.  The image tree's `read_behaviors` (same file, :5-68) applies the rules of the text
    tree's to these dictionaries — it is the function below; only its log lines differ."""
    item_id_to_keys, item_name_to_id = {}, {}
    for index, fields in enumerate(_rows(images_path), start=1):
        item_name_to_id[fields[0]] = index
        item_id_to_keys[index] = fields[0].encode('ascii')
    return item_id_to_keys, item_name_to_id


def read_news_bert(news_path, args, tokenizer):
    """preprocess.py:78-106.  Ids are 1-based in file order (a repeated doc_name keeps its LAST id, every line still takes an
    id); the title is lower-cased and tokenised to exactly --num_words_title entries.  Only the `title` attribute is
    functional in the reference (its `abstract` / `body` branches read variables the two-column TSV never defines and raise
    NameError); they are refused here with the reason instead."""
    unsupported = [a for a in args.news_attributes if a in ('abstract', 'body')]
    if unsupported:
        raise NotImplementedError("news_attributes %r: the reference's reader only defines the title column "
                                  "(preprocess.py:84-100)" % (unsupported,))
    with_title = 'title' in args.news_attributes
    item_id_to_dic, item_name_to_id = {}, {}
    for item_id, (doc_name, title) in enumerate(_rows(news_path), start=1):
        enc = tokenizer(title.lower(), max_length=args.num_words_title, padding='max_length', truncation=True) \
            if with_title else []
        item_name_to_id[doc_name] = item_id
        item_id_to_dic[item_id] = [enc, [], []]
    return item_id_to_dic, item_name_to_id


def read_behaviors(behaviors_path, before_item_id_to_dic, before_item_name_to_id, max_seq_len, min_seq_len, Log_file):
    """preprocess.py:5-61.  Users with fewer than min_seq_len interactions are dropped; the last max_seq_len + 3 interactions
    are kept; items nobody kept are dropped and the rest renumbered 1..item_num in their old order; per user
    train = seq[:-2], valid = seq[-(S+2):-1], test = seq[-(S+1):], histories = train / seq[:-1].  A user name that appears
    twice keeps its first position and its last sequence, while the interactions of BOTH lines count for the item filter —
    as in the reference."""
    Log_file.info("##### news number {} {} (before clearing)#####".format(len(before_item_id_to_dic),
                                                                          len(before_item_name_to_id)))
    Log_file.info("##### min seq len {}, max seq len {}#####".format(min_seq_len, max_seq_len))
    before_item_num = len(before_item_name_to_id)
    used = np.zeros(before_item_num + 1, dtype=bool)
    user_seqs, seq_num = {}, 0
    for fields in _rows(behaviors_path):
        names = fields[1].split(' ')
        if len(names) < min_seq_len:
            continue
        seq = np.fromiter((before_item_name_to_id[n] for n in names[-(max_seq_len + 3):]), dtype=np.int64)
        user_seqs[fields[0]] = seq
        used[seq] = True
        seq_num += 1
    used[0] = False
    kept = np.flatnonzero(used)                                  # old ids that survive, ascending
    new_id = np.zeros(before_item_num + 1, dtype=np.int64)
    new_id[kept] = np.arange(1, kept.size + 1)
    item_num = int(kept.size)
    item_id_to_dic = {i + 1: before_item_id_to_dic[int(old)] for i, old in enumerate(kept)}
    Log_file.info("##### items after clearing {}, {}, {} #####".format(item_num, item_num, len(item_id_to_dic)))

    users_train, users_valid, users_test, hist_valid, hist_test = {}, {}, {}, {}, {}
    for user_id, seq in enumerate(user_seqs.values()):
        s = new_id[seq].tolist()
        users_train[user_id] = s[:-2]
        users_valid[user_id] = s[-(max_seq_len + 2):-1]
        users_test[user_id] = s[-(max_seq_len + 1):]
        hist_valid[user_id] = torch.LongTensor(np.array(s[:-2]))
        hist_test[user_id] = torch.LongTensor(np.array(s[:-1]))
    Log_file.info("##### user seqs after clearing {}, {}, {}, {}, {}#####".
                  format(seq_num, len(user_seqs), len(users_train), len(users_valid), len(users_test)))
    return item_num, item_id_to_dic, users_train, users_valid, users_test, hist_valid, hist_test


def get_doc_input_bert(item_id_to_content, args):
    """preprocess.py:109-151: int32 [I+1, L] token ids and attention masks per attribute (row 0 stays all zero: the padding
    item), None for the attributes not in --news_attributes."""
    item_num = len(item_id_to_content) + 1
    if 'title' not in args.news_attributes:
        return None, None, None, None, None, None
    news_title = np.zeros((item_num, args.num_words_title), dtype='int32')
    news_title_attmask = np.zeros((item_num, args.num_words_title), dtype='int32')
    for item_id in range(1, item_num):
        title = item_id_to_content[item_id][0]
        news_title[item_id] = title['input_ids']
        news_title_attmask[item_id] = title['attention_mask']
    return news_title, news_title_attmask, None, None, None, None


def load_text_data(args, tokenizer, Log_file, use_modal=True):
    """The reader block of run.py:319-341 in one call: the namespace `train(args, use_modal, local_rank, data)` of
    adapter4rec_b200.run / adapter4rec_b200.pretraining.text_run takes (item_content = the concatenation of the present
    token / mask matrices, run.py:336-341).  use_modal = False (the id tower): the catalogue is read by name only
    (read_news, no tokenizer) and item_content is None."""
    import os
    root = os.path.join(args.root_data_dir, args.dataset)
    if use_modal:
        before_dic, before_name_to_id = read_news_bert(os.path.join(root, args.news), args, tokenizer)
    else:
        before_dic, before_name_to_id = read_news(os.path.join(root, args.news))
    item_num, item_id_to_dic, users_train, users_valid, users_test, hist_valid, hist_test = read_behaviors(
        os.path.join(root, args.behaviors), before_dic, before_name_to_id, args.max_seq_len, args.min_seq_len, Log_file)
    item_content = None
    if use_modal:
        item_content = np.concatenate([x for x in get_doc_input_bert(item_id_to_dic, args) if x is not None], axis=1)
    return types.SimpleNamespace(item_content=item_content, item_num=item_num, users_train=users_train,
                                 users_valid=users_valid, users_test=users_test, users_history_for_valid=hist_valid,
                                 users_history_for_test=hist_test)
