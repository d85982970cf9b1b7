"""CPU: adapter4rec_b200.data_utils.preprocess (news / behaviours TSV -> item_content, user sequences, histories) against what
the UNMODIFIED reference readers returned on the same fixture (tests/golden/make_golden_preprocess.py ran
Downstream/Text/data_utils/preprocess.py here; golden.json holds its outputs).  Integer work: everything must be equal."""
import json
import logging
import os
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import preprocess_fixture as F  # noqa: E402


def _args(attrs=('title',)):
    return types.SimpleNamespace(news_attributes=list(attrs), num_words_title=F.NUM_WORDS, num_words_abstract=50,
                                 num_words_body=50, root_data_dir=os.path.dirname(F.DIR), dataset=os.path.basename(F.DIR),
                                 news=os.path.basename(F.NEWS), behaviors=os.path.basename(F.BEHAVIORS),
                                 max_seq_len=F.MAX_SEQ_LEN, min_seq_len=F.MIN_SEQ_LEN)


@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(F.DIR, "golden.json")))


def _int_keys(d):
    return {int(k): v for k, v in d.items()}


def test_readers_equal_the_reference(gold):
    from adapter4rec_b200.data_utils import preprocess as P
    log = logging.getLogger("preprocess_test")
    args = _args()
    before_dic, before_name_to_id = P.read_news_bert(F.NEWS, args, F.toy_tokenizer)
    assert len(before_name_to_id) == gold["before_item_num"] and list(before_dic) == list(range(1, 121))
    item_num, item_id_to_dic, tr, va, te, hv, ht = P.read_behaviors(F.BEHAVIORS, before_dic, before_name_to_id,
                                                                    F.MAX_SEQ_LEN, F.MIN_SEQ_LEN, log)
    assert item_num == gold["item_num"] == len(item_id_to_dic)
    assert tr == _int_keys(gold["users_train"]) and va == _int_keys(gold["users_valid"]) and te == _int_keys(gold["users_test"])
    assert list(tr) == list(range(len(tr)))                                       # user ids in file order
    for got, ref in ((hv, gold["users_history_for_valid"]), (ht, gold["users_history_for_test"])):
        assert {k: v.tolist() for k, v in got.items()} == _int_keys(ref)
        assert all(v.dtype == torch.int64 for v in got.values())
    title, mask, *rest = P.get_doc_input_bert(item_id_to_dic, args)
    assert all(r is None for r in rest)
    content = np.concatenate([title, mask], axis=1)
    assert str(content.dtype) == gold["item_content_dtype"] == "int32"
    assert content.tolist() == gold["item_content"]
    assert not content[0].any()                                                   # row 0: the padding item
    ids, names = P.read_news(F.NEWS)
    assert len(ids) == gold["read_news"]["ids"] and ids[1] == gold["read_news"]["first"] and names[ids[7]] == 7


def test_load_text_data_feeds_the_entry_scripts(gold):
    """the reader block of Downstream/Text/run.py:319-341 in one call, in the shape run.train / text_run.train consume"""
    from adapter4rec_b200.data_utils import preprocess as P
    from adapter4rec_b200.run import build_train_batch
    data = P.load_text_data(_args(), F.toy_tokenizer, logging.getLogger("preprocess_test"))
    assert data.item_num == gold["item_num"] and data.item_content.tolist() == gold["item_content"]
    assert data.users_test == _int_keys(gold["users_test"])
    users = sorted(data.users_train)[:5]
    items, log_mask = build_train_batch(users, data.users_train, data.item_content, data.item_num, F.MAX_SEQ_LEN)
    assert tuple(items.shape) == (5, F.MAX_SEQ_LEN + 1, 2, 2 * F.NUM_WORDS) and tuple(log_mask.shape) == (5, F.MAX_SEQ_LEN)
    for b, u in enumerate(users):
        n = len(data.users_train[u])
        assert int(log_mask[b].sum()) == n - 1
        assert items[b, F.MAX_SEQ_LEN + 1 - n:, 0].tolist() == data.item_content[data.users_train[u]].tolist()


def test_edge_cases(tmp_path):
    """sequence-length filter and left truncation, renumbering of the surviving items, a repeated user name, the reference's
    non-functional attributes, unknown item names"""
    from adapter4rec_b200.data_utils import preprocess as P
    log = logging.getLogger("preprocess_test")
    news = tmp_path / "news.tsv"
    news.write_text("".join("d%d\tTitle %d\n" % (i, i) for i in range(1, 13)))
    beh = tmp_path / "b.tsv"
    beh.write_text("a\td1 d2 d3\n"                                   # 3 < min_seq_len 4: dropped
                   "b\td12 d11 d10 d9 d8 d7 d6 d5 d4\n"              # 9 > S + 3 = 7: the last 7 kept
                   "c\td2 d4 d6 d8\n"
                   "b\td5 d6 d7 d8\n")                               # b again: first position, last sequence
    args = _args()
    dic, name_to_id = P.read_news_bert(str(news), args, F.toy_tokenizer)
    item_num, id_to_dic, tr, va, te, hv, ht = P.read_behaviors(str(beh), dic, name_to_id, 4, 4, log)
    # kept old ids: {10,9,8,7,6,5,4} u {2,4,6,8} u {5,6,7,8} = {2,4,5,6,7,8,9,10} -> new ids 1..8
    assert item_num == 8 and [id_to_dic[i][0]['input_ids'][2] for i in (1, 8)] == \
        [F.toy_tokenizer("title %d" % d, 9, 'max_length', True)['input_ids'][2] for d in (2, 10)]
    assert list(tr) == [0, 1] and te[0] == [3, 4, 5, 6] and te[1] == [1, 2, 4, 6]       # user 0 = b (last line), user 1 = c
    assert tr[0] == [3, 4] and va[0] == [3, 4, 5] and hv[0].tolist() == [3, 4] and ht[0].tolist() == [3, 4, 5]
    with pytest.raises(NotImplementedError):
        P.read_news_bert(str(news), _args(('title', 'abstract')), F.toy_tokenizer)
    beh.write_text("z\td1 d2 d3 nope\n")
    with pytest.raises(KeyError):
        P.read_behaviors(str(beh), dic, name_to_id, 4, 4, log)
    assert P.get_doc_input_bert(id_to_dic, _args(())) == (None,) * 6


def test_load_body_and_the_real_tokenizer(tmp_path):
    """run.load_body reads tokenizer + config from the reference's directory layout (Downstream/Text/run.py:295-300); with
    transformers' BertTokenizer the token rows are [CLS] ids [SEP] padded to --num_words_title, mask = 1 on the real tokens —
    the row format the synthetic bench catalogue imitates (SURVEY.md §8d)."""
    from adapter4rec_b200 import run
    from adapter4rec_b200.data_utils import preprocess as P
    name = F.write_tiny_body(str(tmp_path))
    args = _args()
    args.bert_model_load = name
    tokenizer, cfg, state = run.load_body(args, pretrained_root=str(tmp_path))
    assert state is None and cfg.hidden_size == 128 and cfg.num_hidden_layers == 2 and cfg.vocab_size == 18
    data = P.load_text_data(args, tokenizer, logging.getLogger("preprocess_test"))
    L = F.NUM_WORDS
    ids, mask = data.item_content[:, :L], data.item_content[:, L:]
    assert data.item_content.shape == (data.item_num + 1, 2 * L) and not data.item_content[0].any()
    n = mask[1:].sum(1)
    assert (ids[1:, 0] == 2).all() and (ids[np.arange(1, len(ids)), n - 1] == 3).all()       # [CLS] ... [SEP]
    assert ((ids[1:] != 0) == (mask[1:] == 1)).all() and ids.max() < cfg.vocab_size and n.min() >= 2 and n.max() == L
