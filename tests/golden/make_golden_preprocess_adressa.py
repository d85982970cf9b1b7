"""Runs the UNMODIFIED text readers (Downstream/Text/data_utils/preprocess.py: read_news_bert, get_doc_input_bert) with the
REAL tokenizer (transformers' BertTokenizer on the vocab.txt the reference ships under pretrained_models/bert/bert_base_uncased)
on the REAL catalogue the reference ships (Dataset/Adressa/Adressa_news_base.tsv, 20,373 news titles, --num_words_title 30) and
stores a digest of the token matrix in tests/golden/preprocess/adressa_digest.json.  This is the item side of BASELINE.json's
configs[0] plumbing run.  The files are not part of this repository, so the suite does not read the digest: it records what
the unmodified readers produced (DESIGN.md cites its token count)."""
import hashlib
import importlib.util
import json
import os
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
NEWS = "/root/reference/Dataset/Adressa/Adressa_news_base.tsv"
BODY = "/root/reference/Downstream/Text/pretrained_models/bert/bert_base_uncased"
ARGS = types.SimpleNamespace(news_attributes=['title'], num_words_title=30, num_words_abstract=50, num_words_body=50)


def token_matrix(module, tokenizer):
    dic, name_to_id = module.read_news_bert(NEWS, ARGS, tokenizer)
    title, mask, *_ = module.get_doc_input_bert(dic, ARGS)
    return np.concatenate([title, mask], axis=1), name_to_id


def digest(content, name_to_id):
    h = hashlib.sha256()
    h.update(str(content.dtype).encode() + repr(content.shape).encode())
    h.update(np.ascontiguousarray(content).tobytes())
    h.update(repr(sorted(name_to_id.items())[:50]).encode())
    return h.hexdigest()


if __name__ == "__main__":
    from transformers import BertTokenizer
    spec = importlib.util.spec_from_file_location("ref_preprocess", "/root/reference/Downstream/Text/data_utils/preprocess.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    content, name_to_id = token_matrix(ref, BertTokenizer.from_pretrained(BODY))
    rec = {"rows": int(content.shape[0]), "cols": int(content.shape[1]), "names": len(name_to_id),
           "mean_tokens": float(content[1:, 30:].sum(1).mean()), "sha256": digest(content, name_to_id)}
    with open(os.path.join(HERE, "preprocess", "adressa_digest.json"), "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print(rec)
