"""Runs the UNMODIFIED image-tree readers (Downstream/CV/data_utils/preprocess.py: read_images, read_behaviors) on the REAL
catalogue / behaviour files the reference ships (Dataset/Amazon/amazon_2w_{items,users}.tsv) and stores digests of what they
return in tests/golden/preprocess/amazon_digest.json.  The data files are not part of this repository, so the suite does not
read the digest: it records what the unmodified readers returned on them."""
import hashlib
import importlib.util
import json
import logging
import os

HERE = os.path.dirname(os.path.abspath(__file__))
ITEMS = "/root/reference/Dataset/Amazon/amazon_2w_items.tsv"
USERS = "/root/reference/Dataset/Amazon/amazon_2w_users.tsv"


def digest(item_num, item_id_to_keys, tr, va, te, hv, ht):
    h = hashlib.sha256()
    h.update(repr(item_num).encode())
    h.update(repr(sorted(item_id_to_keys.items())).encode())
    for d in (tr, va, te):
        h.update(repr(sorted(d.items())).encode())
    for d in (hv, ht):
        h.update(repr(sorted((k, v.tolist()) for k, v in d.items())).encode())
    return h.hexdigest()


if __name__ == "__main__":
    spec = importlib.util.spec_from_file_location("ref_cv_preprocess", "/root/reference/Downstream/CV/data_utils/preprocess.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    keys, name_to_id = ref.read_images(ITEMS)
    out = ref.read_behaviors(USERS, keys, name_to_id, 10, 5, logging.getLogger("golden"))
    rec = {"max_seq_len": 10, "min_seq_len": 5, "before_items": len(name_to_id), "item_num": out[0], "users": len(out[2]),
           "sha256": digest(*out)}
    with open(os.path.join(HERE, "preprocess", "amazon_digest.json"), "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print(rec)
