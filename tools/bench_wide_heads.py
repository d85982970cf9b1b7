"""Wider SASRec user encoders: what 128-wide attention heads cost.

1. a4r_attn_small_fwd / _bwd at head_dim 32, 64 and 128 at one SASRec-like shape (65,536 histories x L = 20, 2 heads,
   causal, f32 log_mask), with and without probability dropout.  The widths alternate inside every round so that they
   share the card's state; the median over rounds is reported.  Algorithmic bytes: forward q, k, v read + ctx written;
   backward q, k, v, dctx read + dq, dk, dv written (the mask adds 4 B per token in both).  Every working set is above
   the 126 MB L2 (smallest: d = 32 forward, 503 MB of qkv).
2. The C2-shaped train step (bench.make_args: BERT-base + LoRA r = 8, 512 users x 20 positions, dropout 0.1) at D = 64
   and at D = 256 with 2 heads, CUDA events over --steps steps after --warmup.
3. Evaluator scoring at d = 256: a4r_score_topk + merge of 4,096 users against 1 M items (512 MB of bf16 table).
The card name and power limit are read in the same run.

    python tools/bench_wide_heads.py [--out profiles/wide_heads.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from adapter4rec_b200 import lib, ops  # noqa: E402

HBM = 7.7e12     # B/s, HGX B200 data sheet, one GPU

ap = argparse.ArgumentParser()
ap.add_argument("--seqs", type=int, default=65536)
ap.add_argument("--rounds", type=int, default=7)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--users-per-pass", type=int, default=256)
ap.add_argument("--eval-users", type=int, default=4096)
ap.add_argument("--eval-items", type=int, default=1_000_000)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wide_heads.json"))
a = ap.parse_args()

torch.cuda.set_device(0)
lib.get_lib()
dev = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn, reps):
    """device ms per call: CUDA events around `reps` back-to-back calls"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def attention():
    N, L, heads = a.seqs, 20, 2
    g = torch.Generator(device=dev).manual_seed(1)
    lens = torch.randint(1, L + 1, (N,), generator=g, device=dev)
    mask = (torch.arange(L, device=dev)[None, :] >= (L - lens)[:, None]).float()       # left-padded log_mask
    cases = {}
    for dh in (32, 64, 128):
        H = heads * dh
        qkv = (torch.randn((N * L, 3 * H), generator=g, device=dev) * 0.5).to(torch.bfloat16)
        dctx = (torch.randn((N * L, H), generator=g, device=dev) * 0.5).to(torch.bfloat16)
        for drop in (None, (0.1, 1234, 1 << 33)):
            kw = dict(mask=mask, causal=True, mask_neg=-1e9, dropout=drop)
            fwd = (lambda qkv=qkv, kw=kw, dh=dh: ops.attn_small_fwd(qkv, N, L, heads, dh, **kw))
            bwd = (lambda qkv=qkv, dctx=dctx, kw=kw, dh=dh: ops.attn_small_bwd(qkv, dctx, N, L, heads, dh, **kw))
            fwd(), bwd()
            tok = N * L
            cases[(dh, drop is not None)] = dict(fwd=fwd, bwd=bwd, fwd_bytes=4 * tok * H * 2 + tok * 4,
                                                 bwd_bytes=7 * tok * H * 2 + tok * 4, ms_fwd=[], ms_bwd=[])
    torch.cuda.synchronize()
    for _ in range(a.rounds):
        for c in cases.values():          # every width and dropout setting once per round, in turn
            c["ms_fwd"].append(timed(c["fwd"], a.reps))
            c["ms_bwd"].append(timed(c["bwd"], a.reps))
    out = []
    for (dh, drop), c in cases.items():
        row = {"head_dim": dh, "dropout": 0.1 if drop else 0.0, "seqs": N, "L": L, "heads": heads}
        for d in ("fwd", "bwd"):
            ms = statistics.median(c["ms_" + d])
            b = c[d + "_bytes"]
            row[d] = {"ms": ms, "ms_min_max": [min(c["ms_" + d]), max(c["ms_" + d])], "algorithmic_bytes": b,
                      "gb_per_s": b / (ms / 1e3) / 1e9, "share_of_hbm_datasheet": b / (ms / 1e3) / HBM}
        out.append(row)
    return out


def train_step(D):
    from adapter4rec_b200 import surgery
    from adapter4rec_b200.model import BertModel, Model, TextConfigLite
    from adapter4rec_b200.trainer import FlatAdamTrainer
    torch.manual_seed(123456)
    args = bench.make_args()
    args.embedding_dim = D
    model = Model(args, bench.ITEMS, True, BertModel(TextConfigLite())).to(dev)
    surgery.freeze_all(model)
    surgery.insert_adapters(model, args)
    model.train()
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_bert_lr, args.adapter_sasrec_lr,
                              users_per_pass=a.users_per_pass)
    gen = torch.Generator().manual_seed(123456)
    cat = bench.synth_catalogue(gen)
    batches = [tuple(t.to(dev) for t in bench.synth_batch(cat, 512, gen)) for _ in range(3)]
    for i in range(a.warmup):
        trainer.train_step(*batches[i % 3])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps):
        loss = trainer.train_step(*batches[i % 3])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    res = {"embedding_dim": D, "heads": args.num_attention_heads, "head_dim": D // args.num_attention_heads, "users": 512,
           "users_per_pass": a.users_per_pass, "ms_per_step": ms, "user_seqs_per_s": 512 / (ms / 1e3),
           "loss_after_steps": float(loss)}
    del model, trainer, batches
    torch.cuda.empty_cache()
    return res


def scoring():
    U, I, d = a.eval_users, a.eval_items, 256
    g = torch.Generator(device=dev).manual_seed(3)
    users = torch.randn((U, d), generator=g, device=dev).to(torch.bfloat16)
    items = torch.randn((I, d), generator=g, device=dev).to(torch.bfloat16)
    hist = torch.randint(1, I, (U, 20), generator=g, device=dev).int()
    tgt = torch.randint(1, I, (U,), generator=g, device=dev).int()

    def run():
        sc, ids = ops.score_topk(users, items, id_base=0, history=hist, k=10)
        return ops.topk_merge(sc, ids, target=tgt)
    run()
    ms = statistics.median(timed(run, 5) for _ in range(5))
    return {"users": U, "items": I, "dim": d, "ms": ms, "users_per_s": U / (ms / 1e3),
            "what": "a4r_score_topk (history masked, top-10) + merge with HR / NDCG, whole table per call"}


out = {"what": "128-wide SASRec attention heads: kernel bandwidth, C2 train step at D = 64 vs 256, d = 256 scoring",
       "card": card(), "attention_small": attention(), "train_step_c2": [train_step(64), train_step(256)],
       "eval_scoring_d256": scoring()}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
