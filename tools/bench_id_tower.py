"""ID-embedding item tower (--item_tower id): one training step of SASRec over an nn.Embedding item table at B = 512 users,
S = 20, D = 64, for the Adressa catalogue (20,374 items) and a 10 M-item synthetic catalogue, plus the full-ranking
evaluation of 4,096 users against the whole table (C5-style: every item scored, top-10).

Reported per catalogue: step time and user-seqs/s (CUDA events over --steps steps after --warmup, three rotating resident
batches); device time of the gather kernel, of the stable id sort (the one ATen op on the path) and of the table-gradient
kernel, each with its algorithmic bytes and the share of the 7.7 TB/s HBM3e data-sheet bandwidth those bytes would need;
the dense table passes of the step (zero_grad + Adam over the flat buffer: 20 GB per step at 10 M x 64); the evaluation time.
The card name and power limit are read in the same run.

    python tools/bench_id_tower.py [--out profiles/id_tower.json]"""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from adapter4rec_b200 import lib, ops  # noqa: E402
from adapter4rec_b200.data_utils import metrics as M  # noqa: E402
from adapter4rec_b200.model import Model  # noqa: E402
from adapter4rec_b200.trainer import FlatAdamTrainer  # noqa: E402

HBM = 7.7e12     # B/s, HGX B200 data sheet, one GPU

ap = argparse.ArgumentParser()
ap.add_argument("--items", type=int, nargs="+", default=[20374, 10_000_000])
ap.add_argument("--users", type=int, default=512)
ap.add_argument("--seq", type=int, default=20)
ap.add_argument("--dim", type=int, default=64)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=5)
ap.add_argument("--reps", type=int, default=200)
ap.add_argument("--eval-users", type=int, default=4096)
ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "id_tower.json"))
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
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel(name, ms, nbytes):
    return {"what": name, "ms": ms, "algorithmic_bytes": nbytes, "gb_per_s": nbytes / (ms / 1e3) / 1e9,
            "share_of_hbm_datasheet": nbytes / (ms / 1e3) / HBM}


def one(I):
    B, S, D = a.users, a.seq, a.dim
    S1, R = S + 1, a.users * (a.seq + 1) * 2
    args = types.SimpleNamespace(max_seq_len=S, l2_weight=0, embedding_dim=D, num_attention_heads=2, drop_rate=0.1,
                                 transformer_block=2)
    torch.manual_seed(123456)
    model = Model(args, I, False, None).to(dev)
    model.train()
    trainer = FlatAdamTrainer(model, 1e-4, 1e-4, 1e-4, 1e-4, users_per_pass=B, overlap=False)
    g = torch.Generator(device=dev).manual_seed(7)
    batches = []
    for _ in range(3):
        ids = torch.randint(1, I + 1, (B, S1, 2), generator=g, device=dev)
        batches.append((ids.view(B * S1, 2), torch.ones(B, S, device=dev)))
    for i in range(a.warmup):
        trainer.train_step(*batches[i % 3])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps):
        loss = trainer.train_step(*batches[i % 3])
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / a.steps

    w = model.id_embedding.weight.detach()
    ids = batches[0][0].view(B, S1, 2)
    emb, hist = ops.id_embed_fwd(w, ids)
    gather_ms = timed(lambda: ops.id_embed_fwd(w, ids), a.reps)
    sort_ms = timed(lambda: torch.sort(ids.view(-1), stable=True), a.reps)
    sorted_ids, order = torch.sort(ids.view(-1), stable=True)
    distinct = int(torch.unique(sorted_ids).numel())
    grad = trainer.flat_grad[:w.numel()].view(w.shape)       # id_embedding.weight comes first in the --lr group

    def bwd():
        lib.check(lib.get_lib().a4r_id_embed_bwd(ops._p(sorted_ids), ops._p(order), ops._p(emb), ops._p(hist), ops._p(grad),
                                                 w.shape[0], D, B, S1, 0, 1, ops._stream()), "a4r_id_embed_bwd")
    bwd_ms = timed(bwd, a.reps)
    n = trainer.flat_param.numel()
    zero_ms = timed(trainer.zero_grad, 20)

    def adam():
        for _, lr, off, k in trainer.segments:
            ops.adam_step(trainer.flat_param[off:off + k], trainer.flat_grad[off:off + k], trainer.exp_avg[off:off + k],
                          trainer.exp_avg_sq[off:off + k], lr, 0.9, 0.999, 1e-8, 0.0, 1)
    adam_ms = timed(adam, 20)

    U = a.eval_users
    tok = torch.randint(1, I + 1, (U, S), generator=g, device=dev)
    tgt = torch.randint(1, I + 1, (U,), generator=g, device=dev).int()
    mask = torch.ones(U, S, device=dev)

    def evaluate():
        table = M.get_item_embeddings(model, None, 512, args, False, 0)
        return M.eval_arrays(model, tok, mask, tgt, tok.int(), table, 1024)
    eval_ms = timed(evaluate, 3)
    return {
        "items": I, "users": B, "seq": S, "dim": D, "step_ms": step_ms, "user_seqs_per_s": B / (step_ms / 1e3),
        "loss": float(loss), "trainable_params": n, "distinct_ids_in_batch": distinct,
        "gather": kernel("a4r_id_embed_fwd", gather_ms, R * 8 + R * D * 4 + R * D * 2 + B * S * D * 2),
        "sort": kernel("torch.sort(stable=True), int64 keys + int64 indices", sort_ms, R * 8 + 2 * R * 8),
        "backward": kernel("a4r_id_embed_bwd (accumulate)", bwd_ms, 2 * R * 8 + R * D * 2 + B * S * D * 2 + 2 * distinct * D * 4),
        "dense_table_passes": {"zero_grad_ms": zero_ms, "adam_ms": adam_ms,
                               "algorithmic_bytes": 4 * n + 7 * 4 * n,
                               "share_of_hbm_datasheet": (4 * n + 7 * 4 * n) / ((zero_ms + adam_ms) / 1e3) / HBM},
        "eval_full_ranking": {"users": U, "ms": eval_ms, "what": "table cast + user encoder + score/top-10 over all items"},
    }


out = {"what": "ID-embedding item tower, one training step + full-ranking evaluation", "card": card(),
       "runs": [one(I) for I in a.items]}
os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
with open(a.out, "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out))
