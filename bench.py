#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native TransRec hot path.

Workload (BASELINE.json configs[1], "C2" in SURVEY.md §8): SASRec + BERT-base, LoRA r=8 on query/value (and on the
SASRec w_Q/w_V), synthetic MIND-shape data (30-token titles, 20-item histories), bf16 activations with fp32
accumulation, 512 users per GPU per optimizer step, data-parallel.  One "step" = forward + backward + gradient
all-reduce + Adam over one batch of 512 users (= 21,504 item sequences = 645,120 tokens) per GPU.

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      # the reference's CPU arithmetic (oracle port) on the host cores

Prints ONE JSON line on rank 0 (contract in the task statement: metric/value/unit/n_gpus/.../roofline/cpu_baseline).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "train user-sequences/s (SASRec + BERT-base LoRA r=8 adapter-tuning step: fwd+bwd+allreduce+Adam)"
UNIT = "user-seqs/s"
S, L, D = 20, 30, 64
ITEMS = 80000
FLOP_FWD_PER_TOKEN = 12 * (14155776 + 92160 + 49152)   # SURVEY.md §8d: GEMMs + attention + LoRA r=8, per token, forward


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed training steps: of the headline loop and of the loops timed beside it (end to end, layouts, "
                         "graphed step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy: loss (float64) and the "
                         "trainable parameters after its Adam update and their gradients (float32, flat, trainer order)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--users", type=int, default=512, help="users per GPU per step (C2: 512)")
    ap.add_argument("--users-per-pass", type=int, default=512,
                    help="activation-memory pass size (exact gradient accumulation over passes); 512 = the whole batch in one pass "
                         "(112 GB peak of the 180 GB), 256 = two passes (60 GB)")
    ap.add_argument("--cpu-users", type=int, default=0,
                    help="users in the bounded CPU sample (default: 48 for cpu_baseline ~15 s, 16 per step for --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip the extra (non-headline) unpadded-token measurement")
    ap.add_argument("--variants", default="all",
                    help="comma list of the non-headline variants to run: layouts (unpadded / dedup), graphed_step, c1, c3, c4")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def make_args(r=8):
    import types
    return types.SimpleNamespace(
        max_seq_len=S, min_seq_len=5, l2_weight=0, embedding_dim=D, num_attention_heads=2, drop_rate=0.1,
        transformer_block=2, num_words_title=L, num_words_abstract=50, num_words_body=50, news_attributes=["title"],
        word_embedding_dim=768, bert_model_load="bert_base_uncased", bert_adapter_down_size=r, adapter_down_size=r,
        adapter_dropout_rate=0.1, adapter_activation="RELU", num_workers=0, adapter_type="lora", n_tokens=0,
        adding_adapter_to="all", is_serial="True", finetune_layernorm="None", fine_tune_to="None",
        lr=1e-4, fine_tune_lr=1e-5, adapter_bert_lr=5e-4, adapter_sasrec_lr=1e-4)


def synth_catalogue(gen):
    """SURVEY.md §8d: I rows of ids(30) | mask(30); [CLS]=101 at 0, [SEP]=102 at len-1, zeros beyond; row 0 all zero."""
    import torch
    ids = torch.randint(1000, 30522, (ITEMS + 1, L), generator=gen)
    lens = torch.randint(8, L + 1, (ITEMS + 1,), generator=gen)
    pos = torch.arange(L).unsqueeze(0)
    mask = (pos < lens.unsqueeze(1)).long()
    ids = ids * mask
    ids[:, 0] = 101
    ids[torch.arange(ITEMS + 1), lens - 1] = 102
    rows = torch.cat([ids, mask], 1)
    rows[0] = 0
    return rows


def synth_batch(catalogue, users, gen):
    """users x (S+1) distinct items + one sampled negative per position (not in the user's sequence), last negative
    slot = item 0 (dataset.py:24-49); log_mask all ones (no padding: executed work = algorithmic work)."""
    import torch
    seq = torch.stack([torch.randperm(ITEMS, generator=gen)[:S + 1] + 1 for _ in range(users)])
    neg = torch.randint(1, ITEMS + 1, (users, S + 1), generator=gen)
    for _ in range(4):   # rejection: resample negatives that hit the user's own sequence
        clash = (neg.unsqueeze(2) == seq.unsqueeze(1)).any(2)
        if not clash.any():
            break
        neg = torch.where(clash, torch.randint(1, ITEMS + 1, neg.shape, generator=gen), neg)
    neg[:, S] = 0
    ids = torch.stack([seq, neg], 2)                                  # [users, S+1, 2]
    sample_items = catalogue[ids].view(users * (S + 1) * 2, 2 * L)     # int64 ids | mask rows
    log_mask = torch.ones(users, S)
    return sample_items, log_mask


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, mx = [], set(), None
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx = float(p[2])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs run on rank 0 alone (the other ranks idle), so they
    take every core this process may run on.  Returns the thread count actually in use."""
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n))
    return torch.get_num_threads()


def oracle_step_factory(model_sd, users, seed=7):
    """One adapter-tuning step of the reference's arithmetic on the CPU (oracle port, fp32, torch CPU threads):
    forward + backward + torch.optim.Adam over `users` users of the same workload."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import transrec_oracle as O
    cfg = O.TextConfig(hidden=768, layers=12, heads=12, eps=1e-12)
    rec = O.RecConfig(max_seq_len=S, embedding_dim=D, heads=2, blocks=2, num_words_title=L)
    sd = {k: v.detach().float().cpu().clone() for k, v in model_sd.items()}
    train = [k for k in sd if "lora_" in k or (k.endswith("bias") and any(t in k for t in (".query.", ".value.", ".w_Q.", ".w_V.")))]
    for k in train:
        sd[k].requires_grad_(True)
    opt = torch.optim.Adam([sd[k] for k in train], lr=1e-4)
    gen = torch.Generator().manual_seed(seed)
    cat = synth_catalogue(gen)

    def step():
        items, mask = synth_batch(cat, users, gen)
        opt.zero_grad()
        loss = O.model_forward(items, mask, sd, cfg, rec)
        loss.backward()
        opt.step()
        return float(loss)

    return step


def cpu_eval_legs(model_sd, cores):
    """BASELINE.md §3 items 2-3 on the host cores (oracle port, fp32): the item-table encode over 512 catalogue rows, the
    reference evaluator's arithmetic (eval_model, metrics.py:82-116) at I = 100,000 / D = 64 / 256 users, and a clearly
    labelled RESTATEMENT for the C5 shape (chunked matmul + topk, I = 1 M, d = 768, 256 users; the reference evaluator
    itself cannot run C5: 80 MB of float64 labels per user, dataset.py:73-74)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import transrec_oracle as O
    cfg = O.TextConfig(hidden=768, layers=12, heads=12, eps=1e-12)
    rec = O.RecConfig(max_seq_len=S, embedding_dim=D, heads=2, blocks=2, num_words_title=L)
    sd = {k: v.detach().float().cpu() for k, v in model_sd.items()}
    out = {}
    gen = torch.Generator().manual_seed(31)
    cat = synth_catalogue(gen)[:512]
    with torch.no_grad():
        t0 = time.time()
        O.item_embeddings(cat, sd, cfg, rec, batch=512)
        dt = time.time() - t0
    out["item_encode"] = {"value": 512 / dt, "unit": "items/s", "cores": cores, "kind": "port",
                          "sample": "512 catalogue rows x %d tokens, BERT-base + LoRA forward, fp32, %.1f s" % (L, dt)}
    I, U = 100_000, 4096
    emb = torch.randn((I + 1, D), generator=gen) * 0.3
    seqs = [torch.randint(1, I + 1, (S + 1,), generator=gen).tolist() for _ in range(U)]
    hist = [q[:-1] for q in seqs]
    t0 = time.time()
    hit, _ = O.eval_model(seqs, hist, emb, sd, rec)
    dt = time.time() - t0
    out["eval_model_d64"] = {"value": U / dt, "unit": "users/s", "cores": cores, "kind": "port",
                             "sample": "%d users against %d items, D=%d: SASRec user encoder + score row + history mask + rank "
                                       "of the target per user (rank = 1 + #{s_j > s_t}; the reference argsorts every row: 58 users/s on "
                                       "8 cores, BASELINE.md §2), fp32, %.1f s" % (U, I, D, dt)}
    I5, d5, U5, chunk = 1_000_000, 768, 1024, 65536
    table = torch.empty((I5 + 1, d5), dtype=torch.bfloat16)
    for i in range(0, I5 + 1, chunk):
        j = min(I5 + 1, i + chunk)
        table[i:j] = (torch.randn((j - i, d5), generator=gen) * d5 ** -0.5).to(torch.bfloat16)
    users = torch.randn((U5, d5), generator=gen).to(torch.bfloat16).float()
    h5 = torch.randint(1, I5 + 1, (U5, S), generator=gen)
    t0 = time.time()
    best_s = torch.full((U5, 10), -float("inf"))
    best_i = torch.zeros((U5, 10), dtype=torch.long)
    for i in range(0, I5 + 1, chunk):
        j = min(I5 + 1, i + chunk)
        sc = users @ table[i:j].float().t()
        inside = (h5 >= i) & (h5 < j)
        rows = torch.arange(U5).unsqueeze(1).expand_as(h5)[inside]
        sc[rows, (h5 - i)[inside]] = -float("inf")
        if i == 0:
            sc[:, 0] = -float("inf")
        cs, ci = torch.topk(sc, 10, dim=1)
        ms, mi = torch.topk(torch.cat([best_s, cs], 1), 10, dim=1)
        best_i = torch.gather(torch.cat([best_i, ci + i], 1), 1, mi)
        best_s = ms
    dt = time.time() - t0
    out["c5_restatement"] = {"value": U5 / dt, "unit": "users/s", "cores": cores, "kind": "port",
                             "sample": "RESTATEMENT (chunked torch.matmul + torch.topk, history masked, id 0 dropped): %d users x "
                                       "%d items x d=%d, bf16 table -> fp32, %.1f s; C5 (10 M items) is 10x the items per user"
                                       % (U5, I5, d5, dt),
                             "extrapolated_c5_users_per_s": U5 / dt / 10.0}
    return out


def reference_sd():
    """Random-init C2 model on the CPU, only to obtain a state dict with the reference's key names for the oracle."""
    import torch
    from adapter4rec_b200 import surgery
    from adapter4rec_b200.model import BertModel, Model, TextConfigLite
    torch.manual_seed(123456)
    args = make_args()
    model = Model(args, ITEMS, True, BertModel(TextConfigLite()))
    surgery.freeze_all(model)
    surgery.insert_adapters(model, args)
    return model.state_dict()


def run_reference(a):
    """--impl reference: the reference's CPU arithmetic (oracle port) on all host threads, each step a bounded sample of C2
    (a.cpu_users users)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = use_all_host_threads()
    a.cpu_users = a.cpu_users or 16
    step = oracle_step_factory(reference_sd(), a.cpu_users)
    for _ in range(min(a.warmup, 1)):
        step()
    t0 = time.time()
    steps = a.steps
    for _ in range(steps):
        step()
    dt = (time.time() - t0) / steps
    v = a.cpu_users / dt
    sample = "%d users (= %d sequences x %d tokens) per step, fp32, torch CPU" % (a.cpu_users, a.cpu_users * 42, L)
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": min(a.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: SASRec(D=64,2 blocks)+BERT-base, LoRA r=8 on q/v, S=20, 30 tokens, bf16",
                   "users_per_gpu_per_step": 512, "sample": "bounded CPU sample of the same workload: %d users per step, fp32"
                   % a.cpu_users},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def bench_eval(dev, world, rank, steps, warmup):
    """Full-ranking evaluation, BASELINE.json configs[4] ("C5"): 10 M-item bf16 table (d = 768) sharded by item id over
    the ranks (all 10 M on one GPU at N = 1), blocks of 9,472 users with 20 history ids each, top-10 + HR/NDCG.
    User vectors are synthetic bf16 (kernel-level benchmark: score GEMM + mask + top-k + merge [+ all-gather]);
    the d = 64 line runs the COMPLETE evaluator (K10 gather, SASRec user encoder, scores, top-k, metrics) on a
    1 M-item table with the model's real embedding width."""
    import torch
    import torch.distributed as dist
    from adapter4rec_b200 import ops
    out = {}
    # 9,472 users = 37 blocks of 256 (one per CTA pair) x 2 item splits = 74 pairs = all 148 SMs of a B200
    I_total, d, U = 10_000_000, 768, 9472
    per = (I_total + 1 + world - 1) // world
    lo = rank * per
    n_local = max(0, min(I_total + 1, lo + per) - lo)
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    table = torch.empty((n_local, d), dtype=torch.bfloat16, device=dev)
    for i in range(0, n_local, 1 << 20):
        j = min(n_local, i + (1 << 20))
        table[i:j] = (torch.randn((j - i, d), generator=g, device=dev) * d ** -0.5).to(torch.bfloat16)
    gu = torch.Generator(device=dev).manual_seed(7)
    users = [torch.randn((U, d), generator=gu, device=dev).to(torch.bfloat16) for _ in range(2)]
    hist = torch.randint(1, I_total + 1, (U, 20), generator=gu, device=dev, dtype=torch.int32)
    tgt = torch.randint(1, I_total + 1, (U,), generator=gu, device=dev, dtype=torch.int32)

    def block(u):
        sc, ids = ops.score_topk(u, table, id_base=lo, history=hist, k=10)
        if world > 1:
            lsc, lid, _, _ = ops.topk_merge(sc, ids)
            gsc = torch.empty((world,) + tuple(lsc.shape), dtype=lsc.dtype, device=dev)
            gid = torch.empty((world,) + tuple(lid.shape), dtype=lid.dtype, device=dev)
            dist.all_gather_into_tensor(gsc, lsc)
            dist.all_gather_into_tensor(gid, lid)
            sc, ids = gsc, gid
        return ops.topk_merge(sc.contiguous(), ids.contiguous(), target=tgt)

    for i in range(warmup):
        block(users[i % 2])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        res = block(users[i % 2])
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t) / steps
    flops = 2.0 * U * (I_total + 1) * d
    out["c5_score_topk"] = {"users_per_s": U / (ms / 1e3), "ms_per_block": ms, "users_per_block": U, "items": I_total,
                            "d": d, "tflops_per_gpu": flops / world / (ms / 1e3) / 1e12,
                            "note": "synthetic user vectors; score GEMM + history mask + top-10 + merge%s; table larger "
                                    "than L2" % (" + all-gather" if world > 1 else "")}
    # ---- the lists are checked, not just timed: for 24 users of the last block the kernel's partial top-10 over THIS rank's
    # shard must be a valid top-10 of torch's fp32 scores (scores equal to 2e-3, nothing outside the list beating its minimum)
    sc, ids = ops.score_topk(users[0], table, id_base=lo, history=hist, k=10)
    lsc, lid, _, _ = ops.topk_merge(sc, ids)
    sample = torch.arange(0, U, U // 24, device=dev)[:24]
    ref = torch.empty((sample.numel(), n_local), dtype=torch.float32, device=dev)
    for i in range(0, n_local, 1 << 20):
        j = min(n_local, i + (1 << 20))
        ref[:, i:j] = users[0][sample].float() @ table[i:j].float().t()
    gid = torch.arange(lo, lo + n_local, device=dev)
    dead = (gid[None, None, :] == hist[sample].long()[:, :, None]).any(1) | (gid == 0)[None, :]
    ref.masked_fill_(dead, -float("inf"))
    got_sc = torch.gather(ref, 1, (lid[sample].long() - lo).clamp_(0, n_local - 1))
    best10 = torch.topk(ref, 10, dim=1).values
    ok = bool(((got_sc - lsc[sample]).abs() <= 2e-3).all()) and bool((best10[:, -1] <= lsc[sample][:, -1] + 2e-3).all())
    if not ok:
        raise RuntimeError("C5: a4r_score_topk's lists disagree with torch's scores on the sampled users")
    out["c5_score_topk"]["checked"] = "24 users of a block: list scores == torch fp32 scores (2e-3), no outside item beats the list"
    del ref, dead
    # ---- the REAL job once: 1,000,000 users in blocks of 9,472 against the 10 M-item table (every block: score + mask + top-10
    # + merge [+ all-gather]); user vectors synthetic, wall-clock and device time both reported
    n_blocks = (1_000_000 + U - 1) // U
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = time.time()
    e0.record()
    for i in range(n_blocks):
        res = block(users[i % 2])
    e1.record()
    torch.cuda.synchronize()
    wall = time.time() - w0
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out["c5_full_run"] = {"users": n_blocks * U, "items": I_total, "d": d, "blocks": n_blocks, "device_s": float(t) / 1e3, "wall_s": wall,
                          "users_per_s": n_blocks * U / (float(t) / 1e3), "shards": world,
                          "note": "BASELINE.json configs[4] end to end on %d GPU(s): %d blocks of %d users" % (world, n_blocks, U)}
    del table, users
    torch.cuda.empty_cache()
    return out


def bench_eval_full(model, args, dev, world, rank, steps):
    """The COMPLETE evaluator (eval_arrays: K10 item-ID gather -> SASRec user encoder -> K11/K12 score+mask+top-k ->
    K13 merge + HR/NDCG [+ all-gather]) at the model's real embedding width (D = 64), 1 M synthetic items sharded by id,
    blocks of 8,192 users with 20-item histories."""
    import torch
    import torch.distributed as dist
    from adapter4rec_b200.data_utils.metrics import ItemTable, eval_arrays, shard_range
    # blocks of 8,192 users per GPU: the per-block costs (user-encoder launches, three collectives) are latency, so the block
    # grows with the number of ranks that share the items
    blk = 8192 * world
    I, U = 1_000_000, blk * max(2, steps)
    lo, hi = shard_range(I + 1, rank, world)
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    table = ItemTable((torch.randn((hi - lo, D), generator=g, device=dev) * 0.3).to(torch.bfloat16), lo, I + 1, rank, world)
    gu = torch.Generator().manual_seed(11)
    tok = torch.randint(1, I + 1, (U, S), generator=gu)
    mask = torch.ones((U, S))
    tgt = torch.randint(1, I + 1, (U,), generator=gu).int()
    hist = tok.int()
    tok, mask, tgt, hist = [t.pin_memory() for t in (tok, mask, tgt, hist)]
    eval_arrays(model, tok[:blk], mask[:blk], tgt[:blk], hist[:blk], table, blk)       # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    hit, ndcg, _ = eval_arrays(model, tok, mask, tgt, hist, table, blk)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    return {"users_per_s": U / (ms / 1e3), "users": U, "items": I, "d": D, "ms_total": ms, "hr10": float(hit.mean()),
            "ndcg10": float(ndcg.mean()),
            "note": "complete evaluator incl. host->device copy of the per-user arrays; random embeddings => chance-level HR"}


def bench_item_table(model, args, catalogue, dev, world, rank):
    """get_item_embeddings (data_utils/metrics.py:62-79): the item encoder over the whole 80,001-row catalogue under
    no_grad, item ids sharded over the ranks, the table stays on the device (timed separately from the ranking, SURVEY §8d)."""
    import torch
    import torch.distributed as dist
    from adapter4rec_b200.data_utils.metrics import get_item_embeddings
    out = {}
    bert = model.bert_encoder.text_encoders.title.bert_model
    for name, unpad in (("padded", False), ("unpadded_tokens", True)):
        bert.unpad = unpad
        get_item_embeddings(model, catalogue[:8192], 4096, args, True, dev)          # warm-up
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        table = get_item_embeddings(model, catalogue, 4096, args, True, dev)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = {"items_per_s": catalogue.shape[0] / (float(t) / 1e3), "ms_total": float(t)}
    bert.unpad = False
    out["items"] = int(catalogue.shape[0])
    out["note"] = "BERT-base forward over every catalogue row (30 token slots), host rows copied per 4,096-item block"
    return out


_REAL_STDOUT = None


def dump_outputs(path, loss, trainer):
    """What the last timed step computed, as a caller of trainer.train_step receives it: the loss it returns, and the
    parameters and gradients it leaves in the trainer's flat buffers (317,696 fp32 values each for C2, parameter order of
    trainer.names).  Inputs, initial weights and dropout seeds are fixed, so two builds can be compared array for array."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in (("loss", loss.detach().double().reshape(1)), ("params", trainer.flat_param),
                    ("grads", trainer.flat_grad)):
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def _time_steps(trainer, batches, steps, warmup, dev, world):
    """max-over-ranks device time per step of `trainer.train_step` over rotating resident batches"""
    import torch
    import torch.distributed as dist
    for i in range(warmup):
        trainer.train_step(*batches[i % len(batches)])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loss = trainer.train_step(*batches[i % len(batches)])
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t) / steps, float(loss)


def bench_graphed(trainer, a, host, resident, dev, world):
    """SURVEY.md 8e / 8f-2: zero_grad + every pass of forward / backward + Adam recorded ONCE in a CUDA graph (the all-reduce
    stays an eager NCCL call between two graphs when world > 1) and replayed per step — same kernels, same arithmetic
    (tests/test_graph_step_gpu.py: bit-identical to the eager step), one cudaGraphLaunch instead of ~1,800 launches.
    Timed like the headline: resident batches, then end to end with the pinned-host batch copy and the loss read-back."""
    import torch
    import torch.distributed as dist
    n_pool = len(resident)
    torch.cuda.empty_cache()            # the recording allocates one step's activations in its own pool
    from adapter4rec_b200 import lib
    lib_launches0 = lib.launch_count()
    for i in range(2):                  # call 1 records (the trainer has run eager steps already), call 2 replays
        trainer.train_step_graphed(*resident[i % n_pool])
    recorded_launches = lib.launch_count() - lib_launches0
    torch.cuda.synchronize()

    def timed(fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.steps):
            out = fn(i)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t) / a.steps, out

    gms, gloss = timed(lambda i: trainer.train_step_graphed(*resident[i % n_pool]))

    def e2e_step(i):
        x, m = host[i % n_pool]
        return trainer.train_step_graphed(x.to(dev, non_blocking=True), m.to(dev, non_blocking=True)).item()

    ems, eloss = timed(e2e_step)
    mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    trainer.release_graph()
    torch.cuda.empty_cache()
    return {"value": a.users * world / (gms / 1e3), "unit": UNIT, "ms_per_step": gms,
            "e2e": {"value": a.users * world / (ems / 1e3), "ms_per_step": ems},
            "kernels_in_the_recording": recorded_launches, "graph_launches_per_step": 1 if world <= 1 else 2,
            "loss_after_these_steps": float(gloss), "max_mem_gb": mem,
            "note": "trainer.train_step_graphed: the headline step (same batches, dropout on, fresh masks per replay through the "
                    "indirect seed) replayed from one recording; training simply continues; NOT the headline value"}


def bench_c1_houlsby(dev, world, rank, steps, users=256):
    """BASELINE.json configs[0] ("C1") on the GPU: SASRec + BERT-base with serial Houlsby adapters (r = 64 in BERT, 16 in
    SASRec: parameters.py:55,62), S=20, 30 tokens — the configuration that runs the fused adapter block (K5) 24 times per
    forward.  Same synthetic catalogue shapes as the headline; non-headline figure."""
    import torch
    from adapter4rec_b200 import surgery
    from adapter4rec_b200.model import BertModel, Model, TextConfigLite
    from adapter4rec_b200.trainer import FlatAdamTrainer
    args = make_args(r=64)
    args.adapter_type, args.adapter_down_size = "houslby", 16
    torch.manual_seed(123456)
    model = Model(args, ITEMS, True, BertModel(TextConfigLite())).to(dev)
    surgery.freeze_all(model)
    surgery.insert_adapters(model, args)
    model.train()
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_bert_lr, args.adapter_sasrec_lr,
                              users_per_pass=min(users, 128))
    gen = torch.Generator().manual_seed(4242 + rank)
    cat = synth_catalogue(gen)
    batches = [tuple(t.to(dev) for t in synth_batch(cat, users, gen)) for _ in range(2)]
    ms, loss = _time_steps(trainer, batches, steps, 2, dev, world)
    tokens = users * 42 * L
    flops = 2 * 12 * (14155776 + 92160 + 393216) * tokens      # SURVEY.md §8d, C1: forward + data-gradient backward
    return {"value": users * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "users_per_gpu_per_step": users,
            "users_per_pass": min(users, 128), "model_tflops_per_gpu": flops / (ms / 1e3) / 1e12,
            "trainable_params": trainer.num_trainable, "loss": loss,
            "note": "C1 shapes (Houlsby r=64, S=20, 30 tokens) at %d users per GPU per step, dropout on; NOT the headline value" % users}


def bench_c4_roberta_prompt_cpc(dev, world, rank, steps, users=256):
    """BASELINE.json configs[3] ("C4") as a throughput leg: ModelCPC (the last position predicts the target,
    Downstream/Text/model/model.py:73-135) over RoBERTa-base (vocabulary 50,265, position ids from the padding index 1) with a
    SoftEmbedding prefix of 10 learned tokens (model.py:586-630; run.py:429-434) — the configuration whose PARITY is pinned at
    full size in tests/test_fullsize_gpu.py.  Synthetic Adressa-shape titles: 30 token slots, S = 20.  Non-headline figure."""
    import torch
    from adapter4rec_b200 import surgery
    from adapter4rec_b200.model import ModelCPC, RobertaModel, TextConfigLite
    from adapter4rec_b200.trainer import FlatAdamTrainer
    args = make_args()
    args.adapter_type, args.n_tokens, args.bert_model_load = "prompt", 10, "roberta-base"
    torch.manual_seed(123456)
    cfg = TextConfigLite(vocab_size=50265, max_position_embeddings=514, type_vocab_size=1, pad_token_id=1, layer_norm_eps=1e-5)
    model = ModelCPC(args, ITEMS, True, RobertaModel(cfg)).to(dev)
    surgery.freeze_all(model)
    model = surgery.insert_adapters(model, args)
    model.train()
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_bert_lr, args.adapter_sasrec_lr,
                              users_per_pass=min(users, 128))
    gen = torch.Generator().manual_seed(777 + rank)
    cat = synth_catalogue(gen)
    ids, mask = cat[:, :L].clone(), cat[:, L:]
    ids[:, 0] = torch.where(mask[:, 0] > 0, torch.zeros_like(ids[:, 0]), ids[:, 0])        # <s> = 0
    ids = torch.where(mask > 0, torch.where(ids == 102, torch.full_like(ids, 2), ids), torch.ones_like(ids))   # </s> = 2, <pad> = 1
    cat = torch.cat([ids, mask], 1)
    batches = [tuple(t.to(dev) for t in synth_batch(cat, users, gen)) for _ in range(2)]
    ms, loss = _time_steps(trainer, batches, steps, 2, dev, world)
    return {"value": users * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "users_per_gpu_per_step": users,
            "users_per_pass": min(users, 128), "trainable_params": trainer.num_trainable, "loss": loss,
            "token_slots_per_item": L + args.n_tokens,
            "note": "C4 shapes (CPC + RoBERTa-base + 10 soft-prompt tokens, S=20, 30 + 10 token slots per item) at %d users per GPU "
                    "per step, dropout on; the frozen backbone still needs its data gradients down to the prompt; NOT the headline "
                    "value" % users}


def bench_c3_vit(dev, world, rank, steps, users=64):
    """BASELINE.json configs[2] ("C3"): SASRec + ViT-B/16-224 with Houlsby adapters (r = 64), S=10 => 22 images per user,
    synthetic images in (-1, 1) (the post-Normalize(0.5, 0.5) range), bf16.  Non-headline figure."""
    import types
    import torch
    from adapter4rec_b200 import surgery
    from adapter4rec_b200.cv import Model as CVModel, ViTConfigLite, ViTForImageClassification
    from adapter4rec_b200.model.layers import Linear
    from adapter4rec_b200.trainer import FlatAdamTrainer
    S3 = 10
    args = types.SimpleNamespace(max_seq_len=S3, l2_weight=0, embedding_dim=D, num_attention_heads=2, drop_rate=0.1,
                                 transformer_block=2, CV_model_load="vit-base-patch16-224", cv_adapter_down_size=64,
                                 adapter_down_size=16, adapter_dropout_rate=0.1, adapter_activation="RELU", n_tokens=10,
                                 adapter_type="houslby", adding_adapter_to="all", is_serial="True", finetune_layernorm="None")
    torch.manual_seed(12345)
    net = ViTForImageClassification(ViTConfigLite())
    net.classifier = Linear(768, D)
    model = CVModel(args, 1000, True, net).to(dev)
    surgery.freeze_all(model)
    surgery.insert_adapters_cv(model, args)
    model.train()
    trainer = FlatAdamTrainer(model, 1e-4, 1e-5, 5e-4, 1e-4, users_per_pass=32)
    n_img = users * (S3 + 1) * 2
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    batches = [(torch.rand((n_img, 3, 224, 224), generator=g, device=dev) * 2 - 1, torch.ones((users, S3), device=dev))
               for _ in range(2)]
    ms, loss = _time_steps(trainer, batches, steps, 2, dev, world)
    fwd_flops_img = 12 * 197 * (14155776 + 4 * 197 * 768 + 393216) + 196 * 2 * 768 * 768
    return {"value": users * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "users_per_gpu_per_step": users,
            "images_per_gpu_per_step": n_img, "users_per_pass": 32,
            "model_tflops_per_gpu": 2 * fwd_flops_img * n_img / (ms / 1e3) / 1e12,
            "trainable_params": trainer.num_trainable, "loss": loss,
            "note": "C3 shapes (ViT-B/16-224 Houlsby r=64, 197 tokens per image, 22 images per user), images resident in HBM; "
                    "NOT the headline value"}


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line to stdout when
    NCCL_DEBUG is set in the environment), so file descriptor 1 is pointed at stderr for the duration of the run and the
    JSON line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    a = parse()
    _claim_stdout()
    if a.impl == "reference":
        return run_reference(a)
    import torch
    import torch.distributed as dist
    from adapter4rec_b200 import lib, ops, surgery
    from adapter4rec_b200.model import BertModel, Model, TextConfigLite
    from adapter4rec_b200.trainer import FlatAdamTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib.get_lib()   # fail loudly if the CUDA library is missing

    torch.manual_seed(123456)
    args = make_args()
    model = Model(args, ITEMS, True, BertModel(TextConfigLite())).to(dev)
    surgery.freeze_all(model)
    surgery.insert_adapters(model, args)
    model.train()
    trainer = FlatAdamTrainer(model, args.lr, args.fine_tune_lr, args.adapter_bert_lr, args.adapter_sasrec_lr,
                              users_per_pass=a.users_per_pass)

    gen = torch.Generator().manual_seed(123456 + rank)
    cat = synth_catalogue(gen)
    n_pool = 3
    host = [synth_batch(cat, a.users, gen) for _ in range(n_pool)]
    host = [(x.pin_memory(), m.pin_memory()) for x, m in host]
    resident = [(x.to(dev), m.to(dev)) for x, m in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- kernel-resident timing: inputs already in HBM ----------------
    for i in range(a.warmup):
        trainer.train_step(*resident[i % n_pool])
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    ops.gemm_profile_start()
    launches0 = lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(a.steps):
        loss = trainer.train_step(*resident[i % n_pool])
    ev1.record()
    barrier()
    launches = lib.launch_count() - launches0
    max_mem_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    gemm_flops, gemm_ms, gemm_calls, gemm_groups = ops.gemm_profile_stop(by_shape=True)
    clk = clocks.stop()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    ms_per_step = ms / a.steps
    value = a.users * world / (ms_per_step / 1e3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, loss, trainer)

    # ---------------- end-to-end: host (pinned) -> device copy of the batch + loss read-back every step ----------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(a.steps):
        x, m = host[i % n_pool]
        xd, md = x.to(dev, non_blocking=True), m.to(dev, non_blocking=True)
        loss_val = trainer.train_step(xd, md).item()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t) / a.steps
    h2d = host[0][0].numel() * 8 + host[0][1].numel() * 4

    # ---------------- variant: unpadded token layout (same batches, same results, fewer executed tokens) ----------------
    # The synthetic items have 8..30 real tokens in 30 slots; HF BERT (the reference) computes the padded slots and then
    # ignores them.  `unpad` runs the encoder on the kept tokens only — bit-identical embeddings and loss
    # (tests/test_model_gpu.py::test_unpadded_token_layout_gives_the_same_step).  Reported NEXT TO the headline, which
    # executes every padded token exactly as the reference does.
    variants = {}

    def want(name):
        return not a.no_variants and (a.variants == "all" or name in a.variants.split(","))

    if want("layouts"):
        bert = model.bert_encoder.text_encoders.title.bert_model
        bert.unpad = True
        for i in range(2):
            trainer.train_step(*resident[i % n_pool])
        barrier()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        for i in range(a.steps):
            vloss = trainer.train_step(*resident[i % n_pool])
        v1.record()
        barrier()
        t = torch.tensor([v0.elapsed_time(v1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vms = float(t) / a.steps
        kept = sum(int((x[:, L:] != 0).sum()) for x, _ in resident) / n_pool
        variants["unpadded_tokens"] = {
            "value": a.users * world / (vms / 1e3), "unit": UNIT, "ms_per_step": vms,
            "tokens_executed_per_gpu_per_step": kept, "tokens_padded_per_gpu_per_step": a.users * 42 * L,
            "loss_after_these_steps": float(vloss),
            "note": "same batches and per-step results as the headline (training simply continues); only kept tokens are executed "
                                          "(PackedTokens: cu_seqlens attention, [CLS] gather); NOT the headline value"}
        bert.unpad = False
        # ---------------- variant: each distinct item of a pass is encoded once (Model.dedup_items) ----------------
        model.dedup_items = True
        dms, dloss = _time_steps(trainer, resident, a.steps, 2, dev, world)
        uniq = sum(int(torch.unique(x.view(-1, 2 * L), dim=0).shape[0]) for x, _ in resident) / n_pool
        variants["dedup_items"] = {
            "value": a.users * world / (dms / 1e3), "unit": UNIT, "ms_per_step": dms,
            "distinct_item_rows_per_batch": uniq, "item_rows_per_batch": a.users * 42,
            "note": "an item occurring several times in a pass (uniform synthetic sampling over 80 k items: ~10 % of the slots; real "
                    "logs repeat popular items far more) is encoded once and its gradient rows are summed; identical forward "
                    "values, occurrences share one dropout mask; NOT the headline value (the reference encodes every slot)"}
        bert.unpad = True
        cms, closs = _time_steps(trainer, resident, a.steps, 2, dev, world)
        variants["unpadded_dedup"] = {"value": a.users * world / (cms / 1e3), "unit": UNIT, "ms_per_step": cms,
                                      "note": "both of the above together; NOT the headline value"}
        bert.unpad = False
        model.dedup_items = False

    # ---------------- variant: the same step replayed from a CUDA graph (trainer.train_step_graphed) ----------------
    # (default run: one GPU only — a rank-local failure while recording would leave the other ranks inside a collective;
    # `--variants graphed_step` runs it at any N: profiles/r02_bench_graphed_step_n2.json)
    if want("graphed_step") and (world == 1 or a.variants != "all"):
        try:
            variants["graphed_step"] = bench_graphed(trainer, a, host, resident, dev, world)
        except Exception as exc:  # noqa: BLE001 — a failed recording must not take the headline line with it
            variants["graphed_step"] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:300])}
            trainer.release_graph()

    # ---------------- second half of the metric: full-ranking eval users/s ----------------
    del trainer, resident
    model.zero_grad(set_to_none=True)
    torch.cuda.empty_cache()
    eval_out = None
    if not a.no_eval:
        eval_out = bench_eval(dev, world, rank, max(2, a.steps), 2)
        model.eval()
        eval_out["eval_model_d64"] = bench_eval_full(model, args, dev, world, rank, a.steps)
        eval_out["item_table_build"] = bench_item_table(model, args, cat, dev, world, rank)
    # ---------------- the other two training configurations of BASELINE.json (non-headline) ----------------
    if want("c1"):
        torch.cuda.empty_cache()
        variants["c1_bert_houlsby"] = bench_c1_houlsby(dev, world, rank, max(2, min(a.steps, 3)))
    if want("c3"):
        torch.cuda.empty_cache()
        variants["c3_vit_houlsby"] = bench_c3_vit(dev, world, rank, max(2, min(a.steps, 3)))
    if want("c4"):
        torch.cuda.empty_cache()
        variants["c4_roberta_prompt_cpc"] = bench_c4_roberta_prompt_cpc(dev, world, rank, max(2, min(a.steps, 3)))
    torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk, pk_kind = peaks()
    tokens = a.users * 42 * L
    algo_flops_step = 2 * FLOP_FWD_PER_TOKEN * tokens            # forward + data-gradient backward (frozen backbone)
    achieved_all = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
    # the dominant kernel = gemm_tn_kernel over ALL its launches of the timed region (every shape and epilogue: the
    # kernel with the largest share of the step); the per-shape table sits beside it in `by_shape`
    achieved = achieved_all
    epi_names = {0: "linear", 1: "gelu(+pre-activation out)", 2: "relu", 3: "gelu' (dgrad)", 4: "relu' (dgrad)"}
    # DRAM traffic per launch: launch-weighted mean over the shapes of the committed `ncu --set full` captures (profiles/)
    traffic, traffic_note = None, None
    try:
        recs = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_full_gemm_traffic.json")))
        tot_b, tot_a, tot_n = 0.0, 0.0, 0
        for shape, g in gemm_groups.items():
            for rec in recs:
                # captures were taken at a smaller row count; A, C and the streamed epilogue operands are linear in M (the
                # weight operand is L2-resident), so a launch with more rows is scaled by the row ratio
                if tuple(rec["shape"][1:]) == tuple(shape[1:4]):
                    tot_b += rec["dram_bytes_per_launch"] * (shape[0] / float(rec["shape"][0])) * g[2]
                    tot_a += rec["algorithmic_bytes"] * (shape[0] / float(rec["shape"][0])) * g[2]
                    tot_n += g[2]
                    break
        # (the captured shapes are the eight large ones of a pass; the small SASRec-side GEMMs and the two-segment dT GEMM of the
        #  LoRA backward — a quarter of the launches, ~3 % of the GEMM time — have no capture: the mean is over the covered
        #  launches, whose count is reported beside it)
        if tot_n >= 0.7 * gemm_calls:
            traffic = tot_b / tot_n
            traffic_note = {"launches_covered": tot_n, "launches": gemm_calls, "algorithmic_bytes_per_launch": tot_a / tot_n,
                            "ratio": tot_b / tot_a if tot_a else None,
                            "source": "profiles/r02_ncu_full_gemm_traffic.json (ncu --set full, dram__bytes_read + write per shape)"}
    except Exception:
        pass
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "C2: SASRec(D=64,2 blocks)+BERT-base, LoRA r=8 on q/v, S=20, 30 tokens, bf16",
                   "users_per_gpu_per_step": a.users, "sequences_per_gpu_per_step": a.users * 42,
                   "tokens_per_gpu_per_step": tokens, "users_per_pass": a.users_per_pass, "parallelism": "dp%d" % world,
                   "l2": "inputs larger than L2 (>= 1 GB activations per layer per pass); %d rotating batches" % n_pool,
                   "dropout": "on, p=0.1 (BERT hidden + attention-probability, SASRec) as the reference trains: counter-RNG "
                              "kernels, masks regenerated in the backward",
                   "last_layer_tail": "[CLS] rows only (identical results: other rows of the last layer never reach the loss)"},
        "model_tflops_per_gpu": algo_flops_step / (ms_per_step / 1e3) / 1e12,
        "loss": loss_val,
        "gpu_launches": int(launches),
        "max_mem_gb": max_mem_gb,
        "clocks": {"sm_mhz": clk["sm_mhz"], "sm_max_mhz": clk["sm_max_mhz"], "reasons": clk["reasons"]},
        "e2e": {"value": a.users * world / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_detail": traffic_note,
                     "kernel": "gemm_tn_kernel (tcgen05 cta_group::2 + TMA), all %d launches of the timed region (every shape "
                               "and epilogue): %.1f%% of the step; algorithmic FLOPs = sum of 2*M*N*(K+K2) = %.4g per launch "
                               "on average; per-shape figures in by_shape"
                               % (gemm_calls, 100.0 * gemm_ms / ms, gemm_flops / max(1, gemm_calls)),
                     "peak_source": pk_kind + " bf16_tflops_sustained (kernel timed inside a long step)",
                     "all_gemm_launches": {"achieved": achieved_all, "frac": achieved_all / peak if peak else None,
                                           "launches": gemm_calls, "share_of_step": gemm_ms / ms},
                     "by_shape": [{"M": k[0], "N": k[1], "K": k[2], "epilogue": epi_names.get(k[3], "?"), "launches": v[2],
                                   "share_of_step": v[1] / ms, "tflops": v[0] / (v[1] / 1e3) / 1e12,
                                   "frac": v[0] / (v[1] / 1e3) / 1e12 / peak if peak else None}
                                  for k, v in sorted(gemm_groups.items(), key=lambda kv: -kv[1][1])[:12]]},
    }
    if eval_out is not None:
        pk_b = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
        eval_out["c5_score_topk"]["frac_of_peak"] = eval_out["c5_score_topk"]["tflops_per_gpu"] / pk_b
        out["eval"] = eval_out
    if variants:
        out["variants"] = variants
    if not a.no_cpu_baseline and world == 1:
        # rank 0 at N = 1 only (the contract): a bounded sample of the same workload on every host core
        cores = use_all_host_threads()
        a.cpu_users = a.cpu_users or 48
        msd = {k: v for k, v in model.state_dict().items()}
        step = oracle_step_factory(msd, a.cpu_users)
        t0 = time.time()
        step()
        dt = time.time() - t0
        out["cpu_baseline"] = {"value": a.cpu_users / dt, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "1 step over %d users (= %d sequences x %d tokens), fp32 oracle port, %.1f s"
                                         % (a.cpu_users, a.cpu_users * 42, L, dt)}
        if not a.no_eval:
            out["cpu_baseline"]["eval_half"] = cpu_eval_legs(msd, cores)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
