"""Autograd glue: torch.autograd.Function wrappers that call the sm_100a kernels (adapter4rec_b200.ops) for both
directions.  No arithmetic of the path is done by torch here — torch tracks the graph, owns memory and streams.

Backward policy (SURVEY.md §7.3): a frozen weight never gets a weight gradient (only dX = dY·W through a cached bf16
transpose); trainable adapter / LoRA / bias / LayerNorm parameters get theirs from the skinny wgrad, column-sum and
LayerNorm-backward kernels, in fp32."""
import torch

from . import ops

BF16 = torch.bfloat16


PARAM_EPOCH = [0]   # bumped by the trainer after every optimizer step (the Adam kernel writes through raw pointers,
                    # which torch's version counters cannot see)


def bump_param_epoch():
    PARAM_EPOCH[0] += 1


def _param_key(tensors):
    """Staleness key of operands derived from `tensors` (None entries allowed): each tensor's storage and version, and
    the optimizer-step count when any of them trains.  Operands are rebuilt when it changes."""
    return tuple(None if t is None else (t.data_ptr(), t._version, t.device) for t in tensors) + (
        PARAM_EPOCH[0] if any(t is not None and t.requires_grad for t in tensors) else -1,)


class WeightCache:
    """bf16 copies of an fp32 master weight: W [N,K] for the forward GEMM and Wᵀ [K,N] for the data-gradient GEMM.
    Rebuilt when the parameter is modified in place (optimizer step, load_state_dict) or moved."""

    def __init__(self):
        self.key = None
        self.master = None
        self.w = None
        self.wt = None

    def get(self, weight, need_t=False):
        key = _param_key((weight,))
        if key != self.key:
            self.key = key
            self.master = weight.detach()
            if self._fusable(self.master):
                self.w, self.wt = ops.cast_transpose(self.master, True, need_t)   # one pass: bf16 copy (+ transpose)
            else:
                self.w, self.wt = self.master.to(BF16).contiguous(), None
        if need_t and self.wt is None:
            if self._fusable(self.master):
                _, self.wt = ops.cast_transpose(self.master, False, True)
            else:
                self.wt = self.w.t().contiguous()
        return self.w, self.wt

    @staticmethod
    def _fusable(w):
        return w.is_cuda and w.dtype == torch.float32 and w.dim() == 2 and w.stride(1) == 1


def _as2d(x):
    return x.reshape(-1, x.shape[-1])


class LinearFunction(torch.autograd.Function):
    """y = act(x Wᵀ + b) + residual + residual2, act in {none, gelu, relu} fused in the GEMM epilogue;
    {leaky_relu, gelu_new} (bottleneck-only activations of the Pfeiffer / Compacter adapters) run as a stand-alone
    elementwise pass over the r-wide output."""

    @staticmethod
    def forward(ctx, x, weight, bias, residual, residual2, cache, act):
        w, _ = cache.get(weight)
        standalone = act in ("leaky_relu", "gelu_new")
        epi = {None: ops.EPI_LINEAR, "gelu": ops.EPI_GELU, "relu": ops.EPI_RELU}[None if standalone else act]
        b = None if bias is None else bias.detach().float().contiguous()
        need_grad = any(ctx.needs_input_grad[:5])
        aux = None
        if act == "gelu" and need_grad:
            aux = torch.empty((x.shape[0], w.shape[0]), dtype=BF16, device=x.device)
        y = ops.gemm(x, w, bias=b, epilogue=epi, residual=residual, residual2=residual2, aux=aux)
        if standalone:
            aux, y = y, ops.act_fwd(y, act)
        ctx.cache, ctx.act = cache, act
        ctx.has_bias, ctx.has_r1, ctx.has_r2 = bias is not None, residual is not None, residual2 is not None
        save_x = x if ctx.needs_input_grad[1] else None
        act_saved = aux if act in ("gelu", "gelu_new") else (y if act in ("relu", "leaky_relu") else None)
        ctx.save_for_backward(save_x, act_saved, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, act_saved, weight = ctx.saved_tensors
        dy = dy.contiguous()
        if ctx.act is not None:
            dy = ops.act_bwd(dy, act_saved, ctx.act)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            _, wt = ctx.cache.get(weight, need_t=True)
            dx = ops.gemm(dy, wt)
        if ctx.needs_input_grad[1]:
            dw = ops.wgrad(dy, x)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = ops.colsum(dy)
        # the residuals enter after the activation only when act is None (enforced by the callers)
        dr1 = dy if ctx.has_r1 and ctx.needs_input_grad[3] else None
        dr2 = dy if ctx.has_r2 and ctx.needs_input_grad[4] else None
        return dx, dw, db, dr1, dr2, None, None


def linear(x, weight, bias, cache, act=None, residual=None, residual2=None):
    assert act is None or (residual is None and residual2 is None)
    return LinearFunction.apply(x, weight, bias, residual, residual2, cache, act)


def _frozen(dense, intermediate=None):
    """F of a frozen block: ((W, b, cache),) of the dense Linear, or ((Wi, bi, ci), (Wf, bf, cf)) of the GELU FFN pair
    intermediate -> dense.  Frozen weights need no gradient, so they travel in this tuple rather than as node inputs."""
    return tuple((m.weight, m.bias, m._cache) for m in ((dense,) if intermediate is None else (intermediate, dense)))


def _ln_args(ln):
    return (None, None, 0.0) if ln is None else (ln.weight, ln.bias, ln.eps)


def _needs(ctx, names):
    """{argument name: needs a gradient} of a node whose forward takes the arguments `names` in this order"""
    return dict(zip(names, ctx.needs_input_grad))


def _frozen_fwd(x, F, res, rng, need_u):
    """(dropout(F(x)) (+ res), u): dropout (rng = (p, seed, offset) or None) and the residual live in the epilogue of F's
    last GEMM; u is the FFN pair's pre-activation (the GELU′ operand of the backward), kept when need_u, else None."""
    ws = [cache.get(w)[0] for w, _, cache in F]
    u = None
    if len(F) == 2:
        u = torch.empty((x.shape[0], ws[0].shape[0]), dtype=BF16, device=x.device) if need_u else None
        x = ops.gemm(x, ws[0], bias=F[0][1].detach(), epilogue=ops.EPI_GELU, aux=u)
    return ops.gemm(x, ws[-1], bias=F[-1][1].detach(), residual=res, dropout=rng), u


def _frozen_bwd(dh, u, F, fold):
    """dx of _frozen_fwd from dh, the gradient at F's output (already through the dropout).  GELU′ rides in the epilogue
    of the first data-gradient GEMM; fold (the skip gradient when res is x, or None) in that of the last."""
    wts = [cache.get(w, need_t=True)[1] for w, _, cache in F]
    if len(F) == 2:
        dh = ops.gemm(dh, wts[1], epilogue=ops.EPI_DGELU, aux=u)
    return ops.gemm(dh, wts[0], residual=fold)


def _dropout_rng(p, x, F):
    """(p, seed, offset) of the dropout on F's output, or None when p == 0"""
    return (float(p),) + DropoutState.draw((x.shape[0] * F[-1][0].shape[0] + 3) // 4) if p > 0 else None


class FrozenBlockFunction(torch.autograd.Function):
    """A frozen dense layer or FFN pair with its dropout, residual and post-LN LayerNorm in a single autograd node:

        out = tail(dropout(F(x)) + res)       F(x) = x Woᵀ + bo                  (attention.output: BertSelfOutput)
                                             F(x) = GELU(x Wiᵀ + bi) Wfᵀ + bf   (intermediate + output: BertOutput, ViTOutput)

    tail = LayerNorm (gamma given; gamma / beta may be trainable: finetune_layernorm) or nothing (then p must be 0).
    res = None, x itself (its gradient rides in the epilogue of the last data-gradient GEMM) or another tensor.
    Forward: dropout and the residual add live in the epilogue of the last GEMM (counter RNG).  Backward: LayerNorm's
    backward kernel emits dz AND dz ⊙ mask/(1-p) (the gradient through the dropout) in one pass; GELU′ and the skip
    gradient live in the epilogues of the data-gradient GEMMs."""

    ARGS = ("x", "res", "gamma", "beta", "eps", "p", "F")

    @staticmethod
    def forward(ctx, x, res, gamma, beta, eps, p, F):
        assert gamma is not None or p == 0, "dropout without the LayerNorm tail is not fused"
        need = any(_needs(ctx, FrozenBlockFunction.ARGS).values())
        rng = _dropout_rng(p, x, F)
        out, u = _frozen_fwd(x, F, res, rng, need)
        ctx.rng, ctx.F, ctx.fold, ctx.ln = rng, F, res is x, gamma is not None
        z = mean = rstd = g = None
        if ctx.ln:
            z, g, b = out, gamma.detach().float().contiguous(), beta.detach().float().contiguous()
            out, _, mean, rstd = ops.layernorm_fwd(z, g, b, eps, want_stats=need)
        ctx.save_for_backward(z, mean, rstd, g, u)
        return out

    @staticmethod
    def backward(ctx, dout):
        z, mean, rstd, g, u = ctx.saved_tensors
        need = _needs(ctx, FrozenBlockFunction.ARGS)
        grads = {}
        dout = dz = dzm = dout.contiguous()
        if ctx.ln:
            if need["gamma"] or need["beta"]:
                grads["gamma"], grads["beta"] = torch.empty_like(g), torch.empty_like(g)
            r = ops.layernorm_bwd(dout, z, mean, rstd, g, dgamma=grads.get("gamma"), dbeta=grads.get("beta"), masked=ctx.rng)
            dz, dzm = r if ctx.rng is not None else (r, r)
        if need["x"]:
            grads["x"] = _frozen_bwd(dzm, u, ctx.F, dz if ctx.fold else None)
        if need["res"] and not ctx.fold:
            grads["res"] = dz
        return tuple(grads.get(n) for n in FrozenBlockFunction.ARGS)


def frozen_block(x, res, dense, intermediate=None, ln=None, p=0.0):
    """tail(dropout(F(x)) + res) as one node (FrozenBlockFunction).  dense / intermediate: the block's frozen Linear
    modules (intermediate None: F is dense alone); ln: its LayerNorm module, or None for no tail (p must then be 0)."""
    return FrozenBlockFunction.apply(x, res, *_ln_args(ln), p, _frozen(dense, intermediate))


class LayerNormFunction(torch.autograd.Function):
    """y = LN(x + res[row % res_rows]).  res is the bf16 copy of a broadcast table (the SASRec position table) or None;
    `res_param` is its fp32 master when that table is trainable (full fine-tuning): its gradient is the column sum of dz
    over the broadcast axis."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, res, res_param=None):
        need = any(ctx.needs_input_grad[:3]) or (res_param is not None and res_param.requires_grad)
        g, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        if res is not None:
            y, z, mean, rstd = ops.layernorm_fwd(x, g, b, eps, res=res, want_z=need, want_stats=need)
        else:
            y, _, mean, rstd = ops.layernorm_fwd(x, g, b, eps, want_stats=need)
            z = x
        ctx.res_rows = 0 if res is None else res.numel() // res.shape[-1]
        ctx.res_shape = None if res_param is None else tuple(res_param.shape)
        if need:
            ctx.save_for_backward(z, mean, rstd, g)
        return y

    @staticmethod
    def backward(ctx, dy):
        z, mean, rstd, g = ctx.saved_tensors
        dy = dy.contiguous()
        dg = db = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dg, db = torch.empty_like(g), torch.empty_like(g)
        dz = ops.layernorm_bwd(dy, z, mean, rstd, g, dgamma=dg, dbeta=db)
        dres = None
        if ctx.res_shape is not None and ctx.needs_input_grad[5]:
            rows, H = ctx.res_rows, dz.shape[1]
            dres = torch.zeros(ctx.res_shape, dtype=torch.float32, device=dz.device)
            dres[:rows] = ops.colsum(dz.view(-1, rows * H)).view(rows, H)
        return dz, dg, db, None, None, dres


def layer_norm(x, weight, bias, eps, res=None, res_param=None):
    return LayerNormFunction.apply(x, weight, bias, eps, res, res_param)


class LayerNormSkipFunction(torch.autograd.Function):
    """(LN(x), x): a pre-LN block x1 = x + f(LN(x)) takes its skip connection from the SECOND output, so the skip gradient
    is delivered to this node and added inside the LayerNorm-backward kernel (a4r_layernorm_bwd_add) instead of by a
    separate autograd accumulation pass over [M, H].  Same trick as QKVFunction's skip output on the post-LN side."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps):
        need = any(ctx.needs_input_grad[:3])
        g, b = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        y, _, mean, rstd = ops.layernorm_fwd(x, g, b, eps, want_stats=need)
        if need:
            ctx.save_for_backward(x, mean, rstd, g)
        return y, x          # autograd treats a returned input as x.view_as(x)

    @staticmethod
    def backward(ctx, dy, dskip):
        x, mean, rstd, g = ctx.saved_tensors
        want_ln = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        if dy is None:                                   # only the skip output was used downstream
            return dskip, None, None, None
        dy = dy.contiguous()
        if dskip is not None and not want_ln:
            return ops.layernorm_bwd_add(dy, x, mean, rstd, g, dskip.contiguous()), None, None, None
        dg = db = None
        if want_ln:
            dg, db = torch.empty_like(g), torch.empty_like(g)
        dx = ops.layernorm_bwd(dy, x, mean, rstd, g, dgamma=dg, dbeta=db)
        if dskip is not None:
            dx = dx + dskip
        return dx, dg, db, None


def layer_norm_skip(x, weight, bias, eps):
    return LayerNormSkipFunction.apply(x, weight, bias, eps)


class DropoutState:
    """Seed and running counter of the counter-based dropout RNG (a4r_dropout / attention-probability dropout).  Every
    call site draws a fresh counter range, so masks are independent across sites and steps; the backward of a site reuses
    the (seed, offset) its forward drew."""
    seed = 0x5EEDA4D2
    counter = 0
    seed_address = None      # set while a step is being recorded in a CUDA graph: device address of the seed of each replay
    SEED_INDIRECT = 1 << 63  # A4R_SEED_INDIRECT (include/adapter4rec.h)

    @classmethod
    def manual_seed(cls, seed):
        cls.seed, cls.counter = int(seed) & 0xFFFFFFFFFFFF, 0

    @classmethod
    def draw(cls, n_counters):
        off = cls.counter
        cls.counter += int(n_counters)
        if cls.seed_address is not None:
            return cls.SEED_INDIRECT | int(cls.seed_address), off
        return cls.seed, off

    @classmethod
    def replay_seed(cls, step, base=None):
        """seed of replay number `step` of a recorded step: the counter offsets are baked into the graph, so successive replays
        differ by their seed (splitmix64 of the base seed and the step number: unrelated streams, below bit 63)"""
        z = ((cls.seed if base is None else int(base)) + 0x9E3779B97F4A7C15 * (int(step) + 1)) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        return (z ^ (z >> 31)) & 0x7FFFFFFFFFFFFFFF


class DropoutAddFunction(torch.autograd.Function):
    """out = dropout(x) + res   (nn.Dropout followed by the residual add of the reference's post-LN blocks)."""

    @staticmethod
    def forward(ctx, x, res, p):
        ctx.p = p
        ctx.rng = DropoutState.draw((x.numel() + 3) // 4)
        ctx.has_res = res is not None
        return ops.dropout(x.contiguous(), None if res is None else res.contiguous(), p, *ctx.rng)

    @staticmethod
    def backward(ctx, dy):
        dy = dy.contiguous()
        dx = ops.dropout(dy, None, ctx.p, *ctx.rng) if ctx.needs_input_grad[0] else None
        return dx, (dy if ctx.has_res and ctx.needs_input_grad[1] else None), None


def dropout_add(x, res, p):
    """dropout(x) (+ res); identity (+ plain add through the caller's fused path) when p == 0"""
    return DropoutAddFunction.apply(x, res, float(p))


class AddFunction(torch.autograd.Function):
    """out = x + res in bf16 (the p = 0 case of a4r_dropout: every element kept, scale 1)."""

    @staticmethod
    def forward(ctx, x, res):
        return ops.dropout(x.contiguous(), res.contiguous(), 0.0, 0, 0)

    @staticmethod
    def backward(ctx, dy):
        return (dy if ctx.needs_input_grad[0] else None), (dy if ctx.needs_input_grad[1] else None)


def add(x, res):
    return AddFunction.apply(x, res)


class AttentionFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, mask, N, L, heads, head_dim, causal, mask_neg, dropout_p=0.0, scale=None, cu_seqlens=None):
        ctx.cfg = (N, L, heads, head_dim, causal, mask_neg, scale)
        ctx.cu = cu_seqlens
        ctx.mask = mask
        ctx.drop = None
        if dropout_p > 0.0:
            ctx.drop = (dropout_p,) + DropoutState.draw(N * heads * 32 * 8)
        out, lse = ops.attn_small_fwd(qkv, N, L, heads, head_dim, mask=mask, causal=causal, mask_neg=mask_neg, want_lse=True,
                                      dropout=ctx.drop, scale=scale, cu_seqlens=cu_seqlens)
        # the short-sequence kernel recomputes everything from qkv; the mid-length (ViT) kernel reuses lse and the output
        ctx.save_for_backward(qkv, lse, out if lse is not None else None)
        return out

    @staticmethod
    def backward(ctx, dctx):
        qkv, lse, out = ctx.saved_tensors
        N, L, heads, head_dim, causal, mask_neg, scale = ctx.cfg
        dqkv = ops.attn_small_bwd(qkv, dctx.contiguous(), N, L, heads, head_dim, mask=ctx.mask, causal=causal,
                                  mask_neg=mask_neg, lse=lse, ctx=out, dropout=ctx.drop, scale=scale, cu_seqlens=ctx.cu)
        return dqkv, None, None, None, None, None, None, None, None, None, None


def attention(qkv, mask, N, L, heads, head_dim, causal=False, mask_neg=ops.F32_MIN, dropout_p=0.0, scale=None,
              cu_seqlens=None):
    """scale: softmax temperature override (default head_dim ** -0.5); used when narrow heads are zero-padded to a
    kernel-supported width.  cu_seqlens: packed variable-length token layout (short-sequence kernel)."""
    return AttentionFunction.apply(qkv, mask, N, L, heads, head_dim, causal, mask_neg, float(dropout_p), scale, cu_seqlens)


class GatherRowsFunction(torch.autograd.Function):
    """out[i] = x[idx[i]] for UNIQUE row indices (the [CLS] rows of a packed token matrix, or the valid tokens of a padded
    one).  Backward = the inverse placement into zeros: pure data movement."""

    @staticmethod
    def forward(ctx, x, idx):
        ctx.rows = x.shape[0]
        ctx.save_for_backward(idx)
        return ops.gather_rows(x.contiguous(), idx)

    @staticmethod
    def backward(ctx, dy):
        (idx,) = ctx.saved_tensors
        dx = torch.zeros((ctx.rows, dy.shape[1]), dtype=dy.dtype, device=dy.device)
        dx.index_copy_(0, idx, dy.contiguous())
        return dx, None


def gather_rows(x, idx):
    return GatherRowsFunction.apply(x, idx)


class ExpandRowsFunction(torch.autograd.Function):
    """out[i] = x[inverse[i]] where several i may share a row (the item embeddings of a batch in which an item occurs more
    than once: it is encoded ONCE).  Backward = the sum of the gradient rows of every occurrence, formed deterministically:
    the gradient rows are brought into group order (stable sort of `inverse`) and each group is summed sequentially
    (segment reduction over `counts`) — no atomics, no host synchronisation."""

    @staticmethod
    def forward(ctx, x, inverse, counts):
        ctx.save_for_backward(inverse, counts)
        return ops.gather_rows(x.contiguous(), inverse)

    @staticmethod
    def backward(ctx, dy):
        inverse, counts = ctx.saved_tensors
        order = torch.argsort(inverse, stable=True)
        grouped = dy.contiguous()[order].float()
        return torch.segment_reduce(grouped, "sum", lengths=counts, axis=0).to(dy.dtype), None, None


def expand_rows(x, inverse, counts):
    return ExpandRowsFunction.apply(x, inverse, counts)


_ROW_HASH = {}


def unique_rows(rows):
    """(unique rows [U, W], inverse [N], counts [U]) of an int64 matrix.  torch.unique(dim=0) sorts rows lexicographically
    (tens of milliseconds for a 10 k x 60 batch); here rows are compared through a 64-bit multiplicative hash (1-D radix
    sort) and the result is VERIFIED against the rows — on a hash collision the exact routine runs instead."""
    N, W = rows.shape
    key = (rows.device, W)
    if key not in _ROW_HASH:
        g = torch.Generator().manual_seed(0x5EED)
        _ROW_HASH[key] = (torch.randint(-2 ** 62, 2 ** 62, (W,), generator=g, dtype=torch.int64) | 1).to(rows.device)
    h = (rows * _ROW_HASH[key]).sum(1)                      # int64 arithmetic wraps: a hash, not a value
    uh, inverse, counts = torch.unique(h, return_inverse=True, return_counts=True)
    first = torch.full((uh.numel(),), N, dtype=torch.int64, device=rows.device)
    first.scatter_reduce_(0, inverse, torch.arange(N, device=rows.device), reduce="amin")
    uniq = rows[first]
    if not bool((uniq[inverse] == rows).all()):             # two different rows with one hash: vanishingly rare
        uniq, inverse, counts = torch.unique(rows, dim=0, return_inverse=True, return_counts=True)
    return uniq, inverse, counts


LORA_PAD = 64  # the rank-r intermediates of all LoRA'd projections of one fused QKV share one 64-column k-block


def _lora_slots(P):
    """(slots, ones) of P = [(W, b, lora_A, lora_B) per projection]: slot (j, off, r) holds projection j's rank-r
    intermediate in columns [off, off + r) of T; ones: the ranks leave column 63 of T free for a ones column"""
    slots, off = [], 0
    for j, (_, _, A, _) in enumerate(P):
        if A is not None:
            slots.append((j, off, A.shape[0]))
            off += A.shape[0]
    assert off <= LORA_PAD, "the LoRA ranks %s of one fused projection sum to %d, more than %d" % (
        [r for _, _, r in slots], off, LORA_PAD)
    return tuple(slots), bool(slots) and off < LORA_PAD


class QKVCache:
    """Operands of one QKVFunction: the bf16 fused weight [Wq;Wk;Wv], rebuilt when a weight changes (its transpose is
    built by the first backward), and, rebuilt when any parameter changes, the fp32 fused bias (a missing bias is a block
    of zeros) and the bf16 LoRA operands A_cat [64, K], A_catᵀ, B_ext [n·H, 64], B_extᵀ.  The LoRA tensors are written
    into their slots of two persistent fp32 staging matrices (the padding stays zero) and the four operands come out of
    two a4r_cast_transpose_f32_bf16 launches.  With a ones column, the constant bias of T = x·A_catᵀ sets column 63 to 1:
    it adds nothing to qkv (B_ext[:, 63] = 0) and makes the bias gradients one more column of the dqkvᵀ·T gradient."""

    def __init__(self):
        self.w_key = self.key = self.layout = None
        self.w = self.wt = self.bias = self.lora = None

    def get(self, P, slots, ones):
        """(W, bias, (T's bias, A_cat, A_catᵀ, B_ext, B_extᵀ) or None without LoRA)"""
        key = _param_key([W for W, _, _, _ in P])
        if key != self.w_key:
            self.w_key, self.wt = key, None
            self.w = torch.cat([W.detach().to(BF16) for W, _, _, _ in P], 0).contiguous()
        key = _param_key([t for p in P for t in p])
        if key != self.key:
            self.key = key
            self._build(P, slots, ones)
        return self.w, self.bias, self.lora

    def _build(self, P, slots, ones):
        (H, K), dev = P[0][0].shape, P[0][0].device
        layout = (dev, H, K, len(P), slots)
        if layout != self.layout:
            self.layout = layout
            self.zero = torch.zeros(H, dtype=torch.float32, device=dev)
            if slots:
                self.stage = (torch.zeros((LORA_PAD, K), dtype=torch.float32, device=dev),
                              torch.zeros((len(P) * H, LORA_PAD), dtype=torch.float32, device=dev))
                self.t_bias = torch.zeros(LORA_PAD, dtype=torch.float32, device=dev)
                if ones:
                    self.t_bias[LORA_PAD - 1] = 1.0
        self.bias = torch.cat([self.zero if b is None else b.detach().float() for _, b, _, _ in P])
        self.lora = None
        if slots:
            a_stage, b_stage = self.stage
            for j, o, r in slots:
                a_stage[o:o + r].copy_(P[j][2].detach())
                torch.mul(P[j][3].detach(), 1.0 / r, out=b_stage[j * H:(j + 1) * H, o:o + r])
            self.lora = (self.t_bias,) + ops.cast_transpose(a_stage, True, True) + ops.cast_transpose(b_stage, True, True)

    def weight_t(self):
        if self.wt is None:
            self.wt = self.w.t().contiguous()
        return self.wt


class QKVFunction(torch.autograd.Function):
    """Fused q|k|v projection of one attention module:  qkv = x·[Wq;Wk;Wv]ᵀ + [bq;bk;bv]  (one GEMM, N = 3H), where any
    of the three may be a loralib Linear (Downstream/Text/run.py:414-428):  + (x·Aᵀ)·Bᵀ / r.  The low-rank term rides in
    the same tcgen05 tile as a K-extension: T = x·A_catᵀ  [M,64]  is one skinny GEMM, then
    qkv = [x | T]·[W_cat | B_ext]ᵀ with B_ext the block matrix of the (scaled) lora_B factors.

    params = (W, b, lora_A, lora_B) per fused projection (3 for q|k|v, 1 for a stand-alone loralib Linear), None where
    absent; their operands come from `cache` (QKVCache).  with_skip: x is returned as a second output too.  A caller that
    feeds it to the block's skip connection gets the skip gradient delivered to this node, where it rides in the epilogue
    of the data-gradient GEMM instead of costing a separate elementwise add per layer."""

    PARAMS = ("weight", "bias", "lora_A", "lora_B")

    @staticmethod
    def args(n):
        """argument names of the node over n projections; (j, name) is parameter `name` of projection j"""
        return ("x", "cache", "with_skip") + tuple((j, p) for j in range(n) for p in QKVFunction.PARAMS)

    @staticmethod
    def forward(ctx, x, cache, with_skip, *params):
        P = [params[i:i + 4] for i in range(0, len(params), 4)]
        need = _needs(ctx, QKVFunction.args(len(P)))
        slots, ones = _lora_slots(P)
        w, bias, lora = cache.get(P, slots, ones)
        T = a_cat_t = b_ext_t = None
        if lora is None:
            qkv = ops.gemm(x, w, bias=bias)
        else:
            t_bias, a_cat, a_cat_t, b_ext, b_ext_t = lora
            T = ops.gemm(x, a_cat, bias=t_bias)
            qkv = ops.gemm(x, w, bias=bias, a2=T, b2=b_ext)
        ctx.set_materialize_grads(False)
        ctx.cache, ctx.slots, ctx.ones, ctx.n, ctx.H = cache, slots, ones, len(P), P[0][0].shape[0]
        need_x = any(need[(j, "weight")] or need[(j, "lora_A")] for j in range(len(P)))
        ctx.save_for_backward(x if need_x else None, T, a_cat_t, b_ext_t)
        return (qkv, x) if with_skip else qkv          # autograd treats a returned input as x.view_as(x)

    @staticmethod
    def backward(ctx, dqkv, dskip=None):
        x, T, a_cat_t, b_ext_t = ctx.saved_tensors
        names = QKVFunction.args(ctx.n)
        if dqkv is None:                                  # only the skip output was used downstream
            return (dskip,) + (None,) * (len(names) - 1)
        need, grads = _needs(ctx, names), {}
        H, n, slots = ctx.H, ctx.n, ctx.slots
        third = lambda t, j: t[:, j * H:(j + 1) * H]
        dqkv, dskip = dqkv.contiguous(), None if dskip is None else dskip.contiguous()
        wt = ctx.cache.weight_t()
        dT = None
        if slots:
            # dT = dqkv·B_ext [M,64].  B_ext has non-zero rows only in the thirds whose projection carries a LoRA pair, so
            # this HBM-bound skinny GEMM reads those thirds of dqkv (one K-segment, or two through the second operand
            # pair: LoRA on q and v, run.py:414-428, skips the key third), or all of dqkv when every projection has one
            segs = [(dqkv, b_ext_t)] if len(slots) == n else [(third(dqkv, j), third(b_ext_t, j)) for j, _, _ in slots]
            a2, b2 = segs[1] if len(segs) == 2 else (None, None)
            dT = ops.gemm(*segs[0], a2=a2, b2=b2)
        if need["x"]:                                     # dx = [dqkv | dT]·[W_cat ; A_cat] (+ the skip gradient)
            grads["x"] = ops.gemm(dqkv, wt, a2=dT, b2=a_cat_t, residual=dskip)
        if ctx.ones:
            # ONE weight-gradient pass over a third of dqkv (over all of it when every third is wanted) gives that
            # projection's bias and lora_B gradients, dqkvᵀ·[T | 1]; ONE pass over x gives every lora_A, dTᵀ·x (dT carries
            # the 1/r of B_ext).  A third whose bias and lora_B need no gradient (the frozen key) is not read.
            rows = [need[(j, "bias")] or need[(j, "lora_B")] for j in range(n)]
            g1 = [None] * n
            if all(rows):
                full = ops.wgrad(dqkv, T)                                    # [n·H, 64]
                g1 = [full[j * H:(j + 1) * H] for j in range(n)]
            elif any(rows):
                g1 = [ops.wgrad(third(dqkv, j), T) if rows[j] else None for j in range(n)]
            g2 = ops.wgrad(dT, x) if any(need[(j, "lora_A")] for j in range(n)) else None      # [64, K]
            bias_grad = lambda j: g1[j][:, LORA_PAD - 1].contiguous()
            b_grad = lambda j, o, r: g1[j][:, o:o + r] * (1.0 / r)
            a_grad = lambda o, r: g2[o:o + r].contiguous()
        else:
            # no LoRA, or ranks that fill all 64 columns of T: column sums, and weight gradients over aligned windows
            bias_grad = lambda j: ops.colsum(third(dqkv, j))
            b_grad = lambda j, o, r: _pad_cols_wgrad(third(dqkv, j), T, o, r, 1.0 / r, transpose=False)
            a_grad = lambda o, r: _pad_cols_wgrad(dT, x, o, r, 1.0, transpose=True)
        for j in range(n):
            if need[(j, "weight")]:
                grads[(j, "weight")] = ops.wgrad(third(dqkv, j), x)
            if need[(j, "bias")]:
                grads[(j, "bias")] = bias_grad(j)
        for j, o, r in slots:
            if need[(j, "lora_B")]:                      # lora_B [H, r] = (1/r) dq_jᵀ·T_j
                grads[(j, "lora_B")] = b_grad(j, o, r)
            if need[(j, "lora_A")]:                      # lora_A [r, K] = dT_jᵀ·x
                grads[(j, "lora_A")] = a_grad(o, r)
        return tuple(grads.get(k) for k in names)


def qkv(x, modules, cache, skip=False):
    """QKVFunction over the projection modules (query, key, value; any may be a LoRALinear) or one stand-alone
    LoRALinear, with their QKVCache.  skip: returns (qkv, x') where x' is x as the node's second output (x itself when x
    needs no gradient); the caller uses x' as the block's skip input."""
    params = [getattr(m, name, None) for m in modules for name in QKVFunction.PARAMS]
    with_skip = skip and x.requires_grad
    out = QKVFunction.apply(x, cache, with_skip, *params)
    return (out, x) if skip and not with_skip else out


def _pad_cols_wgrad(a, b, off, r, alpha, transpose):
    """Skinny wgrad where the rank-r operand is columns [off, off+r) of a 64-wide buffer.  The kernel wants 16-byte
    aligned column windows, so compute over the aligned window and slice."""
    lo = (off // 8) * 8
    hi = ((off + r + 7) // 8) * 8
    if transpose:      # result [r, K] from a = dT [M,64] (window), b = x [M,K]
        full = ops.wgrad(a[:, lo:hi], b, alpha=alpha)
        return full[off - lo:off - lo + r].contiguous()
    full = ops.wgrad(a, b[:, lo:hi], alpha=alpha)   # result [H, window]
    return full[:, off - lo:off - lo + r].contiguous()


class EmbedLNFunction(torch.autograd.Function):
    """K1 with the soft-prompt substitution.  Adapter tuning trains at most the prompt rows; under full fine-tuning
    (fine_tune_to = all, Pretraining/*) the word / position / token-type tables and the embedding LayerNorm are trainable
    too: `params` = (word_weight, pos_weight, type_weight, ln_weight, ln_bias) are the fp32 masters, passed so autograd can
    hand their gradients back (None entries = frozen)."""

    @staticmethod
    def forward(ctx, ids, L, tables, gamma, beta, eps, roberta_pad_id, prompt, word_pad_idx, *params):
        word, pos, typ = tables
        need_prompt = prompt is not None and prompt.requires_grad
        need_tab = [p is not None and p.requires_grad for p in params] + [False] * (5 - len(params))
        need = need_prompt or any(need_tab)
        p16 = None if prompt is None else prompt.detach().to(BF16).contiguous()
        out, z, mean, rstd = ops.embed_ln_fwd(ids, L, word, pos, typ, gamma, beta, eps, roberta_pad_id=roberta_pad_id,
                                              prompt=p16, want_z=need)
        ctx.L, ctx.need_prompt, ctx.need_tab, ctx.roberta_pad_id, ctx.word_pad_idx = L, need_prompt, need_tab, roberta_pad_id, word_pad_idx
        ctx.n_prompt = 0 if prompt is None else prompt.shape[0]
        ctx.shapes = [None if p is None else tuple(p.shape) for p in params]
        if need:
            ctx.save_for_backward(z, mean, rstd, gamma, ids)
        return out

    @staticmethod
    def backward(ctx, dout):
        z, mean, rstd, gamma, ids = ctx.saved_tensors
        need_word, need_pos, need_typ, need_g, need_b = ctx.need_tab
        dg = db = None
        if need_g or need_b:
            dg, db = torch.empty_like(gamma), torch.empty_like(gamma)
        dz = ops.layernorm_bwd(dout.contiguous(), z, mean, rstd, gamma, dgamma=dg, dbeta=db)
        H = dz.shape[1]
        L, n = ctx.L, ctx.n_prompt
        dp = None
        if ctx.need_prompt:
            # d prompt[t] = sum over items of dz[item, t]: view [N, L*H] and column-sum the first n*H columns
            dp = ops.colsum(dz.view(-1, L * H), width=n * H).view(n, H)
        grads = [None] * len(ctx.shapes)
        tok = ids[:, :L]
        if need_word:
            idx = tok.clone()
            if n > 0:
                idx[:, :n] = -1                                    # positions replaced by the soft prompt read no table row
            grads[0] = ops.scatter_add_rows(dz, idx, ctx.shapes[0][0], skip_idx=ctx.word_pad_idx)
        if need_pos:
            P = ctx.shapes[1][0]
            if ctx.roberta_pad_id >= 0:
                # RobertaEmbeddings: position ids from the token ids (cumsum over non-pad tokens), padding_idx = pad id
                m = (tok != ctx.roberta_pad_id).long()
                pos_ids = torch.cumsum(m, 1) * m + ctx.roberta_pad_id
                grads[1] = ops.scatter_add_rows(dz, pos_ids, P, skip_idx=ctx.roberta_pad_id)
            else:
                g = torch.zeros((P, H), dtype=torch.float32, device=dz.device)
                g[:L] = ops.colsum(dz.view(-1, L * H)).view(L, H)   # position l of every item reads row l
                grads[1] = g
        if need_typ:
            g = torch.zeros(ctx.shapes[2], dtype=torch.float32, device=dz.device)
            g[0] = ops.colsum(dz)                                   # token_type_ids are all zero on this path
            grads[2] = g
        if need_g:
            grads[3] = dg
        if need_b and len(grads) > 4:
            grads[4] = db
        return (None, None, None, None, None, None, None, dp, None) + tuple(grads)


class BceLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, prec, emb, log_mask, cpc):
        loss, count, pos, neg = ops.bce_loss_fwd(prec, emb, log_mask, cpc=cpc)
        ctx.cpc = cpc
        ctx.log_mask = log_mask
        ctx.save_for_backward(prec, emb, pos, neg, count)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad_out):
        prec, emb, pos, neg, count = ctx.saved_tensors
        go = grad_out.reshape(1).float().contiguous()
        d_prec, d_emb = ops.bce_loss_bwd(prec, emb, ctx.log_mask, pos, neg, count, grad_out=go, cpc=ctx.cpc)
        return d_prec, d_emb, None, None


def bce_loss(prec, emb, log_mask, cpc=False):
    return BceLossFunction.apply(prec, emb, log_mask, cpc)


class InbatchCeFunction(torch.autograd.Function):
    """K9-S: in-batch softmax + duplicate-item mask + CE (a4r_inbatch_ce_*); nothing but the row log-sum-exps is saved."""

    @staticmethod
    def forward(ctx, prec, emb, item_ids, log_mask, cand_bias):
        loss, count, lse = ops.inbatch_ce_fwd(prec, emb, item_ids, log_mask, cand_bias)
        ctx.aux = (item_ids, log_mask, cand_bias)
        ctx.save_for_backward(prec, emb, lse, count)
        return loss.view(())

    @staticmethod
    def backward(ctx, grad_out):
        prec, emb, lse, count = ctx.saved_tensors
        item_ids, log_mask, cand_bias = ctx.aux
        go = grad_out.reshape(1).float().contiguous()
        d_prec, d_emb = ops.inbatch_ce_bwd(prec, emb, item_ids, log_mask, lse, count, cand_bias=cand_bias, grad_out=go)
        return d_prec, d_emb, None, None, None


def inbatch_softmax_loss(prec, emb, item_ids, log_mask, cand_bias=None):
    return InbatchCeFunction.apply(prec, emb, item_ids, log_mask, cand_bias)


class AdapterBlockFunction(torch.autograd.Function):
    """K5 as one autograd node, optionally behind a frozen dense layer or FFN pair F (the serial Houlsby wrapper of a
    frozen post-LN block, BertAdaptedSelfOutput.forward, Downstream/Text/model/model.py:292-297):

        h   = dropout(F(x)) when F is given, else x
        out = tail(h + W_u act(W_d h + b_d) + b_u [+ inp])       tail = LayerNorm (gamma given), + inp, or nothing

    Forward: F's GEMMs (dropout in the epilogue of the last one, counter RNG), then the fused a4r_adapter_ln_fwd kernel.
    Backward: LayerNorm backward, two skinny data-gradient GEMMs and the rank-r weight / bias gradients.  The second GEMM
    forms (ds W_d + dz) and, behind F, masks the SUM with the regenerated dropout mask in its epilogue
    (`dropout_after_residual`), so no stand-alone dropout pass exists in either direction; GELU′ and — when `inp` is x
    itself (the feed-forward block) — the skip gradient ride in the epilogues of F's data-gradient GEMMs.  Trainable: the
    adapter and the LayerNorm; F (given only with the LayerNorm tail) is frozen."""

    ARGS = ("x", "inp", "w_down", "b_down", "w_up", "b_up", "gamma", "beta", "eps", "act", "cache_d", "cache_u", "p", "F")

    @staticmethod
    def forward(ctx, x, inp, w_down, b_down, w_up, b_up, gamma, beta, eps, act, cache_d, cache_u, p, F):
        tail = 0 if gamma is not None else (1 if inp is not None else 2)
        assert F is None or tail == 0, "a frozen F is fused only with the LayerNorm tail"
        need = any(_needs(ctx, AdapterBlockFunction.ARGS).values())
        h, u, rng = x, None, None
        if F is not None:
            rng = _dropout_rng(p, x, F)
            h, u = _frozen_fwd(x, F, None, rng, need)
        wd, _ = cache_d.get(w_down)
        wu, _ = cache_u.get(w_up)
        g = b = None
        if tail == 0:
            g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        out, z, mean, rstd, s, u_ad = ops.adapter_ln_fwd(h, inp, wd, b_down.detach().float().contiguous(), wu,
                                                         b_up.detach().float().contiguous(), g, b, eps, act=act, tail=tail,
                                                         save=need)
        ctx.act, ctx.tail, ctx.rng, ctx.F, ctx.caches = act, tail, rng, F, (cache_d, cache_u)
        ctx.fold = F is not None and inp is x
        ctx.save_for_backward(h, z, mean, rstd, g, s, u_ad, u, w_down, w_up)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, z, mean, rstd, g, s, u_ad, u, w_down, w_up = ctx.saved_tensors
        need = _needs(ctx, AdapterBlockFunction.ARGS)
        grads = {}
        dz = dout.contiguous()
        if ctx.tail == 0:
            if need["gamma"] or need["beta"]:
                grads["gamma"], grads["beta"] = torch.empty_like(g), torch.empty_like(g)
            dz = ops.layernorm_bwd(dz, z, mean, rstd, g, dgamma=grads.get("gamma"), dbeta=grads.get("beta"))
        cache_d, cache_u = ctx.caches
        _, wut = cache_u.get(w_up, need_t=True)      # [r, H]
        _, wdt = cache_d.get(w_down, need_t=True)    # [H, r]
        if ctx.act == "gelu":
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DGELU, aux=u_ad)
        else:
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DRELU, aux=s)
        if need["w_down"]:
            grads["w_down"] = ops.wgrad(ds, h)
        if need["b_down"]:
            grads["b_down"] = ops.colsum(ds)
        if need["w_up"] or need["b_up"]:
            full = ops.wgrad(dz, ops.s_ext(s))               # dzᵀ · [s | 1]: weight and bias gradient in one pass over dz
            grads["w_up"], grads["b_up"] = full[:, :s.shape[1]], full[:, s.shape[1]]
        if need["x"]:
            # gradient at h, through F's dropout when there is one: (ds W_d + dz) * mask / (1 - p) in ONE epilogue
            dh = ops.gemm(ds, wdt, residual=dz, dropout=ctx.rng, dropout_after=True)
            grads["x"] = dh if ctx.F is None else _frozen_bwd(dh, u, ctx.F, dz if ctx.fold else None)
        if need["inp"] and not ctx.fold:
            grads["inp"] = dz
        return tuple(grads.get(n) for n in AdapterBlockFunction.ARGS)


def adapter_block(x, inp, adapter, ln=None, dense=None, intermediate=None, p=0.0):
    """AdapterBlockFunction.  adapter: the AdapterBlock (fc_down, fc_up, act); ln: a LayerNorm module or None;
    dense / intermediate: the frozen Linear modules of F (dense None: no F; intermediate None: F is dense alone)."""
    d, up = adapter.fc_down, adapter.fc_up
    return AdapterBlockFunction.apply(x, inp, d.weight, d.bias, up.weight, up.bias, *_ln_args(ln), adapter.act, d._cache,
                                      up._cache, p, None if dense is None else _frozen(dense, intermediate))


class IdEmbeddingFunction(torch.autograd.Function):
    """The id item tower's lookup (nn.Embedding(item_num + 1, D, padding_idx) reached from Model.forward with
    use_modal = False): ids [B, S1, 2] -> (emb [B, S1, 2, D], hist [B, S1-1, D] = emb[:, :-1, 0]) bf16 from the fp32 master.

    The backward adds the table gradient of BOTH outputs straight into `weight.grad` (created as zeros when absent) and
    returns None for the weight: the trainer's `.grad` is a view into its flat buffer, and a returned dense [V, D] tensor
    would make autograd allocate, zero, add and free a full-table temporary per pass for a gradient that touches at most
    B*S1*2 rows.  Rows are summed in fp32 in a fixed order without atomics (bit-identical run to run and under a graph
    replay); row padding_idx is never written."""

    @staticmethod
    def forward(ctx, ids, weight, padding_idx):
        emb, hist = ops.id_embed_fwd(weight.detach(), ids)
        ctx.save_for_backward(ids)
        ctx.weight, ctx.padding_idx = weight, padding_idx
        return emb, hist

    @staticmethod
    def backward(ctx, d_emb, d_hist):
        (ids,) = ctx.saved_tensors
        w = ctx.weight
        if d_emb is None and d_hist is None:
            return None, None, None
        if w.grad is None:
            w.grad = torch.zeros_like(w)
        ref = d_emb if d_emb is not None else d_hist
        B, S1 = ids.shape[0], ids.shape[1]
        if d_emb is None:
            d_emb = torch.zeros((B, S1, 2, w.shape[1]), dtype=ref.dtype, device=ref.device)
        ops.id_embed_bwd(ids, d_emb.contiguous(), None if d_hist is None else d_hist.contiguous(), w.grad,
                         padding_idx=ctx.padding_idx, accumulate=True)
        return None, None, None


def id_embedding(ids, weight, padding_idx=0):
    return IdEmbeddingFunction.apply(ids, weight, padding_idx)
