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


class WeightCache:
    """bf16 copies of an fp32 master weight: W [N,K] for the forward GEMM and Wᵀ [K,N] for the data-gradient GEMM.
    Rebuilt when the parameter is modified in place (optimizer step, load_state_dict) or moved."""

    def __init__(self):
        self.key = None
        self.master = None
        self.w = None
        self.wt = None

    def get(self, weight, need_t=False):
        key = (weight.data_ptr(), weight._version, weight.device, PARAM_EPOCH[0] if weight.requires_grad else -1)
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


class FFNFunction(torch.autograd.Function):
    """Frozen BERT feed-forward: h = GELU(y Wiᵀ + bi) Wfᵀ + bf (+ residual).  The backward fuses GELU' into the epilogue
    of the first data-gradient GEMM and the residual gradient into the second, and keeps only the pre-activation."""

    @staticmethod
    def forward(ctx, y, wi, bi, wf, bf, residual, cache_i, cache_f):
        w1, _ = cache_i.get(wi)
        w2, _ = cache_f.get(wf)
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[5]
        u = torch.empty((y.shape[0], w1.shape[0]), dtype=BF16, device=y.device) if need else None
        f = ops.gemm(y, w1, bias=bi.detach(), epilogue=ops.EPI_GELU, aux=u)
        h = ops.gemm(f, w2, bias=bf.detach(), residual=residual)
        ctx.caches = (cache_i, cache_f)
        ctx.has_res = residual is not None
        ctx.res_is_input = residual is y
        ctx.save_for_backward(u, wi, wf)
        return h

    @staticmethod
    def backward(ctx, dh):
        u, wi, wf = ctx.saved_tensors
        dh = dh.contiguous()
        _, w2t = ctx.caches[1].get(wf, need_t=True)
        _, w1t = ctx.caches[0].get(wi, need_t=True)
        du = ops.gemm(dh, w2t, epilogue=ops.EPI_DGELU, aux=u)
        # when the residual IS the input (post-LN BERT: h = FFN(y) + y) its gradient is folded into the epilogue of the
        # last data-gradient GEMM and nothing is returned for the residual slot (autograd would add them otherwise).
        fold = ctx.has_res and ctx.res_is_input
        dy = ops.gemm(du, w1t, residual=dh if fold else None) if ctx.needs_input_grad[0] else None
        dres = dh if (ctx.has_res and not fold and ctx.needs_input_grad[5]) else None
        return dy, None, None, None, None, dres, None, None


class PostLNBlockFunction(torch.autograd.Function):
    """One frozen post-LN residual block of BERT in a single autograd node:

        out = LayerNorm(dropout(F(x)) + res)       F(x) = x Woᵀ + bo                      (attention.output: BertSelfOutput)
                                                  F(x) = GELU(x Wiᵀ + bi) Wfᵀ + bf       (intermediate + output: BertOutput)

    Forward: dropout and the residual add live in the epilogue of the last GEMM (counter RNG).  Backward: LayerNorm's
    backward kernel emits dz AND dz ⊙ mask/(1-p) (the gradient through the dropout) in one pass; GELU′ and the residual
    gradient live in the epilogues of the data-gradient GEMMs.  Only LayerNorm may be trainable (finetune_layernorm)."""

    @staticmethod
    def forward(ctx, x, res, gamma, beta, eps, p, w1, b1, cache1, w2, b2, cache2):
        ffn = w2 is not None
        need = any(ctx.needs_input_grad[:4])
        rng = (float(p),) + DropoutState.draw((x.shape[0] * (w2 if ffn else w1).shape[0] + 3) // 4) if p > 0 else None
        wa, _ = cache1.get(w1)
        u = None
        if ffn:
            wb, _ = cache2.get(w2)
            u = torch.empty((x.shape[0], wa.shape[0]), dtype=BF16, device=x.device) if need else None
            f = ops.gemm(x, wa, bias=b1.detach(), epilogue=ops.EPI_GELU, aux=u)
            z = ops.gemm(f, wb, bias=b2.detach(), residual=res, dropout=rng)
        else:
            z = ops.gemm(x, wa, bias=b1.detach(), residual=res, dropout=rng)
        g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        out, _, mean, rstd = ops.layernorm_fwd(z, g, b, eps, want_stats=need)
        ctx.rng, ctx.ffn, ctx.caches = rng, ffn, (cache1, cache2)
        ctx.res_is_input = res is x
        if need:
            ctx.save_for_backward(z, mean, rstd, g, u, w1, w2)
        return out

    @staticmethod
    def backward(ctx, dout):
        z, mean, rstd, g, u, w1, w2 = ctx.saved_tensors
        dout = dout.contiguous()
        want_ln = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        dg = db = None
        if want_ln:
            dg, db = torch.empty_like(g), torch.empty_like(g)
        r = ops.layernorm_bwd(dout, z, mean, rstd, g, dgamma=dg, dbeta=db, masked=ctx.rng)
        dz, dzm = r if ctx.rng is not None else (r, r)
        dx = None
        if ctx.needs_input_grad[0]:
            fold = dz if ctx.res_is_input else None      # res is x: the skip gradient rides in the last epilogue
            if ctx.ffn:
                _, w2t = ctx.caches[1].get(w2, need_t=True)
                _, w1t = ctx.caches[0].get(w1, need_t=True)
                du = ops.gemm(dzm, w2t, epilogue=ops.EPI_DGELU, aux=u)
                dx = ops.gemm(du, w1t, residual=fold)
            else:
                _, w1t = ctx.caches[0].get(w1, need_t=True)
                dx = ops.gemm(dzm, w1t, residual=fold)
        dres = dz if (ctx.needs_input_grad[1] and not ctx.res_is_input) else None
        return dx, dres, dg, db, None, None, None, None, None, None, None, None


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
    separate autograd accumulation pass over [M, H].  Same trick as QKVFunction's "skip" output on the post-LN side."""

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


class QKVFunction(torch.autograd.Function):
    """Fused q|k|v projection of one attention module:  qkv = x·[Wq;Wk;Wv]ᵀ + [bq;bk;bv]  (one GEMM, N = 3H), where any
    of the three may be a loralib Linear (Downstream/Text/run.py:414-428):  + (x·Aᵀ)·Bᵀ / r.  The low-rank term rides in
    the same tcgen05 tile as a K-extension: T = x·A_catᵀ  [M,64]  is one skinny GEMM, then
    qkv = [x | T]·[W_cat | B_ext]ᵀ with B_ext the block matrix of the (scaled) lora_B factors.

    params = (W, b, lora_A, lora_B) per fused projection (3 for q|k|v, 1 for a stand-alone loralib Linear), None where absent."""

    @staticmethod
    def forward(ctx, x, cache, *params):
        """params may end with the marker string "skip": the function then ALSO returns x (as a second output).  A caller
        that feeds this second output to the block's skip connection gets the skip gradient delivered to THIS node, where
        it rides in the epilogue of the data-gradient GEMM instead of costing a separate elementwise add per layer."""
        ctx.with_skip = len(params) > 0 and isinstance(params[-1], str) and params[-1] == "skip"
        if ctx.with_skip:
            params = params[:-1]
        ctx.set_materialize_grads(False)
        assert len(params) % 4 == 0
        n = len(params) // 4
        H = params[0].shape[0]
        K = params[0].shape[1]
        dev = x.device
        frozen_w = not any(p is not None and p.requires_grad for p in [params[4 * j] for j in range(n)])
        key = tuple((p.data_ptr(), p._version) for p in [params[4 * j] for j in range(n)]) + (PARAM_EPOCH[0] if not frozen_w else -1,)
        if cache.get("key") != key or not frozen_w:
            cache["key"] = key
            cache["w"] = torch.cat([params[i].detach().to(BF16) for i in range(0, 4 * n, 4)], 0).contiguous()
            cache["wt"] = None
        w = cache["w"]
        # the fused bias and the LoRA operand matrices depend on TRAINABLE tensors: rebuilt once per optimizer step (or
        # whenever a parameter object / version changes), not once per forward
        small = [params[4 * j + i] for j in range(n) for i in (1, 2, 3)]
        skey = (PARAM_EPOCH[0],) + tuple(None if p is None else (p.data_ptr(), p._version) for p in small)
        reuse = cache.get("small_key") == skey
        if reuse:
            bias = cache["bias"]
        else:
            # one concatenation (a missing bias contributes a cached block of zeros)
            zero_h = cache.get("zero_h")
            if zero_h is None or zero_h.device != dev or zero_h.numel() != H:
                zero_h = cache["zero_h"] = torch.zeros(H, dtype=torch.float32, device=dev)
            bias = torch.cat([zero_h if params[4 * j + 1] is None else params[4 * j + 1].detach().float() for j in range(n)])
            cache["small_key"], cache["bias"] = skey, bias
        # LoRA bookkeeping: slot j occupies columns [off_j, off_j + r_j) of the 64-wide T
        slots, off = [], 0
        for j in range(n):
            A = params[4 * j + 2]
            if A is not None:
                r = A.shape[0]
                slots.append((j, off, r))
                off += r
        assert off <= LORA_PAD, "sum of LoRA ranks of one fused projection must be <= 64"
        T = a_cat = b_ext = None
        if slots:
            ctx.ones_col = off < LORA_PAD
            if reuse and "a_cat" in cache:
                a_cat, b_ext, t_bias = cache["a_cat"], cache["b_ext"], cache["t_bias"]
            else:
                # Rebuilt once per optimizer step: the operands are assembled in two persistent fp32 staging matrices (the
                # LoRA tensors are written straight into their slots, the padding stays zero) and every bf16 operand of the step
                # — A_cat, A_catᵀ, B_ext, B_extᵀ — comes out of two a4r_cast_transpose_f32_bf16 launches.
                st = cache.get("lora_stage")
                if st is None or st[0].device != dev or st[0].shape != (LORA_PAD, K) or st[1].shape != (n * H, LORA_PAD):
                    st = cache["lora_stage"] = (torch.zeros((LORA_PAD, K), dtype=torch.float32, device=dev),
                                                torch.zeros((n * H, LORA_PAD), dtype=torch.float32, device=dev))
                    cache["lora_slots"] = None
                if cache.get("lora_slots") != slots:               # a different slot layout: clear what the old one wrote
                    st[0].zero_()
                    st[1].zero_()
                    cache["lora_slots"] = list(slots)
                for j, o, r in slots:
                    st[0][o:o + r].copy_(params[4 * j + 2].detach())
                    torch.mul(params[4 * j + 3].detach(), 1.0 / r, out=st[1][j * H:(j + 1) * H, o:o + r])
                a_cat, a_cat_t = ops.cast_transpose(st[0], True, True)
                b_ext, b_ext_t = ops.cast_transpose(st[1], True, True)
                # column 63 of T is a constant 1 (zero weight row + bias 1): it contributes nothing to qkv (B_ext[:, 63] = 0)
                # and turns the bias gradients into one more column of the fused dqkvᵀ·T weight-gradient below
                tb = cache.get("t_bias_const")                      # (ones_col, tensor): a constant, built once
                if tb is None or tb[0] != ctx.ones_col or tb[1].device != dev:
                    t_bias = torch.zeros(LORA_PAD, dtype=torch.float32, device=dev)
                    if ctx.ones_col:
                        t_bias[LORA_PAD - 1] = 1.0
                    tb = cache["t_bias_const"] = (ctx.ones_col, t_bias)
                t_bias = tb[1]
                cache["a_cat"], cache["b_ext"], cache["t_bias"] = a_cat, b_ext, t_bias
                cache["a_cat_t"], cache["b_ext_t"] = a_cat_t, b_ext_t
            T = ops.gemm(x, a_cat, bias=t_bias)
            qkv = ops.gemm(x, w, bias=bias, a2=T, b2=b_ext)
        else:
            qkv = ops.gemm(x, w, bias=bias)
        ctx.cache, ctx.slots, ctx.H, ctx.n = cache, slots, H, n
        if not slots:
            ctx.ones_col = False
        ctx.n_params = len(params)
        ctx.param_needs = [p is not None and p.requires_grad for p in params]
        need_x = any(ctx.param_needs[4 * j + 2] for j in range(n)) or any(ctx.param_needs[4 * j] for j in range(n))
        ctx.save_for_backward(x if need_x else None, T, a_cat, b_ext)
        if ctx.with_skip:
            return qkv, x          # autograd treats a returned input as x.view_as(x)
        return qkv

    @staticmethod
    def backward(ctx, dqkv, dskip=None):
        x, T, a_cat, b_ext = ctx.saved_tensors
        H, cache, n = ctx.H, ctx.cache, ctx.n
        tail = (None,) if ctx.with_skip else ()
        if dqkv is None:                                  # only the skip output was used downstream
            return (dskip, None) + (None,) * ctx.n_params + tail
        dqkv = dqkv.contiguous()
        if dskip is not None:
            dskip = dskip.contiguous()
        if cache.get("wt") is None:
            cache["wt"] = cache["w"].t().contiguous()
        grads = [None] * ctx.n_params
        dT = None
        if ctx.slots:
            # dT = dqkv·B_ext  [M,64];  dx = [dqkv | dT]·[W_catᵀ | A_catᵀ]ᵀ (+ the skip gradient in the epilogue)
            if cache.get("b_ext") is b_ext and cache.get("b_ext_t") is not None:
                b_ext_t, a_cat_t = cache["b_ext_t"], cache["a_cat_t"]
            else:
                b_ext_t, a_cat_t = b_ext.t().contiguous(), a_cat.t().contiguous()
                if cache.get("b_ext") is b_ext:
                    cache["b_ext_t"], cache["a_cat_t"] = b_ext_t, a_cat_t
            # only the projections that carry a LoRA pair have non-zero rows in B_ext: with q|k|v fused and LoRA on q and v
            # (run.py:414-428) the key third of dqkv is skipped — its products are exact zeros — so this HBM-bound skinny
            # GEMM reads 2/3 of dqkv (two K-segments through the GEMM's second operand pair)
            lj = [j for j, _, _ in ctx.slots]
            if n == 3 and len(lj) == 2:
                (ja, jb) = lj
                dT = ops.gemm(dqkv[:, ja * H:(ja + 1) * H], b_ext_t[:, ja * H:(ja + 1) * H],
                              a2=dqkv[:, jb * H:(jb + 1) * H], b2=b_ext_t[:, jb * H:(jb + 1) * H])
            elif n == 3 and len(lj) == 1:
                dT = ops.gemm(dqkv[:, lj[0] * H:(lj[0] + 1) * H], b_ext_t[:, lj[0] * H:(lj[0] + 1) * H])
            else:
                dT = ops.gemm(dqkv, b_ext_t)
            dx = ops.gemm(dqkv, cache["wt"], a2=dT, b2=a_cat_t, residual=dskip) if ctx.needs_input_grad[0] else None
        else:
            dx = ops.gemm(dqkv, cache["wt"], residual=dskip) if ctx.needs_input_grad[0] else None
        fused = bool(ctx.slots) and ctx.ones_col
        if fused:
            # ONE pass over dqkv gives every lora_B and every bias gradient; ONE pass over x gives every lora_A.  Each pass
            # runs only if one of its results is wanted (x is saved only when a lora_A or a weight trains).
            want_g1 = any(ctx.param_needs[4 * j + 1] for j in range(n)) or any(ctx.param_needs[4 * j + 3] for j, _, _ in ctx.slots)
            want_g2 = any(ctx.param_needs[4 * j + 2] for j, _, _ in ctx.slots)
            # g1 rows of projection j are wanted for its bias or its lora_B; a projection that needs neither (the frozen key
            # projection under LoRA on q and v) is not read: one weight-gradient launch per wanted third of dqkv
            g1_rows = [ctx.param_needs[4 * j + 1] or any(jj == j and ctx.param_needs[4 * j + 3] for jj, _, _ in ctx.slots)
                       for j in range(n)]
            g1 = [None] * n
            if want_g1:
                if all(g1_rows):
                    full = ops.wgrad(dqkv, T)                       # [n*H, 64] = dqkvᵀ · [T | 1]
                    g1 = [full[j * H:(j + 1) * H] for j in range(n)]
                else:
                    g1 = [ops.wgrad(dqkv[:, j * H:(j + 1) * H], T) if g1_rows[j] else None for j in range(n)]
            g2 = ops.wgrad(dT, x) if want_g2 else None              # [64, K]   = dTᵀ · x
        for j in range(n):
            dq = dqkv[:, j * H:(j + 1) * H]
            if ctx.param_needs[4 * j]:
                grads[4 * j] = ops.wgrad(dq, x)
            if ctx.param_needs[4 * j + 1]:
                grads[4 * j + 1] = g1[j][:, LORA_PAD - 1].contiguous() if fused else ops.colsum(dq)
        for j, o, r in ctx.slots:
            dq = dqkv[:, j * H:(j + 1) * H]
            if ctx.param_needs[4 * j + 3]:   # lora_B [H, r] = (1/r) dqᵀ · T_j
                grads[4 * j + 3] = (g1[j][:, o:o + r] * (1.0 / r)) if fused else \
                    _pad_cols_wgrad(dq, T, o, r, 1.0 / r, transpose=False)
            if ctx.param_needs[4 * j + 2]:   # lora_A [r, K] = dT_jᵀ · x   (dT already carries the 1/r of B_ext)
                grads[4 * j + 2] = g2[o:o + r].contiguous() if fused else _pad_cols_wgrad(dT, x, o, r, 1.0, transpose=True)
        return (dx, None) + tuple(grads) + tail


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


class HoulsbyBlockFunction(torch.autograd.Function):
    """K5 as one autograd node: out = tail(h + W_u act(W_d h + b_d) + b_u [+ inp]) with tail = LayerNorm (gamma given),
    or nothing.  Forward = the fused a4r_adapter_ln_fwd kernel; backward = LayerNorm backward, two skinny data-gradient
    GEMMs (act' and the skip gradient in their epilogues) and the rank-r weight / bias gradients — no torch arithmetic."""

    @staticmethod
    def forward(ctx, h, inp, w_down, b_down, w_up, b_up, gamma, beta, eps, act, cache_d, cache_u):
        wd, _ = cache_d.get(w_down)
        wu, _ = cache_u.get(w_up)
        tail = 0 if gamma is not None else (1 if inp is not None else 2)
        need = any(ctx.needs_input_grad[:8])
        g = b = None
        if tail == 0:
            g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        out, z, mean, rstd, s, u = ops.adapter_ln_fwd(h, inp, wd, b_down.detach().float().contiguous(), wu,
                                                      b_up.detach().float().contiguous(), g, b, eps, act=act, tail=tail,
                                                      save=need)
        ctx.act, ctx.tail, ctx.caches, ctx.has_inp = act, tail, (cache_d, cache_u), inp is not None
        if need:
            ctx.save_for_backward(h, z, mean, rstd, g, s, u, w_down, w_up)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, z, mean, rstd, g, s, u, w_down, w_up = ctx.saved_tensors
        dout = dout.contiguous()
        dg = db = None
        if ctx.tail == 0:
            if ctx.needs_input_grad[6] or ctx.needs_input_grad[7]:
                dg, db = torch.empty_like(g), torch.empty_like(g)
            dz = ops.layernorm_bwd(dout, z, mean, rstd, g, dgamma=dg, dbeta=db)
        else:
            dz = dout
        _, wut = ctx.caches[1].get(w_up, need_t=True)      # [r, H]
        _, wdt = ctx.caches[0].get(w_down, need_t=True)    # [H, r]
        if ctx.act == "gelu":
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DGELU, aux=u)
        else:
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DRELU, aux=s)
        dh = ops.gemm(ds, wdt, residual=dz) if ctx.needs_input_grad[0] else None
        dwd = ops.wgrad(ds, h) if ctx.needs_input_grad[2] else None
        dbd = ops.colsum(ds) if ctx.needs_input_grad[3] else None
        dwu = dbu = None
        if ctx.needs_input_grad[4] or ctx.needs_input_grad[5]:
            full = ops.wgrad(dz, ops.s_ext(s))               # dzᵀ · [s | 1]: weight and bias gradient in one pass over dz
            dwu, dbu = full[:, :s.shape[1]], full[:, s.shape[1]]
        dinp = dz if (ctx.has_inp and ctx.needs_input_grad[1]) else None
        return dh, dinp, dwd, dbd, dwu, dbu, dg, db, None, None, None, None


def houlsby_block(h, inp, adapter_down, adapter_up, act, ln=None):
    """adapter_down / adapter_up: the AdapterBlock's Linear modules (weight, bias, _cache); ln: a LayerNorm module or None."""
    return HoulsbyBlockFunction.apply(h, inp, adapter_down.weight, adapter_down.bias, adapter_up.weight, adapter_up.bias,
                                      None if ln is None else ln.weight, None if ln is None else ln.bias,
                                      0.0 if ln is None else ln.eps, act, adapter_down._cache, adapter_up._cache)


class HoulsbyPostLNBlockFunction(torch.autograd.Function):
    """One frozen post-LN block of BERT under a serial Houlsby wrapper (BertAdaptedSelfOutput.forward,
    Downstream/Text/model/model.py:292-297) as a single autograd node:

        h   = dropout(F(x))          F(x) = x Woᵀ + bo  (attention.output)  |  GELU(x Wiᵀ + bi) Wfᵀ + bf  (intermediate + output)
        out = LayerNorm(h + W_u act(W_d h + b_d) + b_u + inp)

    Forward: the dropout lives in the epilogue of F's last GEMM (counter RNG), everything after it is the fused K5 kernel.
    Backward: LayerNorm backward -> two skinny data-gradient GEMMs; the second one forms (ds W_d + dz) and masks the SUM
    with the regenerated dropout mask in its epilogue (`dropout_after_residual`), so no stand-alone dropout pass exists in
    either direction; GELU' and — when `inp` is the block input x itself (the feed-forward block) — the skip gradient
    ride in the epilogues of F's data-gradient GEMMs.  Trainable: the adapter and (finetune_layernorm) the LayerNorm."""

    @staticmethod
    def forward(ctx, x, inp, p, w1, b1, cache1, w2, b2, cache2, w_down, b_down, w_up, b_up, gamma, beta, eps, act,
                cache_d, cache_u):
        ffn = w2 is not None
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1] or any(ctx.needs_input_grad[9:15])
        wa, _ = cache1.get(w1)
        n_out = (w2 if ffn else w1).shape[0]
        rng = (float(p),) + DropoutState.draw((x.shape[0] * n_out + 3) // 4) if p > 0 else None
        u = None
        if ffn:
            wb, _ = cache2.get(w2)
            u = torch.empty((x.shape[0], wa.shape[0]), dtype=BF16, device=x.device) if need else None
            f = ops.gemm(x, wa, bias=b1.detach(), epilogue=ops.EPI_GELU, aux=u)
            h = ops.gemm(f, wb, bias=b2.detach(), dropout=rng)
        else:
            h = ops.gemm(x, wa, bias=b1.detach(), dropout=rng)
        wd, _ = cache_d.get(w_down)
        wu, _ = cache_u.get(w_up)
        g, b = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        out, z, mean, rstd, s, u_ad = ops.adapter_ln_fwd(h, inp, wd, b_down.detach().float().contiguous(), wu,
                                                         b_up.detach().float().contiguous(), g, b, eps, act=act, tail=0,
                                                         save=need)
        ctx.rng, ctx.ffn, ctx.act = rng, ffn, act
        ctx.caches = (cache1, cache2, cache_d, cache_u)
        ctx.inp_is_x = inp is x
        if need:
            ctx.save_for_backward(h, z, mean, rstd, g, s, u_ad, u, w1, w2, w_down, w_up)
        return out

    @staticmethod
    def backward(ctx, dout):
        h, z, mean, rstd, g, s, u_ad, u, w1, w2, w_down, w_up = ctx.saved_tensors
        cache1, cache2, cache_d, cache_u = ctx.caches
        dout = dout.contiguous()
        dg = db = None
        if ctx.needs_input_grad[13] or ctx.needs_input_grad[14]:
            dg, db = torch.empty_like(g), torch.empty_like(g)
        dz = ops.layernorm_bwd(dout, z, mean, rstd, g, dgamma=dg, dbeta=db)
        _, wut = cache_u.get(w_up, need_t=True)      # [r, H]
        _, wdt = cache_d.get(w_down, need_t=True)    # [H, r]
        if ctx.act == "gelu":
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DGELU, aux=u_ad)
        else:
            ds = ops.gemm(dz, wut, epilogue=ops.EPI_DRELU, aux=s)
        dwd = ops.wgrad(ds, h) if ctx.needs_input_grad[9] else None
        dbd = ops.colsum(ds) if ctx.needs_input_grad[10] else None
        dwu = dbu = None
        if ctx.needs_input_grad[11] or ctx.needs_input_grad[12]:
            full = ops.wgrad(dz, ops.s_ext(s))               # dzᵀ · [s | 1]: weight and bias gradient in one pass over dz
            dwu, dbu = full[:, :s.shape[1]], full[:, s.shape[1]]
        dx = None
        if ctx.needs_input_grad[0]:
            # gradient at the dense output, through the dropout: (ds W_d + dz) * mask / (1 - p) in ONE epilogue
            dhm = ops.gemm(ds, wdt, residual=dz, dropout=ctx.rng, dropout_after=True)
            fold = dz if ctx.inp_is_x else None
            _, w1t = cache1.get(w1, need_t=True)
            if ctx.ffn:
                _, w2t = cache2.get(w2, need_t=True)
                du = ops.gemm(dhm, w2t, epilogue=ops.EPI_DGELU, aux=u)
                dx = ops.gemm(du, w1t, residual=fold)
            else:
                dx = ops.gemm(dhm, w1t, residual=fold)
        dinp = dz if (ctx.needs_input_grad[1] and not ctx.inp_is_x) else None
        return (dx, dinp, None, None, None, None, None, None, None, dwd, dbd, dwu, dbu, dg, db, None, None, None, None)


def houlsby_postln_block(x, inp, p, dense, intermediate, adapter, ln):
    """dense / intermediate: the frozen Linear modules of the block (intermediate None for attention.output);
    adapter: the AdapterBlock; ln: the block's LayerNorm module."""
    if intermediate is None:
        w1, b1, c1, w2, b2, c2 = dense.weight, dense.bias, dense._cache, None, None, None
    else:
        w1, b1, c1 = intermediate.weight, intermediate.bias, intermediate._cache
        w2, b2, c2 = dense.weight, dense.bias, dense._cache
    return HoulsbyPostLNBlockFunction.apply(x, inp, p, w1, b1, c1, w2, b2, c2, adapter.fc_down.weight, adapter.fc_down.bias,
                                            adapter.fc_up.weight, adapter.fc_up.bias, ln.weight, ln.bias, ln.eps,
                                            adapter.act, adapter.fc_down._cache, adapter.fc_up._cache)


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
