"""Tensor-level wrappers over the C ABI: every function takes CUDA torch tensors, passes raw device pointers and
the current CUDA stream to libadapter4rec_sm100.so, and returns torch tensors.  PyTorch is only the owner of
device memory and streams here — no arithmetic of the hot path is done by torch ops."""
import ctypes

import torch

from . import lib as _l
from .lib import EPI_DGELU, EPI_DRELU, EPI_GELU, EPI_LINEAR, EPI_RELU  # noqa: F401

BF16 = torch.bfloat16
F32_MIN = -3.4028234663852886e38  # torch.finfo(torch.float32).min: the transformers additive attention mask value


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _rows2d(t, name):
    """[rows, cols] view requirements of the ABI: unit column stride, row stride in elements."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError("%s must be 2-D with unit column stride, got shape %s stride %s" % (name, tuple(t.shape), t.stride()))
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


_workspaces = {}


def workspace(nbytes, device):
    """Grow-only scratch buffer per (device, stream); owned by torch's allocator, handed to the library per call."""
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


_gemm_profile = None


def gemm_profile_start():
    """bench.py: bracket every GEMM launch with CUDA events on the launching stream (roofline.achieved)."""
    global _gemm_profile
    _gemm_profile = []


def gemm_profile_stop(by_shape=False):
    """returns (total algorithmic FLOPs, total device milliseconds, launches) since gemm_profile_start(); with by_shape
    also a dict {(M, N, K+K2, epilogue): [flops, ms, launches]}."""
    global _gemm_profile
    prof, _gemm_profile = _gemm_profile, None
    torch.cuda.synchronize()
    flops = sum(p[0] for p in prof)
    times = [p[1].elapsed_time(p[2]) for p in prof]
    ms = sum(times)
    if not by_shape:
        return flops, ms, len(prof)
    groups = {}
    for p, t in zip(prof, times):
        g = groups.setdefault(p[3], [0.0, 0.0, 0])
        g[0] += p[0]
        g[1] += t
        g[2] += 1
    return flops, ms, len(prof), groups


def gemm(a, b, bias=None, epilogue=EPI_LINEAR, residual=None, residual2=None, aux=None, a2=None, b2=None,
         alpha=1.0, out=None, out_dtype=BF16, block_n=0, dropout=None, dropout_after=False):
    """C[M,N] = epi(alpha * (a @ b.T + a2 @ b2.T) + bias)  — see a4r_gemm_bf16_tn in include/adapter4rec.h.
    dropout = (p, seed, offset): mask on the LINEAR epilogue value before the residuals, or (dropout_after) on the sum."""
    assert a.dtype == BF16 and b.dtype == BF16, "gemm operands must be bf16"
    M, K = a.shape
    N, Kb = b.shape
    assert K == Kb, "gemm: K mismatch %d vs %d" % (K, Kb)
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=a.device)
    g = _l.GemmArgs()
    g.A, g.lda = _p(a), _rows2d(a, "a")
    g.B, g.ldb = _p(b), _rows2d(b, "b")
    if a2 is not None:
        assert a2.dtype == BF16 and b2.dtype == BF16 and a2.shape[0] == M and b2.shape[0] == N and a2.shape[1] == b2.shape[1]
        g.A2, g.lda2, g.B2, g.ldb2, g.K2 = _p(a2), _rows2d(a2, "a2"), _p(b2), _rows2d(b2, "b2"), a2.shape[1]
    g.C, g.ldc = _p(out), _rows2d(out, "out")
    if aux is not None:
        assert aux.dtype == BF16 and tuple(aux.shape) == (M, N)
        g.aux, g.ldaux = _p(aux), _rows2d(aux, "aux")
    if residual is not None:
        assert residual.dtype == BF16 and tuple(residual.shape) == (M, N)
        g.residual, g.ldr = _p(residual), _rows2d(residual, "residual")
    if residual2 is not None:
        assert residual2.dtype == BF16 and tuple(residual2.shape) == (M, N)
        g.residual2, g.ldr2 = _p(residual2), _rows2d(residual2, "residual2")
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N and bias.is_contiguous()
        g.bias = _p(bias)
    g.M, g.N, g.K = M, N, K
    if dropout is not None:
        assert out.is_contiguous(), "epilogue dropout indexes the logical [M, N] output"
        g.dropout_p, g.dropout_seed, g.dropout_offset = float(dropout[0]), int(dropout[1]), int(dropout[2])
        g.dropout_after_residual = int(bool(dropout_after))
    g.alpha, g.epilogue, g.out_f32, g.block_n = float(alpha), int(epilogue), int(out.dtype == torch.float32), int(block_n)
    assert out.dtype in (BF16, torch.float32)
    if _gemm_profile is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _l.check(_l.get_lib().a4r_gemm_bf16_tn(ctypes.byref(g), _stream()), "a4r_gemm_bf16_tn")
        e1.record()
        k2 = a2.shape[1] if a2 is not None else 0
        _gemm_profile.append((2.0 * M * N * (K + k2), e0, e1, (M, N, K + k2, int(epilogue))))
        return out
    _l.check(_l.get_lib().a4r_gemm_bf16_tn(ctypes.byref(g), _stream()), "a4r_gemm_bf16_tn")
    return out


def dropout(x, res, p, seed, offset):
    """out = x * mask / (1 - p) (+ res); the mask is a pure function of (seed, offset, element index)."""
    assert x.dtype == BF16 and x.is_contiguous() and (res is None or (res.dtype == BF16 and res.is_contiguous() and res.shape == x.shape))
    out = torch.empty_like(x)
    _l.check(_l.get_lib().a4r_dropout(_p(x), _p(res), _p(out), x.numel(), float(p), int(seed), int(offset), _stream()),
             "a4r_dropout")
    return out


def _attn_args(qkv, N, L, heads, head_dim, mask, causal, mask_neg, dropout=None, scale=None, cu_seqlens=None):
    a = _l.AttnArgs()
    if cu_seqlens is not None:
        # packed layout: rows [cu[n], cu[n+1]) belong to sequence n; the mask (if any) is per token row
        assert cu_seqlens.dtype == torch.int32 and cu_seqlens.is_contiguous() and cu_seqlens.numel() == N + 1 and L <= 32
        a.cu_seqlens = _p(cu_seqlens)
        if mask is not None:
            assert mask.dim() == 1 and mask.numel() == qkv.shape[0] and mask.is_contiguous()
            a.mask, a.mask_ld = _p(mask), 0
            a.mask_dtype = {torch.int64: 1, torch.float32: 2}[mask.dtype]
    if dropout is not None:
        a.dropout_p, a.dropout_seed, a.dropout_offset = float(dropout[0]), int(dropout[1]), int(dropout[2])
    a.qkv, a.ld_qkv = _p(qkv), _rows2d(qkv, "qkv")
    a.N, a.L, a.heads, a.head_dim = N, L, heads, head_dim
    if mask is None:
        a.mask_dtype = 0
    elif cu_seqlens is None:
        assert mask.dim() == 2 and mask.shape[0] == N and mask.shape[1] >= L and mask.stride(1) == 1
        a.mask, a.mask_ld = _p(mask), mask.stride(0)
        a.mask_dtype = {torch.int64: 1, torch.float32: 2}[mask.dtype]
    a.causal, a.scale, a.mask_neg = int(causal), (float(head_dim) ** -0.5 if scale is None else float(scale)), float(mask_neg)
    return a


def _attn_kernel(L, head_dim, causal, direction):
    """short-sequence kernel for L <= 32, the CTA-per-(sequence, head) kernel for 32 < L <= 256 (ViT)"""
    lib = _l.get_lib()
    if L <= 32:
        return (lib.a4r_attn_small_fwd if direction == "fwd" else lib.a4r_attn_small_bwd), "a4r_attn_small_" + direction
    if L <= 256 and head_dim == 64 and not causal:
        return (lib.a4r_attn_mid_fwd if direction == "fwd" else lib.a4r_attn_mid_bwd), "a4r_attn_mid_" + direction
    raise RuntimeError("attention: unsupported shape L=%d head_dim=%d causal=%s (no fallback exists)" % (L, head_dim, causal))


def attn_small_fwd(qkv, N, L, heads, head_dim, mask=None, causal=False, mask_neg=F32_MIN, want_lse=False, dropout=None,
                   scale=None, cu_seqlens=None):
    """returns ctx, or (ctx, lse) with want_lse (lse is None for the short-sequence kernel, which recomputes it).
    cu_seqlens (int32 [N+1]): packed variable-length layout, L = the longest sequence (<= 32)."""
    assert qkv.dtype == BF16 and (cu_seqlens is not None or qkv.shape[0] == N * L)
    out = torch.empty((qkv.shape[0], heads * head_dim), dtype=BF16, device=qkv.device)
    a = _attn_args(qkv, N, L, heads, head_dim, mask, causal, mask_neg, dropout, scale, cu_seqlens)
    a.out, a.ld_out = _p(out), out.stride(0)
    lse = None
    if want_lse and L > 32:
        lse = torch.empty((N * L, heads), dtype=torch.float32, device=qkv.device)
        a.lse = _p(lse)
    fn, name = _attn_kernel(L, head_dim, causal, "fwd")
    _l.check(fn(ctypes.byref(a), _stream()), name)
    return (out, lse) if want_lse else out


def attn_small_bwd(qkv, dctx, N, L, heads, head_dim, mask=None, causal=False, mask_neg=F32_MIN, lse=None, ctx=None,
                   dropout=None, scale=None, cu_seqlens=None):
    assert qkv.dtype == BF16 and dctx.dtype == BF16 and dctx.shape[0] == qkv.shape[0]
    assert cu_seqlens is not None or qkv.shape[0] == N * L
    dqkv = torch.empty((qkv.shape[0], 3 * heads * head_dim), dtype=BF16, device=qkv.device)
    a = _attn_args(qkv, N, L, heads, head_dim, mask, causal, mask_neg, dropout, scale, cu_seqlens)
    assert _rows2d(qkv, "qkv") == dqkv.stride(0), "attention bwd expects a contiguous qkv"
    a.out, a.dout, a.ld_out = _p(dqkv), _p(dctx), _rows2d(dctx, "dctx")
    if L > 32:
        assert lse is not None and ctx is not None and ctx.is_contiguous() and dctx.is_contiguous()
        a.lse, a.ctx = _p(lse), _p(ctx)
    fn, name = _attn_kernel(L, head_dim, causal, "bwd")
    _l.check(fn(ctypes.byref(a), _stream()), name)
    return dqkv


def layernorm_fwd(x, gamma, beta, eps, res=None, want_z=False, want_stats=True):
    """y = LN(x + res[row % res_rows]); returns (y, z or None, mean or None, rstd or None)."""
    assert x.dtype == BF16 and x.is_contiguous() and x.dim() == 2
    M, H = x.shape
    y = torch.empty_like(x)
    z = torch.empty_like(x) if want_z else None
    mean = torch.empty(M, dtype=torch.float32, device=x.device) if want_stats else None
    rstd = torch.empty(M, dtype=torch.float32, device=x.device) if want_stats else None
    res_rows = 0
    if res is not None:
        assert res.dtype == BF16 and res.is_contiguous() and res.shape[-1] == H
        res_rows = res.numel() // H
    _l.check(_l.get_lib().a4r_layernorm_fwd(_p(x), _p(res), res_rows, _p(gamma), _p(beta), float(eps), _p(y), _p(z),
                                            _p(mean), _p(rstd), M, H, _stream()), "a4r_layernorm_fwd")
    return y, z, mean, rstd


def layernorm_bwd(dy, z, mean, rstd, gamma, dgamma=None, dbeta=None, accumulate=False, masked=None):
    """returns dz, or (dz, dz * dropout_mask / (1 - p)) when masked = (p, seed, offset)"""
    assert dy.dtype == BF16 and z.dtype == BF16 and dy.is_contiguous() and z.is_contiguous()
    M, H = z.shape
    dz = torch.empty_like(z)
    dzm = torch.empty_like(z) if masked is not None else None
    mp, mseed, moff = masked if masked is not None else (0.0, 0, 0)
    ws, wsb = None, 0
    if dgamma is not None:
        wsb = _l.get_lib().a4r_layernorm_bwd_workspace_bytes(H)
        ws = workspace(wsb, z.device)
    _l.check(_l.get_lib().a4r_layernorm_bwd(_p(dy), _p(z), _p(mean), _p(rstd), _p(gamma), _p(dz), _p(dgamma), _p(dbeta),
                                            int(accumulate), _p(ws), wsb, M, H, _p(dzm), float(mp), int(mseed), int(moff),
                                            _stream()), "a4r_layernorm_bwd")
    return (dz, dzm) if masked is not None else dz


def layernorm_bwd_add(dy, z, mean, rstd, gamma, dskip):
    """dz = LayerNorm-backward(dy) + dskip in one pass (pre-LN skip connections); frozen LayerNorm only"""
    assert dy.dtype == BF16 and z.dtype == BF16 and dskip.dtype == BF16
    assert dy.is_contiguous() and z.is_contiguous() and dskip.is_contiguous() and dskip.shape == z.shape
    M, H = z.shape
    dz = torch.empty_like(z)
    _l.check(_l.get_lib().a4r_layernorm_bwd_add(_p(dy), _p(z), _p(mean), _p(rstd), _p(gamma), _p(dskip), _p(dz), M, H,
                                                _stream()), "a4r_layernorm_bwd_add")
    return dz


def embed_ln_fwd(ids, L, word_emb, pos_emb, type_emb, gamma, beta, eps, pos_offset=0, roberta_pad_id=-1, prompt=None,
                 want_z=False):
    """ids: int64 [N, >=L] (row stride arbitrary); returns (out [N*L,H], z, mean, rstd)."""
    assert ids.dtype == torch.int64 and ids.dim() == 2 and ids.stride(1) == 1
    N, H = ids.shape[0], word_emb.shape[1]
    out = torch.empty((N * L, H), dtype=BF16, device=ids.device)
    z = torch.empty_like(out) if want_z else None
    mean = torch.empty(N * L, dtype=torch.float32, device=ids.device) if want_z else None
    rstd = torch.empty(N * L, dtype=torch.float32, device=ids.device) if want_z else None
    a = _l.EmbedArgs()
    a.ids, a.ld_ids = _p(ids), ids.stride(0)
    a.word_emb, a.pos_emb, a.type_emb, a.prompt = _p(word_emb), _p(pos_emb), _p(type_emb), _p(prompt)
    a.gamma, a.beta, a.out, a.z_out, a.mean_out, a.rstd_out = _p(gamma), _p(beta), _p(out), _p(z), _p(mean), _p(rstd)
    a.N, a.L, a.H, a.pos_offset, a.roberta_pad_id = N, L, H, pos_offset, roberta_pad_id
    a.n_prompt = 0 if prompt is None else prompt.shape[0]
    a.eps = float(eps)
    _l.check(_l.get_lib().a4r_embed_ln_fwd(ctypes.byref(a), _stream()), "a4r_embed_ln_fwd")
    return out, z, mean, rstd


def scatter_add_rows(src, idx, num_rows, skip_idx=-1):
    """f32 [num_rows, H] with out[idx[r]] += src[r] (bf16 src [R, H], int64 idx [R]); idx < 0 / == skip_idx skipped."""
    assert src.dtype == BF16 and src.dim() == 2 and src.stride(1) == 1 and idx.dtype == torch.int64
    idx = idx.contiguous().view(-1)
    assert idx.numel() == src.shape[0]
    out = torch.zeros((num_rows, src.shape[1]), dtype=torch.float32, device=src.device)
    _l.check(_l.get_lib().a4r_scatter_add_rows(_p(src), src.stride(0), _p(idx), _p(out), src.shape[0], src.shape[1],
                                               int(num_rows), int(skip_idx), _stream()), "a4r_scatter_add_rows")
    return out


ACT_KINDS = {"gelu": 0, "relu": 1, "leaky_relu": 2, "gelu_new": 3}


def act_bwd(dy, u, kind):
    """dy * act'(u): 'gelu' / 'gelu_new' (u = pre-activation) or 'relu' / 'leaky_relu' (u = activation output)."""
    assert dy.dtype == BF16 and u.dtype == BF16 and dy.is_contiguous() and u.is_contiguous() and dy.shape == u.shape
    out = torch.empty_like(dy)
    _l.check(_l.get_lib().a4r_act_bwd(_p(dy), _p(u), _p(out), dy.numel(), ACT_KINDS[kind], _stream()), "a4r_act_bwd")
    return out


def cast_transpose(w, want=True, want_t=False):
    """bf16 copy and / or bf16 transpose of an fp32 2-D weight in one kernel (the weight caches of functional.WeightCache)"""
    assert w.dtype == torch.float32 and w.dim() == 2 and w.stride(1) == 1
    rows, cols = w.shape
    out = torch.empty((rows, cols), dtype=BF16, device=w.device) if want else None
    out_t = torch.empty((cols, rows), dtype=BF16, device=w.device) if want_t else None
    _l.check(_l.get_lib().a4r_cast_transpose_f32_bf16(_p(w), w.stride(0), _p(out), _p(out_t), rows, cols, _stream()),
             "a4r_cast_transpose_f32_bf16")
    return out, out_t


def act_fwd(u, kind):
    """act(u) stand-alone (activations that have no GEMM-epilogue mode: leaky_relu, gelu_new)."""
    assert u.dtype == BF16 and u.is_contiguous()
    out = torch.empty_like(u)
    _l.check(_l.get_lib().a4r_act_fwd(_p(u), _p(out), u.numel(), ACT_KINDS[kind], _stream()), "a4r_act_fwd")
    return out


def colsum(x, width=None, out=None, accumulate=False):
    assert x.dtype == BF16 and x.dim() == 2
    M = x.shape[0]
    width = x.shape[1] if width is None else width
    if out is None and width == x.shape[1] and width <= 128 and x.is_contiguous() and M >= 4096:
        # narrow matrices (rank-r bottleneck gradients): a row is one or two 128-byte lines, so the row-per-step kernel
        # idles most of a warp; fold f rows into one (a contiguous reshape) and add the f partial sums afterwards
        f = 16
        while f > 1 and M % f:
            f //= 2
        if f > 1:
            return colsum(x.view(M // f, f * width)).view(f, width).sum(0)
    if out is None:
        out = torch.empty(width, dtype=torch.float32, device=x.device)
        accumulate = False
    wsb = _l.get_lib().a4r_colsum_workspace_bytes(width)
    ws = workspace(wsb, x.device)
    _l.check(_l.get_lib().a4r_colsum(_p(x), _rows2d(x, "x"), M, width, _p(out), int(accumulate), _p(ws), wsb, _stream()),
             "a4r_colsum")
    return out


def wgrad_mma_sync(a, b, alpha=1.0, out=None, accumulate=False, n=None, k=None):
    """dW[N,K] (+)= alpha * a[:, :N].T @ b[:, :K]   (a = dY [M,>=N], b = X [M,>=K]; fp32 result) on the round-1
    mma.sync split-M kernel (a4r_wgrad_bf16).  Kept as an ABI entry point and as the cross-check of the tcgen05 kernel
    in the tests; the product path (`wgrad` below) is the tcgen05 kernel."""
    assert a.dtype == BF16 and b.dtype == BF16 and a.shape[0] == b.shape[0]
    M = a.shape[0]
    N = a.shape[1] if n is None else n
    K = b.shape[1] if k is None else k
    if out is None:
        out = torch.empty((N, K), dtype=torch.float32, device=a.device)
        accumulate = False
    assert out.dtype == torch.float32 and tuple(out.shape) == (N, K) and out.stride(1) == 1
    wsb = _l.get_lib().a4r_wgrad_workspace_bytes(M, N, K)
    ws = workspace(wsb, a.device)
    _l.check(_l.get_lib().a4r_wgrad_bf16(_p(a), _rows2d(a, "a"), _p(b), _rows2d(b, "b"), _p(out), out.stride(0), M, N, K,
                                         float(alpha), int(accumulate), _p(ws), wsb, _stream()), "a4r_wgrad_bf16")
    return out


def wgrad_tc(a, b, alpha=1.0, out=None, accumulate=False, n=None, k=None):
    """dW[N,K] (+)= alpha * a[:, :N].T @ b[:, :K] on tcgen05 (MN-major operands, split over tokens, fp32 result)."""
    assert a.dtype == BF16 and b.dtype == BF16 and a.shape[0] == b.shape[0]
    M = a.shape[0]
    N = a.shape[1] if n is None else n
    K = b.shape[1] if k is None else k
    if out is None:
        out = torch.empty((N, K), dtype=torch.float32, device=a.device)
        accumulate = False
    assert out.dtype == torch.float32 and tuple(out.shape) == (N, K) and out.stride(1) == 1
    wsb = _l.get_lib().a4r_wgrad_tc_workspace_bytes(M, N, K)
    ws = workspace(wsb, a.device)
    _l.check(_l.get_lib().a4r_wgrad_tc_bf16(_p(a), _rows2d(a, "a"), _p(b), _rows2d(b, "b"), _p(out), out.stride(0), M, N, K,
                                            float(alpha), int(accumulate), _p(ws), wsb, _stream()), "a4r_wgrad_tc_bf16")
    return out


wgrad = wgrad_tc   # every weight gradient of the path: 2-5x faster than the mma.sync kernel at every shape measured


def _bce_args(prec, emb, log_mask, pos, neg, loss, count, cpc):
    B, S, D = prec.shape
    assert prec.dtype == BF16 and emb.dtype == BF16 and prec.is_contiguous() and emb.is_contiguous()
    assert emb.numel() == B * (S + 1) * 2 * D
    a = _l.BceArgs()
    a.prec, a.emb, a.log_mask = _p(prec), _p(emb), _p(log_mask)
    a.pos_score, a.neg_score, a.loss, a.count = _p(pos), _p(neg), _p(loss), _p(count)
    a.B, a.S, a.D, a.cpc = B, S, D, int(cpc)
    return a


def bce_loss_fwd(prec, emb, log_mask, cpc=False):
    """returns (loss [1] f32, count [1] f32, pos_score [B,S], neg_score [B,S])."""
    B, S, _ = prec.shape
    dev = prec.device
    pos = torch.empty((B, S), dtype=torch.float32, device=dev)
    neg = torch.empty((B, S), dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    count = torch.empty(1, dtype=torch.float32, device=dev)
    if log_mask is not None:
        assert log_mask.dtype == torch.float32 and log_mask.is_contiguous() and tuple(log_mask.shape) == (B, S)
    a = _bce_args(prec, emb, log_mask, pos, neg, loss, count, cpc)
    wsb = _l.get_lib().a4r_bce_workspace_bytes()
    ws = workspace(wsb, dev)
    _l.check(_l.get_lib().a4r_bce_loss_fwd(ctypes.byref(a), _p(ws), wsb, _stream()), "a4r_bce_loss_fwd")
    return loss, count, pos, neg


def bce_loss_bwd(prec, emb, log_mask, pos, neg, count, grad_out=None, cpc=False):
    d_prec = torch.empty_like(prec)
    d_emb = torch.empty_like(emb)
    loss = torch.empty(1, dtype=torch.float32, device=prec.device)
    a = _bce_args(prec, emb, log_mask, pos, neg, loss, count, cpc)
    if grad_out is not None:
        assert grad_out.dtype == torch.float32 and grad_out.numel() == 1
    _l.check(_l.get_lib().a4r_bce_loss_bwd(ctypes.byref(a), _p(grad_out), _p(d_prec), _p(d_emb), _stream()),
             "a4r_bce_loss_bwd")
    return d_prec, d_emb


def adapter_ln_supported(H, r):
    return bool(_l.get_lib().a4r_adapter_ln_supported(int(H), int(r)))


def adapter_ln_fwd(h, inp, w_down, b_down, w_up, b_up, gamma=None, beta=None, eps=0.0, act="relu", tail=0, save=False,
                   impl=0):
    """K5 in one kernel: out = tail(h + W_u act(W_d h + b_d) + b_u [+ inp]); tail 0 = LayerNorm, 1 = +inp, 2 = nothing.
    returns (out, z, mean, rstd, s, u): with save=True the tensors the backward reads (z/mean/rstd for tail 0, s always,
    u = pre-activation for GELU), else None.  s is a [M, r] VIEW of a [M, r + 16] buffer (32-byte aligned rows) whose column r holds ones
    (s_ext(s) returns it): dzᵀ · [s | 1] is d(fc_up.weight) and d(fc_up.bias) in one weight-gradient GEMM."""
    assert h.dtype == BF16 and h.dim() == 2 and w_down.dtype == BF16 and w_up.dtype == BF16
    assert w_down.is_contiguous() and w_up.is_contiguous()
    M, H = h.shape
    r = w_down.shape[0]
    assert tuple(w_down.shape) == (r, H) and tuple(w_up.shape) == (H, r)
    for t in (b_down, b_up) + ((gamma, beta) if tail == 0 else ()):
        assert t.dtype == torch.float32 and t.is_contiguous()
    dev = h.device
    out = torch.empty((M, H), dtype=BF16, device=dev)
    z = mean = rstd = s = u = None
    if save:
        s = torch.empty((M, r + 16), dtype=BF16, device=dev)[:, :r]
        if act == "gelu":
            u = torch.empty((M, r), dtype=BF16, device=dev)
        if tail == 0:
            z = torch.empty((M, H), dtype=BF16, device=dev)
            mean = torch.empty(M, dtype=torch.float32, device=dev)
            rstd = torch.empty(M, dtype=torch.float32, device=dev)
    a = _l.AdapterArgs()
    a.h, a.ldh = _p(h), _rows2d(h, "h")
    if inp is not None:
        assert inp.dtype == BF16 and tuple(inp.shape) == (M, H)
        a.input, a.ldi = _p(inp), _rows2d(inp, "input")
    a.w_down, a.b_down, a.w_up, a.b_up = _p(w_down), _p(b_down), _p(w_up), _p(b_up)
    a.gamma, a.beta, a.out, a.z_out, a.mean, a.rstd, a.s_out, a.u_out = (_p(gamma), _p(beta), _p(out), _p(z), _p(mean),
                                                                         _p(rstd), _p(s), _p(u))
    a.M, a.H, a.r, a.act, a.tail, a.eps = M, H, r, {"relu": 0, "gelu": 1}[act], int(tail), float(eps)
    a.lds = 0 if s is None else s.stride(0)
    a.impl = int(impl)       # 0 = default, 2 = staged kernel, 3 = row-per-thread kernel (include/adapter4rec.h)
    _l.check(_l.get_lib().a4r_adapter_ln_fwd(ctypes.byref(a), _stream()), "a4r_adapter_ln_fwd")
    return out, z, mean, rstd, s, u


def s_ext(s):
    """[s | 1 0 .. 0]: the [M, r + 8] window of the padded buffer behind the s view that adapter_ln_fwd returned"""
    M, r = s.shape
    assert s.stride(0) == r + 16 and s.storage_offset() == 0
    return s.as_strided((M, r + 8), (r + 16, 1))


MASKED_LOGIT = -1e4  # the constant the in-batch softmax head writes over excluded candidates


def _inbatch_args(prec, emb, item_ids, log_mask, cand_bias, lse, loss, count):
    B, S, D = prec.shape
    assert prec.dtype == BF16 and emb.dtype == BF16 and prec.is_contiguous() and emb.is_contiguous()
    assert emb.numel() == B * (S + 1) * 2 * D, "emb must be Model.forward's encoder output [B, S+1, 2, D]"
    assert item_ids.dtype == torch.int64 and item_ids.is_contiguous() and tuple(item_ids.shape) == (B, S + 1)
    assert log_mask.dtype == torch.float32 and log_mask.is_contiguous() and tuple(log_mask.shape) == (B, S)
    if cand_bias is not None:
        assert cand_bias.dtype == torch.float32 and cand_bias.is_contiguous() and cand_bias.numel() == B * (S + 1)
    a = _l.InbatchCeArgs()
    a.prec, a.cand, a.ld_cand = _p(prec), _p(emb), 2 * D     # candidate c = history slot (b, j) = emb[b, j, 0, :]
    a.item_ids, a.log_mask, a.cand_bias = _p(item_ids), _p(log_mask), _p(cand_bias)
    a.lse, a.loss, a.count = _p(lse), _p(loss), _p(count)
    a.B, a.S, a.D, a.masked_logit = B, S, D, MASKED_LOGIT
    return a


def inbatch_ce_fwd(prec, emb, item_ids, log_mask, cand_bias=None):
    """returns (loss [1] f32, count [1] f32, lse [B*S] f32) — see a4r_inbatch_ce_fwd in include/adapter4rec.h."""
    B, S, _ = prec.shape
    dev = prec.device
    lse = torch.empty(B * S, dtype=torch.float32, device=dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    count = torch.empty(1, dtype=torch.float32, device=dev)
    a = _inbatch_args(prec, emb, item_ids, log_mask, cand_bias, lse, loss, count)
    wsb = _l.get_lib().a4r_inbatch_ce_workspace_bytes(B, S)
    ws = workspace(wsb, dev)
    _l.check(_l.get_lib().a4r_inbatch_ce_fwd(ctypes.byref(a), _p(ws), wsb, _stream()), "a4r_inbatch_ce_fwd")
    return loss, count, lse


def inbatch_ce_bwd(prec, emb, item_ids, log_mask, lse, count, cand_bias=None, grad_out=None):
    """returns (d_prec [B,S,D], d_emb [B,S+1,2,D]); the sampled-negative half of d_emb is zero (this head ignores it)."""
    d_prec = torch.empty_like(prec)
    d_emb = torch.zeros_like(emb)
    loss = torch.empty(1, dtype=torch.float32, device=prec.device)
    a = _inbatch_args(prec, emb, item_ids, log_mask, cand_bias, lse, loss, count)
    if grad_out is not None:
        assert grad_out.dtype == torch.float32 and grad_out.numel() == 1
    _l.check(_l.get_lib().a4r_inbatch_ce_bwd(ctypes.byref(a), _p(grad_out), _p(d_prec), _p(d_emb), 2 * prec.shape[2],
                                             _stream()), "a4r_inbatch_ce_bwd")
    return d_prec, d_emb


def adam_step(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
    for t in (p, g, m, v):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    _l.check(_l.get_lib().a4r_adam_step(_p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
                                        float(eps), float(weight_decay), int(step), float(grad_scale), _stream()),
             "a4r_adam_step")


def adam_step_dev(p, g, m, v, lr, beta1, beta2, eps, weight_decay, bias_corr, grad_scale=1.0):
    """adam_step with (1 - beta1^t, sqrt(1 - beta2^t)) read from the device tensor bias_corr (f32 [2]): the form a CUDA-graph
    replay needs, bit-identical to adam_step for the same t."""
    for t in (p, g, m, v):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    assert bias_corr.dtype == torch.float32 and bias_corr.numel() == 2 and bias_corr.is_cuda
    _l.check(_l.get_lib().a4r_adam_step_dev(_p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2),
                                            float(eps), float(weight_decay), _p(bias_corr), float(grad_scale), _stream()),
             "a4r_adam_step_dev")


def adam_bias_corrections(beta1, beta2, step):
    """the two factors a4r_adam_step derives from the step number (in double, as the library does)"""
    import math
    import struct
    b1, b2 = (struct.unpack("f", struct.pack("f", float(b)))[0] for b in (beta1, beta2))   # the ABI takes the betas as float
    return 1.0 - math.pow(b1, int(step)), math.sqrt(1.0 - math.pow(b2, int(step)))


def gather_rows(table, ids):
    """out[..., :] = table[ids[...], :]  (bf16 table [R, D], int64 ids of any shape)."""
    assert table.dtype == BF16 and table.is_contiguous() and ids.dtype == torch.int64
    ids_c = ids.contiguous()
    out = torch.empty(tuple(ids.shape) + (table.shape[1],), dtype=BF16, device=table.device)
    _l.check(_l.get_lib().a4r_gather_rows(_p(table), _p(ids_c), _p(out), ids_c.numel(), table.shape[1], _stream()),
             "a4r_gather_rows")
    return out


def sample_train_batch(seqs, item_content, item_num, seed, offset, neg_in=None):
    """seqs int64 [B, S1] (left-padded ids), item_content int64 [I+1, W] -> (sample_items [B, S1, 2, W] int64,
    log_mask [B, S1-1] f32, neg ids [B, S1] int64, fail flag [1] int32 — left on the device, no sync here).
    item_content None: ids-only mode, sample_items is None (the id tower's sample is stack([seqs, neg], -1))."""
    assert seqs.dtype == torch.int64 and seqs.is_contiguous() and seqs.dim() == 2
    B, S1 = seqs.shape
    dev = seqs.device
    if item_content is None:
        W, out = 0, None
    else:
        assert item_content.dtype == torch.int64 and item_content.is_contiguous() and item_content.dim() == 2
        W = item_content.shape[1]
        out = torch.empty((B, S1, 2, W), dtype=torch.int64, device=dev)
    log_mask = torch.empty((B, S1 - 1), dtype=torch.float32, device=dev)
    neg = torch.empty((B, S1), dtype=torch.int64, device=dev)
    fail = torch.zeros(1, dtype=torch.int32, device=dev)
    if neg_in is not None:
        assert neg_in.dtype == torch.int64 and neg_in.is_contiguous() and neg_in.shape == seqs.shape
    _l.check(_l.get_lib().a4r_sample_train_batch(_p(seqs), _p(item_content), _p(neg_in), _p(out), _p(log_mask), _p(neg),
                                                 _p(fail), B, S1, W, int(item_num), int(seed) & (2 ** 64 - 1),
                                                 int(offset) & (2 ** 64 - 1), _stream()), "a4r_sample_train_batch")
    return out, log_mask, neg, fail


def id_embed_fwd(table, ids, want_hist=True):
    """table f32 [V, D] (the fp32 master), ids int64 [B, S1, 2] -> (emb bf16 [B, S1, 2, D], hist bf16 [B, S1-1, D] or
    None): bf16_rne(table[ids]) and its history slots, in one pass."""
    assert table.dtype == torch.float32 and table.dim() == 2 and table.is_contiguous()
    assert ids.dtype == torch.int64 and ids.dim() == 3 and ids.shape[2] == 2 and ids.is_contiguous()
    B, S1, _ = ids.shape
    V, D = table.shape
    emb = torch.empty((B, S1, 2, D), dtype=BF16, device=table.device)
    hist = torch.empty((B, S1 - 1, D), dtype=BF16, device=table.device) if want_hist else None
    _l.check(_l.get_lib().a4r_id_embed_fwd(_p(table), V, D, _p(ids), B, S1, _p(emb), _p(hist), _stream()),
             "a4r_id_embed_fwd")
    return emb, hist


def id_embed_bwd(ids, d_emb, d_hist, grad, padding_idx=0, accumulate=True):
    """grad f32 [V, D] (+)= the table gradient of id_embed_fwd's two outputs (d_hist may be None), summed per row in fp32 in
    ascending occurrence order.  The occurrences are grouped by a stable device sort of the ids (no host sync)."""
    assert ids.dtype == torch.int64 and ids.dim() == 3 and ids.shape[2] == 2 and ids.is_contiguous()
    B, S1, _ = ids.shape
    V, D = grad.shape
    assert grad.dtype == torch.float32 and grad.is_contiguous()
    assert d_emb.dtype == BF16 and d_emb.is_contiguous() and d_emb.numel() == B * S1 * 2 * D
    if d_hist is not None:
        assert d_hist.dtype == BF16 and d_hist.is_contiguous() and d_hist.numel() == B * (S1 - 1) * D
    sorted_ids, order = torch.sort(ids.view(-1), stable=True)
    _l.check(_l.get_lib().a4r_id_embed_bwd(_p(sorted_ids), _p(order), _p(d_emb), _p(d_hist), _p(grad), V, D, B, S1,
                                           int(padding_idx), int(bool(accumulate)), _stream()), "a4r_id_embed_bwd")
    return grad


def score_topk(users, items, id_base=0, history=None, k=10):
    """Partial top-k lists of users @ items.T over one item shard: returns (scores [P,U,k] f32, ids [P,U,k] i32)."""
    assert users.dtype == BF16 and items.dtype == BF16 and users.shape[1] == items.shape[1]
    U, d = users.shape
    I = items.shape[0]
    P = _l.get_lib().a4r_score_topk_partials(U, I)
    sc = torch.empty((P, U, k), dtype=torch.float32, device=users.device)
    ids = torch.empty((P, U, k), dtype=torch.int32, device=users.device)
    hl = 0
    if history is not None:
        assert history.dtype == torch.int32 and history.is_contiguous() and history.shape[0] == U
        hl = history.shape[1]
    _l.check(_l.get_lib().a4r_score_topk(_p(users), _rows2d(users, "users"), _p(items), _rows2d(items, "items"), U, I, d,
                                         int(id_base), _p(history), hl, int(k), _p(sc), _p(ids), _stream()),
             "a4r_score_topk")
    return sc, ids


def topk_merge(scores, ids, target=None):
    """Merge [P,U,k] partial lists -> (scores [U,k], ids [U,k], hit [U] or None, ndcg [U] or None)."""
    P, U, k = scores.shape
    assert scores.dtype == torch.float32 and ids.dtype == torch.int32 and scores.is_contiguous() and ids.is_contiguous()
    osc = torch.empty((U, k), dtype=torch.float32, device=scores.device)
    oid = torch.empty((U, k), dtype=torch.int32, device=scores.device)
    hit = ndcg = None
    if target is not None:
        assert target.dtype == torch.int32 and target.numel() == U and target.is_contiguous()
        hit = torch.empty(U, dtype=torch.float32, device=scores.device)
        ndcg = torch.empty(U, dtype=torch.float32, device=scores.device)
    _l.check(_l.get_lib().a4r_topk_merge(_p(scores), _p(ids), P, U, k, _p(osc), _p(oid), _p(target), _p(hit), _p(ndcg),
                                         _stream()), "a4r_topk_merge")
    return osc, oid, hit, ndcg


def patchify(images, patch_size):
    """[N,C,R,R] f32 -> [N*P, C*ps*ps] bf16 (im2col of the non-overlapping patch convolution)."""
    assert images.dtype == torch.float32 and images.is_contiguous() and images.dim() == 4 and images.shape[2] == images.shape[3]
    N, C, R, _ = images.shape
    P = (R // patch_size) ** 2
    out = torch.empty((N * P, C * patch_size * patch_size), dtype=BF16, device=images.device)
    _l.check(_l.get_lib().a4r_patchify(_p(images), _p(out), N, C, R, patch_size, _stream()), "a4r_patchify")
    return out


def vit_assemble(patch_emb, cls, pos, prompt, N, P):
    """[cls + pos[0] | patch_emb + pos[1..P] | prompt] -> [N*(1+P+T), H] bf16."""
    H = patch_emb.shape[1]
    T = 0 if prompt is None else prompt.shape[0]
    for t in (patch_emb, cls, pos) + ((prompt,) if prompt is not None else ()):
        assert t.dtype == BF16 and t.is_contiguous()
    out = torch.empty((N * (1 + P + T), H), dtype=BF16, device=patch_emb.device)
    _l.check(_l.get_lib().a4r_vit_assemble(_p(patch_emb), _p(cls), _p(pos), _p(prompt), _p(out), N, P, T, H, _stream()),
             "a4r_vit_assemble")
    return out
