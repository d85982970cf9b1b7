"""Leaf modules with the parameter names of torch.nn / loralib (so reference checkpoints load unchanged) whose
forward runs on the sm_100a kernels."""
import math

import torch
import torch.nn as nn

from .. import functional as Fn

BF16 = torch.bfloat16


def to_2d_bf16(x):
    x2 = x.reshape(-1, x.shape[-1])
    return x2 if x2.dtype == BF16 else x2.to(BF16)


def frozen_ffn_dense(intermediate, output):
    """The output dense Linear of a transformer layer's feed-forward pair (intermediate -> GELU -> output.dense) when
    both Linears are frozen, else None.  `output` may be an adapter wrapper that keeps the original module as
    `self_output`."""
    dense = getattr(getattr(output, "self_output", output), "dense", None)
    if dense is None or any(t.requires_grad for t in (intermediate.weight, intermediate.bias, dense.weight, dense.bias)):
        return None
    return dense


class Linear(nn.Module):
    """nn.Linear replacement: parameters `weight` [out,in], `bias` [out] (fp32 masters), tcgen05 GEMM forward."""

    def __init__(self, in_features, out_features, bias=True):
        super().__init__()
        self.in_features, self.out_features = in_features, out_features
        self.weight = nn.Parameter(torch.empty(out_features, in_features))
        self.bias = nn.Parameter(torch.empty(out_features)) if bias else None
        self.reset_parameters()
        self._cache = Fn.WeightCache()

    def reset_parameters(self):
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            bound = 1 / math.sqrt(self.in_features)
            nn.init.uniform_(self.bias, -bound, bound)

    def forward(self, x, act=None, residual=None, residual2=None):
        shape = x.shape
        y = Fn.linear(to_2d_bf16(x), self.weight, self.bias, self._cache, act=act, residual=residual, residual2=residual2)
        return y.view(*shape[:-1], self.out_features)

    def extra_repr(self):
        return "in_features=%d, out_features=%d, bias=%s" % (self.in_features, self.out_features, self.bias is not None)


class LoRALinear(Linear):
    """loralib 0.1.1 `Linear` as the reference constructs it (Downstream/Text/run.py:418-428:
    lora.Linear(in, out, r=r)): a NEW linear whose `weight` is re-initialised and frozen, whose `bias` is new and
    trainable, plus lora_A [r,in] (kaiming-uniform, a=sqrt(5)) and lora_B [out,r] (zeros); lora_alpha = 1, so
    scaling = 1/r; no dropout; never merged by the reference's train/eval loop (SURVEY.md Appendix B-3)."""

    def __init__(self, in_features, out_features, r=0, lora_alpha=1, bias=True, **kwargs):
        super().__init__(in_features, out_features, bias=bias)
        self.r, self.lora_alpha = r, lora_alpha
        if r > 0:
            self.lora_A = nn.Parameter(self.weight.new_zeros((r, in_features)))
            self.lora_B = nn.Parameter(self.weight.new_zeros((out_features, r)))
            self.scaling = lora_alpha / r
            self.weight.requires_grad = False
            nn.init.kaiming_uniform_(self.lora_A, a=math.sqrt(5))
            nn.init.zeros_(self.lora_B)
        self._qkv_cache = Fn.QKVCache()

    def forward(self, x, act=None, residual=None, residual2=None):
        if self.r == 0:
            return super().forward(x, act=act, residual=residual, residual2=residual2)
        assert act is None and residual is None and residual2 is None
        assert self.lora_alpha == 1, "only the reference's lora_alpha = 1 is implemented"
        shape = x.shape
        # stand-alone use: run the fused-projection function with a single slot
        y = Fn.qkv(to_2d_bf16(x), (self,), self._qkv_cache)
        return y.view(*shape[:-1], self.out_features)


class PHMLinear(nn.Module):
    """Parameterised hypercomplex multiplication layer as HyperComplexAdapterBlock configures it
    (Downstream/Text/model/layers.py:25-166 with shared_phm_rule=True, factorized_phm=True, phm_rank=1, bias=True,
    w_init="glorot-uniform"; modules.py:218-245): y = x·H + b with H = Σ_i phm_rule[i] ⊗ (W_left[i]·W_right[i])
    ([in, out], rebuilt every forward, kronecker.py:23-34).  Parameter names: W_left [n, in/n, 1], W_right
    [n, 1, out/n], b [out]; `phm_rule` [n, n, n] is the single tensor shared by every PHMLinear of the model, assigned by
    CompacterModel through set_phm_rule (run.py:70-81) — being an nn.Parameter it is registered here too, so the
    reference's state_dict repeats it under every layer.

    H has in·out <= 768·64 elements, i.e. it is parameter-space work independent of the batch: it is synthesised with
    torch tensor ops on the device (autograd carries dH back to W_left / W_right / phm_rule); every per-token
    operation — the projection, bias, activation, the data gradient and dH = xᵀ·dy — runs in the sm_100a kernels."""

    def __init__(self, in_features, out_features, phm_dim, bias=True, phm_rank=1, **unused):
        super().__init__()
        assert in_features % phm_dim == 0, "Argument `in_features`=%d is not divisble be `phm_dim`%d" % (in_features, phm_dim)
        assert out_features % phm_dim == 0, "Argument `out_features`=%d is not divisble be `phm_dim`%d" % (out_features, phm_dim)
        self.in_features, self.out_features, self.phm_dim, self.phm_rank = in_features, out_features, phm_dim, phm_rank
        self.W_left = nn.Parameter(torch.empty(phm_dim, in_features // phm_dim, phm_rank))
        self.W_right = nn.Parameter(torch.empty(phm_dim, phm_rank, out_features // phm_dim))
        self.b = nn.Parameter(torch.zeros(out_features)) if bias else None
        for i in range(phm_dim):                                   # glorot_uniform, inits.py:10-11
            nn.init.xavier_uniform_(self.W_left.data[i], gain=math.sqrt(2))
            nn.init.xavier_uniform_(self.W_right.data[i], gain=math.sqrt(2))

    def set_phm_rule(self, phm_rule=None, phm_rule_left=None, phm_rule_right=None):
        self.phm_rule = phm_rule

    def weight(self):
        """H transposed to the [out, in] layout of nn.Linear.weight (fp32, differentiable)."""
        n = self.phm_dim
        W = torch.bmm(self.W_left, self.W_right)                                        # [n, in/n, out/n]
        H = torch.einsum('bac,bkp->akcp', self.phm_rule, W).reshape(self.in_features, self.out_features)
        return H.t().contiguous()

    def forward(self, x, act=None, residual=None):
        shape = x.shape
        y = Fn.linear(to_2d_bf16(x), self.weight(), self.b, Fn.WeightCache(), act=act, residual=residual)
        return y.view(*shape[:-1], self.out_features)


class LayerNorm(nn.Module):
    def __init__(self, normalized_shape, eps=1e-5):
        super().__init__()
        n = normalized_shape if isinstance(normalized_shape, int) else normalized_shape[-1]
        self.normalized_shape, self.eps = (n,), eps
        self.weight = nn.Parameter(torch.ones(n))
        self.bias = nn.Parameter(torch.zeros(n))

    def forward(self, x, res=None, res_param=None):
        shape = x.shape
        return Fn.layer_norm(to_2d_bf16(x), self.weight, self.bias, self.eps, res=res, res_param=res_param).view(shape)

    def forward_skip(self, x2d):
        """(LN(x), x') for pre-LN blocks: use x' as the skip input so its gradient is added inside the LN-backward kernel"""
        if not (x2d.requires_grad and x2d.is_contiguous()):
            return self.forward(x2d), x2d
        return Fn.layer_norm_skip(x2d, self.weight, self.bias, self.eps)


class Embedding(nn.Module):
    """A frozen lookup table (`weight` [V,H]); gathers happen inside the fused embedding kernel."""

    def __init__(self, num_embeddings, embedding_dim, padding_idx=None):
        super().__init__()
        self.num_embeddings, self.embedding_dim, self.padding_idx = num_embeddings, embedding_dim, padding_idx
        self.weight = nn.Parameter(torch.empty(num_embeddings, embedding_dim))
        nn.init.normal_(self.weight)
        self._cache = Fn.WeightCache()

    def table_bf16(self):
        return self._cache.get(self.weight)[0]


class IdEmbedding(nn.Module):
    """The id item tower's table: nn.Embedding(num_embeddings, embedding_dim, padding_idx=0) with the parameter name
    `weight` [V, D] (fp32 master, xavier_normal_ as the reference initialises id_embedding; row padding_idx is zero and is
    never written by the backward).  forward(ids [B, S1, 2] int64) -> (emb bf16 [B, S1, 2, D], hist bf16 [B, S1-1, D]):
    the lookup and the user-encoder input in one kernel (Fn.IdEmbeddingFunction)."""

    def __init__(self, num_embeddings, embedding_dim, padding_idx=0):
        super().__init__()
        self.num_embeddings, self.embedding_dim, self.padding_idx = num_embeddings, embedding_dim, padding_idx
        self.weight = nn.Parameter(torch.empty(num_embeddings, embedding_dim))
        nn.init.xavier_normal_(self.weight)
        with torch.no_grad():
            self.weight[padding_idx].zero_()

    def forward(self, ids):
        ids = ids.to(device=self.weight.device, dtype=torch.int64).contiguous()
        return Fn.id_embedding(ids, self.weight, self.padding_idx)

    def extra_repr(self):
        return "%d, %d, padding_idx=%d" % (self.num_embeddings, self.embedding_dim, self.padding_idx)
