"""SASRec user-encoder building blocks and the adapter bottleneck, mirroring Downstream/Text/model/modules.py
(class names, constructor signatures, attribute and parameter names), running on the sm_100a kernels."""
import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .layers import BF16, Embedding, LayerNorm, Linear, PHMLinear, to_2d_bf16

SASREC_MASK_NEG = -1e9   # encoders.py:28


class PositionwiseFeedForward(nn.Module):
    """modules.py:16-28: LayerNorm(x + w_2(relu(w_1(x)))), eps 1e-6."""

    def __init__(self, d_model, d_inner, dropout):
        super().__init__()
        self.w_1 = Linear(d_model, d_inner)
        self.w_2 = Linear(d_inner, d_model)
        self.layer_norm = LayerNorm(d_model, eps=1e-6)
        self.dropout = nn.Dropout(dropout)
        self.activate = nn.ReLU()

    def presum(self, x2, adapter=None, extra=None):
        """x2 + dropout(w_2(relu(w_1 x2))) (+ extra) — the argument of the block's LayerNorm.  `adapter` (serial
        Houlsby) is applied to the dropped-out FFN output before the skip connection; `extra` (parallel Houlsby) is a
        second summand that already contains what the caller wants added."""
        h = self.w_1(x2, act="relu")
        p = self.dropout.p if self.training else 0.0
        res = x2.contiguous() if extra is None else extra
        if adapter is None:
            if p > 0:
                z = Fn.dropout_add(self.w_2(h), res, p)
                return z
            return self.w_2(h, residual=res)
        assert extra is None
        o = self.w_2(h)
        return adapter(Fn.dropout_add(o, None, p) if p > 0 else o, extra_residual=x2)

    def forward(self, x, adapter=None):
        return self.layer_norm(self.presum(to_2d_bf16(x), adapter)).view(x.shape)


class SelfAttention(nn.Module):
    """modules.py:31-42; the arithmetic runs inside the fused attention kernel."""

    def __init__(self, temperature, dropout):
        super().__init__()
        self.temperature = temperature
        self.dropout = nn.Dropout(dropout)


class MultiHeadedAttention(nn.Module):
    """modules.py:45-74: bias-free w_Q/w_K/w_V/fc (w_Q / w_V may be swapped for loralib Linears), LayerNorm eps 1e-6."""

    def __init__(self, n_heads, d_model, dropout):
        super().__init__()
        assert d_model % n_heads == 0
        self.d_model, self.d_k, self.n_heads = d_model, d_model // n_heads, n_heads
        self.d_v = self.d_k
        self.w_Q = Linear(d_model, n_heads * self.d_k, bias=False)
        self.w_K = Linear(d_model, n_heads * self.d_k, bias=False)
        self.w_V = Linear(d_model, n_heads * self.d_v, bias=False)
        self.fc = Linear(n_heads * self.d_v, d_model, bias=False)
        self.self_attention = SelfAttention(temperature=self.d_k ** 0.5, dropout=dropout)
        self.dropout = nn.Dropout(p=dropout)
        self.layer_norm = LayerNorm(d_model, eps=1e-6)
        self._qkv_cache = Fn.QKVCache()

    def presum(self, x2, mask, B, S, adapter=None, extra=None):
        """x2 + dropout(fc(attention(x2))) (+ extra) — the argument of the block's LayerNorm (see
        PositionwiseFeedForward.presum for `adapter` / `extra`)."""
        qkv = Fn.qkv(x2, (self.w_Q, self.w_K, self.w_V), self._qkv_cache)
        pd = self.self_attention.dropout.p if self.training else 0.0
        w = self.kernel_width(self.d_k)
        if w == self.d_k:
            ctx = Fn.attention(qkv, mask, B, S, self.n_heads, self.d_k, causal=self.causal, mask_neg=SASREC_MASK_NEG,
                               dropout_p=pd)
        else:
            # other widths (the K-adapter inside SASRec: d = 16, 2 heads -> d_k = 8; D = 192 with 4 heads -> 48): every
            # head is zero-padded to the next width the attention kernel handles (q·k and p·v are unchanged by zero
            # columns) with the softmax temperature of the TRUE head width; pad / slice are pure data movement
            h3 = 3 * self.n_heads
            qp = torch.nn.functional.pad(qkv.view(-1, h3, self.d_k), (0, w - self.d_k)).reshape(-1, h3 * w)
            cp = Fn.attention(qp, mask, B, S, self.n_heads, w, causal=self.causal, mask_neg=SASREC_MASK_NEG,
                              dropout_p=pd, scale=self.d_k ** -0.5)
            ctx = cp.view(-1, self.n_heads, w)[:, :, :self.d_k].reshape(-1, self.n_heads * self.d_k)
        p = self.dropout.p if self.training else 0.0
        res = x2.contiguous() if extra is None else extra
        if adapter is None:
            return Fn.dropout_add(self.fc(ctx), res, p) if p > 0 else self.fc(ctx, residual=res)
        assert extra is None
        o = self.fc(ctx)
        return adapter(Fn.dropout_add(o, None, p) if p > 0 else o, extra_residual=x2)

    KERNEL_WIDTHS = (32, 64, 128)   # head widths the short-sequence attention kernel runs natively

    @classmethod
    def kernel_width(cls, d_k):
        """the kernel width a d_k-wide head runs at: d_k itself if native, else the next native width (zero-padded)"""
        for w in cls.KERNEL_WIDTHS:
            if d_k <= w:
                return w
        raise AssertionError("head width %d: the attention kernel supports head widths up to 128 (natively 32, 64 and "
                             "128; narrower heads are zero-padded to the next of these)" % d_k)

    causal = True    # User_Encoder's mask (encoders.py:24-28); KAdapterBlock runs the same block with an all-ones mask

    def forward(self, query, key, value, mask, adapter=None):
        """query is key is value = block input [B,S,D]; mask = the [B,S] float log_mask (non-zero = valid key); the
        causal structure of User_Encoder.forward's additive mask is applied inside the kernel."""
        assert query is key and key is value, "SASRec self-attention only"
        B, S, D = query.shape
        z = self.presum(to_2d_bf16(query), mask, B, S, adapter)
        return self.layer_norm(z).view(B, S, D)


class TransformerBlock(nn.Module):
    def __init__(self, d_model, n_heads, d_inner, dropout):
        super().__init__()
        self.multi_head_attention = MultiHeadedAttention(n_heads=n_heads, d_model=d_model, dropout=dropout)
        self.feed_forward = PositionwiseFeedForward(d_model=d_model, d_inner=d_inner, dropout=dropout)

    def forward(self, block_input, mask):
        output = self.multi_head_attention(block_input, block_input, block_input, mask)
        return self.feed_forward(output)


class TransformerEncoder(nn.Module):
    """modules.py:90-113: LayerNorm(input + position_embedding) then the blocks."""

    def __init__(self, n_vocab, n_position, d_model, n_heads, dropout, n_layers):
        super().__init__()
        self.position_embedding = Embedding(n_position, d_model)
        self.dropout = nn.Dropout(p=dropout)
        self.layer_norm = LayerNorm(d_model, eps=1e-6)
        self.transformer_blocks = nn.ModuleList(
            [TransformerBlock(d_model=d_model, n_heads=n_heads, d_inner=d_model * 4, dropout=dropout)
             for _ in range(n_layers)])

    def forward(self, input_embs, log_mask, att_mask):
        B, S, D = input_embs.shape
        pos = self.position_embedding.table_bf16()[:S].contiguous()
        pe = self.position_embedding.weight
        output = self.layer_norm(to_2d_bf16(input_embs).contiguous(), res=pos, res_param=pe if pe.requires_grad else None)
        if self.training and self.dropout.p > 0:
            output = Fn.dropout_add(output, None, self.dropout.p)
        output = output.view(B, S, D)
        if "SASRecKAdaptedTransformerBlocks" in str(type(self.transformer_blocks)):      # modules.py:108-109
            return self.transformer_blocks(output, att_mask)
        for transformer in self.transformer_blocks:
            output = transformer.forward(output, att_mask)
        return output


class AdapterBlock(nn.Module):
    """modules.py:116-134: fc_up(act(fc_down(x))) + x; N(0, 0.01²) weights, zero biases; `dropout` is constructed but
    never applied by the reference (SURVEY.md Appendix B-1)."""

    def __init__(self, args, input_size, down_size, dropout=0.1):
        super().__init__()
        self.fc_down = Linear(input_size, down_size)
        nn.init.normal_(self.fc_down.weight, std=1e-2)
        nn.init.zeros_(self.fc_down.bias)
        self.act = "gelu" if args.adapter_activation == "GELU" else "relu"
        self.activate = nn.GELU() if self.act == "gelu" else nn.ReLU()
        self.fc_up = Linear(down_size, input_size)
        nn.init.normal_(self.fc_up.weight, std=1e-2)
        nn.init.zeros_(self.fc_up.bias)
        self.dropout = nn.Dropout(dropout)

    def forward(self, input_embs, extra_residual=None):
        """Returns fc_up(act(fc_down(x))) + x (+ extra_residual: the enclosing block's skip connection, fused into
        the same GEMM epilogue)."""
        x2 = to_2d_bf16(input_embs)
        if self.fused_ok(x2):
            return self.fused(x2, extra_residual).view(input_embs.shape)
        s = self.fc_down(x2, act=self.act)
        out = self.fc_up(s, residual=x2, residual2=extra_residual)
        return out.view(input_embs.shape)

    def fused_ok(self, x2):
        """the one-pass K5 kernel covers H % 64 == 0, H <= 768, r % 8 == 0, r <= 64 (BERT / ViT adapters); other shapes
        (the D = 64 SASRec adapters sit inside a 64-wide block that is launch-bound anyway) compose GEMM kernels"""
        return x2.is_contiguous() and ops.adapter_ln_supported(self.fc_down.in_features, self.fc_down.out_features)

    def fused(self, x2, extra_residual=None, ln=None):
        """tail(x + fc_up(act(fc_down(x))) [+ extra_residual]) in one kernel; tail = ln (a LayerNorm module) or identity"""
        return Fn.adapter_block(x2, extra_residual, self, ln=ln)


class AdapterPfeifferBlock(nn.Module):
    """modules.py:137-158: fc_up(act(fc_down(x))) WITHOUT the inner residual; default nn.Linear initialisation (the
    N(0, 0.01²) lines are commented out in the reference); act from args.adapter_activation in {"GELU", "leaky_relu",
    "relu"} — any other value (including the flag's default "RELU") leaves `activate` undefined in the reference and
    its forward raises AttributeError; the same happens here, at construction time, with a message."""

    def __init__(self, args, input_size, down_size, dropout=0.1):
        super().__init__()
        self.fc_down = Linear(input_size, down_size)
        kinds = {"GELU": ("gelu", nn.GELU), "leaky_relu": ("leaky_relu", nn.LeakyReLU), "relu": ("relu", nn.ReLU)}
        if args.adapter_activation not in kinds:
            raise AttributeError("'AdapterPfeifferBlock' object has no attribute 'activate' (adapter_activation=%r; the "
                                 "reference defines it only for GELU / leaky_relu / relu, modules.py:144-149)"
                                 % args.adapter_activation)
        self.act, cls = kinds[args.adapter_activation]
        self.activate = cls()
        self.fc_up = Linear(down_size, input_size)
        self.dropout = nn.Dropout(dropout)

    def forward(self, input_embs, extra_residual=None):
        """fc_up(act(fc_down(x))) (+ extra_residual, fused into the up-projection's epilogue)"""
        x2 = to_2d_bf16(input_embs)
        s = self.fc_down(x2, act=self.act)
        return self.fc_up(s, residual=extra_residual).view(input_embs.shape)


class HyperComplexAdapterBlock(nn.Module):
    """modules.py:209-250 (Compacter): up_sampler(gelu_new(down_sampler(x))) — two PHMLinear layers sharing the
    model-wide phm_rule, tanh-GELU in between, NO inner residual."""

    def __init__(self, args, input_size, down_size):
        super().__init__()
        self.args = args
        self.input_dim, self.down_sample_size = input_size, down_size
        self.down_sampler = PHMLinear(in_features=input_size, out_features=down_size, bias=True,
                                      phm_dim=args.hypercomplex_division, phm_rank=1)
        self.up_sampler = PHMLinear(in_features=down_size, out_features=input_size, bias=True,
                                    phm_dim=args.hypercomplex_division, phm_rank=1)

    def forward(self, x, extra_residual=None):
        """up(gelu_new(down(x))) (+ extra_residual: the enclosing block's skip connection, fused in the epilogue)"""
        x2 = to_2d_bf16(x)
        z = self.down_sampler(x2, act="gelu_new")
        return self.up_sampler(z, residual=extra_residual).view(x.shape)


class KAdapterBlock(nn.Module):
    """modules.py:161-206: down_project -> two TransformerBlocks of width down_size over the whole sequence with an
    all-ones mask (additive 0: NOT causal, padding positions attend and are attended) -> up_project, + the input.
    Projections ~ N(0, 2e-4²), zero biases."""

    def __init__(self, args, num_head, input_size, down_size, dropout=0.1):
        super().__init__()
        self.args = args
        self.down_project = Linear(input_size, down_size)
        self.up_project = Linear(down_size, input_size)
        self.init_weights()
        self.transformer_blocks = nn.ModuleList(
            [TransformerBlock(d_model=down_size, n_heads=num_head, d_inner=down_size * 4, dropout=dropout)
             for _ in range(2)])
        for blk in self.transformer_blocks:
            blk.multi_head_attention.causal = False

    def forward(self, hidden_states):
        """hidden_states [N, L, H] -> [N, L, H]"""
        N, L, H = hidden_states.shape
        x2 = to_2d_bf16(hidden_states).contiguous()
        output = self.down_project(x2).view(N, L, -1)
        for transformer in self.transformer_blocks:
            output = transformer.forward(output, None)
        return self.up_project(to_2d_bf16(output), residual=x2).view(N, L, H)

    def init_weights(self):
        self.down_project.weight.data.normal_(mean=0.0, std=2e-4)
        self.down_project.bias.data.zero_()
        self.up_project.weight.data.normal_(mean=0.0, std=2e-4)
        self.up_project.bias.data.zero_()
