"""ViT item encoder with the module tree and parameter names of transformers' ViTForImageClassification (so the surgery
of Downstream/CV/run_adapter.py:367-470 — `vit.encoder.layer[i].attention.output = VITAdaptedSelfOutput(...)`,
`.output = VITAdaptedOutput(...)`, `attention.attention.query/value = lora.Linear(768, 768, r=12)`,
`vit.embeddings = SoftPrompt(...)`, `classifier = nn.Linear(768, D)` — and reference checkpoints work unchanged),
executing on the sm_100a kernels.  Pre-LN layer algebra of SURVEY.md Appendix A3."""
import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from ..model.layers import BF16, LayerNorm, Linear, frozen_ffn_dense, to_2d_bf16


class ViTConfigLite:
    def __init__(self, hf_config=None, **kw):
        src = {} if hf_config is None else {k: getattr(hf_config, k) for k in dir(hf_config) if not k.startswith("_")
                                            and isinstance(getattr(hf_config, k, None), (int, float, str, bool, type(None)))}
        src.update(kw)
        self.hidden_size = src.get("hidden_size", 768)
        self.num_hidden_layers = src.get("num_hidden_layers", 12)
        self.num_attention_heads = src.get("num_attention_heads", 12)
        self.intermediate_size = src.get("intermediate_size", 3072)
        self.image_size = src.get("image_size", 224)
        self.patch_size = src.get("patch_size", 16)
        self.num_channels = src.get("num_channels", 3)
        self.layer_norm_eps = src.get("layer_norm_eps", 1e-12)
        self.hidden_dropout_prob = src.get("hidden_dropout_prob", 0.0)
        self.attention_probs_dropout_prob = src.get("attention_probs_dropout_prob", 0.0)
        # ViT-base's defaults (and every checkpoint the reference loads, Downstream/CV/run_adapter.py:283-297) have both
        # dropouts at 0.0, and the serial wrappers / plain ViT blocks of this package do not apply them: refuse a config
        # that asks for dropout rather than train silently without it.
        if self.hidden_dropout_prob != 0.0 or self.attention_probs_dropout_prob != 0.0:
            raise NotImplementedError("ViT hidden_dropout_prob / attention_probs_dropout_prob must be 0.0 (got %r / %r)"
                                      % (self.hidden_dropout_prob, self.attention_probs_dropout_prob))
        self.initializer_range = src.get("initializer_range", 0.02)
        self.num_labels = src.get("num_labels", 2)


class PatchProjection(nn.Module):
    """Parameters of nn.Conv2d(C, H, kernel_size=ps, stride=ps): weight [H,C,ps,ps], bias [H]."""

    def __init__(self, in_channels, out_channels, patch_size):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels, patch_size, patch_size))
        self.bias = nn.Parameter(torch.zeros(out_channels))
        nn.init.normal_(self.weight, std=0.02)
        self._cache = Fn.WeightCache()


class ViTPatchEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.image_size, self.patch_size, self.num_channels = config.image_size, config.patch_size, config.num_channels
        self.num_patches = (config.image_size // config.patch_size) ** 2
        self.projection = PatchProjection(config.num_channels, config.hidden_size, config.patch_size)

    def forward(self, pixel_values):
        """[N,C,R,R] f32 -> patch embeddings [N*P, H] bf16: im2col kernel + tcgen05 GEMM.  With a trainable projection
        (full fine-tuning: Downstream/CV/run_adapter.py `fine_tune_to=all`, Pretraining/CV) the conv's weight gradient is
        the weight-gradient GEMM d_embᵀ · patches over the saved im2col rows, its bias gradient a column sum."""
        pr = self.projection
        patches = ops.patchify(pixel_values.float().contiguous(), self.patch_size)
        w2d = pr.weight.view(pr.weight.shape[0], -1)
        if pr.weight.requires_grad or pr.bias.requires_grad:
            return Fn.linear(patches, w2d, pr.bias, pr._cache)
        return ops.gemm(patches, pr._cache.get(w2d)[0], bias=pr.bias.detach().float().contiguous())


class _AssembleFunction(torch.autograd.Function):
    """Token assembly out[n] = [cls + pos[0] | patch_emb[n] + pos[1:] | prompt].  Adapter tuning trains the appended
    soft-prompt tokens only; full fine-tuning also needs d_patch_emb (a row slice of d_out), d_pos = the sum of d_out over
    the images (deterministic two-stage column sum) and d_cls = d_pos[0] (cls and pos[0] feed the same token)."""

    @staticmethod
    def forward(ctx, patch_emb, cls, pos, prompt, N, P, cls16, pos16):
        p16 = None if prompt is None else prompt.detach().reshape(-1, prompt.shape[-1]).to(BF16).contiguous()
        out = ops.vit_assemble(patch_emb.detach(), cls16, pos16, p16, N, P)
        ctx.dims = (N, P, 0 if p16 is None else p16.shape[0], patch_emb.shape[1])
        ctx.shapes = (cls.shape, pos.shape, None if prompt is None else prompt.shape)
        return out

    @staticmethod
    def backward(ctx, dout):
        N, P, T, H = ctx.dims
        cls_shape, pos_shape, prompt_shape = ctx.shapes
        L = 1 + P + T
        dout = dout.contiguous()
        d2 = dout.view(N, L * H)
        dpe = dcls = dpos = dprompt = None
        if ctx.needs_input_grad[0]:
            dpe = dout.view(N, L, H)[:, 1:1 + P].reshape(N * P, H)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dsum = ops.colsum(d2, width=(1 + P) * H)
            if ctx.needs_input_grad[1]:
                dcls = dsum[:H].clone().view(cls_shape)
            if ctx.needs_input_grad[2]:
                dpos = dsum.view(pos_shape)
        if T > 0 and ctx.needs_input_grad[3]:
            dprompt = ops.colsum(d2[:, (1 + P) * H:], width=T * H).view(prompt_shape)
        return dpe, dcls, dpos, dprompt, None, None, None, None


class ViTEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.cls_token = nn.Parameter(torch.randn(1, 1, config.hidden_size))
        self.patch_embeddings = ViTPatchEmbeddings(config)
        self.position_embeddings = nn.Parameter(torch.randn(1, self.patch_embeddings.num_patches + 1, config.hidden_size))
        self.dropout = nn.Dropout(config.hidden_dropout_prob)
        self._cls_cache, self._pos_cache = Fn.WeightCache(), Fn.WeightCache()

    def tokens(self, pixel_values, prompt=None):
        N = pixel_values.shape[0]
        P = self.patch_embeddings.num_patches
        pe = self.patch_embeddings(pixel_values)
        cls16 = self._cls_cache.get(self.cls_token.view(1, -1))[0].view(-1)
        pos16 = self._pos_cache.get(self.position_embeddings.view(P + 1, -1))[0]
        x = _AssembleFunction.apply(pe, self.cls_token, self.position_embeddings, prompt, N, P, cls16, pos16)
        T = 0 if prompt is None else prompt.shape[-2]
        return x, 1 + P + T

    def forward(self, pixel_values, bool_masked_pos=None, interpolate_pos_encoding=None):
        x, L = self.tokens(pixel_values)
        return x.view(pixel_values.shape[0], L, -1)


class ViTSelfAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.num_attention_heads = config.num_attention_heads
        self.attention_head_size = config.hidden_size // config.num_attention_heads
        self.query = Linear(config.hidden_size, config.hidden_size)
        self.key = Linear(config.hidden_size, config.hidden_size)
        self.value = Linear(config.hidden_size, config.hidden_size)
        self._qkv_cache = Fn.QKVCache()

    def forward(self, x2d, N, L):
        # query / value may be loralib Linears (run_adapter.py:383-388)
        qkv = Fn.qkv(x2d, (self.query, self.key, self.value), self._qkv_cache)
        return Fn.attention(qkv, None, N, L, self.num_attention_heads, self.attention_head_size, causal=False)


class ViTSelfOutput(nn.Module):
    """transformers' ViTSelfOutput: dense (+ dropout); the residual is added by ViTLayer."""

    def __init__(self, config):
        super().__init__()
        self.dense = Linear(config.hidden_size, config.hidden_size)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_states, input_tensor=None):
        return self.dense(hidden_states)

    def forward_fused(self, hidden_states, residual):
        """dense(hidden) + residual with the skip connection fused into the GEMM epilogue"""
        return self.dense(to_2d_bf16(hidden_states), residual=to_2d_bf16(residual))


class ViTAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.attention = ViTSelfAttention(config)
        self.output = ViTSelfOutput(config)


class ViTIntermediate(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = Linear(config.hidden_size, config.intermediate_size)

    def forward(self, x):
        return self.dense(x, act="gelu")


class ViTOutput(nn.Module):
    """transformers' ViTOutput: dense(hidden) + input_tensor."""

    def __init__(self, config):
        super().__init__()
        self.dense = Linear(config.intermediate_size, config.hidden_size)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_states, input_tensor):
        return self.dense(to_2d_bf16(hidden_states), residual=to_2d_bf16(input_tensor)).view(input_tensor.shape)


class ViTLayer(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.attention = ViTAttention(config)
        self.intermediate = ViTIntermediate(config)
        self.output = ViTOutput(config)
        self.layernorm_before = LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.layernorm_after = LayerNorm(config.hidden_size, eps=config.layer_norm_eps)

    def forward(self, x2d, N, L, cls_only=False):
        """x1 = x + A1(dense(attn(LN(x)))),  x2 = x1 + A2(dense(GELU(dense(LN(x1)))))   (A = identity without adapters).
        cls_only (last layer, classifier reads token 0 only): the row-wise tail runs on the [CLS] rows alone."""
        H = x2d.shape[1]
        ln0, res = self.layernorm_before.forward_skip(x2d)      # the skip gradient is added inside LN-backward
        ctx = self.attention.attention(ln0, N, L)
        if cls_only:
            ctx, res = ctx.view(N, L, H)[:, 0], res.view(N, L, H)[:, 0]
        ao = self.attention.output
        x1 = ao.forward_fused(ctx, res) if hasattr(ao, "forward_fused") else (to_2d_bf16(ao(ctx, res)) + res)
        y, x1 = self.layernorm_after.forward_skip(x1)
        out = self.output
        wi = self.intermediate.dense
        wf = frozen_ffn_dense(wi, out)
        if wf is not None and type(out) is ViTOutput:
            return Fn.frozen_block(y, x1, wf, intermediate=wi)
        if wf is not None and hasattr(out, "forward_from_dense"):
            h = Fn.frozen_block(y, None, wf, intermediate=wi)
            return to_2d_bf16(out.forward_from_dense(h, x1))
        return to_2d_bf16(out(self.intermediate(y), x1))


class ViTEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.layer = nn.ModuleList([ViTLayer(config) for _ in range(config.num_hidden_layers)])


class ViTModel(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.embeddings = ViTEmbeddings(config)
        self.encoder = ViTEncoder(config)
        self.layernorm = LayerNorm(config.hidden_size, eps=config.layer_norm_eps)

    def forward(self, pixel_values, cls_only=False, **unused):
        N = pixel_values.shape[0]
        emb = self.embeddings
        if hasattr(emb, "tokens"):
            x, L = emb.tokens(pixel_values)
        else:
            raise TypeError("vit.embeddings must be ViTEmbeddings or SoftPrompt")
        last = len(self.encoder.layer) - 1
        for i, layer in enumerate(self.encoder.layer):
            x = layer(x, N, L, cls_only=cls_only and i == last)
        x = self.layernorm(x)
        return (x.view(N, 1 if cls_only else L, -1),)


class ViTForImageClassification(nn.Module):
    """forward(pixel_values, return_dict=None) -> (logits [N, num_labels],), as the reference consumes it
    (Vit_Encoder.forward, Downstream/CV/model/encoders.py:31-32).  `classifier` is replaced by the caller with
    nn.Linear(768, embedding_dim) (run_adapter.py:291-297); any module with weight/bias works."""

    def __init__(self, config):
        super().__init__()
        self.config = config if isinstance(config, ViTConfigLite) else ViTConfigLite(config)
        self.vit = ViTModel(self.config)
        self.classifier = Linear(self.config.hidden_size, self.config.num_labels)
        self.apply(self._init_weights)

    def _init_weights(self, module):
        std = self.config.initializer_range
        if isinstance(module, Linear):
            nn.init.trunc_normal_(module.weight, mean=0.0, std=std)
            if module.bias is not None:
                nn.init.zeros_(module.bias)
        elif isinstance(module, LayerNorm):
            nn.init.ones_(module.weight)
            nn.init.zeros_(module.bias)
        elif isinstance(module, ViTEmbeddings):
            nn.init.trunc_normal_(module.position_embeddings, mean=0.0, std=std)
            nn.init.trunc_normal_(module.cls_token, mean=0.0, std=std)

    def forward(self, pixel_values=None, return_dict=None, **unused):
        hidden = self.vit(pixel_values, cls_only=True)[0]
        cls = hidden[:, 0]
        clf = self.classifier
        if not hasattr(clf, "_cache"):
            clf._cache = Fn.WeightCache()
        logits = Fn.linear(to_2d_bf16(cls), clf.weight, clf.bias, clf._cache)
        return (logits,)
