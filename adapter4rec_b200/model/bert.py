"""BERT / RoBERTa encoder body with the module tree and parameter names of transformers' BertModel / RobertaModel
(so `model.bert_encoder.text_encoders.title.bert_model.encoder.layer[i].attention.output = ...` surgery from
Downstream/Text/run.py:414-465 and reference checkpoints work unchanged), executing on the sm_100a kernels.

Numerics follow the layer algebra of SURVEY.md Appendix A2: bf16 activations, fp32 accumulation/statistics.
Dropout (train mode): hidden-state dropouts run in a4r_dropout fused with the residual add that follows them, the
attention-probability dropout inside the attention kernel; both use a counter-based RNG whose masks the backward
regenerates.  eval() / p = 0 is the deterministic arithmetic the parity tests are defined on."""
import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .layers import BF16, Embedding, LayerNorm, Linear, LoRALinear, frozen_ffn_dense, to_2d_bf16


class TextConfigLite:
    """Subset of transformers' BertConfig / RobertaConfig used by the path.  Accepts a transformers config object
    (duck-typed) or keyword arguments."""

    def __init__(self, hf_config=None, **kw):
        src = {} if hf_config is None else {k: getattr(hf_config, k) for k in dir(hf_config) if not k.startswith("_")
                                            and isinstance(getattr(hf_config, k, None), (int, float, str, bool, type(None)))}
        src.update(kw)
        self.vocab_size = src.get("vocab_size", 30522)
        self.hidden_size = src.get("hidden_size", 768)
        self.num_hidden_layers = src.get("num_hidden_layers", 12)
        self.num_attention_heads = src.get("num_attention_heads", 12)
        self.intermediate_size = src.get("intermediate_size", 3072)
        self.max_position_embeddings = src.get("max_position_embeddings", 512)
        self.type_vocab_size = src.get("type_vocab_size", 2)
        self.layer_norm_eps = src.get("layer_norm_eps", 1e-12)
        self.pad_token_id = src.get("pad_token_id", 0)
        self.model_type = src.get("model_type", "bert")
        self.hidden_dropout_prob = src.get("hidden_dropout_prob", 0.1)
        self.attention_probs_dropout_prob = src.get("attention_probs_dropout_prob", 0.1)
        self.initializer_range = src.get("initializer_range", 0.02)


class BertEmbeddings(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.word_embeddings = Embedding(config.vocab_size, config.hidden_size, padding_idx=config.pad_token_id)
        self.position_embeddings = Embedding(config.max_position_embeddings, config.hidden_size)
        self.token_type_embeddings = Embedding(config.type_vocab_size, config.hidden_size)
        self.LayerNorm = LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)
        self._typ_cache = Fn.WeightCache()

    def forward(self, input_ids):
        """input_ids: int64 [N, L] (may be a strided view of the reference's [ids | mask] rows) -> bf16 [N*L, H]."""
        N, L = input_ids.shape
        we = self.word_embeddings
        prompt = None
        if hasattr(we, "learned_embedding"):          # SoftEmbedding (Downstream/Text/model/model.py:586-630)
            prompt, table = we.learned_embedding, we.wte.table_bf16()
            assert we.n_tokens <= L
        else:
            table = we.table_bf16()
        roberta_pad = self.config.pad_token_id if self.config.model_type == "roberta" else -1
        typ = self._typ_cache.get(self.token_type_embeddings.weight)[0][0]
        tables = (table, self.position_embeddings.table_bf16(), typ)
        g, b = self.LayerNorm.weight.detach().float(), self.LayerNorm.bias.detach().float()
        # fp32 masters of whatever is trainable here (full fine-tuning); the word table's padding_idx row never gets a
        # gradient (transformers builds it with nn.Embedding(..., padding_idx=pad_token_id))
        wmaster = we.wte.weight if hasattr(we, "learned_embedding") else we.weight
        masters = [wmaster, self.position_embeddings.weight, self.token_type_embeddings.weight, self.LayerNorm.weight,
                   self.LayerNorm.bias]
        masters = [m if m.requires_grad else None for m in masters]
        x = Fn.EmbedLNFunction.apply(input_ids, L, tables, g, b, self.LayerNorm.eps, roberta_pad, prompt,
                                     int(self.config.pad_token_id), *masters)
        if self.training and self.dropout.p > 0:
            x = Fn.dropout_add(x, None, self.dropout.p)
        return x


class BertSelfAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.num_attention_heads = config.num_attention_heads
        self.attention_head_size = config.hidden_size // config.num_attention_heads
        self.all_head_size = config.hidden_size
        self.query = Linear(config.hidden_size, config.hidden_size)
        self.key = Linear(config.hidden_size, config.hidden_size)
        self.value = Linear(config.hidden_size, config.hidden_size)
        self.dropout = nn.Dropout(config.attention_probs_dropout_prob)
        self._qkv_cache = Fn.QKVCache()

    def forward(self, x2d, attention_mask, N, L, packed=None, want_skip=False):
        """x2d bf16 [N*L, H]; attention_mask int64/f32 [N, L] (non-zero = attend) or None -> context [N*L, H].
        packed = PackedTokens: x2d holds only the kept tokens [T, H]; the mask is per token row.
        want_skip: also return x2d as an output of the projection's autograd node — the caller uses THAT tensor as the
        sub-layer's skip input, so the skip gradient is added inside the data-gradient GEMM's epilogue."""
        # any of query / key / value may have been replaced by a loralib Linear
        out = Fn.qkv(x2d, (self.query, self.key, self.value), self._qkv_cache, skip=want_skip)
        qkv, skip = out if want_skip else (out, None)
        if packed is not None:
            ctx = Fn.attention(qkv, packed.token_mask, N, L, self.num_attention_heads, self.attention_head_size,
                               causal=False, mask_neg=ops.F32_MIN, dropout_p=self.dropout.p if self.training else 0.0,
                               cu_seqlens=packed.cu_seqlens)
        else:
            ctx = Fn.attention(qkv, attention_mask, N, L, self.num_attention_heads, self.attention_head_size,
                               causal=False, mask_neg=ops.F32_MIN, dropout_p=self.dropout.p if self.training else 0.0)
        return (ctx, skip) if want_skip else ctx


class BertSelfOutput(nn.Module):
    """dense -> dropout -> LayerNorm(h + input).  Used for attention.output and (as BertOutput) for output."""

    def __init__(self, config, in_features=None):
        super().__init__()
        self.dense = Linear(in_features or config.hidden_size, config.hidden_size)
        self.LayerNorm = LayerNorm(config.hidden_size, eps=config.layer_norm_eps)
        self.dropout = nn.Dropout(config.hidden_dropout_prob)

    def forward(self, hidden_states, input_tensor):
        shape = input_tensor.shape
        p = self.dropout.p if self.training else 0.0
        d = self.dense
        if not (d.weight.requires_grad or d.bias.requires_grad):
            # frozen dense: dense -> dropout -> + input -> LayerNorm as ONE autograd node (fused epilogues both ways)
            out = Fn.frozen_block(to_2d_bf16(hidden_states), to_2d_bf16(input_tensor), d, ln=self.LayerNorm, p=p)
            return out.view(shape)
        if p > 0:
            z = Fn.dropout_add(d(to_2d_bf16(hidden_states)), to_2d_bf16(input_tensor).contiguous(), p)
        else:
            z = d(to_2d_bf16(hidden_states), residual=to_2d_bf16(input_tensor))   # residual fused in the epilogue
        return self.LayerNorm(z).view(shape)


class BertOutput(BertSelfOutput):
    def __init__(self, config):
        super().__init__(config, in_features=config.intermediate_size)


class BertAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.self = BertSelfAttention(config)
        self.output = BertSelfOutput(config)

    def forward(self, x2d, attention_mask, N, L, packed=None):
        ctx, skip = self.self(x2d, attention_mask, N, L, packed, want_skip=True)
        return self.output(ctx, skip)


class BertIntermediate(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = Linear(config.hidden_size, config.intermediate_size)

    def forward(self, x):
        return self.dense(x, act="gelu")


class BertLayer(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.attention = BertAttention(config)
        self.intermediate = BertIntermediate(config)
        self.output = BertOutput(config)

    def forward(self, x2d, attention_mask, N, L, cls_only=False, packed=None):
        """cls_only (last layer when the caller reads hidden[:, 0] only, as Text_Encoder does, encoders.py:55): every
        op after the attention is row-wise, so only the [CLS] row of each item is pushed through the output
        projection, the feed-forward and the LayerNorms (1/L of the work); K and V still cover all tokens."""
        if cls_only:
            H = x2d.shape[1]
            ctx, skip = self.attention.self(x2d, attention_mask, N, L, packed, want_skip=True)
            if packed is not None:   # the [CLS] token is the first row of every packed sequence
                y = self.attention.output(Fn.gather_rows(ctx, packed.cls_rows), Fn.gather_rows(skip, packed.cls_rows))
            else:
                y = self.attention.output(ctx.view(N, L, H)[:, 0], skip.view(N, L, H)[:, 0])   # strided [N,H] views, no copies
        else:
            y = self.attention(x2d, attention_mask, N, L, packed)
        out = self.output
        wi = self.intermediate.dense
        wf = frozen_ffn_dense(wi, out)
        if wf is not None and type(out) is BertOutput:
            # frozen feed-forward + dropout + residual + LayerNorm: one autograd node (GELU', dropout and the residual
            # gradient all live in GEMM / LayerNorm-backward epilogues)
            p = out.dropout.p if self.training else 0.0
            return Fn.frozen_block(y, y, wf, intermediate=wi, ln=out.LayerNorm, p=p)
        if wf is not None and hasattr(out, "forward_block"):
            # serial Houlsby wrapper: FFN pair + dropout + adapter + LayerNorm in one autograd node
            fused = out.forward_block(y, y, wi)
            if fused is not None:
                return to_2d_bf16(fused)
        if wf is not None and hasattr(out, "forward_from_dense"):
            # adapter-wrapped output: the frozen FFN pair stays fused, the wrapper continues from the dense output
            h = Fn.frozen_block(y, None, wf, intermediate=wi)
            return to_2d_bf16(out.forward_from_dense(h, y))
        return out(self.intermediate(y), y)                 # foreign or trainable output module


class PackedTokens:
    """Variable-length ("unpadded") token layout of one forward pass: only the tokens the attention mask keeps exist, the
    sequences lie back to back.  Exact for what Text_Encoder consumes (hidden[:, 0], encoders.py:53-55): a padded token is
    never a key (additive finfo.min mask) and every other op of the layer is row-wise, so it cannot influence a kept
    token.  An item whose mask is ALL zero (the padding item, row 0 of item_content) keeps its L tokens and its zero
    mask: with every key masked the additive mask yields the uniform softmax of the reference (SURVEY.md Appendix B-6).

    token_rows: int64 [T] rows of the padded [N*L] layout that are kept; cu_seqlens: int32 [N+1]; token_mask: f32 [T];
    cls_rows: int64 [N] first packed row of every sequence."""

    def __init__(self, attention_mask):
        m = attention_mask != 0
        keep = m | (~m.any(dim=1, keepdim=True))
        flat = keep.reshape(-1)
        self.token_rows = flat.nonzero().squeeze(1)                      # (one host sync: T is data dependent)
        lens = keep.sum(dim=1)
        cu = torch.zeros(m.shape[0] + 1, dtype=torch.int32, device=m.device)
        cu[1:] = torch.cumsum(lens, 0)
        self.cu_seqlens = cu
        self.cls_rows = cu[:-1].long()
        self.token_mask = m.reshape(-1)[self.token_rows].float().contiguous()
        self.num_tokens = int(self.token_rows.numel())


class BertEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.layer = nn.ModuleList([BertLayer(config) for _ in range(config.num_hidden_layers)])


class BertPooler(nn.Module):
    """Kept for state_dict compatibility; the reference computes it and discards the result
    (SURVEY.md Appendix B-5), so it is never evaluated here."""

    def __init__(self, config):
        super().__init__()
        self.dense = Linear(config.hidden_size, config.hidden_size)


class BertModel(nn.Module):
    """forward(input_ids=, attention_mask=) -> (last_hidden_state [N, L, H] bf16,) like transformers' BertModel[0]."""

    def __init__(self, config, add_pooling_layer=True):
        super().__init__()
        self.config = config if isinstance(config, TextConfigLite) else TextConfigLite(config)
        self.embeddings = BertEmbeddings(self.config)
        self.encoder = BertEncoder(self.config)
        self.pooler = BertPooler(self.config) if add_pooling_layer else None
        self.apply(self._init_weights)

    def _init_weights(self, module):
        std = self.config.initializer_range
        if isinstance(module, (Linear, Embedding)):
            nn.init.normal_(module.weight, mean=0.0, std=std)
            if getattr(module, "bias", None) is not None:
                nn.init.zeros_(module.bias)
        elif isinstance(module, LayerNorm):
            nn.init.ones_(module.weight)
            nn.init.zeros_(module.bias)

    def get_input_embeddings(self):
        return self.embeddings.word_embeddings

    def set_input_embeddings(self, value):
        self.embeddings.word_embeddings = value

    supports_cls_only = True

    def forward(self, input_ids=None, attention_mask=None, cls_only=False, output_hidden_states=None, **unused):
        """cls_only=True returns [N, 1, H] (the [CLS] position only), skipping the row-wise tail of the last layer for
        all other tokens; values at position 0 are identical to the full computation.
        output_hidden_states (default: config.output_hidden_states, which the reference sets when loading,
        run.py:286-297) -> (last_hidden_state, None, (embedding output, layer 1 output, ..., layer n output)) — the
        transformers tuple layout BertKAdaptedBertModel reads as outputs[2] (the pooler output, outputs[1], is never
        evaluated: SURVEY.md Appendix B-5)."""
        N, L = input_ids.shape
        if output_hidden_states is None:
            output_hidden_states = bool(getattr(self.config, "output_hidden_states", False))
        x = self.embeddings(input_ids)
        all_hidden = [x.view(N, L, -1)] if output_hidden_states else None
        last = len(self.encoder.layer) - 1
        # `unpad` (opt-in attribute): run the layers on the kept tokens only.  Needs the [CLS]-only consumer (nothing else
        # reads per-token outputs), the short-sequence attention kernel, and embeddings that are not being trained (their
        # gradient would have to be scattered back to the padded layout; adapter tuning never needs it)
        packed = None
        if (getattr(self, "unpad", False) and cls_only and not output_hidden_states and attention_mask is not None
                and L <= 32 and not x.requires_grad):
            packed = PackedTokens(attention_mask)
            x = Fn.gather_rows(x, packed.token_rows)
        for i, layer in enumerate(self.encoder.layer):
            x = layer(x, attention_mask, N, L, cls_only=cls_only and i == last and not output_hidden_states, packed=packed)
            if output_hidden_states:
                all_hidden.append(x.view(N, L, -1))
        if output_hidden_states:
            return (x.view(N, L, -1), None, tuple(all_hidden))
        return (x.view(N, 1 if cls_only else L, -1),)


class RobertaModel(BertModel):
    def __init__(self, config, add_pooling_layer=True):
        cfg = config if isinstance(config, TextConfigLite) else TextConfigLite(config)
        cfg.model_type = "roberta"
        super().__init__(cfg, add_pooling_layer)
