"""Model / ModelCPC and the adapter wrapper classes, mirroring Downstream/Text/model/model.py (names, constructor and
forward signatures, state_dict keys).  The loss is the reference's BCE-with-logits over one sampled negative per
position (model.py:30,62-68), computed by the fused K9 kernel."""
import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .encoders import Bert_Encoder, User_Encoder
from .layers import BF16, Embedding, IdEmbedding, to_2d_bf16
from .layers import LayerNorm
from .layers import PHMLinear
from .layers import Linear
from .modules import AdapterBlock, AdapterPfeifferBlock, HyperComplexAdapterBlock, KAdapterBlock


def _word_dim(args):
    """The reference sizes BERT adapters from the model NAME (model.py:275-286)."""
    name = args.bert_model_load
    for key, dim in (("tiny", 128), ("mini", 256), ("medium", 512), ("base", 768), ("large", 1024)):
        if key in name:
            return dim
    raise AssertionError("The pretrained model name should be defined correctly. such as bert-base-uncased so on")


def check_trainable_supported(module):
    """Fail loudly instead of silently leaving a gradient at zero.  The sm_100a path differentiates adapters, LoRA factors,
    biases, LayerNorms, prompt embeddings, every Linear weight and — for full fine-tuning — the BERT / RoBERTa / SASRec
    embedding tables and the ViT patch projection / cls token / position embeddings.  The BERT pooler is kept for
    state_dict compatibility but never evaluated (the reference computes and discards it, SURVEY.md Appendix B-5;
    Pretraining/Text/run.py:48-64 freezes it): left trainable it simply receives no gradient, as in the reference.
    Nothing on the modality-encoder path is refused today; the hook stays so that a future parameter kind without a
    gradient kernel can be rejected here."""
    return None


class _ModelBase(nn.Module):
    cpc = False

    def __init__(self, args, item_num, use_modal, bert_model):
        super().__init__()
        self.args = args
        self.use_modal = use_modal
        self.max_seq_len = args.max_seq_len + 1
        self.l2_weight = args.l2_weight / 2
        if self.use_modal:
            self.bert_encoder = Bert_Encoder(args=args, bert_model=bert_model)
        else:                                           # --item_tower id: the item table is a trainable embedding
            self.id_embedding = IdEmbedding(item_num + 1, args.embedding_dim, padding_idx=0)
        self.user_encoder = User_Encoder(item_num=item_num, max_seq_len=args.max_seq_len, item_dim=args.embedding_dim,
                                         num_attention_heads=args.num_attention_heads, dropout=args.drop_rate,
                                         n_layers=args.transformer_block)
        self.criterion = nn.BCEWithLogitsLoss()   # structural parity only; the fused kernel computes the loss
        self._checked = None

    def forward(self, sample_items, log_mask, local_rank=None, sample_items_id=None, cand_bias=None):
        """sample_items int64 [B*(S+1)*2, 2L] (ids | mask rows), log_mask f32 [B,S] -> scalar loss.  The id tower
        (use_modal = False) takes the item ids themselves: int64 [B*(S+1)*2] or [B, S+1, 2].

        Extension beyond the reference signature (model.py:48): with `args.loss_type == "inbatch_softmax"` (an attribute,
        not a command-line flag — the flag set stays the reference's) the BCE head is replaced by the in-batch softmax
        head with duplicate-item masking (K9-S); it needs `sample_items_id` int64 [B, S+1] (the item id of every history
        slot, 0 = padding) and optionally `cand_bias` f32 [B*(S+1)] (log-popularity debias)."""
        if self.training:
            sig = tuple(p.requires_grad for p in self.parameters())
            if sig != self._checked:
                check_trainable_supported(self)
                self._checked = sig
        D = self.args.embedding_dim
        if not self.use_modal:
            input_embs, input_logs_embs = self.id_embedding(sample_items.reshape(-1, self.max_seq_len, 2))
        elif getattr(self, "dedup_items", False):
            # Optional (off by default, not what the reference executes): an item that occurs several times in the batch
            # — as a positive of several users, as a sampled negative, as the padding row — is encoded ONCE and its
            # embedding row is shared; the backward sums the gradient rows of its occurrences.  Identical forward values
            # (every op of the encoder is independent across items); in train mode the occurrences now share one dropout
            # mask where the reference draws one per occurrence.
            uniq, inverse, counts = Fn.unique_rows(sample_items)
            input_embs_all = Fn.expand_rows(self.bert_encoder(uniq), inverse, counts)
        else:
            input_embs_all = self.bert_encoder(sample_items)                   # [N, D] bf16
        if self.use_modal:
            input_embs = input_embs_all.view(-1, self.max_seq_len, 2, D)
            input_logs_embs = input_embs[:, :-1, 0, :].contiguous()            # history items 0..S-1 as user-encoder input
        log_mask = log_mask.to(device=input_embs.device, dtype=torch.float32).contiguous()
        prec_vec = self.user_encoder(input_logs_embs, log_mask, local_rank)
        if getattr(self.args, "loss_type", "bce") == "inbatch_softmax":
            if self.cpc or sample_items_id is None:
                raise ValueError("loss_type='inbatch_softmax' needs sample_items_id [B, S+1] and is not defined for ModelCPC")
            ids = sample_items_id.to(device=input_embs.device, dtype=torch.int64).view(-1, self.max_seq_len).contiguous()
            return Fn.inbatch_softmax_loss(prec_vec.contiguous(), input_embs.contiguous(), ids, log_mask, cand_bias)
        return Fn.bce_loss(prec_vec.contiguous(), input_embs.contiguous(), None if self.cpc else log_mask, cpc=self.cpc)


class Model(_ModelBase):
    """Downstream/Text/model/model.py:9-70."""
    cpc = False


class ModelCPC(_ModelBase):
    """Downstream/Text/model/model.py:73-135: the loss uses the last position only, without a validity mask."""
    cpc = True


class BertAdaptedSelfOutput(nn.Module):
    """model.py:273-297 (Houlsby serial; wraps BOTH attention.output and output, run.py:456-460):
    dense -> dropout -> adapter -> LayerNorm(h + input)."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, _word_dim(args), args.bert_adapter_down_size, args.adapter_dropout_rate)

    def forward(self, hidden_states, input_tensor):
        out = self.forward_block(to_2d_bf16(hidden_states), input_tensor, None)
        if out is not None:
            return out
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_block(self, x2, input_tensor, intermediate):
        """dense (or intermediate -> GELU -> dense when `intermediate` is given) -> dropout -> adapter -> LayerNorm as ONE
        autograd node (Fn.HoulsbyPostLNBlockFunction) when the block's dense layers are frozen and the adapter has the
        fused kernel's shape; None otherwise (the caller composes the pieces)."""
        d = self.self_output.dense
        inp = x2 if input_tensor is x2 else to_2d_bf16(input_tensor)   # identity matters: inp is x folds the skip gradient
        mods = (d,) if intermediate is None else (d, intermediate)
        if any(m.weight.requires_grad or m.bias.requires_grad for m in mods):
            return None
        if inp is not x2 and not inp.is_contiguous():
            # the [CLS]-only tail of the padded layout hands in a strided [N, H] view of the skip rows: one small copy keeps
            # it on the fused kernel, i.e. on the same instruction sequence as the unpadded layout (bit-equal results)
            inp = inp.contiguous()
        if not (ops.adapter_ln_supported(self.adapter.fc_down.in_features, self.adapter.fc_down.out_features)
                and inp.is_contiguous() and x2.shape[0] == inp.shape[0]):
            return None
        p = self.self_output.dropout.p if self.training else 0.0
        out = Fn.houlsby_postln_block(x2, inp, p, d, intermediate, self.adapter, self.self_output.LayerNorm)
        return out.view(input_tensor.shape)

    def forward_from_dense(self, h, input_tensor):
        """everything after self_output.dense (the encoder layer fuses that dense with the GELU GEMM before it)"""
        h = to_2d_bf16(h)
        drop = self.self_output.dropout
        if self.training and drop.p > 0:
            h = Fn.dropout_add(h, None, drop.p)                   # model.py:294: dropout BEFORE the adapter
        inp = to_2d_bf16(input_tensor)
        if self.adapter.fused_ok(h) and inp.is_contiguous():
            return self.adapter.fused(h, inp, ln=self.self_output.LayerNorm).view(input_tensor.shape)
        z = self.adapter(h, extra_residual=inp)
        return self.self_output.LayerNorm(z).view(input_tensor.shape)


class BertAdaptedParallelSelfOutput(nn.Module):
    """model.py:246-270 (Houlsby parallel, is_serial = 'None', run.py:466-479): the adapter reads the block INPUT;
    LayerNorm(adapter(input) + dropout(dense(h)) + input) where adapter(x) = fc_up(act(fc_down(x))) + x, i.e. the
    input enters the sum twice, as in the reference."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, _word_dim(args), args.bert_adapter_down_size, args.adapter_dropout_rate)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        inp = to_2d_bf16(input_tensor).contiguous()
        a = to_2d_bf16(self.adapter(inp, extra_residual=inp))             # up(act(down(inp))) + inp + inp
        h = to_2d_bf16(h)
        drop = self.self_output.dropout
        z = Fn.dropout_add(h, a, drop.p) if (self.training and drop.p > 0) else Fn.add(h, a)
        return self.self_output.LayerNorm(z).view(input_tensor.shape)


class BertPfeifferAdaptedSelfOutput(nn.Module):
    """model.py:300-329 (wraps layer.output only, run.py:403-406): h = dropout(dense(x)); t = LayerNorm(h + input);
    LN(adapter(t) + h + input) with a residual-free bottleneck (AdapterPfeifferBlock) and a NEW LayerNorm `LN`
    (eps 1e-6)."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterPfeifferBlock(args, _word_dim(args), args.bert_adapter_down_size, args.adapter_dropout_rate)
        self.LN = LayerNorm(_word_dim(args), eps=1e-06)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        inp = to_2d_bf16(input_tensor).contiguous()
        h = to_2d_bf16(h)
        drop = self.self_output.dropout
        hi = Fn.dropout_add(h, inp, drop.p) if (self.training and drop.p > 0) else Fn.add(h, inp)   # h + input
        t = self.self_output.LayerNorm(hi)
        return self.LN(self.adapter(t, extra_residual=hi)).view(input_tensor.shape)


class SASRecAdaptedSelfOutput(nn.Module):
    """model.py:332-376: the SASRec block with adapter1 after fc and adapter2 after the feed-forward, both before the
    LayerNorms."""

    def __init__(self, transformer_block, args):
        super().__init__()
        self.transformer_block = transformer_block
        self.adapter1 = AdapterBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)
        self.adapter2 = AdapterBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)

    def forward(self, block_input, mask):
        tb = self.transformer_block
        h = tb.multi_head_attention(block_input, block_input, block_input, mask, adapter=self.adapter1)
        return tb.feed_forward(h, adapter=self.adapter2)


class SASRecPfeifferVer2AdaptedSelfOutput(nn.Module):
    """model.py:379-423 (adapter_type 'pfeiffer_ver2', run.py:389-399): only adapter1 (after the attention's fc); the
    feed-forward half is the plain block."""

    def __init__(self, transformer_block, args):
        super().__init__()
        self.transformer_block = transformer_block
        self.adapter1 = AdapterBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)

    def forward(self, block_input, mask):
        tb = self.transformer_block
        h = tb.multi_head_attention(block_input, block_input, block_input, mask, adapter=self.adapter1)
        return tb.feed_forward(h)


class SASRecPfeifferAdaptedSelfOutput(nn.Module):
    """model.py:426-471: plain attention half; feed-forward half h = dropout(ffn(y)), t = layer_norm(y + h),
    LN(adapter(t) + h + y) with AdapterPfeifferBlock and a new LayerNorm `LN` (eps 1e-6)."""

    def __init__(self, transformer_block, args):
        super().__init__()
        self.transformer_block = transformer_block
        self.adapter = AdapterPfeifferBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)
        self.LN = LayerNorm(args.embedding_dim, eps=1e-06)

    def forward(self, block_input, mask):
        tb = self.transformer_block
        y = tb.multi_head_attention(block_input, block_input, block_input, mask)
        ff = tb.feed_forward
        hy = ff.presum(to_2d_bf16(y))                                   # y + dropout(ffn(y))
        t = ff.layer_norm(hy)
        return self.LN(self.adapter(t, extra_residual=hy)).view(block_input.shape)


class SASRecParallelAdaptedSelfOutput(nn.Module):
    """model.py:474-520: both adapters read the sub-block INPUT: layer_norm(adapter1(x) + x + dropout(fc(attn(x)))),
    then layer_norm(adapter2(y) + y + dropout(ffn(y))); adapter(x) already contains + x."""

    def __init__(self, transformer_block, args):
        super().__init__()
        self.transformer_block = transformer_block
        self.adapter1 = AdapterBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)
        self.adapter2 = AdapterBlock(args, args.embedding_dim, args.adapter_down_size, args.adapter_dropout_rate)

    def forward(self, block_input, mask):
        tb = self.transformer_block
        B, S, D = block_input.shape
        x2 = to_2d_bf16(block_input).contiguous()
        a1 = to_2d_bf16(self.adapter1(x2, extra_residual=x2))           # up(act(down(x))) + x + x
        mha, ff = tb.multi_head_attention, tb.feed_forward
        y = mha.layer_norm(mha.presum(x2, mask, B, S, extra=a1))
        a2 = to_2d_bf16(self.adapter2(y, extra_residual=y))
        return ff.layer_norm(ff.presum(y, extra=a2)).view(B, S, D)


class BertCompacterAdaptedSelfOutput(nn.Module):
    """model.py:696-720: LayerNorm(adapter(dropout(dense(x))) + input) with the residual-free HyperComplexAdapterBlock
    (the dense output reaches the LayerNorm only THROUGH the adapter, as in the reference)."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = HyperComplexAdapterBlock(args, _word_dim(args), args.bert_adapter_down_size)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        h = to_2d_bf16(h)
        drop = self.self_output.dropout
        if self.training and drop.p > 0:
            h = Fn.dropout_add(h, None, drop.p)
        z = self.adapter(h, extra_residual=to_2d_bf16(input_tensor).contiguous())
        return self.self_output.LayerNorm(z).view(input_tensor.shape)


class SASRecCompacterAdaptedSelfOutput(nn.Module):
    """model.py:650-693: the serial-Houlsby placement with HyperComplexAdapterBlocks (no inner residual)."""

    def __init__(self, transformer_block, args):
        super().__init__()
        self.transformer_block = transformer_block
        self.adapter1 = HyperComplexAdapterBlock(args, args.embedding_dim, args.adapter_down_size)
        self.adapter2 = HyperComplexAdapterBlock(args, args.embedding_dim, args.adapter_down_size)

    def forward(self, block_input, mask):
        tb = self.transformer_block
        h = tb.multi_head_attention(block_input, block_input, block_input, mask, adapter=self.adapter1)
        return tb.feed_forward(h, adapter=self.adapter2)


class CompacterModel(nn.Module):
    """Downstream/Text/run.py:70-81 (the reference defines it in the entry script): owns the shared phm_rule
    [n, n, n] ~ N(0, phm_init_range²), hands it to every PHMLinear, and forwards to the wrapped model (reached as
    `.model` by data_utils/metrics.py:72-73,101-102)."""

    def __init__(self, args, model):
        super().__init__()
        phm_dim = args.hypercomplex_division
        self.model = model
        self.phm_rule = nn.Parameter(torch.empty(phm_dim, phm_dim, phm_dim).normal_(mean=0, std=args.phm_init_range))
        for name, sub_module in model.named_modules():
            if isinstance(sub_module, PHMLinear):
                sub_module.set_phm_rule(phm_rule=self.phm_rule)

    def forward(self, sample_items, log_mask, local_rank=None):
        return self.model(sample_items, log_mask, local_rank)


class BertKAdaptedBertModel(nn.Module):
    """model.py:523-561 (K-Adapter; replaces `text_encoders.title.bert_model` itself, run.py:410-411): adapters run
    OUTSIDE the frozen body on its intermediate hidden states: for k in k_adapter_bert_list (+1, i.e. the OUTPUT of that
    layer): last = adapter_k(hidden_states[k] + last); result = com_dense([sequence_output | last])."""

    def __init__(self, bert_model, args):
        super().__init__()
        word_embedding_dim = _word_dim(args)
        self.bert_model = bert_model
        self.k_adapter_num_list = [int(i) + 1 for i in list(args.k_adapter_bert_list.split(","))]
        self.bert_adapter_list = nn.ModuleList([KAdapterBlock(args, args.num_adapter_heads_bert, word_embedding_dim,
                                                              args.k_adapter_bert_hidden_dim, args.adapter_dropout_rate)
                                                for i in self.k_adapter_num_list])
        self.com_dense = Linear(word_embedding_dim * 2, word_embedding_dim)

    def forward(self, input_ids, attention_mask):
        outputs = self.bert_model(input_ids, attention_mask, output_hidden_states=True)
        sequence_output, hidden_states = outputs[0], outputs[2]
        hidden_states_last = None                                  # the reference starts from zeros: x + 0 == x
        for index, adapter in enumerate(self.bert_adapter_list):
            hs = hidden_states[self.k_adapter_num_list[index]]
            fusion_state = hs if hidden_states_last is None else Fn.add(to_2d_bf16(hs), to_2d_bf16(hidden_states_last)).view(hs.shape)
            hidden_states_last = adapter(fusion_state)
        if hidden_states_last is None:
            hidden_states_last = torch.zeros_like(sequence_output)
        input_embs_all = self.com_dense(torch.cat([sequence_output, hidden_states_last], dim=2))
        return input_embs_all, outputs[1], outputs[2]


class SASRecKAdaptedTransformerBlocks(nn.Module):
    """model.py:564-583 (replaces `transformer_encoder.transformer_blocks`, run.py:412-413): before each block,
    last = adapter_i(output + last); after the blocks, com_dense2([output | last])."""

    def __init__(self, transformer_blocks, args):
        super().__init__()
        self.transformer_blocks = transformer_blocks
        self.len_transformer_blocks = self.transformer_blocks.__len__()
        self.adapter_list = nn.ModuleList([KAdapterBlock(args, args.num_adapter_heads_sasrec, args.embedding_dim,
                                                         args.adapter_down_size, args.drop_rate)
                                           for _ in range(self.len_transformer_blocks)])
        self.com_dense2 = Linear(args.embedding_dim * 2, args.embedding_dim)

    def forward(self, output, att_mask):
        hidden_states_last = None
        for index, transformer in enumerate(self.transformer_blocks):
            fusion_state = output if hidden_states_last is None else \
                Fn.add(to_2d_bf16(output), to_2d_bf16(hidden_states_last)).view(output.shape)
            hidden_states_last = self.adapter_list[index](fusion_state)
            output = transformer(output, att_mask)
        return self.com_dense2(torch.cat([output, hidden_states_last], dim=2))


class SoftEmbedding(nn.Module):
    """model.py:586-630: the first n_tokens word embeddings of every item are REPLACED by learned vectors
    (tokens[:, n_tokens:] keeps the rest).  The substitution happens inside the fused embedding kernel; this module
    owns the parameters (`wte.weight`, `learned_embedding`)."""

    def __init__(self, wte, n_tokens=100, random_range=0.5, initialize_from_vocab=True):
        super().__init__()
        self.wte = wte
        self.n_tokens = n_tokens
        self.learned_embedding = nn.parameter.Parameter(
            self.initialize_embedding(wte, n_tokens, random_range, initialize_from_vocab))

    def initialize_embedding(self, wte, n_tokens=100, random_range=0.5, initialize_from_vocab=True):
        if initialize_from_vocab:
            return self.wte.weight[:n_tokens].clone().detach()
        return torch.FloatTensor(n_tokens, wte.weight.size(1)).uniform_(-random_range, random_range)
