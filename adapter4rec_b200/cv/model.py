"""CV (image) TransRec model classes, mirroring Downstream/CV/model/{model,encoders}.py."""
import torch
import torch.nn as nn

from .. import functional as Fn
from ..model.encoders import User_Encoder
from ..model.layers import BF16, IdEmbedding, to_2d_bf16
from ..model.model import (CompacterModel, SASRecAdaptedSelfOutput, SASRecCompacterAdaptedSelfOutput,  # noqa: F401
                           SASRecParallelAdaptedSelfOutput, SASRecPfeifferVer2AdaptedSelfOutput,
                           check_trainable_supported)   # the SASRec wrappers are the text tree's classes (CV model.py:235-372,465-510)
from ..model.modules import AdapterBlock, HyperComplexAdapterBlock

SASRecPfeifferV2AdaptedSelfOutput = SASRecPfeifferVer2AdaptedSelfOutput   # the CV tree's spelling (CV model.py:283)


class _Act:
    """GELU applied to the classifier output: evaluated by the elementwise kernel pair (forward inside a GEMM epilogue is
    not possible here because `classifier` is a caller-provided module)."""


class Vit_Encoder(nn.Module):
    """encoders.py:25-32: GELU(image_net(images)[0])."""

    def __init__(self, image_net):
        super().__init__()
        self.image_net = image_net
        self.activate = nn.GELU()

    def forward(self, item_content):
        net = self.image_net
        # fuse the GELU into the classifier GEMM's epilogue when the classifier is one of our Linear-compatible modules
        hidden = net.vit(item_content, cls_only=True)[0]
        clf = net.classifier
        if not hasattr(clf, "_cache"):
            clf._cache = Fn.WeightCache()
        return Fn.linear(to_2d_bf16(hidden[:, 0]), clf.weight, clf.bias, clf._cache, act="gelu")


class _ModelBase(nn.Module):
    cpc = False

    def __init__(self, args, item_num, use_modal, image_net):
        super().__init__()
        self.args = args
        self.use_modal = use_modal
        self.max_seq_len = args.max_seq_len
        self.l2_weight = args.l2_weight / 2
        self.user_encoder = User_Encoder(item_num=item_num, max_seq_len=args.max_seq_len, item_dim=args.embedding_dim,
                                         num_attention_heads=args.num_attention_heads, dropout=args.drop_rate,
                                         n_layers=args.transformer_block)
        if not use_modal:                               # --item_tower id: the item table is a trainable embedding
            self.id_embedding = IdEmbedding(item_num + 1, args.embedding_dim, padding_idx=0)
        elif 'vit' not in args.CV_model_load:
            raise NotImplementedError("only the ViT image encoder is on the hot path (CV_model_load=%r)" % args.CV_model_load)
        else:
            self.cv_encoder = Vit_Encoder(image_net=image_net)
        self.criterion = nn.BCEWithLogitsLoss()
        self._checked = None

    def forward(self, sample_items, log_mask, local_rank=None):
        """sample_items f32 [B*(S+1)*2, 3, R, R] (the id tower: int64 item ids [B*(S+1)*2] or [B, S+1, 2]); log_mask f32
        [B,S] -> scalar loss (Downstream/CV/model/model.py:54-77)."""
        if self.training:
            sig = tuple(p.requires_grad for p in self.parameters())
            if sig != self._checked:
                check_trainable_supported(self)
                self._checked = sig
        if not self.use_modal:
            input_embs, input_logs_embs = self.id_embedding(sample_items.reshape(-1, self.max_seq_len + 1, 2))
        else:
            input_embs_all = self.cv_encoder(sample_items)
            input_embs = input_embs_all.view(-1, self.max_seq_len + 1, 2, self.args.embedding_dim)
            input_logs_embs = input_embs[:, :-1, 0, :].contiguous()
        log_mask = log_mask.to(device=input_embs.device, dtype=torch.float32).contiguous()
        prec_vec = self.user_encoder(input_logs_embs, log_mask, local_rank)
        return Fn.bce_loss(prec_vec.contiguous(), input_embs.contiguous(), None if self.cpc else log_mask, cpc=self.cpc)


class Model(_ModelBase):
    cpc = False


class ModelCPC(_ModelBase):
    cpc = True


class VITAdaptedSelfOutput(nn.Module):
    """Downstream/CV/model/model.py:182-195: adapter(dense(x)); no residual, no LayerNorm (ViT is pre-LN)."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, 768, args.cv_adapter_down_size, args.adapter_dropout_rate)

    def _dense(self, hidden_states):
        """dense + the wrapped module's nn.Dropout (model.py:191-193; ViT's default probability is 0: then nothing is launched)"""
        h = self.self_output.dense(hidden_states)
        p = self.self_output.dropout.p if self.training else 0.0
        return Fn.dropout_add(to_2d_bf16(h), None, p).view(h.shape) if p > 0 else h

    def forward(self, hidden_states, input_tensor=None):
        return self.adapter(self._dense(hidden_states))

    def forward_fused(self, hidden_states, residual):
        h = self._dense(to_2d_bf16(hidden_states))
        return to_2d_bf16(self.adapter(h, extra_residual=to_2d_bf16(residual)))


class VITAdaptedOutput(nn.Module):
    """Downstream/CV/model/model.py:198-212: adapter(dense(x)) + input."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, 768, args.cv_adapter_down_size, args.adapter_dropout_rate)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        h = to_2d_bf16(h)
        p = self.self_output.dropout.p if self.training else 0.0     # model.py:207-209: dropout sits between dense and the adapter
        if p > 0:
            h = Fn.dropout_add(h, None, p)
        return self.adapter(h, extra_residual=to_2d_bf16(input_tensor)).view(input_tensor.shape)


class VITAdaptedParallelSelfOutput(nn.Module):
    """Downstream/CV/model/model.py:149-162: adapter(input) + dropout(dense(x)) (the layer adds its skip afterwards).
    Defined by the reference but not dispatched by run_adapter.py (its use at :240 is commented out)."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, 768, args.cv_adapter_down_size, args.adapter_dropout_rate)

    def forward_fused(self, hidden_states, residual):
        inp = to_2d_bf16(residual).contiguous()
        a = to_2d_bf16(self.adapter(inp, extra_residual=inp))         # adapter(inp) + the layer's skip connection
        h = self.self_output.dense(to_2d_bf16(hidden_states))
        p = self.self_output.dropout.p if self.training else 0.0
        return Fn.dropout_add(h, a, p) if p > 0 else Fn.add(h, a)

    def forward(self, hidden_states, input_tensor):
        inp = to_2d_bf16(input_tensor).contiguous()
        a = to_2d_bf16(self.adapter(inp))
        h = self.self_output.dense(to_2d_bf16(hidden_states))
        p = self.self_output.dropout.p if self.training else 0.0
        return (Fn.dropout_add(h, a, p) if p > 0 else Fn.add(h, a)).view(input_tensor.shape)


class VITAdaptedParallelOutput(nn.Module):
    """Downstream/CV/model/model.py:165-179 (is_serial = 'None' wraps layer.output ONLY, run_adapter.py:236-241):
    dropout(dense(x)) + input + adapter(input), adapter(x) = fc_up(act(fc_down(x))) + x."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = AdapterBlock(args, 768, args.cv_adapter_down_size, args.adapter_dropout_rate)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        inp = to_2d_bf16(input_tensor).contiguous()
        a = to_2d_bf16(self.adapter(inp, extra_residual=inp))
        h = to_2d_bf16(h)
        p = self.self_output.dropout.p if self.training else 0.0
        return (Fn.dropout_add(h, a, p) if p > 0 else Fn.add(h, a)).view(input_tensor.shape)


class VITCompacterAdaptedSelfOutput(nn.Module):
    """Downstream/CV/model/model.py:432-445: adapter(dropout(dense(x))) with the residual-free HyperComplexAdapterBlock."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = HyperComplexAdapterBlock(args, 768, args.cv_adapter_down_size)

    def _dense(self, hidden_states):
        h = self.self_output.dense(to_2d_bf16(hidden_states))
        p = self.self_output.dropout.p if self.training else 0.0
        return Fn.dropout_add(h, None, p) if p > 0 else h

    def forward(self, hidden_states, input_tensor=None):
        return self.adapter(self._dense(hidden_states))

    def forward_fused(self, hidden_states, residual):
        return to_2d_bf16(self.adapter(self._dense(hidden_states), extra_residual=to_2d_bf16(residual).contiguous()))


class VITCompacterAdaptedOutput(nn.Module):
    """Downstream/CV/model/model.py:448-462: adapter(dropout(dense(x))) + input."""

    def __init__(self, self_output, args):
        super().__init__()
        self.self_output = self_output
        self.adapter = HyperComplexAdapterBlock(args, 768, args.cv_adapter_down_size)

    def forward(self, hidden_states, input_tensor):
        return self.forward_from_dense(self.self_output.dense(to_2d_bf16(hidden_states)), input_tensor)

    def forward_from_dense(self, h, input_tensor):
        h = to_2d_bf16(h)
        p = self.self_output.dropout.p if self.training else 0.0
        if p > 0:
            h = Fn.dropout_add(h, None, p)
        return self.adapter(h, extra_residual=to_2d_bf16(input_tensor).contiguous()).view(input_tensor.shape)


class SoftPrompt(nn.Module):
    """Downstream/CV/model/model.py:512-535: n learned tokens appended after [cls | patches] + positions."""

    def __init__(self, wte, n_tokens=10, embed_dim=768):
        super().__init__()
        self.wte = wte
        self.patch_embeddings = wte.patch_embeddings
        self.n_tokens = n_tokens
        self.Prompt_Tokens = nn.Parameter(torch.zeros(1, n_tokens, embed_dim))

    def tokens(self, pixel_values):
        return self.wte.tokens(pixel_values, prompt=self.Prompt_Tokens)

    def forward(self, pixel_values, bool_masked_pos=None, interpolate_pos_encoding=None):
        x, L = self.tokens(pixel_values)
        return x.view(pixel_values.shape[0], L, -1)


class VITKAdaptedCVModel(nn.Module):
    """Name kept so that run_adapter.py's import line (Downstream/CV/run_adapter.py:17-22) resolves.  The reference's own class
    (Downstream/CV/model/model.py:374-404) does not run under the installed transformers (its wrapped encoder is called with a
    signature that library no longer accepts; SURVEY.md §8c, probe p4), so there is nothing to pin an implementation to:
    constructing it says so, exactly as `surgery.insert_adapters_cv` does for --adapter_type kadapter."""

    def __init__(self, cv_model=None, args=None):
        super().__init__()
        raise NotImplementedError("VITKAdaptedCVModel: the reference's own class does not run under the installed "
                                  "transformers; the text tree's K-Adapter (BertKAdaptedBertModel) is implemented")


class VITPfeifferAdaptedSelfOutput(nn.Module):
    """Name kept for the same import line.  In the reference (model.py:215-232) the class is only reached through
    `add_pfeiffer_adapter_to_vit` (run_adapter.py:44-45), which no branch of the adapter dispatch calls (:367-445 has
    pfeiffer_ver2 / kadapter / lora / compacter / prompt / houslby): dead code there, not built here."""

    def __init__(self, self_output=None, args=None):
        super().__init__()
        raise NotImplementedError("VITPfeifferAdaptedSelfOutput is unreachable from run_adapter.py's dispatch "
                                  "(--adapter_type pfeiffer_ver2 uses VITAdaptedSelfOutput + SASRecPfeifferV2AdaptedSelfOutput)")
