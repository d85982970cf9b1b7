"""Adapter insertion, mirroring the in-place module surgery of Downstream/Text/run.py:367-479 (which lives inside
train() in the reference and is therefore restated here as a function with the same flag semantics)."""
from .model.layers import LoRALinear
from .model.model import (BertAdaptedParallelSelfOutput, BertAdaptedSelfOutput, BertCompacterAdaptedSelfOutput,
                          BertKAdaptedBertModel, SASRecKAdaptedTransformerBlocks,
                          BertPfeifferAdaptedSelfOutput, CompacterModel, SASRecCompacterAdaptedSelfOutput,
                          SASRecAdaptedSelfOutput, SASRecParallelAdaptedSelfOutput, SASRecPfeifferAdaptedSelfOutput,
                          SASRecPfeifferVer2AdaptedSelfOutput, SoftEmbedding)


ID_TOWER_ADAPTERS = ("item_tower 'id' has no item-encoder body to insert adapters into: use --adding_adapter_to None "
                     "(an id run trains the embedding table and the user encoder, --fine_tune_to all)")


def freeze_all(model):
    """fine_tune_to = 'None' (run.py:368-371)."""
    for _, param in model.named_parameters():
        param.requires_grad = False


def insert_adapters(model, args, log=None):
    """Dispatch on args.adapter_type by SUBSTRING, in the reference's order and with its spelling 'houslby'
    (run.py:389-452; SURVEY.md Appendix B-2).  New modules are trainable by default."""
    if 'None' in getattr(args, "adding_adapter_to", "bert"):
        return model
    if not getattr(model, "use_modal", True):
        raise ValueError(ID_TOWER_ADAPTERS)
    bert = model.bert_encoder.text_encoders.title.bert_model
    layers = bert.encoder.layer
    blocks = model.user_encoder.transformer_encoder.transformer_blocks
    t = args.adapter_type
    dev = next(model.parameters()).device
    if "pfeiffer_ver2" in t:                                           # run.py:389-399
        for lm in layers:
            lm.attention.output = BertAdaptedSelfOutput(lm.attention.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = SASRecPfeifferVer2AdaptedSelfOutput(blocks[i], args).to(dev)
    elif "pfeiffer" in t:                                              # run.py:400-409
        for lm in layers:
            lm.output = BertPfeifferAdaptedSelfOutput(lm.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = SASRecPfeifferAdaptedSelfOutput(blocks[i], args).to(dev)
    elif 'kadapter' in t:                                              # run.py:409-413
        title = model.bert_encoder.text_encoders.title
        title.bert_model = BertKAdaptedBertModel(title.bert_model, args).to(dev)
        te = model.user_encoder.transformer_encoder
        te.transformer_blocks = SASRecKAdaptedTransformerBlocks(te.transformer_blocks, args).to(dev)
    elif "lora" in t:                                                  # run.py:414-428
        for lm in layers:
            lm.attention.self.query = LoRALinear(args.word_embedding_dim, args.word_embedding_dim,
                                                 r=args.bert_adapter_down_size).to(dev)
            lm.attention.self.value = LoRALinear(args.word_embedding_dim, args.word_embedding_dim,
                                                 r=args.bert_adapter_down_size).to(dev)
        for i in range(len(blocks)):
            blocks[i].multi_head_attention.w_Q = LoRALinear(args.embedding_dim, args.embedding_dim,
                                                            r=args.adapter_down_size).to(dev)
            blocks[i].multi_head_attention.w_V = LoRALinear(args.embedding_dim, args.embedding_dim,
                                                            r=args.adapter_down_size).to(dev)
    elif "prompt" in t:                                                # run.py:429-434
        s_wte = SoftEmbedding(bert.get_input_embeddings(), n_tokens=args.n_tokens, initialize_from_vocab=True)
        bert.set_input_embeddings(s_wte.to(dev))
    elif "compacter" in t:                                             # run.py:435-450: returns the WRAPPED model
        for lm in layers:
            lm.attention.output = BertCompacterAdaptedSelfOutput(lm.attention.output, args).to(dev)
            lm.output = BertCompacterAdaptedSelfOutput(lm.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = SASRecCompacterAdaptedSelfOutput(blocks[i], args).to(dev)
        model = CompacterModel(args, model).to(dev)
    elif "houslby" in t:                                               # run.py:452-465
        serial = "None" not in getattr(args, "is_serial", "True")       # run.py:454 vs :466
        bert_cls = BertAdaptedSelfOutput if serial else BertAdaptedParallelSelfOutput
        rec_cls = SASRecAdaptedSelfOutput if serial else SASRecParallelAdaptedSelfOutput
        for lm in layers:
            lm.attention.output = bert_cls(lm.attention.output, args).to(dev)
            lm.output = bert_cls(lm.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = rec_cls(blocks[i], args).to(dev)
    return model


def unfreeze_layernorm(model, args):
    """finetune_layernorm (run.py:494-501)."""
    if "None" not in getattr(args, "adding_adapter_to", "bert") and 'None' not in getattr(args, "finetune_layernorm", "None"):
        for name, param in model.named_parameters():
            if "adapter" not in name and ("LayerNorm" in name or "layer_norm" in name):
                param.requires_grad = True


def insert_adapters_cv(model, args):
    """Image tree: Downstream/CV/run_adapter.py:367-470 (houslby serial, lora with its hard-coded ranks r=12 / r=4 / r=0,
    prompt which also unfreezes the classifier)."""
    from .cv.model import SASRecAdaptedSelfOutput as _SAS
    from .cv.model import (SoftPrompt, VITAdaptedOutput, VITAdaptedParallelOutput, VITAdaptedSelfOutput,
                           VITCompacterAdaptedOutput, VITCompacterAdaptedSelfOutput)
    if 'None' in getattr(args, "adding_adapter_to", "all"):
        return model
    if not getattr(model, "use_modal", True):
        raise ValueError(ID_TOWER_ADAPTERS)
    net = model.cv_encoder.image_net
    layers = net.vit.encoder.layer
    blocks = model.user_encoder.transformer_encoder.transformer_blocks
    t = args.adapter_type
    dev = next(model.parameters()).device
    if "pfeiffer_ver2" in t:                                           # run_adapter.py:367-377
        for lm in layers:
            lm.attention.output = VITAdaptedSelfOutput(lm.attention.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = SASRecPfeifferVer2AdaptedSelfOutput(blocks[i], args).to(dev)
    elif "kadapter" in t:
        # run_adapter.py:378-382 replaces vit.encoder by VITKAdaptedCVModel, whose forward calls the transformers ViT
        # encoder with a signature the installed transformers no longer has (SURVEY.md §8c probe p4: the reference itself
        # fails here), so there is no reference output to pin this variant to
        raise NotImplementedError("adapter_type 'kadapter' on the image tree: the reference's own VITKAdaptedCVModel does "
                                  "not run under the installed transformers; text-tree kadapter is implemented")
    elif "lora" in t:                                                  # run_adapter.py:383-395
        for lm in layers:
            lm.attention.attention.query = LoRALinear(768, 768, r=12).to(dev)
            lm.attention.attention.value = LoRALinear(768, 768, r=12).to(dev)
        for i in range(len(blocks)):
            blocks[i].multi_head_attention.w_Q = LoRALinear(args.embedding_dim, args.embedding_dim, r=4).to(dev)
            blocks[i].multi_head_attention.w_V = LoRALinear(args.embedding_dim, args.embedding_dim).to(dev)   # r = 0
    elif "compacter" in t:                                             # run_adapter.py:396-411: returns the WRAPPED model
        for lm in layers:
            lm.attention.output = VITCompacterAdaptedSelfOutput(lm.attention.output, args).to(dev)
            lm.output = VITCompacterAdaptedOutput(lm.output, args).to(dev)
        for i in range(len(blocks)):
            blocks[i] = SASRecCompacterAdaptedSelfOutput(blocks[i], args).to(dev)
        model = CompacterModel(args, model).to(dev)
    elif "prompt" in t:                                                # run_adapter.py:413-421
        net.vit.embeddings = SoftPrompt(net.vit.embeddings, n_tokens=args.n_tokens, embed_dim=768).to(dev)
        for name, param in model.named_parameters():
            if "cv_encoder.image_net.classifier" in name:
                param.requires_grad = True
    elif "houslby" in t:                                               # run_adapter.py:423-445
        if "None" not in getattr(args, "is_serial", "True"):
            for lm in layers:
                lm.attention.output = VITAdaptedSelfOutput(lm.attention.output, args).to(dev)
                lm.output = VITAdaptedOutput(lm.output, args).to(dev)
            for i in range(len(blocks)):
                blocks[i] = _SAS(blocks[i], args).to(dev)
        else:                                                          # parallel: layer.output only (:236-247)
            for lm in layers:
                lm.output = VITAdaptedParallelOutput(lm.output, args).to(dev)
            for i in range(len(blocks)):
                blocks[i] = SASRecParallelAdaptedSelfOutput(blocks[i], args).to(dev)
    return model
