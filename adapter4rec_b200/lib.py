"""ctypes binding of libadapter4rec_sm100.so (the C ABI declared in include/adapter4rec.h).

There is no fallback: if the shared library is missing, or a call fails, a RuntimeError is raised."""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libadapter4rec_sm100.so")

A4R_OK, A4R_EINVAL, A4R_ECUDA, A4R_EARCH, A4R_EWORKSPACE = 0, -1, -2, -3, -4
EPI_LINEAR, EPI_GELU, EPI_RELU, EPI_DGELU, EPI_DRELU = 0, 1, 2, 3, 4


class GemmArgs(Structure):
    _fields_ = [
        ("A", c_void_p), ("lda", c_int64), ("B", c_void_p), ("ldb", c_int64),
        ("A2", c_void_p), ("lda2", c_int64), ("B2", c_void_p), ("ldb2", c_int64), ("K2", c_int64),
        ("C", c_void_p), ("ldc", c_int64), ("aux", c_void_p), ("ldaux", c_int64),
        ("residual", c_void_p), ("ldr", c_int64), ("residual2", c_void_p), ("ldr2", c_int64),
        ("bias", c_void_p), ("M", c_int64), ("N", c_int64), ("K", c_int64),
        ("alpha", c_float), ("epilogue", c_int32), ("out_f32", c_int32), ("block_n", c_int32),
        ("dropout_p", c_float), ("dropout_seed", ctypes.c_uint64), ("dropout_offset", ctypes.c_uint64),
        ("dropout_after_residual", c_int32),
    ]


class AttnArgs(Structure):
    _fields_ = [
        ("qkv", c_void_p), ("out", c_void_p), ("dout", c_void_p), ("mask", c_void_p),
        ("ld_qkv", c_int64), ("ld_out", c_int64), ("mask_ld", c_int64),
        ("N", c_int64), ("L", c_int64), ("heads", c_int64), ("head_dim", c_int64),
        ("mask_dtype", c_int32), ("causal", c_int32), ("scale", c_float), ("mask_neg", c_float),
        ("lse", c_void_p), ("ctx", c_void_p),
        ("dropout_p", c_float), ("dropout_seed", ctypes.c_uint64), ("dropout_offset", ctypes.c_uint64),
        ("cu_seqlens", c_void_p),
    ]


class EmbedArgs(Structure):
    _fields_ = [
        ("ids", c_void_p), ("ld_ids", c_int64), ("word_emb", c_void_p), ("pos_emb", c_void_p),
        ("type_emb", c_void_p), ("prompt", c_void_p), ("gamma", c_void_p), ("beta", c_void_p),
        ("out", c_void_p), ("z_out", c_void_p), ("mean_out", c_void_p), ("rstd_out", c_void_p),
        ("N", c_int64), ("L", c_int64), ("H", c_int64), ("pos_offset", c_int64),
        ("roberta_pad_id", c_int64), ("n_prompt", c_int64), ("eps", c_float),
    ]


class BceArgs(Structure):
    _fields_ = [
        ("prec", c_void_p), ("emb", c_void_p), ("log_mask", c_void_p), ("pos_score", c_void_p),
        ("neg_score", c_void_p), ("loss", c_void_p), ("count", c_void_p),
        ("B", c_int64), ("S", c_int64), ("D", c_int64), ("cpc", c_int32),
    ]


class AdapterArgs(Structure):
    _fields_ = [
        ("h", c_void_p), ("ldh", c_int64), ("input", c_void_p), ("ldi", c_int64),
        ("w_down", c_void_p), ("b_down", c_void_p), ("w_up", c_void_p), ("b_up", c_void_p),
        ("gamma", c_void_p), ("beta", c_void_p), ("out", c_void_p), ("z_out", c_void_p),
        ("mean", c_void_p), ("rstd", c_void_p), ("s_out", c_void_p), ("u_out", c_void_p),
        ("M", c_int64), ("H", c_int64), ("r", c_int64), ("act", c_int32), ("tail", c_int32), ("eps", c_float),
        ("lds", c_int64),
    ]


class InbatchCeArgs(Structure):
    _fields_ = [
        ("prec", c_void_p), ("cand", c_void_p), ("ld_cand", c_int64), ("item_ids", c_void_p), ("log_mask", c_void_p),
        ("cand_bias", c_void_p), ("lse", c_void_p), ("loss", c_void_p), ("count", c_void_p),
        ("B", c_int64), ("S", c_int64), ("D", c_int64), ("masked_logit", c_float),
    ]


# name -> (restype, argtypes); every symbol include/adapter4rec.h declares must appear here
# (tests/test_abi.py checks header <-> table <-> .so agreement).
PROTOTYPES = {
    "a4r_version": (c_int32, []),
    "a4r_last_error_string": (c_char_p, []),
    "a4r_device_check": (c_int32, []),
    "a4r_launch_count": (c_int64, []),
    "a4r_gemm_bf16_tn": (c_int32, [POINTER(GemmArgs), c_void_p]),
    "a4r_attn_small_fwd": (c_int32, [POINTER(AttnArgs), c_void_p]),
    "a4r_attn_small_bwd": (c_int32, [POINTER(AttnArgs), c_void_p]),
    "a4r_attn_mid_fwd": (c_int32, [POINTER(AttnArgs), c_void_p]),
    "a4r_attn_mid_bwd": (c_int32, [POINTER(AttnArgs), c_void_p]),
    "a4r_layernorm_fwd": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "a4r_layernorm_bwd_workspace_bytes": (c_size_t, [c_int64]),
    "a4r_layernorm_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_int32, c_void_p, c_size_t, c_int64, c_int64, c_void_p, c_float, ctypes.c_uint64,
                                    ctypes.c_uint64, c_void_p]),
    "a4r_layernorm_bwd_add": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                        c_void_p]),
    "a4r_adapter_ln_supported": (c_int32, [c_int64, c_int64]),
    "a4r_adapter_ln_fwd": (c_int32, [POINTER(AdapterArgs), c_void_p]),
    "a4r_embed_ln_fwd": (c_int32, [POINTER(EmbedArgs), c_void_p]),
    "a4r_act_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "a4r_act_fwd": (c_int32, [c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "a4r_scatter_add_rows": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "a4r_cast_transpose_f32_bf16": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "a4r_dropout": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_float, ctypes.c_uint64, ctypes.c_uint64, c_void_p]),
    "a4r_colsum_workspace_bytes": (c_size_t, [c_int64]),
    "a4r_colsum": (c_int32, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int32, c_void_p, c_size_t, c_void_p]),
    "a4r_wgrad_tc_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "a4r_wgrad_tc_bf16": (c_int32, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                    c_float, c_int32, c_void_p, c_size_t, c_void_p]),
    "a4r_bce_workspace_bytes": (c_size_t, []),
    "a4r_bce_loss_fwd": (c_int32, [POINTER(BceArgs), c_void_p, c_size_t, c_void_p]),
    "a4r_bce_loss_bwd": (c_int32, [POINTER(BceArgs), c_void_p, c_void_p, c_void_p, c_void_p]),
    "a4r_inbatch_ce_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "a4r_inbatch_ce_fwd": (c_int32, [POINTER(InbatchCeArgs), c_void_p, c_size_t, c_void_p]),
    "a4r_inbatch_ce_bwd": (c_int32, [POINTER(InbatchCeArgs), c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "a4r_adam_step": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                                c_float, c_int64, c_float, c_void_p]),
    "a4r_adam_step_dev": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                                    c_float, c_void_p, c_float, c_void_p]),
    "a4r_patchify": (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "a4r_vit_assemble": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                   c_void_p]),
    "a4r_gather_rows": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "a4r_sample_train_batch": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                         c_int64, c_int64, c_int64, ctypes.c_uint64, ctypes.c_uint64, c_void_p]),
    "a4r_id_embed_fwd": (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "a4r_id_embed_bwd": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                   c_int64, c_int32, c_void_p]),
    "a4r_score_topk_partials": (c_int32, [c_int64, c_int64]),
    "a4r_score_topk": (c_int32, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_void_p,
                                 c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "a4r_topk_merge": (c_int32, [c_void_p, c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
}

_lib = None


def get_lib():
    """Load the shared library once; fail loudly if it has not been built (run `python -m adapter4rec_b200._build`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "adapter4rec_b200: %s is missing — build it with __graft_entry__.build() "
                "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def check(rc, what):
    if rc != A4R_OK:
        msg = get_lib().a4r_last_error_string()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else ""))


def launch_count():
    return int(get_lib().a4r_launch_count())
