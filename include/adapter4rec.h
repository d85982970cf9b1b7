/*
 * adapter4rec.h — C ABI of libadapter4rec_sm100.so
 *
 * B200 (sm_100a) kernels for the TransRec train + full-ranking-eval hot path of
 * westlake-repl/Adapter4Rec.  The reference is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md §2: "no native components"), so each entry point cites the reference Python
 * symbol (file:line under /root/reference) whose arithmetic it replaces; INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add at each of those call sites.
 *
 * Conventions (SURVEY.md §8b):
 *   - every pointer is a DEVICE pointer into caller-owned memory (the library never allocates
 *     or frees device memory and keeps no global state besides a per-process attribute cache);
 *   - tensors are contiguous row-major unless a leading dimension (`ld*`, in ELEMENTS) is given;
 *   - "bf16" = __nv_bfloat16, "f32" = float, ids are int64 (the reference passes LongTensor);
 *   - 16-byte alignment of every base pointer and of every row (ld * sizeof(elem) % 16 == 0);
 *   - kernels are enqueued asynchronously on `stream` (a cudaStream_t); no implicit sync;
 *   - return 0 on success, a negative A4R_E* code otherwise; a4r_last_error_string() gives the
 *     message (thread-local).  No exceptions cross the ABI.  There is NO CPU fallback and no
 *     dispatch to other architectures: on a device that is not sm_100 every call fails with
 *     A4R_EARCH.
 */
#ifndef ADAPTER4REC_H_
#define ADAPTER4REC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define A4R_OK 0
#define A4R_EINVAL (-1)     /* bad shape / alignment / null pointer / unsupported flag */
#define A4R_ECUDA (-2)      /* a CUDA runtime/driver call failed */
#define A4R_EARCH (-3)      /* current device is not compute capability 10.x */
#define A4R_EWORKSPACE (-4) /* workspace too small */

typedef void* a4r_stream_t; /* cudaStream_t */

#define A4R_API __attribute__((visibility("default")))

/* library version: major*10000 + minor*100 + patch */
A4R_API int a4r_version(void);
/* message of the last failing call on this thread ("" if none) */
A4R_API const char* a4r_last_error_string(void);
/* 0 if the current CUDA device can run this library (sm_100), A4R_EARCH otherwise */
A4R_API int a4r_device_check(void);
/* number of kernels this library has launched in this process (monotonic; bench.py's gpu_launches) */
A4R_API int64_t a4r_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * K2 / K4 / K7 / K11-dense: tcgen05 + TMA GEMM   C[M,N] = epi(alpha * (A·Bᵀ + A2·B2ᵀ) + bias)
 *
 * Replaces every nn.Linear on the path: BertSelfAttention.query/key/value (fused, N=2304),
 * BertSelfOutput.dense, BertIntermediate.dense(+GELU), BertOutput.dense (transformers, called from
 * Downstream/Text/model/encoders.py:53), Text_Encoder.fc(+GELU) (encoders.py:55-57), the SASRec
 * w_Q/w_K/w_V/fc/w_1/w_2 (modules.py:54-57,19-20), AdapterBlock.fc_down/fc_up (modules.py:131-134),
 * loralib.Linear (run.py:414-428: the rank-r term enters as the K-extension A2·B2ᵀ), and — with
 * B = Wᵀ stored [K_out, N_in] — their data gradients dX = dY·W.
 *
 * A [M,K] bf16 (lda), B [N,K] bf16 (ldb)  — both "K-major", i.e. nn.Linear's native [out,in].
 * Optional K-extension A2 [M,K2], B2 [N,K2] (K2 % 8 == 0) accumulated into the same tile.
 * Epilogue, with v = alpha*acc + bias[n] (bias f32 [N] or NULL):
 *   A4R_EPI_LINEAR : C = v + residual + residual2           (either may be NULL)
 *   A4R_EPI_GELU   : aux = v (if aux != NULL), C = gelu_erf(v)
 *   A4R_EPI_RELU   : C = max(v, 0)
 *   A4R_EPI_DGELU  : C = v * gelu_erf'(aux)                 (aux = saved pre-activation, bf16 [M,N]; bias must be NULL)
 *   A4R_EPI_DRELU  : C = aux > 0 ? v : 0                    (aux = saved ReLU output,   bf16 [M,N]; bias must be NULL)
 * C is bf16 (out_f32 = 0) or f32 (out_f32 = 1).  K % 8 == 0, N % 8 == 0; M, N, K tails are handled.
 * ------------------------------------------------------------------------------------------------ */
enum {
  A4R_EPI_LINEAR = 0,
  A4R_EPI_GELU = 1,
  A4R_EPI_RELU = 2,
  A4R_EPI_DGELU = 3,
  A4R_EPI_DRELU = 4
};

typedef struct a4r_gemm_args {
  const void* A;
  int64_t lda;
  const void* B;
  int64_t ldb;
  const void* A2;
  int64_t lda2;
  const void* B2;
  int64_t ldb2;
  int64_t K2;
  void* C;
  int64_t ldc;
  void* aux;
  int64_t ldaux;
  const void* residual;
  int64_t ldr;
  const void* residual2;
  int64_t ldr2;
  const float* bias;
  int64_t M, N, K;
  float alpha;
  int32_t epilogue;
  int32_t out_f32;
  int32_t block_n; /* 0 = auto; else 64, 128, 256 (one CTA per tile) or 512 (256 x 256 tile on a CTA pair, cta_group::2) */
  /* LINEAR epilogue only: dropout on v BEFORE the residuals (the `dense -> dropout -> + input` of BertSelfOutput /
   * BertOutput); element (row, col) uses the counter indexing of a4r_dropout over the logical [M, N] output */
  float dropout_p;
  uint64_t dropout_seed;
  uint64_t dropout_offset;
  /* 0: the mask is applied to v BEFORE the residuals (forward).  1: to v + residual + residual2 — the gradient through
   * a dropout whose input gradient is a sum that this GEMM forms in its epilogue (the fused Houlsby block's backward:
   * d_dense_out = (ds W_d + dz) * mask / (1 - p), Downstream/Text/model/model.py:293-295 read backwards) */
  int32_t dropout_after_residual;
} a4r_gemm_args;

A4R_API int a4r_gemm_bf16_tn(const a4r_gemm_args* args, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K3: whole-sequence attention for short sequences (L <= 32; head_dim 32 or 64), forward / backward.
 *
 * Replaces BertSelfAttention's softmax(q·kᵀ/√d + mask)·v (transformers, reached from
 * Downstream/Text/model/encoders.py:53) and SASRec's SelfAttention.forward
 * (Downstream/Text/model/modules.py:38-42) with the mask of User_Encoder.forward (encoders.py:25-28).
 *
 * qkv  [N*L, ld_qkv] bf16, columns q | k | v each heads*head_dim wide (the fused-QKV GEMM output).
 * mask [N, mask_ld]: non-zero = valid key; mask_dtype 0 none / 1 int64 / 2 f32.  The mask is ADDITIVE:
 *      score += mask_neg once if the key is masked or (causal and key index > query index).
 * fwd: out = ctx  [N*L, ld_out] bf16.
 * bwd: dout = dctx [N*L, ld_out] bf16, out = dqkv [N*L, ld_qkv] bf16 (dq | dk | dv); probabilities are
 *      recomputed from qkv, nothing else is saved by the forward.
 * ------------------------------------------------------------------------------------------------ */
typedef struct a4r_attn_args {
  const void* qkv;
  void* out;
  const void* dout;
  const void* mask;
  int64_t ld_qkv, ld_out, mask_ld;
  int64_t N, L, heads, head_dim;
  int32_t mask_dtype;
  int32_t causal;
  float scale;
  float mask_neg;
  float* lse;      /* mid-length kernel only: [N*L, heads] f32 log-sum-exp rows, written by fwd, required by bwd */
  const void* ctx; /* mid-length bwd only: the forward output [N*L, ld_out] */
  /* dropout on the attention probabilities (BertSelfAttention.dropout, SelfAttention.dropout modules.py:35,41; train
   * mode only): p = 0 disables it; the backward must be given the same (seed, offset) to regenerate the mask.
   * Short-sequence kernel only (ViT's dropout probability is 0). */
  float dropout_p;
  uint64_t dropout_seed;
  uint64_t dropout_offset;
  /* short-sequence kernel only — packed (variable-length) token layout: sequence n owns token rows
   * [cu_seqlens[n], cu_seqlens[n+1]) (int32 [N+1], device), each at most 32 long (L = that maximum); the mask, if given, is
   * indexed by token row.  Padded tokens — which HF BERT computes and then ignores (they are masked as keys and only
   * position 0 is read, encoders.py:53-55) — simply do not exist in this layout.  NULL = fixed length L per sequence. */
  const int32_t* cu_seqlens;
} a4r_attn_args;

A4R_API int a4r_attn_small_fwd(const a4r_attn_args* args, a4r_stream_t stream);
A4R_API int a4r_attn_small_bwd(const a4r_attn_args* args, a4r_stream_t stream);

/* Same contract for mid-length sequences (L <= 256, head_dim 64, causal = 0): ViT-B/16 attention with L = 197 (+ soft
 * prompt tokens), transformers' ViTSelfAttention reached from Vit_Encoder.forward (Downstream/CV/model/encoders.py:31-32).
 * One CTA per (sequence, head) keeps q, k, v (and dctx) in shared memory; flash-style online softmax. */
A4R_API int a4r_attn_mid_fwd(const a4r_attn_args* args, a4r_stream_t stream);
A4R_API int a4r_attn_mid_bwd(const a4r_attn_args* args, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K6: LayerNorm (biased variance, fp32 statistics) with an optional fused residual, forward / backward.
 *
 * Replaces nn.LayerNorm in BertSelfOutput/BertOutput (eps 1e-12; RoBERTa 1e-5), in the SASRec blocks and
 * TransformerEncoder (eps 1e-6; Downstream/Text/model/modules.py:21,61,96 and :105 where the residual is the
 * position embedding broadcast over users: res_rows = S).
 *
 * fwd: z = x + res[row % res_rows] (res may be NULL); y = LN(z).  x, res, y, z_out bf16 [M,H]; gamma/beta f32.
 *      z_out (optional) receives z rounded to bf16 — the tensor the backward reads; mean/rstd f32 [M] optional.
 * bwd: dz from dy, z, mean, rstd, gamma.  If dgamma/dbeta are non-NULL (finetune_layernorm,
 *      Downstream/Text/run.py:496-501) they receive (accumulate=0) or accumulate (=1) the parameter
 *      gradients via a deterministic two-stage reduction through `workspace`.  If dz_masked is non-NULL it receives
 *      dz * mask / (1 - p) with the a4r_dropout mask of (dropout_seed, dropout_offset): the gradient flowing through
 *      the dropout that precedes this LayerNorm's residual add (saves a separate pass over dz).
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_layernorm_fwd(const void* x, const void* res, int64_t res_rows, const float* gamma, const float* beta,
                      float eps, void* y, void* z_out, float* mean, float* rstd, int64_t M, int64_t H,
                      a4r_stream_t stream);
A4R_API size_t a4r_layernorm_bwd_workspace_bytes(int64_t H);
A4R_API int a4r_layernorm_bwd(const void* dy, const void* z, const float* mean, const float* rstd, const float* gamma,
                      void* dz, float* dgamma, float* dbeta, int32_t accumulate, void* workspace,
                      size_t workspace_bytes, int64_t M, int64_t H, void* dz_masked, float dropout_p,
                      uint64_t dropout_seed, uint64_t dropout_offset, a4r_stream_t stream);
/* dz = LayerNorm-backward(dy) + dskip: pre-LN blocks (ViT: x1 = x + f(LN(x)), transformers' ViTLayer reached from
 * Downstream/CV/model/encoders.py:31-32) deliver the skip-connection gradient to the LayerNorm's input; adding it here
 * replaces a separate elementwise pass over [M, H].  Frozen LayerNorm only (no dgamma / dbeta). */
A4R_API int a4r_layernorm_bwd_add(const void* dy, const void* z, const float* mean, const float* rstd, const float* gamma,
                          const void* dskip, void* dz, int64_t M, int64_t H, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K5: the Houlsby adapter block fused into one pass (tcgen05 down/up projections + residuals + LayerNorm).
 * Replaces everything after `self_output.dense` / `dropout` in BertAdaptedSelfOutput.forward
 * (Downstream/Text/model/model.py:292-297): AdapterBlock.forward (modules.py:131-134) + the residual add + LayerNorm;
 * and, with tail 1 / 2, VITAdaptedOutput.forward / VITAdaptedSelfOutput.forward (Downstream/CV/model/model.py:182-212).
 *
 *   s = act(h·W_dᵀ + b_d)          act 0 = ReLU, 1 = erf-GELU (args.adapter_activation, modules.py:122-125)
 *   z = s·W_uᵀ + b_u + h (+ input)
 *   tail 0: out = LayerNorm(z; gamma, beta, eps)     tail 1: out = z (input added)     tail 2: out = z (no input)
 *
 * h [M,H] bf16 (ldh), input [M,H] bf16 (ldi), w_down [r,H] bf16, w_up [H,r] bf16 (both contiguous, nn.Linear layout),
 * biases / gamma / beta f32, out [M,H] bf16 contiguous.  Optional outputs for the backward: z_out [M,H] bf16 (pre-LN sum,
 * tail 0), mean / rstd [M] f32 (tail 0), s_out [M,r] bf16 (activation output), u_out [M,r] bf16 (pre-activation; GELU).
 * lds (0 = r) is the row stride of s_out in elements; with lds >= r + 8 the kernel also writes [1, 0, ..., 0] into columns
 * [r, r + 8) of every row, so that ONE weight-gradient GEMM dzᵀ·[s | 1] yields d(fc_up.weight) and d(fc_up.bias) together.
 * Shapes: H %% 64 == 0, H <= 768, r %% 8 == 0, r <= 64 (a4r_adapter_ln_supported); other shapes compose
 * a4r_gemm_bf16_tn + a4r_layernorm_fwd.
 * impl selects the kernel formulation explicitly (no environment variables, no process state): 0 = default (the
 * row-per-thread TMA kernel where the shape allows it, else the staged kernel), 2 = staged kernel, 3 = row-per-thread kernel
 * (A4R_EINVAL if the shape is outside a4r_adapter_rows_supported).  Both formulations produce the same tensors.
 * ------------------------------------------------------------------------------------------------ */
typedef struct a4r_adapter_args {
  const void* h;
  int64_t ldh;
  const void* input;
  int64_t ldi;
  const void* w_down;
  const float* b_down;
  const void* w_up;
  const float* b_up;
  const float* gamma;
  const float* beta;
  void* out;
  void* z_out;
  float* mean;
  float* rstd;
  void* s_out;
  void* u_out;
  int64_t M, H, r;
  int32_t act;
  int32_t tail;
  float eps;
  int64_t lds;
  int32_t impl;
} a4r_adapter_args;
A4R_API int a4r_adapter_ln_supported(int64_t H, int64_t r);
A4R_API int a4r_adapter_ln_fwd(const a4r_adapter_args* args, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K1: token + position + token-type embedding gather fused with LayerNorm (BertEmbeddings /
 * RobertaEmbeddings, reached from Downstream/Text/model/encoders.py:53), with the soft-prompt
 * substitution of SoftEmbedding.forward (Downstream/Text/model/model.py:620-630).
 *
 * ids [N, ld_ids] int64 (the first L columns of the reference's [ids | mask] item rows).
 * word_emb [V,H], pos_emb [P,H], type_emb [H] (row 0; may be NULL) bf16.  Position id = t + pos_offset, or
 * — if roberta_pad_id >= 0 — pad + cumsum(ids != pad) for non-pad tokens and pad otherwise (L <= 32).
 * prompt [n_prompt,H] bf16 (may be NULL) replaces the word embedding of the first n_prompt positions.
 * out [N*L,H] bf16; z_out (pre-LN sum), mean_out, rstd_out optional (needed for the prompt gradient).
 * ------------------------------------------------------------------------------------------------ */
typedef struct a4r_embed_args {
  const int64_t* ids;
  int64_t ld_ids;
  const void* word_emb;
  const void* pos_emb;
  const void* type_emb;
  const void* prompt;
  const float* gamma;
  const float* beta;
  void* out;
  void* z_out;
  float* mean_out;
  float* rstd_out;
  int64_t N, L, H;
  int64_t pos_offset;
  int64_t roberta_pad_id;
  int64_t n_prompt;
  float eps;
} a4r_embed_args;
A4R_API int a4r_embed_ln_fwd(const a4r_embed_args* args, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K15 support: ViT patch embedding = im2col (this kernel) + a4r_gemm_bf16_tn.  ViTPatchEmbeddings.projection is a
 * ps x ps convolution with stride ps (transformers, reached from Vit_Encoder.forward,
 * Downstream/CV/model/encoders.py:31-32): images [N,C,R,R] f32 -> out [N*(R/ps)^2, C*ps*ps] bf16 with column order
 * (c, py, px) = the flattening of the conv weight [out, C, ps, ps].  ps %% 8 == 0, R %% ps == 0.
 * a4r_vit_assemble builds the token sequence of ViTEmbeddings.forward / SoftPrompt.forward
 * (Downstream/CV/model/model.py:523-535): out [N, 1+P+T, H] bf16 = [cls + pos[0] | patch_emb + pos[1..P] | prompt].
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_patchify(const float* images, void* out, int64_t N, int64_t C, int64_t R, int64_t ps, a4r_stream_t stream);
A4R_API int a4r_vit_assemble(const void* patch_emb, const void* cls, const void* pos, const void* prompt, void* out,
                             int64_t N, int64_t P, int64_t T, int64_t H, a4r_stream_t stream);

/* Embedding-table gradient (full fine-tuning, SURVEY.md 8f-3): dst[idx[r], :] += src[r, :] for r < R, skipping idx < 0,
 * idx >= V and idx == skip_idx (nn.Embedding's padding_idx — BertEmbeddings.word_embeddings / RobertaEmbeddings'
 * word and position tables, reached from Text_Encoder.forward, Downstream/Text/model/encoders.py:53).  src bf16 [R, ld],
 * dst f32 [V, H] (the caller zeroes it), H %% 8 == 0.  fp32 vector atomics: summation order unspecified. */
A4R_API int a4r_scatter_add_rows(const void* src, int64_t ld, const int64_t* idx, float* dst, int64_t R, int64_t H,
                                 int64_t V, int64_t skip_idx, a4r_stream_t stream);

/* out = dy * act'(u) elementwise over n bf16 values; kind 0: erf-GELU with u = pre-activation
 * (Text_Encoder.activate, encoders.py:46,57), kind 1: ReLU with u = activation output, kind 2: LeakyReLU(0.01) with
 * u = activation output (AdapterPfeifferBlock, Downstream/Text/model/modules.py:146-147), kind 3: tanh-GELU
 * ("gelu_new", HyperComplexAdapterBlock, modules.py:217) with u = pre-activation.
 * a4r_act_fwd: out = act(u) for the same kinds (the activations without a GEMM-epilogue mode run stand-alone on the
 * r-wide bottleneck). */
A4R_API int a4r_act_bwd(const void* dy, const void* u, void* out, int64_t n, int32_t kind, a4r_stream_t stream);
A4R_API int a4r_act_fwd(const void* u, void* out, int64_t n, int32_t kind, a4r_stream_t stream);

/* Weight caches: dst [rows, cols] = bf16(src) and / or dst_t [cols, rows] = bf16(src)^T from an fp32 master [rows, cols] (row
 * stride ld_src) in one pass; either output may be NULL.  Replaces the per-forward half-precision weight copies that
 * torch.cuda.amp.autocast makes in the reference (Downstream/CV/run_adapter.py:588, Downstream/CV/run.py:261; the text tree
 * trains in fp32) and the explicit transposes of the data-gradient GEMMs: the copies are cached per parameter version. */
A4R_API int a4r_cast_transpose_f32_bf16(const float* src, int64_t ld_src, void* dst, void* dst_t, int64_t rows, int64_t cols,
                                        a4r_stream_t stream);

/* Dropout (+ residual): out = x * mask / (1 - p) (+ res), n bf16 elements (n %% 8 == 0).  Replaces nn.Dropout on the
 * hidden states (BertSelfOutput.dropout / BertOutput.dropout / BertEmbeddings.dropout, SASRec modules.py:27,72,107)
 * fused with the residual add that follows it.  Counter-based RNG: element i is decided by (seed, offset + i / 4), so
 * the backward regenerates the mask by calling the same function on the gradient with the same (seed, offset). */
A4R_API int a4r_dropout(const void* x, const void* res, void* out, int64_t n, float p, uint64_t seed, uint64_t offset,
                        a4r_stream_t stream);
/* (nn.Dropout draws from torch's global generator, advanced by every call: BertSelfOutput.dropout etc. as above, SASRec
 * modules.py:27,72,107; the reference checkpoints that generator's state, Downstream/Text/data_utils/utils.py:109-115.)
 * Every dropout seed of this header (a4r_dropout, a4r_gemm_args.dropout_seed, a4r_attention_args.dropout_seed, the
 * dropout_seed of a4r_layernorm_bwd) may be given indirectly: with bit 63 set, the low 63 bits are the DEVICE address of
 * the 64-bit seed (8-byte aligned), read when the kernel runs.  A step recorded in a CUDA graph keeps its (baked)
 * counter offsets and draws fresh masks on every replay from the seed the host stores there before the replay. */
#define A4R_SEED_INDIRECT (1ull << 63)

/* out[j] (+)= sum_m x[m, j] for a bf16 [M, ld] matrix, j < width: bias gradients of trainable biases
 * (lora.Linear bias, Downstream/Text/run.py:414-428; AdapterBlock biases, Downstream/Text/model/modules.py:117-127).  Deterministic two-stage reduction through `workspace`. */
A4R_API size_t a4r_colsum_workspace_bytes(int64_t width);
A4R_API int a4r_colsum(const void* x, int64_t ld, int64_t M, int64_t width, float* out, int32_t accumulate,
               void* workspace, size_t workspace_bytes, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Weight gradient of a TRAINABLE low-rank module:  dW[N,K] (+)= alpha * A[M,N]ᵀ · B[M,K]   (f32 out)
 *
 * A = dY (bf16 [M,lda]), B = X (bf16 [M,ldb]) gives nn.Linear's dW[out,in]: AdapterBlock.fc_down / fc_up
 * (Downstream/Text/model/modules.py:117-127) and loralib's lora_B = dYᵀ·(x·Aᵀ), lora_A = (dY·B)ᵀ·x
 * (Downstream/Text/run.py:414-428).  One of N, K is small (<= 64): HBM-bound, deterministic split-M.
 * ------------------------------------------------------------------------------------------------ */
A4R_API size_t a4r_wgrad_workspace_bytes(int64_t M, int64_t N, int64_t K);
A4R_API int a4r_wgrad_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, float* dW, int64_t ldw, int64_t M,
                   int64_t N, int64_t K, float alpha, int32_t accumulate, void* workspace, size_t workspace_bytes,
                   a4r_stream_t stream);

/* The same contraction on tcgen05 (MN-major operand descriptors: the activations are read in place, no transposes),
 * split over the token axis with a fixed-order reduction: dW[N,K] (+)= alpha * A[M,N]^T . B[M,K], any N, K multiple of 8.
 * Serves full fine-tuning — every nn.Linear weight of the encoder when fine_tune_to = all
 * (Pretraining/Text/run.py:241-253, Downstream/Text/run.py:372-376) — and the skinny LoRA / adapter gradients.
 * dW 16-byte aligned, ldw % 4 == 0. */
A4R_API size_t a4r_wgrad_tc_workspace_bytes(int64_t M, int64_t N, int64_t K);
A4R_API int a4r_wgrad_tc_bf16(const void* A, int64_t lda, const void* B, int64_t ldb, float* dW, int64_t ldw, int64_t M,
                              int64_t N, int64_t K, float alpha, int32_t accumulate, void* workspace,
                              size_t workspace_bytes, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K9: fused masked dot + BCE-with-logits + mean, forward / backward.
 * Replaces Model.forward's loss (Downstream/Text/model/model.py:53-68) and, with cpc = 1,
 * ModelCPC.forward's (model.py:120-133).
 *
 * prec [B,S,D] bf16 (user-encoder output), emb [B,S+1,2,D] bf16 (encoder output; [:,:,0] history item,
 * [:,:,1] sampled negative), log_mask [B,S] f32.  fwd writes pos_score/neg_score [B,S] f32, loss [1] f32 and
 * count [1] f32 (= |valid positions|).  bwd (grad_out: device f32 scalar or NULL = 1) writes d_prec [B,S,D]
 * and the LOSS part of d_emb [B,S+1,2,D] (bf16); the gradient through the user-encoder input is separate.
 * ------------------------------------------------------------------------------------------------ */
typedef struct a4r_bce_args {
  const void* prec;
  const void* emb;
  const float* log_mask;
  float* pos_score;
  float* neg_score;
  float* loss;
  float* count;
  int64_t B, S, D;
  int32_t cpc;
} a4r_bce_args;
A4R_API size_t a4r_bce_workspace_bytes(void);
A4R_API int a4r_bce_loss_fwd(const a4r_bce_args* args, void* workspace, size_t workspace_bytes, a4r_stream_t stream);
A4R_API int a4r_bce_loss_bwd(const a4r_bce_args* args, const float* grad_out, void* d_prec, void* d_emb,
                     a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K9-S: in-batch softmax loss with duplicate-item masking, forward / backward (north-star head; SURVEY.md §8a row L2).
 * The reference itself trains with BCE (a4r_bce_loss_*; Downstream/Text/model/model.py:62-68) and has no softmax head,
 * so this entry point has no reference symbol to replace: its semantics are the in-batch debiased cross-entropy of the
 * same group's IDvs.MoRec trainer, restated by oracle/transrec_oracle.py:inbatch_softmax_loss ("parity unpinned").
 *
 * prec [B,S,D] bf16 (user-encoder output); candidates = the B*(S+1) history items of the batch, candidate
 * c = b*(S+1)+j read at cand + c*ld_cand (ld_cand = 2*D reads emb[:, :, 0, :] of Model.forward's encoder output in
 * place); item_ids [B,S+1] int64 (0 = padding); log_mask [B,S] f32; cand_bias [B*(S+1)] f32 or NULL (log-popularity).
 *   logit[(b,s), c] = <prec[b,s], cand[c]> - cand_bias[c]
 *   logit := masked_logit  if candidate slot (b',j) is padding (j < S and log_mask[b',j] == 0)
 *                          or item_ids[c] occurs in item_ids[b, :] and c != target(b,s) = b*(S+1)+s+1
 *   loss = mean over {(b,s): log_mask[b,s] != 0} of  logsumexp_c logit - logit[target]
 * fwd writes lse [B*S] f32 (kept for the backward), loss [1], count [1].  bwd (grad_out: device f32 scalar or NULL = 1)
 * writes d_prec [B,S,D] bf16 and d_cand (row c at d_cand + c*ld_dcand, D columns) bf16; the [B*S, B*(S+1)] logit matrix
 * is never materialised and there are no atomics (deterministic).  D = 64 or 128.
 * ------------------------------------------------------------------------------------------------ */
typedef struct a4r_inbatch_ce_args {
  const void* prec;
  const void* cand;
  int64_t ld_cand;
  const int64_t* item_ids;
  const float* log_mask;
  const float* cand_bias;
  float* lse;
  float* loss;
  float* count;
  int64_t B, S, D;
  float masked_logit; /* -1e4 in the MoRec statement */
} a4r_inbatch_ce_args;
A4R_API size_t a4r_inbatch_ce_workspace_bytes(int64_t B, int64_t S);
A4R_API int a4r_inbatch_ce_fwd(const a4r_inbatch_ce_args* args, void* workspace, size_t workspace_bytes, a4r_stream_t stream);
A4R_API int a4r_inbatch_ce_bwd(const a4r_inbatch_ce_args* args, const float* grad_out, void* d_prec, void* d_cand,
                               int64_t ld_dcand, a4r_stream_t stream);

/* K14: torch.optim.Adam semantics (Downstream/Text/run.py:524-529) over one flat f32 segment.
 * step is 1-based; the gradient is multiplied by grad_scale first (1/world_size after a sum all-reduce). */
A4R_API int a4r_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int64_t step, float grad_scale, a4r_stream_t stream);
/* The same update (optim.Adam(...).step(), Downstream/Text/run.py:524-529,600) with the two step-dependent factors read from
 * device memory: bias_corr[0] = 1 - beta1^step, bias_corr[1] = sqrt(1 - beta2^step).  For a train step recorded in a CUDA
 * graph (SURVEY.md 8e / 8f-2: "the step under one CUDA graph"): kernel arguments are baked at capture, so what changes
 * between replays is uploaded before each replay.
 * Given the factors a4r_adam_step computes for the same step the result is bit-identical. */
A4R_API int a4r_adam_step_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                              float eps, float weight_decay, const float* bias_corr, float grad_scale, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K10: item-ID gather  out[r,:] = table[ids[r],:]  (bf16 rows of D elements).  Replaces the CPU fancy-index
 * `self.item_content[pad_tokens]` of BuildEvalDataset.__getitem__ (Downstream/Text/data_utils/dataset.py:72).
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_gather_rows(const void* table, const int64_t* ids, void* out, int64_t rows, int64_t D,
                            a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Train-batch assembly on the device (SURVEY.md 8f-1).  Replaces BuildTrainDataset.__getitem__
 * (Downstream/Text/data_utils/dataset.py:24-49) for a whole batch: per user, one uniform negative in [1, item_num]
 * per real history slot except the last, redrawn while it occurs in the user's own sequence (:36-40), then
 * out[b, j, 0, :] = item_content[seqs[b, j]], out[b, j, 1, :] = item_content[neg[b, j]] (:46) and
 * log_mask[b, j] = (seqs[b, j] != 0) for j < S (:31).
 *   seqs [B, S1] int64 left-padded item ids (0 = padding), S1 = max_seq_len + 1;  item_content [item_num+1, W] int64
 *   (W = 2L: ids | attention mask; row 0 = the padding item);  out [B, S1, 2, W] int64;  log_mask [B, S1-1] f32;
 *   neg_out [B, S1] int64 (the negatives used);  fail_flag: one int32 set to 1 if some slot found no admissible
 *   negative in 64 draws (item_num <= S1; the reference's loop would not terminate);  neg_in: NULL to sample, or
 *   [B, S1] int64 negatives to use instead (replay / parity against the reference's Python RNG).
 * Draw a of slot (b, j) is a pure function of (seed, offset + (b*S1 + j)*64 + a): a caller advances offset by
 * B*S1*64 per batch.  All pointers are device pointers; item_content and out 16-byte aligned, W even.
 * Ids-only mode (item_content = NULL, W = 0, out may be NULL): the id item tower's sample (BuildTrainDataset with
 * use_modal = False returns the ids [S1, 2] themselves) is [seqs | neg_out]; only log_mask and neg_out are written, and
 * neg_out is exactly what the full call returns for the same (seed, offset).
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_sample_train_batch(const int64_t* seqs, const int64_t* item_content, const int64_t* neg_in, int64_t* out,
                                   float* log_mask, int64_t* neg_out, int32_t* fail_flag, int64_t B, int64_t S1, int64_t W,
                                   int64_t item_num, uint64_t seed, uint64_t offset, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * ID item tower (--item_tower id): nn.Embedding(item_num + 1, D, padding_idx=0) reached from Model.forward
 * (`input_embs_all = self.id_embedding(sample_items)`, the use_modal = False branch of Downstream/Text/model/model.py's
 * Model / ModelCPC and of Downstream/CV/model/model.py's), forward and backward.
 *
 * a4r_id_embed_fwd: ids int64 [B, S1, 2] (S1 = max_seq_len + 1), table f32 [V, D] (the fp32 master, 16-byte aligned,
 *   D %% 4 == 0) -> emb bf16 [B, S1, 2, D] = bf16_rne(table[ids]) and, if hist != NULL, hist bf16 [B, S1-1, D] =
 *   emb[:, :S1-1, 0] (the user-encoder input).  An id outside [0, V) reads as a zero row.  No bf16 copy of the table is
 *   made: the traffic is the gathered rows only.
 * a4r_id_embed_bwd: the table gradient of both outputs.  sorted_ids [R] / order [R] (R = B*S1*2) are a STABLE ascending
 *   sort of the flat ids (order = the flat occurrence index of each sorted entry).  For every id in [0, V) other than
 *   padding_idx that occurs, row id of grad f32 [V, D] receives the fp32 sum of its occurrences r in ascending r, where
 *   occurrence r = (b, j, t) contributes d_emb[r] and then, if t == 0 and j < S1-1 and d_hist != NULL, d_hist[b, j]
 *   (d_emb bf16 [B, S1, 2, D], d_hist bf16 [B, S1-1, D]); grad[id] = sum (accumulate = 0) or grad[id] + sum
 *   (accumulate = 1).  Rows of ids that do not occur are not touched.  No atomics: bit-identical run to run.
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_id_embed_fwd(const float* table, int64_t V, int64_t D, const int64_t* ids, int64_t B, int64_t S1,
                             void* emb, void* hist, a4r_stream_t stream);
A4R_API int a4r_id_embed_bwd(const int64_t* sorted_ids, const int64_t* order, const void* d_emb, const void* d_hist,
                             float* grad, int64_t V, int64_t D, int64_t B, int64_t S1, int64_t padding_idx,
                             int32_t accumulate, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K11 + K12: full-ranking scores fused with the history mask and per-user top-k.
 * Replaces `scores = torch.matmul(prec_emb, item_embeddings.t())`, `score[history] = -inf`, `score[1:]` and the
 * argsort of metrics_topK (Downstream/Text/data_utils/metrics.py:105-111,51-59).
 *
 * users [U, ld_users] bf16 (d columns), items [I, ld_items] bf16 = one shard of the item table whose row r is item
 * id id_base + r.  history [U, hist_len] int32 ids to exclude (0 = unused slot; may be NULL); item id 0 is always
 * excluded.  Writes P = a4r_score_topk_partials(U, I) partial lists, each sorted by (score desc, id asc):
 * out_scores [P, U, k] f32 (-inf = empty slot), out_ids [P, U, k] int32.  k <= 16.
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_score_topk_partials(int64_t U, int64_t I);
A4R_API int a4r_score_topk(const void* users, int64_t ld_users, const void* items, int64_t ld_items, int64_t U, int64_t I,
                           int64_t d, int64_t id_base, const int32_t* history, int64_t hist_len, int32_t k,
                           float* out_scores, int32_t* out_ids, a4r_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K13: merge P sorted partial top-k lists per user (item splits of one GPU, or the all-gathered lists of all
 * item shards) under (score desc, id asc); if target != NULL also HR@k and NDCG@k per user exactly as
 * metrics_topK (metrics.py:51-59): hit = [target in top-k], ndcg = hit / log2(rank + 1).  P <= 64.
 * ------------------------------------------------------------------------------------------------ */
A4R_API int a4r_topk_merge(const float* in_scores, const int32_t* in_ids, int32_t P, int64_t U, int32_t k,
                           float* out_scores, int32_t* out_ids, const int32_t* target, float* hit, float* ndcg,
                           a4r_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ADAPTER4REC_H_ */
