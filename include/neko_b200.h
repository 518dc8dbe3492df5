/*
 * neko_b200 -- C ABI of the B200-native Gato training hot path.
 *
 * The reference (ManifoldRG/NEKO) has no FFI: its hot path is the Python class
 * gato/policy/gato_policy.py:18 (GatoPolicy) calling torch ops.  This header declares the
 * operator-level entry points a maintainer binds (ctypes, see INTEGRATION.md) to replace those
 * torch call sites.  Every function cites the reference lines it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named host_*;
 *   - the caller owns every buffer (outputs and workspaces included); nothing is allocated,
 *     nothing synchronises, everything is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return 0 on success, a negative NEKO_E* code otherwise; neko_last_error() gives the
 *     thread-local message;  sm_100 only -- other devices get NEKO_EDEVICE (no CPU fallback);
 *   - bf16 buffers are raw uint16_t bit patterns (__nv_bfloat16).
 */
#ifndef NEKO_B200_H
#define NEKO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NEKO_OK 0
#define NEKO_EINVAL (-1)   /* bad argument (shape / alignment / null pointer) */
#define NEKO_ECUDA (-2)    /* CUDA runtime / driver error                      */
#define NEKO_EDEVICE (-3)  /* current device is not sm_100                     */

int neko_version(void);
const char* neko_last_error(void);
/* 0 when the current CUDA device is a compute-capability-10.x part. */
int neko_device_check(void);
int neko_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * Dropout (nn.Dropout at trajectory_gpt2.py:179 attention weights, :254 and :278 residual branches, :707
 * embeddings; p = --dropout, and 0.1 for the embeddings whatever --dropout says).  Masks are counter based: the keep
 * decision of element (row, col) of site `stream` is a pure function of (seed, stream, row, col), so backward kernels
 * regenerate them.  `seed` points to two uint32 words in DEVICE memory that the host refreshes before every forward
 * (a replayed CUDA graph therefore draws fresh masks).  NULL pointer, NULL seed or thr16 == 0 disable dropout.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  const uint32_t* seed;  /* device pointer to 2 words                                        */
  uint32_t stream;       /* site id: 0 embeddings, 4*layer+1 attention, +2 attn residual, +3 mlp residual */
  uint32_t thr16;        /* round(p * 65536): an element is dropped when its 16 random bits < thr16   */
  float scale;           /* 65536 / (65536 - thr16), applied to kept elements                */
  uint32_t reserved;
} neko_dropout;

/* x[rows, cols] (fp32, row pitch ld) *= mask * scale, in place.  Used for embd dropout and its backward. */
int neko_dropout_apply(float* x, int64_t ld, int rows, int cols, const neko_dropout* drop, void* stream);
/* keep[rows, cols] (uint8 0/1): the mask the kernels use -- for tests and for replaying a step in a reference. */
int neko_dropout_mask(uint8_t* keep, int rows, int cols, const neko_dropout* drop, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tokenise + embed + interleave: GatoPolicy.tokenize_input_dicts, gato_policy.py:195-432,
 * with ContinuousTokenizer.encode / mu_law (input_tokenizers.py:5-30) inlined.
 * One descriptor per sample; the host packs all continuous values into `fvals`, all integer
 * inputs (text ids, discrete obs / actions) into `ivals`.
 * ------------------------------------------------------------------------------------------- */
typedef struct neko_sample_desc {
  int32_t n_timesteps;   /* T                                                            */
  int32_t n_patches;     /* image patches per timestep (ids 0, target 0)                 */
  int32_t n_text;        /* text tokens per timestep (target 1)                          */
  int32_t n_cobs;        /* continuous observation scalars per timestep (mu-law, tgt 0)  */
  int32_t n_dobs;        /* discrete observation tokens per timestep (target 0)          */
  int32_t n_cact;        /* continuous action scalars per timestep (no mu-law, tgt 1)    */
  int32_t n_dact;        /* discrete action tokens per timestep (target 1)               */
  int32_t seq_off;       /* left padding = S - T * tokens_per_timestep                   */
  int32_t text_off;      /* offsets (elements) of this sample's [T, n_*] blocks          */
  int32_t cobs_off;      /*   text/dobs/dact index ivals, cobs/cact index fvals          */
  int32_t dobs_off;
  int32_t cact_off;
  int32_t dact_off;
  int32_t patch_off;     /* first row of this sample in patch_emb [P_total, d]           */
  int32_t row_base;      /* packed layout: first row of this sample (prefix sum of lengths) */
  int32_t reserved1;
} neko_sample_desc;

typedef struct neko_tok_params {
  float mu;              /* 100   */
  float M;               /* 256   */
  int32_t n_bins;        /* 1024  */
  int32_t cont_start;    /* token_starts['continuous'] = 50257, gato_policy.py:66-70 */
  int32_t disc_start;    /* token_starts['discrete']   = 51281 */
  int32_t vocab;         /* rows of embed_table */
  int32_t use_pos;       /* add pos_embed_observation to observation tokens (:381-385) */
  int32_t seq_len;       /* S: left-padded length (max over samples)                  */
  int32_t width;         /* output row length (= S, or context_len with pad_seq)      */
  int32_t ctx_rows;      /* rows of pos_table */
} neko_tok_params;

/* ids, masks and embeddings in one pass.  tokens int64 [B,width]; target/token masks fp32
 * [B,width]; token_embeddings fp32 [B,width,d] (may be NULL: ids/masks only).
 * err_flag (nullable, int32): set to 1 when an id falls outside [0,vocab). */
int neko_tokenize_embed_fwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                            const float* fvals, const int32_t* ivals, const float* patch_emb,
                            const float* embed_table, const float* pos_table, const float* sep_vec,
                            int64_t* tokens, float* target_masks, float* token_masks,
                            float* token_embeddings, int32_t* err_flag, void* stream);

/* Packed (padding-free) layout: the same ids / masks / embeddings, but sample b's valid position s is written to row
 * descs[b].row_base + (s - seq_off) of tokens [T], target/token masks [T] and token_embeddings [T,d] (T = sum of the
 * sample lengths); padding positions write nothing.  seq_len / width of host_params as in the padded call. */
int neko_tokenize_embed_packed_fwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                                   const float* fvals, const int32_t* ivals, const float* patch_emb,
                                   const float* embed_table, const float* pos_table, const float* sep_vec,
                                   int64_t* tokens, float* target_masks, float* token_masks,
                                   float* token_embeddings, int32_t* err_flag, void* stream);

/* Backward of the embedding half (autograd of gato_policy.py:275-393): scatter-adds into
 * d_embed_table [vocab,d], d_pos_table [ctx_rows,d], d_sep [d] (all fp32, accumulated) and writes
 * d_patch_emb [P_total,d] (nullable). */
int neko_embed_bwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                   const int64_t* tokens, const float* d_token_embeddings,
                   float* d_embed_table, float* d_pos_table, float* d_sep, float* d_patch_emb,
                   void* stream);
/* neko_embed_bwd on the packed layout: tokens [T], d_token_embeddings [T,d] (rows as in the packed forward). */
int neko_embed_packed_bwd(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                          const int64_t* tokens, const float* d_token_embeddings,
                          float* d_embed_table, float* d_pos_table, float* d_sep, float* d_patch_emb,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * LayerNorm (ln_1 / ln_2 / ln_f, trajectory_gpt2.py:323,353,779). x fp32 [N,d] -> y bf16 (fp16 if out_f16).
 * d % 4 == 0, d <= 2048; rows are dense (pitch d).  x, gamma, beta 16-byte aligned; y, y2 8-byte aligned.
 * ------------------------------------------------------------------------------------------- */
int neko_layernorm_fwd(const float* x, const float* gamma, const float* beta, uint16_t* y_16,
                       uint16_t* y2_bf16 /* nullable second copy */, float* mean, float* rstd, int N, int d,
                       float eps, int out_f16, void* stream);
/* dx_resid (fp32 [N,d]) += LN'(dy); optional bf16 copy of the updated dx_resid; dgamma/dbeta
 * fp32 [d] are accumulated (caller zeroes them).  dx_colsum (nullable, fp32 [d], accumulated): column sums
 * of the bf16 copy = the bias gradient of the Conv1D whose output was added into this residual.
 * branch_drop (nullable): the residual branch that produced x went through dropout (x = x_prev + dropout(branch)); the
 * bf16 copy and dx_colsum then carry mask * scale * dx_resid, i.e. the gradient entering that branch.
 * x, dx_resid, gamma 16-byte aligned; dy, dx_bf16 8-byte aligned (the alignment neko_layernorm_bwd_ordered requires).
 * Kernel: warp-per-row when d % 128 == 0 and d <= 1024; otherwise a column-owner kernel over NEKO_LN_CTAS row ranges
 * (default 2 per SM; values below 1 keep the default): staged (cp.async.bulk ring) when d % 8 == 0, dy is 16-byte
 * aligned and the ring has >= 2 stages, else register.  NEKO_LN_BWD_COLUMNS / NEKO_LN_BWD_REGISTER (read once per
 * process) force the column-owner / register kernels. */
int neko_layernorm_bwd(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean,
                       const float* rstd, float* dx_resid, uint16_t* dx_bf16, float* dgamma,
                       float* dbeta, float* dx_colsum, int N, int d, const neko_dropout* branch_drop, void* stream);
/* The backward kernel neko_layernorm_bwd would run for these arguments (same argument checks, same environment knobs),
 * decided on the host without launching anything: 0 = warp-per-row, 1 = staged, 2 = register, < 0 = the call is
 * rejected.  out (nullable) receives the launch shape. */
typedef struct neko_layernorm_bwd_path_info {
  int32_t grid;                 /* CTAs launched                                                   */
  int32_t rows_per_cta;         /* column-owner kernels: consecutive rows per CTA; 0 for warp-per-row (grid-stride rows) */
  int32_t stages;               /* staged kernel: shared-memory ring depth (2..4); 0 otherwise      */
} neko_layernorm_bwd_path_info;
int neko_layernorm_bwd_path(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean,
                            const float* rstd, const float* dx_resid, const uint16_t* dx_bf16, const float* dgamma,
                            const float* dbeta, const float* dx_colsum, int N, int d, const neko_dropout* branch_drop,
                            neko_layernorm_bwd_path_info* out);

/* ---------------------------------------------------------------------------------------------
 * Dense GEMM on tcgen05 tensor cores (HF Conv1D addmm trajectory_gpt2.py:222,253,274,277;
 * predict_token gato_policy.py:172; post_embedding_projection embeddings.py:53; and their
 * autograd dgrad / wgrad).   C[M,N] = epilogue( sum_k A[m,k] * B[n,k] ).
 * The operand buffers must cover the full (tile-padded is NOT required; TMA zero-fills past M/N/K) logical
 * extents given by M, N, K.
 * a_mn / b_mn = 0: operand is K-major (row m / n is contiguous in k, leading dimension ld);
 *             = 1: operand is MN-major (stored [K, M] / [K, N] row-major, leading dimension ld).
 * ------------------------------------------------------------------------------------------- */
enum neko_epilogue {
  NEKO_EPI_BF16 = 0,            /* C 16-bit = acc (+bias)                                       */
  NEKO_EPI_F32 = 1,             /* C fp32 = acc (+bias) (+= C when accumulate)                  */
  NEKO_EPI_GELU_BF16 = 2,       /* C 16-bit = acc+bias (pre-activation), C2 16-bit = gelu_erf() */
  NEKO_EPI_RESID_F32 = 3,       /* C fp32 = acc + bias + aux_f32[m,n]   (residual add)          */
  NEKO_EPI_DGELU_BF16 = 4,      /* C 16-bit = acc * gelu_erf'(aux_bf16[m,n]); bias must be NULL */
  NEKO_EPI_RESID_F32_BF16 = 5   /* as 3, plus C2 16-bit copy of the result                      */
};
/* 16-bit operands / outputs are bf16 unless the matching flag selects IEEE fp16 (same tensor-core rate,
 * 3 more mantissa bits: the forward pass uses fp16 operands to meet the logits tolerance, gradients stay
 * bf16 for range).  tcgen05 kind::f16 traps on mixed A/B formats, so NEKO_GEMM_A_F16 and NEKO_GEMM_B_F16 must
 * be set together. */
#define NEKO_GEMM_A_F16 1
#define NEKO_GEMM_B_F16 2
#define NEKO_GEMM_C_F16 4
#define NEKO_GEMM_C2_F16 8
#define NEKO_GEMM_GELU_TANH 16 /* GELU / GELU' epilogues use the tanh form (HF "gelu_new", pretrained GPT-2) instead of erf */
#define NEKO_GEMM_DETERMINISTIC 32 /* bitwise reproducible: splits = 1 and no stream-K whatever NEKO_GEMM_SPLITS / NEKO_GEMM_STREAMK
                                    * say, so each element is summed by one CTA in k order (the result does not depend on the grid) */

typedef struct neko_gemm_desc {
  int32_t M, N, K;
  int32_t a_mn, b_mn;           /* operand majors, see above                                    */
  int32_t epilogue;             /* enum neko_epilogue                                           */
  int32_t accumulate;           /* NEKO_EPI_F32 only: C += result                               */
  int32_t flags;                /* NEKO_GEMM_*_F16; A and B must share one 16-bit format         */
  const void* A; int64_t lda;   /* leading dimensions in elements, multiples of 8               */
  const void* B; int64_t ldb;
  void* C;  int64_t ldc;
  void* C2; int64_t ldc2;       /* second output of the GELU / RESID_F32_BF16 epilogues          */
  void* C3; int64_t ldc3;       /* optional bf16 copy of C2 (GELU epilogue): the wgrad operand   */
  const float* bias;            /* [N] or NULL                                                  */
  const void* aux; int64_t ld_aux;
  neko_dropout drop;            /* RESID epilogues: C = aux + dropout(acc + bias) (resid_dropout, trajectory_gpt2.py:254,278) */
  void* workspace;              /* optional, zero-initialised ONCE by the caller and then left to the library: lets launches whose  */
  int64_t workspace_bytes;      /* tile count is a poor multiple of the SM count run stream-K (a tile's k-range shared by two CTAs /
                                 * CTA pairs, partial accumulators and their counters live here).  neko_gemm_workspace_bytes() is
                                 * enough for any problem; NULL / too small = classic tile scheduling.  One workspace per stream. */
} neko_gemm_desc;

int neko_gemm(const neko_gemm_desc* host_desc, void* stream);

/* The schedule neko_gemm would launch for this descriptor (same argument checks, same NEKO_GEMM_* environment knobs),
 * computed on the host without launching anything. */
typedef struct neko_gemm_plan_info {
  int32_t BN;                   /* tile width: 128, 192 or 256 columns                          */
  int32_t pair;                 /* 1: cta_group::2 CTA pair (256-row tile), 0: single CTA (128)  */
  int32_t splits;               /* split-K factor (fp32 reduce-add into C when > 1)              */
  int32_t epi_warps;            /* epilogue warps per CTA: 8 or 16                              */
  int32_t streamk;              /* 1: stream-K work distribution (needs the workspace)          */
  int32_t tma_store;            /* 1: outputs through shared-memory staging + TMA stores, 0: direct stores */
  int32_t tma_aux;              /* 1: RESID_F32 / DGELU aux operand through TMA boxes, 0: per-thread loads */
  int32_t vec_ok;               /* 1: 16-byte epilogue accesses, 0: per-element (scalar) path   */
  int32_t n_fast;               /* tile rasterisation walks N first                             */
  int32_t stages;               /* shared-memory ring depth of the main loop                    */
} neko_gemm_plan_info;
int neko_gemm_plan(const neko_gemm_desc* host_desc, neko_gemm_plan_info* out);
/* Bytes of neko_gemm_desc.workspace that cover every problem on this device (148 partial 128 x 256 fp32 tiles + counters). */
int64_t neko_gemm_workspace_bytes(void);

/* ---------------------------------------------------------------------------------------------
 * Causal self-attention with left padding (Attention._attn, trajectory_gpt2.py:163-188, with the
 * additive -1e4 padding bias of :663-679 realised as a per-sample first valid key).
 * qkv bf16 [B,S,3*H*dh] (q | k | v as c_attn emits them), out bf16 [B,S,H*dh], lse fp32 [B,H,S].
 * Sample b attends keys in [first_valid[b], min(query, S_valid-1)]; rows outside [first_valid[b], S_valid)
 * (left padding, right padding of --pad_seq) are written as zeros.
 * drop (nullable): attn_dropout on the softmax weights (:179); mask element (row = (b*H + h)*S + query, col = key).
 */
int neko_attention_fwd(const uint16_t* qkv, const int32_t* first_valid, uint16_t* out,
                       uint16_t* out2_bf16 /* nullable second copy */, float* lse, int B, int S, int S_valid,
                       int H, int dh, int out_f16, const neko_dropout* drop, void* stream);
/* The forward kernel neko_attention_fwd would run for these arguments (same argument checks, same NEKO_ATTN_TC knob),
 * decided on the host without launching anything: 0 = mma.sync kernel, 1 = tcgen05 kernel, < 0 = the call is rejected. */
int neko_attention_fwd_path(const uint16_t* qkv, const int32_t* first_valid, const uint16_t* out,
                            const uint16_t* out2_bf16, const float* lse, int B, int S, int S_valid, int H, int dh,
                            int out_f16, const neko_dropout* drop);
/* Single-query attention against a key/value cache (KV-cached decode for the predict_* loops, gato_policy.py:452-476 --
 * the reference re-runs the whole context per generated token).  q bf16 [H*dh] (the new position's query), k_cache /
 * v_cache bf16 [len, H*dh] (all visible keys incl. the new one), out 16-bit [H*dh].  len <= 8192; dh even and dividing 128;
 * q and k_cache 4-byte aligned. */
int neko_attention_decode(const uint16_t* q, const uint16_t* k_cache, const uint16_t* v_cache, int len, int H, int dh,
                          uint16_t* out, int out_f16, void* stream);
/* dqkv bf16 [B,S,3*H*dh]; delta fp32 [B,H,S] is caller-provided scratch. */
int neko_attention_bwd(const uint16_t* qkv, const uint16_t* out, const uint16_t* dout, const float* lse,
                       const int32_t* first_valid, uint16_t* dqkv, float* delta, int B, int S, int S_valid,
                       int H, int dh, int out_f16, const neko_dropout* drop, void* stream);
/* Variable-length (packed) causal attention: sample b owns rows [cu_seqlens[b], cu_seqlens[b+1]) of qkv bf16 [T,3*H*dh],
 * out bf16 [T,H*dh] and lse fp32 [H,T]; query q of a sample attends its own keys [0, q].  S_max = longest sample (grid
 * extent).  Attention dropout keeps the padded layout's coordinates so the masks equal neko_attention_fwd's bit for bit:
 * row (b*H + h)*S_width + first_valid[b] + q, column first_valid[b] + k, where S_width is the padded row length (S, or
 * context_len with --pad_seq) and first_valid[b] = S - length of b.  Head dims 16, 32, 64, 128 (mma.sync kernels). */
int neko_attention_varlen_fwd(const uint16_t* qkv, const int32_t* cu_seqlens, const int32_t* first_valid, uint16_t* out,
                              uint16_t* out2_bf16 /* nullable second copy */, float* lse, int B, int T, int S_max, int S_width,
                              int H, int dh, int out_f16, const neko_dropout* drop, void* stream);
/* dqkv bf16 [T,3*H*dh]; delta fp32 [H,T] is caller-provided scratch. */
int neko_attention_varlen_bwd(const uint16_t* qkv, const uint16_t* out, const uint16_t* dout, const float* lse,
                              const int32_t* cu_seqlens, const int32_t* first_valid, uint16_t* dqkv, float* delta, int B, int T,
                              int S_max, int S_width, int H, int dh, int out_f16, const neko_dropout* drop, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Masked cross entropy (gato_policy.py:174-186).  rows int32 [n_rows]: flat source positions
 * b*S_width+s whose target is tokens[row+1]; loss = mean over rows (written to *loss).
 * ------------------------------------------------------------------------------------------- */
#define NEKO_CE_LOGITS_COMPACT 1   /* logits row r (not rows[r]) holds position rows[r]            */
#define NEKO_CE_DLOGITS_COMPACT 2  /* dlogits row r (not rows[r]) receives position rows[r]         */
#define NEKO_CE_ZERO_PAD 4         /* bwd also zeroes dlogits columns V..ld_dlogits of the rows it writes */
/* A target outside [0, V) (e.g. -1) is not an error: nothing outside the row is read, the row's loss is 0 (it still counts
 * in the mean's n_rows), and its gradient row is softmax * g / n_rows with no one-hot term. */
int neko_masked_ce_fwd(const float* logits, int64_t ld_logits, int V, const int32_t* rows, int n_rows,
                       const int64_t* tokens, float* row_lse, float* row_loss, float* loss, int flags,
                       void* stream);
/* dlogits bf16 rows get (softmax - onehot) * (*gscale) / n_rows; in the dense layout the caller
 * zero-fills the buffer beforehand.  gscale: device fp32 scalar (upstream d loss). */
/* Training forward: loss AND the gradient operand in one pass over the selected rows (each row is read from HBM once and
 * kept in shared memory): dlogits = (softmax - onehot) / n_rows as bf16, i.e. neko_masked_ce_bwd with gscale = 1.
 * Returns 1 (nothing launched) when a row does not fit the shared memory of one CTA or the buffers are not vector-aligned:
 * the caller then uses neko_masked_ce_fwd / neko_masked_ce_bwd.  neko_ce_scale_grad multiplies the stored gradient by the
 * upstream scalar in backward and is a no-op on the device when that scalar is exactly 1. */
int neko_masked_ce_fused(const float* logits, int64_t ld_logits, int V, const int32_t* rows, int n_rows,
                         const int64_t* tokens, float* row_lse, float* row_loss, float* loss,
                         uint16_t* dlogits, int64_t ld_dlogits, int flags, void* stream);
/* The same pass over fp16 logits (the head GEMM of the training path that returns no logits writes them in 16 bits): V*2
 * bytes read per row instead of V*4; statistics in fp32.  Same return convention. */
int neko_masked_ce_fused_f16(const uint16_t* logits_f16, int64_t ld_logits, int V, const int32_t* rows, int n_rows,
                             const int64_t* tokens, float* row_lse, float* row_loss, float* loss, uint16_t* dlogits,
                             int64_t ld_dlogits, int flags, void* stream);
int neko_ce_scale_grad(uint16_t* dlogits, int64_t n, const float* gscale, void* stream);
int neko_masked_ce_bwd(const float* logits, int64_t ld_logits, int V, const int32_t* rows, int n_rows,
                       const int64_t* tokens, const float* row_lse, const float* gscale,
                       uint16_t* dlogits, int64_t ld_dlogits, int flags, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Small memory-bound helpers around the GEMMs.
 * ------------------------------------------------------------------------------------------- */
int neko_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream);
int neko_cast_f32_to_f16(const float* src, uint16_t* dst, int64_t n, void* stream);
/* one read, two 16-bit copies (fp16 forward operand + bf16 backward operand of the weights) */
int neko_cast_f32_to_f16_bf16(const float* src, uint16_t* dst_f16, uint16_t* dst_bf16, int64_t n, void* stream);
/* GEGLU gate (--activation_fn geglu; MLP.forward, trajectory_gpt2.py:267-276): h = gelu(c_fc(x)) * gated_layer(x).
 * fwd: out (fp16 if out_f16 else bf16, + optional bf16 copy) = act (fp16 if act_f16 else bf16) * gate (bf16), n elements.
 * bwd: d_gate = dh * gelu_erf(pre), d_pre = dh * gate * gelu_erf'(pre); all bf16. */
int neko_geglu_fwd(const uint16_t* act, const uint16_t* gate_bf16, uint16_t* out, uint16_t* out_bf16 /* nullable */,
                   int64_t n, int act_f16, int out_f16, void* stream);
int neko_geglu_bwd(const uint16_t* dh_bf16, const uint16_t* pre_bf16, const uint16_t* gate_bf16, uint16_t* d_gate_bf16,
                   uint16_t* d_pre_bf16, int64_t n, void* stream);
/* out[n] (+)= sum_m X[m,n]; X bf16 [M, ld]  (bias gradients of Conv1D / Linear). */
int neko_colsum_bf16(const uint16_t* X, int64_t ld, int M, int N, float* out, int accumulate, void* stream);
/* rows: dst[i,:] = src[rows[i],:] (gather) or dst[rows[i],:] = src[i,:] (scatter), bf16 width n. */
int neko_gather_rows_bf16(const uint16_t* src, int64_t ld_src, const int32_t* rows, int n_rows, int n,
                          uint16_t* dst, int64_t ld_dst, void* stream);
int neko_scatter_rows_bf16(const uint16_t* src, int64_t ld_src, const int32_t* rows, int n_rows, int n,
                           uint16_t* dst, int64_t ld_dst, void* stream);
int neko_scatter_rows_add_f32(const uint16_t* src_bf16, int64_t ld_src, const int32_t* rows, int n_rows,
                              int n, float* dst, int64_t ld_dst, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Image patch embedding: ImageEmbedding.forward / ResidualBlock_V2 (embeddings.py:28-61,111-131)
 * up to (not including) post_embedding_projection, which is a neko_gemm_bf16 call.
 * images: `n_img` frames [3,Himg,Wimg] of fp32 (is_u8=0) or uint8 (is_u8=1), 0..255.
 * patches_out fp16 [n_img*n_h*n_w, 3*p*p]  (c p1 p2 flattening, embeddings.py:50).
 * Saved for backward: gn_stats fp32 [P, groups, 2] (mean, rstd).
 * ------------------------------------------------------------------------------------------- */
int neko_patch_resblock_fwd(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch,
                            int C, int groups, const float* conv1_w, const float* conv1_b,
                            const float* gn_w, const float* gn_b, const float* conv2_w,
                            const float* conv2_b, uint16_t* patches_out, uint16_t* patches_out_bf16 /* nullable */,
                            float* gn_stats, void* stream);
int neko_patch_resblock_bwd(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch,
                            int C, int groups, const float* conv1_w, const float* conv1_b,
                            const float* gn_w, const float* gn_b, const float* conv2_w,
                            const float* gn_stats, const uint16_t* d_patches_bf16,
                            float* d_conv1_w, float* d_conv1_b, float* d_gn_w, float* d_gn_b,
                            float* d_conv2_w, float* d_conv2_b, void* stream);
/* x[p,:] += row_tab[row_bin[p]] + col_tab[col_bin[p]] (embeddings.py:56-57,102-110) on fp32 [P,d]; the
 * bins are computed by the host with the reference's own torch calls (keeps the train-mode RNG stream). */
int neko_patch_pos_add(float* x, int P, int d, const int32_t* row_bin, const int32_t* col_bin,
                       const float* row_tab, const float* col_tab, void* stream);
int neko_patch_pos_bwd(const float* dx, int P, int d, const int32_t* row_bin, const int32_t* col_bin,
                       float* d_row_tab, float* d_col_tab, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Optimiser step (train.py:127-133, trainer.py:181-186): global-norm clip + AdamW over one flat
 * fp32 parameter / gradient arena.
 * ------------------------------------------------------------------------------------------- */
int neko_sumsq_f32(const float* x, int64_t n, float* out_accum, void* stream);
/* w_f16 / w_bf16 (nullable): 16-bit operand copies of the first n_cast parameters (the GEMM weights), rewritten in the
 * same pass so that the next forward needs no cast kernel. */
int neko_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                    float lr, float beta1, float beta2, float eps, float weight_decay, int step,
                    const float* grad_sumsq, float max_norm, float grad_div,
                    uint16_t* w_f16, uint16_t* w_bf16, int64_t n_cast, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Ordered reductions (deterministic training mode, DESIGN.md "Deterministic training mode").  Each entry point computes what
 * its default twin computes, but every floating-point sum has a fixed order that depends on the problem shape only -- not on
 * the grid, the SM count, NEKO_*_CTAS caps or timing -- so the result is bitwise reproducible.  It differs from the default
 * twin by reassociation only.  Scratch memory comes from `workspace` (device, at least *_workspace_bytes bytes, no
 * initialisation needed; 256-byte aligned for the sorting entry points, 16-byte for the others); nothing is allocated or
 * synchronised, so the calls can be captured in a CUDA graph.  The *_workspace_bytes queries return the size, or a negative
 * NEKO_E* code.  Argument checks return NEKO_EINVAL before any CUDA call; the sorting entry points (embed, patch_pos) query
 * the radix sort's scratch size before they compare it with workspace_bytes.
 * NEKO_ORDERED_CTAS (environment) caps the grid of these kernels; it changes no result.
 * ------------------------------------------------------------------------------------------- */
/* neko_layernorm_bwd with dgamma / dbeta / dx_colsum summed over fixed 64-row blocks (block partials in the workspace, then
 * folded in a fixed order, one writer per element).  d % 4 == 0, d <= 2048; x, dx_resid, gamma 16-byte and dy, dx_bf16
 * 8-byte aligned.  dx_resid and dx_bf16 are computed row by row exactly as the warp-per-row default kernel does. */
int64_t neko_layernorm_bwd_ordered_workspace_bytes(int N, int d);
int neko_layernorm_bwd_ordered(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean,
                               const float* rstd, float* dx_resid, uint16_t* dx_bf16, float* dgamma, float* dbeta,
                               float* dx_colsum, int N, int d, const neko_dropout* branch_drop, void* workspace,
                               int64_t workspace_bytes, void* stream);
/* neko_colsum_bf16 over fixed 64-row blocks. */
int64_t neko_colsum_bf16_ordered_workspace_bytes(int M, int N);
int neko_colsum_bf16_ordered(const uint16_t* X, int64_t ld, int M, int N, float* out, int accumulate, void* workspace,
                             int64_t workspace_bytes, void* stream);
/* neko_embed_bwd / neko_embed_packed_bwd as a sorted scatter-add: (table row, source row) keys are built on the device and
 * radix-sorted (stable), and every embed_token / pos_embed_observation row and the separator is summed by one writer in
 * ascending source-row order.  d_patch_emb rows are copied.  Ids outside [0, vocab) and position slots >= ctx_rows are
 * skipped.  Gradient buffers 16-byte aligned.  One workspace size covers both layouts. */
int64_t neko_embed_bwd_ordered_workspace_bytes(int B, const neko_tok_params* host_params);
int neko_embed_bwd_ordered(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                           const int64_t* tokens, const float* d_token_embeddings, float* d_embed_table, float* d_pos_table,
                           float* d_sep, float* d_patch_emb, void* workspace, int64_t workspace_bytes, void* stream);
int neko_embed_packed_bwd_ordered(const neko_sample_desc* descs, int B, int d, const neko_tok_params* host_params,
                                  const int64_t* tokens, const float* d_token_embeddings, float* d_embed_table,
                                  float* d_pos_table, float* d_sep, float* d_patch_emb, void* workspace,
                                  int64_t workspace_bytes, void* stream);
/* neko_patch_resblock_bwd with the patches cut into fixed chunks of 8: each chunk stores its weight / GroupNorm gradient
 * partials to a workspace slot, and the slots are folded in a fixed order. */
int64_t neko_patch_resblock_bwd_ordered_workspace_bytes(int n_img, int Himg, int Wimg, int patch);
int neko_patch_resblock_bwd_ordered(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch,
                                    int C, int groups, const float* conv1_w, const float* conv1_b,
                                    const float* gn_w, const float* gn_b, const float* conv2_w,
                                    const float* gn_stats, const uint16_t* d_patches_bf16,
                                    float* d_conv1_w, float* d_conv1_b, float* d_gn_w, float* d_gn_b,
                                    float* d_conv2_w, float* d_conv2_b, void* workspace, int64_t workspace_bytes,
                                    void* stream);
/* neko_patch_pos_bwd as a sorted scatter-add (d % 4 == 0).  n_row_bins / n_col_bins: rows of d_row_tab / d_col_tab; bins
 * outside them are skipped. */
int64_t neko_patch_pos_bwd_ordered_workspace_bytes(int P, int n_row_bins, int n_col_bins);
int neko_patch_pos_bwd_ordered(const float* dx, int P, int d, const int32_t* row_bin, const int32_t* col_bin,
                               float* d_row_tab, int n_row_bins, float* d_col_tab, int n_col_bins, void* workspace,
                               int64_t workspace_bytes, void* stream);
/* neko_sumsq_f32 over fixed 8192-element blocks, then one CTA folds the block partials in a fixed order. */
int64_t neko_sumsq_f32_ordered_workspace_bytes(int64_t n);
int neko_sumsq_f32_ordered(const float* x, int64_t n, float* out_accum, void* workspace, int64_t workspace_bytes,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Data-parallel gradient all-reduce over NVLink peer memory (replaces the DDP bucket all-reduce the reference gets from
 * Accelerate: train.py:26-40,107; trainer.py:176-186 -- SUM over ranks, then / world).  One process per GPU; every
 * rank's gradient arena and a small signal buffer are mapped into every process with the two ipc calls below.
 * neko_p2p_allreduce_f32 is a two-shot, in-place, deterministic fp32 all-reduce of arena elements [lo, hi) whose CTAs
 * (128 threads, no shared memory) are sized to co-reside with the persistent GEMM CTAs of backward; it must be
 * called by every rank with the same (lo, hi) in the same order.  `state`: two zero-initialised uint32 words private to
 * the rank (launch counter, CTA arrival counter) -- all barrier bookkeeping is device state, so the launch replays from a
 * CUDA graph.  host_bufs / host_sigs are HOST arrays of `world` device pointers (index = rank, own pointers included);
 * each signal buffer holds `world` zero-initialised uint32 words.
 * ------------------------------------------------------------------------------------------- */
/* Measurement aid: n_ctas CTAs of `threads` threads that idle for `ns` nanoseconds (no shared memory).  Used to queue a whole
 * step behind a blocker so that per-kernel CUDA events see no launch gaps (bench.py), and to test which kernels co-reside. */
int neko_debug_spin(int n_ctas, int threads, long long ns, int max_shared_carveout, void* stream);
/* Device-wide shared-memory carveout preference (cudaDeviceSetCacheConfig) for kernels without one of their own: with
 * on != 0 every kernel of the step runs in the split the all-reduce CTAs hold, so none waits for an SM to drain. */
int neko_prefer_shared_carveout(int on);
int neko_ipc_export(const void* dev_ptr, unsigned char* handle_out /* 64 bytes */, long long* offset_out);
int neko_ipc_import(const unsigned char* handle /* 64 bytes */, long long offset, void** dev_ptr_out);
int neko_ipc_close(void* dev_ptr, long long offset);
/* Copy-engine flavour of the same all-reduce (what neko_b200/dp.py runs by default): NVLink traffic is moved by
 * neko_memcpy_async between peer-mapped buffers (DMA engines, no SM), neko_p2p_signal_wait is the one-warp cross-rank
 * barrier between the steps (per channel c: signal words 32 + 8c .. of the 64-word signal buffers, launch counter in state[2 + c] of the 8-word state) and
 * neko_reduce_planes_f32 sums the staged contributions: dst[i] = scale * sum_q (q == self ? dst[i] : stage[q*plane+i]). */
int neko_memcpy_async(void* dst, const void* src, long long bytes, void* stream);
int neko_p2p_signal_wait(void* const* host_sigs, unsigned* state, int rank, int world, int channel /* 0..3 */, void* stream);
int neko_reduce_planes_f32(float* dst, const float* stage, long long plane, int n_planes, int self, long long n, float scale, void* stream);
/* host_stage (nullable): HOST array of `world` device pointers to every rank's staging buffer (world planes of stage_plane
 * floats each).  When given, the exchange runs push style -- contributions are WRITTEN into the owner's staging planes
 * at stage_off (the caller advances it by ceil((hi-lo)/world) + 4 per call within a step), reduced there, and the result is
 * written into every arena: no loads cross NVLink.  NULL: pull style (peer loads, in place, no staging memory). */
int neko_p2p_allreduce_f32(void* const* host_bufs, void* const* host_sigs, void* const* host_stage, long long stage_plane,
                           long long stage_off, unsigned* state, int rank, int world, long long lo, long long hi, float scale,
                           int n_ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NEKO_B200_H */
