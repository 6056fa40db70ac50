/*
 * ymp.h - C ABI of libymp_b200.so: the sm_100a kernels behind the mPLUG-Video (Youku-mPLUG)
 * pre-training hot path.
 *
 * The reference (X-PLUG/Youku-mPLUG) has no native boundary of its own: every device op on the
 * path is a PyTorch library call made from models/{vision_transformer,modeling_distributed_gpt3,
 * distributed_gpt3}.py.  Each entry point below therefore cites the reference *call site* whose
 * device computation it replaces (file:line, relative to the reference repo root).
 *
 * Contract (all entry points):
 *   - plain pointers + sizes only; device pointers unless stated otherwise; no torch types
 *   - never allocates, never frees, never synchronises; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*), so every call is CUDA-graph capturable
 *   - returns 0 on success, a negative YMP_E* code on failure; ymp_last_error() returns a
 *     thread-local human-readable message for the last failure on this thread
 *   - bf16 tensors are raw uint16 storage (__nv_bfloat16), fp32 tensors are float
 */
#ifndef YMP_H_
#define YMP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YMP_OK 0
#define YMP_EINVAL (-1)  /* bad argument (shape, alignment, null pointer) */
#define YMP_ECUDA (-2)   /* CUDA runtime / driver error (message has the CUDA string) */
#define YMP_ENOSUP (-3)  /* configuration not supported by the compiled kernels */

const char* ymp_last_error(void);
/* ABI version of this header; bumped on any struct change. */
int ymp_abi_version(void);
/* Number of kernel launches this process has enqueued through the library (for gpu_launches). */
uint64_t ymp_launch_count(void);
/* Programmatic dependent launch for the calling thread's next launches of ymp_gemm_skinny, ymp_layernorm_fwd and the
 * mma.sync ymp_attn_fwd (the single-token decoding step): each of those kernels may then start while its predecessor in
 * the stream drains (it waits on the device before reading the predecessor's output).  Returns the previous setting. */
int ymp_set_pdl(int on);

/* ------------------------------------------------------------------------------------------
 * Dropout of the GPT-3 decoder (the reference keeps the frozen decoder in train() mode, so
 * hidden_dropout / attention_dropout = 0.1 are live: models/modeling_distributed_gpt3.py:631 embedding,
 * :732 attention probabilities, :1056-1078 the two bias-dropout-adds).  No mask tensor exists: a keep
 * decision is Philox4x32-10(key = seed, counter = (column >> 2, row, site, offset)).word[column & 3]
 * >= floor(p * 2^32), kept values are scaled by 1 / (1 - p), and the backward kernels regenerate the same
 * bits (csrc/philox.cuh; CPU restatement for the parity tests: oracle/philox.py).
 *   rng    : DEVICE pointer to {seed, offset} (uint64 x 2), read when the kernel runs - a captured CUDA
 *            graph therefore draws fresh masks on every replay; NULL (or p == 0) disables dropout
 *   site   : which dropout call of the decoder pass (YMP_DROP_SITE_*)
 *   row / column: logical coordinates - hidden states [B*S, H]: row = b*S + s, column = feature;
 *            attention probabilities: row = (seq*heads + head)*s_q + query, column = key
 * ------------------------------------------------------------------------------------------ */
typedef struct ymp_dropout_spec {
  const uint64_t* rng;
  uint32_t site;
  float p;
} ymp_dropout_spec;
#define YMP_DROP_SITE_EMBED 0u                              /* embedding dropout (:631) */
#define YMP_DROP_SITE_ATTN(layer) (4u * (layer) + 1u)       /* attention probabilities of layer (:732) */
#define YMP_DROP_SITE_BDA_ATTN(layer) (4u * (layer) + 2u)   /* bias-dropout-add after attention (:1056-1062) */
#define YMP_DROP_SITE_BDA_MLP(layer) (4u * (layer) + 3u)    /* bias-dropout-add after the MLP (:1072-1078) */

/* ------------------------------------------------------------------------------------------
 * GEMM  D[M,N] = epilogue( alpha * op(A)[M,K] . op(B)[N,K]^T )          tcgen05 + TMA + TMEM
 *
 * Replaces: F.linear in ViT Attention qkv/proj (models/vision_transformer.py:171-176,205),
 * temporal_fc (:250), Mlp fc1/fc2 (:103-110), AttentionPool in/out proj + MLP (:368-374),
 * visual_fc (models/distributed_gpt3.py:136), GPT-3 query_key_value / dense / dense_h_to_4h /
 * dense_4h_to_h (models/modeling_distributed_gpt3.py:843-857,562-578), the tied LM head
 * (:1348-1350), and every dgrad / wgrad GEMM autograd derives from them.
 *
 * Operand storage (bf16):
 *   a_mn_major = 0: A is [M,K] row-major, row stride lda  ("K-major")
 *   a_mn_major = 1: A is stored transposed, [K,M] row-major, row stride lda ("MN-major")
 *   b_mn_major = 0: B is [N,K] row-major, row stride ldb  (a torch nn.Linear weight)
 *   b_mn_major = 1: B is [K,N] row-major, row stride ldb
 *   All leading dimensions must be multiples of 8 elements and base pointers 16-byte aligned.
 * Epilogue, applied in this order to v = alpha * acc:
 *   v += bias[n]                         (bias: bf16 [N], optional)
 *   if aux_out: aux_out[m,n] = bf16(act'(v)) when act != NONE (what the backward pass multiplies by),
 *                            = bf16(v)       when act == NONE                       (ld = ldd)
 *   v = act(v)                           (YMP_ACT_*; skipped when aux_in is set)
 *   if aux_in:  v *= aux_in[m,n]         (backward of an activation: aux_in is the act' saved above,
 *                                          so the backward epilogue needs no transcendental)
 *   if drop:    v = dropout(v)           (row = m, column = n; bias-dropout-add: residual + dropout(x + bias))
 *   v += residual[m,n]                   (bf16 or fp32 [M,N], row stride ldr, optional)
 *   D[m,n] = v  (bf16 or fp32) ; or atomically D[m,n] += v (fp32, accumulate=1, used by split-K)
 * ------------------------------------------------------------------------------------------ */
#define YMP_ACT_NONE 0
#define YMP_ACT_GELU_ERF 1  /* nn.GELU() exact: ViT / abstractor MLP (vision_transformer.py:94) */
#define YMP_ACT_GELU_TANH 2 /* Megatron bias_gelu_impl: GPT-3 MLP (modeling_distributed_gpt3.py:586) */

#define YMP_DT_BF16 0
#define YMP_DT_F32 1

typedef struct ymp_gemm_args {
  const void* A;
  const void* B;
  void* D;
  int32_t M, N, K;
  int32_t lda, ldb, ldd;
  int32_t a_mn_major, b_mn_major;
  const void* bias;     /* bf16 [N] or NULL */
  const void* residual; /* bf16 or fp32 (residual_dtype) [M,N] or NULL */
  int32_t ldr;
  int32_t act;          /* YMP_ACT_* */
  void* aux_out;        /* bf16 [M,N] (ld = ldd) or NULL: act'(pre-activation) (or the value if act=NONE) */
  const void* aux_in;   /* bf16 [M,N] (ld = ldd) or NULL: element-wise multiplier */
  int32_t out_dtype;    /* YMP_DT_BF16 | YMP_DT_F32 */
  int32_t accumulate;   /* 1: D (fp32) += result using atomics */
  int32_t split_k;      /* >=1; >1 requires accumulate=1 and out_dtype=F32; 0 = library picks */
  float alpha;
  int32_t tile_n;       /* 0 = auto, else 128 or 256 */
  int32_t res_row_mod;  /* >0: residual row = m % res_row_mod (broadcast tables: position embeddings) */
  int32_t d_row_block;  /* >0: D row = (m / d_row_block) * d_row_stride + m % d_row_block           */
  int32_t d_row_stride; /*     (writes [B*Q] rows into a [B, S>=Q] buffer without a copy)           */
  int32_t residual_dtype; /* YMP_DT_BF16 (default) | YMP_DT_F32: the residual streams are kept in fp32 */
  ymp_dropout_spec drop;  /* dropout before the residual add (not together with aux_out) */
  /* Fused im2col (the patch embedding, models/vision_transformer.py:392-398: `(b t) c h w` rearrange + Conv2d(k = stride
   * = P) as ONE GEMM): when im2col_P > 0, A is not a matrix but the video [B, C, T, H, W] (bf16, contiguous); row
   * m = (b*N + n)*T + t (n = py*(W/P) + px: the encoder's patch-major token order), column k = (c, iy, ix) as in
   * conv_weight.flatten(1).  The TMA producer gathers each 128-row x 64-column operand tile straight from the video as
   * four 16-column sub-tiles (one pixel row of every patch: 5-D boxes {16 px, 1 row, T frames} = T rows x 32 bytes, i.e.
   * SWIZZLE_32B atoms; one tcgen05.mma K-step per sub-tile); no patch matrix is written.  Needs P = 16, T % 8 == 0,
   * 128 % T == 0, M = B*N*T, K = C*P*P, a_mn_major = 0. */
  int32_t im2col_P, im2col_B, im2col_C, im2col_T, im2col_H, im2col_W;
} ymp_gemm_args;

int ymp_gemm(const ymp_gemm_args* a, void* stream);

/* Skinny GEMM for single-token decoding (KV-cache steps of sample() / beam_search(),
 * models/modeling_distributed_gpt3.py:1620-1886): y[M, N] = epilogue(x[M, K] . w[N, K]^T), 1 <= M <= 8.  One pass over the
 * weights, HBM-bound, mma.sync fed straight from global memory (csrc/gemv.cu).  Epilogue: + bias[n], act (YMP_ACT_*),
 * + residual[m, n], store.  ymp_gemm_skinny_batch takes the same arguments with 1 <= M <= 64 (the step of a batch of beam
 * searches: n_samples x beam rows); both compute row m of y from row m of x only, bit for bit, whatever M is (the kernel
 * layout is chosen from N and K), so the two agree on every row. */
typedef struct ymp_gemm_skinny_args {
  const void* x;         /* bf16 [M, K], row stride ldx */
  const void* w;         /* bf16 [N, K], row stride ldw (an nn.Linear weight) */
  const void* bias;      /* bf16 [N] or NULL */
  const void* residual;  /* bf16 / fp32 [M, N] (residual_dtype), row stride ldr, or NULL */
  void* y;               /* bf16 / fp32 [M, N] (out_dtype), row stride ldy */
  int32_t M, N, K, ldx, ldw, ldr, ldy;
  int32_t act, residual_dtype, out_dtype;
  /* optional second copy of the bf16 result at a row offset read on the device: y2[m * ldy2 + *y2_off_dev * y2_off_stride + n]
   * (the new token's K/V row written straight into the KV cache at the device-side cache length) */
  void* y2;
  const int64_t* y2_off_dev;
  int64_t ldy2, y2_off_stride;
  /* optional fused LayerNorm of the complete fp32 result (the next sub-layer's input): the CTA that finishes last
   * (ticket in *ln_counter, which must be 0 at launch and is reset to 0) writes ln_out[m, :] = LN(y[m, :]) in bf16 with
   * exactly the arithmetic of ymp_layernorm_fwd - one kernel boundary less per sub-layer of the decoding step.  M <= 8 only. */
  const void* ln_gamma;  /* bf16 [N] */
  const void* ln_beta;   /* bf16 [N] */
  void* ln_out;          /* bf16 [M, N], row stride ld_ln */
  uint32_t* ln_counter;
  int32_t ld_ln;
  float ln_eps;
} ymp_gemm_skinny_args;
int ymp_gemm_skinny(const ymp_gemm_skinny_args* a, void* stream);
int ymp_gemm_skinny_batch(const ymp_gemm_skinny_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * LayerNorm (fp32 statistics, bf16 in/out), one warp per row.
 * Replaces LayerNormWithForceFP32.forward (models/vision_transformer.py:69-71: cast->LN->cast,
 * three kernels) and megatron MixedFusedLayerNorm (models/modeling_distributed_gpt3.py:1002-1020,
 * 1131-1135) plus their autograd backward.
 *   in_rows (optional int32 [rows]): output row r normalises input row in_rows[r]; used for the
 *   final TimeSformer norm to emit the reference's (t n) token order (vision_transformer.py:582-585).
 * ------------------------------------------------------------------------------------------ */
typedef struct ymp_layernorm_args {
  const void* x;      /* bf16 [*, D], row stride ldx */
  const void* gamma;  /* bf16 [D] */
  const void* beta;   /* bf16 [D] */
  void* y;            /* bf16 [rows, D], row stride ldy */
  float* mean;        /* fp32 [rows] or NULL (saved for backward) */
  float* rstd;        /* fp32 [rows] or NULL */
  const int32_t* in_rows;
  int32_t rows, D, ldx, ldy;
  float eps;
  int32_t x_dtype;    /* YMP_DT_BF16 | YMP_DT_F32 (fp32 residual stream in) */
  int32_t y_dtype;    /* YMP_DT_BF16 | YMP_DT_F32 */
} ymp_layernorm_args;
int ymp_layernorm_fwd(const ymp_layernorm_args* a, void* stream);

typedef struct ymp_layernorm_bwd_args {
  const void* dy;     /* bf16 [rows, D], stride lddy */
  const void* x;      /* bf16, the forward input (stride ldx) */
  const void* gamma;
  const float* mean;
  const float* rstd;
  const void* add;    /* optional bf16 [*, D] (stride ldadd): gradient of the skip branch, added to dx */
  void* dx;           /* bf16, same indexing/stride as x */
  float* dgamma;      /* fp32 [D], ACCUMULATED (atomics); NULL (with dbeta) when the affine is frozen */
  float* dbeta;
  const int32_t* in_rows;
  int32_t rows, D, ldx, lddy, ldadd;
  int32_t x_dtype;    /* dtype of x (dx is always bf16, same row stride in elements) */
  void* dx_drop;      /* optional second output, bf16, indexed like dx: dropout_backward(dx) = dx * mask / (1-p) for the
                         dropout site that produced this LayerNorm's input stream (row = x row, column = feature):
                         the A operand of the dgrad GEMM below that bias-dropout-add */
  ymp_dropout_spec drop;
} ymp_layernorm_bwd_args;
int ymp_layernorm_bwd(const ymp_layernorm_bwd_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused attention: O = softmax(scale * Q K^T [causal]) V, scores never materialised.
 * Replaces Attention.forward core (models/vision_transformer.py:179-204), nn.MultiheadAttention
 * inside AttentionPool (:371) and GPT3CoreAttention.forward (models/modeling_distributed_gpt3.py:
 * 734-817: baddbmm -> scale/mask(-10000)/softmax -> bmm) and their backward.
 *
 * Rows of a sequence are found through a ymp_seqmap, so Q/K/V are read in place from packed QKV
 * GEMM outputs:  row(s, i) =
 *     i <  n_prefix : prefix_base + (prefix_per_seq ? s : s / seq_div) * prefix_stride + i
 *     i >= n_prefix : (s / seq_div) * outer_stride + (s % seq_div) * inner_stride
 *                     + (i - n_prefix) * pos_stride
 * element(s, i, head, d) = base[row(s,i) * ld + head * head_stride + d].
 *   dense [n_seq, S] rows:           seq_div=1, outer_stride=S, pos_stride=1
 *   TimeSformer frame (b,t) tokens stored (b, n, t) with one cls row per b appended after all
 *   tokens (vision_transformer.py:254-267):  seq_div=T, outer_stride=N*T, inner_stride=1,
 *   pos_stride=T, n_prefix=1, prefix_base=B*N*T, prefix_stride=1
 * lse: fp32 [n_seq, n_heads, s_q] (natural log), needed by the backward.
 * ------------------------------------------------------------------------------------------ */
#define YMP_MASK_NONE 0
#define YMP_MASK_CAUSAL 1
#define YMP_MASK_BLOCK 2

typedef struct ymp_seqmap {
  int32_t seq_div;
  int32_t n_prefix;
  int32_t prefix_per_seq;
  int32_t _pad;
  int64_t outer_stride, inner_stride, pos_stride;
  int64_t prefix_base, prefix_stride;
} ymp_seqmap;

typedef struct ymp_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* o;
  float* lse;
  int32_t ldq, ldk, ldv, ldo;
  int32_t q_head_stride, k_head_stride, v_head_stride, o_head_stride;
  ymp_seqmap map_q, map_kv, map_o;
  int32_t n_seq, n_heads, head_dim, s_q, s_kv;
  int32_t mask;        /* YMP_MASK_NONE | YMP_MASK_CAUSAL | YMP_MASK_BLOCK */
  int32_t mask_block;  /* YMP_MASK_BLOCK: position i attends j iff i / mask_block == j / mask_block.
                          Packs many short sequences (TimeSformer temporal attention over T frames,
                          vision_transformer.py:246-248) into one tensor-core tile. */
  int64_t total_rows;  /* >0 (dense packed sequences only): rows beyond total_rows do not exist, so
                          the last sequence may be shorter than s_q */
  float scale;
  ymp_dropout_spec drop;  /* dropout of the attention probabilities (tcgen05 kernels only): O = dropout(P) V, the
                             softmax statistics (lse) stay those of the undropped P */
  const int32_t* s_kv_dev; /* optional DEVICE scalar: only the first min(s_kv, *s_kv_dev) keys exist.  Lets a captured
                             CUDA graph of the single-token decoding step follow the growing KV cache (forward only,
                             served by the mma.sync kernels) */
  const int32_t* kv_rows;  /* optional DEVICE table [n_seq, ld_kv_rows] (single-query decoding only, s_q == 1): key j of
                             sequence s is row kv_rows[s * ld_kv_rows + j] of the k and v buffers (map_kv unused).  A beam
                             reorder of a batched beam search then moves table entries, not cached keys; every entry
                             below s_kv must be a valid row even past *s_kv_dev */
  int32_t ld_kv_rows;
} ymp_attn_args;
int ymp_attn_fwd(const ymp_attn_args* a, void* stream);

typedef struct ymp_attn_bwd_args {
  ymp_attn_args fwd;      /* the forward call's arguments (q,k,v,o,lse and maps) */
  const void* dout;       /* bf16, addressed by map_do / lddo / do_head_stride */
  void* dq;               /* bf16 outputs; every addressed element is written exactly once */
  void* dk;
  void* dv;
  float* delta_ws;        /* workspace fp32 [n_seq * n_heads * s_q] (rowsum(dO*O), written then read) */
  int32_t lddo, lddq, lddk, lddv;
  int32_t do_head_stride, dq_head_stride, dk_head_stride, dv_head_stride;
  ymp_seqmap map_do, map_dq, map_dkv;
} ymp_attn_bwd_args;
int ymp_attn_bwd(const ymp_attn_bwd_args* a, void* stream);
/* Diagnostic: which kernel family served the last ymp_attn_fwd / ymp_attn_bwd call of this thread (-1: none yet).
 * tcgen05 tiles serve head_dim 64 / 80 / 88 / 96 at any key range; warp-per-sequence kernels the packed
 * block-diagonal (temporal, T <= 16) case; the mma.sync kernels remain for head_dim 128 and for a few query
 * rows against a long cache (single-token decoding). */
#define YMP_ATTN_PATH_MMA_SYNC 0
#define YMP_ATTN_PATH_TCGEN05 1
#define YMP_ATTN_PATH_SMALL 2
#define YMP_ATTN_PATH_DECODE 3  /* one query row per sequence: streaming kernel of the decoding step */
int ymp_attn_last_path(void);

/* ------------------------------------------------------------------------------------------
 * Patch-embedding im2col: video [B,C,T,H,W] bf16 -> patches [(b,n,t), C*P*P] (the A operand of
 * the conv-as-GEMM).  Replaces the `(b t) c h w` rearrange + Conv2d(k=stride=P)
 * (models/vision_transformer.py:546-548,397).
 * ------------------------------------------------------------------------------------------ */
typedef struct ymp_im2col_args {
  const void* video;
  void* out;
  int32_t B, C, T, H, W, P, ldo;
} ymp_im2col_args;
int ymp_im2col(const ymp_im2col_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Input pipeline tail on the GPU (SURVEY.md 8f N4): uint8 clips [B,T,H,W,C] (decoded, resized and
 * augmented frames) -> normalised bf16 model input [B,C,T,H,W].  Replaces
 * volume_transforms.ClipToTensor (`clip / 255.`, dataset/video_utils/volume_transforms.py:25-37) +
 * video_transforms.Normalize (`sub_(mean).div_(std)`, dataset/video_utils/functional.py:125-137) +
 * the default collate + `.to(device)` + bf16 cast (dataset/__init__.py:60-85), and cuts the
 * host->device traffic 4x (1 byte per value instead of an fp32).
 * lut[c*256 + v] is the bf16 result for channel c and pixel value v; the host fills it with the
 * reference's own fp32 op order, so the kernel is bit-exact by construction (a gather).
 * ------------------------------------------------------------------------------------------ */
typedef struct ymp_clip_args {
  const void* frames;  /* uint8 [B,T,H,W,C] contiguous */
  void* out;           /* bf16 [B,C,T,H,W] contiguous */
  const void* lut;     /* bf16 [C*256] (device memory) */
  int32_t B, T, H, W, C;
} ymp_clip_args;
int ymp_clip_normalize(const ymp_clip_args* a, void* stream);

/* y = dropout(x) over a [rows, cols] matrix (bf16 or fp32, in place allowed): the embedding dropout
 * (models/modeling_distributed_gpt3.py:631; logical row = row0 + r) and the mask export used by the parity tests. */
typedef struct ymp_dropout_args {
  const void* x;
  void* y;
  int32_t rows, cols, ldx, ldy;
  int32_t dtype;   /* YMP_DT_BF16 | YMP_DT_F32 (both x and y) */
  int64_t row0;
  ymp_dropout_spec drop;
} ymp_dropout_args;
int ymp_dropout(const ymp_dropout_args* a, void* stream);

/* Word-embedding gather + learned position add, written straight into the decoder input
 * buffer [B, S, hidden] at rows row_offset..row_offset+L-1 of each sample.  Replaces
 * word_embeddings(ids) + cat + position add (models/distributed_gpt3.py:155-156,
 * models/modeling_distributed_gpt3.py:640-650).  Index work is bit-exact. */
typedef struct ymp_embed_args {
  const int64_t* ids;  /* [B, L] */
  const void* table;   /* bf16 [vocab, hidden] */
  const void* pos;     /* bf16 [max_pos, hidden] or NULL */
  void* out;           /* bf16 [B*S, hidden] rows of stride ldo */
  int32_t B, L, S, row_offset, hidden, vocab, ldo;
  int32_t out_dtype;   /* YMP_DT_BF16 | YMP_DT_F32 */
} ymp_embed_args;
int ymp_embed_gather(const ymp_embed_args* a, void* stream);

/* Softmax cross entropy over the vocabulary, per-token (unreduced) losses.  Replaces
 * logits.clone().float() + vocab_parallel_cross_entropy (modeling_distributed_gpt3.py:1353-1359).
 * bwd: dlogits = grad_rows[row] * (softmax - onehot), may alias logits. */
typedef struct ymp_ce_args {
  const void* logits;      /* bf16 [rows, V], stride ld */
  const int64_t* labels;   /* [rows] */
  float* loss;             /* fp32 [rows] (fwd) */
  float* lse;              /* fp32 [rows] (fwd out / bwd in) */
  const float* grad_rows;  /* fp32 [rows] (bwd) */
  void* dlogits;           /* bf16 [rows, V] (bwd) */
  int32_t rows, V, ld;
} ymp_ce_args;
int ymp_ce_fwd(const ymp_ce_args* a, void* stream);
int ymp_ce_bwd(const ymp_ce_args* a, void* stream);

/* out[c] += sum_r in[r,c]  (bias gradients, batch sums).  out is fp32 and ACCUMULATED. */
typedef struct ymp_colsum_args {
  const void* in;  /* bf16 [R, C], stride ld */
  float* out;      /* fp32 [C] */
  int32_t R, C, ld;
} ymp_colsum_args;
int ymp_colsum(const ymp_colsum_args* a, void* stream);

/* broadcast=0: out[g,:] = scale * sum_t in[g,t,:]   (cls mean over frames, vision_transformer.py:262)
 * broadcast=1: out[g,t,:] = scale * in[g,:]          (its backward) */
typedef struct ymp_group_args {
  const void* in;
  void* out;
  int32_t G, T, C, ld_in, ld_out, broadcast;
  float scale;
} ymp_group_args;
int ymp_group_reduce(const ymp_group_args* a, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer step on flat buffers (next row N1 of SURVEY.md section 8f; needed so that the timed
 * training step skips no work).  Replaces DeepSpeed FusedAdam(adam_w_mode) + global-norm clipping
 * (reference utils.py:490-526; invoked by model.step(), run_pretrain_distributed_gpt3.py:137).
 *   ymp_sumsq : *out += sum(g[i]^2)            (fp32, atomics; the caller zeroes *out)
 *   ymp_adamw : g' = g * grad_scale * min(1, max_grad_norm / (sqrt(*sumsq)*grad_scale + 1e-6))
 *               AdamW on the fp32 master weights, bf16 model weights refreshed in the same pass
 *               (128-bit accesses, 26 bytes of HBM traffic per parameter incl. the optional gradient reset).
 * ------------------------------------------------------------------------------------------ */
int ymp_sumsq(const float* g, int64_t n, float* out, void* stream);

typedef struct ymp_adamw_args {
  float* master;        /* fp32 [n] */
  void* param;          /* bf16 [n] */
  const float* grad;    /* fp32 [n] */
  float* m;             /* fp32 [n] */
  float* v;             /* fp32 [n] */
  const float* sumsq;   /* device scalar or NULL (no clipping) */
  int64_t n;
  int32_t step;         /* 1-based step count for bias correction */
  float lr, beta1, beta2, eps, weight_decay;
  float grad_scale;     /* e.g. 1/world_size after a summing all-reduce */
  float max_grad_norm;  /* <= 0: no clipping */
  const float* hyper;   /* optional DEVICE array {lr, weight_decay, 1-beta1^t, 1-beta2^t}; when set it
                           overrides lr / weight_decay / step so a captured CUDA graph can follow an
                           lr schedule without re-capture */
  int32_t zero_grad;    /* 1: the kernel also writes zeros to grad (it is the accumulator of the next step) */
} ymp_adamw_args;
int ymp_adamw(const ymp_adamw_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* YMP_H_ */
