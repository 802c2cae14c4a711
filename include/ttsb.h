/*
 * ttsb.h -- C ABI of libttsb.so, the B200 (sm_100a) kernels behind the ForwardTransformer text->mel hot path
 * of as-ideas/TransformerTTS.
 *
 * The reference has no FFI/plugin interface: its boundary is the Python API (model/models.py:344-642,
 * data/audio.py:88-92).  The host-side mirror of that API lives in transformertts_b200/ and binds these entry
 * points with ctypes (transformertts_b200/lib.py); INTEGRATION.md shows the stub a maintainer of the reference
 * would add.  Each entry point names the reference lines it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative TTSB_ERR_* otherwise; ttsb_last_error() gives the text
 *     (thread-local);
 *   - all pointers are CALLER-OWNED DEVICE pointers unless the name ends in _host; nothing is allocated inside;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, no hidden synchronisation;
 *   - activations are row-major (B, T, C) channels-last as in Keras; "hi/lo" pairs are the bf16 split of an fp32
 *     tensor (x ~= hi + lo) used by the 3-pass bf16 tensor-core mode; lo pointers may be NULL in single-pass mode;
 *   - packed weights are bf16 [N_pad, K] (K contiguous), produced from the Keras (K, N) / (k, Cin, Cout) layout by
 *     ttsb_pack_weight.
 */
#ifndef TTSB_H_
#define TTSB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTSB_OK 0
#define TTSB_ERR_INVALID_ARGUMENT (-1)
#define TTSB_ERR_CUDA (-2)
#define TTSB_ERR_UNSUPPORTED (-3)

#define TTSB_ABI_VERSION 3

/* precision of the tensor-core products */
#define TTSB_PREC_BF16 0   /* single bf16 pass, fp32 accumulate */
#define TTSB_PREC_BF16X3 1 /* hi*hi + lo*hi + hi*lo, fp32 accumulate (fp32-class accuracy) */
#define TTSB_PREC_FP16 2   /* ttsb_mha_fwd only: single IEEE fp16 pass (11-bit mantissa), q/k/vT hold fp16 */

/* implementation selector (debug): tcgen05/TMA kernels, or the plain SIMT CUDA kernels kept for bring-up */
#define TTSB_IMPL_TCGEN05 0
#define TTSB_IMPL_SIMT 1

const char* ttsb_last_error(void);
int ttsb_abi_version(void);
/* number of kernels this library has launched since load / since the last reset (bench.py "gpu_launches") */
int64_t ttsb_launch_count(void);
void ttsb_reset_launch_count(void);
/* a host that replays a captured CUDA graph of N library launches adds N per replay, so the counter keeps meaning
 * "kernels of this library that ran" */
void ttsb_add_launch_count(int64_t n);

/* Dropout decisions are a stateless hash of (seed, site, element index); `seed` is a by-value argument of every kernel that
 * draws them.  The 32-bit word *salt_dev (DEVICE memory) is XORed into that seed by all kernels launched afterwards on the
 * stream (stream-ordered device-to-device copies into the library's constant memory; 0 after load).  A host that replays a
 * captured training step puts this call at the head of the capture and rewrites *salt_dev before every replay, which gives
 * each step its own masks although the captured `seed` arguments never change. */
int ttsb_set_dropout_salt(const uint32_t* salt_dev, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Weight / activation preparation
 * ------------------------------------------------------------------------------------------------------- */
/* Keras kernel (K, N) fp32 (Conv1D (k, Cin, Cout) is the same memory with K = k*Cin) -> packed bf16 hi/lo
 * [n_pad, K], rows >= N zero.  w_lo may be NULL. */
int ttsb_pack_weight(const float* w_kn, int K, int N, int n_pad, void* w_hi, void* w_lo, void* stream);
/* Batched refresh of packed operands (training: the weights change every step).  One descriptor per destination block:
 *   dst[r][c] = (r < R && c % cb < cb_valid) ? src[r*sr + (c / cb)*s_outer + (c % cb)*s_inner] : 0,   r < R_pad, c < C_cols
 * which covers the forward packing (K,N)->[N_pad,K], the data-gradient packings of Dense ((K,N)->[K_pad,N_pad]) and Conv1D
 * ((k,Cin,Cout)->[Cin_pad, k*Cout_pad]) and zero-padded fp32 vectors (bias, LayerNorm gamma/beta).  The descriptor array
 * lives in DEVICE memory (built once); one launch refreshes everything. */
typedef struct ttsb_pack_desc {
  const float* src;
  void* dst;
  int R, R_pad, C_cols;
  int cb, cb_valid;
  long long sr, s_outer, s_inner;
  int dst_ld;
  int dst_f32; /* 1: destination is fp32, 0: bf16 */
} ttsb_pack_desc;
int ttsb_repack_batched(const ttsb_pack_desc* descs_device, int n, void* stream);
/* fp32 [n] -> bf16 hi (and lo when non-NULL) */
int ttsb_split_bf16(const float* x, int64_t n, void* x_hi, void* x_lo, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Encoder prologue: Embedding + LayerNorm + scalar*PE   (model/models.py:522, model/layers.py:299-300)
 * tokens int32 (B,T); emb (vocab,d); pe (max_pos,d) fp32; pos_scalar device scalar.
 * ------------------------------------------------------------------------------------------------------- */
int ttsb_embed_ln_pe_fwd(const int32_t* tokens, const float* emb, const float* gamma, const float* beta,
                         const float* pe, const float* pos_scalar, int B, int T, int d, int vocab, float eps,
                         float* out_f32, void* out_hi, void* out_lo, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Tensor-core GEMM family:  Dense, dual-input Dense (concat projection) and Conv1D(k, 'same')
 *   (model/layers.py:134-136,149 MHA projections; :93-94 FFN; :19-26 Conv1D; model/models.py:422 mel Dense)
 *
 *   out[b,t,:] = epilogue( bias + sum_s  A_{src[s]}[b, t + shift[s], :] @ W[koff_s : koff_s + K_s, :] )
 *
 * Segments: a Dense has one segment (shift 0); the concat projection has two sources; a k-tap 'same' conv has k
 * segments over the same source with shifts -(k-1)/2 ... ; rows outside [0,T) read as zero.
 * Epilogue (in this order): +bias, relu?, +residual?, LayerNorm over the first ln_n columns?, zero rows t >= row_len[b]?.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct ttsb_gemm_args {
  int B, T;                 /* rows = B*T */
  int N;                    /* logical output columns */
  int block_n;              /* N tile (multiple of 16, <= 256); packed W has n_tiles*block_n rows */
  int num_segments;         /* 1..4 */
  int seg_src[4];           /* 0 or 1: which A source */
  int seg_shift[4];         /* time shift of the source rows */
  int seg_k[4];             /* K of the segment (multiple of 64) */
  const void* a_hi[2];      /* bf16 (B,T,lda) sources */
  const void* a_lo[2];      /* NULL in TTSB_PREC_BF16 */
  int lda[2];               /* row stride in elements */
  int a_col0[2];            /* first column of the source inside its row */
  const void* w_hi;         /* packed bf16 [n_tiles*block_n, K_total] */
  const void* w_lo;
  const float* bias;        /* [n_tiles*block_n] (zero padded past N) or NULL */
  int relu;
  const float* residual;    /* fp32 (B,T,ld_res) or NULL */
  int ld_res;
  const float* ln_gamma;    /* LayerNorm params [block_n] (padded) or NULL */
  const float* ln_beta;
  float ln_eps;
  const int32_t* row_len;   /* [B] valid lengths or NULL */
  float* out_f32;           /* any of the three may be NULL */
  void* out_hi;
  void* out_lo;
  int ld_out;               /* row stride of all outputs, >= n_tiles*block_n, multiple of 8 (16 with 16-bit outputs) */
  int out_fp16;             /* 1: out_hi receives IEEE fp16 (single plane) instead of bf16 hi/lo */
  float* out_preln;         /* optional fp32 (B,T,ld_out): value before the LayerNorm (saved for the backward pass) */
  /* training dropout (keras semantics, stateless mask from (seed, site, element index)): drop_pre on the GEMM output
   * after bias/ReLU and before the residual add; drop_post on the LayerNorm output.  The element index of output column
   * n of row (b, t) is (b*T + t)*ld_out + n for both sites (the offset of the element in out_f32 / out_preln). */
  float drop_pre_p, drop_post_p;
  uint32_t drop_pre_site, drop_post_site, drop_seed;
  int precision;            /* TTSB_PREC_* */
  int impl;                 /* TTSB_IMPL_* */
  /* residual given as a bf16 hi/lo pair instead of fp32 (residual == NULL): value = hi + lo, row stride ld_res.  In
   * bf16x3 inference the activation pair IS the residual stream (16 mantissa bits), so the LayerNorm GEMMs neither write
   * nor re-read an fp32 copy of every activation (LayerNorm epilogue only). */
  const void* residual_hi;
  const void* residual_lo;
} ttsb_gemm_args;

int ttsb_linear_fwd(const ttsb_gemm_args* args, void* stream);

/* Stand-alone LayerNorm (+ row mask) over rows of fp32 x (B,T,ld)[:, :, :d]  (model/layers.py:27,96,207: epsilon 1e-6).
 * Used when a row is wider than one 256-column accumulator tile (model dimension 384): the GEMM then writes the
 * pre-norm value and this kernel produces the fp32 + bf16 hi/lo activation triple. */
int ttsb_layernorm_fwd(const float* x, const float* gamma, const float* beta, int B, int T, int d, int ld, float eps,
                       const int32_t* row_len, float* out_f32, void* out_hi, void* out_lo, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused variable-length attention  (model/layers.py:138-147 split/merge heads, :176-195 scaled dot product)
 *   self-attention (kv_hi == NULL): q,k,v are columns q_col0 + h*dh / k_col0 + h*dh / v_col0 + h*dh of ONE buffer
 *     (B,T,ld_qk), the QKV GEMM output; Tk = T.
 *   cross-attention (kv_hi != NULL; model/layers.py:315-327 CrossAttentionResnorm): q from (B,T,ld_qk) at q_col0,
 *     k and v from a second buffer (B,Tk,ld_kv) at k_col0 / v_col0 (the K|V GEMM of the encoder output).
 *   out: bf16 hi (and lo when out_lo != NULL) (B,T,ld_out), head h at columns h*dh.
 *   Masking follows the reference's additive -1e9 masks: keys t >= kv_len[b] (padding mask, transformer_utils.py:24-32)
 *   and, with causal = 1, keys t > query index (look-ahead mask, transformer_utils.py:35-37; the Aligner passes
 *   max(padding, look-ahead), models.py:136-138).
 *   full_queries = 0: query rows >= kv_len[b] are written as zeros (ForwardTransformer blocks multiply them by the
 *   mask right after, layers.py:228-230); 1: every query row is computed from the unmasked keys as the reference does
 *   (Aligner decoder blocks never re-mask their rows).
 *   precision TTSB_PREC_FP16: the buffers hold IEEE fp16 (written by ttsb_linear_fwd with out_fp16 = 1), one
 *   tensor-core pass.  Head dims 64, 128 (all precisions), 192, 256 (single-pass precisions).
 * ------------------------------------------------------------------------------------------------------- */
typedef struct ttsb_mha_args {
  int B, T, H, dh;
  const void* qk_hi;
  const void* qk_lo;
  int ld_qk, q_col0, k_col0, v_col0;
  const int32_t* kv_len; /* [B] */
  void* out_hi;
  void* out_lo;
  int ld_out;
  /* optional: materialised softmax weights, reference-exact fp32 (logits + mask * -1e9, softmax).
   * weights_all = 0: ONE batch row, (H,T,Tk) (the ForwardTransformer's callers read item 0 only);
   * weights_all = 1: every row, (B,H,T,Tk) (the Aligner's cross-attention is a model output, models.py:150-153) */
  float* weights_out;
  int weights_batch_index;
  int precision;
  int impl;
  /* ---- ABI 2 ---- */
  const void* kv_hi;     /* NULL: self-attention */
  const void* kv_lo;
  int ld_kv, Tk;
  int causal;
  int full_queries;
  int weights_all;
} ttsb_mha_args;

int ttsb_mha_fwd(const ttsb_mha_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Training-step GEMMs (single-pass bf16, fp32 accumulate) -- gradients of the layers above
 *
 * ttsb_bgemm: per-(batch row b, head h) products  out_z[m][n] = alpha * sum_k A_z[m][k] * B_z[n][k]  where both operands
 *   are activations: S = Q K^T, O = P V, dP = dO V^T, dQ = dS K, dK = dS^T Q, dV = P^T dO (model/layers.py:179-193 and
 *   its gradient).  Each operand is a bf16 tensor described as (dim0 contiguous, dim1 rows, dim2 batches) with element
 *   strides.  K-major operand (x_mn_major = 0): dim0 is the contraction axis, dim1 the M (or N) axis; MN-major operand
 *   (x_mn_major = 1): dim0 is the M (or N) axis, dim1 the contraction axis -- so a transposed operand (P^T, dS^T, dO^T,
 *   V^T, K^T) is the SAME tensor read MN-major and no transposed copies exist.  The tile origin of problem z = (b,h) is
 *   (c0 + h*h_col, c1 + h*h_row, z_batch ? z : b).
 * ttsb_wgrad: weight gradients  dW[seg*Cin + c][n] += sum_{b,t} X_seg[b][t + shift_seg][c] * G[b][t][n]  for Dense
 *   (1 segment), concat-Dense (2 sources) and Conv1D (k segments with the tap shifts); X and G are the row-major bf16
 *   activations / output gradients (B, T, ld) read MN-major; dW is fp32 in the Keras (K, N) layout and is ACCUMULATED
 *   into.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct ttsb_bgemm_args {
  int B, H, M, N, K;
  const void* a;
  long long a_dim0, a_dim1, a_dim2, a_stride1, a_stride2;
  int a_h_col, a_h_row, a_z_batch, a_mn_major;
  const void* b;
  long long b_dim0, b_dim1, b_dim2, b_stride1, b_stride2;
  int b_h_col, b_h_row, b_z_batch, b_mn_major;
  float alpha;
  float* out_f32;            /* either or both */
  void* out_bf16;
  int ld_out;                /* row stride (elements), multiple of 16 */
  long long out_batch_stride;/* elements between consecutive z (or b when out_by_b) */
  int out_h_col;             /* column offset per head */
  int out_by_b;              /* 1: output batch index is b (heads side by side in the columns) */
  int out_cols;              /* writable columns per row of one problem (multiple of 16); columns >= N are written 0 */
  const int32_t* row_len;    /* optional [B]: rows m >= row_len[b] are written as zeros */
  const int32_t* col_len;    /* optional [B]: columns n >= col_len[b] are written as zeros */
  /* ---- ABI 2: fused softmax backward.  With sm_P != NULL the product is dP = dO V^T of an attention backward and the
   * epilogue writes dS = sm_scale * P_pre * (dropout(dP) - D) (bf16, out_bf16) instead of dP, with the masking rules and
   * dropout hash of ttsb_softmax_bwd: sm_P = P_pre bf16 in the OUTPUT layout (requires out_by_b = 0, out_h_col = 0,
   * out_batch_stride = M * ld_out), sm_D fp32 [B*H*M] = rowsum(P_drop * dP) = dO . O per (row, head)
   * (ttsb_rowdot_heads), sm_len = key lengths [B], sm_flags as ttsb_softmax_bwd. */
  const void* sm_P;
  const float* sm_D;
  float sm_scale, sm_drop_p;
  uint32_t sm_seed, sm_site;
  int sm_flags;
  const int32_t* sm_len;
  const void* sm_Pdrop;      /* optional: the saved post-dropout probabilities (same layout); the dropout decision is then
                              * read back from it (kept <=> P_drop != 0 where P_pre != 0) instead of re-hashed */
} ttsb_bgemm_args;

int ttsb_bgemm(const ttsb_bgemm_args* args, void* stream);

typedef struct ttsb_wgrad_args {
  int B, T, Cin, N;
  int num_segments;          /* 1..4 */
  int seg_src[4];            /* which x source */
  int seg_shift[4];          /* time shift of the source rows (conv taps); rows outside [0,T) read as zero */
  const void* x[2];          /* bf16 (B, T, ldx[i]); the first Cin columns are used */
  int ldx[2];
  const void* g;             /* bf16 (B, T, ldg); the first N columns are used */
  int ldg;
  float* dw;                 /* fp32 (num_segments*Cin, N), accumulated */
} ttsb_wgrad_args;

int ttsb_wgrad(const ttsb_wgrad_args* args, void* stream);

/* out[(b*H + h)*T + t] = sum_c x[b,t,h*dh+c] * y[b,t,h*dh+c]  (bf16 (B,T,ld) inputs, fp32 out): the row statistic
 * D = dO . O of the attention backward (equals rowsum(P_drop * dP), so dP never has to be materialised). */
int ttsb_rowdot_heads(const void* x_bf16, const void* y_bf16, int B, int T, int H, int dh, int ld, float* out, void* stream);

/* Row softmax of materialised, pre-scaled scores S fp32 (B*H, T, ld) with key masking (model/layers.py:186-192) and
 * attention dropout: P_pre = softmax, P_drop = dropout(P_pre) (pass the same pointer twice when drop_p == 0).  Dropout
 * element index of key k in row t of problem z = b*H + h: (z*T + t)*ld + k (ttsb_softmax_bwd regenerates the same mask). */
/* flags: bit 0 = look-ahead mask (keys > query index masked, transformer_utils.py:35-37); bit 1 = every query row is live
 * (Aligner blocks); without it query rows >= kv_len[b] are written as zeros (they are masked downstream). */
int ttsb_softmax_fwd(const float* S, int B, int H, int T, int Tk, int ld, const int32_t* kv_len, float drop_p,
                     uint32_t seed, uint32_t site, int flags, void* P_pre, void* P_drop, void* stream);
/* The two calls above (logits GEMM + ttsb_softmax_fwd) fused for self-attention with flags == 0: P_pre = softmax(scale *
 * Q K^T) over keys < kv_len[b], P_drop = dropout(P_pre), both bf16 (B*H, T, ld_p); the logits stay in tensor memory.
 * qkv is a bf16 (B, T, ld) activation tensor holding head h of Q at columns q_col0 + h*dh and of K at k_col0 + h*dh.
 * Needs dh in {64, 128, 192} and fewer than 2^33 probabilities (ttsb_attn_probs_supported; otherwise use the two calls
 * above); pass P_drop == P_pre when drop_p == 0.
 * Same dropout element index as ttsb_softmax_fwd: (z*T + t)*ld_p + key. */
int ttsb_attn_probs_supported(int dh, int ld_p);
int ttsb_attn_probs_fwd(const void* qkv, int ld, int q_col0, int k_col0, int B, int H, int T, int dh, const int32_t* kv_len,
                        float scale, float drop_p, uint32_t seed, uint32_t site, void* P_pre, void* P_drop, int ld_p,
                        void* stream);
/* Backward counterpart (the same kernel, one pass): dS = scale * P_pre * (dropout(dO V^T) - D) bf16 (B*H, T, ld_p), the
 * softmax gradient of model/layers.py:186-192 fused into the dP product -- what ttsb_bgemm does with sm_P set, with sixteen
 * epilogue warps and no fp32 dP in HBM.  dO bf16 (B, T, ld_do) holds head h at columns do_col0 + h*dh, v bf16 (B, T, ld_v)
 * at v_col0 + h*dh; D fp32 (B*H*T) from ttsb_rowdot_heads; keys >= kv_len[b] and query rows >= kv_len[b] give zeros. */
int ttsb_attn_ds_bwd(const void* dO, int ld_do, int do_col0, const void* v, int ld_v, int v_col0, int B, int H, int T, int dh,
                     const int32_t* kv_len, const void* P_pre, const float* D, float scale, float drop_p, uint32_t seed,
                     uint32_t site, void* dS, int ld_p, void* stream);
int ttsb_softmax_bwd(const void* P_pre, const float* dP, int B, int H, int T, int Tk, int ld, const int32_t* kv_len,
                     float scale, float drop_p, uint32_t seed, uint32_t site, int flags, void* dS, void* stream);
/* LayerNorm backward from the saved pre-norm values u (keras LayerNormalization, model/layers.py:27,96,207,295,508).
 * post_drop regenerates the mask of a dropout on the LayerNorm output (applied to dz), pre_drop that of ttsb_linear_fwd's
 * drop_pre (applied to g_bf16, the gradient of the GEMM output); both use element index (b*T + t)*ld + c, the index
 * ttsb_linear_fwd uses with ld_out = ld. */
int ttsb_layernorm_bwd(const float* dz, const float* u, const float* gamma, int B, int T, int C, int ld, float eps,
                       const int32_t* row_len, int relu_mask, float pre_drop_p, uint32_t pre_site, float post_drop_p,
                       uint32_t post_site, uint32_t seed, float* du, void* g_bf16, float* dgamma, float* dbeta, float* dbias,
                       void* stream);
/* column sums of bf16 (rows, ld)[:, :C] accumulated into fp32 out[C] (bias gradients) */
int ttsb_colsum_bf16(const void* x, int64_t rows, int C, int ld, float* out, void* stream);
/* three adjacent column segments of width seg -> three outputs (the q / k / v bias gradients from the (rows, 3d) buffer) */
int ttsb_colsum_bf16_x3(const void* x, int64_t rows, int seg, int ld, float* out0, float* out1, float* out2, void* stream);
int ttsb_relu_bwd(void* dy_bf16, const void* h_bf16, int64_t n, void* stream);
/* ttsb_relu_bwd plus the bias gradient of the layer that produced h, in the same pass: colsum[c] += sum_rows (masked dy)
 * (dy, h bf16 (rows, C) contiguous). */
int ttsb_relu_bwd_colsum(void* dy, const void* h, int64_t rows, int C, float* colsum, void* stream);
/* fp32 (rows, C) -> bf16 (rows, ld_out >= C) with zero padding columns */
int ttsb_cast_bf16_pad(const float* x, int64_t rows, int C, void* out_bf16, int ld_out, void* stream);
/* mean |pred - target| over ALL elements of pred[:, :Tt] (utils/losses.py:41-49 as called with mask=None), added to
 * *loss_out; grad = weight * sign(pred - target) / numel (zero for rows >= Tt). */
int ttsb_mae_loss(const float* pred, int B, int Tp, int Tt, int C, const float* target_f32, const int32_t* target_i32,
                  float weight, float* loss_out, float* grad, void* stream);
/* Duration extraction from the Aligner's attention maps (utils/alignments.py:103-143; the producer of the durations the
 * ForwardTransformer trains on).  Lengths are the reference's "mel_lengths(mels) - 1" / "phoneme_lengths(phonemes) - 1".
 * ttsb_attention_scores: utils/metrics.py:5-44 -> scores (B,H,3) = jumpiness, peakiness, 3 / diagonality.
 * ttsb_durations_from_attention: reference matrix = att[b, best head, 1:mel_len, 1:phon_len] (or the score-weighted sum of
 *   the heads), shortest monotonic path through (max - attention) (utils/alignments.py:58-91: scipy Dijkstra; here the
 *   equivalent anti-diagonal dynamic programme in float64), durations int32 (B,Tk) (zero beyond phon_len - 1).
 *   scratch: B*Tq*Tk bytes. */
int ttsb_attention_scores(const float* att, int B, int H, int Tq, int Tk, const int32_t* mel_len, const int32_t* phon_len, int r,
                          float* scores, void* stream);
int ttsb_durations_from_attention(const float* att, int B, int H, int Tq, int Tk, const int32_t* mel_len, const int32_t* phon_len,
                                  const float* scores, int weighted, uint8_t* scratch, int32_t* durations, void* stream);

/* Aligner losses (SURVEY 8(f) row 1).
 * ttsb_scaled_ce_loss: utils/losses.py:4-21 new_scaled_crossentropy -- sparse softmax CE of logits (B,Tp,ld)[:, :Tt, :C] against
 *   int targets (B,Tt); sample weight (target != 0) + (target == index) * (scaling - 1); Keras SUM_OVER_BATCH_SIZE
 *   (sum / (B*Tt)); added to *loss_out.
 * ttsb_diag_loss: utils/metrics.py:47-70 batch_diagonal_mask + models.py:189-205 -- mean over (b,h) of
 *   sum_{q<q_len, k<k_len} att[b,h,q,k] * |k/k_len - q/q_len|, divided by 10; added to *loss_out. */
int ttsb_scaled_ce_loss(const float* logits, int B, int Tp, int Tt, int C, int ld, const int32_t* targets, int index,
                        float scaling, float* loss_out, float grad_weight, float* grad /* optional (B,Tp,ld_grad) */, int ld_grad,
                        void* stream);
/* training form of ttsb_diag_loss on the post-dropout probabilities P (bf16, (B*H,Tq,ld)): *loss_out += loss_scale * loss,
 * dP (fp32, same layout, optional) += grad_scale * d loss / d P */
int ttsb_diag_loss_train(const void* P_bf16, int B, int H, int Tq, int Tk, int ld, const int32_t* q_len, const int32_t* k_len,
                         float loss_scale, float* loss_out, float grad_scale, float* dP, void* stream);
int ttsb_diag_loss(const float* att, int B, int H, int Tq, int Tk, const int32_t* q_len, const int32_t* k_len,
                   float* loss_out, void* stream);
/* Expand (length regulator) backward: dx[b,i,:] = sum of dm[b,t,:] over the frames t in [start_i, start_i + dur[b,i]) with
 * start_i = sum_{j<i} max(dur[b,j], 0); negative durations count as 0 and frames >= Tm are dropped.  dm fp32 (B,Tm,d), dx fp32
 * (B,Tp,d) (every element written); d must be a multiple of 4 and dm, dx 16-byte aligned (float4 rows). */
int ttsb_expand_bwd(const float* dm, const int32_t* dur_int, int B, int Tp, int Tm, int d, float* dx, void* stream);
int ttsb_embedding_bwd(const float* dx, const int32_t* tokens, int B, int T, int d, int vocab, float* demb, void* stream);
/* d(pos_encoding_scalar) = sum dropout(g) * PE[t]; (drop_p, seed, site) regenerate the prologue dropout mask (element index
 * (b*T + t)*d + c, the flat index of the prologue output) */
int ttsb_pe_scalar_bwd(const float* g, const float* pe, int B, int T, int d, float drop_p, uint32_t seed, uint32_t site,
                       float* dscalar, void* stream);
/* training variants of the two stack prologues: keras Dropout after LayerNorm + PE (model/layers.py:301); dropout element
 * index = flat output index (b*T + t)*d + c (T = Tm for the expand form) */
int ttsb_embed_ln_pe_train_fwd(const int32_t* tokens, const float* emb, const float* gamma, const float* beta,
                               const float* pe, const float* pos_scalar, int B, int T, int d, int vocab, float eps,
                               float drop_p, uint32_t seed, uint32_t site, float* out_f32, void* out_hi, void* out_lo,
                               void* stream);
int ttsb_expand_ln_pe_train_fwd(const float* x, const int32_t* idx, const float* gamma, const float* beta, const float* pe,
                                const float* pos_scalar, int B, int Tp, int Tm, int d, float eps, float drop_p, uint32_t seed,
                                uint32_t site, float* out_f32, void* out_hi, void* out_lo, void* stream);
int ttsb_pitch_embed_bwd(const float* g, const float* pitch, const float* w, const float* bias, int B, int T, int d,
                         float* dw, float* db, void* stream);
int ttsb_statpred_head_bwd(const float* gout, const float* out, const float* h, int ldh, int C, const float* w, int relu,
                           const int32_t* row_len, int B, int T, float* dh, float* dw, float* db, void* stream);
/* Keras/TF-2.2 Adam (utils/training_config_manager.py:102-106): theta -= lr_t * m / (sqrt(v) + eps) with
 * lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t) computed by the caller; grad is multiplied by grad_scale first. */
int ttsb_adam_tf_step(float* param, const float* grad, float* m, float* v, int64_t n, float lr_t, float beta1, float beta2,
                      float eps, float grad_scale, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * StatPredictor head  Dense(C->1, relu|linear) * mask   (model/layers.py:479-485)
 *   h fp32 (B,T,ldh) -> out fp32 (B,T)
 * ------------------------------------------------------------------------------------------------------- */
int ttsb_statpred_head_fwd(const float* h, int ldh, int C, const float* w, const float* bias, int relu,
                           const int32_t* row_len, int B, int T, float* out, void* stream);

/* x + relu(pitch*w + b)  (model/models.py:527-531; Dense(1->d, relu)) -> fp32 (B,T,d) */
int ttsb_pitch_embed_add_fwd(const float* x, const float* pitch, const float* w, const float* bias, int B, int T,
                             int d, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Length regulator  (model/models.py:532-540, model/layers.py:549-565)
 * ------------------------------------------------------------------------------------------------------- */
/* durations (B,Tp) fp32 * scalar -> min(max_mask) -> max(min_mask) -> round-half-even -> int32.
 * max_mask / min_mask may be NULL.  Also writes per-row totals to out_len[B]; a row that holds a negative duration gets
 * out_len = -1 (the reference's ragged-tensor construction raises on it; the host checks this one array). */
int ttsb_durations_to_int(const float* dur, float scalar, const float* max_mask, const float* min_mask, int B, int Tp,
                          int32_t* out_int, int32_t* out_len, void* stream);
/* int durations (B,Tp) -> frame->phoneme index map (B,Tm) (-1 at padded frames); row totals must be <= Tm */
int ttsb_expand_indices(const int32_t* dur_int, int B, int Tp, int Tm, int32_t* out_idx, void* stream);
/* out[b,t,:] = idx[b,t] >= 0 ? x[b, idx[b,t], :] : 0     (Expand; fp32, d multiple of 4) */
int ttsb_length_regulate_fwd(const float* x, const int32_t* idx, int B, int Tp, int Tm, int d, float* out, void* stream);
/* fused Expand + decoder prologue LN + scalar*PE (model/layers.py:299-300): writes fp32 + bf16 hi/lo */
int ttsb_expand_ln_pe_fwd(const float* x, const int32_t* idx, const float* gamma, const float* beta, const float* pe,
                          const float* pos_scalar, int B, int Tp, int Tm, int d, float eps, float* out_f32, void* out_hi,
                          void* out_lo, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * utils/spectrogram_ops.py:8-17
 * ------------------------------------------------------------------------------------------------------- */
int ttsb_mel_lengths(const float* mel, int B, int T, int C, float padding_value, int32_t* out, void* stream);
int ttsb_phoneme_lengths(const int32_t* phonemes, int B, int T, int32_t padding, int32_t* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * STFT -> mel filterbank -> log   (data/audio.py:72-92, 209-231)
 *   wav fp32 (n_clips, n_samples); out fp32 (n_clips, n_frames, n_mels), n_frames = 1 + n_samples/hop.
 *   n_fft must be 1024 (the reference's config), hop 256, window = periodic Hann(1024), reflect padding.
 *   mel_basis fp32 (n_mels, 513) dense (the kernel uses its band structure); normalizer 0 = MelGAN log(clip 1e-5),
 *   1 = WaveRNN.
 * ------------------------------------------------------------------------------------------------------- */
int ttsb_stft_mel_log(const float* wav, int n_clips, int n_samples, const float* mel_basis, int n_mels,
                      int normalizer, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * mel -> waveform  (Audio.reconstruct_waveform, data/audio.py:94-110: librosa mel_to_stft(power=1) + griffinlim(32, momentum .99))
 *   n_fft 1024, hop 256, periodic Hann, centred frames with reflect padding (the reference configuration).
 * ------------------------------------------------------------------------------------------------------- */
/* mel amplitudes (n_frames, n_mels) -> non-negative linear magnitudes (n_frames, 513): per frame min_{x>=0} |A x - m|^2 for the
 * mel basis A (n_mels, 513), from the start max(pinv(A) m, 0) that librosa's nnls uses, with n_iter FISTA steps of size `step`
 * (1 / |A|_2^2).  band[2*j], band[2*j+1] = first / past-last non-zero bin of basis row j; bin_mels[2*k], [2*k+1] = first /
 * past-last mel row that is non-zero at bin k.  basis_pinv is (513, n_mels). */
int ttsb_mel_to_linear(const float* mel_amp, int n_frames, int n_mels, const float* mel_basis, const float* basis_pinv,
                       const int32_t* band, const int32_t* bin_mels, float step, int n_iter, float* out, void* stream);
/* librosa.stft: wav (n_samples) -> complex64 (1 + n_samples/256, 513) as interleaved (re, im) floats */
int ttsb_stft_complex(const float* wav, int n_samples, float* spec_out, void* stream);
/* librosa.istft: complex64 (n_frames, 513) -> wav (256 * (n_frames - 1)).  workspace: ttsb_istft_workspace_bytes(n_frames) bytes
 * of device memory (the windowed time frames before the overlap-add). */
int64_t ttsb_istft_workspace_bytes(int n_frames);
int ttsb_istft(const float* spec, int n_frames, void* workspace, int64_t workspace_bytes, float* wav_out, void* stream);
/* one phase update of fast Griffin-Lim over n complex bins: a = rebuilt - momentum/(1+momentum) * previous (previous may be
 * NULL: first iteration); a /= |a| + 1e-16; projected_out = magnitude * a.  rebuilt / previous / projected_out are complex64. */
int ttsb_griffinlim_update(const float* rebuilt, const float* previous, const float* magnitude, float momentum, int64_t n,
                           float* projected_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange (BASELINE.json: "NCCL allreduce over NVLink on gradient buckets only"; the reference has
 * no distributed code).  One communicator per process / GPU.  NCCL is loaded at run time (libnccl.so.2 of the host
 * process, or $TTSB_NCCL_LIB); without it these return TTSB_ERR_UNSUPPORTED.
 *   ttsb_dp_unique_id       : rank 0 fills a 128-byte id that the host distributes to all ranks (any side channel)
 *   ttsb_dp_init            : collective; binds to the calling thread's current CUDA device
 *   ttsb_dp_allreduce_bucket: in-place SUM of buf[0:count] (fp32, device) across ranks, enqueued on `stream`; the 1/N
 *                             factor is applied by ttsb_adam_tf_step(grad_scale).  Call it as soon as a contiguous slice of
 *                             the flat gradient buffer is final, on a second stream, to overlap it with the remaining
 *                             backward kernels.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct ttsb_dp_comm ttsb_dp_comm;
int ttsb_dp_unique_id(void* id_out_128_bytes);
int ttsb_dp_init(const void* unique_id_128_bytes, int rank, int world, ttsb_dp_comm** out);
int ttsb_dp_allreduce_bucket(ttsb_dp_comm* comm, float* buf, int64_t count, void* stream);
int ttsb_dp_destroy(ttsb_dp_comm* comm);

#ifdef __cplusplus
}
#endif
#endif /* TTSB_H_ */
