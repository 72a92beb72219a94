/* apla_b200 -- C ABI of the B200-native APLA fine-tune step.
 *
 * The reference (MoeinSorkhei/APLA) is 100 % Python/PyTorch and has no FFI; every entry point below replaces a
 * span of ATen/cuBLAS calls issued by the reference file:line cited next to it (paths relative to the reference
 * root).  All functions:
 *   - take raw DEVICE pointers + sizes + a cudaStream_t (passed as void*), never torch types;
 *   - return 0 on success, non-zero on error (message via apla_last_error(), thread-local);
 *   - never allocate, never synchronise, never take ownership;
 *   - require an sm_100 device (apla_device_check()).
 * Dtypes: "bf16" = __nv_bfloat16, "f32" = float.  Matrices are row-major with an explicit leading dimension
 * (elements).  T = tokens, D = embedding dim, H = heads (head dim is 64 everywhere).
 */
#ifndef APLA_B200_H_
#define APLA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* apla_stream_t; /* cudaStream_t */

/* --- library ------------------------------------------------------------------------------------------- */
const char* apla_last_error(void);
int apla_version(void);
/* kernels launched by this library since it was loaded (every launcher counts its own launches) */
int64_t apla_launch_count(void);
/* 0 iff the current device is compute capability 10.x (B200); the product path has no other backend. */
int apla_device_check(void);

/* --- GEMMs (tcgen05 + TMA), y = x W^T with W = [out, in] like nn.Linear ----------------------------------- */
/* out_bf16[M,N] = A_bf16[M,K] . W_bf16[N,K]^T + bias_f32[N] (bias may be NULL).
 * Replaces nn.Linear forward of frozen layers: self.qkv(x) src/apla/appla_attn.py:53; also used for every
 * input-gradient GEMM dX = dY . W by passing the pre-transposed weight (apla_gemm_dgrad). */
int apla_gemm_bias_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* out, int ldo, int M,
                       int N, int K, apla_stream_t stream);
/* h_bf16 = A . W^T + bias ; g_bf16 = gelu_erf(h).  Mlp.fc1 + nn.GELU, src/utils/transformers/vit.py:163-164. */
int apla_gemm_bias_gelu_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* h, void* g,
                            int ldo, int M, int N, int K, apla_stream_t stream);
/* out_f32[M,N] = resid_f32[M,N] + gamma_f32[N] * (A . W^T + bias)   (gamma NULL = 1; out may alias resid).
 * The two F.linear + two scatter_ of src/apla/appla_attn.py:64-79 (W is the full-layout projection), or Mlp.fc2
 * vit.py:166, followed by LayerScale vit.py:243-244 and the residual add vit.py:284-285. */
int apla_gemm_bias_ls_residual_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                   const float* gamma, const float* resid, float* out, int ldo, int M, int N, int K,
                                   apla_stream_t stream);
/* The residual update above with one scale per group of rows_per_scale rows (stochastic depth, vit.py drop_path):
 * out_f32[m,n] = resid_f32[m,n] + row_scale_f32[m / rows_per_scale] * gamma_f32[n] * (A . W^T + bias)   (gamma NULL = 1).
 * rows_per_scale = N scales the token rows of an image, 1 scales one row per image (the CLS rows, row stride ldo).
 * A scale of 1 gives apla_gemm_bias_ls_residual_fwd's bits.  The default (2-CTA) GEMM only: refused under
 * APLA_GEMM_IMPL=1.  NULL A, W, resid, row_scale or out, an empty shape or rows_per_scale < 1 are refused. */
int apla_gemm_bias_ls_residual_scaled_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                          const float* gamma, const float* resid, const float* row_scale,
                                          int rows_per_scale, float* out, int ldo, int M, int N, int K,
                                          apla_stream_t stream);
/* The residual update above FOLLOWED BY the LayerNorm that reads it, in one launch:
 *   out_f32 = resid_f32 + gamma * (A . W^T + bias);  ln_out_bf16[M,N] = (out - mean) * rstd * ln_w + ln_b
 * i.e. vit.py:284 + the norm2 of vit.py:285 (projection), or vit.py:285 + the norm1 of the next block's vit.py:280 (fc2).
 * one_launch = 0: the two kernels back to back.  one_launch = 1 and N = 384 / 768 / 1024: ONE launch -- the CTA that
 * completes the last column tile of a 128-row slab normalises the slab while it is still in L2 (bit-identical results;
 * measured slower on the C2 step, DESIGN.md section 4).  one_launch < 0: the default = two kernels unless
 * APLA_GEMM_LN_FUSE=1.  One-launch calls on one device must be stream-ordered (shared arrival counters). */
int apla_gemm_bias_ls_residual_ln_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                      const float* gamma, const float* resid, float* out, int ldo, const float* ln_w,
                                      const float* ln_b, void* ln_out, int ld_ln, float eps, int M, int N, int K,
                                      int one_launch, apla_stream_t stream);
/* out_f32[M,N] += gamma_f32[N] * (A . W^T + bias): the same residual update performed IN PLACE -- the epilogue hands
 * the scaled tile to the L2 as a TMA reduce-add, so the fp32 residual never passes through shared memory. */
int apla_gemm_bias_ls_accumulate(const void* A, int lda, const void* W, int ldw, const float* bias, const float* gamma,
                                 float* out, int ldo, int M, int N, int K, apla_stream_t stream);
/* dX_bf16[M,K_in] = dY_bf16[M,N_out] . Wt_bf16[K_in,N_out]^T : input gradient of a frozen Linear; Wt is the
 * transposed weight ([in, out], prepared once because the weight is frozen).  No weight gradient is computed or
 * allocated (autograd prunes it the same way for requires_grad=False, SURVEY.md 2.3 K24). */
int apla_gemm_dgrad(const void* dY, int ldy, const void* Wt, int ldwt, void* dX, int ldx, int M, int K_in, int N_out,
                    apla_stream_t stream);
/* dH_bf16 = (dY . Wt^T) * gelu_erf'(h_bf16): fc2 input gradient fused with GELU backward (vit.py:164-166). */
int apla_gemm_dgrad_gelu_bwd(const void* dY, int ldy, const void* Wt, int ldwt, const void* h, void* dH, int ldh,
                             int M, int K_in, int N_out, apla_stream_t stream);
/* Training variant of the pair above (what the step engine runs): the forward saves the GELU derivative instead of
 * the pre-activation -- dgelu_f16 = gelu_erf'(A . W^T + bias), g_bf16 = gelu_erf(A . W^T + bias), both from the fp32
 * accumulator -- and the fc2 input gradient becomes dH_bf16 = (dY . Wt^T) * mul_f16.  Same autograd result as
 * nn.GELU backward (vit.py:164), one multiply in the epilogue instead of an erf evaluation. */
int apla_gemm_bias_gelu_dgelu_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* dgelu,
                                  void* g, int ldo, int M, int N, int K, apla_stream_t stream);
int apla_gemm_dgrad_mul(const void* dY, int ldy, const void* Wt, int ldwt, const void* mul, void* dH, int ldh, int M,
                        int K_in, int N_out, apla_stream_t stream);
/* Forward-only fc1 (evaluation, or any forward that autograd will not differentiate): g_bf16 = gelu_erf(A . W^T + bias),
 * bit-identical to the g output of apla_gemm_bias_gelu_dgelu_fwd; no derivative is written. */
int apla_gemm_bias_gelu_only_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* g, int ldo,
                                 int M, int N, int K, apla_stream_t stream);
/* dO_bf16[M,D] = dY_bf16[M,D_out] . Wt^T  and  delta_f32[M, D/64] = rowsum over each 64-wide head of dO * O_bf16:
 * the input gradient of the attention projection (backward of appla_attn.py:64-79) fused with the softmax-backward
 * row term of the attention that produced O (appla_attn.py:58-62); pass the result to apla_attn_bwd with out = NULL. */
int apla_gemm_dgrad_delta(const void* dY, int ldy, const void* Wt, int ldwt, const void* O, void* dO, int ldo,
                          float* delta, int M, int D, int N_out, apla_stream_t stream);
/* APLA weight gradient.  dW1_f32[r, D_in] += dYsub^T . X  where dYsub_bf16[T, n_pad] holds the r gathered
 * output-gradient columns (n_pad = r rounded up to 64, zero padded) and X_bf16[T, D_in] is the projection input.
 * With rowmap != NULL, dYsub is the full [T, D_out] gradient and rowmap[n] (int32, -1 = frozen) is the
 * trainable slot of output feature n (the partial_size == dim case).  Split-K fp32 atomics: dW1 must be zeroed
 * by the caller.  This is autograd's backward of F.linear(x, proj_weight1) + scatter_ (appla_attn.py:64,70-74). */
int apla_proj_wgrad_gather(const void* dYsub, int ldy, const void* X, int ldx, const int32_t* rowmap, float* dW1,
                           int ldw, int T, int D_in, int n_pad, int r, apla_stream_t stream);
/* db_f32[map(j)] += sum_t dY_bf16[t, j]  (bias gradient of the trainable rows). */
int apla_colsum(const void* dY, int64_t ld, int T, int n, const int32_t* rowmap, float* db, apla_stream_t stream);

/* --- LayerNorm ----------------------------------------------------------------------------------------- */
/* y_bf16 = LayerNorm(x_f32; w, b, eps).  nn.LayerNorm(eps=1e-6) vit.py:280,285,417 (factories :519-571). */
int apla_layernorm_fwd(const float* x, int64_t ldx, const float* w, const float* b, void* y, int64_t ldy, int rows,
                       int D, float eps, apla_stream_t stream);
/* dx_f32 = dres_f32 + LayerNorm'(dy_bf16) (dres NULL = 0; dx may alias dres);
 * dxb_bf16 = gamma * dx (optional); sub_bf16[t, j<r] = gamma[idx[j]] * dx[t, idx[j]], zero for r <= j < r_pad
 * (optional): residual-gradient add + LayerScale backward + APLA column gather in one pass. */
int apla_layernorm_bwd(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w, const float* dres,
                       int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb, const float* gamma,
                       void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad, int rows, int D, float eps,
                       apla_stream_t stream);
/* sub_bf16[t, j] = dy_bf16[t, idx[j]] (j < r), 0 (r <= j < r_pad). */
/* apla_layernorm_bwd with dxb and sub of row t also multiplied by row_scale_f32[t / rows_per_scale] -- the
 * stochastic-depth scale of the branch that reads them; dx_f32 (the residual-stream gradient) is not scaled.  A scale
 * of 1 gives apla_layernorm_bwd's bits.  D a multiple of 128 only.  NULL dy, x, w, dx, dxb or row_scale, an empty shape
 * or rows_per_scale < 1 are refused. */
int apla_layernorm_bwd_scaled(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w,
                              const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb,
                              const float* gamma, void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad,
                              const float* row_scale, int rows_per_scale, int rows, int D, float eps,
                              apla_stream_t stream);
int apla_gather_cols(const void* dy, int64_t ld, void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad,
                     int rows, apla_stream_t stream);

/* out_bf16 = gamma * x_f32 (gamma NULL = 1): LayerScale backward (vit.py:243-244) + down-cast of a residual-stream
 * gradient entering the fused block from autograd (Block.forward vit.py:279-288 seen from its output). */
int apla_ls_cast(const float* x, int64_t ldx, const float* gamma, void* out, int64_t ldo, int rows, int D,
                 apla_stream_t stream);

/* --- attention ------------------------------------------------------------------------------------------ */
/* out_bf16[T, H*64] = softmax(scale * q k^T) v per sequence and head; lse_f32[T, H] saved for backward.
 * qkv_bf16[T, 3*H*64] laid out (3, H, 64) along the last dim (appla_attn.py:53-54).  cu_seqlens = NULL: num_seqs
 * sequences of max_seqlen tokens (appla_attn.py:56-60); otherwise int32[num_seqs+1] packed offsets = the
 * BlockDiagonalMask of appla_attn_mem_eff.py:37-43 / dinov2/layers/block.py:191-217. */
int apla_attn_fwd(const void* qkv, void* out, float* lse, const int32_t* cu_seqlens, int num_seqs, int max_seqlen,
                  int total_tokens,
                  int H, float scale, apla_stream_t stream);
/* dqkv_bf16[T, 3*H*64] from dout_bf16[T, H*64]; delta_f32[T, H] is workspace, or -- with out == NULL -- the
 * precomputed rowsum(dout * out) per (token, head) from apla_gemm_dgrad_delta. */
int apla_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
                  const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
                  apla_stream_t stream);

/* Attention of the LAST block for the CLS query only (dense batch of B sequences of N tokens): only norm(x)[:, 0]
 * reaches the classifier (vit.py:417-419, models.py:87), so only row b*N of out / lse is produced, and backward takes
 * the gradient of that row alone: dqkv gets dK / dV of every key, dQ of the CLS rows and zeros for every other dQ row --
 * exactly what apla_attn_fwd / apla_attn_bwd return for those rows and for a dout that is zero elsewhere. */
int apla_attn_cls_fwd(const void* qkv, void* out, float* lse, int B, int N, int H, float scale, apla_stream_t stream);
int apla_attn_cls_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int B, int N,
                      int H, float scale, apla_stream_t stream);

/* Attention probabilities (the [B,H,N,N] `attn` of appla_attn.py:56-60,83, or its first q_rows query rows):
 * probs_f32[B, H, q_rows, N] = exp(scale * q k^T - lse) for B dense sequences of N tokens, from the qkv and the lse that
 * apla_attn_fwd wrote (or, for q_rows = 1, apla_attn_cls_fwd: only the lse of rows b*N is read).  One pass, no softmax
 * re-normalisation: each row sums to 1 up to rounding.  Refuses NULL pointers, B / N / H < 1 and q_rows outside [1, N]. */
int apla_attn_probs(const void* qkv, const float* lse, float* probs, int B, int N, int H, int q_rows, float scale,
                    apla_stream_t stream);

/* --- step ends ------------------------------------------------------------------------------------------ */
/* patches_bf16[B*P, kpad] from images_f32[B,3,S,S], k = (c, py, px): PatchEmbed conv as a GEMM, vit.py:302-306. */
int apla_patchify(const float* images, void* patches, int B, int S, int patch, int kpad, apla_stream_t stream);
/* x_f32[B, P+1, D] = cat(cls, patch_bf16) + pos_f32[P+1, D]   (vit.py:392-396; pos already interpolated). */
int apla_assemble_tokens(const void* patch, const float* cls, const float* pos, float* x, int B, int P, int D,
                         apla_stream_t stream);
/* logits_f32[B,C] = xn_bf16[B,D] . W_f32[C,D]^T + bias   (Classifier.fc, src/defaults/models.py:87). */
int apla_head_fwd(const void* xn, const float* W, const float* bias, float* logits, int B, int D, int C,
                  apla_stream_t stream);
/* *loss += loss_scale * sum_b CE_b ; dlogits = grad_scale * (softmax - onehot)   (wrappers.py:314). */
int apla_cross_entropy(const float* logits, const int64_t* labels, float* dlogits, float* loss, int B, int C,
                       float grad_scale, float loss_scale, apla_stream_t stream);
/* Probability targets (nn.CrossEntropyLoss with fp32 [B, C] targets, wrappers.py:314, as timm Mixup / CutMix with label
 * smoothing yields them, src/utils/_utils.py:424): with tsum_b = sum_c t[b,c] and tz_b = sum_c t[b,c] z[b,c],
 * *loss += loss_scale * sum_b (tsum_b lse_b - tz_b) ; dlogits = grad_scale * (tsum_b softmax - t).  Targets are neither
 * normalised nor validated (torch does neither).  For one-hot rows dlogits equals apla_cross_entropy's bit for bit.
 * Refuses NULL pointers and B or C < 1. */
int apla_cross_entropy_soft(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                            float grad_scale, float loss_scale, apla_stream_t stream);
/* Evaluation sums of one batch (Trainer.evaluate, trainer.py:162-245): acc_f32[0] += sum_b CE_b, acc_f32[1] += number of
 * rows whose argmax (first maximum) equals the label.  One launch, fixed summation order, no host synchronisation; a
 * label outside [0, C) makes acc[0] NaN. */
int apla_eval_accumulate(const float* logits, const int64_t* labels, int B, int C, float* acc, apla_stream_t stream);
/* Multi-label targets (nn.BCEWithLogitsLoss, wrappers.py:310-320, without weight or pos_weight): per element
 * l = max(z, 0) - z t + log1p(exp(-|z|)) in fp32, finite for every finite z;  *loss += loss_scale * sum_{b,c} l (one
 * atomicAdd per row) ; dlogits = grad_scale * (sigmoid(z) - t).  Targets f32[B, C] are neither clamped nor checked (torch
 * does neither).  BCEWithLogitsLoss's mean is loss_scale = grad_scale = 1 / (B C).  Refuses NULL pointers and B or C < 1. */
int apla_bce_with_logits(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                         float grad_scale, float loss_scale, apla_stream_t stream);
/* Multi-label evaluation sums of one batch: acc_f64[0] += sum_{b,c} l (as apla_bce_with_logits), acc_f64[1] += number of
 * elements with (z > 0) == (t >= 0.5).  double, because element counts of a validation set pass 2^24.  One launch, fixed
 * summation order, no host synchronisation.  Refuses NULL pointers and B or C < 1. */
int apla_eval_accumulate_bce(const float* logits, const float* targets, int B, int C, double* acc, apla_stream_t stream);
/* dW_f32[C,D], db_f32[C] (overwritten) and dxn_bf16[B,D]. */
int apla_head_bwd(const float* dlogits, const void* xn, const float* W, float* dW, float* db, void* dxn, int B, int D,
                  int C, apla_stream_t stream);

/* --- optimiser tail over one contiguous fp32 arena -------------------------------------------------------- */
/* out[0] = sum (scale*g)^2, bit-reproducible (fixed summation order: every data-parallel rank must derive the same clip
 * coefficient from the same all-reduced gradients).  `out` is a ZERO-INITIALISED buffer of APLA_SUMSQ_FLOATS floats owned by
 * the caller: out[0] is the result, the rest is scratch that every call leaves zeroed. */
#define APLA_SUMSQ_FLOATS 600
int apla_grad_sumsq(const float* g, int64_t n, float scale, float* out, apla_stream_t stream);
/* clip_grad_norm_(max_norm) (trainer.py:136) + torch.optim.AdamW step (wrappers.py:199-221): elements
 * [0,n_decay) are decayed.  gscale pre-multiplies the gradients (1/world for the DDP mean). */
int apla_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, int64_t n_decay, const float* sumsq,
                    float gscale, float max_norm, float lr, float wd, float beta1, float beta2, float eps, int step,
                    apla_stream_t stream);
/* Scatter trainable rows into the dense bf16 projection copies (appla_attn.py:70-79 done once per update). */
int apla_proj_refresh(const float* w1, const float* b1, const int32_t* idx, void* wfull, void* wfullT, float* bfull,
                      int L, int r, int D, int64_t w1_block_stride, int64_t b1_block_stride, apla_stream_t stream);

/* --- DINOv2 self-supervised objective: HBM-bound row kernels (SURVEY 8f row f2, BASELINE config C4) ------- */
/* Paths below are relative to src/self_supervised/dinov2/.  K = number of prototypes (65 536 in the shipped configs),
 * K % 4 == 0, rows 16-byte aligned.  All tensors f32 unless a name says bf16.  Reductions are fixed-order.
 * Validated on the B200 against oracle/ssl_oracle.py (tests/test_ssl_gpu.py, strict). */
/* out[rows,K] = softmax((t - center[K]) * inv_temp): DINOLoss.softmax_center_teacher loss/dino_clstoken_loss.py:28-31,
 * iBOTPatchLoss.softmax_center_teacher loss/ibot_patch_loss.py:39-51. */
int apla_softmax_center(const float* t, int64_t ldt, const float* center, float inv_temp, int rows, int K, float* out,
                        int64_t ldo, apla_stream_t stream);
/* out[K] = scale * sum over rows of a[rows,K]; ws = workspace of splits*K floats: torch.sum(teacher_output, dim=0)
 * loss/dino_clstoken_loss.py:84 (scale 1) and torch.sum(teacher_patch_tokens.mean(1), dim=0) loss/ibot_patch_loss.py:131
 * (scale 1/n).  The data-parallel all-reduce of out sits between this and apla_center_ema. */
int apla_colsum_f32(const float* a, int64_t ld, int rows, int K, float* ws, int splits, float scale, float* out,
                    apla_stream_t stream);
/* center = center * momentum + batch_sum * inv_count * (1 - momentum): apply_center_update
 * loss/dino_clstoken_loss.py:88-98, loss/ibot_patch_loss.py:134-145 (inv_count = 1 / (len * world)). */
int apla_center_ema(float* center, const float* batch_sum, int K, float inv_count, float momentum,
                    apla_stream_t stream);
/* Soft-target cross-entropy rows: q = t0[row % t_rows] (+ t1[row % t_rows] if t1 != NULL), z = s * inv_temp,
 * row_loss[row] = -w (sum_k q_k z_k - mass lse(z)), w = w_uniform * (w_row ? w_row[row] : 1); lse / mass [rows] are
 * kept for the backward.  One launch covers DINOLoss.forward over all crop pairs (loss/dino_clstoken_loss.py:62-74)
 * or iBOTPatchLoss.forward_masked (loss/ibot_patch_loss.py:102-121). */
int apla_soft_ce_fwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                     int t_rows, const float* w_row, float w_uniform, float inv_temp, float* row_loss, float* lse,
                     float* mass, apla_stream_t stream);
/* ds[rows,K] (f32, or bf16 if ds_is_bf16) = -w inv_temp *gscale (q - mass softmax(z)); gscale = device scalar with the
 * upstream gradient (NULL = 1).  What autograd produces for the two losses above. */
int apla_soft_ce_bwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                     int t_rows, const float* w_row, float w_uniform, float inv_temp, const float* lse,
                     const float* mass, const float* gscale, void* ds, int64_t ldd, int ds_is_bf16,
                     apla_stream_t stream);
/* apla_soft_ce_fwd + apla_soft_ce_bwd of the same rows in ONE launch, for callers that know the upstream gradient when the
 * loss is taken (apla_ssl_objective): the second pass walks each row backwards so that it re-reads from L2 what the first
 * pass just streamed.  row_loss uses w_fwd, ds uses w_bwd (loss_dict scale vs. scale x loss weight). */
int apla_soft_ce_fwd_bwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                         int t_rows, const float* w_row, float w_fwd, float w_bwd, float inv_temp, const float* gscale,
                         float* row_loss, void* ds, int64_t ldd, int ds_is_bf16, apla_stream_t stream);
/* Sinkhorn-Knopp teacher targets, sinkhorn_knopp_teacher loss/dino_clstoken_loss.py:33-60, loss/ibot_patch_loss.py:53-83,
 * in the [samples, K] layout: out = exp(t * inv_temp); then per iteration apla_colsum_f32 (+ all-reduce) and
 * apla_sk_normalize: p[b,k] <- p[b,k] * col_scale / colsum[k] (col_scale = 1/K), then p[b,:] <- p[b,:] * row_scale / sum_k p[b,k]
 * (row_scale = 1/B between iterations, 1 after the last so that every sample's targets sum to 1). */
int apla_sk_exp(const float* t, int64_t ldt, float inv_temp, int rows, int K, float* out, int64_t ldo,
                apla_stream_t stream);
int apla_sk_normalize(float* p, int64_t ld, int rows, int K, const float* colsum, float col_scale, float row_scale,
                      apla_stream_t stream);
/* out[0] = scale * sum a[0..n) (single CTA, fixed order): the .mean() / .sum() that end the losses. */
int apla_sum_f32(const float* a, int n, float scale, float* out, apla_stream_t stream);
/* y = x / max(||x||, eps) per row of x[rows,d] (f32 or bf16), y as bf16 and / or f32 (either may be NULL):
 * F.normalize in DINOHead.forward layers/dino_head.py:38-39; also the first line of KoLeoLoss loss/koleo_loss.py:41. */
int apla_l2norm_fwd(const void* x, int64_t ldx, int x_is_f32, int rows, int d, float eps, void* y_bf16, float* y_f32,
                    int64_t ldy, apla_stream_t stream);
/* dx = (dy - y (y . dy)) / ||x||; dy and dx share one dtype (f32 or bf16). */
int apla_l2norm_bwd(const void* x, int64_t ldx, int x_is_f32, const void* dy, int64_t ld_dy, int grads_are_f32,
                    int rows, int d, float eps, void* dx, int64_t ld_dx, apla_stream_t stream);
/* W[K,d] = g[K] v[K,d] / ||v[k,:]|| as bf16 and / or f32: weight_norm(nn.Linear(bottleneck, K, bias=False))
 * layers/dino_head.py:27-31, and its backward from dW[K,d] (dg or dv may be NULL: weight_g is frozen when
 * norm_last_layer is set). */
int apla_weightnorm_fwd(const float* g, const float* v, int K, int d, void* w_bf16, float* w_f32,
                        apla_stream_t stream);
int apla_weightnorm_bwd(const float* g, const float* v, const float* dW, int64_t ld_dw, int K, int d, float* dg,
                        float* dv, apla_stream_t stream);
/* KoLeoLoss.forward loss/koleo_loss.py:23-45 on already L2-normalised rows xn[groups*n, D] (each group of n rows is
 * one call of the reference): nn[i] = argmax_j!=i xn_i . xn_j, dist[i] = ||xn_i - xn_nn + 1e-8||,
 * row_loss[i] = -w log(dist + eps) / n.  The backward returns the gradient for the UN-normalised rows x. */
int apla_koleo_fwd(const float* xn, int groups, int n, int D, float eps, float w, int32_t* nn, float* dist,
                   float* row_loss, apla_stream_t stream);
int apla_koleo_bwd(const float* x, const float* xn, int groups, int n, int D, float eps, float norm_eps, float w,
                   const int32_t* nn, const float* dist, const float* gscale, float* dx, apla_stream_t stream);
/* teacher[n] = m teacher + (1 - m) student: DINOv2.update_teacher models.py:437-447. */
int apla_ema_update(float* teacher, const float* student, int64_t n, float m, apla_stream_t stream);
/* The objective of one self-supervised step on given head outputs as ONE native launch sequence (12 launches, no host code
 * between them): teacher targets + centre statistics + forward and backward of dino_local / dino_global / ibot with the
 * scales of DINOv2.forward (models.py:227-234, 237-318, 374-433; two global crops, shared head, "centering").
 *   s_scores [n_local*B + 2B + n_masked, K]: student head output = local CLS rows (crop-major), global CLS rows, masked rows;
 *   t_scores [2B + n_masked, K]: teacher head output, global CLS rows already swapped (models.py:244), masked rows;
 *   t_probs: workspace of t_scores' shape; row_ws: 3 * student-rows floats; col_ws: splits * K floats;
 *   dino_center / ibot_center [K]: the centres to USE this step (pending update applied);
 *   masks_weight [n_masked]: dinov2_utils.py:48;  ds (f32 or bf16, may be NULL): gradient of
 *   dino_weight (local + global) + ibot_weight * ibot with respect to s_scores, times *gscale (NULL = 1);
 *   losses[3] = dino_local_crops_loss, dino_global_crops_loss, 2 * ibot_loss as loss_dict reports them;
 *   dino_batch_sum [K] / ibot_batch_mean [K]: all-reduce (sum) over the ranks, then apla_center_ema with
 *   inv_count = 1 / (2B * world) and 1 / world respectively. */
int apla_ssl_objective(const float* s_scores, int64_t lds, const float* t_scores, int64_t ldt, float* t_probs, int64_t ldp,
                       const float* dino_center, const float* ibot_center, const float* masks_weight, int B, int n_local,
                       int n_masked, int K, float teacher_temp, float student_temp, float dino_weight, float ibot_weight,
                       float* row_ws, float* col_ws, int splits, void* ds, int64_t ldd, int ds_is_bf16,
                       const float* gscale, float* losses, float* dino_batch_sum, float* ibot_batch_mean,
                       apla_stream_t stream);

/* --- one block, two calls -------------------------------------------------------------------------------- */
/* Block.forward (src/utils/transformers/vit.py:279-288: x += ls1(attn(norm1(x))); x += ls2(mlp(norm2(x)))) around an
 * APLA attention (src/apla/appla_attn.py:50-83) and its backward, as the launch sequences the step engine runs per
 * block.  cu_seqlens != NULL: packed crops, block-diagonal attention (dinov2/layers/block.py:274-288).
 * Weights: bf16 [out,in] and pre-transposed [in,out] copies of the frozen Linears, the dense projection copy with the
 * trainable rows scattered in (apla_proj_refresh), fp32 biases / LayerNorm / LayerScale vectors (g1, g2 NULL = none).
 * idx: the r trainable rows (compact path, r <= 128, r_pad = r rounded up to 64); rowmap: int32[D] row -> slot of dW1
 * or -1 (dense path); exactly one of the two is set when a weight gradient is requested. */
typedef struct apla_block_weights {
  const void *wqkv, *wqkvT, *wproj, *wprojT, *wfc1, *wfc1T, *wfc2, *wfc2T;
  const float *bqkv, *bproj, *bfc1, *bfc2, *ln1w, *ln1b, *ln2w, *ln2b, *g1, *g2;
  const int32_t *idx, *rowmap;
  int32_t D, H, hidden, r, r_pad;
  float eps1, eps2, scale;
} apla_block_weights;
int apla_block_weights_size(void);
/* x_in f32[T,D] -> x_mid f32[T,D] (after the attention branch) -> x_out f32[T,D]; saves qkv bf16[T,3D], ao bf16[T,D],
 * lse f32[T,H], dgelu f16[T,hidden] for backward; ln_tmp bf16[T,D] and gelu_tmp bf16[T,hidden] are scratch. */
int apla_block_fwd(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp, void* qkv,
                   void* ao, float* lse, void* dgelu, void* gelu_tmp, const int32_t* cu_seqlens, int num_seqs,
                   int max_seqlen, int T, apla_stream_t stream);
/* The same forward keeping nothing for backward (no autograd, evaluation, a frozen teacher): fc1 writes gelu(h) only and
 * there is no dgelu.  lse_tmp f32[T,H], ln_tmp, qkv, ao and gelu_tmp are scratch.  x_out may alias x_in (x_in is last
 * read by the projection); x_mid may alias neither. */
int apla_block_fwd_infer(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp,
                         void* qkv, void* ao, float* lse_tmp, void* gelu_tmp, const int32_t* cu_seqlens, int num_seqs,
                         int max_seqlen, int T, apla_stream_t stream);
/* dx_out f32[T,D] -> dx_in f32[T,D] (NULL: no input gradient wanted; may alias dx_mid) and dw1 f32[r,D] / db1 f32[r]
 * (NULL: no weight gradient; zeroed here).  dx_mid f32[T,D], dyb bf16[T,D], dh bf16[T,hidden], dln bf16[T,D],
 * dsub bf16[T,r_pad] (compact path), d_ao bf16[T,D], delta f32[T,H], dqkv bf16[T,3D] are scratch.
 * Chaining consecutive blocks: a block's backward starts by forming dyb = bf16(g2 * dx_out), a pass over the fp32
 * gradient the block BEHIND it has just written.  That block can write it instead, from the LayerNorm-1 backward that
 * produces dx_in: give it dyb_prev bf16[T,D] and gamma_prev = the g2 of the block in front (NULL = 1); the block in front
 * is then called with dyb_ready = 1 and that buffer as dyb.  dyb_prev NULL / dyb_ready 0: the stand-alone behaviour. */
int apla_block_bwd(const apla_block_weights* w, const float* dx_out, const float* x_in, const float* x_mid,
                   const void* qkv, const void* ao, const float* lse, const void* dgelu, float* dx_mid, float* dx_in,
                   void* dyb, void* dh, void* dln, void* dsub, void* d_ao, float* delta, void* dqkv, float* dw1,
                   float* db1, const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int T, int dyb_ready,
                   void* dyb_prev, const float* gamma_prev, apla_stream_t stream);

/* --- step engine: the whole fine-tune step as one native call sequence ------------------------------------ */
/* Replaces Trainer.global_step's device work (src/defaults/trainer.py:106-138): Classifier.forward
 * (src/defaults/models.py:81-92), CrossEntropyLoss, loss.backward() restricted to the APLA rows + head,
 * clip_grad_norm_ and AdamW.  The engine owns no memory; every buffer is a caller-allocated device pointer
 * registered by name (global: block = -1; per block: block = 0..L-1).  See apla_b200/engine.py for the table. */
typedef void* apla_engine_t;
apla_engine_t apla_engine_create(int B, int N, int D, int H, int L, int hidden, int C, int patch, int img, int kpad,
                                 int r, int r_pad, int full_rows, float eps, float scale);
void apla_engine_destroy(apla_engine_t e);
/* Optional global buffers (NULL = unset): "hyper" f32[3] -- {lr, 1 - beta1^t, sqrt(1 - beta2^t)} read by the AdamW
 * kernel instead of its arguments (replayable graphs); "drop_path" f32[L, 2, B] -- stochastic depth (vit.py drop_path):
 * the scale (0 or 1/keep) of block l's attention (0) and MLP (1) branch for image b.  With it set, the training forward
 * computes x_mid = x_in + s[l,0,b] * ls1(attn) and x_out = x_mid + s[l,1,b] * ls2(mlp) for the first n_img images, and the
 * backward scales the bf16 gradient each branch reads by the same s (the fp32 residual gradient is not scaled); unset,
 * the step runs exactly its launches without it.  The evaluation entries never read it. */
int apla_engine_set_ptr(apla_engine_t e, const char* name, int block, void* p);
/* Options (default in brackets): "infer_batch" [0] -- images per apla_engine_infer call (its workspace capacity);
 * "cls_only_last_block" [2] -- evaluate the per-token tail of the LAST block (projection,
 * LayerNorm 2, MLP and their input gradients; value >= 1) and its attention (value 2: apla_attn_cls_*) for the CLS
 * rows only, because only norm(x)[:, 0] reaches the head (vit.py:417-419, models.py:87); 0 = every token.  Values 0 and
 * 1 give bit-identical logits / loss; 2 replaces bf16 tensor-core attention of that row by fp32 arithmetic;
 * "criterion" [0] -- the training loss: 0 = cross-entropy (nn.CrossEntropyLoss), 1 = BCE-with-logits
 * (nn.BCEWithLogitsLoss, multi-label: apla_engine_forward_n reads `targets` as f32[n_img, C] BCE targets and refuses
 * int64 labels, as apla_engine_forward does); any other value is refused. */
int apla_engine_set_option(apla_engine_t e, const char* name, int value);
/* Trainable arena layout (fp32): [proj_weight1 x L | fc.weight | proj_bias1 x L | fc.bias]; the first
 * apla_engine_arena_decay_size() elements are weight-decayed (src/defaults/wrappers.py:205-221). */
int64_t apla_engine_arena_size(apla_engine_t e);
int64_t apla_engine_arena_decay_size(apla_engine_t e);
/* logits (+ loss and dlogits when labels != NULL): loss += loss_scale * sum CE, dlogits *= grad_scale. */
int apla_engine_forward(apla_engine_t e, const float* images, const int64_t* labels, float loss_scale,
                        float grad_scale, apla_stream_t stream);
/* The same forward over the first 1 <= n_img <= B images of the step's buffers (the partial last batch of an epoch), with
 * hard labels int64[n_img] or probability targets f32[n_img, C] (apla_cross_entropy_soft), at most one of the two; with
 * neither, logits only.  Every GEMM, attention, LayerNorm and the head run over n_img*N rows (n_img CLS rows); the xs
 * checkpoints keep their capacity stride B*N*D and rows beyond n_img*N of any buffer are neither read nor written.  The
 * engine records n_img: the next apla_engine_backward runs over the same rows.  apla_engine_forward(...) is
 * apla_engine_forward_n(e, images, B, labels, NULL, ...).  Under option "criterion" = 1 the loss is BCE-with-logits:
 * `targets` are f32[n_img, C] multi-label targets (apla_bce_with_logits) and int64 `labels` are refused before any launch;
 * the backward consumes dlogits whichever criterion produced them. */
int apla_engine_forward_n(apla_engine_t e, const float* images, int n_img, const int64_t* labels, const float* targets,
                          float loss_scale, float grad_scale, apla_stream_t stream);
/* Evaluation forward: logits_f32[n_img, C] (and, with emb != NULL, the bf16 final-norm CLS rows emb[n_img, D] the head
 * reads) for 1 <= n_img <= "infer_batch" images with the CURRENT weights (arena + refreshed projection copies).  Runs the
 * forward's launch sequence with the forward-only fc1 over its own workspace, registered by name (block = -1):
 * "infer_x" f32[2, cap*N, D], "infer_ln" bf16[cap*N, D], "infer_qkv" bf16[cap*N, 3D], "infer_ao" bf16[cap*N, D],
 * "infer_lse" f32[cap*N, H], "infer_gelu" bf16[cap*N, hidden], "infer_patches" bf16[cap*P, kpad],
 * "infer_pe_out" bf16[cap*P, D], "infer_cls_ln" bf16[cap, D].  Reads no buffer of the step but the weights and writes
 * none: captured step graphs stay valid. */
int apla_engine_infer(apla_engine_t e, const float* images, int n_img, float* logits, void* emb, apla_stream_t stream);
/* CLS attention map of the last block (vit.py get_last_selfattention(x)[:, :, 0, :]): probs_f32[n_img, H, N] for
 * 1 <= n_img <= "infer_batch" images with the CURRENT weights.  The launch sequence of apla_engine_infer up to and
 * including the last block's attention (any "cls_only_last_block" mode), then apla_attn_probs with q_rows = 1; that
 * block's tail, the final norm and the head are not run.  Same workspace and the same argument checks as
 * apla_engine_infer. */
int apla_engine_cls_attention(apla_engine_t e, const float* images, int n_img, float* probs, apla_stream_t stream);
/* Backward through blocks block_from, block_from-1, ..., block_to (block_from == L-1 also zeroes the gradient arena
 * and runs the head / final-norm backward first).  Splitting the range lets the host start the data-parallel
 * all-reduce of the upper blocks' gradients while the lower blocks are still running.  It runs over the n_img images of
 * the last apla_engine_forward / apla_engine_forward_n, whose saved activations it consumes. */
int apla_engine_backward(apla_engine_t e, int block_from, int block_to, apla_stream_t stream);
/* clip + AdamW over the arena, then refresh of the dense bf16 projection copies */
int apla_engine_optim(apla_engine_t e, float gscale, float max_norm, float lr, float wd, float beta1, float beta2,
                      float eps, int step, apla_stream_t stream);

/* --- data-parallel gradient exchange -------------------------------------------------------------------- */
/* In-place sum all-reduce of arena[offset, offset + count) across the `world` GPUs of one node, as ONE kernel launch
 * (capturable in a CUDA graph): replaces the DDP reducer's NCCL all-reduce of the trainable gradients
 * (src/defaults/wrappers.py:182-183; SURVEY.md 8b `apla_grad_arena_allreduce`).  peer_bufs[i] / peer_flags[i] are HOST
 * arrays of DEVICE pointers to rank i's arena and flag words as mapped into THIS process (symmetric / peer memory);
 * flags hold apla_grad_arena_allreduce_flag_words() zero-initialised uint32 per rank; `epochs` is a LOCAL zero-initialised
 * device buffer of apla_grad_arena_allreduce_epoch_words() uint32.  offset and count are multiples of 4 floats.
 * A second slice [offset_b, offset_b + count_b) (count_b may be 0) is reduced by the same launch.  `multicast` is the
 * NVLS multicast mapping of the arena (NULL: plain peer loads / stores).
 * Every rank must issue the same sequence of calls per channel (0..3); calls on different channels may overlap.
 * The result is bit-identical on all ranks (one owner per element). `ctas` <= 148 (0 = 32), 128 threads each. */
int apla_grad_arena_allreduce(const void* const* peer_bufs, const void* const* peer_flags, void* multicast, void* epochs,
                              int rank, int world, int64_t offset_floats, int64_t count_floats, int64_t offset_b,
                              int64_t count_b, int channel, int ctas, apla_stream_t stream);
int apla_grad_arena_allreduce_flag_words(void);
int apla_grad_arena_allreduce_epoch_words(void);

#ifdef __cplusplus
}
#endif
#endif /* APLA_B200_H_ */
