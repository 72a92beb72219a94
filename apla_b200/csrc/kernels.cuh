// Internal (C++) declarations of the kernel launchers; the C ABI in capi.cu and the step engine call these.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace apla {

enum { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_RESID = 2, EPI_GELU_BWD = 3, EPI_F32_T = 4, EPI_DELTA = 5, EPI_BIAS_GELU_D = 6,
       EPI_MUL_F16 = 7, EPI_RED = 8, EPI_RESID_LN = 9, EPI_BIAS_GELU_G = 10, EPI_RESID_SCALED = 11 };

// gemm.cu
int gemm_tn(int epi, const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
            const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream, int bn_override);
int gemm2_tn(int epi, const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
             const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream, int bn);
int gemm_wgrad_nt(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* dW, int ldw,
                  const int* rowmap, int n_valid, cudaStream_t stream);
// out_f32 = resid + gamma * (A B^T + bias) and ln_out_bf16 = LayerNorm(out_f32): one launch when the 2-CTA kernel covers
// the width (gemm2.cu, EPI_RESID_LN), otherwise the residual GEMM followed by layernorm_fwd.  With row_scale set, the
// branch of row m is scaled by row_scale[m / rows_per_scale] (gemm_resid_scaled), always in the two-launch form.
int gemm_resid_ln(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                  const float* gamma, const float* resid, int ldo, const float* ln_w, const float* ln_b, void* ln_out,
                  int ld_ln, float eps, cudaStream_t stream, int fuse_mode = -1, const float* row_scale = nullptr,
                  int rows_per_scale = 1);
// out_f32 = resid + row_scale[m / rows_per_scale] * gamma * (A B^T + bias): the residual epilogue with a per-row-group
// scale (stochastic depth), 2-CTA kernel only (gemm2.cu, EPI_RESID_SCALED)
int gemm_resid_scaled(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                      const float* gamma, const float* resid, int ldo, const float* row_scale, int rows_per_scale,
                      cudaStream_t stream);
int gemm2_resid_scaled(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                       const float* gamma, const float* resid, int ldo, const float* row_scale, int rows_per_scale,
                       cudaStream_t stream, int bn);
bool gemm2_resid_ln_supported(int N);
int gemm2_resid_ln(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                   const float* gamma, const float* resid, int ldo, const float* ln_w, const float* ln_b, void* ln_out,
                   int ld_ln, float eps, cudaStream_t stream);

// attention.cu (dispatch), attention_tc.cu / attention_tc_bwd.cu (streaming tcgen05 kernels, any sequence length)
int attn_fwd(const void* qkv, void* out, float* lse, const int* cu_seqlens, int num_seqs, int max_seqlen,
             int total_tokens, int H,
             float scale, cudaStream_t stream);
int attn_fwd_tc(const void* qkv, void* out, float* lse, const int* cu_seqlens, int num_seqs, int max_seqlen,
                int total_tokens, int H, float scale, cudaStream_t stream);
int attn_bwd_tc(const void* qkv, const void* dout, const float* lse, const float* delta, void* dqkv,
                const int* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
                cudaStream_t stream);
// attention_fwd_sr.cu: persistent sequence-resident forward, max_seqlen <= 272
int attn_fwd_sr(const void* qkv, void* out, float* lse, const int* cu_seqlens, int num_seqs, int max_seqlen,
                int total_tokens, int H, float scale, cudaStream_t stream);
// attention_fused.cu: single-pass fused backward (dQ, dK, dV in one launch), max_seqlen <= 272
bool attn_fused_supported(int max_seqlen);
int attn_bwd_fused(const void* qkv, const void* dout, const float* lse, const float* delta, void* dqkv,
                   const int* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
                   cudaStream_t stream);
// attention_bwd2.cu: second-generation fused backward (odd token on CUDA cores, event-driven issuer), max_seqlen <= 257
bool attn_bwd2_supported(int max_seqlen);
int attn_bwd2(const void* qkv, const void* dout, const float* lse, const float* delta, void* dqkv,
              const int* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
              cudaStream_t stream);
int attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
             const int* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
             cudaStream_t stream);

// attention_cls.cu: the last block's attention for the CLS query only (rows b*N of out / lse / dout; dqkv dense)
int attn_cls_fwd(const void* qkv, void* out, float* lse, int B, int N, int H, float scale, cudaStream_t stream);
int attn_cls_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int B, int N, int H,
                 float scale, cudaStream_t stream);

// attention_probs.cu: probs_f32[B, H, q_rows, N] = exp(scale q k^T - lse) of the first q_rows queries per sequence
int attn_probs(const void* qkv, const float* lse, float* probs, int B, int N, int H, int q_rows, float scale,
               cudaStream_t stream);

// rowwise.cu
int layernorm_fwd(const float* x, int64_t ldx, const float* w, const float* b, void* y, int64_t ldy, int rows, int D,
                  float eps, cudaStream_t stream);
// row_scale set: dxb and sub of row t are also scaled by row_scale[t / rows_per_scale] (dx is not); D % 128 == 0 only
int layernorm_bwd(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w, const float* dres,
                  int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb, const float* gamma, void* sub,
                  int64_t ld_sub, const int* idx, int r, int r_pad, int rows, int D, float eps, cudaStream_t stream,
                  const float* row_scale = nullptr, int rows_per_scale = 1);
int gather_cols(const void* dy, int64_t ld, void* sub, int64_t ld_sub, const int* idx, int r, int r_pad, int rows,
                cudaStream_t stream);
// row_scale set: row t is also scaled by row_scale[t / rows_per_scale]
int ls_cast(const float* x, int64_t ldx, const float* gamma, void* out, int64_t ldo, int rows, int D,
            cudaStream_t stream, const float* row_scale = nullptr, int rows_per_scale = 1);
int colsum(const void* a, int64_t ld, int rows, int n, float* out, const int* rowmap, cudaStream_t stream);
int patchify(const float* img, void* out, int B, int S, int p, int kpad, cudaStream_t stream);
int assemble_tokens(const void* patch, const float* cls, const float* pos, float* x, int B, int P, int D,
                    cudaStream_t stream);

// head_optim.cu
int head_fwd(const void* xn, const float* W, const float* bias, float* logits, int B, int D, int C, cudaStream_t s);
int cross_entropy(const float* logits, const int64_t* labels, float* dlogits, float* loss, int B, int C,
                  float grad_scale, float loss_scale, cudaStream_t s);
int cross_entropy_soft(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                       float grad_scale, float loss_scale, cudaStream_t s);
int eval_accumulate(const float* logits, const int64_t* labels, int B, int C, float* acc, cudaStream_t s);
int bce_with_logits(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                    float grad_scale, float loss_scale, cudaStream_t s);
int eval_accumulate_bce(const float* logits, const float* targets, int B, int C, double* acc, cudaStream_t s);
int head_bwd(const float* dlogits, const void* xn, const float* W, float* dW, float* db, void* dxn, int B, int D, int C,
             cudaStream_t s);
int grad_sumsq(const float* g, int64_t n, float scale, float* out, cudaStream_t s);
int adamw_step(float* p, const float* g, float* m, float* v, int64_t n, int64_t n_decay, const float* sumsq,
               float gscale, float max_norm, float lr, float wd, float b1, float b2, float eps, int step,
               cudaStream_t s, const float* hyper = nullptr);
int proj_refresh(const float* w1, const float* b1, const int* idx, void* wfull, void* wfullT, float* bfull, int L,
                 int r, int D, int64_t w1_block_stride, int64_t b1_block_stride, cudaStream_t s);

// dp_allreduce.cu: two-shot all-reduce of the gradient arena over symmetric (peer-mapped) memory, graph-capturable
int grad_arena_allreduce(float* const* peer_bufs, uint32_t* const* peer_flags, float* multicast, uint32_t* epochs, int rank,
                         int world, int64_t offset_floats, int64_t count_floats, int64_t offset_b, int64_t count_b,
                         int channel, int ctas, cudaStream_t stream);
int grad_arena_allreduce_flag_words();
int grad_arena_allreduce_epoch_words();

// ssl.cu: row kernels of the DINOv2 self-supervised objective (SURVEY 8f row f2)
int ssl_softmax_center(const float* t, int64_t ldt, const float* center, float inv_temp, int rows, int K, float* out,
                       int64_t ldo, cudaStream_t s);
int ssl_colsum_f32(const float* a, int64_t ld, int rows, int K, float* ws, int splits, float scale, float* out,
                   cudaStream_t s);
int ssl_center_ema(float* center, const float* batch_sum, int K, float inv_count, float momentum, cudaStream_t s);
int ssl_soft_ce_fwd(const float* sp, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                    int t_rows, const float* w_row, float w_uniform, float inv_temp, float* row_loss, float* lse,
                    float* mass, cudaStream_t s);
int ssl_soft_ce_bwd(const float* sp, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                    int t_rows, const float* w_row, float w_uniform, float inv_temp, const float* lse, const float* mass,
                    const float* gscale, void* ds, int64_t ldd, int ds_is_bf16, cudaStream_t s);
int ssl_soft_ce_fwd_bwd(const float* sp, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                        int t_rows, const float* w_row, float w_fwd, float w_bwd, float inv_temp, const float* gscale,
                        float* row_loss, void* ds, int64_t ldd, int ds_is_bf16, cudaStream_t s);
int ssl_sk_exp(const float* t, int64_t ldt, float inv_temp, int rows, int K, float* out, int64_t ldo, cudaStream_t s);
int ssl_sk_normalize(float* p, int64_t ld, int rows, int K, const float* colsum, float col_scale, float row_scale,
                     cudaStream_t s);
int ssl_sum_f32(const float* a, int n, float scale, float* out, cudaStream_t s);
int ssl_l2norm_fwd(const void* x, int64_t ldx, int x_is_f32, int rows, int d, float eps, void* y_bf16, float* y_f32,
                   int64_t ldy, cudaStream_t s);
int ssl_l2norm_bwd(const void* x, int64_t ldx, int x_is_f32, const void* dy, int64_t ld_dy, int grads_are_f32, int rows,
                   int d, float eps, void* dx, int64_t ld_dx, cudaStream_t s);
int ssl_weightnorm_fwd(const float* g, const float* v, int K, int d, void* w_bf16, float* w_f32, cudaStream_t s);
int ssl_weightnorm_bwd(const float* g, const float* v, const float* dW, int64_t ld_dw, int K, int d, float* dg, float* dv,
                       cudaStream_t s);
int ssl_koleo_fwd(const float* xn, int groups, int n, int D, float eps, float w, int* nn, float* dist, float* row_loss,
                  cudaStream_t s);
int ssl_koleo_bwd(const float* x, const float* xn, int groups, int n, int D, float eps, float norm_eps, float w,
                  const int* nn, const float* dist, const float* gscale, float* dx, cudaStream_t s);
int ssl_ema(float* t, const float* sp, int64_t n, float m, cudaStream_t s);
int ssl_objective(const float* s_scores, int64_t lds, const float* t_scores, int64_t ldt, float* t_probs, int64_t ldp,
                  const float* dino_center, const float* ibot_center, const float* masks_weight, int B, int n_local,
                  int n_masked, int K, float teacher_temp, float student_temp, float dino_weight, float ibot_weight,
                  float* row_ws, float* col_ws, int splits, void* ds, int64_t ldd, int ds_is_bf16, const float* gscale,
                  float* losses, float* dino_batch_sum, float* ibot_batch_mean, cudaStream_t s);

}  // namespace apla
