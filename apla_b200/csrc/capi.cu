// extern "C" surface declared in include/apla_b200.h: thin argument checks + forwarding to the kernels.
#include "../../include/apla_b200.h"

#include "common.cuh"
#include "kernels.cuh"

using namespace apla;

#define S(stream) reinterpret_cast<cudaStream_t>(stream)

extern "C" {

const char* apla_last_error(void) { return get_error(); }
int apla_version(void) { return 100; }
int64_t apla_launch_count(void) { return launch_count(); }

int apla_device_check(void) {
  int dev = 0, major = 0, minor = 0;
  APLA_CUDA(cudaGetDevice(&dev));
  APLA_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  APLA_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  APLA_CHECK(major == 10, "apla_b200 needs an sm_100 (B200) device, found compute capability %d.%d", major, minor);
  return 0;
}

int apla_gemm_bias_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* out, int ldo, int M,
                       int N, int K, apla_stream_t stream) {
  return gemm_tn(EPI_BIAS, A, W, M, N, K, lda, ldw, out, nullptr, bias, nullptr, nullptr, ldo, S(stream), 0);
}
int apla_gemm_bias_gelu_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* h, void* g,
                            int ldo, int M, int N, int K, apla_stream_t stream) {
  return gemm_tn(EPI_BIAS_GELU, A, W, M, N, K, lda, ldw, h, g, bias, nullptr, nullptr, ldo, S(stream), 0);
}
int apla_gemm_bias_ls_residual_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                   const float* gamma, const float* resid, float* out, int ldo, int M, int N, int K,
                                   apla_stream_t stream) {
  return gemm_tn(EPI_RESID, A, W, M, N, K, lda, ldw, out, nullptr, bias, gamma, resid, ldo, S(stream), 0);
}
int apla_gemm_bias_ls_residual_scaled_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                          const float* gamma, const float* resid, const float* row_scale,
                                          int rows_per_scale, float* out, int ldo, int M, int N, int K,
                                          apla_stream_t stream) {
  if (!A || !W || !resid || !row_scale || !out) {
    set_error("apla_gemm_bias_ls_residual_scaled_fwd: null A, W, resid, row_scale or out");
    return 1;
  }
  APLA_CHECK(M > 0 && N > 0 && K > 0, "apla_gemm_bias_ls_residual_scaled_fwd: empty problem %dx%dx%d", M, N, K);
  APLA_CHECK(rows_per_scale >= 1, "apla_gemm_bias_ls_residual_scaled_fwd: rows_per_scale=%d must be >= 1", rows_per_scale);
  return gemm_resid_scaled(A, W, M, N, K, lda, ldw, out, bias, gamma, resid, ldo, row_scale, rows_per_scale, S(stream));
}
int apla_gemm_bias_ls_residual_ln_fwd(const void* A, int lda, const void* W, int ldw, const float* bias,
                                      const float* gamma, const float* resid, float* out, int ldo, const float* ln_w,
                                      const float* ln_b, void* ln_out, int ld_ln, float eps, int M, int N, int K,
                                      int one_launch, apla_stream_t stream) {
  return gemm_resid_ln(A, W, M, N, K, lda, ldw, out, bias, gamma, resid, ldo, ln_w, ln_b, ln_out, ld_ln, eps, S(stream),
                       one_launch);
}
int apla_gemm_bias_ls_accumulate(const void* A, int lda, const void* W, int ldw, const float* bias, const float* gamma,
                                 float* out, int ldo, int M, int N, int K, apla_stream_t stream) {
  return gemm_tn(EPI_RED, A, W, M, N, K, lda, ldw, out, nullptr, bias, gamma, nullptr, ldo, S(stream), 0);
}
int apla_gemm_dgrad(const void* dY, int ldy, const void* Wt, int ldwt, void* dX, int ldx, int M, int K_in, int N_out,
                    apla_stream_t stream) {
  return gemm_tn(EPI_BIAS, dY, Wt, M, K_in, N_out, ldy, ldwt, dX, nullptr, nullptr, nullptr, nullptr, ldx, S(stream), 0);
}
int apla_gemm_dgrad_gelu_bwd(const void* dY, int ldy, const void* Wt, int ldwt, const void* h, void* dH, int ldh,
                             int M, int K_in, int N_out, apla_stream_t stream) {
  return gemm_tn(EPI_GELU_BWD, dY, Wt, M, K_in, N_out, ldy, ldwt, dH, nullptr, nullptr, nullptr, h, ldh, S(stream), 0);
}
int apla_gemm_bias_gelu_dgelu_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* dgelu, void* g,
                                  int ldo, int M, int N, int K, apla_stream_t stream) {
  return gemm_tn(EPI_BIAS_GELU_D, A, W, M, N, K, lda, ldw, dgelu, g, bias, nullptr, nullptr, ldo, S(stream), 0);
}
int apla_gemm_bias_gelu_only_fwd(const void* A, int lda, const void* W, int ldw, const float* bias, void* g, int ldo,
                                 int M, int N, int K, apla_stream_t stream) {
  if (!A || !W || !g) {
    set_error("apla_gemm_bias_gelu_only_fwd: null A, W or g");
    return 1;
  }
  return gemm_tn(EPI_BIAS_GELU_G, A, W, M, N, K, lda, ldw, g, nullptr, bias, nullptr, nullptr, ldo, S(stream), 0);
}
int apla_gemm_dgrad_mul(const void* dY, int ldy, const void* Wt, int ldwt, const void* mul, void* dH, int ldh, int M,
                        int K_in, int N_out, apla_stream_t stream) {
  return gemm_tn(EPI_MUL_F16, dY, Wt, M, K_in, N_out, ldy, ldwt, dH, nullptr, nullptr, nullptr, mul, ldh, S(stream), 0);
}
int apla_gemm_dgrad_delta(const void* dY, int ldy, const void* Wt, int ldwt, const void* O, void* dO, int ldo,
                          float* delta, int M, int D, int N_out, apla_stream_t stream) {
  return gemm_tn(EPI_DELTA, dY, Wt, M, D, N_out, ldy, ldwt, dO, delta, nullptr, nullptr, O, ldo, S(stream), 0);
}
int apla_proj_wgrad_gather(const void* dYsub, int ldy, const void* X, int ldx, const int32_t* rowmap, float* dW1,
                           int ldw, int T, int D_in, int n_pad, int r, apla_stream_t stream) {
  // dW1^T[D_in, n] = X^T[D_in, T] . dYsub[T, n]: D_in on the MMA M dimension, the (small) r on N
  return gemm_wgrad_nt(X, dYsub, D_in, n_pad, T, ldx, ldy, dW1, ldw, rowmap, rowmap ? n_pad : r, S(stream));
}
int apla_colsum(const void* dY, int64_t ld, int T, int n, const int32_t* rowmap, float* db, apla_stream_t stream) {
  return colsum(dY, ld, T, n, db, rowmap, S(stream));
}

int apla_layernorm_fwd(const float* x, int64_t ldx, const float* w, const float* b, void* y, int64_t ldy, int rows,
                       int D, float eps, apla_stream_t stream) {
  return layernorm_fwd(x, ldx, w, b, y, ldy, rows, D, eps, S(stream));
}
int apla_layernorm_bwd(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w, const float* dres,
                       int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb, const float* gamma,
                       void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad, int rows, int D, float eps,
                       apla_stream_t stream) {
  return layernorm_bwd(dy, ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx, dxb, ld_dxb, gamma, sub, ld_sub, idx, r, r_pad,
                       rows, D, eps, S(stream));
}
int apla_layernorm_bwd_scaled(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w,
                              const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb,
                              const float* gamma, void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad,
                              const float* row_scale, int rows_per_scale, int rows, int D, float eps,
                              apla_stream_t stream) {
  if (!dy || !x || !w || !dx || !dxb || !row_scale) {
    set_error("apla_layernorm_bwd_scaled: null dy, x, w, dx, dxb or row_scale");
    return 1;
  }
  APLA_CHECK(rows > 0 && D > 0, "apla_layernorm_bwd_scaled: empty problem rows=%d D=%d", rows, D);
  APLA_CHECK(rows_per_scale >= 1, "apla_layernorm_bwd_scaled: rows_per_scale=%d must be >= 1", rows_per_scale);
  return layernorm_bwd(dy, ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx, dxb, ld_dxb, gamma, sub, ld_sub, idx, r, r_pad,
                       rows, D, eps, S(stream), row_scale, rows_per_scale);
}
int apla_gather_cols(const void* dy, int64_t ld, void* sub, int64_t ld_sub, const int32_t* idx, int r, int r_pad,
                     int rows, apla_stream_t stream) {
  return gather_cols(dy, ld, sub, ld_sub, idx, r, r_pad, rows, S(stream));
}

int apla_ls_cast(const float* x, int64_t ldx, const float* gamma, void* out, int64_t ldo, int rows, int D,
                 apla_stream_t stream) {
  return ls_cast(x, ldx, gamma, out, ldo, rows, D, S(stream));
}

int apla_attn_fwd(const void* qkv, void* out, float* lse, const int32_t* cu_seqlens, int num_seqs, int max_seqlen,
                  int total_tokens,
                  int H, float scale, apla_stream_t stream) {
  return attn_fwd(qkv, out, lse, cu_seqlens, num_seqs, max_seqlen, total_tokens, H, scale, S(stream));
}
int apla_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, float* delta, void* dqkv,
                  const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int total_tokens, int H, float scale,
                  apla_stream_t stream) {
  return attn_bwd(qkv, out, dout, lse, delta, dqkv, cu_seqlens, num_seqs, max_seqlen, total_tokens, H, scale, S(stream));
}

int apla_attn_cls_fwd(const void* qkv, void* out, float* lse, int B, int N, int H, float scale, apla_stream_t stream) {
  return attn_cls_fwd(qkv, out, lse, B, N, H, scale, S(stream));
}
int apla_attn_cls_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, int B, int N,
                      int H, float scale, apla_stream_t stream) {
  return attn_cls_bwd(qkv, out, dout, lse, dqkv, B, N, H, scale, S(stream));
}

int apla_attn_probs(const void* qkv, const float* lse, float* probs, int B, int N, int H, int q_rows, float scale,
                    apla_stream_t stream) {
  return attn_probs(qkv, lse, probs, B, N, H, q_rows, scale, S(stream));
}

int apla_patchify(const float* images, void* patches, int B, int Simg, int patch, int kpad, apla_stream_t stream) {
  return patchify(images, patches, B, Simg, patch, kpad, S(stream));
}
int apla_assemble_tokens(const void* patch, const float* cls, const float* pos, float* x, int B, int P, int D,
                         apla_stream_t stream) {
  return assemble_tokens(patch, cls, pos, x, B, P, D, S(stream));
}
int apla_head_fwd(const void* xn, const float* W, const float* bias, float* logits, int B, int D, int C,
                  apla_stream_t stream) {
  return head_fwd(xn, W, bias, logits, B, D, C, S(stream));
}
int apla_cross_entropy(const float* logits, const int64_t* labels, float* dlogits, float* loss, int B, int C,
                       float grad_scale, float loss_scale, apla_stream_t stream) {
  return cross_entropy(logits, labels, dlogits, loss, B, C, grad_scale, loss_scale, S(stream));
}
int apla_cross_entropy_soft(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                            float grad_scale, float loss_scale, apla_stream_t stream) {
  return cross_entropy_soft(logits, targets, dlogits, loss, B, C, grad_scale, loss_scale, S(stream));
}
int apla_eval_accumulate(const float* logits, const int64_t* labels, int B, int C, float* acc, apla_stream_t stream) {
  return eval_accumulate(logits, labels, B, C, acc, S(stream));
}
int apla_bce_with_logits(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                         float grad_scale, float loss_scale, apla_stream_t stream) {
  return bce_with_logits(logits, targets, dlogits, loss, B, C, grad_scale, loss_scale, S(stream));
}
int apla_eval_accumulate_bce(const float* logits, const float* targets, int B, int C, double* acc,
                             apla_stream_t stream) {
  return eval_accumulate_bce(logits, targets, B, C, acc, S(stream));
}
int apla_head_bwd(const float* dlogits, const void* xn, const float* W, float* dW, float* db, void* dxn, int B, int D,
                  int C, apla_stream_t stream) {
  return head_bwd(dlogits, xn, W, dW, db, dxn, B, D, C, S(stream));
}

int apla_grad_sumsq(const float* g, int64_t n, float scale, float* out, apla_stream_t stream) {
  return grad_sumsq(g, n, scale, out, S(stream));
}
int apla_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, int64_t n_decay, const float* sumsq,
                    float gscale, float max_norm, float lr, float wd, float beta1, float beta2, float eps, int step,
                    apla_stream_t stream) {
  return adamw_step(p, g, m, v, n, n_decay, sumsq, gscale, max_norm, lr, wd, beta1, beta2, eps, step, S(stream));
}
int apla_proj_refresh(const float* w1, const float* b1, const int32_t* idx, void* wfull, void* wfullT, float* bfull,
                      int L, int r, int D, int64_t w1_block_stride, int64_t b1_block_stride, apla_stream_t stream) {
  return proj_refresh(w1, b1, idx, wfull, wfullT, bfull, L, r, D, w1_block_stride, b1_block_stride, S(stream));
}

// --- DINOv2 self-supervised objective (ssl.cu) ---
int apla_softmax_center(const float* t, int64_t ldt, const float* center, float inv_temp, int rows, int K, float* out,
                        int64_t ldo, apla_stream_t stream) {
  return ssl_softmax_center(t, ldt, center, inv_temp, rows, K, out, ldo, S(stream));
}
int apla_colsum_f32(const float* a, int64_t ld, int rows, int K, float* ws, int splits, float scale, float* out,
                    apla_stream_t stream) {
  return ssl_colsum_f32(a, ld, rows, K, ws, splits, scale, out, S(stream));
}
int apla_center_ema(float* center, const float* batch_sum, int K, float inv_count, float momentum,
                    apla_stream_t stream) {
  return ssl_center_ema(center, batch_sum, K, inv_count, momentum, S(stream));
}
int apla_soft_ce_fwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                     int t_rows, const float* w_row, float w_uniform, float inv_temp, float* row_loss, float* lse,
                     float* mass, apla_stream_t stream) {
  return ssl_soft_ce_fwd(s, lds, rows, K, t0, t1, ldt, t_rows, w_row, w_uniform, inv_temp, row_loss, lse, mass,
                         S(stream));
}
int apla_soft_ce_bwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                     int t_rows, const float* w_row, float w_uniform, float inv_temp, const float* lse,
                     const float* mass, const float* gscale, void* ds, int64_t ldd, int ds_is_bf16,
                     apla_stream_t stream) {
  return ssl_soft_ce_bwd(s, lds, rows, K, t0, t1, ldt, t_rows, w_row, w_uniform, inv_temp, lse, mass, gscale, ds, ldd,
                         ds_is_bf16, S(stream));
}
int apla_soft_ce_fwd_bwd(const float* s, int64_t lds, int rows, int K, const float* t0, const float* t1, int64_t ldt,
                         int t_rows, const float* w_row, float w_fwd, float w_bwd, float inv_temp, const float* gscale,
                         float* row_loss, void* ds, int64_t ldd, int ds_is_bf16, apla_stream_t stream) {
  return ssl_soft_ce_fwd_bwd(s, lds, rows, K, t0, t1, ldt, t_rows, w_row, w_fwd, w_bwd, inv_temp, gscale, row_loss, ds, ldd,
                             ds_is_bf16, S(stream));
}
int apla_sk_exp(const float* t, int64_t ldt, float inv_temp, int rows, int K, float* out, int64_t ldo,
                apla_stream_t stream) {
  return ssl_sk_exp(t, ldt, inv_temp, rows, K, out, ldo, S(stream));
}
int apla_sk_normalize(float* p, int64_t ld, int rows, int K, const float* colsum, float col_scale, float row_scale,
                      apla_stream_t stream) {
  return ssl_sk_normalize(p, ld, rows, K, colsum, col_scale, row_scale, S(stream));
}
int apla_sum_f32(const float* a, int n, float scale, float* out, apla_stream_t stream) {
  return ssl_sum_f32(a, n, scale, out, S(stream));
}
int apla_l2norm_fwd(const void* x, int64_t ldx, int x_is_f32, int rows, int d, float eps, void* y_bf16, float* y_f32,
                    int64_t ldy, apla_stream_t stream) {
  return ssl_l2norm_fwd(x, ldx, x_is_f32, rows, d, eps, y_bf16, y_f32, ldy, S(stream));
}
int apla_l2norm_bwd(const void* x, int64_t ldx, int x_is_f32, const void* dy, int64_t ld_dy, int grads_are_f32,
                    int rows, int d, float eps, void* dx, int64_t ld_dx, apla_stream_t stream) {
  return ssl_l2norm_bwd(x, ldx, x_is_f32, dy, ld_dy, grads_are_f32, rows, d, eps, dx, ld_dx, S(stream));
}
int apla_weightnorm_fwd(const float* g, const float* v, int K, int d, void* w_bf16, float* w_f32,
                        apla_stream_t stream) {
  return ssl_weightnorm_fwd(g, v, K, d, w_bf16, w_f32, S(stream));
}
int apla_weightnorm_bwd(const float* g, const float* v, const float* dW, int64_t ld_dw, int K, int d, float* dg,
                        float* dv, apla_stream_t stream) {
  return ssl_weightnorm_bwd(g, v, dW, ld_dw, K, d, dg, dv, S(stream));
}
int apla_koleo_fwd(const float* xn, int groups, int n, int D, float eps, float w, int32_t* nn, float* dist,
                   float* row_loss, apla_stream_t stream) {
  return ssl_koleo_fwd(xn, groups, n, D, eps, w, nn, dist, row_loss, S(stream));
}
int apla_koleo_bwd(const float* x, const float* xn, int groups, int n, int D, float eps, float norm_eps, float w,
                   const int32_t* nn, const float* dist, const float* gscale, float* dx, apla_stream_t stream) {
  return ssl_koleo_bwd(x, xn, groups, n, D, eps, norm_eps, w, nn, dist, gscale, dx, S(stream));
}
int apla_ema_update(float* teacher, const float* student, int64_t n, float m, apla_stream_t stream) {
  return ssl_ema(teacher, student, n, m, S(stream));
}
int apla_ssl_objective(const float* s_scores, int64_t lds, const float* t_scores, int64_t ldt, float* t_probs, int64_t ldp,
                       const float* dino_center, const float* ibot_center, const float* masks_weight, int B, int n_local,
                       int n_masked, int K, float teacher_temp, float student_temp, float dino_weight, float ibot_weight,
                       float* row_ws, float* col_ws, int splits, void* ds, int64_t ldd, int ds_is_bf16,
                       const float* gscale, float* losses, float* dino_batch_sum, float* ibot_batch_mean,
                       apla_stream_t stream) {
  return ssl_objective(s_scores, lds, t_scores, ldt, t_probs, ldp, dino_center, ibot_center, masks_weight, B, n_local,
                       n_masked, K, teacher_temp, student_temp, dino_weight, ibot_weight, row_ws, col_ws, splits, ds, ldd,
                       ds_is_bf16, gscale, losses, dino_batch_sum, ibot_batch_mean, S(stream));
}

int apla_grad_arena_allreduce(const void* const* peer_bufs, const void* const* peer_flags, void* multicast, void* epochs,
                              int rank, int world, int64_t offset_floats, int64_t count_floats, int64_t offset_b,
                              int64_t count_b, int channel, int ctas, apla_stream_t stream) {
  if (!peer_bufs || !peer_flags || !epochs) {
    set_error("apla_grad_arena_allreduce: null argument");
    return 1;
  }
  return grad_arena_allreduce(reinterpret_cast<float* const*>(const_cast<void* const*>(peer_bufs)),
                              reinterpret_cast<uint32_t* const*>(const_cast<void* const*>(peer_flags)),
                              reinterpret_cast<float*>(multicast), reinterpret_cast<uint32_t*>(epochs), rank, world,
                              offset_floats, count_floats, offset_b, count_b, channel, ctas, S(stream));
}
int apla_grad_arena_allreduce_flag_words(void) { return grad_arena_allreduce_flag_words(); }
int apla_grad_arena_allreduce_epoch_words(void) { return grad_arena_allreduce_epoch_words(); }

}  // extern "C"
