// One transformer block around an APLA attention as TWO native calls (forward, backward): the launch sequences the step
// engine runs per block (engine.cu), exposed for callers that keep their own autograd graph -- the block-level drop-in
// apla_b200/apla/apla_block.py.  Replaces Block.forward (src/utils/transformers/vit.py:279-288) and, with cu_seqlens,
// NestedTensorBlock.forward_nested (src/self_supervised/dinov2/layers/block.py:274-288), plus what autograd derives
// from them: input gradients for every token, weight gradients only for the r trainable projection rows
// (src/apla/appla_attn.py:64-79).  No allocation, no synchronisation: every buffer is the caller's.
#include "../../include/apla_b200.h"

#include "common.cuh"
#include "kernels.cuh"

using namespace apla;

namespace {

int check_weights(const apla_block_weights* w, const char* who) {
  APLA_CHECK(w != nullptr, "%s: null weights", who);
  APLA_CHECK(w->D > 0 && w->D % 64 == 0 && w->H > 0 && w->H * 64 == w->D && w->hidden > 0 && w->hidden % 64 == 0,
             "%s: bad geometry D=%d H=%d hidden=%d (head dim must be 64)", who, w->D, w->H, w->hidden);
  APLA_CHECK(w->wqkv && w->wproj && w->wfc1 && w->wfc2 && w->ln1w && w->ln1b && w->ln2w && w->ln2b,
             "%s: missing weight pointers", who);
  return 0;
}

// Stochastic depth: branch_scale = f32[2, T / rows_per_scale]; element b of branch 0 (attention) or 1 (MLP) scales the
// rows_per_scale token rows of image b.  NULL: no drop path.
int check_scale(const float* branch_scale, int rows_per_scale, int T, const char* who) {
  APLA_CHECK(rows_per_scale >= 1, "%s: rows_per_scale=%d must be >= 1", who, rows_per_scale);
  APLA_CHECK(branch_scale == nullptr || T % rows_per_scale == 0,
             "%s: T=%d is not a whole number of images of rows_per_scale=%d rows", who, T, rows_per_scale);
  return 0;
}

// One branch's residual update, out = resid + gamma * (A W^T + bias), with the branch output of image b scaled by
// scale[b] when there is a scale (EPI_RESID_SCALED)
int resid_gemm(const void* A, const void* W, int T, int D, int K, float* out, const float* bias, const float* gamma,
               const float* resid, const float* scale, int rows_per_scale, cudaStream_t s) {
  if (scale) return gemm_resid_scaled(A, W, T, D, K, K, K, out, bias, gamma, resid, D, scale, rows_per_scale, s);
  return gemm_tn(EPI_RESID, A, W, T, D, K, K, K, out, nullptr, bias, gamma, resid, D, s, 0);
}

// The forward of both entries.  dgelu set: fc1 also saves gelu' for backward; NULL: it writes gelu(h) only.
int block_fwd(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp, void* qkv,
              void* ao, float* lse, void* dgelu, void* gelu_tmp, const int32_t* cu_seqlens, int num_seqs, int max_seqlen,
              int T, const float* branch_scale, int rows_per_scale, cudaStream_t s) {
  const int D = w->D, Hd = w->hidden;
  const float* s0 = branch_scale;
  const float* s1 = branch_scale ? branch_scale + T / rows_per_scale : nullptr;
  if (int rc = layernorm_fwd(x_in, D, w->ln1w, w->ln1b, ln_tmp, D, T, D, w->eps1, s)) return rc;
  if (int rc = gemm_tn(EPI_BIAS, ln_tmp, w->wqkv, T, 3 * D, D, D, D, qkv, nullptr, w->bqkv, nullptr, nullptr, 3 * D, s, 0))
    return rc;
  if (int rc = attn_fwd(qkv, ao, lse, cu_seqlens, num_seqs, max_seqlen, T, w->H, w->scale, s)) return rc;
  if (int rc = resid_gemm(ao, w->wproj, T, D, D, x_mid, w->bproj, w->g1, x_in, s0, rows_per_scale, s)) return rc;
  if (int rc = layernorm_fwd(x_mid, D, w->ln2w, w->ln2b, ln_tmp, D, T, D, w->eps2, s)) return rc;
  if (dgelu) {
    if (int rc = gemm_tn(EPI_BIAS_GELU_D, ln_tmp, w->wfc1, T, Hd, D, D, D, dgelu, gelu_tmp, w->bfc1, nullptr, nullptr, Hd,
                         s, 0))
      return rc;
  } else if (int rc = gemm_tn(EPI_BIAS_GELU_G, ln_tmp, w->wfc1, T, Hd, D, D, D, gelu_tmp, nullptr, w->bfc1, nullptr,
                              nullptr, Hd, s, 0)) {
    return rc;
  }
  return resid_gemm(gelu_tmp, w->wfc2, T, D, Hd, x_out, w->bfc2, w->g2, x_mid, s1, rows_per_scale, s);
}

}  // namespace

extern "C" {

int apla_block_weights_size(void) { return (int)sizeof(apla_block_weights); }

int apla_block_fwd(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp, void* qkv,
                   void* ao, float* lse, void* dgelu, void* gelu_tmp, const int32_t* cu_seqlens, int num_seqs,
                   int max_seqlen, int T, apla_stream_t stream) {
  return apla_block_fwd_scaled(w, x_in, x_mid, x_out, ln_tmp, qkv, ao, lse, dgelu, gelu_tmp, cu_seqlens, num_seqs,
                               max_seqlen, T, nullptr, 1, stream);
}

int apla_block_fwd_scaled(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp,
                          void* qkv, void* ao, float* lse, void* dgelu, void* gelu_tmp, const int32_t* cu_seqlens,
                          int num_seqs, int max_seqlen, int T, const float* branch_scale, int rows_per_scale,
                          apla_stream_t stream) {
  if (int rc = check_weights(w, "apla_block_fwd")) return rc;
  APLA_CHECK(T > 0 && num_seqs > 0 && max_seqlen > 0, "apla_block_fwd: empty problem");
  if (int rc = check_scale(branch_scale, rows_per_scale, T, "apla_block_fwd")) return rc;
  APLA_CHECK(x_in && x_mid && x_out && ln_tmp && qkv && ao && lse && dgelu && gelu_tmp, "apla_block_fwd: null buffer");
  return block_fwd(w, x_in, x_mid, x_out, ln_tmp, qkv, ao, lse, dgelu, gelu_tmp, cu_seqlens, num_seqs, max_seqlen, T,
                   branch_scale, rows_per_scale, reinterpret_cast<cudaStream_t>(stream));
}

int apla_block_fwd_infer(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out, void* ln_tmp,
                         void* qkv, void* ao, float* lse_tmp, void* gelu_tmp, const int32_t* cu_seqlens, int num_seqs,
                         int max_seqlen, int T, apla_stream_t stream) {
  return apla_block_fwd_infer_scaled(w, x_in, x_mid, x_out, ln_tmp, qkv, ao, lse_tmp, gelu_tmp, cu_seqlens, num_seqs,
                                     max_seqlen, T, nullptr, 1, stream);
}

int apla_block_fwd_infer_scaled(const apla_block_weights* w, const float* x_in, float* x_mid, float* x_out,
                                void* ln_tmp, void* qkv, void* ao, float* lse_tmp, void* gelu_tmp,
                                const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int T,
                                const float* branch_scale, int rows_per_scale, apla_stream_t stream) {
  if (int rc = check_weights(w, "apla_block_fwd_infer")) return rc;
  APLA_CHECK(T > 0 && num_seqs > 0 && max_seqlen > 0, "apla_block_fwd_infer: empty problem");
  if (int rc = check_scale(branch_scale, rows_per_scale, T, "apla_block_fwd_infer")) return rc;
  APLA_CHECK(x_in && x_mid && x_out && ln_tmp && qkv && ao && lse_tmp && gelu_tmp, "apla_block_fwd_infer: null buffer");
  APLA_CHECK(x_mid != x_in && x_mid != x_out, "apla_block_fwd_infer: x_mid may not alias x_in or x_out");
  // apla_block_fwd's sequence; fc1 writes gelu(h) only.  x_in is last read by the projection, so x_out may alias it.
  return block_fwd(w, x_in, x_mid, x_out, ln_tmp, qkv, ao, lse_tmp, nullptr, gelu_tmp, cu_seqlens, num_seqs, max_seqlen,
                   T, branch_scale, rows_per_scale, reinterpret_cast<cudaStream_t>(stream));
}

int apla_block_bwd(const apla_block_weights* w, const float* dx_out, const float* x_in, const float* x_mid,
                   const void* qkv, const void* ao, const float* lse, const void* dgelu, float* dx_mid, float* dx_in,
                   void* dyb, void* dh, void* dln, void* dsub, void* d_ao, float* delta, void* dqkv, float* dw1,
                   float* db1, const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int T, int dyb_ready,
                   void* dyb_prev, const float* gamma_prev, apla_stream_t stream) {
  return apla_block_bwd_scaled(w, dx_out, x_in, x_mid, qkv, ao, lse, dgelu, dx_mid, dx_in, dyb, dh, dln, dsub, d_ao, delta,
                               dqkv, dw1, db1, cu_seqlens, num_seqs, max_seqlen, T, dyb_ready, dyb_prev, gamma_prev,
                               nullptr, 1, stream);
}

int apla_block_bwd_scaled(const apla_block_weights* w, const float* dx_out, const float* x_in, const float* x_mid,
                          const void* qkv, const void* ao, const float* lse, const void* dgelu, float* dx_mid,
                          float* dx_in, void* dyb, void* dh, void* dln, void* dsub, void* d_ao, float* delta, void* dqkv,
                          float* dw1, float* db1, const int32_t* cu_seqlens, int num_seqs, int max_seqlen, int T,
                          int dyb_ready, void* dyb_prev, const float* gamma_prev, const float* branch_scale,
                          int rows_per_scale, apla_stream_t stream) {
  if (int rc = check_weights(w, "apla_block_bwd")) return rc;
  APLA_CHECK(T > 0 && num_seqs > 0 && max_seqlen > 0, "apla_block_bwd: empty problem");
  if (int rc = check_scale(branch_scale, rows_per_scale, T, "apla_block_bwd")) return rc;
  APLA_CHECK(dx_out && x_mid && dgelu && dx_mid && dyb && dh && dln && w->wfc1T && w->wfc2T, "apla_block_bwd: null buffer");
  // a hand-over from the block behind holds bf16(gamma2 * dx_out), without this block's MLP-branch scale
  APLA_CHECK(!(branch_scale && dyb_ready), "apla_block_bwd: with branch scales the block forms dyb itself (dyb_ready = 0)");
  APLA_CHECK(branch_scale == nullptr || w->D % 128 == 0,
             "apla_block_bwd: with branch scales D=%d must be a multiple of 128 (the row-scaled LayerNorm backward)", w->D);
  const bool want_w = dw1 != nullptr;
  const bool compact = want_w && w->rowmap == nullptr;         // r <= 128: gathered columns; else dense dY + row map
  APLA_CHECK(!want_w || (db1 && ao && w->r > 0 && w->r <= w->D), "apla_block_bwd: weight gradient needs db1, ao, 0 < r <= D");
  APLA_CHECK(!compact || (dsub && w->idx && w->r_pad >= w->r && w->r_pad % 64 == 0),
             "apla_block_bwd: the compact path needs dsub, idx and r_pad (multiple of 64) >= r");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int D = w->D, Hd = w->hidden, r = w->r;
  // drop path: the bf16 gradient a branch reads carries that branch's scale (s1: MLP, s0: attention); the fp32 residual
  // gradients dx_mid / dx_in do not
  const float* s0 = branch_scale;
  const float* s1 = branch_scale ? branch_scale + T / rows_per_scale : nullptr;
  // MLP branch: dyb = bf16(s1 * gamma2 * dx_out) -> fc2 dgrad x gelu' -> fc1 dgrad
  // (dyb_ready: the block behind this one already wrote it from its LayerNorm-1 backward, see the header)
  if (!dyb_ready) {
    if (int rc = ls_cast(dx_out, D, w->g2, dyb, D, T, D, s, s1, rows_per_scale)) return rc;
  }
  if (int rc = gemm_tn(EPI_MUL_F16, dyb, w->wfc2T, T, Hd, D, D, D, dh, nullptr, nullptr, nullptr, dgelu, Hd, s, 0)) return rc;
  if (int rc = gemm_tn(EPI_BIAS, dh, w->wfc1T, T, D, Hd, Hd, Hd, dln, nullptr, nullptr, nullptr, nullptr, D, s, 0)) return rc;
  // dx_mid = dx_out + LN2'(dln); dyb = bf16(s0 * gamma1 * dx_mid) = gradient at the projection output (+ its APLA columns)
  if (int rc = layernorm_bwd(dln, D, x_mid, D, w->ln2w, dx_out, D, dx_mid, D, dyb, D, w->g1, compact ? dsub : nullptr,
                             compact ? w->r_pad : 0, compact ? w->idx : nullptr, compact ? r : 0, compact ? w->r_pad : 0,
                             T, D, w->eps2, s, s0, rows_per_scale))
    return rc;
  if (want_w) {
    APLA_CUDA(cudaMemsetAsync(dw1, 0, size_t(r) * D * sizeof(float), s));
    APLA_CUDA(cudaMemsetAsync(db1, 0, size_t(r) * sizeof(float), s));
    if (compact) {
      if (int rc = gemm_wgrad_nt(ao, dsub, D, w->r_pad, T, D, w->r_pad, dw1, D, nullptr, r, s)) return rc;
      if (int rc = colsum(dsub, w->r_pad, T, r, db1, nullptr, s)) return rc;
    } else {
      if (int rc = gemm_wgrad_nt(ao, dyb, D, D, T, D, D, dw1, D, w->rowmap, D, s)) return rc;
      if (int rc = colsum(dyb, D, T, D, db1, w->rowmap, s)) return rc;
    }
  }
  if (dx_in == nullptr) return 0;      // nothing upstream wants a gradient (block 0 behind a frozen embedding)
  APLA_CHECK(x_in && qkv && ao && lse && d_ao && delta && dqkv && w->wprojT && w->wqkvT, "apla_block_bwd: null buffer");
  if (int rc = gemm_tn(EPI_DELTA, dyb, w->wprojT, T, D, D, D, D, d_ao, delta, nullptr, nullptr, ao, D, s, 0)) return rc;
  if (int rc = attn_bwd(qkv, nullptr, d_ao, lse, delta, dqkv, cu_seqlens, num_seqs, max_seqlen, T, w->H, w->scale, s))
    return rc;
  if (int rc = gemm_tn(EPI_BIAS, dqkv, w->wqkvT, T, D, 3 * D, 3 * D, 3 * D, dln, nullptr, nullptr, nullptr, nullptr, D, s, 0))
    return rc;
  // dx_in = dx_mid + LN1'(dln); optionally also bf16(gamma_prev * dx_in) for the block in front
  return layernorm_bwd(dln, D, x_in, D, w->ln1w, dx_mid, D, dx_in, D, dyb_prev, dyb_prev ? D : 0, dyb_prev ? gamma_prev : nullptr,
                       nullptr, 0, nullptr, 0, 0, T, D, w->eps1, s);
}

}  // extern "C"
