// Step engine: the whole APLA fine-tune step (Trainer.global_step, src/defaults/trainer.py:106-138, over
// Classifier.forward src/defaults/models.py:81-92 and Block.forward src/utils/transformers/vit.py:279-288) as ONE
// native call sequence on one stream -- no Python between kernels, capturable in a CUDA graph.
//
// The engine owns no memory: the host side (apla_b200/engine.py) allocates every buffer (torch tensors), hands the
// device pointers over by name, and keeps them alive.  Gradient flow implemented here = exactly what autograd
// computes for the reference: input gradients everywhere a trainable tensor sits upstream, weight gradients only
// for the APLA rows of every projection and for the classifier head; block 0's attention / qkv / proj input
// gradients are skipped because nothing upstream of them is trainable (SURVEY.md 2.3 K24).
#include <map>
#include <string>
#include <vector>

#include "../../include/apla_b200.h"
#include "common.cuh"
#include "kernels.cuh"

namespace apla {

struct BlockPtrs {
  // frozen weights (bf16 working copies, [out,in] and pre-transposed [in,out]) and fp32 vectors
  const void *wqkv = nullptr, *wqkvT = nullptr, *wfc1 = nullptr, *wfc1T = nullptr, *wfc2 = nullptr, *wfc2T = nullptr;
  void *wproj = nullptr, *wprojT = nullptr;  // dense projection copies, refreshed after every update
  const float *bqkv = nullptr, *bfc1 = nullptr, *bfc2 = nullptr, *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr,
              *ln2b = nullptr, *g1 = nullptr, *g2 = nullptr;
  float* bproj = nullptr;
  // saved activations
  void *qkv = nullptr, *ao = nullptr, *hpre = nullptr;  // hpre: fp16 GELU derivative of the fc1 pre-activation
  float* lse = nullptr;
};

struct Engine {
  // shape
  int B = 0, N = 0, D = 0, H = 0, L = 0, hidden = 0, C = 0, P = 0, patch = 0, img = 0, kpad = 0;
  int r = 0, r_pad = 0, full_rows = 0;  // full_rows: partial_size == dim handled through rowmap on the dense dY
  // Only the CLS token of the last block's output reaches the head (forward_features returns norm(x)[:, 0],
  // src/utils/transformers/vit.py:417-419; Classifier.fc models.py:87).  Everything in the last block that is
  // per-token -- the projection, LayerNorm 2, the whole MLP branch and, on the way back, their input gradients -- is
  // therefore evaluated on the B CLS rows only (row stride N*D); all other rows of those tensors are dead values in
  // the forward pass and exact zeros in the backward pass.  Attention itself still needs every token's K and V.
  int cls_last = 2;   // 0 = every token everywhere, 1 = CLS-only per-token tail, 2 = also CLS-only attention (default)
  float eps = 1e-6f, scale = 0.125f;
  std::vector<BlockPtrs> blk;
  std::map<std::string, void*> g;  // global buffers by name
  std::string err;
  // The APLA weight / bias gradient of a block (a small GEMM + a column sum) depends only on that block's LayerNorm-2
  // backward and feeds nothing before the optimiser, so it runs on a side stream beside the projection dgrad, the
  // attention backward and the qkv dgrad -- persistent kernels whose last round leaves most SMs idle (768 (image, head)
  // groups over 148 CTAs = 5.19 rounds).  Fork / join are events, so the pattern is capturable in the step's CUDA graph.
  // side_wgrad = number of dsub slots the host allocated (2 enables the side stream for partial_size < dim; the
  // full-rows path reads dxb and needs none).
  int side_wgrad = 0;
  // evaluation forward (apla_engine_infer): images per call at most, set by option "infer_batch"; 0 = no workspace
  int infer_cap = 0;
  // images of the last training forward (apla_engine_forward_n; B for apla_engine_forward): the backward consumes that
  // forward's saved activations, so it runs over the same n_cur * N rows
  int n_cur = 0;
  // training loss, option "criterion": 0 = cross-entropy (int64 labels or fp32 class probabilities), 1 = BCE-with-logits
  // (fp32 multi-label targets only)
  int criterion = 0;
  cudaStream_t side = nullptr;
  std::vector<cudaEvent_t> ev_fork, ev_done;
  ~Engine() {
    for (cudaEvent_t ev : ev_fork) cudaEventDestroy(ev);
    for (cudaEvent_t ev : ev_done) cudaEventDestroy(ev);
    if (side) cudaStreamDestroy(side);
  }
  int side_ready() {
    if (side) return 0;
    int lo = 0, hi = 0;
    APLA_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    APLA_CUDA(cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, lo));   // lowest: the main chain's CTAs go first
    ev_fork.resize(L);
    ev_done.resize(L);
    for (int l = 0; l < L; ++l) {
      APLA_CUDA(cudaEventCreateWithFlags(&ev_fork[l], cudaEventDisableTiming));
      APLA_CUDA(cudaEventCreateWithFlags(&ev_done[l], cudaEventDisableTiming));
    }
    return 0;
  }
  int T() const { return B * N; }
  template <class Tp>
  Tp* get(const char* name) {
    auto it = g.find(name);
    return it == g.end() ? nullptr : reinterpret_cast<Tp*>(it->second);
  }
};

static const char* kGlobalNames[] = {
    // inputs / embedding
    "patches", "wpe", "bpe", "pe_out", "cls", "pos",
    // residual stream checkpoints xs[0..2L] as one [2L+1, T, D] fp32 buffer
    "xs",
    // transients
    "ln_out", "gelu_out", "dx", "dxb", "dsub", "dO", "dqkv", "delta",
    // final norm + head
    "lnfw", "lnfb", "cls_ln", "logits", "dlogits", "loss", "dcls",
    // trainable arena (params / grads / adam moments), index tables, scratch
    "params", "grads", "exp_avg", "exp_avg_sq", "idx", "rowmap", "sumsq",
};

// optional global buffers (not checked by check_ready): "hyper" = float[3] {lr, 1 - beta1^t, sqrt(1 - beta2^t)} read by
// the AdamW kernel instead of its launch arguments, so that a captured step can be replayed with new values;
// "drop_path" = float[L, 2, B] stochastic-depth scales s[l, branch, image] in {0, 1/keep} (vit.py drop_path), written by
// the host before every training forward (see drop_path_scale)
static const char* kOptionalNames[] = {"hyper", "drop_path"};

// Scales of block l's branch (0 = attention, 1 = MLP) for the images of a step, or NULL without drop path.  The branch
// output of image b is multiplied by s[l, branch, b] in the forward (EPI_RESID_SCALED), and so is the bf16 gradient the
// branch reads in the backward (the row-scaled LayerNorm backward); the fp32 residual gradient passes unscaled.
static const float* drop_path_scale(Engine* e, int l, int branch) {
  const float* s = e->get<float>("drop_path");
  return s ? s + size_t(2 * l + branch) * e->B : nullptr;
}

// evaluation workspace (apla_engine_infer), sized for infer_cap images of N tokens; none of it is used by the step.
// "infer_x" holds two fp32 [cap*N, D] residual buffers: the block input (overwritten by the block output) and the stream
// after the attention branch -- two buffers whatever the depth.
static const char* kInferNames[] = {"infer_x", "infer_ln", "infer_qkv", "infer_ao", "infer_lse", "infer_gelu",
                                    "infer_patches", "infer_pe_out", "infer_cls_ln"};

static int check_ready(Engine* e) {
  for (const char* n : kGlobalNames) {
    if (std::string(n) == "rowmap" && !e->full_rows) continue;
    if (std::string(n) == "dsub" && e->full_rows) continue;
    APLA_CHECK(e->g.count(n) && e->g[n] != nullptr, "engine: buffer '%s' was not set", n);
  }
  for (int l = 0; l < e->L; ++l) {
    const BlockPtrs& b = e->blk[l];
    APLA_CHECK(b.wqkv && b.wqkvT && b.wfc1 && b.wfc1T && b.wfc2 && b.wfc2T && b.wproj && b.wprojT && b.bproj &&
                   b.bfc1 && b.bfc2 && b.ln1w && b.ln1b && b.ln2w && b.ln2b && b.qkv && b.ao && b.hpre && b.lse,
               "engine: block %d has unset pointers", l);
  }
  return 0;
}

// arena layout: [W1 (L x r x D) | fc.weight (C x D) | b1 (L x r) | fc.bias (C)]
struct Arena {
  int64_t w1, fcw, b1, fcb, n, n_decay;
};
static Arena arena_of(const Engine* e) {
  Arena a;
  a.w1 = 0;
  a.fcw = int64_t(e->L) * e->r * e->D;
  a.b1 = a.fcw + int64_t(e->C) * e->D;
  a.fcb = a.b1 + int64_t(e->L) * e->r;
  a.n = a.fcb + e->C;
  a.n_decay = a.b1;
  return a;
}

// The step's forward over the first n images of its buffers (n = B: the full batch).  Every launch covers n*N token rows
// or n CLS rows, so rows beyond them -- stale from an earlier, larger batch -- are never read; only the xs checkpoints
// keep their capacity stride TD.
static int engine_forward(Engine* e, const float* images, int n, const int64_t* labels, const float* targets,
                          float loss_scale, float grad_scale, cudaStream_t s) {
  APLA_CHECK(n >= 1 && n <= e->B, "apla_engine_forward_n: n_img=%d outside [1, %d]", n, e->B);
  APLA_CHECK(!(labels && targets), "apla_engine_forward_n: labels and targets are both set");
  APLA_CHECK(!(labels && e->criterion == 1),
             "apla_engine_forward: criterion 1 (BCE-with-logits) takes fp32 targets [n_img, C], not int64 labels");
  if (int rc = check_ready(e)) return rc;
  const int D = e->D, B = n, N = e->N, L = e->L, Hd = e->hidden, T = B * N;
  const size_t TD = size_t(e->T()) * D;
  e->n_cur = n;
  float* xs = e->get<float>("xs");
  void* ln_out = e->get<void>("ln_out");
  void* gelu_out = e->get<void>("gelu_out");
  const Arena ar = arena_of(e);
  float* params = e->get<float>("params");

  // ---- patch embedding + cls + pos (vit.py:389-396) ----
  if (int rc = patchify(images, e->get<void>("patches"), B, e->img, e->patch, e->kpad, s)) return rc;
  if (int rc = gemm_tn(EPI_BIAS, e->get<void>("patches"), e->get<void>("wpe"), B * e->P, D, e->kpad, e->kpad, e->kpad,
                       e->get<void>("pe_out"), nullptr, e->get<float>("bpe"), nullptr, nullptr, D, s, 0))
    return rc;
  if (int rc = assemble_tokens(e->get<void>("pe_out"), e->get<float>("cls"), e->get<float>("pos"), xs, B, e->P, D, s))
    return rc;

  // ---- blocks (vit.py:279-288) ----
  for (int l = 0; l < L; ++l) {
    const BlockPtrs& b = e->blk[l];
    float* x_in = xs + size_t(2 * l) * TD;
    float* x_mid = xs + size_t(2 * l + 1) * TD;
    float* x_out = xs + size_t(2 * l + 2) * TD;
    // LayerNorm 1: block 0 normalises the embedded tokens; later blocks get it from the previous block's fc2 launch
    if (l == 0) {
      if (int rc = layernorm_fwd(x_in, D, b.ln1w, b.ln1b, ln_out, D, T, D, e->eps, s)) return rc;
    }
    if (int rc = gemm_tn(EPI_BIAS, ln_out, b.wqkv, T, 3 * D, D, D, D, b.qkv, nullptr, b.bqkv, nullptr, nullptr, 3 * D, s, 0))
      return rc;
    // rows / row strides of the per-token tail of the block: every token, or the CLS rows of the last block
    const bool cls = e->cls_last && l == L - 1;
    if (cls && e->cls_last >= 2) {   // one query row per (image, head); the other rows of ao stay zero
      if (int rc = attn_cls_fwd(b.qkv, b.ao, b.lse, B, N, e->H, e->scale, s)) return rc;
    } else {
      if (int rc = attn_fwd(b.qkv, b.ao, b.lse, nullptr, B, N, T, e->H, e->scale, s)) return rc;
    }
    const int R = cls ? B : T;
    const int sD = cls ? N * D : D, sH = cls ? N * Hd : Hd;
    const int rps = cls ? 1 : N;   // rows per image: the scale of drop path is one per image
    // projection (+bias, LayerScale, residual) and LayerNorm 2 in one launch
    if (int rc = gemm_resid_ln(b.ao, b.wproj, R, D, D, sD, D, x_mid, b.bproj, b.g1, x_in, sD, b.ln2w, b.ln2b, ln_out, sD,
                               e->eps, s, -1, drop_path_scale(e, l, 0), rps))
      return rc;
    if (int rc = gemm_tn(EPI_BIAS_GELU_D, ln_out, b.wfc1, R, Hd, D, sD, D, b.hpre, gelu_out, b.bfc1, nullptr, nullptr, sH, s, 0))
      return rc;
    if (l + 1 < L) {
      // fc2 (+bias, LayerScale, residual) and the NEXT block's LayerNorm 1 in one launch
      const BlockPtrs& nb = e->blk[l + 1];
      if (int rc = gemm_resid_ln(gelu_out, b.wfc2, R, D, Hd, sH, Hd, x_out, b.bfc2, b.g2, x_mid, sD, nb.ln1w, nb.ln1b, ln_out,
                                 sD, e->eps, s, -1, drop_path_scale(e, l, 1), rps))
        return rc;
    } else if (const float* dp = drop_path_scale(e, l, 1)) {
      if (int rc = gemm_resid_scaled(gelu_out, b.wfc2, R, D, Hd, sH, Hd, x_out, b.bfc2, b.g2, x_mid, sD, dp, rps, s))
        return rc;
    } else {
      if (int rc = gemm_tn(EPI_RESID, gelu_out, b.wfc2, R, D, Hd, sH, Hd, x_out, nullptr, b.bfc2, b.g2, x_mid, sD, s, 0))
        return rc;
    }
  }

  // ---- final norm on the CLS rows only (vit.py:417-419), head, loss ----
  const float* x_fin = xs + size_t(2 * L) * TD;
  if (int rc = layernorm_fwd(x_fin, int64_t(N) * D, e->get<float>("lnfw"), e->get<float>("lnfb"), e->get<void>("cls_ln"),
                             D, B, D, e->eps, s))
    return rc;
  if (int rc = head_fwd(e->get<void>("cls_ln"), params + ar.fcw, params + ar.fcb, e->get<float>("logits"), B, D, e->C, s))
    return rc;
  if (labels || targets) {
    APLA_CUDA(cudaMemsetAsync(e->get<float>("loss"), 0, sizeof(float), s));
    if (labels) {
      if (int rc = cross_entropy(e->get<float>("logits"), labels, e->get<float>("dlogits"), e->get<float>("loss"), B, e->C,
                                 grad_scale, loss_scale, s))
        return rc;
    } else if (e->criterion == 1) {
      if (int rc = bce_with_logits(e->get<float>("logits"), targets, e->get<float>("dlogits"), e->get<float>("loss"), B,
                                   e->C, grad_scale, loss_scale, s))
        return rc;
    } else {
      if (int rc = cross_entropy_soft(e->get<float>("logits"), targets, e->get<float>("dlogits"), e->get<float>("loss"), B,
                                      e->C, grad_scale, loss_scale, s))
        return rc;
    }
  }
  return 0;
}

static int check_infer_ready(Engine* e, int n_img) {
  APLA_CHECK(e->infer_cap > 0, "apla_engine_infer: no evaluation workspace (option 'infer_batch' is 0)");
  APLA_CHECK(n_img >= 1 && n_img <= e->infer_cap, "apla_engine_infer: n_img=%d outside [1, %d]", n_img, e->infer_cap);
  for (const char* n : kInferNames)
    APLA_CHECK(e->g.count(n) && e->g[n] != nullptr, "apla_engine_infer: workspace '%s' was not set", n);
  for (const char* n : {"wpe", "bpe", "cls", "pos", "lnfw", "lnfb", "params"})
    APLA_CHECK(e->g.count(n) && e->g[n] != nullptr, "apla_engine_infer: buffer '%s' was not set", n);
  for (int l = 0; l < e->L; ++l) {
    const BlockPtrs& b = e->blk[l];
    APLA_CHECK(b.wqkv && b.wfc1 && b.wfc2 && b.wproj && b.bproj && b.bfc1 && b.bfc2 && b.ln1w && b.ln1b && b.ln2w && b.ln2b,
               "apla_engine_infer: block %d has unset weights", l);
  }
  return 0;
}

// Classifier.forward (models.py:81-92) for n_img images with the engine's current weights, in the launch sequence of
// engine_forward (same kernels, same gemm_resid_ln pairing, same CLS-only last block), but over its own workspace and
// with the forward-only fc1 epilogue: nothing is kept for a backward pass.  With cls_probs set it stops after the last
// block's attention and writes that attention's CLS-query probabilities cls_probs_f32[n_img, H, N] instead of logits.
static int engine_infer(Engine* e, const float* images, int n_img, float* logits, void* emb, cudaStream_t s,
                        float* cls_probs = nullptr) {
  if (int rc = check_infer_ready(e, n_img)) return rc;
  const int B = n_img, N = e->N, D = e->D, L = e->L, Hd = e->hidden, T = B * N;
  float* xa = e->get<float>("infer_x");                       // block input, then block output
  float* xb = xa + size_t(e->infer_cap) * N * D;              // after the attention branch
  void* ln = e->get<void>("infer_ln");
  void* qkv = e->get<void>("infer_qkv");
  void* ao = e->get<void>("infer_ao");
  float* lse = e->get<float>("infer_lse");
  void* gelu = e->get<void>("infer_gelu");
  void* patches = e->get<void>("infer_patches");
  void* pe_out = e->get<void>("infer_pe_out");
  void* cls_ln = emb ? emb : e->get<void>("infer_cls_ln");
  const Arena ar = arena_of(e);
  const float* params = e->get<float>("params");

  if (int rc = patchify(images, patches, B, e->img, e->patch, e->kpad, s)) return rc;
  if (int rc = gemm_tn(EPI_BIAS, patches, e->get<void>("wpe"), B * e->P, D, e->kpad, e->kpad, e->kpad, pe_out, nullptr,
                       e->get<float>("bpe"), nullptr, nullptr, D, s, 0))
    return rc;
  if (int rc = assemble_tokens(pe_out, e->get<float>("cls"), e->get<float>("pos"), xa, B, e->P, D, s)) return rc;
  for (int l = 0; l < L; ++l) {
    const BlockPtrs& b = e->blk[l];
    if (l == 0) {
      if (int rc = layernorm_fwd(xa, D, b.ln1w, b.ln1b, ln, D, T, D, e->eps, s)) return rc;
    }
    if (int rc = gemm_tn(EPI_BIAS, ln, b.wqkv, T, 3 * D, D, D, D, qkv, nullptr, b.bqkv, nullptr, nullptr, 3 * D, s, 0))
      return rc;
    const bool cls = e->cls_last && l == L - 1;
    if (cls && e->cls_last >= 2) {
      if (int rc = attn_cls_fwd(qkv, ao, lse, B, N, e->H, e->scale, s)) return rc;
    } else {
      if (int rc = attn_fwd(qkv, ao, lse, nullptr, B, N, T, e->H, e->scale, s)) return rc;
    }
    if (cls_probs && l == L - 1) return attn_probs(qkv, lse, cls_probs, B, N, e->H, 1, e->scale, s);
    const int R = cls ? B : T;
    const int sD = cls ? N * D : D, sH = cls ? N * Hd : Hd;
    if (int rc = gemm_resid_ln(ao, b.wproj, R, D, D, sD, D, xb, b.bproj, b.g1, xa, sD, b.ln2w, b.ln2b, ln, sD, e->eps, s))
      return rc;
    if (int rc = gemm_tn(EPI_BIAS_GELU_G, ln, b.wfc1, R, Hd, D, sD, D, gelu, nullptr, b.bfc1, nullptr, nullptr, sH, s, 0))
      return rc;
    if (l + 1 < L) {
      const BlockPtrs& nb = e->blk[l + 1];
      if (int rc = gemm_resid_ln(gelu, b.wfc2, R, D, Hd, sH, Hd, xa, b.bfc2, b.g2, xb, sD, nb.ln1w, nb.ln1b, ln, sD, e->eps, s))
        return rc;
    } else {
      if (int rc = gemm_tn(EPI_RESID, gelu, b.wfc2, R, D, Hd, sH, Hd, xa, nullptr, b.bfc2, b.g2, xb, sD, s, 0)) return rc;
    }
  }
  if (int rc = layernorm_fwd(xa, int64_t(N) * D, e->get<float>("lnfw"), e->get<float>("lnfb"), cls_ln, D, B, D, e->eps, s))
    return rc;
  return head_fwd(cls_ln, params + ar.fcw, params + ar.fcb, logits, B, D, e->C, s);
}

static int engine_backward(Engine* e, int l_from, int l_to, cudaStream_t s) {
  if (int rc = check_ready(e)) return rc;
  // rows of the last forward (n_cur images); the xs checkpoints and the two dsub slots keep their capacity strides
  const int D = e->D, B = e->n_cur, N = e->N, L = e->L, Hd = e->hidden, r = e->r, T = B * N;
  const size_t TD = size_t(e->T()) * D, Tn_D = size_t(T) * D;
  float* xs = e->get<float>("xs");
  void* dln = e->get<void>("ln_out");      // reused: gradient w.r.t. a LayerNorm output
  void* dH = e->get<void>("gelu_out");     // reused: gradient w.r.t. the fc1 pre-activation
  float* dx = e->get<float>("dx");
  void* dxb = e->get<void>("dxb");
  char* dsub0 = e->full_rows ? nullptr : e->get<char>("dsub");
  const size_t dsub_slot = size_t(e->T()) * e->r_pad * 2, dsub_bytes = size_t(T) * e->r_pad * 2;
  const bool side = e->side_wgrad >= 2 || (e->side_wgrad >= 1 && e->full_rows);
  if (side) {
    if (int rc = e->side_ready()) return rc;
  }
  const int* idx = e->get<int>("idx");
  const int* rowmap = e->full_rows ? e->get<int>("rowmap") : nullptr;
  const Arena ar = arena_of(e);
  float* params = e->get<float>("params");
  float* grads = e->get<float>("grads");

  APLA_CHECK(0 <= l_to && l_to <= l_from && l_from < L, "engine_backward: bad block range [%d..%d]", l_from, l_to);
  if (l_from == L - 1) {
  APLA_CUDA(cudaMemsetAsync(grads, 0, size_t(ar.n) * sizeof(float), s));
  // head: dW, db, and the gradient of the normalised CLS token
  if (int rc = head_bwd(e->get<float>("dlogits"), e->get<void>("cls_ln"), params + ar.fcw, grads + ar.fcw, grads + ar.fcb,
                        e->get<void>("dcls"), B, D, e->C, s))
    return rc;
  // final norm backward: only CLS rows carry gradient; everything else in dx / dxb is zero
  APLA_CUDA(cudaMemsetAsync(dx, 0, Tn_D * sizeof(float), s));
  APLA_CUDA(cudaMemsetAsync(dxb, 0, Tn_D * 2, s));
  if (int rc = layernorm_bwd(e->get<void>("dcls"), D, xs + size_t(2 * L) * TD, int64_t(N) * D, e->get<float>("lnfw"),
                             nullptr, 0, dx, int64_t(N) * D, dxb, int64_t(N) * D, e->blk[L - 1].g2, nullptr, 0, nullptr, 0,
                             0, B, D, e->eps, s, drop_path_scale(e, L - 1, 1), 1))
    return rc;
  }

  for (int l = l_from; l >= l_to; --l) {
    const BlockPtrs& b = e->blk[l];
    const float* x_in = xs + size_t(2 * l) * TD;
    const float* x_mid = xs + size_t(2 * l + 1) * TD;
    // MLP branch: dxb holds bf16(s[l,1] * gamma2 * dx_out); hpre holds gelu'(fc1 pre-activation) in fp16.  In the last block only
    // the CLS rows of dx_out are non-zero (see Engine::cls_last): its MLP input gradients and LayerNorm-2 backward run on
    // those B rows; dx / dxb / dsub of all other rows stay the zeros they were initialised with.
    const bool cls = e->cls_last && l == L - 1;
    const int R = cls ? B : T;
    const int sD = cls ? N * D : D, sH = cls ? N * Hd : Hd;
    if (int rc = gemm_tn(EPI_MUL_F16, dxb, b.wfc2T, R, Hd, D, sD, D, dH, nullptr, nullptr, nullptr, b.hpre, sH, s, 0))
      return rc;
    if (int rc = gemm_tn(EPI_BIAS, dH, b.wfc1T, R, D, Hd, sH, Hd, dln, nullptr, nullptr, nullptr, nullptr, sD, s, 0))
      return rc;
    // dsub alternates between two slots when the weight gradient runs beside the main chain: block l's LayerNorm-2
    // backward may only overwrite the slot after block l+2's weight gradient has read it
    void* dsub = dsub0 ? dsub0 + ((side && (l & 1)) ? dsub_slot : 0) : nullptr;
    if (side && dsub && l + 2 <= l_from) APLA_CUDA(cudaStreamWaitEvent(s, e->ev_done[l + 2], 0));
    if (cls && dsub) APLA_CUDA(cudaMemsetAsync(dsub, 0, dsub_bytes, s));
    // dx_mid = dx_out + LN2'(dln); dxb = bf16(s[l,0] * gamma1 * dx_mid); dsub = its APLA columns
    if (int rc = layernorm_bwd(dln, sD, x_mid, sD, b.ln2w, dx, sD, dx, sD, dxb, sD, b.g1, dsub,
                               cls ? int64_t(N) * e->r_pad : e->r_pad, idx + size_t(l) * r, r, e->r_pad, R, D, e->eps, s,
                               drop_path_scale(e, l, 0), cls ? 1 : N))
      return rc;
    // APLA weight gradient: only the trainable rows of the projection (appla_attn.py:64,70-74)
    float* dW1 = grads + ar.w1 + size_t(l) * r * D;
    float* db1 = grads + ar.b1 + size_t(l) * r;
    cudaStream_t ws = s;
    if (side) {
      ws = e->side;
      APLA_CUDA(cudaEventRecord(e->ev_fork[l], s));
      APLA_CUDA(cudaStreamWaitEvent(ws, e->ev_fork[l], 0));
    }
    if (e->full_rows) {
      if (int rc = gemm_wgrad_nt(b.ao, dxb, D, D, T, D, D, dW1, D, rowmap + size_t(l) * D, D, ws)) return rc;
      if (int rc = colsum(dxb, D, T, D, db1, rowmap + size_t(l) * D, ws)) return rc;
    } else {
      if (int rc = gemm_wgrad_nt(b.ao, dsub, D, e->r_pad, T, D, e->r_pad, dW1, D, nullptr, r, ws)) return rc;
      if (int rc = colsum(dsub, e->r_pad, T, r, db1, nullptr, ws)) return rc;
    }
    if (side) APLA_CUDA(cudaEventRecord(e->ev_done[l], ws));
    if (l == 0) break;  // nothing trainable upstream of block 0's attention
    void* dO = e->get<void>("dO");
    if (cls && e->cls_last >= 2) {
      // last block: dO and dQ exist for the CLS rows only; dK / dV of every key come from that one row
      if (int rc = gemm_tn(EPI_BIAS, dxb, b.wprojT, B, D, D, N * D, D, dO, nullptr, nullptr, nullptr, nullptr, N * D, s, 0))
        return rc;
      if (int rc = attn_cls_bwd(b.qkv, b.ao, dO, b.lse, e->get<void>("dqkv"), B, N, e->H, e->scale, s)) return rc;
    } else {
      // dO = dY Wproj, and delta = rowsum(dO * O) per (token, head) from the same epilogue
      if (int rc = gemm_tn(EPI_DELTA, dxb, b.wprojT, T, D, D, D, D, dO, e->get<float>("delta"), nullptr, nullptr, b.ao, D, s, 0))
        return rc;
      if (int rc = attn_bwd(b.qkv, nullptr, dO, b.lse, e->get<float>("delta"), e->get<void>("dqkv"), nullptr, B, N, T, e->H,
                            e->scale, s))
        return rc;
    }
    if (int rc = gemm_tn(EPI_BIAS, e->get<void>("dqkv"), b.wqkvT, T, D, 3 * D, 3 * D, 3 * D, dln, nullptr, nullptr, nullptr,
                         nullptr, D, s, 0))
      return rc;
    if (side && e->full_rows) APLA_CUDA(cudaStreamWaitEvent(s, e->ev_done[l], 0));   // its weight gradient reads dxb
    // dx_in = dx_mid + LN1'(dln); dxb = bf16(s[l-1,1] * gamma2[l-1] * dx_in) feeds block l-1's MLP branch
    if (int rc = layernorm_bwd(dln, D, x_in, D, b.ln1w, dx, D, dx, D, dxb, D, e->blk[l - 1].g2, nullptr, 0, nullptr, 0, 0,
                               T, D, e->eps, s, drop_path_scale(e, l - 1, 1), N))
      return rc;
  }
  // join: the side stream is serial, so the last block's event covers every weight gradient of this range
  if (side) APLA_CUDA(cudaStreamWaitEvent(s, e->ev_done[l_to], 0));
  return 0;
}

static int engine_optim(Engine* e, float gscale, float max_norm, float lr, float wd, float b1, float b2, float eps,
                        int step, cudaStream_t s) {
  if (int rc = check_ready(e)) return rc;
  const Arena ar = arena_of(e);
  float* params = e->get<float>("params");
  float* grads = e->get<float>("grads");
  float* sumsq = e->get<float>("sumsq");
  if (int rc = grad_sumsq(grads, ar.n, gscale, sumsq, s)) return rc;
  if (int rc = adamw_step(params, grads, e->get<float>("exp_avg"), e->get<float>("exp_avg_sq"), ar.n, ar.n_decay, sumsq,
                          gscale, max_norm, lr, wd, b1, b2, eps, step, s, e->get<float>("hyper")))
    return rc;
  // refresh the dense bf16 projection copies from the updated fp32 rows: one launch when the host laid the per-block
  // copies out back to back (apla_b200/engine.py does), one launch per block otherwise
  const int L = e->L, r = e->r, D = e->D;
  bool packed = true;
  for (int l = 1; l < L; ++l) {
    packed = packed && reinterpret_cast<char*>(e->blk[l].wproj) == reinterpret_cast<char*>(e->blk[0].wproj) + size_t(l) * D * D * 2 &&
             reinterpret_cast<char*>(e->blk[l].wprojT) == reinterpret_cast<char*>(e->blk[0].wprojT) + size_t(l) * D * D * 2 &&
             e->blk[l].bproj == e->blk[0].bproj + size_t(l) * D;
  }
  if (packed)
    return proj_refresh(params + ar.w1, params + ar.b1, e->get<int>("idx"), e->blk[0].wproj, e->blk[0].wprojT,
                        e->blk[0].bproj, L, r, D, int64_t(r) * D, r, s);
  for (int l = 0; l < L; ++l) {
    if (int rc = proj_refresh(params + ar.w1 + size_t(l) * r * D, params + ar.b1 + size_t(l) * r,
                              e->get<int>("idx") + size_t(l) * r, e->blk[l].wproj, e->blk[l].wprojT, e->blk[l].bproj, 1, r,
                              D, 0, 0, s))
      return rc;
  }
  return 0;
}

}  // namespace apla

using namespace apla;

extern "C" {

apla_engine_t apla_engine_create(int B, int N, int D, int H, int L, int hidden, int C, int patch, int img, int kpad, int r,
                                 int r_pad, int full_rows, float eps, float scale) {
  if (B <= 0 || N <= 1 || D % 128 != 0 || H * 64 != D || L <= 0 || hidden % 32 != 0 || C <= 0 || r <= 0 || r > D ||
      img % patch != 0 || (img / patch) * (img / patch) + 1 != N || kpad % 8 != 0 || kpad < 3 * patch * patch ||
      (!full_rows && (r_pad % 64 != 0 || r_pad < r))) {
    set_error("apla_engine_create: invalid configuration (B=%d N=%d D=%d H=%d L=%d hidden=%d C=%d patch=%d img=%d kpad=%d "
              "r=%d r_pad=%d full_rows=%d)", B, N, D, H, L, hidden, C, patch, img, kpad, r, r_pad, full_rows);
    return nullptr;
  }
  Engine* e = new Engine();
  e->B = B; e->N = N; e->D = D; e->H = H; e->L = L; e->hidden = hidden; e->C = C; e->P = N - 1; e->patch = patch;
  e->img = img; e->kpad = kpad; e->r = r; e->r_pad = r_pad; e->full_rows = full_rows; e->eps = eps; e->scale = scale;
  e->n_cur = B;
  e->blk.resize(L);
  return e;
}

void apla_engine_destroy(apla_engine_t h) { delete reinterpret_cast<Engine*>(h); }

/* block < 0: global buffer `name`; otherwise per-block pointer `name` of block `block`. */
int apla_engine_set_ptr(apla_engine_t h, const char* name, int block, void* p) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && name != nullptr, "apla_engine_set_ptr: null handle or name");
  const std::string n(name);
  if (block < 0) {
    bool known = false;
    for (const char* k : kGlobalNames) known |= (n == k);
    for (const char* k : kOptionalNames) known |= (n == k);
    for (const char* k : kInferNames) known |= (n == k);
    APLA_CHECK(known, "apla_engine_set_ptr: unknown global buffer '%s'", name);
    e->g[n] = p;
    return 0;
  }
  APLA_CHECK(block < e->L, "apla_engine_set_ptr: block %d out of range", block);
  BlockPtrs& b = e->blk[block];
#define SETP(field)                                              \
  if (n == #field) {                                             \
    b.field = reinterpret_cast<decltype(b.field)>(p);            \
    return 0;                                                    \
  }
  SETP(wqkv) SETP(wqkvT) SETP(wfc1) SETP(wfc1T) SETP(wfc2) SETP(wfc2T) SETP(wproj) SETP(wprojT) SETP(bqkv) SETP(bfc1)
  SETP(bfc2) SETP(ln1w) SETP(ln1b) SETP(ln2w) SETP(ln2b) SETP(g1) SETP(g2) SETP(bproj) SETP(qkv) SETP(ao) SETP(hpre)
  SETP(lse)
#undef SETP
  set_error("apla_engine_set_ptr: unknown block pointer '%s'", name);
  return 1;
}

int apla_engine_set_option(apla_engine_t h, const char* name, int value) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && name != nullptr, "apla_engine_set_option: null handle or name");
  if (std::string(name) == "cls_only_last_block") {
    e->cls_last = value < 0 ? 0 : (value > 2 ? 2 : value);
    return 0;
  }
  if (std::string(name) == "infer_batch") {   // capacity of the evaluation workspace in images (0 = none)
    APLA_CHECK(value >= 0, "apla_engine_set_option: infer_batch=%d is negative", value);
    e->infer_cap = value;
    return 0;
  }
  if (std::string(name) == "side_wgrad") {   // 0 = off, 1 = on for partial_size == dim, 2 = on, "dsub" holds two slots
    e->side_wgrad = value < 0 ? 0 : (value > 2 ? 2 : value);
    return 0;
  }
  if (std::string(name) == "criterion") {   // 0 = cross-entropy, 1 = BCE-with-logits
    APLA_CHECK(value == 0 || value == 1,
               "apla_engine_set_option: criterion=%d is neither 0 (cross-entropy) nor 1 (BCE-with-logits)", value);
    e->criterion = value;
    return 0;
  }
  set_error("apla_engine_set_option: unknown option '%s'", name);
  return 1;
}

int64_t apla_engine_arena_size(apla_engine_t h) {
  Engine* e = reinterpret_cast<Engine*>(h);
  return e ? arena_of(e).n : -1;
}
int64_t apla_engine_arena_decay_size(apla_engine_t h) {
  Engine* e = reinterpret_cast<Engine*>(h);
  return e ? arena_of(e).n_decay : -1;
}

int apla_engine_forward(apla_engine_t h, const float* images, const int64_t* labels, float loss_scale, float grad_scale,
                        apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && images != nullptr, "apla_engine_forward: null handle or images");
  return engine_forward(e, images, e->B, labels, nullptr, loss_scale, grad_scale, reinterpret_cast<cudaStream_t>(stream));
}
int apla_engine_forward_n(apla_engine_t h, const float* images, int n_img, const int64_t* labels, const float* targets,
                          float loss_scale, float grad_scale, apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && images != nullptr, "apla_engine_forward_n: null handle or images");
  return engine_forward(e, images, n_img, labels, targets, loss_scale, grad_scale, reinterpret_cast<cudaStream_t>(stream));
}
int apla_engine_infer(apla_engine_t h, const float* images, int n_img, float* logits, void* emb, apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && images != nullptr && logits != nullptr, "apla_engine_infer: null handle, images or logits");
  return engine_infer(e, images, n_img, logits, emb, reinterpret_cast<cudaStream_t>(stream));
}
int apla_engine_cls_attention(apla_engine_t h, const float* images, int n_img, float* probs, apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr && images != nullptr && probs != nullptr,
             "apla_engine_cls_attention: null handle, images or probs");
  return engine_infer(e, images, n_img, nullptr, nullptr, reinterpret_cast<cudaStream_t>(stream), probs);
}
int apla_engine_backward(apla_engine_t h, int block_from, int block_to, apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr, "apla_engine_backward: null handle");
  return engine_backward(e, block_from, block_to, reinterpret_cast<cudaStream_t>(stream));
}
int apla_engine_optim(apla_engine_t h, float gscale, float max_norm, float lr, float wd, float beta1, float beta2,
                      float eps, int step, apla_stream_t stream) {
  Engine* e = reinterpret_cast<Engine*>(h);
  APLA_CHECK(e != nullptr, "apla_engine_optim: null handle");
  return engine_optim(e, gscale, max_norm, lr, wd, beta1, beta2, eps, step, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
