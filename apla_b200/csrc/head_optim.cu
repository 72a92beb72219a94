// Step tail: classifier head (Classifier.fc, src/defaults/models.py:87), CrossEntropyLoss(mean)
// (src/defaults/wrappers.py:314), and the optimiser tail of Trainer.global_step (src/defaults/trainer.py:133-138):
// clip_grad_norm_(1.0) + AdamW over ONE contiguous fp32 arena of all trainable tensors, followed by the refresh of
// the bf16 working copies of the projection (trainable rows scattered back to their index positions,
// src/apla/appla_attn.py:64-79).  All tiny next to the block GEMMs; written for few launches, not peak rates.
#include "common.cuh"
#include "ptx.cuh"

namespace apla {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// logits[b,c] = sum_d xn[b,d] * W[c,d] + bias[c]   (xn bf16 = LayerNorm output of the CLS token)
__global__ void head_fwd_kernel(const __nv_bfloat16* __restrict__ xn, const float* __restrict__ W,
                                const float* __restrict__ bias, float* __restrict__ logits, int B, int D, int C) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= B * C) return;
  const int b = gw / C, c = gw % C;
  float acc = 0.f;
  for (int d = lane; d < D; d += 32) acc += __bfloat162float(xn[size_t(b) * D + d]) * __ldg(W + size_t(c) * D + d);
  acc = warp_sum(acc);
  if (lane == 0) logits[gw] = acc + bias[c];
}

// per row: loss_b = logsumexp - logit[label]; dlogits = (softmax - onehot) * grad_scale; loss += loss_b * loss_scale
__global__ void ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                          float* __restrict__ dlogits, float* __restrict__ loss, int C, float grad_scale,
                          float loss_scale) {
  const int b = blockIdx.x;
  const float* lr = logits + size_t(b) * C;
  __shared__ float red[32];
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) mx = fmaxf(mx, lr[c]);
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < (blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) s += expf(lr[c] - mx);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  s = 0.f;
  for (int i = 0; i < (blockDim.x >> 5); ++i) s += red[i];
  const float lse = mx + logf(s);
  const int y = (int)labels[b];
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    dlogits[size_t(b) * C + c] = (expf(lr[c] - lse) - (c == y ? 1.f : 0.f)) * grad_scale;
  if (threadIdx.x == 0) atomicAdd(loss, (lse - lr[y]) * loss_scale);
}

// Probability targets t[b, :] (F.cross_entropy(z, t) with fp32 [B, C] targets: mixup / cutmix / label smoothing), neither
// normalised nor validated, as torch does neither:  loss_b = tsum lse - tz with tsum = sum_c t_c, tz = sum_c t_c z_c;
// dlogits = (tsum softmax - t) * grad_scale.  The max / exponential-sum passes and the block reductions are ce_kernel's,
// with tsum and tz reduced beside the sum: for a one-hot row tsum == 1.0f and every zero term adds exactly, so lse, the
// row loss and (1.0f * p - t) * grad_scale are ce_kernel's bit for bit.
__global__ void ce_soft_kernel(const float* __restrict__ logits, const float* __restrict__ targets,
                               float* __restrict__ dlogits, float* __restrict__ loss, int C, float grad_scale,
                               float loss_scale) {
  const int b = blockIdx.x;
  const float* lr = logits + size_t(b) * C;
  const float* tr = targets + size_t(b) * C;
  __shared__ float red[32], red_t[32], red_tz[32];
  float mx = -INFINITY;
  for (int c = threadIdx.x; c < C; c += blockDim.x) mx = fmaxf(mx, lr[c]);
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < (blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float s = 0.f, ts = 0.f, tz = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float z = lr[c], t = tr[c];
    s += expf(z - mx);
    ts += t;
    tz += t * z;
  }
  s = warp_sum(s);
  ts = warp_sum(ts);
  tz = warp_sum(tz);
  if ((threadIdx.x & 31) == 0) {
    red[threadIdx.x >> 5] = s;
    red_t[threadIdx.x >> 5] = ts;
    red_tz[threadIdx.x >> 5] = tz;
  }
  __syncthreads();
  s = 0.f;
  ts = 0.f;
  tz = 0.f;
  for (int i = 0; i < (blockDim.x >> 5); ++i) {
    s += red[i];
    ts += red_t[i];
    tz += red_tz[i];
  }
  const float lse = mx + logf(s);
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    dlogits[size_t(b) * C + c] = (ts * expf(lr[c] - lse) - tr[c]) * grad_scale;
  if (threadIdx.x == 0) atomicAdd(loss, (ts * lse - tz) * loss_scale);
}

// BCEWithLogitsLoss (pos_weight 1) of one element in fp32, finite for every finite z: with e = exp(-|z|) <= 1,
// l = max(z, 0) - z t + log1p(e) and sigma(z) = 1 / (1 + e) for z >= 0, e / (1 + e) otherwise.
__device__ __forceinline__ float bce_term(float z, float t, float& sig) {
  const float e = expf(-fabsf(z));
  const float inv = 1.f / (1.f + e);
  sig = z >= 0.f ? inv : e * inv;
  return fmaxf(z, 0.f) - z * t + log1pf(e);
}

// Multi-label targets t[b, :] (nn.BCEWithLogitsLoss, wrappers.py:310-320), neither clamped nor checked, as torch does
// neither: per row, loss += loss_scale * sum_c l(z, t); dlogits = (sigma(z) - t) * grad_scale.  One CTA per row with the
// block reduction of ce_kernel, one atomicAdd per row.
__global__ void bce_kernel(const float* __restrict__ logits, const float* __restrict__ targets,
                           float* __restrict__ dlogits, float* __restrict__ loss, int C, float grad_scale,
                           float loss_scale) {
  const int b = blockIdx.x;
  const float* lr = logits + size_t(b) * C;
  const float* tr = targets + size_t(b) * C;
  __shared__ float red[32];
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float t = tr[c];
    float sig;
    s += bce_term(lr[c], t, sig);
    dlogits[size_t(b) * C + c] = (sig - t) * grad_scale;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    s = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) s += red[i];
    atomicAdd(loss, s * loss_scale);
  }
}

// Evaluation sums over one batch, one CTA: acc[0] += sum_b CE_b (the row softmax of ce_kernel, one warp per row),
// acc[1] += #{b : argmax_c logits[b,c] == labels[b]} with the first maximum winning, as torch.argmax picks it.  Each warp
// walks its rows in order and the warps' partial sums are added in warp order: the result does not depend on timing.
// A label outside [0, C) makes the loss NaN rather than reading outside the row.
constexpr int kEvalThreads = 512;
__global__ void __launch_bounds__(kEvalThreads) eval_acc_kernel(const float* __restrict__ logits,
                                                               const int64_t* __restrict__ labels, int B, int C,
                                                               float* __restrict__ acc) {
  constexpr int kWarps = kEvalThreads / 32;
  __shared__ float ce_w[kWarps], hit_w[kWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float ce_sum = 0.f, hits = 0.f;
  for (int b = warp; b < B; b += kWarps) {
    const float* lr = logits + size_t(b) * C;
    float mx = -INFINITY;
    int arg = C;
    for (int c = lane; c < C; c += 32) {
      const float v = lr[c];
      if (v > mx || arg == C) { mx = v; arg = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, mx, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
    }
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += expf(lr[c] - mx);
    s = warp_sum(s);
    const int64_t y = labels[b];
    const bool valid = y >= 0 && y < C;
    const float lse = mx + logf(s);
    ce_sum += valid ? lse - lr[valid ? y : 0] : NAN;
    hits += (valid && arg == int(y)) ? 1.f : 0.f;
  }
  if (lane == 0) {
    ce_w[warp] = ce_sum;
    hit_w[warp] = hits;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, h = 0.f;
    for (int w = 0; w < kWarps; ++w) {
      a += ce_w[w];
      h += hit_w[w];
    }
    acc[0] += a;
    acc[1] += h;
  }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Multi-label evaluation sums over one batch of n = B*C elements, one CTA: acc[0] += sum l (bce_term),
// acc[1] += #{(b, c) : (z > 0) == (t >= 0.5)}.  The accumulator is double: a validation set's element count passes 2^24,
// beyond which an fp32 counter stops counting.  Each thread walks its elements in order and sums in double, the warps
// reduce in a fixed shuffle pattern and thread 0 adds the warps in warp order: the result does not depend on timing.
__global__ void __launch_bounds__(kEvalThreads) eval_acc_bce_kernel(const float* __restrict__ logits,
                                                                   const float* __restrict__ targets, int64_t n,
                                                                   double* __restrict__ acc) {
  constexpr int kWarps = kEvalThreads / 32;
  __shared__ double l_w[kWarps], hit_w[kWarps];
  double l_sum = 0.0;
  int64_t hits = 0;
  for (int64_t i = threadIdx.x; i < n; i += kEvalThreads) {
    const float z = logits[i], t = targets[i];
    float sig;
    l_sum += double(bce_term(z, t, sig));
    hits += (z > 0.f) == (t >= 0.5f);
  }
  l_sum = warp_sum_d(l_sum);
  double h = warp_sum_d(double(hits));
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    l_w[warp] = l_sum;
    hit_w[warp] = h;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0;
    h = 0.0;
    for (int w = 0; w < kWarps; ++w) {
      a += l_w[w];
      h += hit_w[w];
    }
    acc[0] += a;
    acc[1] += h;
  }
}

// dW[c,d] = sum_b dlogits[b,c] * xn[b,d] ; db[c] = sum_b dlogits[b,c]
__global__ void head_wgrad_kernel(const float* __restrict__ dlogits, const __nv_bfloat16* __restrict__ xn,
                                  float* __restrict__ dW, float* __restrict__ db, int B, int D, int C) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * D) return;
  const int c = i / D, d = i % D;
  float acc = 0.f, accb = 0.f;
  for (int b = 0; b < B; ++b) {
    const float g = __ldg(dlogits + size_t(b) * C + c);
    acc += g * __bfloat162float(xn[size_t(b) * D + d]);
    accb += g;
  }
  dW[i] = acc;
  if (d == 0) db[c] = accb;
}

// dxn[b,d] = sum_c dlogits[b,c] * W[c,d]  -> bf16 (gradient w.r.t. the final LayerNorm output)
// One block per (64-column slice of d, image b): 4 groups of 64 threads split the classes, 8 independent loads in
// flight per thread (the first version ran one 555-step dependent loop per output and took 80 us).
__global__ void __launch_bounds__(256)
head_dgrad_kernel(const float* __restrict__ dlogits, const float* __restrict__ W, __nv_bfloat16* __restrict__ dxn, int B,
                  int D, int C) {
  __shared__ float red[4][64];
  const int b = blockIdx.y, d = blockIdx.x * 64 + (threadIdx.x & 63), part = threadIdx.x >> 6;
  const float* dl = dlogits + size_t(b) * C;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (d < D) {
    int c = part;
    for (; c + 28 < C; c += 32) {
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] = fmaf(__ldg(dl + c + 4 * u), __ldg(W + size_t(c + 4 * u) * D + d), acc[u]);
    }
    for (; c < C; c += 4) acc[0] = fmaf(__ldg(dl + c), __ldg(W + size_t(c) * D + d), acc[0]);
  }
  red[part][threadIdx.x & 63] = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
  __syncthreads();
  if (part == 0 && d < D)
    dxn[size_t(b) * D + d] = __float2bfloat16_rn((red[0][threadIdx.x] + red[1][threadIdx.x]) + (red[2][threadIdx.x] + red[3][threadIdx.x]));
}

// ---- second-generation head kernels: the first ones re-read the whole weight matrix per image (109 MB of L2 traffic for
// a 27 MFLOP product) and took 36 + 50 us of an 8.2 ms step; these keep the reused operand in shared memory: 9.5 + ~20 us.
// (A one-warp-per-class forward with the weight row in registers was 10x SLOWER than head_fwd_kernel -- four warps per SM
// cannot hide the load latency -- and was dropped.)

// dW tile of 32 classes x 64 features per block, the two operand tiles of 64 images staged in shared memory
__global__ void __launch_bounds__(256)
head_wgrad2_kernel(const float* __restrict__ dlogits, const __nv_bfloat16* __restrict__ xn, float* __restrict__ dW,
                   float* __restrict__ db, int B, int D, int C) {
  __shared__ float sdl[64][32];
  __shared__ __align__(16) float sxn[64][64];
  const int c_tile = blockIdx.x * 32, d_tile = blockIdx.y * 64;
  const int tc = threadIdx.x >> 4, td = threadIdx.x & 15;       // 2 classes x 4 features per thread
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  float accb[2] = {0.f, 0.f};
  for (int b0 = 0; b0 < B; b0 += 64) {
    for (int i = threadIdx.x; i < 64 * 32; i += 256) {
      const int b = i >> 5, c = i & 31;
      sdl[b][c] = (b0 + b < B && c_tile + c < C) ? __ldg(dlogits + size_t(b0 + b) * C + c_tile + c) : 0.f;
    }
    for (int i = threadIdx.x; i < 64 * 64; i += 256) {
      const int b = i >> 6, d = i & 63;
      sxn[b][d] = (b0 + b < B && d_tile + d < D) ? __bfloat162float(xn[size_t(b0 + b) * D + d_tile + d]) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int b = 0; b < 64; ++b) {
      const float g0 = sdl[b][2 * tc], g1 = sdl[b][2 * tc + 1];
      const float4 x = *reinterpret_cast<const float4*>(&sxn[b][4 * td]);
      acc[0][0] = fmaf(g0, x.x, acc[0][0]); acc[0][1] = fmaf(g0, x.y, acc[0][1]);
      acc[0][2] = fmaf(g0, x.z, acc[0][2]); acc[0][3] = fmaf(g0, x.w, acc[0][3]);
      acc[1][0] = fmaf(g1, x.x, acc[1][0]); acc[1][1] = fmaf(g1, x.y, acc[1][1]);
      acc[1][2] = fmaf(g1, x.z, acc[1][2]); acc[1][3] = fmaf(g1, x.w, acc[1][3]);
      accb[0] += g0;
      accb[1] += g1;
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int c = c_tile + 2 * tc + i;
    if (c >= C) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int d = d_tile + 4 * td + j;
      if (d < D) dW[size_t(c) * D + d] = acc[i][j];
    }
    if (blockIdx.y == 0 && td == 0) db[c] = accb[i];
  }
}

// dxn for IMG images per block: the images' dlogits rows sit in shared memory, a weight element is loaded once per IMG uses
constexpr int kHeadImg = 4;
__global__ void __launch_bounds__(256)
head_dgrad2_kernel(const float* __restrict__ dlogits, const float* __restrict__ W, __nv_bfloat16* __restrict__ dxn, int B,
                   int D, int C) {
  extern __shared__ float sdl2[];                 // [kHeadImg][C], then the reduction scratch [4][kHeadImg][64]
  float* red = sdl2 + kHeadImg * C;
  const int b0 = blockIdx.y * kHeadImg, col = threadIdx.x & 63, d = blockIdx.x * 64 + col, part = threadIdx.x >> 6;
  for (int i = threadIdx.x; i < kHeadImg * C; i += 256) {
    const int b = i / C, c = i - b * C;
    sdl2[i] = b0 + b < B ? __ldg(dlogits + size_t(b0 + b) * C + c) : 0.f;
  }
  __syncthreads();
  float acc[kHeadImg];
#pragma unroll
  for (int i = 0; i < kHeadImg; ++i) acc[i] = 0.f;
  if (d < D) {
    int c = part;
    for (; c + 12 < C; c += 16) {                 // four independent weight loads in flight
      float w[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) w[u] = __ldg(W + size_t(c + 4 * u) * D + d);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < kHeadImg; ++i) acc[i] = fmaf(sdl2[i * C + c + 4 * u], w[u], acc[i]);
    }
    for (; c < C; c += 4) {
      const float w = __ldg(W + size_t(c) * D + d);
#pragma unroll
      for (int i = 0; i < kHeadImg; ++i) acc[i] = fmaf(sdl2[i * C + c], w, acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < kHeadImg; ++i) red[(part * kHeadImg + i) * 64 + col] = acc[i];
  __syncthreads();
  if (part == 0 && d < D) {
#pragma unroll
    for (int i = 0; i < kHeadImg; ++i)
      if (b0 + i < B)
        dxn[size_t(b0 + i) * D + d] = __float2bfloat16_rn((red[i * 64 + col] + red[(kHeadImg + i) * 64 + col]) +
                                                          (red[(2 * kHeadImg + i) * 64 + col] + red[(3 * kHeadImg + i) * 64 + col]));
  }
}

// ------------------------------------------------------------------------------------------------
// optimiser tail over the arena
// ------------------------------------------------------------------------------------------------
// Deterministic: every block leaves its partial sum in ws[block]; the block that finishes last adds the partials in
// index order.  (An atomicAdd of the partials gave a run-to-run different last bit, hence a different clip coefficient
// on every data-parallel rank: the ranks' parameters drifted apart by an ulp per step -- found by tools/dp_check.py.)
// out[0] = result, out[1 .. kSumsqBlocks] = partials, out[kSumsqBlocks + 1] = arrival counter (reset by the last block).
constexpr int kSumsqBlocks = 592;
static_assert(kSumsqBlocks + 2 <= 600, "APLA_SUMSQ_FLOATS (include/apla_b200.h) must cover result + partials + counter");
__global__ void sumsq_kernel(const float* __restrict__ g, int64_t n, float scale, float* __restrict__ out) {
  float acc = 0.f;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float v = g[i] * scale;
    acc += v * v;
  }
  acc = warp_sum(acc);
  __shared__ float red[32];
  __shared__ bool last;
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) {
      out[1 + blockIdx.x] = v;
      __threadfence();
      unsigned* counter = reinterpret_cast<unsigned*>(out + 1 + kSumsqBlocks);
      last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  // fixed order: thread t sums partials t, t + 256, ... ; then the same warp / block tree as above
  float v = 0.f;
  for (int i = threadIdx.x; i < int(gridDim.x); i += blockDim.x) v += __ldcg(out + 1 + i);
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) {
      out[0] = t;
      *reinterpret_cast<unsigned*>(out + 1 + kSumsqBlocks) = 0u;   // ready for the next launch (also under graph replay)
    }
  }
}

// torch.optim.AdamW semantics (decoupled decay first, then bias-corrected update), gradients pre-scaled by
// `gscale` (1/world for the data-parallel mean) and by the clip coefficient min(1, max_norm/(norm+1e-6)).
// Elements [0, n_decay) get weight decay (2-D tensors), the rest do not (biases; wrappers.py:205-221).
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, int64_t n, int64_t n_decay, const float* __restrict__ sumsq,
                             float gscale, float max_norm, float lr, float wd, float b1, float b2, float eps, float bc1,
                             float bc2_sqrt, const float* __restrict__ hyper) {
  if (hyper) {   // {lr, 1 - beta1^t, sqrt(1 - beta2^t)} from device memory: the launch can be replayed from a CUDA graph
    lr = hyper[0];
    bc1 = hyper[1];
    bc2_sqrt = hyper[2];
  }
  float coef = gscale;
  if (max_norm > 0.f) {
    const float norm = sqrtf(*sumsq);
    coef *= fminf(1.f, max_norm / (norm + 1e-6f));
  }
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const float gi = g[i] * coef;
    float pi = p[i];
    if (i < n_decay) pi *= (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

// scatter the trainable projection rows back into the dense bf16 working copies:
//   Wfull[l][idx[l][j], :] = bf16(W1[l][j, :]);  WfullT[l][:, idx[l][j]] = same;  bfull[l][idx[l][j]] = b1[l][j]
__global__ void proj_refresh_kernel(const float* __restrict__ w1, const float* __restrict__ b1,
                                    const int* __restrict__ idx, __nv_bfloat16* __restrict__ wfull,
                                    __nv_bfloat16* __restrict__ wfullT, float* __restrict__ bfull, int L, int r, int D,
                                    int64_t w1_block_stride, int64_t b1_block_stride) {
  const int l = blockIdx.y, j = blockIdx.x;
  const int row = idx[size_t(l) * r + j];
  const float* src = w1 + l * w1_block_stride + size_t(j) * D;
  __nv_bfloat16* wf = wfull + size_t(l) * D * D;
  __nv_bfloat16* wt = wfullT + size_t(l) * D * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const __nv_bfloat16 v = __float2bfloat16_rn(src[d]);
    wf[size_t(row) * D + d] = v;
    wt[size_t(d) * D + row] = v;
  }
  if (threadIdx.x == 0) bfull[size_t(l) * D + row] = b1[l * b1_block_stride + j];
}

}  // namespace

int head_fwd(const void* xn, const float* W, const float* bias, float* logits, int B, int D, int C, cudaStream_t s) {
  APLA_CHECK(B > 0 && D > 0 && C > 0, "head_fwd: empty");
  const int64_t threads = int64_t(B) * C * 32;
  head_fwd_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(xn), W, bias,
                                                                    logits, B, D, C);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int cross_entropy(const float* logits, const int64_t* labels, float* dlogits, float* loss, int B, int C, float grad_scale,
                  float loss_scale, cudaStream_t s) {
  APLA_CHECK(B > 0 && C > 0, "cross_entropy: empty");
  ce_kernel<<<B, 256, 0, s>>>(logits, labels, dlogits, loss, C, grad_scale, loss_scale);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int cross_entropy_soft(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                       float grad_scale, float loss_scale, cudaStream_t s) {
  APLA_CHECK(B > 0 && C > 0, "cross_entropy_soft: empty problem B=%d C=%d", B, C);
  APLA_CHECK(logits && targets && dlogits && loss, "cross_entropy_soft: null buffer");
  ce_soft_kernel<<<B, 256, 0, s>>>(logits, targets, dlogits, loss, C, grad_scale, loss_scale);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int bce_with_logits(const float* logits, const float* targets, float* dlogits, float* loss, int B, int C,
                    float grad_scale, float loss_scale, cudaStream_t s) {
  APLA_CHECK(B > 0 && C > 0, "bce_with_logits: empty problem B=%d C=%d", B, C);
  APLA_CHECK(logits && targets && dlogits && loss, "bce_with_logits: null buffer");
  bce_kernel<<<B, 256, 0, s>>>(logits, targets, dlogits, loss, C, grad_scale, loss_scale);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int eval_accumulate_bce(const float* logits, const float* targets, int B, int C, double* acc, cudaStream_t s) {
  APLA_CHECK(B > 0 && C > 0, "apla_eval_accumulate_bce: empty problem B=%d C=%d", B, C);
  APLA_CHECK(logits && targets && acc, "apla_eval_accumulate_bce: null buffer");
  eval_acc_bce_kernel<<<1, kEvalThreads, 0, s>>>(logits, targets, int64_t(B) * C, acc);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int eval_accumulate(const float* logits, const int64_t* labels, int B, int C, float* acc, cudaStream_t s) {
  APLA_CHECK(B > 0 && C > 0, "apla_eval_accumulate: empty problem B=%d C=%d", B, C);
  APLA_CHECK(logits && labels && acc, "apla_eval_accumulate: null buffer");
  eval_acc_kernel<<<1, kEvalThreads, 0, s>>>(logits, labels, B, C, acc);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int head_bwd(const float* dlogits, const void* xn, const float* W, float* dW, float* db, void* dxn, int B, int D, int C,
             cudaStream_t s) {
  APLA_CHECK(B > 0 && D > 0 && C > 0, "head_bwd: empty");
  head_wgrad2_kernel<<<dim3(cdiv(C, 32), cdiv(D, 64)), 256, 0, s>>>(dlogits, reinterpret_cast<const __nv_bfloat16*>(xn), dW, db,
                                                                    B, D, C);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  const size_t smem = (size_t(kHeadImg) * C + 4 * kHeadImg * 64) * sizeof(float);
  if (smem <= 48 * 1024) {
    head_dgrad2_kernel<<<dim3(cdiv(D, 64), cdiv(B, kHeadImg)), 256, smem, s>>>(dlogits, W, reinterpret_cast<__nv_bfloat16*>(dxn),
                                                                               B, D, C);
  } else {   // very wide heads: the per-image kernel
    head_dgrad_kernel<<<dim3(cdiv(D, 64), B), 256, 0, s>>>(dlogits, W, reinterpret_cast<__nv_bfloat16*>(dxn), B, D, C);
  }
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int grad_sumsq(const float* g, int64_t n, float scale, float* out, cudaStream_t s) {
  APLA_CHECK(n > 0, "grad_sumsq: empty");
  // `out` holds APLA_SUMSQ_FLOATS floats (include/apla_b200.h): result, per-block partials, arrival counter.  The counter
  // is zero on entry: the caller zero-initialises the buffer once and every launch leaves it at zero.
  const int grid = (int)((n + 1023) / 1024 < kSumsqBlocks ? (n + 1023) / 1024 : kSumsqBlocks);
  sumsq_kernel<<<grid, 256, 0, s>>>(g, n, scale, out);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int adamw_step(float* p, const float* g, float* m, float* v, int64_t n, int64_t n_decay, const float* sumsq,
               float gscale, float max_norm, float lr, float wd, float b1, float b2, float eps, int step,
               cudaStream_t s, const float* hyper) {
  APLA_CHECK(n > 0 && step >= 1, "adamw_step: empty arena or step < 1");
  const double bc1 = 1.0 - pow((double)b1, step);
  const double bc2 = 1.0 - pow((double)b2, step);
  const int grid = (int)((n + 1023) / 1024 < 1184 ? (n + 1023) / 1024 : 1184);
  adamw_kernel<<<grid, 256, 0, s>>>(p, g, m, v, n, n_decay, sumsq, gscale, max_norm, lr, wd, b1, b2, eps, (float)bc1,
                                    (float)sqrt(bc2), hyper);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int proj_refresh(const float* w1, const float* b1, const int* idx, void* wfull, void* wfullT, float* bfull, int L, int r,
                 int D, int64_t w1_block_stride, int64_t b1_block_stride, cudaStream_t s) {
  APLA_CHECK(L > 0 && r > 0 && D > 0, "proj_refresh: empty");
  proj_refresh_kernel<<<dim3(r, L), 256, 0, s>>>(w1, b1, idx, reinterpret_cast<__nv_bfloat16*>(wfull),
                                                 reinterpret_cast<__nv_bfloat16*>(wfullT), bfull, L, r, D,
                                                 w1_block_stride, b1_block_stride);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace apla
