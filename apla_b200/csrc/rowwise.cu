// HBM-bound row kernels of the ViT block: LayerNorm forward / backward with the residual-gradient add,
// the bf16 (LayerScale-scaled) gradient copy and the APLA column gather fused in; patch extraction; token
// assembly (cls + pos-embed).  One warp per row, 128-bit loads/stores, row kept in registers.
// Reference ops replaced: nn.LayerNorm(eps=1e-6) src/utils/transformers/vit.py:519,536,554,571 and :280,:285;
// LayerScale backward vit.py:243-244; scatter_ backward (= gather) src/apla/appla_attn.py:70-79;
// PatchEmbed / cls / pos add vit.py:304-307, :389-396.
#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"

namespace apla {

namespace {

constexpr int kMaxV4 = 8;  // D <= 1024 : up to 8 float4 per lane

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// LayerNorm forward: y_bf16 = (x - mean) * rstd * w + b
// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256)
ln_fwd_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w, const float* __restrict__ bias,
              __nv_bfloat16* __restrict__ y, int64_t ldy, int rows, float eps) {
  constexpr int D = NV * 128;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i] = __ldcs(xr + lane + 32 * i);
    s += v[i].x + v[i].y + v[i].z + v[i].w;
  }
  const float mean = warp_sum(s) * (1.f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.f / D) + eps);
  uint2* yr = reinterpret_cast<uint2*>(y + row * ldy);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 ww = __ldg(reinterpret_cast<const float4*>(w) + lane + 32 * i);
    const float4 bb = __ldg(reinterpret_cast<const float4*>(bias) + lane + 32 * i);
    yr[lane + 32 * i] = make_uint2(pack_bf16(v[i].x * rstd * ww.x + bb.x, v[i].y * rstd * ww.y + bb.y),
                                   pack_bf16(v[i].z * rstd * ww.z + bb.z, v[i].w * rstd * ww.w + bb.w));
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward (input gradient only; weight/bias are frozen), fused with
//   dx      = dres + LN'(dy)                      -> fp32 residual-stream gradient
//   dxb     = bf16(gamma * dx)                    -> A operand of the next dgrad GEMM (LayerScale folded in)
//   sub[j]  = bf16(gamma[idx[j]] * dx[idx[j]])    -> compact gathered columns for the APLA weight gradient
// mean / rstd are recomputed from x (the row is read anyway).
// kScaled (ln_bwd_scaled_kernel): dxb and sub are also multiplied by the row's scale row_scale[row / rows_per_scale] --
// the stochastic-depth mask of the branch that reads them; dx, the residual-stream gradient, is not.
// ------------------------------------------------------------------------------------------------
template <int NV, bool kScaled>
__device__ __forceinline__ void
ln_bwd_row(const __nv_bfloat16* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x, int64_t ldx,
           const float* __restrict__ w, const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx,
           __nv_bfloat16* __restrict__ dxb, int64_t ld_dxb, const float* __restrict__ gamma,
           __nv_bfloat16* __restrict__ sub, int64_t ld_sub, const int* __restrict__ idx, int r, int r_pad, int rows,
           float eps, const float* __restrict__ row_scale, int rows_per_scale) {
  constexpr int D = NV * 128;
  extern __shared__ float srow[];  // [warps][D], only used when sub != nullptr
  const int wib = threadIdx.x >> 5;
  const int row = blockIdx.x * (blockDim.x >> 5) + wib;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  [[maybe_unused]] float rscale = 1.f;
  if constexpr (kScaled) rscale = __ldg(row_scale + row / rows_per_scale);
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  const uint2* dyr = reinterpret_cast<const uint2*>(dy + row * ld_dy);
  const float4* rr = dres ? reinterpret_cast<const float4*>(dres + row * ld_dres) : nullptr;
  // all three input streams of the row are requested up front (14 x 512 B in flight per warp): the kernel is HBM-bound
  // and the reductions below would otherwise sit between three dependent DRAM round trips
  float4 v[NV], g[NV], r4[NV];
  uint2 dr[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = __ldcs(xr + lane + 32 * i);
#pragma unroll
  for (int i = 0; i < NV; ++i) dr[i] = __ldcs(dyr + lane + 32 * i);
  if (rr) {
#pragma unroll
    for (int i = 0; i < NV; ++i) r4[i] = __ldcs(rr + lane + 32 * i);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += v[i].x + v[i].y + v[i].z + v[i].w;
  const float mean = warp_sum(s) * (1.f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q += v[i].x * v[i].x + v[i].y * v[i].y + v[i].z * v[i].z + v[i].w * v[i].w;
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.f / D) + eps);
  float sg = 0.f, sgx = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const uint2 d = dr[i];
    const float4 ww = __ldg(reinterpret_cast<const float4*>(w) + lane + 32 * i);
    v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;   // xhat
    g[i] = make_float4(bf16_lo(d.x) * ww.x, bf16_hi(d.x) * ww.y, bf16_lo(d.y) * ww.z, bf16_hi(d.y) * ww.w);
    sg += g[i].x + g[i].y + g[i].z + g[i].w;
    sgx += g[i].x * v[i].x + g[i].y * v[i].y + g[i].z * v[i].z + g[i].w * v[i].w;
  }
  const float mg = warp_sum(sg) * (1.f / D), mgx = warp_sum(sgx) * (1.f / D);
  float4* outr = reinterpret_cast<float4*>(dx + row * ld_dx);
  uint2* outb = dxb ? reinterpret_cast<uint2*>(dxb + row * ld_dxb) : nullptr;
  float* sr = srow + wib * D;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float4 o;
    o.x = rstd * (g[i].x - mg - v[i].x * mgx);
    o.y = rstd * (g[i].y - mg - v[i].y * mgx);
    o.z = rstd * (g[i].z - mg - v[i].z * mgx);
    o.w = rstd * (g[i].w - mg - v[i].w * mgx);
    if (rr) {
      o.x += r4[i].x; o.y += r4[i].y; o.z += r4[i].z; o.w += r4[i].w;
    }
    outr[lane + 32 * i] = o;
    if (outb || sub) {
      if (gamma) {
        const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * i);
        o.x *= gm.x; o.y *= gm.y; o.z *= gm.z; o.w *= gm.w;
      }
      if constexpr (kScaled) {
        o.x *= rscale; o.y *= rscale; o.z *= rscale; o.w *= rscale;
      }
      if (outb) outb[lane + 32 * i] = make_uint2(pack_bf16(o.x, o.y), pack_bf16(o.z, o.w));
      if (sub) reinterpret_cast<float4*>(sr)[lane + 32 * i] = o;
    }
  }
  if (sub) {
    __syncwarp();
    __nv_bfloat16* so = sub + row * ld_sub;
    for (int j = lane; j < r_pad; j += 32) so[j] = __float2bfloat16_rn(j < r ? sr[__ldg(idx + j)] : 0.f);
  }
}

template <int NV>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x, int64_t ldx,
              const float* __restrict__ w, const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx,
              __nv_bfloat16* __restrict__ dxb, int64_t ld_dxb, const float* __restrict__ gamma,
              __nv_bfloat16* __restrict__ sub, int64_t ld_sub, const int* __restrict__ idx, int r, int r_pad, int rows,
              float eps) {
  ln_bwd_row<NV, false>(dy, ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx, dxb, ld_dxb, gamma, sub, ld_sub, idx, r, r_pad,
                        rows, eps, nullptr, 1);
}

template <int NV>
__global__ void __launch_bounds__(256)
ln_bwd_scaled_kernel(const __nv_bfloat16* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x, int64_t ldx,
                     const float* __restrict__ w, const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx,
                     __nv_bfloat16* __restrict__ dxb, int64_t ld_dxb, const float* __restrict__ gamma,
                     __nv_bfloat16* __restrict__ sub, int64_t ld_sub, const int* __restrict__ idx, int r, int r_pad,
                     int rows, float eps, const float* __restrict__ row_scale, int rows_per_scale) {
  ln_bwd_row<NV, true>(dy, ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx, dxb, ld_dxb, gamma, sub, ld_sub, idx, r, r_pad,
                       rows, eps, row_scale, rows_per_scale);
}

// ------------------------------------------------------------------------------------------------
// Generic-width LayerNorm (any D % 4 == 0 that is not a multiple of 128, e.g. the 64-wide toy models of the parity
// fixtures): same arithmetic, one warp per row, the row re-read from L1/L2 instead of held in registers.  Not a
// performance path.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ln_fwd_generic_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                      const float* __restrict__ bias, __nv_bfloat16* __restrict__ y, int64_t ldy, int rows, int D,
                      float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * ldx;
  float s = 0.f;
  for (int k = lane; k < D; k += 32) s += xr[k];
  const float mean = warp_sum(s) / D;
  float q = 0.f;
  for (int k = lane; k < D; k += 32) q += (xr[k] - mean) * (xr[k] - mean);
  const float rstd = rsqrtf(warp_sum(q) / D + eps);
  for (int k = lane; k < D; k += 32) y[row * ldy + k] = __float2bfloat16_rn((xr[k] - mean) * rstd * w[k] + bias[k]);
}

__global__ void __launch_bounds__(256)
ln_bwd_generic_kernel(const __nv_bfloat16* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x, int64_t ldx,
                      const float* __restrict__ w, const float* dres, int64_t ld_dres, float* dx, int64_t ld_dx,
                      __nv_bfloat16* __restrict__ dxb, int64_t ld_dxb, const float* __restrict__ gamma,
                      __nv_bfloat16* __restrict__ sub, int64_t ld_sub, const int* __restrict__ idx, int r, int r_pad,
                      int rows, int D, float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * ldx;
  const __nv_bfloat16* dyr = dy + row * ld_dy;
  float s = 0.f;
  for (int k = lane; k < D; k += 32) s += xr[k];
  const float mean = warp_sum(s) / D;
  float q = 0.f;
  for (int k = lane; k < D; k += 32) q += (xr[k] - mean) * (xr[k] - mean);
  const float rstd = rsqrtf(warp_sum(q) / D + eps);
  float sg = 0.f, sgx = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float g = __bfloat162float(dyr[k]) * w[k];
    sg += g;
    sgx += g * (xr[k] - mean) * rstd;
  }
  const float mg = warp_sum(sg) / D, mgx = warp_sum(sgx) / D;
  // (dres may alias dx: every element is read and written by the same thread, reads first)
  for (int k = lane; k < D; k += 32) {
    const float g = __bfloat162float(dyr[k]) * w[k];
    float o = rstd * (g - mg - (xr[k] - mean) * rstd * mgx);
    if (dres) o += dres[row * ld_dres + k];
    dx[row * ld_dx + k] = o;
    if (dxb) dxb[row * ld_dxb + k] = __float2bfloat16_rn(gamma ? o * gamma[k] : o);
  }
  if (sub) {
    __syncwarp();
    __threadfence_block();
    for (int j = lane; j < r_pad; j += 32) {
      float v = 0.f;
      if (j < r) {
        const int c = idx[j];
        v = dx[row * ld_dx + c] * (gamma ? gamma[c] : 1.f);
      }
      sub[row * ld_sub + j] = __float2bfloat16_rn(v);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// scaled fp32 -> bf16 copy with the same gather (used where no LayerNorm precedes: nothing on the C2 path,
// kept for the module-level API where dY arrives from autograd)
// ------------------------------------------------------------------------------------------------
__global__ void gather_cols_kernel(const __nv_bfloat16* __restrict__ dy, int64_t ld, __nv_bfloat16* __restrict__ sub,
                                   int64_t ld_sub, const int* __restrict__ idx, int r, int r_pad, int rows) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= int64_t(rows) * r_pad) return;
  const int row = int(i / r_pad), j = int(i % r_pad);
  sub[row * ld_sub + j] = j < r ? dy[row * ld + __ldg(idx + j)] : __float2bfloat16_rn(0.f);
}

// out_bf16[t, d] = gamma[d] * x_f32[t, d] (gamma NULL = 1): LayerScale backward + down-cast of a residual gradient that
// arrives from outside the fused chain (autograd handing the block-level Function its dY); 4 elements per thread
__global__ void ls_cast_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ gamma,
                               __nv_bfloat16* __restrict__ out, int64_t ldo, int rows, int D4) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= int64_t(rows) * D4) return;
  const int row = int(i / D4), c = int(i % D4) * 4;
  float4 v = *reinterpret_cast<const float4*>(x + row * ldx + c);
  if (gamma) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    v.x *= g.x; v.y *= g.y; v.z *= g.z; v.w *= g.w;
  }
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&lo);
  pk.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(out + row * ldo + c) = pk;
}

// column sums of a bf16 [rows, n] matrix -> fp32 out[map(j)] (+=): bias gradient of the trainable rows
__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ a, int64_t ld, int rows, int n, float* __restrict__ out,
                              const int* __restrict__ rowmap, int rows_per_block) {
  // block = 32 x 8 threads: x over columns, y over row slices
  __shared__ float red[8][33];
  const int col = blockIdx.x * 32 + threadIdx.x;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(rows, r0 + rows_per_block);
  float acc = 0.f;
  if (col < n)
    for (int r = r0 + threadIdx.y; r < r1; r += 8) acc += __bfloat162float(a[r * ld + col]);
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && col < n) {
#pragma unroll
    for (int k = 1; k < 8; ++k) acc += red[k][threadIdx.x];
    const int o = rowmap ? rowmap[col] : col;
    if (o >= 0) atomicAdd(out + o, acc);
  }
}

// The same for a WIDE matrix (partial_size == dim: n = 768 / 1024 columns of the dense dY): 16-byte loads, a warp covers 256
// consecutive columns of a row (512 contiguous bytes), 8 warps x `rows_per_block / 8` rows each with four loads in flight,
// one fp32 atomic per column and block.  (The narrow kernel above reads 2 bytes per thread: 1.5 TB/s on this shape.)
__global__ void __launch_bounds__(256)
colsum_wide_kernel(const __nv_bfloat16* __restrict__ a, int64_t ld, int rows, int n, float* __restrict__ out,
                   const int* __restrict__ rowmap, int rows_per_block) {
  __shared__ float red[8][256 + 8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int col0 = blockIdx.x * 256 + lane * 8;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(rows, r0 + rows_per_block);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (col0 < n) {
    const __nv_bfloat16* base = a + col0;
    int r = r0 + w;
    for (; r + 24 < r1; r += 32) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldcs(reinterpret_cast<const uint4*>(base + int64_t(r + 8 * u) * ld));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t q[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          acc[2 * t] += bf16_lo(q[t]);
          acc[2 * t + 1] += bf16_hi(q[t]);
        }
      }
    }
    for (; r < r1; r += 8) {
      const uint4 v = __ldcs(reinterpret_cast<const uint4*>(base + int64_t(r) * ld));
      const uint32_t q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        acc[2 * t] += bf16_lo(q[t]);
        acc[2 * t + 1] += bf16_hi(q[t]);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 8; ++t) red[w][lane * 8 + t] = acc[t];
  __syncthreads();
  const int c = threadIdx.x;                       // one column of the block's 256 per thread
  const int col = blockIdx.x * 256 + c;
  if (col < n) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sum += red[k][c];
    const int o = rowmap ? rowmap[col] : col;
    if (o >= 0) atomicAdd(out + o, sum);
  }
}

// ------------------------------------------------------------------------------------------------
// patch extraction: images fp32 [B,3,S,S] -> bf16 [B*P, kpad], k = (c, py, px)  (conv k=s=p as a GEMM)
// ------------------------------------------------------------------------------------------------
// One block per (image b, patch row gy, channel c): it reads p full image rows (every fetched line is consumed by the
// block) and writes, for each of the S/p patches of that patch row, the p*p contiguous bf16 of channel c -- consecutive
// threads write consecutive bytes.  (The first version walked image rows and scattered 28-byte runs: 46 us.)
// Blocks past those zero the kpad - 3*p*p padding columns of the patch matrix.
__global__ void __launch_bounds__(256)
patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int S, int p, int kpad) {
  const int g = S / p;
  const int kk = 3 * p * p;
  const int n_main = B * g * 3;
  if (int(blockIdx.x) < n_main) {
    const int c = blockIdx.x % 3, gy = (blockIdx.x / 3) % g, b = blockIdx.x / (3 * g);
    const float* src = img + (size_t(b) * 3 + c) * S * S + size_t(gy) * p * S;
    __nv_bfloat16* dst = out + (size_t(b) * g * g + size_t(gy) * g) * kpad + c * p * p;
    const int pp = p * p;
    if ((p & 1) == 0 && (kpad & 1) == 0) {
      const int half = pp >> 1;
      for (int i = threadIdx.x; i < g * half; i += blockDim.x) {
        const int gx = i / half, rem = 2 * (i - gx * half), py = rem / p, px = rem - py * p;
        const float2 v = __ldg(reinterpret_cast<const float2*>(src + size_t(py) * S + gx * p + px));
        *reinterpret_cast<uint32_t*>(dst + size_t(gx) * kpad + rem) = pack_bf16(v.x, v.y);
      }
    } else {
      for (int i = threadIdx.x; i < g * pp; i += blockDim.x) {
        const int gx = i / pp, rem = i - gx * pp, py = rem / p, px = rem - py * p;
        dst[size_t(gx) * kpad + rem] = __float2bfloat16_rn(__ldg(src + size_t(py) * S + gx * p + px));
      }
    }
  } else {
    const int pad = kpad - kk;
    const int64_t total = int64_t(B) * g * g * pad;
    for (int64_t i = int64_t(blockIdx.x - n_main) * blockDim.x + threadIdx.x; i < total;
         i += int64_t(gridDim.x - n_main) * blockDim.x)
      out[(i / pad) * kpad + kk + (i % pad)] = __float2bfloat16_rn(0.f);
  }
}

// tokens: x[b,0,:] = cls + pos[0];  x[b,1+i,:] = patch[b*P+i,:] + pos[1+i]      (fp32 residual stream)
__global__ void assemble_tokens_kernel(const __nv_bfloat16* __restrict__ patch, const float* __restrict__ cls,
                                       const float* __restrict__ pos, float* __restrict__ x, int B, int P, int D) {
  const int64_t total = int64_t(B) * (P + 1) * (D / 4);
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int d4 = int(i % (D / 4));
    const int64_t tok = i / (D / 4);
    const int n = int(tok % (P + 1)), b = int(tok / (P + 1));
    float4 v = __ldg(reinterpret_cast<const float4*>(pos) + int64_t(n) * (D / 4) + d4);
    if (n == 0) {
      const float4 c = __ldg(reinterpret_cast<const float4*>(cls) + d4);
      v.x += c.x; v.y += c.y; v.z += c.z; v.w += c.w;
    } else {
      const uint2 pv = __ldg(reinterpret_cast<const uint2*>(patch) + (int64_t(b) * P + n - 1) * (D / 4) + d4);
      v.x += bf16_lo(pv.x); v.y += bf16_hi(pv.x); v.z += bf16_lo(pv.y); v.w += bf16_hi(pv.y);
    }
    reinterpret_cast<float4*>(x)[i] = v;
  }
}

}  // namespace

#define LN_DISPATCH(NV_, CALL)            \
  switch (NV_) {                          \
    case 1: { constexpr int NV = 1; CALL; } break; \
    case 2: { constexpr int NV = 2; CALL; } break; \
    case 3: { constexpr int NV = 3; CALL; } break; \
    case 4: { constexpr int NV = 4; CALL; } break; \
    case 6: { constexpr int NV = 6; CALL; } break; \
    case 8: { constexpr int NV = 8; CALL; } break; \
    default: set_error("layernorm: unsupported width %d (supported: 128,256,384,512,768,1024)", (NV_)*128); return 1; \
  }

int layernorm_fwd(const float* x, int64_t ldx, const float* w, const float* b, void* y, int64_t ldy, int rows, int D,
                  float eps, cudaStream_t stream) {
  APLA_CHECK(rows > 0, "layernorm_fwd: no rows");
  APLA_CHECK(D > 0 && D % 4 == 0 && D <= 128 * kMaxV4, "layernorm_fwd: D=%d must be a multiple of 4 and <= 1024", D);
  APLA_CHECK(ldx % 4 == 0 && ldy % 4 == 0, "layernorm_fwd: leading dimensions must be multiples of 4");
  const int grid = cdiv(rows, 8);
  if (D % 128 != 0) {
    ln_fwd_generic_kernel<<<grid, 256, 0, stream>>>(x, ldx, w, b, reinterpret_cast<__nv_bfloat16*>(y), ldy, rows, D, eps);
    APLA_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  LN_DISPATCH(D / 128, (ln_fwd_kernel<NV><<<grid, 256, 0, stream>>>(x, ldx, w, b, reinterpret_cast<__nv_bfloat16*>(y),
                                                                    ldy, rows, eps)));
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int layernorm_bwd(const void* dy, int64_t ld_dy, const float* x, int64_t ldx, const float* w, const float* dres,
                  int64_t ld_dres, float* dx, int64_t ld_dx, void* dxb, int64_t ld_dxb, const float* gamma, void* sub,
                  int64_t ld_sub, const int* idx, int r, int r_pad, int rows, int D, float eps, cudaStream_t stream,
                  const float* row_scale, int rows_per_scale) {
  APLA_CHECK(rows > 0, "layernorm_bwd: no rows");
  APLA_CHECK(D > 0 && D % 4 == 0 && D <= 128 * kMaxV4, "layernorm_bwd: D=%d must be a multiple of 4 and <= 1024", D);
  APLA_CHECK(ld_dy % 4 == 0 && ldx % 4 == 0 && ld_dx % 4 == 0 && ld_dres % 4 == 0 && ld_dxb % 4 == 0,
             "layernorm_bwd: leading dimensions must be multiples of 4");
  APLA_CHECK(sub == nullptr || (idx != nullptr && r <= r_pad && r_pad <= ld_sub), "layernorm_bwd: bad gather arguments");
  const int grid = cdiv(rows, 8);
  if (row_scale) {
    APLA_CHECK(D % 128 == 0, "layernorm_bwd: the row-scaled backward needs D a multiple of 128, got %d", D);
    APLA_CHECK(rows_per_scale >= 1, "layernorm_bwd: rows_per_scale=%d must be >= 1", rows_per_scale);
    const size_t smem = sub ? size_t(8) * D * sizeof(float) : 0;
    LN_DISPATCH(D / 128, (ln_bwd_scaled_kernel<NV><<<grid, 256, smem, stream>>>(
                             reinterpret_cast<const __nv_bfloat16*>(dy), ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx,
                             reinterpret_cast<__nv_bfloat16*>(dxb), ld_dxb, gamma, reinterpret_cast<__nv_bfloat16*>(sub),
                             ld_sub, idx, r, r_pad, rows, eps, row_scale, rows_per_scale)));
    APLA_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  if (D % 128 != 0) {
    ln_bwd_generic_kernel<<<grid, 256, 0, stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(dy), ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx,
        reinterpret_cast<__nv_bfloat16*>(dxb), ld_dxb, gamma, reinterpret_cast<__nv_bfloat16*>(sub), ld_sub, idx, r, r_pad,
        rows, D, eps);
    APLA_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  const size_t smem = sub ? size_t(8) * D * sizeof(float) : 0;
  LN_DISPATCH(D / 128, (ln_bwd_kernel<NV><<<grid, 256, smem, stream>>>(
                           reinterpret_cast<const __nv_bfloat16*>(dy), ld_dy, x, ldx, w, dres, ld_dres, dx, ld_dx,
                           reinterpret_cast<__nv_bfloat16*>(dxb), ld_dxb, gamma, reinterpret_cast<__nv_bfloat16*>(sub),
                           ld_sub, idx, r, r_pad, rows, eps)));
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int gather_cols(const void* dy, int64_t ld, void* sub, int64_t ld_sub, const int* idx, int r, int r_pad, int rows,
                cudaStream_t stream) {
  const int64_t total = int64_t(rows) * r_pad;
  APLA_CHECK(total > 0, "gather_cols: empty");
  gather_cols_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(dy), ld, reinterpret_cast<__nv_bfloat16*>(sub), ld_sub, idx, r, r_pad, rows);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int ls_cast(const float* x, int64_t ldx, const float* gamma, void* out, int64_t ldo, int rows, int D,
            cudaStream_t stream) {
  APLA_CHECK(rows > 0 && D > 0 && D % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0, "ls_cast: bad shape rows=%d D=%d", rows, D);
  const int64_t total = int64_t(rows) * (D / 4);
  ls_cast_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(x, ldx, gamma, reinterpret_cast<__nv_bfloat16*>(out),
                                                                      ldo, rows, D / 4);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int colsum(const void* a, int64_t ld, int rows, int n, float* out, const int* rowmap, cudaStream_t stream) {
  APLA_CHECK(rows > 0 && n > 0, "colsum: empty");
  static const bool narrow_only = [] { const char* e = getenv("APLA_COLSUM_NARROW"); return e && atoi(e) != 0; }();   // A/B switch
  if (!narrow_only && n >= 256 && n % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a) & 15) == 0) {
    // enough row slices to put ~8 blocks on every SM, at least 32 rows (4 per warp) each
    const int col_blocks = cdiv(n, 256);
    int rpb = cdiv(rows, cdiv(sm_count() * 8, col_blocks));
    rpb = rpb < 32 ? 32 : (rpb + 7) / 8 * 8;
    dim3 grid(col_blocks, cdiv(rows, rpb));
    colsum_wide_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(a), ld, rows, n, out, rowmap, rpb);
    APLA_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  const int rows_per_block = 64;
  dim3 grid(cdiv(n, 32), cdiv(rows, rows_per_block));
  colsum_kernel<<<grid, dim3(32, 8), 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(a), ld, rows, n, out, rowmap,
                                                  rows_per_block);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int patchify(const float* img, void* out, int B, int S, int p, int kpad, cudaStream_t stream) {
  APLA_CHECK(B > 0 && S % p == 0 && kpad >= 3 * p * p, "patchify: bad shape B=%d S=%d p=%d kpad=%d", B, S, p, kpad);
  const int pad_blocks = kpad > 3 * p * p ? 64 : 0;
  patchify_kernel<<<B * (S / p) * 3 + pad_blocks, 256, 0, stream>>>(img, reinterpret_cast<__nv_bfloat16*>(out), B, S, p, kpad);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int assemble_tokens(const void* patch, const float* cls, const float* pos, float* x, int B, int P, int D,
                    cudaStream_t stream) {
  APLA_CHECK(B > 0 && P > 0 && D % 4 == 0, "assemble_tokens: bad shape");
  const int64_t total = int64_t(B) * (P + 1) * (D / 4);
  const int grid = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  assemble_tokens_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(patch), cls, pos, x, B, P, D);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace apla
