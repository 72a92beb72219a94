// Persistent warp-specialised tcgen05 GEMM for sm_100a.
//
//   D[M,N] = A[M,K] * B[N,K]^T           (both operands K-contiguous: y = x W^T with W = [out,in])
//   D[M,N] = A^T * B  with A = [K,M], B = [K,N] both MN-contiguous ("NT", the weight-gradient form)
//
// bf16 operands arrive by TMA into 128B-swizzled shared-memory stages, one elected thread issues
// tcgen05.mma (128 x BN x 16, fp32 accumulation in TMEM), the accumulator is double-buffered in TMEM so
// the epilogue warps (tcgen05.ld -> registers -> fused epilogue -> global) overlap the next tile's MMAs.
//
// Fused epilogues (what the reference runs as separate ATen kernels, SURVEY.md 2.3 K2/K14/K15/K17-K20):
//   EPI_BIAS       out_bf16 = acc + bias[n]
//   EPI_BIAS_GELU  out_bf16 = h = acc + bias[n];  out2_bf16 = gelu_erf(h)        (Mlp.fc1 + act, vit.py:163-164)
//   EPI_RESID      out_f32  = aux_f32[m,n] + gamma[n] * (acc + bias[n])          (proj/fc2 + LayerScale + residual)
//   EPI_GELU_BWD   out_bf16 = acc * gelu_erf'(aux_bf16[m,n])                     (fc2 dgrad fused with GELU backward)
//   EPI_F32_T      atomicAdd(out_f32[rowmap(n), m], acc)                         (split-K weight gradient, transposed)
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

#include <stdlib.h>

namespace apla {

struct GemmEpi {
  void* out;
  void* out2;
  const float* bias;
  const float* gamma;
  const void* aux;
  const int* rowmap;  // EPI_F32_T: output row for column n (negative = skip); null = identity
  int ldo;            // leading dimension (elements) of out / out2 / aux
  int n_valid;        // EPI_F32_T: columns >= n_valid are padding
};

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + kEpiWarps * 32;

template <int BN>
struct GemmCfg {
  static constexpr int kStages = BN == 256 ? 4 : (BN == 128 ? 6 : 8);
  static constexpr uint32_t kABytes = BM * BK * 2;
  static constexpr uint32_t kBBytes = BN * BK * 2;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kTmemCols = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr size_t kSmemBytes = 1024 + size_t(kStages) * kStageBytes + 256;
};

template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[32], int row, int col0, int M, const GemmEpi& ep) {
  // one thread = one output row, 32 consecutive columns starting at col0
  if constexpr (EPI == EPI_F32_T) {
    float* out = reinterpret_cast<float*>(ep.out);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int n = col0 + j;
      if (n < ep.n_valid && row < M) {
        const int r = ep.rowmap ? __ldg(ep.rowmap + n) : n;
        if (r >= 0) atomicAdd(out + size_t(r) * ep.ldo + row, __uint_as_float(v[j]));
      }
    }
    return;
  } else {
    if (row >= M) return;
    const size_t off = size_t(row) * ep.ldo + col0;
    float x[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]);
    if constexpr (EPI == EPI_BIAS || EPI == EPI_BIAS_GELU || EPI == EPI_RESID) {
      if (ep.bias) {
        const float4* b4 = reinterpret_cast<const float4*>(ep.bias + col0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b = __ldg(b4 + j);
          x[4 * j + 0] += b.x; x[4 * j + 1] += b.y; x[4 * j + 2] += b.z; x[4 * j + 3] += b.w;
        }
      }
    }
    if constexpr (EPI == EPI_BIAS) {
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(ep.out) + off);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        o[j] = make_uint4(pack_bf16(x[8 * j], x[8 * j + 1]), pack_bf16(x[8 * j + 2], x[8 * j + 3]),
                          pack_bf16(x[8 * j + 4], x[8 * j + 5]), pack_bf16(x[8 * j + 6], x[8 * j + 7]));
    } else if constexpr (EPI == EPI_BIAS_GELU) {
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(ep.out) + off);
      uint4* o2 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(ep.out2) + off);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t h[4], g[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          h[t] = pack_bf16(x[8 * j + 2 * t], x[8 * j + 2 * t + 1]);
          // GELU of the bf16-rounded pre-activation (what autocast feeds nn.GELU)
          g[t] = pack_bf16(gelu_erf(bf16_lo(h[t])), gelu_erf(bf16_hi(h[t])));
        }
        o[j] = make_uint4(h[0], h[1], h[2], h[3]);
        o2[j] = make_uint4(g[0], g[1], g[2], g[3]);
      }
    } else if constexpr (EPI == EPI_RESID) {
      const float4* r4 = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ep.aux) + off);
      float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + off);
      const float4* g4 = reinterpret_cast<const float4*>(ep.gamma ? ep.gamma + col0 : nullptr);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 r = __ldcs(r4 + j);
        float4 g = ep.gamma ? __ldg(g4 + j) : make_float4(1.f, 1.f, 1.f, 1.f);
        r.x += g.x * x[4 * j + 0]; r.y += g.y * x[4 * j + 1]; r.z += g.z * x[4 * j + 2]; r.w += g.w * x[4 * j + 3];
        o[j] = r;
      }
    } else if constexpr (EPI == EPI_GELU_BWD) {
      const uint4* h4 = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(ep.aux) + off);
      uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(ep.out) + off);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint4 h = __ldcs(h4 + j);
        const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
        uint32_t d[4];
#pragma unroll
        for (int t = 0; t < 4; ++t)
          d[t] = pack_bf16(x[8 * j + 2 * t] * gelu_erf_grad(bf16_lo(hw[t])),
                           x[8 * j + 2 * t + 1] * gelu_erf_grad(bf16_hi(hw[t])));
        o[j] = make_uint4(d[0], d[1], d[2], d[3]);
      }
    }
  }
}

// A_MN / B_MN: operand is MN-contiguous in global memory ([K, M] / [K, N] row-major)
template <int BN, int EPI, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, int M, int N, int K,
            int k_splits, GemmEpi ep) {
  using Cfg = GemmCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::kStageBytes);
  uint64_t* empty = full + kStages;
  uint64_t* tfull = empty + kStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_m = (M + BM - 1) / BM;
  const int num_n = (N + BN - 1) / BN;
  const int num_kb_total = (K + BK - 1) / BK;
  const int kb_per_split = (num_kb_total + k_splits - 1) / k_splits;
  const int num_tiles = num_m * num_n * k_splits;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int split = tile / (num_m * num_n);
        const int mn = tile - split * (num_m * num_n);
        const int m0 = (mn / num_n) * BM;
        const int n0 = (mn % num_n) * BN;
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, num_kb_total);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + Cfg::kABytes;
          mbar_arrive_expect_tx(&full[stage], Cfg::kStageBytes);
          if constexpr (!A_MN) {
            tma_load_2d(sa, &tma_a, &full[stage], kb * BK, m0);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j) tma_load_2d(sa + j * (BK * 128), &tma_a, &full[stage], m0 + j * 64, kb * BK);
          }
          if constexpr (!B_MN) {
            tma_load_2d(sb, &tma_b, &full[stage], kb * BK, n0);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * (BK * 128), &tma_b, &full[stage], n0 + j * 64, kb * BK);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int split = tile / (num_m * num_n);
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, num_kb_total);
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t b_base = a_base + Cfg::kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // K-major: 16 bf16 = 32 B along the swizzled row, SBO = 8 rows * 128 B.
            // MN-major: 16 k-rows = 2048 B, LBO = one 64-wide MN box (BK*128 B), SBO = 8 k-rows * 128 B.
            const uint64_t adesc = A_MN ? make_sdesc_sw128(a_base + k * 2048, BK * 128, 1024)
                                        : make_sdesc_sw128(a_base + k * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? make_sdesc_sw128(b_base + k * 2048, BK * 128, 1024)
                                        : make_sdesc_sw128(b_base + k * 32, 16, 1024);
            umma_bf16<1>(d_tmem, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty[stage]);  // frees the smem stage when these MMAs retire
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[as]);  // accumulator ready
        as ^= 1;
        if (as == 0) aphase ^= 1;
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int ew = warp - 2;
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int half = ew >> 2;          // warps sharing a quarter split the column chunks
    int as = 0;
    uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int split = tile / (num_m * num_n);
      const int mn = tile - split * (num_m * num_n);
      const int m0 = (mn / num_n) * BM;
      const int n0 = (mn % num_n) * BN;
      const bool has_k = split * kb_per_split < num_kb_total;
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const int row = m0 + q * 32 + lane;
      if (has_k) {
#pragma unroll 1
        for (int c = half; c < BN / 32; c += kEpiWarps / 4) {
          const int col0 = n0 + c * 32;
          if (col0 >= N) break;
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(as * BN + c * 32), v);
          tmem_ld_wait();
          epilogue_chunk<EPI>(v, row, col0, M, ep);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int EPI, bool A_MN, bool B_MN>
static int launch(const void* A, const void* B, int M, int N, int K, int lda, int ldb, int k_splits, const GemmEpi& ep,
                  cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  CUtensorMap ta, tb;
  int rc;
  if (!A_MN) rc = make_tmap_2d(&ta, A, 2, M, K, lda, BM, BK, true);
  else rc = make_tmap_2d(&ta, A, 2, K, M, lda, BK, 64, true);
  if (rc) return rc;
  if (!B_MN) rc = make_tmap_2d(&tb, B, 2, N, K, ldb, BN, BK, true);
  else rc = make_tmap_2d(&tb, B, 2, K, N, ldb, BK, 64, true);
  if (rc) return rc;
  auto kern = gemm_kernel<BN, EPI, A_MN, B_MN>;
  static bool attr_set = false;
  if (!attr_set) {
    APLA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes));
    attr_set = true;
  }
  const int tiles = cdiv(M, BM) * cdiv(N, BN) * k_splits;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  kern<<<grid, kThreads, Cfg::kSmemBytes, stream>>>(ta, tb, M, N, K, k_splits, ep);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

static int pick_bn(int M, int N) {
  // widest tile whose last wave is reasonably full; 256 keeps shared-memory operand traffic lowest
  const int sms = sm_count();
  int best = 256;
  double best_cost = 1e30;
  const int cands[3] = {256, 128, 64};
  for (int i = 0; i < 3; ++i) {
    const int bn = cands[i];
    if (bn > 64 && bn / 2 >= N) continue;
    const int tiles = cdiv(M, BM) * cdiv(N, bn);
    const int waves = cdiv(tiles, sms);
    // cost ~ waves * per-tile time; narrower tiles pay more smem traffic per flop (A re-read)
    const double tile_t = bn * (bn == 256 ? 1.0 : (bn == 128 ? 1.08 : 1.35));
    const double cost = waves * tile_t;
    if (cost < best_cost - 1e-9) { best_cost = cost; best = bn; }
  }
  return best;
}

template <int EPI>
static int dispatch_tn(const void* A, const void* B, int M, int N, int K, int lda, int ldb, const GemmEpi& ep,
                       cudaStream_t stream, int bn_override) {
  int bn = bn_override;
  if (bn <= 0) {
    const char* e = getenv("APLA_GEMM_BN");   // test hook: force one tile width
    bn = e ? atoi(e) : 0;
  }
  if (bn <= 0) bn = pick_bn(M, N);
  switch (bn) {
    case 256: return launch<256, EPI, false, false>(A, B, M, N, K, lda, ldb, 1, ep, stream);
    case 128: return launch<128, EPI, false, false>(A, B, M, N, K, lda, ldb, 1, ep, stream);
    case 64: return launch<64, EPI, false, false>(A, B, M, N, K, lda, ldb, 1, ep, stream);
  }
  set_error("unsupported BN %d", bn);
  return 1;
}

// ------------------------------------------------------------------------------------------------
// public entry (used by capi.cu and engine.cu)
// ------------------------------------------------------------------------------------------------
int gemm_tn(int epi, const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
            const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream, int bn_override) {
  APLA_CHECK(M > 0 && N > 0 && K > 0, "gemm_tn: empty problem %dx%dx%d", M, N, K);
  APLA_CHECK(N % 32 == 0, "gemm_tn: N=%d must be a multiple of 32", N);
  APLA_CHECK(K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0, "gemm_tn: K/lda/ldb (%d/%d/%d) must be multiples of 8", K, lda,
             ldb);
  APLA_CHECK(ldo % 8 == 0, "gemm_tn: ldo=%d must be a multiple of 8", ldo);
  APLA_CHECK(epi != EPI_BIAS_GELU || out2 != nullptr, "gemm_tn: EPI_BIAS_GELU needs out2");
  APLA_CHECK((epi != EPI_RESID && epi != EPI_GELU_BWD && epi != EPI_DELTA) || aux != nullptr,
             "gemm_tn: this epilogue needs aux");
  APLA_CHECK(epi != EPI_MUL_F16 || aux != nullptr, "gemm_tn: EPI_MUL_F16 needs the fp16 multiplier in aux");
  APLA_CHECK(epi != EPI_BIAS_GELU_D || out2 != nullptr, "gemm_tn: EPI_BIAS_GELU_D needs out2");
  if (epi == EPI_DELTA || epi == EPI_BIAS_GELU_D || epi == EPI_BIAS_GELU_G || epi == EPI_MUL_F16 || epi == EPI_RED) {   // 2-CTA kernel only
    APLA_CHECK(epi != EPI_DELTA || (out2 != nullptr && N % 64 == 0),
               "gemm_tn: EPI_DELTA needs the delta buffer in out2 and N %% 64 == 0");
    int bn = bn_override;
    if (bn <= 0) { const char* e = getenv("APLA_GEMM_BN"); bn = e ? atoi(e) : 0; }
    return gemm2_tn(epi, A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
  }
  {
    // default: the 2-CTA kernel with TMA-store epilogues (gemm2.cu); APLA_GEMM_IMPL=1 selects the 1-CTA kernel below
    // (kept for A/B measurements and as the weight-gradient kernel).
    static const int impl = [] { const char* e = getenv("APLA_GEMM_IMPL"); return e ? atoi(e) : 2; }();
    if (impl == 2) {
      int bn = bn_override;
      if (bn <= 0) { const char* e = getenv("APLA_GEMM_BN"); bn = e ? atoi(e) : 0; }
      return gemm2_tn(epi, A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    }
  }
  GemmEpi ep{out, out2, bias, gamma, aux, nullptr, ldo, N};
  switch (epi) {
    case EPI_BIAS: return dispatch_tn<EPI_BIAS>(A, B, M, N, K, lda, ldb, ep, stream, bn_override);
    case EPI_BIAS_GELU:
      APLA_CHECK(out2 != nullptr, "gemm_tn: EPI_BIAS_GELU needs out2");
      return dispatch_tn<EPI_BIAS_GELU>(A, B, M, N, K, lda, ldb, ep, stream, bn_override);
    case EPI_RESID:
      APLA_CHECK(aux != nullptr, "gemm_tn: EPI_RESID needs the residual in aux");
      return dispatch_tn<EPI_RESID>(A, B, M, N, K, lda, ldb, ep, stream, bn_override);
    case EPI_GELU_BWD:
      APLA_CHECK(aux != nullptr, "gemm_tn: EPI_GELU_BWD needs the pre-activation in aux");
      return dispatch_tn<EPI_GELU_BWD>(A, B, M, N, K, lda, ldb, ep, stream, bn_override);
  }
  set_error("gemm_tn: unknown epilogue %d", epi);
  return 1;
}

int gemm_resid_scaled(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                      const float* gamma, const float* resid, int ldo, const float* row_scale, int rows_per_scale,
                      cudaStream_t stream) {
  APLA_CHECK(M > 0 && N > 0 && K > 0, "gemm_resid_scaled: empty problem %dx%dx%d", M, N, K);
  APLA_CHECK(N % 32 == 0, "gemm_resid_scaled: N=%d must be a multiple of 32", N);
  APLA_CHECK(K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldo % 8 == 0,
             "gemm_resid_scaled: K/lda/ldb/ldo (%d/%d/%d/%d) must be multiples of 8", K, lda, ldb, ldo);
  APLA_CHECK(resid != nullptr && row_scale != nullptr && rows_per_scale >= 1,
             "gemm_resid_scaled: needs the residual, the row scales and rows_per_scale >= 1 (got %d)", rows_per_scale);
  static const int impl = [] { const char* e = getenv("APLA_GEMM_IMPL"); return e ? atoi(e) : 2; }();
  APLA_CHECK(impl == 2, "gemm_resid_scaled: the row-scaled residual epilogue exists in the 2-CTA kernel only; "
             "APLA_GEMM_IMPL=%d selects the 1-CTA kernel", impl);
  const char* e = getenv("APLA_GEMM_BN");
  return gemm2_resid_scaled(A, B, M, N, K, lda, ldb, out, bias, gamma, resid, ldo, row_scale, rows_per_scale, stream,
                            e ? atoi(e) : 0);
}

int gemm_resid_ln(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                  const float* gamma, const float* resid, int ldo, const float* ln_w, const float* ln_b, void* ln_out,
                  int ld_ln, float eps, cudaStream_t stream, int fuse_mode, const float* row_scale, int rows_per_scale) {
  // fuse_mode: 1 = one launch, 0 = two launches, < 0 = default, which is one launch only with APLA_GEMM_LN_FUSE=1.  Measured on the C2 step (B200, 50 steps): 8.69 ms fused against 7.93 ms with
  // the two launches -- results bit-identical, but the LayerNorm of a slab lands on the epilogue warps of whichever CTA
  // finishes the slab's last column tile, and those warps are what the K = 768 residual GEMM is already bound by (tensor
  // pipe 36 % busy); the stand-alone row kernel at full occupancy streams the same bytes at 6.3 TB/s.  Kept as an option.
  static const bool fuse = [] { const char* e = getenv("APLA_GEMM_LN_FUSE"); return e && atoi(e) != 0; }();
  static const int impl = [] { const char* e = getenv("APLA_GEMM_IMPL"); return e ? atoi(e) : 2; }();
  const bool want = fuse_mode < 0 ? fuse : fuse_mode != 0;
  if (row_scale) {
    APLA_CHECK(!want, "gemm_resid_ln: the one-launch residual + LayerNorm epilogue (APLA_GEMM_LN_FUSE=1) has no row-scaled "
               "form; unset APLA_GEMM_LN_FUSE to train with drop path");
    if (int rc = gemm_resid_scaled(A, B, M, N, K, lda, ldb, out, bias, gamma, resid, ldo, row_scale, rows_per_scale, stream))
      return rc;
    return layernorm_fwd(out, ldo, ln_w, ln_b, ln_out, ld_ln, M, N, eps, stream);
  }
  if (want && impl == 2 && gemm2_resid_ln_supported(N) && K % 8 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldo % 8 == 0)
    return gemm2_resid_ln(A, B, M, N, K, lda, ldb, out, bias, gamma, resid, ldo, ln_w, ln_b, ln_out, ld_ln, eps, stream);
  if (int rc = gemm_tn(EPI_RESID, A, B, M, N, K, lda, ldb, out, nullptr, bias, gamma, resid, ldo, stream, 0)) return rc;
  return layernorm_fwd(out, ldo, ln_w, ln_b, ln_out, ld_ln, M, N, eps, stream);
}

// Weight gradient  dW[rowmap(n), m] += sum_k A[k, m] * B[k, n]   (A = layer input X [K=T, M=D_in],
// B = output gradient dY [K=T, N]); fp32 atomics over k_splits partial sums, dW must be zero-initialised.
int gemm_wgrad_nt(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* dW, int ldw,
                  const int* rowmap, int n_valid, cudaStream_t stream) {
  APLA_CHECK(M > 0 && N > 0 && K > 0, "gemm_wgrad_nt: empty problem %dx%dx%d", M, N, K);
  APLA_CHECK(M % 64 == 0 && N % 64 == 0, "gemm_wgrad_nt: M=%d and N=%d must be multiples of 64", M, N);
  APLA_CHECK(lda % 8 == 0 && ldb % 8 == 0, "gemm_wgrad_nt: lda/ldb must be multiples of 8");
  const int bn = N % 256 == 0 ? 256 : (N % 128 == 0 ? 128 : 64);
  const int mn_tiles = cdiv(M, BM) * cdiv(N, bn);
  const int num_kb = cdiv(K, BK);
  int splits = sm_count() / mn_tiles;
  if (splits < 1) splits = 1;
  if (splits > num_kb) splits = num_kb;
  // every split must own at least one k-block
  while (splits > 1 && (splits - 1) * cdiv(num_kb, splits) >= num_kb) --splits;
  GemmEpi ep{dW, nullptr, nullptr, nullptr, nullptr, rowmap, ldw, n_valid};
  switch (bn) {
    case 256: return launch<256, EPI_F32_T, true, true>(A, B, M, N, K, lda, ldb, splits, ep, stream);
    case 128: return launch<128, EPI_F32_T, true, true>(A, B, M, N, K, lda, ldb, splits, ep, stream);
    default: return launch<64, EPI_F32_T, true, true>(A, B, M, N, K, lda, ldb, splits, ep, stream);
  }
}

}  // namespace apla
