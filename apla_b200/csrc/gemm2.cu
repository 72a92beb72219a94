// 2-CTA (cta_group::2) persistent tcgen05 GEMM with TMA-store epilogues -- the main GEMM of the step.
//
//   D[M,N] = A[M,K] * B[N,K]^T, bf16 operands, fp32 accumulation in TMEM, 256 x BN tile per CTA pair.
//
// Each CTA of a 2-CTA cluster loads its own 128 rows of A and its own half of the B tile by TMA (128B swizzle); the
// leader CTA's single MMA thread issues tcgen05.mma.cta_group::2 (M=256) that reads both CTAs' shared memory and
// writes both CTAs' TMEM, so every operand byte in shared memory feeds twice the math of a 1-CTA MMA.  Pipelines:
//   smem ring   (TMA -> MMA)   full[] on the leader (tx bytes of both CTAs), empty[] per CTA via multicast commit
//   TMEM ring   (MMA -> epilogue) two accumulator stages; tfull[] per CTA via multicast commit, tempty[] on the leader
//   epilogue    8 warps per CTA; each warp owns a private 2 x 4 KB swizzled staging ring: auxiliary tiles (residual /
//               saved pre-activation) arrive by TMA load one chunk ahead, results leave by TMA store, so global
//               memory only ever sees full 128-byte rows (the first version of this kernel wrote registers straight
//               to global memory, 32 rows per instruction, and was LSU-wavefront-bound in every fused epilogue).
// Epilogues: see kernels.cuh / gemm.cu header (EPI_BIAS, EPI_BIAS_GELU, EPI_RESID, EPI_GELU_BWD), plus
//   EPI_BIAS_GELU_D  h = acc + bias[n] (fp32, not stored);  out_f16 = gelu_erf'(h);  out2_bf16 = gelu_erf(h)
//   EPI_BIAS_GELU_G  out_bf16 = gelu_erf(acc + bias[n]), bit-identical to out2 of EPI_BIAS_GELU_D: the forward-only
//                    fc1, with the EPI_BIAS data path (one 128-byte staging row and one TMA store per 64-column chunk)
//   EPI_MUL_F16      out_bf16 = acc * aux_f16[m,n]   (fc2 dgrad times the saved GELU derivative)
//   EPI_RESID_LN     EPI_RESID, then the LayerNorm that reads the new residual stream: the CTA that completes the LAST
//                    column tile of a 128-row slab (a self-resetting arrival counter per slab in global memory)
//                    re-reads the slab -- still in L2 -- and writes bf16((x - mean) * rstd * w + b), the A operand of
//                    the next GEMM.  Same arithmetic as ln_fwd_kernel (rowwise.cu), minus its launch and its DRAM pass.
//   EPI_RESID_SCALED  out_f32 = aux_f32[m,n] + row_scale[m / rows_per_scale] * gamma[n] * (acc + bias[n]): EPI_RESID
//                    with one scale per group of rows (stochastic depth: per image; 0 or 1/keep), folded into gamma, so
//                    a scale of 1 gives EPI_RESID's bits
//   EPI_DELTA  out_bf16 = acc;  rowstat[m, n/64] = sum over the 64-wide head of bf16(acc) * aux_bf16[m, n]
//              (attention-projection dgrad fused with FlashAttention's delta = rowsum(dO * O); one staging chunk is
//              exactly one head and one thread owns one row of it, so the reduction needs no shuffles).
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

#include <stdlib.h>

namespace apla {
namespace g2 {

constexpr int BM = 128;  // rows per CTA; the CTA pair computes 256
constexpr int BK = 64;
constexpr int kEpiWarps = 8;
constexpr int kThreads = 64 + kEpiWarps * 32;
constexpr uint32_t kStgBuf = 4096;  // one staging buffer: 32 rows x 128 B

template <int BN>
struct Cfg {
  static constexpr uint32_t kABytes = BM * BK * 2;
  static constexpr uint32_t kBBytes = (BN / 2) * BK * 2;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = BN == 256 ? 5 : 6;
  static constexpr uint32_t kStagingBytes = kEpiWarps * 2 * kStgBuf;
  static constexpr uint32_t kTmemCols = 2 * BN;
  static constexpr size_t kSmemBytes = 1024 + size_t(kStages) * kStageBytes + kStagingBytes + 512;
};

__device__ __forceinline__ uint32_t stg_addr(uint32_t buf, int row, int chunk) {
  return buf + row * 128 + ((chunk ^ (row & 7)) << 4);
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t mapa_rank0(uint32_t addr) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(addr));
  return r;
}

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory"); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// arguments of the epilogues beyond the GEMM's: the LayerNorm of EPI_RESID_LN, the row scales of EPI_RESID_SCALED
struct LnArgs {
  const float* x;   // the fp32 output of this GEMM (read back by generic loads)
  int64_t ldx;
  const float* w;
  const float* b;
  __nv_bfloat16* out;
  int* counters;   // [row slabs of 128] arrival counters, zero between launches (the last arriver resets its slab's)
  int ld;
  float eps;
  const float* row_scale;   // EPI_RESID_SCALED: row m is scaled by row_scale[m / rows_per_scale]
  int rows_per_scale;
};

// LayerNorm of `nrows` consecutive rows (two at a time: the loads of both are in flight together) by one warp;
// D = NV * 128.  ld.global.cg: the rows were just written through L2 by TMA stores of this and other CTAs.
template <int NV>
__device__ __forceinline__ void ln_rows(const LnArgs& ln, int row0, int nrows, int M, int lane) {
  const float* x = ln.x;
  const int64_t ldx = ln.ldx;
  constexpr float inv_d = 1.f / float(NV * 128);
  for (int r = 0; r < nrows; r += 2) {
    float4 v[2][NV];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int row = row0 + r + t;
      const float4* xr = reinterpret_cast<const float4*>(x + int64_t(row) * ldx);
#pragma unroll
      for (int i = 0; i < NV; ++i) v[t][i] = (row < M && r + t < nrows) ? __ldcg(xr + lane + 32 * i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int row = row0 + r + t;
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) s += v[t][i].x + v[t][i].y + v[t][i].z + v[t][i].w;
      const float mean = warp_sum(s) * inv_d;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        v[t][i].x -= mean; v[t][i].y -= mean; v[t][i].z -= mean; v[t][i].w -= mean;
        q += v[t][i].x * v[t][i].x + v[t][i].y * v[t][i].y + v[t][i].z * v[t][i].z + v[t][i].w * v[t][i].w;
      }
      const float rstd = rsqrtf(warp_sum(q) * inv_d + ln.eps);
      if (row < M && r + t < nrows) {
        uint2* yr = reinterpret_cast<uint2*>(ln.out + int64_t(row) * ln.ld);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const float4 ww = __ldg(reinterpret_cast<const float4*>(ln.w) + lane + 32 * i);
          const float4 bb = __ldg(reinterpret_cast<const float4*>(ln.b) + lane + 32 * i);
          yr[lane + 32 * i] = make_uint2(pack_bf16(v[t][i].x * rstd * ww.x + bb.x, v[t][i].y * rstd * ww.y + bb.y),
                                         pack_bf16(v[t][i].z * rstd * ww.z + bb.z, v[t][i].w * rstd * ww.w + bb.w));
        }
      }
    }
  }
}

template <int BN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
             const __grid_constant__ CUtensorMap tma_out, const __grid_constant__ CUtensorMap tma_out2,
             const __grid_constant__ CUtensorMap tma_aux, int M, int N, int K, const float* __restrict__ bias,
             const float* __restrict__ gamma, float* __restrict__ rowstat, const LnArgs ln) {
  using C = Cfg<BN>;
  constexpr int kStages = C::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + kStages * C::kStageBytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(staging + C::kStagingBytes);
  uint64_t* empty = full + kStages;
  uint64_t* tfull = empty + kStages;
  uint64_t* tempty = tfull + 2;
  uint64_t* aux_full = tempty + 2;  // [kEpiWarps][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aux_full + 2 * kEpiWarps);
  [[maybe_unused]] volatile uint32_t* ln_flag = tmem_slot + 1;   // EPI_RESID_LN: "this CTA completed the slab"

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = ((M + 2 * BM - 1) / (2 * BM)) * num_n;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    tma_prefetch_desc(&tma_out);
    if constexpr (EPI == EPI_BIAS_GELU || EPI == EPI_BIAS_GELU_D) tma_prefetch_desc(&tma_out2);
    if constexpr (EPI == EPI_RESID || EPI == EPI_RESID_LN || EPI == EPI_RESID_SCALED || EPI == EPI_GELU_BWD || EPI == EPI_DELTA || EPI == EPI_MUL_F16) tma_prefetch_desc(&tma_aux);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull[a], 1);
      mbar_init(&tempty[a], 2 * kEpiWarps);  // epilogue warps of BOTH CTAs release the accumulator (leader's copy is used)
    }
    for (int i = 0; i < 2 * kEpiWarps; ++i) mbar_init(&aux_full[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc<2>(tmem_slot, C::kTmemCols);
    tmem_relinquish<2>();
  }
  tc_fence_before();
  cluster_sync_all();  // barrier inits of both CTAs are visible before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        const int m0 = (tile / num_n) * (2 * BM) + int(cta_rank) * BM;
        const int n0 = (tile % num_n) * BN + int(cta_rank) * (BN / 2);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * C::kStageBytes;
          uint8_t* sb = sa + C::kABytes;
          const uint32_t full_leader = mapa_rank0(smem_u32(&full[stage]));
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * C::kStageBytes);
          tma_load_2d_2sm(sa, &tma_a, full_leader, kb * BK, m0);
          tma_load_2d_2sm(sb, &tma_b, full_leader, kb * BK, n0);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * BM, BN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        mbar_wait_cluster(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait_cluster(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_base = smem_u32(smem + stage * C::kStageBytes);
          const uint32_t b_base = a_base + C::kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adesc = make_sdesc_sw128(a_base + k * 32, 16, 1024);
            const uint64_t bdesc = make_sdesc_sw128(b_base + k * 32, 16, 1024);
            umma_bf16<2>(d_tmem, adesc, bdesc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit_2sm(&empty[stage], 3);  // frees this smem stage in both CTAs
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&tfull[as], 3);  // accumulator ready in both CTAs
        as ^= 1;
        if (as == 0) aphase ^= 1;
      }
    }
  } else {
    // ===================== epilogue warps (both CTAs) =====================
    constexpr bool kLN = (EPI == EPI_RESID_LN);
    constexpr bool kF32 = (EPI == EPI_RESID || kLN || EPI == EPI_RED || EPI == EPI_RESID_SCALED);
    constexpr bool kAux = (EPI == EPI_RESID || kLN || EPI == EPI_RESID_SCALED || EPI == EPI_GELU_BWD || EPI == EPI_DELTA ||
                           EPI == EPI_MUL_F16);
    constexpr bool kBias = (EPI != EPI_GELU_BWD && EPI != EPI_DELTA && EPI != EPI_MUL_F16);
    constexpr bool kTwoOut = (EPI == EPI_BIAS_GELU || EPI == EPI_BIAS_GELU_D);
    // the bias is read at its use, not one sub-load ahead: the prefetch holds 32 registers, which the LayerNorm and the
    // row scale need (without this, both spill)
    constexpr bool kBiasAtUse = (kLN || EPI == EPI_RESID_SCALED);
    // the GELU epilogues in packed fp32 add the bias inside gelu_erf_both_x2, not to the accumulator beforehand
    constexpr bool kGeluX2 = (EPI == EPI_BIAS_GELU_D || EPI == EPI_BIAS_GELU_G);
    // columns per chunk: one 128-byte staging row, except the two-output GELU epilogue which packs a 64-byte row of
    // each output (h | g) into one 4 KB buffer (64B swizzle) so that chunks can still ping-pong between buffers
    constexpr int CW = (kF32 || kTwoOut) ? 32 : 64;
    constexpr int NCH = BN / CW / 2;         // chunks per warp per tile
    constexpr int SUBS = CW / 32;            // 32-column TMEM loads per chunk
    constexpr int NSUB = NCH * SUBS;
    const int ew = warp - 2;
    const int q = warp & 3;                  // TMEM lane quarter of this warp
    const int half = ew >> 2;
    const uint32_t stg = smem_u32(staging + ew * 2 * kStgBuf);
    uint64_t* abar = aux_full + ew * 2;
    uint32_t aux_phase = 0;
    uint32_t cnt = 0;  // running chunk counter: staging buffer = cnt & 1 (alternates across tiles too)
    int as = 0;
    uint32_t aphase = 0;
    // EPI_RESID_LN: the arrival for a tile's 128-row slab is made one tile late (or at the end), when its stores have
    // drained anyway; whoever brings a slab's count to num_n normalises it.
    [[maybe_unused]] int pend_slab = -1;
    for (int tile = cluster_id; kLN || tile < num_tiles; tile += num_clusters) {
      const int row0 = (tile / num_n) * (2 * BM) + int(cta_rank) * BM + q * 32;  // this warp's 32-row slab
      const int n0 = (tile % num_n) * BN;
      // 32-column sub-loads of this warp that lie inside the matrix (warp-uniform; N % 32 == 0)
      int nvalid = 0;
      if (row0 < M && tile < num_tiles) {
#pragma unroll
        for (int i = 0; i < NSUB; ++i) nvalid += (n0 + (half + 2 * (i / SUBS)) * CW + (i % SUBS) * 32 < N) ? 1 : 0;
      }
      if constexpr (kAux) {
        // first chunk's auxiliary tile travels while the MMAs of this tile are still running
        if (nvalid > 0 && lane == 0) {
          const uint32_t b0 = cnt & 1;
          tma_store_wait_read<0>();
          mbar_arrive_expect_tx(&abar[b0], kStgBuf);
          tma_load_2d(reinterpret_cast<void*>(staging + ew * 2 * kStgBuf + b0 * kStgBuf), &tma_aux, &abar[b0],
                      n0 + half * CW, row0);
        }
      }
      if constexpr (kLN) {
        // (one call site, written out: a lambda called from two places was not inlined and put its captures in local memory)
        if (pend_slab >= 0) {
          const int slab = pend_slab;
          if (lane == 0) {
            tma_store_wait<0>();                                   // this warp's rows of the slab are in global memory
            asm volatile("fence.proxy.async.global;" ::: "memory");
            __threadfence();
          }
          __syncwarp();
          epi_bar_sync();
          if (ew == 0 && lane == 0) {
            const int old = atomicAdd(ln.counters + slab, 1);
            const bool last = old == num_n - 1;
            if (last) ln.counters[slab] = 0;                        // ready for the next launch
            __threadfence();
            *ln_flag = last ? 1u : 0u;
          }
          epi_bar_sync();
          if (*ln_flag != 0) {   // rewritten only behind the next epi_bar_sync, which every warp reaches after this read
            const int r0 = slab * BM + ew * (BM / kEpiWarps);
            switch (N >> 7) {
              case 3: ln_rows<3>(ln, r0, BM / kEpiWarps, M, lane); break;
              case 6: ln_rows<6>(ln, r0, BM / kEpiWarps, M, lane); break;
              default: ln_rows<8>(ln, r0, BM / kEpiWarps, M, lane); break;
            }
          }
        }
        if (tile >= num_tiles) break;
        pend_slab = (tile / num_n) * 2 + int(cta_rank);
      }
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(as * BN + half * CW);
      // The accumulator is read in a two-deep software pipeline: the tcgen05.ld (and the bias fetch) of sub-load
      // i+1 is in flight while sub-load i goes through the epilogue math, and the TMEM stage goes back to the MMA
      // thread as soon as the LAST sub-load has landed in registers -- not after the math and stores of the tile.
      uint32_t v[2][32];
      [[maybe_unused]] float4 bb[8];   // bias of the NEXT sub-load, fetched right after the current one is consumed
      if constexpr (kGeluX2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) bb[i] = make_float4(0.f, 0.f, 0.f, 0.f);   // stays zero when there is no bias
      }
      if (nvalid > 0) {
        tmem_ld_32x32(t_base, v[0]);
        if constexpr (kBias && !kBiasAtUse) {
          if (bias) {
#pragma unroll
            for (int i = 0; i < 8; ++i) bb[i] = __ldg(reinterpret_cast<const float4*>(bias + n0 + half * CW) + i);
          }
        }
      } else {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster_relaxed(&tempty[as], 0);
      }
      [[maybe_unused]] float dot = 0.f;  // EPI_DELTA: this row's sum over the chunk (= one 64-wide head)
      int b = 0;
      uint32_t buf = stg;
#pragma unroll
      for (int idx = 0; idx < NSUB; ++idx) {
        if (idx < nvalid) {
          const int j = idx / SUBS, s = idx % SUBS;
          const int cidx = half + 2 * j;
          const int col0 = n0 + cidx * CW;
          if (s == 0) {
            b = int(cnt & 1);
            ++cnt;
            buf = stg + b * kStgBuf;
            if constexpr (kAux) {
              if (j + 1 < NCH && col0 + 2 * CW < N && lane == 0) {
                tma_store_wait_read<0>();  // the other buffer's last store has drained
                mbar_arrive_expect_tx(&abar[b ^ 1], kStgBuf);
                tma_load_2d(reinterpret_cast<void*>(staging + ew * 2 * kStgBuf + (b ^ 1) * kStgBuf), &tma_aux,
                            &abar[b ^ 1], col0 + 2 * CW, row0);
              }
              mbar_wait(&abar[b], (aux_phase >> b) & 1);
              aux_phase ^= (1u << b);
            } else {
              if (lane == 0) tma_store_wait_read<1>();  // the store issued two chunks ago (same buffer) has drained
              __syncwarp();
            }
            dot = 0.f;
          }
          tmem_ld_wait_regs(v[idx & 1]);
          if (idx + 1 < NSUB && idx + 1 < nvalid) {
            const int j1 = (idx + 1) / SUBS, s1 = (idx + 1) % SUBS;
            tmem_ld_32x32(t_base + uint32_t(2 * j1 * CW + s1 * 32), v[(idx + 1) & 1]);
          }
          if (idx + 1 == nvalid) {
            // every tcgen05.ld of this tile has completed: hand the accumulator stage back to the leader's MMA thread
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster_relaxed(&tempty[as], 0);
          }
          float x[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(v[idx & 1][i]);
          const int col = col0 + s * 32;
          [[maybe_unused]] float bv[32];   // the GELU epilogues add the bias inside their packed-fp32 math
          if constexpr (kBias) {
            if constexpr (kGeluX2) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 t4 = bb[i];
                bv[4 * i] = t4.x; bv[4 * i + 1] = t4.y; bv[4 * i + 2] = t4.z; bv[4 * i + 3] = t4.w;
              }
            }
            if (bias) {
              if constexpr (kBiasAtUse) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float4 t4 = __ldg(reinterpret_cast<const float4*>(bias + col) + i);
                  x[4 * i] += t4.x; x[4 * i + 1] += t4.y; x[4 * i + 2] += t4.z; x[4 * i + 3] += t4.w;
                }
              } else if constexpr (!kGeluX2) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const float4 t4 = bb[i];
                  x[4 * i] += t4.x; x[4 * i + 1] += t4.y; x[4 * i + 2] += t4.z; x[4 * i + 3] += t4.w;
                }
              }
              if (!kBiasAtUse && idx + 1 < NSUB && idx + 1 < nvalid) {
                const int j1 = (idx + 1) / SUBS, s1 = (idx + 1) % SUBS;
                const float4* b4 = reinterpret_cast<const float4*>(bias + n0 + (half + 2 * j1) * CW + s1 * 32);
#pragma unroll
                for (int i = 0; i < 8; ++i) bb[i] = __ldg(b4 + i);
              }
            }
          }
          if constexpr (EPI == EPI_BIAS) {
#pragma unroll
            for (int c = 0; c < 4; ++c)
              sts128(stg_addr(buf, lane, 4 * s + c), pack_bf16(x[8 * c], x[8 * c + 1]), pack_bf16(x[8 * c + 2], x[8 * c + 3]),
                     pack_bf16(x[8 * c + 4], x[8 * c + 5]), pack_bf16(x[8 * c + 6], x[8 * c + 7]));
          } else if constexpr (EPI == EPI_BIAS_GELU) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t h[4], g[4];
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                h[t] = pack_bf16(x[8 * c + 2 * t], x[8 * c + 2 * t + 1]);
                g[t] = pack_bf16(gelu_erf(bf16_lo(h[t])), gelu_erf(bf16_hi(h[t])));
              }
              const uint32_t off = lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4);   // 64B-swizzled row of 32 bf16
              sts128(buf + off, h[0], h[1], h[2], h[3]);
              sts128(buf + kStgBuf / 2 + off, g[0], g[1], g[2], g[3]);
            }
          } else if constexpr (EPI == EPI_BIAS_GELU_D) {
            // saves gelu'(h) in fp16 (|gelu'| <= 1.13: 11 mantissa bits, better than gelu' of a bf16-rounded h) so that the
            // fc2 input-gradient epilogue is one multiply; this epilogue is store-bound, the extra math is hidden
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t dd[4], g[4];
#pragma unroll
              for (int t = 0; t < 4; ++t)
                gelu_erf_both_x2(x[8 * c + 2 * t], x[8 * c + 2 * t + 1], bv[8 * c + 2 * t], bv[8 * c + 2 * t + 1], g[t], dd[t]);
              const uint32_t off = lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4);   // 64B-swizzled row of 32 x 2 bytes
              sts128(buf + off, dd[0], dd[1], dd[2], dd[3]);
              sts128(buf + kStgBuf / 2 + off, g[0], g[1], g[2], g[3]);
            }
          } else if constexpr (EPI == EPI_BIAS_GELU_G) {
            // the same packed-fp32 evaluation as EPI_BIAS_GELU_D, so that g is bit-identical to the training forward's;
            // the instructions that only feed the derivative are dead and the compiler drops them
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint32_t g[4], dd;
#pragma unroll
              for (int t = 0; t < 4; ++t)
                gelu_erf_both_x2(x[8 * c + 2 * t], x[8 * c + 2 * t + 1], bv[8 * c + 2 * t], bv[8 * c + 2 * t + 1], g[t], dd);
              sts128(stg_addr(buf, lane, 4 * s + c), g[0], g[1], g[2], g[3]);
            }
          } else if constexpr (EPI == EPI_MUL_F16) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint32_t a = stg_addr(buf, lane, 4 * s + c);
              const uint4 hv = lds128(a);
              const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
              uint32_t d[4];
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 m = unpack_f16(hw[t]);
                d[t] = pack_bf16(x[8 * c + 2 * t] * m.x, x[8 * c + 2 * t + 1] * m.y);
              }
              sts128(a, d[0], d[1], d[2], d[3]);
            }
          } else if constexpr (EPI == EPI_RED) {
            // out += gamma * (acc + bias): the residual never enters shared memory, the L2 adds (TMA reduce)
            const float4* g4 = reinterpret_cast<const float4*>(gamma ? gamma + col : nullptr);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float4 g = gamma ? __ldg(g4 + c) : make_float4(1.f, 1.f, 1.f, 1.f);
              sts128(stg_addr(buf, lane, c), __float_as_uint(g.x * x[4 * c]), __float_as_uint(g.y * x[4 * c + 1]),
                     __float_as_uint(g.z * x[4 * c + 2]), __float_as_uint(g.w * x[4 * c + 3]));
            }
          } else if constexpr (EPI == EPI_RESID || EPI == EPI_RESID_LN || EPI == EPI_RESID_SCALED) {
            const float4* g4 = reinterpret_cast<const float4*>(gamma ? gamma + col : nullptr);
            // EPI_RESID_SCALED: the scale of this thread's row (lane = row of the slab), read at its use -- holding it
            // across the tile costs a register this kernel does not have
            [[maybe_unused]] float rscale = 0.f;
            if constexpr (EPI == EPI_RESID_SCALED) {
              if (row0 + lane < M) rscale = __ldg(ln.row_scale + (row0 + lane) / ln.rows_per_scale);
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const uint32_t a = stg_addr(buf, lane, c);
              const uint4 rv = lds128(a);
              float4 g = gamma ? __ldg(g4 + c) : make_float4(1.f, 1.f, 1.f, 1.f);
              if constexpr (EPI == EPI_RESID_SCALED) {
                g.x *= rscale; g.y *= rscale; g.z *= rscale; g.w *= rscale;
              }
              sts128(a, __float_as_uint(__uint_as_float(rv.x) + g.x * x[4 * c]),
                     __float_as_uint(__uint_as_float(rv.y) + g.y * x[4 * c + 1]),
                     __float_as_uint(__uint_as_float(rv.z) + g.z * x[4 * c + 2]),
                     __float_as_uint(__uint_as_float(rv.w) + g.w * x[4 * c + 3]));
            }
          } else if constexpr (EPI == EPI_GELU_BWD) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint32_t a = stg_addr(buf, lane, 4 * s + c);
              const uint4 hv = lds128(a);
              const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
              uint32_t d[4];
#pragma unroll
              for (int t = 0; t < 4; ++t)
                d[t] = pack_bf16(x[8 * c + 2 * t] * gelu_erf_grad(bf16_lo(hw[t])),
                                 x[8 * c + 2 * t + 1] * gelu_erf_grad(bf16_hi(hw[t])));
              sts128(a, d[0], d[1], d[2], d[3]);
            }
          } else if constexpr (EPI == EPI_DELTA) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const uint32_t a = stg_addr(buf, lane, 4 * s + c);
              const uint4 ov = lds128(a);
              const uint32_t ow[4] = {ov.x, ov.y, ov.z, ov.w};
              uint32_t d[4];
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                d[t] = pack_bf16(x[8 * c + 2 * t], x[8 * c + 2 * t + 1]);
                dot = fmaf(bf16_lo(d[t]), bf16_lo(ow[t]), dot);   // the rounded dO the attention backward will read
                dot = fmaf(bf16_hi(d[t]), bf16_hi(ow[t]), dot);
              }
              sts128(a, d[0], d[1], d[2], d[3]);
            }
          }
          if (s == SUBS - 1 || idx + 1 == nvalid) {
            if constexpr (EPI == EPI_DELTA) {
              if (row0 + lane < M) rowstat[size_t(row0 + lane) * (N >> 6) + (col0 >> 6)] = dot;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if constexpr (kTwoOut) {
                const uint8_t* sb = staging + ew * 2 * kStgBuf + b * kStgBuf;
                tma_store_2d(&tma_out, reinterpret_cast<const void*>(sb), col0, row0);
                tma_store_2d(&tma_out2, reinterpret_cast<const void*>(sb + kStgBuf / 2), col0, row0);
              } else if constexpr (EPI == EPI_RED) {
                tma_reduce_add_2d(&tma_out, reinterpret_cast<const void*>(staging + ew * 2 * kStgBuf + b * kStgBuf), col0, row0);
              } else {
                tma_store_2d(&tma_out, reinterpret_cast<const void*>(staging + ew * 2 * kStgBuf + b * kStgBuf), col0, row0);
              }
              tma_store_commit();
            }
          }
        }
      }
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
    if (lane == 0) tma_store_wait<0>();
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync_all();  // the peer's smem / TMEM stay alive until every MMA and remote arrive has landed
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<2>(tmem_base, C::kTmemCols);
  }
}

template <int BN, int EPI>
static int launch(const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
                  const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream,
                  const LnArgs& ln = LnArgs{}) {
  float* rowstat = EPI == EPI_DELTA ? reinterpret_cast<float*>(out2) : nullptr;
  using C = Cfg<BN>;
  CUtensorMap ta, tb, to, to2, tx;
  if (int rc = make_tmap_2d(&ta, A, 2, M, K, lda, BM, BK, true)) return rc;
  if (int rc = make_tmap_2d(&tb, B, 2, N, K, ldb, BN / 2, BK, true)) return rc;
  constexpr int oelt = (EPI == EPI_RESID || EPI == EPI_RESID_LN || EPI == EPI_RESID_SCALED || EPI == EPI_RED) ? 4 : 2;
  if (EPI == EPI_BIAS_GELU || EPI == EPI_BIAS_GELU_D) {
    if (int rc = make_tmap_2d_sw(&to, out, 2, M, N, ldo, 32, 32, 64)) return rc;
    if (int rc = make_tmap_2d_sw(&to2, out2, 2, M, N, ldo, 32, 32, 64)) return rc;
  } else {
    if (int rc = make_tmap_2d(&to, out, oelt, M, N, ldo, 32, 128 / oelt, true)) return rc;
    to2 = to;
  }
  tx = to;
  if (EPI == EPI_RESID || EPI == EPI_RESID_LN || EPI == EPI_RESID_SCALED || EPI == EPI_GELU_BWD || EPI == EPI_DELTA ||
      EPI == EPI_MUL_F16)
    if (int rc = make_tmap_2d(&tx, aux, oelt, M, N, ldo, 32, 128 / oelt, true)) return rc;
  auto kern = gemm2_kernel<BN, EPI>;
  static bool attr_set = false;
  if (!attr_set) {
    APLA_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmemBytes));
    attr_set = true;
  }
  const int tiles = cdiv(M, 2 * BM) * cdiv(N, BN);
  const int max_clusters = sm_count() / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  kern<<<2 * clusters, kThreads, C::kSmemBytes, stream>>>(ta, tb, to, to2, tx, M, N, K, bias, gamma, rowstat, ln);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

static int pick_bn(int M, int N) {
  if (N <= 128) return 128;
  const int clusters = sm_count() / 2;
  const int t256 = cdiv(M, 2 * BM) * cdiv(N, 256), t128 = cdiv(M, 2 * BM) * cdiv(N, 128);
  const double c256 = cdiv(t256, clusters) * 1.0, c128 = cdiv(t128, clusters) * 0.76;   // measured: 77.8 vs 51.2 us on 16448x2304x768
  return c128 < c256 ? 128 : 256;
}

template <int EPI>
static int dispatch(const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
                    const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream, int bn) {
  if (bn != 128 && bn != 256) bn = pick_bn(M, N);
  if (bn == 256) return launch<256, EPI>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream);
  return launch<128, EPI>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream);
}

}  // namespace g2

// out_f32 = resid + gamma * (A B^T + bias), ln_out_bf16 = LayerNorm(out_f32; ln_w, ln_b) in the same launch.
bool gemm2_resid_ln_supported(int N) { return N == 384 || N == 768 || N == 1024; }

int gemm2_resid_ln(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                   const float* gamma, const float* resid, int ldo, const float* ln_w, const float* ln_b, void* ln_out,
                   int ld_ln, float eps, cudaStream_t stream) {
  APLA_CHECK(gemm2_resid_ln_supported(N), "gemm2_resid_ln: N=%d is not 384 / 768 / 1024", N);
  APLA_CHECK(ln_w && ln_b && ln_out && resid && ld_ln % 4 == 0 && ldo % 4 == 0, "gemm2_resid_ln: bad LayerNorm arguments");
  // arrival counters, one per 128-row slab: zero at allocation, every launch leaves them zero again.  One allocation per
  // device; launches that use it must be stream-ordered with respect to each other (they are: one step, one stream).
  constexpr int kMaxSlabs = 1 << 16;
  static int* counters[64] = {};
  int dev = 0;
  APLA_CUDA(cudaGetDevice(&dev));
  APLA_CHECK(dev < 64 && cdiv(M, g2::BM) <= kMaxSlabs, "gemm2_resid_ln: device %d / M=%d out of range", dev, M);
  if (!counters[dev]) {
    APLA_CUDA(cudaMalloc(&counters[dev], kMaxSlabs * sizeof(int)));
    APLA_CUDA(cudaMemset(counters[dev], 0, kMaxSlabs * sizeof(int)));
  }
  g2::LnArgs ln{out, int64_t(ldo), ln_w, ln_b, reinterpret_cast<__nv_bfloat16*>(ln_out), counters[dev], ld_ln, eps};
  return g2::launch<256, EPI_RESID_LN>(A, B, M, N, K, lda, ldb, out, nullptr, bias, gamma, resid, ldo, stream, ln);
}

int gemm2_resid_scaled(const void* A, const void* B, int M, int N, int K, int lda, int ldb, float* out, const float* bias,
                       const float* gamma, const float* resid, int ldo, const float* row_scale, int rows_per_scale,
                       cudaStream_t stream, int bn) {
  g2::LnArgs ex{};
  ex.row_scale = row_scale;
  ex.rows_per_scale = rows_per_scale;
  if (bn != 128 && bn != 256) bn = g2::pick_bn(M, N);
  if (bn == 256)
    return g2::launch<256, EPI_RESID_SCALED>(A, B, M, N, K, lda, ldb, out, nullptr, bias, gamma, resid, ldo, stream, ex);
  return g2::launch<128, EPI_RESID_SCALED>(A, B, M, N, K, lda, ldb, out, nullptr, bias, gamma, resid, ldo, stream, ex);
}

int gemm2_tn(int epi, const void* A, const void* B, int M, int N, int K, int lda, int ldb, void* out, void* out2,
             const float* bias, const float* gamma, const void* aux, int ldo, cudaStream_t stream, int bn) {
  switch (epi) {
    case EPI_BIAS: return g2::dispatch<EPI_BIAS>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_BIAS_GELU:
      return g2::dispatch<EPI_BIAS_GELU>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_RESID: return g2::dispatch<EPI_RESID>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_GELU_BWD:
      return g2::dispatch<EPI_GELU_BWD>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_DELTA:
      return g2::dispatch<EPI_DELTA>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_BIAS_GELU_D:
      return g2::dispatch<EPI_BIAS_GELU_D>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_RED:
      return g2::dispatch<EPI_RED>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_MUL_F16:
      return g2::dispatch<EPI_MUL_F16>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
    case EPI_BIAS_GELU_G:
      return g2::dispatch<EPI_BIAS_GELU_G>(A, B, M, N, K, lda, ldb, out, out2, bias, gamma, aux, ldo, stream, bn);
  }
  set_error("gemm2_tn: unknown epilogue %d", epi);
  return 1;
}

}  // namespace apla
