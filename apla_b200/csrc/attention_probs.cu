// Attention probabilities: probs_f32[B, H, q_rows, N] = exp(scale * q k^T - lse) for the first q_rows queries of each
// of B dense sequences of N tokens -- the `attn` tensor the reference's APLA_Attention.forward returns
// (appla_attn.py:56-60, 83), rebuilt from what the forward already computed: the packed qkv and the natural-log
// log-sum-exp of every query row (attention_tc.cu, attention_fwd_sr.cu, attention_cls.cu).  Because lse is known, each
// probability is one exponential of one score: a single pass over the keys, no online rescale, any N.
//
// Skeleton: the score stage of attention_tc.cu without its P.V half.  One CTA per (sequence, head, 128-query tile):
//   warp 4   TMA producer: the 128x64 Q tile once, then 128-key K tiles out of the packed qkv (128B swizzle, K stages)
//   warp 5   MMA issuer (one thread): S = Q K^T into TMEM, two 128-column accumulators so that tile j+1's MMA runs
//            while the epilogue drains tile j
//   warps 0-3  one TMEM lane (= query row) per thread: tcgen05.ld -> exp2(s scale log2e - lse log2e) in fp32 -> a
//            32x32 fp32 staging tile per warp in shared memory -> coalesced rows, one warp store per 32 keys of a row.
// TMA cannot write the output: a row is N * 4 bytes (1028 B at N = 257), not a multiple of 16.
// Masking: the MMA N is sized to the valid keys (multiple of 16); keys >= N and queries >= q_rows are never stored and
// the lse of a query >= q_rows is never read (with q_rows = 1 only the CLS rows of lse need to exist).
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace apla {
namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr int kThreads = 192;
constexpr int BQ = 128, BK = 128, KSTAGES = 3;
constexpr uint32_t TILE = 128 * 128;                      // 128 rows x 64 bf16
constexpr uint32_t STAGE_STRIDE = 33;                     // floats per staged row: conflict-free row and column access
constexpr uint32_t STAGE_BYTES = 32 * STAGE_STRIDE * 4;   // per epilogue warp
constexpr uint32_t SMEM = 1024 + TILE + KSTAGES * TILE + 4 * STAGE_BYTES + 128;
constexpr uint32_t TMEM_COLS = 2 * BK;

__device__ __forceinline__ uint64_t desc_kmajor(uint32_t base, int k) { return make_sdesc_sw128(base + k * 32, 16, 1024); }

__global__ void __launch_bounds__(kThreads, 2)
attn_probs_kernel(const __grid_constant__ CUtensorMap tma_qk, const float* __restrict__ lse, float* __restrict__ probs,
                  int N, int H, int q_rows, float scale) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = smem + TILE;                                              // [KSTAGES]
  const uint32_t stage_base = smem_u32(smem + TILE + KSTAGES * TILE);     // [4 warps][32][33] fp32
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TILE + KSTAGES * TILE + 4 * STAGE_BYTES);
  uint64_t* bar_q = bars;
  uint64_t* k_full = bars + 1;                  // [KSTAGES]
  uint64_t* k_empty = bars + 1 + KSTAGES;       // [KSTAGES]
  uint64_t* s_full = bars + 1 + 2 * KSTAGES;    // [2]
  uint64_t* s_empty = bars + 3 + 2 * KSTAGES;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5 + 2 * KSTAGES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const int q0 = blockIdx.y * BQ;
  const int row0 = b * N;                       // first token of this sequence in qkv / lse
  const int D = H * 64;
  const int nk = (N + BK - 1) / BK;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tma_qk);
    mbar_init(bar_q, 1);
    for (int i = 0; i < KSTAGES; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_empty[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 5) {
    tmem_alloc<1>(tmem_slot, TMEM_COLS);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      mbar_arrive_expect_tx(bar_q, TILE);
      tma_load_2d(sQ, &tma_qk, bar_q, h * 64, row0 + q0);
      for (int t = 0; t < nk; ++t) {
        const int s = t % KSTAGES;
        mbar_wait(&k_empty[s], ((t / KSTAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&k_full[s], TILE);
        tma_load_2d(sK + s * TILE, &tma_qk, &k_full[s], D + h * 64, row0 + t * BK);
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      mbar_wait(bar_q, 0);
      const uint32_t q_base = smem_u32(sQ);
      for (int t = 0; t < nk; ++t) {
        const int s = t % KSTAGES, buf = t & 1;
        const int valid = min(BK, N - t * BK);
        const uint32_t idesc = make_idesc_bf16(128, (valid + 15) & ~15, 0, 0);
        mbar_wait(&k_full[s], (t / KSTAGES) & 1);
        mbar_wait(&s_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t k_base = smem_u32(sK + s * TILE);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_bf16<1>(tmem + buf * BK, desc_kmajor(q_base, k), desc_kmajor(k_base, k), idesc, k > 0);
        umma_commit(&s_full[buf]);
        umma_commit(&k_empty[s]);
      }
    }
  } else {
    // this warp's 32 query rows; warps whose rows are all >= q_rows only keep the barrier protocol going
    const int wrow0 = q0 + warp * 32;
    const int n_rows = min(32, q_rows - wrow0);
    const uint32_t lane_addr = tmem + (uint32_t(warp * 32) << 16);
    const uint32_t st = stage_base + warp * STAGE_BYTES;
    const float sl2 = scale * LOG2E;
    const float l2 = lane < n_rows ? __ldg(lse + size_t(row0 + wrow0 + lane) * H + h) * LOG2E : 0.f;
    float* out0 = probs + (size_t(blockIdx.x) * q_rows + (n_rows > 0 ? wrow0 : 0)) * size_t(N);
    for (int t = 0; t < nk; ++t) {
      const int buf = t & 1;
      const int valid = min(BK, N - t * BK);
      mbar_wait(&s_full[buf], (t >> 1) & 1);
      tc_fence_after();
      if (n_rows > 0) {
        for (int c = 0; c * 32 < valid; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(lane_addr + buf * BK + c * 32, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) sts_f32(st + (lane * STAGE_STRIDE + j) * 4, exp2f(fmaf(__uint_as_float(v[j]), sl2, -l2)));
          __syncwarp();
          const int key = t * BK + c * 32 + lane;
          if (key < N) {
            float* dst = out0 + key;
            for (int r = 0; r < n_rows; ++r) dst[size_t(r) * N] = lds_f32(st + (r * STAGE_STRIDE + lane) * 4);
          }
          __syncwarp();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[buf]);
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc<1>(tmem, TMEM_COLS);
  }
}

}  // namespace

int attn_probs(const void* qkv, const float* lse, float* probs, int B, int N, int H, int q_rows, float scale,
               cudaStream_t stream) {
  APLA_CHECK(qkv != nullptr && lse != nullptr && probs != nullptr, "apla_attn_probs: null qkv, lse or probs");
  APLA_CHECK(B >= 1 && N >= 1 && H >= 1, "apla_attn_probs: bad shape B=%d N=%d H=%d", B, N, H);
  APLA_CHECK(q_rows >= 1 && q_rows <= N, "apla_attn_probs: q_rows=%d outside [1, N=%d]", q_rows, N);
  APLA_CHECK(int64_t(B) * N <= INT32_MAX, "apla_attn_probs: B=%d N=%d too large", B, N);
  CUtensorMap tm;
  if (int rc = make_tmap_2d(&tm, qkv, 2, uint64_t(B) * N, 3 * H * 64, 3 * H * 64, 128, 64, true)) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    APLA_CUDA(cudaFuncSetAttribute(attn_probs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
    attr_set = true;
  }
  dim3 grid(B * H, cdiv(q_rows, BQ));
  attn_probs_kernel<<<grid, kThreads, SMEM, stream>>>(tm, lse, probs, N, H, q_rows, scale);
  APLA_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace apla
