// tcgen05 split-K GEMM with selectable operand majorness:  D[M,N] (f32) = sum_k A(m,k) * B(n,k)
//   A_MN = 0: A is [M,K] row-major (K-major operand)      A_MN = 1: A is [K,M] row-major (MN-major operand)
//   B_MN = 0: B is [N,K] row-major (K-major operand)      B_MN = 1: B is [K,N] row-major (MN-major operand)
// The (1,1) form is the weight gradient of a Linear layer, dW[out,in] = dY[T,out]^T X[T,in] (autograd of F.linear at
// swin_block.py:51,53): the reduction runs over the T tokens, so K is huge and M,N are small -- K is split across
// CTAs, each CTA accumulates its slice in TMEM and writes an f32 partial tile; a fixed-order fold sums the slices
// (deterministic, and f32 all the way, unlike a bf16-output library GEMM).
#include "tc.cuh"

namespace b200 {
namespace tc {
namespace {

constexpr int BM = 128, BN = 128, BK = 64, UK = 16, STAGES = 5;
constexpr int kThreads = 192;
constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
constexpr int ONES_BYTES = 16 * 128;  // [16 n-rows][64 k] K-major tile of 1.0 (swizzle-invariant)
constexpr int SMEM_TOTAL = STAGES * (A_BYTES + B_BYTES) + ONES_BYTES + 256 + 1024;
constexpr int TMEM_COLS = 256;        // BN accumulator columns + 16 for the fused column sums

struct SplitParams {
  float* part;     // [splits][M*N + M]: per split the f32 tile partials followed by the column-sum partials
  int with_cs;     // 1: also produce sum_k A(m,k) (bias gradients)
  int M, N, K, m_tiles, n_tiles, kb_total, kb_per_split, fmt;
};

template <int A_MN, int B_MN>
__global__ void __launch_bounds__(kThreads, 1)
gemm_splitk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, SplitParams P) {
  extern __shared__ unsigned char smem_raw_[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw_) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = smem;
  unsigned char* sB = smem + STAGES * A_BYTES;
  unsigned char* sOnes = smem + STAGES * (A_BYTES + B_BYTES);
  uint64_t* full = reinterpret_cast<uint64_t*>(sOnes + ONES_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x, split = blockIdx.y;
  const int m0 = (tile / P.n_tiles) * BM, n0 = (tile % P.n_tiles) * BN;
  const int kb0 = split * P.kb_per_split;
  const int kb1 = min(kb0 + P.kb_per_split, P.kb_total);

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmA); prefetch_tmap(&tmB);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tfull, 1);
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  const bool do_cs = P.with_cs && n0 == 0;
  const size_t split_stride = (size_t)P.M * P.N + P.M;
  if (do_cs && warp >= 2) {
    const uint32_t one2 = P.fmt == 1 ? 0x3f803f80u : 0x3c003c00u;
    for (int i = threadIdx.x - 64; i < ONES_BYTES / 4; i += 128) reinterpret_cast<uint32_t*>(sOnes)[i] = one2;
    fence_proxy_async();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        mbar_expect_tx(&full[stage], A_BYTES + B_BYTES);
        unsigned char* a = sA + stage * A_BYTES;
        unsigned char* b = sB + stage * B_BYTES;
        if (A_MN) {  // global [K,M]: boxes [64 k-rows][64 m-cols], two of them side by side in M
          tma_load_2d(a, &tmA, &full[stage], m0, kb * BK);
          tma_load_2d(a + BK * 128, &tmA, &full[stage], m0 + 64, kb * BK);
        } else {     // global [M,K]: one box [128 m-rows][64 k-cols]
          tma_load_2d(a, &tmA, &full[stage], kb * BK, m0);
        }
        if (B_MN) {
          tma_load_2d(b, &tmB, &full[stage], n0, kb * BK);
          tma_load_2d(b + BK * 128, &tmB, &full[stage], n0 + 64, kb * BK);
        } else {
          tma_load_2d(b, &tmB, &full[stage], kb * BK, n0);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = idesc_f16(BM, BN, P.fmt, A_MN, B_MN);
      const uint32_t idesc_cs = idesc_f16(BM, 16, P.fmt, A_MN, 0);
      const uint64_t d_ones = smem_desc_k_sw128(sOnes);
      int stage = 0; uint32_t phase = 0;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full[stage], phase);
        fence_after_sync();
        const unsigned char* a = sA + stage * A_BYTES;
        const unsigned char* b = sB + stage * B_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UK; ++k) {
          const uint64_t da = A_MN ? smem_desc_mn_sw128(a + k * UK * 128, BK * 128) : smem_desc_k_sw128(a + k * UK * 2);
          const uint64_t db = B_MN ? smem_desc_mn_sw128(b + k * UK * 128, BK * 128) : smem_desc_k_sw128(b + k * UK * 2);
          umma_f16(tmem_base, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          if (do_cs) umma_f16(tmem_base + BN, da, d_ones, idesc_cs, (kb > kb0 || k > 0) ? 1u : 0u);  // sum_k A(m,k) * 1
        }
        umma_commit(&empty[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      umma_commit(tfull);
    }
  } else {
    const int q = warp & 3, row = q * 32 + lane;
    if (kb1 > kb0) {
      mbar_wait(tfull, 0);
      fence_after_sync();
    }
    const int gm = m0 + row;
    if (do_cs) {  // warp-uniform: tcgen05.ld is .sync.aligned and must be executed by all 32 lanes
      float cs = 0.f;
      if (kb1 > kb0) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + BN, v);
        tmem_ld_wait();
        cs = __uint_as_float(v[0]);
      }
      if (gm < P.M) P.part[(size_t)split * split_stride + (size_t)P.M * P.N + gm] = cs;
    }
    float* dst = P.part + (size_t)split * split_stride + (size_t)gm * P.N + n0;
#pragma unroll 1
    for (int ch = 0; ch < BN / 32; ++ch) {
      uint32_t v[32];
      if (kb1 > kb0) {
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + ch * 32, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0u;
      }
      if (gm < P.M) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int c = n0 + ch * 32 + i * 4;
          if (c + 3 < P.N)
            *reinterpret_cast<uint4*>(dst + ch * 32 + i * 4) = make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          else
            for (int e = 0; e < 4; ++e)
              if (c + e < P.N) dst[ch * 32 + i * 4 + e] = __uint_as_float(v[4 * i + e]);
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) { fence_after_sync(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// out[i] = sum over splits (fixed order); the last `ncs` entries of every split go to `colsum`
__global__ void fold_splits_kernel(const float* __restrict__ part, float* __restrict__ out, float* __restrict__ colsum, int splits,
                                   size_t n, size_t ncs) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n + ncs) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int k = 0;
  for (; k + 3 < splits; k += 4) {
    s0 += part[(size_t)k * (n + ncs) + i];
    s1 += part[(size_t)(k + 1) * (n + ncs) + i];
    s2 += part[(size_t)(k + 2) * (n + ncs) + i];
    s3 += part[(size_t)(k + 3) * (n + ncs) + i];
  }
  for (; k < splits; ++k) s0 += part[(size_t)k * (n + ncs) + i];
  const float s = (s0 + s1) + (s2 + s3);
  if (i < n) out[i] = s;
  else if (colsum) colsum[i - n] = s;
}

int choose_splits(int tiles, int kb_total) {
  int s = (sm_count() + tiles - 1) / tiles;
  if (s > kb_total) s = kb_total;
  if (s > 64) s = 64;
  return s < 1 ? 1 : s;
}

}  // namespace
}  // namespace tc
}  // namespace b200

using namespace b200;
using namespace b200::tc;

extern "C" B200_API size_t b200_gemm_splitk_workspace_bytes(int32_t M, int32_t N, int64_t K) {
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int kb_total = (int)((K + BK - 1) / BK);
  return (size_t)choose_splits(tiles, kb_total) * ((size_t)M * N + M) * sizeof(float);
}

extern "C" B200_API int b200_gemm_splitk(const void* A, const void* B, float* D, float* colsum, void* workspace,
                                         size_t workspace_bytes, int32_t M, int32_t N, int64_t K, int32_t a_mn, int32_t b_mn,
                                         int32_t dtype, void* stream) {
  B200_REQUIRE(dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "gemm_splitk: 16-bit dtypes only");
  B200_REQUIRE(A && B && D && M > 0 && N > 0 && K > 0, B200_ERR_SHAPE, "gemm_splitk: bad arguments");
  B200_REQUIRE(M % 8 == 0 && N % 8 == 0 && K % 8 == 0, B200_ERR_ALIGN, "gemm_splitk: M, N, K must be multiples of 8");
  B200_REQUIRE((((uintptr_t)A | (uintptr_t)B | (uintptr_t)D) & 15) == 0, B200_ERR_ALIGN, "gemm_splitk: 16-byte alignment required");
  const size_t need = b200_gemm_splitk_workspace_bytes(M, N, K);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "gemm_splitk: workspace %zu < %zu", workspace_bytes, need);
  const CUtensorMap* mA = a_mn ? tensor_map_2d(A, (uint64_t)K, (uint64_t)M, (uint64_t)M, BK, 64, dtype)
                               : tensor_map_2d(A, (uint64_t)M, (uint64_t)K, (uint64_t)K, BM, BK, dtype);
  const CUtensorMap* mB = b_mn ? tensor_map_2d(B, (uint64_t)K, (uint64_t)N, (uint64_t)N, BK, 64, dtype)
                               : tensor_map_2d(B, (uint64_t)N, (uint64_t)K, (uint64_t)K, BN, BK, dtype);
  if (!mA || !mB) return B200_ERR_LAUNCH;
  SplitParams P;
  P.part = (float*)workspace; P.M = M; P.N = N; P.K = (int)K;
  P.with_cs = colsum != nullptr;
  P.m_tiles = (M + BM - 1) / BM; P.n_tiles = (N + BN - 1) / BN;
  P.kb_total = (int)((K + BK - 1) / BK);
  const int tiles = P.m_tiles * P.n_tiles;
  const int splits = choose_splits(tiles, P.kb_total);
  P.kb_per_split = (P.kb_total + splits - 1) / splits;
  P.fmt = dtype == B200_BF16 ? 1 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(tiles, splits);
#define LAUNCH_SK(AM, BMN)                                                                        \
  {                                                                                               \
    auto k = gemm_splitk_kernel<AM, BMN>;                                                         \
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL);             \
    k<<<grid, kThreads, SMEM_TOTAL, st>>>(*mA, *mB, P);                                           \
  }
  if (a_mn && b_mn) LAUNCH_SK(1, 1) else if (a_mn) LAUNCH_SK(1, 0) else if (b_mn) LAUNCH_SK(0, 1) else LAUNCH_SK(0, 0)
#undef LAUNCH_SK
  if (int rc = check_launch("gemm_splitk")) return rc;
  const size_t n = (size_t)M * N;
  fold_splits_kernel<<<(unsigned)((n + M + 255) / 256), 256, 0, st>>>((const float*)workspace, D, colsum, splits, n, (size_t)M);
  return check_launch("gemm_splitk_fold");
}
