// tcgen05 GEMM for the SwinBlock's dense contractions:  D[M,N] = epi(A[M,K] * B[N,K]^T + bias[N]).
// Replaces F.linear at swin_block.py:51 (in_proj / out_proj inside nn.MultiheadAttention) and :53 (mlp.0, mlp.2).
//
// Persistent, warp-specialised kernel (one CTA per SM, 320 threads):
//   warp 0   : TMA producer  -- A and B tiles [128|BLOCK_N rows][64 K-elements] with 128-byte swizzle into a
//              STAGES-deep shared-memory ring (mbarrier full/empty pairs)
//   warp 1   : TMEM allocator + MMA issuer -- one elected lane issues tcgen05.mma (cta_group::1, kind::f16,
//              UMMA 128 x BLOCK_N x 16), accumulators in TMEM, double-buffered (2 x BLOCK_N columns) so the
//              epilogue of tile i overlaps the MMAs of tile i+1; tcgen05.commit releases smem slots / signals tiles
//   warps 2-9: epilogue -- tcgen05.ld (lane = row) -> bias / GELU(erf) / residual in registers -> bf16 -> swizzled
//              staging tile in shared memory -> TMA store (rows beyond M are clipped by the tensor map)
// Both operands are K-major (activations [tokens, K]; nn.Linear weights [N, K]) so no transposes are needed.
#include <mutex>
#include <unordered_map>

#include "tc.cuh"

namespace b200 {
namespace tc {

// ---- tensor-map cache ---------------------------------------------------------------------------------------
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    return q == cudaDriverEntryPointSuccess ? (EncodeTiledFn)p : nullptr;
  }();
  return fn;
}
struct Key {
  const void* base;
  uint64_t rows, cols, stride;
  uint32_t br, bc;
  int dtype;
  bool operator==(const Key& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && stride == o.stride && br == o.br && bc == o.bc && dtype == o.dtype;
  }
};
struct KeyHash {
  size_t operator()(const Key& k) const {
    size_t h = (size_t)k.base;
    for (uint64_t v : {k.rows, k.cols, k.stride, (uint64_t)k.br, (uint64_t)k.bc, (uint64_t)k.dtype}) h = h * 1000003u ^ (size_t)v;
    return h;
  }
};
std::mutex g_mu;
std::unordered_map<Key, CUtensorMap*, KeyHash> g_maps;
}  // namespace

const CUtensorMap* tensor_map_2d(const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems, uint32_t box_rows,
                                 uint32_t box_cols, int dtype) {
  Key key{base, rows, cols, row_stride_elems, box_rows, box_cols, dtype};
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) return it->second;
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable (driver too old?)"); return nullptr; }
  if (g_maps.size() > 4096) {  // pointers churn (caching allocator): keep the table bounded
    for (auto& kv : g_maps) delete kv.second;
    g_maps.clear();
  }
  CUtensorMap* m = new CUtensorMap;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {row_stride_elems * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, dtype == B200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu stride=%llu box=%ux%u", (int)r, (unsigned long long)rows,
              (unsigned long long)cols, (unsigned long long)row_stride_elems, box_rows, box_cols);
    delete m;
    return nullptr;
  }
  g_maps.emplace(key, m);
  return m;
}

const CUtensorMap* tensor_map_nhwc(const void* base, uint64_t B, uint64_t H, uint64_t W, uint64_t C, uint32_t box_h, uint32_t box_w,
                                   int dtype) {
  // shares the 2-D cache: (rows, cols, stride) = (B*H, W, C) cannot collide with a 2-D key of the same base because box_cols = 0 marks it
  Key key{base, B * H, W, C | (H << 32), box_h * 1024u + box_w, 0u, dtype};
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_maps.find(key);
  if (it != g_maps.end()) return it->second;
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable (driver too old?)"); return nullptr; }
  if (g_maps.size() > 4096) {
    for (auto& kv : g_maps) delete kv.second;
    g_maps.clear();
  }
  CUtensorMap* m = new CUtensorMap;
  cuuint64_t dims[4] = {C, W, H, B};
  cuuint64_t strides[3] = {C * 2, W * C * 2, H * W * C * 2};
  cuuint32_t box[4] = {64, box_w, box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, dtype == B200_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (NHWC) failed (%d) B=%llu H=%llu W=%llu C=%llu box=%ux%u", (int)r, (unsigned long long)B,
              (unsigned long long)H, (unsigned long long)W, (unsigned long long)C, box_h, box_w);
    delete m;
    return nullptr;
  }
  g_maps.emplace(key, m);
  return m;
}

namespace {

constexpr int BLOCK_M = 128, BLOCK_K = 64, UMMA_K = 16;
// warp 0 TMA, warp 1 MMA, warps 2.. epilogue: EW = 8 (two per TMEM lane quadrant, 64 columns each) or 16 (four per quadrant,
// 32 columns each -- the GELU epilogues are bound by their FP32/MUFU work, so they get twice the warps to hide its latency)
template <int EW> struct Thr { static constexpr int kThreads = 64 + EW * 32, kEpiThreads = EW * 32; };
enum { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RES = 2, EPI_MUL_GELUGRAD = 3 };

struct GemmParams {
  const float* bias;  // [N] or null
  const void* R;      // residual [M,N] (EPI_BIAS_RES)
  long long M;
  int N, K, m_tiles, n_tiles, k_blocks, fmt, has_d2;
};

// NBUF = 2: the output staging tile(s) are double-buffered, so the epilogue of tile i+1 fills one buffer while the TMA
// engine still reads tile i out of the other (the epilogue warps otherwise idle ~30 % of the time at the store hand-off)
template <int BLOCK_N, int STAGES, int NBUF = 1, int NB2 = NBUF> struct Smem {
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
  static constexpr int D_BYTES = BLOCK_M * BLOCK_N * 2;
  static constexpr int OFF_A = 0;
  static constexpr int OFF_B = OFF_A + STAGES * A_BYTES;
  static constexpr int OFF_D = OFF_B + STAGES * B_BYTES;
  static constexpr int OFF_D2 = OFF_D + NBUF * D_BYTES;
  static constexpr int OFF_BAR = OFF_D2 + NB2 * D_BYTES;   // second area: D2 (GELU pre-activation) or the R tile; absent for EPI_BIAS
  static constexpr int TOTAL = OFF_BAR + 256 + 1024;  // + alignment slack
};

// erf via Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7 with 5 terms) on MUFU.RCP + MUFU.EX2 (approximate forms: no
// slow-path subroutine calls) instead of the ~35-instruction erff; far below the rounding step of the 16-bit
// outputs this epilogue produces.
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// returns Phi(a) (standard normal cdf) and writes e = exp(-a^2/2)
__device__ __forceinline__ float normal_cdf(float a, float* e_out) {
  const float ax = fabsf(a) * 0.70710678118654752440f;
  const float t = rcp_approx(fmaf(0.3275911f, ax, 1.f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = ex2_approx(-0.72134752044448170368f * a * a);  // exp(-a^2/2) = exp(-(a/sqrt2)^2)
  *e_out = e;
  const float erf_abs = fmaf(-p * t, e, 1.f);
  return 0.5f * (1.f + copysignf(erf_abs, a));
}
__device__ __forceinline__ float gelu_erf(float a) { float e; return a * normal_cdf(a, &e); }
__device__ __forceinline__ float gelu_erf_grad(float a) {
  float e;
  const float cdf = normal_cdf(a, &e);
  return fmaf(a * 0.39894228040143267794f, e, cdf);
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi, int fmt) {
  if (fmt == 1) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
  }
  __half2 p = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
__device__ __forceinline__ float unpack_lo(uint32_t w, int fmt) {
  return fmt == 1 ? __uint_as_float(w << 16) : __half2float(__ushort_as_half((unsigned short)(w & 0xffff)));
}
__device__ __forceinline__ float unpack_hi(uint32_t w, int fmt) {
  return fmt == 1 ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
}

template <int BLOCK_N, int STAGES, int EPI, int EW, int NBUF>
__global__ void __launch_bounds__(Thr<EW>::kThreads, 1)
gemm_nt_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmD2,
               const __grid_constant__ CUtensorMap tmR, GemmParams P) {
  using S = Smem<BLOCK_N, STAGES, NBUF, (EPI == EPI_BIAS ? 0 : NBUF)>;
  constexpr int kEpiThreads = Thr<EW>::kEpiThreads;
  extern __shared__ unsigned char smem_raw_[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw_) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;   // [2] accumulator ready
  uint64_t* tempty = tfull + 2;       // [2] accumulator drained
  uint64_t* rfull = tempty + 2;       // [2] R tile landed (TMA_R)
  uint64_t* rempty = rfull + 2;       // [2] R tile consumed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + 2);
  // the GELU-backward epilogue reads a whole [128 x BLOCK_N] tile of R: fetched by TMA into the (otherwise unused) second
  // staging area instead of 32 scattered 64-byte row segments per warp load
  constexpr bool TMA_R = ((EPI == EPI_MUL_GELUGRAD || EPI == EPI_BIAS_RES) && NBUF == 2);
  constexpr int R_TILE_BYTES = BLOCK_M * BLOCK_N * 2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = P.m_tiles * P.n_tiles;

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmA); prefetch_tmap(&tmB); prefetch_tmap(&tmD);
    if (P.has_d2) prefetch_tmap(&tmD2);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], kEpiThreads); }
    for (int i = 0; i < 2; ++i) { mbar_init(&rfull[i], 1); mbar_init(&rempty[i], kEpiThreads); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N); tmem_relinquish(); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0; int rb = 0; uint32_t rphase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile / P.n_tiles) * BLOCK_M, n0 = (tile % P.n_tiles) * BLOCK_N;
        if (TMA_R) {
          mbar_wait(&rempty[rb], rphase ^ 1);
          mbar_expect_tx(&rfull[rb], R_TILE_BYTES);
#pragma unroll
          for (int b = 0; b < BLOCK_N / 64; ++b)
            tma_load_2d(smem + S::OFF_D2 + rb * S::D_BYTES + b * (BLOCK_M * 128), &tmR, &rfull[rb], n0 + b * 64, m0);
          if (++rb == 2) { rb = 0; rphase ^= 1; }
        }
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], S::A_BYTES + S::B_BYTES);
          tma_load_2d(smem + S::OFF_A + stage * S::A_BYTES, &tmA, &full[stage], kb * BLOCK_K, m0);
          tma_load_2d(smem + S::OFF_B + stage * S::B_BYTES, &tmB, &full[stage], kb * BLOCK_K, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      const uint32_t idesc = idesc_f16(BLOCK_M, BLOCK_N, P.fmt);
      int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t aphase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait(&tempty[acc], aphase ^ 1);
        fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < P.k_blocks; ++kb) {
          mbar_wait(&full[stage], phase);
          fence_after_sync();
          const uint64_t da = smem_desc_k_sw128(smem + S::OFF_A + stage * S::A_BYTES);
          const uint64_t db = smem_desc_k_sw128(smem + S::OFF_B + stage * S::B_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
            umma_f16(d_tmem, da + (uint64_t)(k * UMMA_K * 2 >> 4), db + (uint64_t)(k * UMMA_K * 2 >> 4), idesc, (kb | k) != 0);
          umma_commit(&empty[stage]);  // smem slot free once these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[acc]);      // accumulator complete
        if (++acc == 2) { acc = 0; aphase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..) =====================
    const int q = warp & 3;                      // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;            // which slice of the tile's columns this warp converts
    const int row = q * 32 + lane;               // row within the tile
    const int et = threadIdx.x - 64;             // 0..kEpiThreads-1
    constexpr int HALF_N = BLOCK_N / (EW / 4);   // columns per thread
    int acc = 0; uint32_t aphase = 0;
    // R operand (residual / GELU pre-activation) of this thread's 32-column chunk, software-prefetched one chunk ahead so
    // its L2/HBM latency hides behind the previous chunk's epilogue arithmetic
    constexpr bool kHasR = (EPI == EPI_BIAS_RES || EPI == EPI_MUL_GELUGRAD);
    auto load_R = [&](int tile_, int ch_, uint32_t (&dst)[16]) {
      const int m0_ = (tile_ / P.n_tiles) * BLOCK_M, n0_ = (tile_ % P.n_tiles) * BLOCK_N;
      const long long grow_ = (long long)m0_ + row;
      const int col0_ = half * HALF_N + ch_ * 32;
      const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(P.R) + grow_ * P.N + n0_ + col0_);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint4 t = make_uint4(0, 0, 0, 0);
        if (tile_ < total_tiles && grow_ < P.M && n0_ + col0_ + i * 8 < P.N) t = rp[i];
        dst[4 * i] = t.x; dst[4 * i + 1] = t.y; dst[4 * i + 2] = t.z; dst[4 * i + 3] = t.w;
      }
    };
    uint32_t rres[16], rnext[16];
    if (kHasR && !TMA_R) load_R(blockIdx.x, 0, rnext);
    int rb = 0; uint32_t rphase = 0;
    int dbuf = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m0 = (tile / P.n_tiles) * BLOCK_M, n0 = (tile % P.n_tiles) * BLOCK_N;
      unsigned char* sD = smem + S::OFF_D + dbuf * S::D_BYTES;
      unsigned char* sD2 = smem + S::OFF_D2 + dbuf * S::D_BYTES;
      if (NBUF == 2) {   // this buffer was last used two tiles ago: at most the previous tile's stores may still be reading
        if (et == 0) bulk_wait_read_1();
        named_bar_sync(2, kEpiThreads);
      }
      mbar_wait(&tfull[acc], aphase);
      fence_after_sync();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BLOCK_N + half * HALF_N;
      const long long grow = (long long)m0 + row;
#pragma unroll
      for (int ch = 0; ch < HALF_N / 32; ++ch) {
        const int col0 = half * HALF_N + ch * 32;  // first column (within the tile) of this 32-wide chunk
        uint32_t v[32];
        tmem_ld32(taddr + ch * 32, v);
        if (TMA_R) {
          if (ch == 0) mbar_wait(&rfull[rb], rphase);
          const unsigned char* sR = smem + S::OFF_D2 + rb * S::D_BYTES + (col0 / 64) * (BLOCK_M * 128);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint4 t = *reinterpret_cast<const uint4*>(sR + sw128_offset(row, (col0 % 64) / 8 + i));
            rres[4 * i] = t.x; rres[4 * i + 1] = t.y; rres[4 * i + 2] = t.z; rres[4 * i + 3] = t.w;
          }
        } else if (kHasR) {
#pragma unroll
          for (int i = 0; i < 16; ++i) rres[i] = rnext[i];
          if (ch + 1 < HALF_N / 32) load_R(tile, ch + 1, rnext);
          else load_R(tile + (int)gridDim.x, 0, rnext);
        }
        float bv[32];
        if (P.bias) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n0 + col0 + 4 * i < P.N) b4 = __ldg(reinterpret_cast<const float4*>(P.bias + n0 + col0) + i);
            bv[4 * i] = b4.x; bv[4 * i + 1] = b4.y; bv[4 * i + 2] = b4.z; bv[4 * i + 3] = b4.w;
          }
        }
        tmem_ld_wait();
        uint32_t o[16], o2[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float a0 = __uint_as_float(v[2 * i]), a1 = __uint_as_float(v[2 * i + 1]);
          if (P.bias) { a0 += bv[2 * i]; a1 += bv[2 * i + 1]; }
          if (EPI == EPI_BIAS_GELU) {
            o2[i] = pack2(a0, a1, P.fmt);
            // GELU sees the stored (rounded) pre-activation so forward and backward agree bit-for-bit on `a`
            a0 = gelu_erf(unpack_lo(o2[i], P.fmt));
            a1 = gelu_erf(unpack_hi(o2[i], P.fmt));
          }
          if (EPI == EPI_BIAS_RES) { a0 += unpack_lo(rres[i], P.fmt); a1 += unpack_hi(rres[i], P.fmt); }
          if (EPI == EPI_MUL_GELUGRAD) { a0 *= gelu_erf_grad(unpack_lo(rres[i], P.fmt)); a1 *= gelu_erf_grad(unpack_hi(rres[i], P.fmt)); }
          o[i] = pack2(a0, a1, P.fmt);
        }
        // 32 columns = 4 x 16-byte chunks of the [128 rows][64 cols] swizzled box number col0/64
        const int box = col0 / 64, c16 = (col0 % 64) / 8;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t off = box * (BLOCK_M * 128) + sw128_offset(row, c16 + i);
          *reinterpret_cast<uint4*>(sD + off) = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
          if (EPI == EPI_BIAS_GELU)
            *reinterpret_cast<uint4*>(sD2 + off) = make_uint4(o2[4 * i], o2[4 * i + 1], o2[4 * i + 2], o2[4 * i + 3]);
        }
      }
      if (TMA_R) { mbar_arrive(&rempty[rb]); if (++rb == 2) { rb = 0; rphase ^= 1; } }   // R tile consumed
      // accumulator drained -> MMA warp may overwrite it
      fence_before_sync();
      mbar_arrive(&tempty[acc]);
      if (++acc == 2) { acc = 0; aphase ^= 1; }
      // staging complete -> one thread stores the boxes
      fence_proxy_async();
      named_bar_sync(1, kEpiThreads);
      if (et == 0) {
#pragma unroll
        for (int b = 0; b < BLOCK_N / 64; ++b) {
          if (n0 + b * 64 < P.N) {
            tma_store_2d(&tmD, sD + b * (BLOCK_M * 128), n0 + b * 64, m0);
            if (EPI == EPI_BIAS_GELU && P.has_d2) tma_store_2d(&tmD2, sD2 + b * (BLOCK_M * 128), n0 + b * 64, m0);
          }
        }
        bulk_commit();
        if (NBUF == 1) bulk_wait_read_all();  // staging may be rewritten once the TMA engine has read it
      }
      if (NBUF == 1) named_bar_sync(1, kEpiThreads);
      dbuf ^= (NBUF - 1);
    }
    if (et == 0) bulk_wait_all();
  }
  // teardown
  fence_before_sync();
  __syncthreads();
  if (warp == 1) { fence_after_sync(); tmem_dealloc(tmem_base, 2 * BLOCK_N < 32 ? 32 : 2 * BLOCK_N); }
}

template <int BLOCK_N, int STAGES, int EPI, int EW = 8, int NBUF = 1>
int launch(const void* A, const void* B, const float* bias, void* D, void* D2, const void* R, long long M, int N, int K,
           int dtype, cudaStream_t st) {
  using S = Smem<BLOCK_N, STAGES, NBUF, (EPI == EPI_BIAS ? 0 : NBUF)>;
  const CUtensorMap* mA = tensor_map_2d(A, (uint64_t)M, (uint64_t)K, (uint64_t)K, BLOCK_M, BLOCK_K, dtype);
  const CUtensorMap* mB = tensor_map_2d(B, (uint64_t)N, (uint64_t)K, (uint64_t)K, BLOCK_N, BLOCK_K, dtype);
  const CUtensorMap* mD = tensor_map_2d(D, (uint64_t)M, (uint64_t)N, (uint64_t)N, BLOCK_M, 64, dtype);
  const CUtensorMap* mD2 = D2 ? tensor_map_2d(D2, (uint64_t)M, (uint64_t)N, (uint64_t)N, BLOCK_M, 64, dtype) : mD;
  const CUtensorMap* mR = R ? tensor_map_2d(R, (uint64_t)M, (uint64_t)N, (uint64_t)N, BLOCK_M, 64, dtype) : mD;
  if (!mA || !mB || !mD || !mD2 || !mR) return B200_ERR_LAUNCH;
  GemmParams P;
  P.bias = bias; P.R = R; P.M = M; P.N = N; P.K = K;
  P.m_tiles = (int)((M + BLOCK_M - 1) / BLOCK_M);
  P.n_tiles = (N + BLOCK_N - 1) / BLOCK_N;
  P.k_blocks = (K + BLOCK_K - 1) / BLOCK_K;
  P.fmt = dtype == B200_BF16 ? 1 : 0;
  P.has_d2 = D2 != nullptr;
  auto kern = gemm_nt_kernel<BLOCK_N, STAGES, EPI, EW, NBUF>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  int grid = P.m_tiles * P.n_tiles;
  if (grid > sm_count()) grid = sm_count();
  kern<<<grid, Thr<EW>::kThreads, S::TOTAL, st>>>(*mA, *mB, *mD, *mD2, *mR, P);
  return check_launch("gemm_nt");
}

}  // namespace
}  // namespace tc
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_gemm_nt_supported(int64_t M, int32_t N, int32_t K, int32_t dtype) {
  return (dtype == B200_BF16 || dtype == B200_F16) && M > 0 && N >= 16 && K >= 16 && N % 8 == 0 && K % 8 == 0;
}

extern "C" B200_API int b200_gemm_nt(const void* A, const void* B, const float* bias, void* D, void* D2, const void* R,
                                     int64_t M, int32_t N, int32_t K, int32_t dtype, int32_t epi, void* stream) {
  B200_REQUIRE(b200_gemm_nt_supported(M, N, K, dtype), B200_ERR_UNSUPPORTED,
               "gemm_nt: unsupported problem M=%lld N=%d K=%d dtype=%d (16-bit dtypes, N and K multiples of 8)", (long long)M, N, K, dtype);
  B200_REQUIRE(A && B && D, B200_ERR_SHAPE, "gemm_nt: null pointer");
  B200_REQUIRE((((uintptr_t)A | (uintptr_t)B | (uintptr_t)D | (uintptr_t)D2 | (uintptr_t)R) & 15) == 0, B200_ERR_ALIGN,
               "gemm_nt: pointers must be 16-byte aligned");
  B200_REQUIRE(epi >= 0 && epi <= 3, B200_ERR_SHAPE, "gemm_nt: bad epilogue %d", epi);
  B200_REQUIRE(epi < 2 || R, B200_ERR_SHAPE, "gemm_nt: epilogue %d needs R", epi);
  cudaStream_t st = (cudaStream_t)stream;
  using namespace b200::tc;
  if (N >= 128) {
    if (epi == 0) return launch<128, 4, EPI_BIAS, 8, 2>(A, B, bias, D, nullptr, nullptr, M, N, K, dtype, st);
    if (epi == 1) return launch<128, 3, EPI_BIAS_GELU, 8, 2>(A, B, bias, D, D2, nullptr, M, N, K, dtype, st);
    if (epi == 3) return launch<128, 3, EPI_MUL_GELUGRAD, 8, 2>(A, B, bias, D, nullptr, R, M, N, K, dtype, st);
    return launch<128, 3, EPI_BIAS_RES, 8, 2>(A, B, bias, D, nullptr, R, M, N, K, dtype, st);
  }
  if (epi == 0) return launch<64, 4, EPI_BIAS>(A, B, bias, D, nullptr, nullptr, M, N, K, dtype, st);
  if (epi == 1) return launch<64, 4, EPI_BIAS_GELU>(A, B, bias, D, D2, nullptr, M, N, K, dtype, st);
  if (epi == 3) return launch<64, 4, EPI_MUL_GELUGRAD>(A, B, bias, D, nullptr, R, M, N, K, dtype, st);
  return launch<64, 4, EPI_BIAS_RES>(A, B, bias, D, nullptr, R, M, N, K, dtype, st);
}
