// Fused MLP half of the SwinBlock on tcgen05 tensor cores (bf16 / f16 activations, C = 128):
//     out = y1 + mlp.2(GELU(mlp.0(LayerNorm2(y1))))                                  (swin_block.py:53)
// on dense pixel-major rows y1[P, C] (P = B*H*W real tokens -- the MLP half is per token, so padded window tokens are
// never touched and the `window_reverse` + crop of swin_block.py:55-58 is the row order itself).  The [P, 4C] hidden
// activation never leaves the SM: it is produced 128 columns at a time into TMEM, turned into GELU(.) bf16 tiles in
// shared memory by the epilogue warps and consumed from there as the A operand of the second GEMM, whose accumulator was
// pre-loaded with the residual y1 (tcgen05.st) -- no [P,4C] tensor, no separate bias / GELU / residual / LayerNorm pass.
//
// Persistent CTA per SM, 28 warps:
//   warp 0      W1' producer: K halves [128 hidden rows x 64] of a chunk through a 2-stage TMA ring (weights stay L2 resident)
//   warp 1      TMEM allocator + MMA issuer (one lane).  Two streams over the chunk index g = 4*tile + j, issued in whichever
//               order their inputs become ready (non-blocking mbarrier.test_wait probes):
//                   MMA1(g): H[g&1]   = xhat(tile) * W1'[j]^T          (128x128x128)
//                   MMA2(g): OUT[t&1] += gelu(H)(g) * W2[:, j]^T       (OUT pre-loaded with the residual y1)
//   warps 2-5   LayerNorm warps (thread = token row = TMEM lane): TMA-loaded y1 tile -> statistics -> xhat (16 bit, in place:
//               the A operand) + y1 (f32) into the OUT accumulator (tcgen05.st)
//   warps 6-9   output warps: OUT + b2 -> 16 bit -> staging tile -> TMA store (two 64-column halves)
//   warps 10-25 GELU warps, two groups of 8 on alternate chunks: tcgen05.ld 2 x 32 columns -> + b1' -> GELU -> 16 bit -> swizzled
//               A tile of MMA2
//   warp 26     y1 tile loader (a tile's A buffer is reloaded as soon as its four MMA1 have retired)
//   warp 27     W2 producer: K halves [128 x 64 hidden columns] of a chunk through a 2-stage TMA ring
// LayerNorm's affine part is folded into the first GEMM by a tiny prep kernel (W1' = W1 * gamma, b1' = b1 + W1 beta), so
// the A operand is the normalised row itself -- which is also what the backward kernel needs again.
//
// GELU: a * Phi(a) with Phi(a) = 0.5 (1 + tanh(q(a))), q an odd degree-5 polynomial fitted to atanh(erf(a / sqrt 2))
// (max |error| of a*Phi(a) against erf-GELU: 3e-5, far below the 16-bit rounding of the tile it feeds) -- ONE MUFU
// (tanh.approx) per element instead of two (rcp + ex2), which halves the SFU time that bounds this epilogue.
#include "tc.cuh"

long long* g_mlp_dbg = nullptr;   // debugging aid, see b200_debug_set_mlp_timeline

namespace b200 {
namespace tc {
namespace {

constexpr int kC = 128, kHid = 512, kTileM = 128;
constexpr int kLnWarps = 4, kOutWarps = 4, kGeluWarps = 16;
constexpr int kFirstOutWarp = 2 + kLnWarps, kFirstGeluWarp = kFirstOutWarp + kOutWarps;
constexpr int kLoaderWarp = kFirstGeluWarp + kGeluWarps;       // warp 26: y1 tiles
constexpr int kW2Warp = kLoaderWarp + 1;                       // warp 27: W2 ring
constexpr int kThreads = 32 * (kW2Warp + 1);                   // 896
constexpr int kRing = 2;                                       // stages per weight ring
constexpr int kTileBytes = kTileM * kC * 2;                    // 32 KB: [2 K-blocks][128 rows][128 B]
constexpr int kHalfBytes = kTileM * 64 * 2;                    // 16 KB: one K-block [128 rows][128 B]

struct MlpSmem {
  static constexpr int OFF_U = 0;                               // 2 x 32 KB: y1 tile -> xhat (A of MMA1)
  static constexpr int OFF_H = OFF_U + 2 * kTileBytes;          // 2 x 32 KB: gelu(H) tiles (A of MMA2)
  static constexpr int OFF_O = OFF_H + 2 * kTileBytes;          // 32 KB: output staging tile (TMA store source)
  static constexpr int OFF_W1 = OFF_O + kTileBytes;             // kRing x 16 KB: W1' K halves [128 hidden rows][128 B]
  static constexpr int OFF_W2 = OFF_W1 + kRing * kHalfBytes;    // kRing x 16 KB: W2 K halves [128 rows][128 B]
  static constexpr int OFF_B1 = OFF_W2 + kRing * kHalfBytes;    // b1' [512] f32
  static constexpr int OFF_B2 = OFF_B1 + kHid * 4;              // b2 [128] f32
  static constexpr int OFF_BAR = OFF_B2 + kC * 4;
  static constexpr int TOTAL = OFF_BAR + 256;   // the dynamic shared memory window itself is 1024-byte aligned (checked at run time)
};
static_assert(MlpSmem::TOTAL <= 232448, "shared memory budget");

struct MlpParams {
  const float* b1f;   // [512] folded bias
  const float* b2;    // [128]
  void* out;          // [P, 128]
  long long P;        // rows
  long long* dbg;     // optional timeline of CTA 0 (profiles/mlp_timeline.py): [role][event][index] SM clock stamps
  int n_tiles, fmt, save_h;   // save_h: also write 2*gelu(a) [P, 512] (training: operand of the mlp.2 weight gradient)
  float eps;
};

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]),
        "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]),
        "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tanh_approx(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// q(a) of the header comment; z is clamped so the (non-monotone beyond |a| ~ 10) polynomial saturates tanh instead
constexpr float kG0 = 0.797458471f, kG1 = 0.0370503451f, kG2 = -3.58732361e-4f;
__device__ __forceinline__ float gelu_tanh5(float a) {
  const float z = fminf(a * a, 64.f);
  const float q = a * fmaf(z, fmaf(z, kG2, kG1), kG0);
  const float hlf = 0.5f * a;
  return fmaf(hlf, tanh_approx(q), hlf);
}
// 2 * gelu(a) = a (1 + tanh(q(a))): the factor 0.5 is folded into W2 by the prep kernel (exact: a power of two)
__device__ __forceinline__ float gelu2_tanh5(float a) {
  const float z = fminf(a * a, 64.f);
  return fmaf(a, tanh_approx(a * fmaf(z, fmaf(z, kG2, kG1), kG0)), a);
}
// d/da [2 gelu(a)] = d/da [a (1 + t)] of the SAME approximation: (1 + t) + a (1 - t^2) q'(a)
__device__ __forceinline__ float gelu2_tanh5_grad(float a) {
  const float a2 = a * a;
  const float z = fminf(a2, 64.f);
  const float inner = fmaf(z, fmaf(z, kG2, kG1), kG0);
  const float t = tanh_approx(a * inner);
  const float qd = a2 < 64.f ? fmaf(z, fmaf(z, 5.f * kG2, 3.f * kG1), kG0) : inner;   // q'(a); constant slope beyond the clamp
  return fmaf(a * qd, fmaf(-t, t, 1.f), 1.f + t);
}
// d/da [a * Phi(a)] of the SAME approximation: Phi + a * 0.5 (1 - t^2) q'(a); also returns the forward value
__device__ __forceinline__ float gelu_tanh5_grad(float a, float* fwd) {
  const float a2 = a * a;
  const float z = fminf(a2, 64.f);
  const float inner = fmaf(z, fmaf(z, kG2, kG1), kG0);
  const float t = tanh_approx(a * inner);
  // q'(a) = k0 + 3 k1 z + 5 k2 z^2 inside the clamp, = inner (constant slope) outside
  const float qd = a2 < 64.f ? fmaf(z, fmaf(z, 5.f * kG2, 3.f * kG1), kG0) : inner;
  const float phi = fmaf(0.5f, t, 0.5f);
  *fwd = a * phi;
  return fmaf(0.5f * a * qd, fmaf(-t, t, 1.f), phi);
}

// debug timeline (CTA 0 only, dbg != nullptr): role r in [0,4), event e in [0,4), index i < 64
template <typename PT> __device__ __forceinline__ void stamp(const PT& P, int r, int e, int i) {
  if (P.dbg != nullptr && blockIdx.x == 0 && i < 64) {
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t));
    P.dbg[(r * 4 + e) * 64 + i] = t;
  }
}

template <int FMT> __device__ __forceinline__ uint32_t pack2h(float lo, float hi) {
  if (FMT == 1) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
  }
  __half2 p = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
template <int FMT> __device__ __forceinline__ float up_lo(uint32_t w) {
  return FMT == 1 ? __uint_as_float(w << 16) : __half2float(__ushort_as_half((unsigned short)(w & 0xffff)));
}
template <int FMT> __device__ __forceinline__ float up_hi(uint32_t w) {
  return FMT == 1 ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
}

// one 128-column row of a [2][128 rows][128 B] swizzled tile: 16-byte chunk c (0..15)
__device__ __forceinline__ uint4* row_chunk(unsigned char* tile, int row, int c) {
  return reinterpret_cast<uint4*>(tile + (c >> 3) * (kTileM * 128) + sw128_offset(row, c & 7));
}

// FMT: 1 = bf16, 0 = f16 (compile-time: the unpack / pack sequences sit in every inner loop)
template <int FMT>
__global__ void __launch_bounds__(kThreads, 1)
swin_mlp_fwd_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmOut,
                    const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmH, MlpParams P) {
  using S = MlpSmem;
  extern __shared__ __align__(1024) unsigned char smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();   // 128-byte swizzle atoms need a 1024-byte aligned base: no slack is budgeted
  float* sb1 = reinterpret_cast<float*>(smem + S::OFF_B1);
  float* sb2 = reinterpret_cast<float*>(smem + S::OFF_B2);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* y_full = bars;            // [2] y1 tile landed (TMA)
  uint64_t* u_ready = bars + 2;       // [2] xhat written + OUT accumulator pre-loaded (128 LayerNorm threads)
  uint64_t* u_free = bars + 4;        // [2] the tile's four MMA1 have read the A tile (commit): it may be reloaded
  uint64_t* w1_full = bars + 6;       // [kRing]
  uint64_t* w1_empty = w1_full + kRing;
  uint64_t* w2_full = w1_empty + kRing;
  uint64_t* w2_empty = w2_full + kRing;
  uint64_t* h_full = w2_empty + kRing;  // [2] H accumulator complete (commit)
  uint64_t* h_tfree = h_full + 2;     // [2] H accumulator read back (256 GELU threads)
  uint64_t* hs_full = h_full + 4;     // [2] gelu(H) tile written (256 GELU threads)
  uint64_t* hs_free = h_full + 6;     // [2] gelu(H) tile consumed by MMA2 (commit)
  uint64_t* o_full = h_full + 8;      // [2] OUT accumulator complete (commit)
  uint64_t* o_free = h_full + 10;     // [2] OUT accumulator read back (128 output threads): it may be pre-loaded again
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h_full + 12);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_local = (int)blockIdx.x < P.n_tiles ? (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int n_chunks = 4 * n_local;
  auto ubuf = [&](int b) { return smem + S::OFF_U + b * kTileBytes; };
  auto hbuf = [&](int b) { return smem + S::OFF_H + b * kTileBytes; };
  unsigned char* obuf = smem + S::OFF_O;

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmY); prefetch_tmap(&tmOut); prefetch_tmap(&tmW1); prefetch_tmap(&tmW2); prefetch_tmap(&tmH);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&y_full[i], 1); mbar_init(&u_ready[i], 32 * kLnWarps); mbar_init(&u_free[i], 1);
      mbar_init(&h_full[i], 1); mbar_init(&h_tfree[i], 16 * kGeluWarps);     // each H accumulator belongs to one group of 8 GELU warps
      mbar_init(&hs_full[i], 1); mbar_init(&hs_free[i], 1); mbar_init(&o_full[i], 1);
      mbar_init(&o_free[i], 32 * kOutWarps);
    }
    for (int i = 0; i < kRing; ++i) {
      mbar_init(&w1_full[i], 1); mbar_init(&w1_empty[i], 1); mbar_init(&w2_full[i], 1); mbar_init(&w2_empty[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  for (int i = threadIdx.x; i < kHid; i += kThreads) sb1[i] = P.b1f[i];
  for (int i = threadIdx.x; i < kC; i += kThreads) sb2[i] = P.b2[i];
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  auto tH = [&](int i) { return tmem_base + i * 128; };          // columns [0,256): two H accumulators
  auto tOut = [&](int b) { return tmem_base + 256 + b * 128; };  // columns [256,512): two OUT accumulators

  if (warp == 0) {
    // ===================== W1' producer: chunk g = rows (g&3)*128 .. +128 of W1', two K halves of 64 columns =====================
    if (elect_one()) {
      int st = 0; uint32_t ph = 0;
      for (int h2 = 0; h2 < 2 * n_chunks; ++h2) {
        mbar_wait(&w1_empty[st], ph ^ 1);
        mbar_expect_tx(&w1_full[st], kHalfBytes);
        tma_load_2d(smem + S::OFF_W1 + st * kHalfBytes, &tmW1, &w1_full[st], (h2 & 1) * 64, ((h2 >> 1) & 3) * 128);
        if (++st == kRing) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == kW2Warp) {
    // ===================== W2 producer: chunk g = columns (g&3)*128 .. +128 of W2, two K halves of 64 columns =====================
    if (elect_one()) {
      int st = 0; uint32_t ph = 0;
      for (int h2 = 0; h2 < 2 * n_chunks; ++h2) {
        mbar_wait(&w2_empty[st], ph ^ 1);
        mbar_expect_tx(&w2_full[st], kHalfBytes);
        tma_load_2d(smem + S::OFF_W2 + st * kHalfBytes, &tmW2, &w2_full[st], ((h2 >> 1) & 3) * 128 + (h2 & 1) * 64, 0);
        if (++st == kRing) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == kLoaderWarp) {
    // ===================== y1 tile loader =====================
    if (elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int b = n & 1;
        const int tile = blockIdx.x + n * gridDim.x;
        mbar_wait(&u_free[b], ((n >> 1) & 1) ^ 1);
        mbar_expect_tx(&y_full[b], kTileBytes);
        tma_load_2d(ubuf(b), &tmY, &y_full[b], 0, tile * kTileM);
        tma_load_2d(ubuf(b) + kTileM * 128, &tmY, &y_full[b], 64, tile * kTileM);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: two streams, issued as their inputs become ready =====================
    if (elect_one()) {
      const uint32_t idesc = idesc_f16(128, 128, FMT);
      int s1 = 0, s2 = 0; uint32_t p1 = 0, p2 = 0;
      int a = 0, b = 0;            // next chunk of the MMA1 / MMA2 stream
      while (b < n_chunks) {
        if (b < a && mbar_poll(&hs_full[b & 1], (b >> 1) & 1)) {
          // ---- MMA2(b): OUT[t&1] += gelu(H)(b) * W2[:, chunk]^T, two K halves of 64 ----
          const int t = b >> 2;
          fence_after_sync();
          stamp(P, 0, 2, b);
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            mbar_wait(&w2_full[s2], p2);
            fence_after_sync();
            const uint64_t da = smem_desc_k_sw128(hbuf(b & 1) + kk * kHalfBytes), db = smem_desc_k_sw128(smem + S::OFF_W2 + s2 * kHalfBytes);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16(tOut(t & 1), da + 2 * k, db + 2 * k, idesc, 1u);
            umma_commit(&w2_empty[s2]);
            if (++s2 == kRing) { s2 = 0; p2 ^= 1; }
          }
          umma_commit(&hs_free[b & 1]);
          if ((b & 3) == 3) umma_commit(&o_full[t & 1]);
          stamp(P, 0, 3, b);
          ++b;
        }
        if (a < n_chunks) {
          const int t = a >> 2;
          if (((a & 3) != 0 || mbar_poll(&u_ready[t & 1], (t >> 1) & 1)) && mbar_poll(&h_tfree[a & 1], ((a >> 1) & 1) ^ 1)) {
            // ---- MMA1(a): H[a&1] = xhat * W1'[chunk]^T, two K halves of 64 ----
            fence_after_sync();
            stamp(P, 0, 0, a);
#pragma unroll
            for (int kk = 0; kk < 2; ++kk) {
              mbar_wait(&w1_full[s1], p1);
              fence_after_sync();
              const uint64_t da = smem_desc_k_sw128(ubuf(t & 1) + kk * kHalfBytes), db = smem_desc_k_sw128(smem + S::OFF_W1 + s1 * kHalfBytes);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_f16(tH(a & 1), da + 2 * k, db + 2 * k, idesc, (kk | k) ? 1u : 0u);
              umma_commit(&w1_empty[s1]);
              if (++s1 == kRing) { s1 = 0; p1 ^= 1; }
            }
            umma_commit(&h_full[a & 1]);
            if ((a & 3) == 3) umma_commit(&u_free[t & 1]);
            stamp(P, 0, 1, a);
            ++a;
          }
        }
      }
    }
  } else if (warp < kFirstOutWarp) {
    // ===================== LayerNorm warps (thread = row = TMEM lane) =====================
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      unsigned char* u = ubuf(b);
      if (row == 0) stamp(P, 1, 0, n);
      mbar_wait(&y_full[b], (n >> 1) & 1);
      if (row == 0) stamp(P, 1, 1, n);
      // one pass, shifted by the row's first element (no cancellation unless |mean - x0| >> std): sum d, sum d^2
      const float x0 = up_lo<FMT>(row_chunk(u, row, 0)->x);
      float s = 0.f, ss = 0.f;
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const uint4 w = *row_chunk(u, row, c);
        const float d0 = up_lo<FMT>(w.x) - x0, d1 = up_hi<FMT>(w.x) - x0, d2 = up_lo<FMT>(w.y) - x0, d3 = up_hi<FMT>(w.y) - x0;
        const float d4 = up_lo<FMT>(w.z) - x0, d5 = up_hi<FMT>(w.z) - x0, d6 = up_lo<FMT>(w.w) - x0, d7 = up_hi<FMT>(w.w) - x0;
        s += ((d0 + d1) + (d2 + d3)) + ((d4 + d5) + (d6 + d7));
        ss += fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3) + (fmaf(d4, d4, d5 * d5) + fmaf(d6, d6, d7 * d7));
      }
      const float md = s * (1.f / kC);
      const float rstd = rsqrtf(fmaxf(ss * (1.f / kC) - md * md, 0.f) + P.eps);
      const float shift = -(x0 + md) * rstd;
      mbar_wait(&o_free[b], ((n >> 1) & 1) ^ 1);   // tile n-2's output warps have read OUT[b]
      fence_after_sync();
#pragma unroll 2
      for (int ch = 0; ch < 4; ++ch) {          // 32 columns at a time: residual -> TMEM, xhat -> A tile (in place)
        uint32_t f[32];
        uint4 w4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) w4[c] = *row_chunk(u, row, ch * 4 + c);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t ww[4] = {w4[c].x, w4[c].y, w4[c].z, w4[c].w};
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float x0_ = up_lo<FMT>(ww[e]), x1_ = up_hi<FMT>(ww[e]);
            f[c * 8 + 2 * e] = __float_as_uint(x0_);
            f[c * 8 + 2 * e + 1] = __float_as_uint(x1_);
            o[e] = pack2h<FMT>(fmaf(x0_, rstd, shift), fmaf(x1_, rstd, shift));
          }
          *row_chunk(u, row, ch * 4 + c) = make_uint4(o[0], o[1], o[2], o[3]);
        }
        tmem_st32(tOut(b) + lane_sel + ch * 32, f);
      }
      tmem_st_wait();
      fence_proxy_async();
      fence_before_sync();
      mbar_arrive(&u_ready[b]);
      if (row == 0) stamp(P, 1, 2, n);
    }
  } else if (warp < kFirstGeluWarp) {
    // ===================== output warps: OUT + b2 -> 16 bit -> staging half tile -> TMA store =====================
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool leader = (warp == kFirstOutWarp && lane == 0);
    bool pending = false;
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      if (row == 0) stamp(P, 2, 0, n);
      mbar_wait(&o_full[b], (n >> 1) & 1);
      fence_after_sync();
      if (row == 0) stamp(P, 2, 1, n);
      if (pending) {                       // the previous tile's stores must have finished reading the staging tile
        if (leader) bulk_wait_read_all();
        named_bar_sync(1, 32 * kOutWarps);
      }
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t v[32];
        tmem_ld32(tOut(b) + lane_sel + ch * 32, v);
        tmem_ld_wait();
        if (ch == 3) { fence_before_sync(); mbar_arrive(&o_free[b]); }     // OUT[b] fully read by this thread
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float* bp = sb2 + ch * 32 + c * 8;
          const float4 ba = *reinterpret_cast<const float4*>(bp), bb = *reinterpret_cast<const float4*>(bp + 4);
          uint4 o;
          o.x = pack2h<FMT>(__uint_as_float(v[c * 8 + 0]) + ba.x, __uint_as_float(v[c * 8 + 1]) + ba.y);
          o.y = pack2h<FMT>(__uint_as_float(v[c * 8 + 2]) + ba.z, __uint_as_float(v[c * 8 + 3]) + ba.w);
          o.z = pack2h<FMT>(__uint_as_float(v[c * 8 + 4]) + bb.x, __uint_as_float(v[c * 8 + 5]) + bb.y);
          o.w = pack2h<FMT>(__uint_as_float(v[c * 8 + 6]) + bb.z, __uint_as_float(v[c * 8 + 7]) + bb.w);
          *row_chunk(obuf, row, ch * 4 + c) = o;
        }
      }
      fence_proxy_async();
      named_bar_sync(1, 32 * kOutWarps);
      if (leader) {
        tma_store_2d(&tmOut, obuf, 0, tile * kTileM);
        tma_store_2d(&tmOut, obuf + kHalfBytes, 64, tile * kTileM);
        bulk_commit();
      }
      pending = true;
      if (row == 0) stamp(P, 2, 2, n);
    }
    if (leader) bulk_wait_all();
  } else if (warp < kLoaderWarp) {
    // ===================== GELU warps: H (TMEM) -> + b1' -> GELU -> 16-bit A tile of MMA2 =====================
    // two groups of 8 warps on alternate chunks (group = H accumulator = A tile): one group's wait / tcgen05.ld / store /
    // fence latencies are covered by the other group's arithmetic
    const int gw = warp - kFirstGeluWarp;
    const int grp = gw >> 3;                         // 0: even chunks, 1: odd chunks
    const int q = warp & 3, cs = (gw >> 2) & 1;      // TMEM lane quadrant, 64-column half of the 128-column chunk
    const int row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    unsigned char* h = hbuf(grp) + cs * kHalfBytes;  // this thread's 64 columns = K-block cs of the group's A tile
    const bool leader = ((gw & 7) == 0 && lane == 0);
    bool pending = false;
    for (int g = grp; g < n_chunks; g += 2) {
      const uint32_t ph = (g >> 1) & 1;
      const float* bias = sb1 + (g & 3) * 128 + cs * 64;
      if (leader) stamp(P, 3, 0, g);
      mbar_wait(&h_full[grp], ph);
      fence_after_sync();
      if (leader) stamp(P, 3, 1, g);
      mbar_wait(&hs_free[grp], ph ^ 1);
      if (pending) {                                 // the TMA store of chunk g-2 has read the tile
        if (leader) bulk_wait_read_all();
        named_bar_sync(2 + grp, 16 * kGeluWarps);
      }
#pragma unroll 1
      for (int r2 = 0; r2 < 2; ++r2) {
        uint32_t v[32];
        tmem_ld32(tH(grp) + lane_sel + cs * 64 + r2 * 32, v);
        tmem_ld_wait();
        if (r2 == 1) { fence_before_sync(); mbar_arrive(&h_tfree[grp]); }
        uint32_t o[16];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float4 bv = *reinterpret_cast<const float4*>(bias + r2 * 32 + 4 * e);
          o[2 * e] = pack2h<FMT>(gelu2_tanh5(__uint_as_float(v[4 * e]) + bv.x), gelu2_tanh5(__uint_as_float(v[4 * e + 1]) + bv.y));
          o[2 * e + 1] = pack2h<FMT>(gelu2_tanh5(__uint_as_float(v[4 * e + 2]) + bv.z), gelu2_tanh5(__uint_as_float(v[4 * e + 3]) + bv.w));
        }
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<uint4*>(h + sw128_offset(row, r2 * 4 + c)) = make_uint4(o[4 * c], o[4 * c + 1], o[4 * c + 2], o[4 * c + 3]);
      }
      if (leader) stamp(P, 3, 2, g);
      fence_proxy_async();
      named_bar_sync(2 + grp, 16 * kGeluWarps);
      if (leader) {
        mbar_arrive(&hs_full[grp]);
        if (P.save_h) {
          const int r0 = (blockIdx.x + (g >> 2) * gridDim.x) * kTileM;
          tma_store_2d(&tmH, hbuf(grp), (g & 3) * 128, r0);
          tma_store_2d(&tmH, hbuf(grp) + kHalfBytes, (g & 3) * 128 + 64, r0);
          bulk_commit();
        }
        stamp(P, 3, 3, g);
      }
      pending = P.save_h != 0;
    }
    if (leader) bulk_wait_all();
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) { fence_after_sync(); tmem_dealloc(tmem_base, 512); }
}

// =====================================================================================================================
// backward of the fused MLP half.  Per 128-row tile, with the hidden dimension in 8 chunks of 64 columns:
//     xhat = LN2 statistics of y1 (recomputed; also written out for the weight-gradient GEMM)
//     A(g) = xhat * W1'[chunk]^T,  G(g) = g_out * W2'[:, chunk]            (MMA_a, MMA_g -> TMEM)
//     a = A + b1',  g_a = G * d[2 gelu](a) -> shared (A of MMA_u) -> global (TMA store)      (h = 2 gelu(a) was saved by the forward)
//     U += g_a(g) * W1'[chunk]                                             (MMA_u; W1' = W1 gamma, so U = dL/dxhat)
//     g_y1' = rstd * (U - mean(U) - xhat * mean(U * xhat))                 (LayerNorm backward; the residual "+ g_out" is added
//                                                                           by the consumer, b200_swin_partition)
// The W1' chunk of a ring stage serves MMA_a (K-major B) and MMA_u (MN-major B) from the same bytes.  Parameter gradients are
// contractions over ALL rows and are left to b200_gemm_splitk on the three tensors written here (see include/).
// Warp roles as in the forward kernel: 0 W1' producer | 1 MMA issuer | 2-5 LayerNorm warps | 6-9 final (g_y1) warps |
// 10-25 two groups of 8 GELU-backward warps on alternate chunks | 26 y1 / g_out tile loader | 27 W2' producer.
// =====================================================================================================================
constexpr int kRingW1B = 4;                                    // W1' stages are held from MMA_a(g) to MMA_u(g): a deep ring
struct MlpBwdSmem {
  static constexpr int OFF_X = 0;                               // 2 x 32 KB: y1 tile -> xhat (A of MMA_a) -> g_y1 staging
  static constexpr int OFF_G = OFF_X + 2 * kTileBytes;          // 32 KB: g_out tile (A of MMA_g)
  static constexpr int OFF_GA = OFF_G + kTileBytes;             // 2 x 16 KB: g_a chunk tiles (A of MMA_u, TMA store source)
  static constexpr int OFF_W1 = OFF_GA + 2 * kHalfBytes;        // kRingW1B x 16 KB: W1' chunks [64 hidden rows][2 x 128 B]
  static constexpr int OFF_W2 = OFF_W1 + kRingW1B * kHalfBytes; // kRing x 16 KB: W2' chunks [128 rows][128 B]
  static constexpr int OFF_RS = OFF_W2 + kRing * kHalfBytes;    // rstd [2][128] f32
  static constexpr int OFF_BAR = OFF_RS + 2 * kTileM * 4;
  static constexpr int TOTAL = OFF_BAR + 384;   // 32 mbarriers + the TMEM slot
};
static_assert(MlpBwdSmem::TOTAL <= 232448, "shared memory budget");

struct MlpBwdParams {
  const float* b1f;
  long long P;
  long long* dbg;
  int n_tiles;
  float eps;
};

// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}

template <int FMT>
__global__ void __launch_bounds__(kThreads, 1)
swin_mlp_bwd_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmG,
                    const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmXhat, const __grid_constant__ CUtensorMap tmGa,
                    const __grid_constant__ CUtensorMap tmGy, MlpBwdParams P) {
  using S = MlpBwdSmem;
  extern __shared__ __align__(1024) unsigned char smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  float* srs = reinterpret_cast<float*>(smem + S::OFF_RS);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* y_full = bars;                 // [2] y1 tile landed
  uint64_t* u_ready = bars + 2;            // [2] xhat written (128 LayerNorm threads)
  uint64_t* x_free = bars + 4;             // [2] tile buffer reusable: the xhat store and the g_y1 store have both read it
  uint64_t* g_full = bars + 6;             // g_out tile landed
  uint64_t* g_free = bars + 7;             // the tile's eight MMA_g have read it (commit)
  uint64_t* w1_full = bars + 8;            // [kRingW1B]
  uint64_t* w1_empty = w1_full + kRingW1B;
  uint64_t* w2_full = w1_empty + kRingW1B; // [kRing]
  uint64_t* w2_empty = w2_full + kRing;
  uint64_t* ag_full = w2_empty + kRing;    // [2] A and G accumulators of a chunk complete (commit)
  uint64_t* ag_tfree = ag_full + 2;        // [2] ... read back (256 threads of the group)
  uint64_t* ga_full = ag_full + 4;         // [2] g_a tile written (group leader, after the group's barrier)
  uint64_t* ga_free = ag_full + 6;         // [2] g_a tile consumed by MMA_u (commit)
  uint64_t* tu_full = ag_full + 8;         // [2] U accumulator of a tile complete (commit)
  uint64_t* tu_free = ag_full + 10;        // [2] ... read back (128 final threads)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ag_full + 12);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_local = (int)blockIdx.x < P.n_tiles ? (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int n_chunks = 8 * n_local;
  auto xbuf = [&](int b) { return smem + S::OFF_X + b * kTileBytes; };
  unsigned char* gbuf = smem + S::OFF_G;
  auto gabuf = [&](int i) { return smem + S::OFF_GA + i * kHalfBytes; };

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmY); prefetch_tmap(&tmG); prefetch_tmap(&tmW1); prefetch_tmap(&tmW2); prefetch_tmap(&tmXhat); prefetch_tmap(&tmGa);
    prefetch_tmap(&tmGy);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&y_full[i], 1); mbar_init(&u_ready[i], 32 * kLnWarps); mbar_init(&x_free[i], 2);
      mbar_init(&ag_full[i], 1); mbar_init(&ag_tfree[i], 16 * kGeluWarps); mbar_init(&ga_full[i], 1); mbar_init(&ga_free[i], 1);
      mbar_init(&tu_full[i], 1); mbar_init(&tu_free[i], 32 * kOutWarps);
    }
    mbar_init(g_full, 1); mbar_init(g_free, 1);
    for (int i = 0; i < kRingW1B; ++i) { mbar_init(&w1_full[i], 1); mbar_init(&w1_empty[i], 1); }
    for (int i = 0; i < kRing; ++i) { mbar_init(&w2_full[i], 1); mbar_init(&w2_empty[i], 1); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  auto tA = [&](int i) { return tmem_base + i * 64; };            // [0,128): A accumulators of the two groups
  auto tG = [&](int i) { return tmem_base + 128 + i * 64; };      // [128,256): G accumulators
  auto tU = [&](int b) { return tmem_base + 256 + b * 128; };     // [256,512): U accumulators of two tiles

  if (warp == 0) {
    // ===================== W1' producer: chunk g = rows (g&7)*64 .. +64, all 128 columns (two K blocks) =====================
    if (elect_one()) {
      int st = 0; uint32_t ph = 0;
      for (int g = 0; g < n_chunks; ++g) {
        unsigned char* dst = smem + S::OFF_W1 + st * kHalfBytes;
        mbar_wait(&w1_empty[st], ph ^ 1);
        mbar_expect_tx(&w1_full[st], kHalfBytes);
        tma_load_2d(dst, &tmW1, &w1_full[st], 0, (g & 7) * 64);
        tma_load_2d(dst + 64 * 128, &tmW1, &w1_full[st], 64, (g & 7) * 64);
        if (++st == kRingW1B) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == kW2Warp) {
    // ===================== W2' producer: chunk g = columns (g&7)*64 .. +64, all 128 rows =====================
    if (elect_one()) {
      int st = 0; uint32_t ph = 0;
      for (int g = 0; g < n_chunks; ++g) {
        mbar_wait(&w2_empty[st], ph ^ 1);
        mbar_expect_tx(&w2_full[st], kHalfBytes);
        tma_load_2d(smem + S::OFF_W2 + st * kHalfBytes, &tmW2, &w2_full[st], (g & 7) * 64, 0);
        if (++st == kRing) { st = 0; ph ^= 1; }
      }
    }
  } else if (warp == kLoaderWarp) {
    // ===================== y1 / g_out tile loader =====================
    if (elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int b = n & 1;
        const int tile = blockIdx.x + n * gridDim.x;
        mbar_wait(&x_free[b], ((n >> 1) & 1) ^ 1);
        mbar_expect_tx(&y_full[b], kTileBytes);
        tma_load_2d(xbuf(b), &tmY, &y_full[b], 0, tile * kTileM);
        tma_load_2d(xbuf(b) + kHalfBytes, &tmY, &y_full[b], 64, tile * kTileM);
        mbar_wait(g_free, (n & 1) ^ 1);
        mbar_expect_tx(g_full, kTileBytes);
        tma_load_2d(gbuf, &tmG, g_full, 0, tile * kTileM);
        tma_load_2d(gbuf + kHalfBytes, &tmG, g_full, 64, tile * kTileM);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: stream 1 = MMA_a + MMA_g per chunk, stream 2 = MMA_u per chunk =====================
    if (elect_one()) {
      const uint32_t id_a = idesc_f16(128, 64, FMT, 0, 0), id_g = idesc_f16(128, 64, FMT, 0, 1), id_u = idesc_f16(128, 128, FMT, 0, 1);
      int s1a = 0, s1u = 0, s2 = 0; uint32_t p1a = 0, p2 = 0;
      int a = 0, b = 0;            // next chunk of stream 1 / stream 2
      while (b < n_chunks) {
        if (b < a && mbar_poll(&ga_full[b & 1], (b >> 1) & 1)) {
          // ---- MMA_u(b): U[t&1] (+)= g_a(b) [128 x 64] * W1'[chunk] [64 x 128] (B MN-major, from the stage MMA_a(b) used) ----
          const int t = b >> 3;
          bool go = true;
          if ((b & 7) == 0) go = mbar_poll(&tu_free[t & 1], ((t >> 1) & 1) ^ 1);   // fresh accumulator: tile t-2's final warps are done
          if (go) {
            fence_after_sync();
            stamp(P, 0, 2, b);
            unsigned char* A = gabuf(b & 1);
            unsigned char* B = smem + S::OFF_W1 + s1u * kHalfBytes;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16(tU(t & 1), smem_desc_k_sw128(A + k * 32), smem_desc_mn_sw128(B + k * 2048, 64 * 128), id_u, ((b & 7) | k) ? 1u : 0u);
            umma_commit(&w1_empty[s1u]);
            umma_commit(&ga_free[b & 1]);
            if ((b & 7) == 7) umma_commit(&tu_full[t & 1]);
            if (++s1u == kRingW1B) s1u = 0;
            ++b;
          }
        }
        if (a < n_chunks && a < b + kRingW1B) {   // a W1' stage stays held until MMA_u of its chunk: never wait on a stage the ring cannot supply
          const int t = a >> 3;
          bool go = mbar_poll(&ag_tfree[a & 1], ((a >> 1) & 1) ^ 1);
          if (go && (a & 7) == 0) go = mbar_poll(&u_ready[t & 1], (t >> 1) & 1) && mbar_poll(g_full, t & 1);
          if (go) {
            fence_after_sync();
            stamp(P, 0, 0, a);
            mbar_wait(&w1_full[s1a], p1a);
            mbar_wait(&w2_full[s2], p2);
            fence_after_sync();
            stamp(P, 0, 1, a);
            unsigned char* X = xbuf(t & 1);
            unsigned char* W1s = smem + S::OFF_W1 + s1a * kHalfBytes;
            unsigned char* W2s = smem + S::OFF_W2 + s2 * kHalfBytes;
#pragma unroll
            for (int k = 0; k < 8; ++k)      // A(g) = xhat [128 x 128] * W1'[chunk]^T : B K-major [64 rows][2 K blocks]
              umma_f16(tA(a & 1), smem_desc_k_sw128(X + (k >> 2) * kHalfBytes + (k & 3) * 32),
                       smem_desc_k_sw128(W1s + (k >> 2) * (64 * 128) + (k & 3) * 32), id_a, k ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < 8; ++k)      // G(g) = g_out [128 x 128] * W2'[:, chunk] : B MN-major [128 K rows][64]
              umma_f16(tG(a & 1), smem_desc_k_sw128(gbuf + (k >> 2) * kHalfBytes + (k & 3) * 32),
                       smem_desc_mn_sw128(W2s + k * 2048, kHalfBytes), id_g, k ? 1u : 0u);
            umma_commit(&w2_empty[s2]);
            umma_commit(&ag_full[a & 1]);
            if ((a & 7) == 7) umma_commit(g_free);
            if (++s1a == kRingW1B) { s1a = 0; p1a ^= 1; }
            if (++s2 == kRing) { s2 = 0; p2 ^= 1; }
            ++a;
          }
        }
      }
    }
  } else if (warp < kFirstOutWarp) {
    // ===================== LayerNorm warps: y1 -> xhat (in place) + rstd; the tile also leaves as xhat[P,128] =====================
    const int q = warp & 3, row = q * 32 + lane;
    const bool leader = (warp == 2 && lane == 0);
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      unsigned char* u = xbuf(b);
      if (leader && n > 0) {               // the previous tile's xhat store has read its buffer: one of its x_free arrivals
        bulk_wait_read_all();
        mbar_arrive(&x_free[(n - 1) & 1]);
      }
      if (row == 0) stamp(P, 1, 0, n);
      mbar_wait(&y_full[b], (n >> 1) & 1);
      if (row == 0) stamp(P, 1, 1, n);
      const float x0 = up_lo<FMT>(row_chunk(u, row, 0)->x);
      float s = 0.f, ss = 0.f;
#pragma unroll
      for (int c = 0; c < 16; ++c) {
        const uint4 w = *row_chunk(u, row, c);
        const float d0 = up_lo<FMT>(w.x) - x0, d1 = up_hi<FMT>(w.x) - x0, d2 = up_lo<FMT>(w.y) - x0, d3 = up_hi<FMT>(w.y) - x0;
        const float d4 = up_lo<FMT>(w.z) - x0, d5 = up_hi<FMT>(w.z) - x0, d6 = up_lo<FMT>(w.w) - x0, d7 = up_hi<FMT>(w.w) - x0;
        s += ((d0 + d1) + (d2 + d3)) + ((d4 + d5) + (d6 + d7));
        ss += fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3) + (fmaf(d4, d4, d5 * d5) + fmaf(d6, d6, d7 * d7));
      }
      const float md = s * (1.f / kC);
      const float rstd = rsqrtf(fmaxf(ss * (1.f / kC) - md * md, 0.f) + P.eps);
      const float shift = -(x0 + md) * rstd;
      srs[b * kTileM + row] = rstd;
#pragma unroll 4
      for (int c = 0; c < 16; ++c) {
        uint4* p = row_chunk(u, row, c);
        const uint4 w = *p;
        uint4 o;
        o.x = pack2h<FMT>(fmaf(up_lo<FMT>(w.x), rstd, shift), fmaf(up_hi<FMT>(w.x), rstd, shift));
        o.y = pack2h<FMT>(fmaf(up_lo<FMT>(w.y), rstd, shift), fmaf(up_hi<FMT>(w.y), rstd, shift));
        o.z = pack2h<FMT>(fmaf(up_lo<FMT>(w.z), rstd, shift), fmaf(up_hi<FMT>(w.z), rstd, shift));
        o.w = pack2h<FMT>(fmaf(up_lo<FMT>(w.w), rstd, shift), fmaf(up_hi<FMT>(w.w), rstd, shift));
        *p = o;
      }
      fence_proxy_async();
      mbar_arrive(&u_ready[b]);
      if (row == 0) stamp(P, 1, 2, n);
      named_bar_sync(1, 32 * kLnWarps);
      if (leader) {
        tma_store_2d(&tmXhat, u, 0, tile * kTileM);
        tma_store_2d(&tmXhat, u + kHalfBytes, 64, tile * kTileM);
        bulk_commit();
      }
    }
    if (leader && n_local > 0) { bulk_wait_all(); mbar_arrive(&x_free[(n_local - 1) & 1]); }
  } else if (warp < kFirstGeluWarp) {
    // ===================== final warps: U = dL/dxhat -> LayerNorm backward -> g_y1 row, in place over the xhat tile =====================
    // (thread = row = TMEM lane; the residual "+ g_out" is added by the consumer of g_y1, b200_swin_partition)
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool leader = (warp == kFirstOutWarp && lane == 0);
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      unsigned char* u = xbuf(b);
      if (row == 0) stamp(P, 2, 0, n);
      mbar_wait(&tu_full[b], (n >> 1) & 1);
      fence_after_sync();
      if (row == 0) stamp(P, 2, 1, n);
      const float rstd = srs[b * kTileM + row];
      float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t v[32];
        tmem_ld32(tU(b) + lane_sel + ch * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint4 w = *row_chunk(u, row, ch * 4 + c);
          const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float g0 = __uint_as_float(v[c * 8 + 2 * e]), g1 = __uint_as_float(v[c * 8 + 2 * e + 1]);
            s1 += g0 + g1;
            s2 = fmaf(g0, up_lo<FMT>(ww[e]), s2);
            s2 = fmaf(g1, up_hi<FMT>(ww[e]), s2);
          }
        }
      }
      const float m1 = s1 * (1.f / kC), m2 = s2 * (1.f / kC);
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t v[32];
        tmem_ld32(tU(b) + lane_sel + ch * 32, v);
        tmem_ld_wait();
        if (ch == 3) { fence_before_sync(); mbar_arrive(&tu_free[b]); }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4* p = row_chunk(u, row, ch * 4 + c);
          const uint4 w = *p;
          const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
          uint32_t o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e)
            o[e] = pack2h<FMT>(rstd * (__uint_as_float(v[c * 8 + 2 * e]) - m1 - up_lo<FMT>(ww[e]) * m2),
                               rstd * (__uint_as_float(v[c * 8 + 2 * e + 1]) - m1 - up_hi<FMT>(ww[e]) * m2));
          *p = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
      fence_proxy_async();
      named_bar_sync(4, 32 * kOutWarps);
      if (leader) {
        tma_store_2d(&tmGy, u, 0, tile * kTileM);
        tma_store_2d(&tmGy, u + kHalfBytes, 64, tile * kTileM);
        bulk_commit();
        bulk_wait_read_all();
        mbar_arrive(&x_free[b]);
      }
      if (row == 0) stamp(P, 2, 2, n);
    }
    if (leader) bulk_wait_all();
  } else if (warp < kLoaderWarp) {
    // ===================== GELU-backward warps: two groups of 8 on alternate 64-column chunks =====================
    const int gw = warp - kFirstGeluWarp;
    const int grp = gw >> 3;
    const int q = warp & 3, cs = (gw >> 2) & 1;      // TMEM lane quadrant, 32-column half of the chunk
    const int row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool leader = ((gw & 7) == 0 && lane == 0);
    unsigned char* ga = gabuf(grp);
    bool pending = false;
    for (int g = grp; g < n_chunks; g += 2) {
      const uint32_t ph = (g >> 1) & 1;
      const int t = g >> 3, j = g & 7;
      const float4* bias = reinterpret_cast<const float4*>(P.b1f + j * 64 + cs * 32);   // 2 KB, L1 resident
      if (leader) stamp(P, 3, 0, g);
      mbar_wait(&ag_full[grp], ph);
      fence_after_sync();
      if (leader) stamp(P, 3, 1, g);
      mbar_wait(&ga_free[grp], ph ^ 1);              // MMA_u(g-2) has consumed the g_a tile ...
      if (pending) {                                 // ... and the TMA stores of chunk g-2 have read both staging tiles
        if (leader) bulk_wait_read_all();
        named_bar_sync(2 + grp, 16 * kGeluWarps);
      }
#pragma unroll 1
      for (int r2 = 0; r2 < 2; ++r2) {
        uint32_t va[16], vg[16];
        tmem_ld16(tA(grp) + lane_sel + cs * 32 + r2 * 16, va);
        tmem_ld16(tG(grp) + lane_sel + cs * 32 + r2 * 16, vg);
        tmem_ld_wait();
        if (r2 == 1) { fence_before_sync(); mbar_arrive(&ag_tfree[grp]); }
        uint32_t og[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float4 bv = __ldg(bias + r2 * 4 + e);
          const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
          float dd[4];
#pragma unroll
          for (int z = 0; z < 4; ++z) dd[z] = gelu2_tanh5_grad(__uint_as_float(va[4 * e + z]) + bb[z]) * __uint_as_float(vg[4 * e + z]);
          og[2 * e] = pack2h<FMT>(dd[0], dd[1]); og[2 * e + 1] = pack2h<FMT>(dd[2], dd[3]);
        }
        const uint32_t o0 = sw128_offset(row, cs * 4 + r2 * 2), o1 = sw128_offset(row, cs * 4 + r2 * 2 + 1);
        *reinterpret_cast<uint4*>(ga + o0) = make_uint4(og[0], og[1], og[2], og[3]);
        *reinterpret_cast<uint4*>(ga + o1) = make_uint4(og[4], og[5], og[6], og[7]);
      }
      if (leader) stamp(P, 3, 2, g);
      fence_proxy_async();
      named_bar_sync(2 + grp, 16 * kGeluWarps);
      if (leader) {
        stamp(P, 3, 3, g);
        mbar_arrive(&ga_full[grp]);
        const int r0 = (blockIdx.x + t * gridDim.x) * kTileM;
        tma_store_2d(&tmGa, ga, j * 64, r0);
        bulk_commit();
      }
      pending = true;
    }
    if (leader) bulk_wait_all();
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) { fence_after_sync(); tmem_dealloc(tmem_base, 512); }
}

// W1' = W1 * gamma (16-bit), b1' = b1 + W1 beta (f32), W2' = W2 / 2 (16-bit; the kernels produce 2 * gelu).  One warp per W1 row; W2 converted by the same grid.
__global__ void swin_mlp_prep_kernel(const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const float* __restrict__ w2, uint16_t* __restrict__ w1f,
                                     float* __restrict__ b1f, uint16_t* __restrict__ w2h, int C, int hid, int fmt) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp < hid) {
    float acc = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float w = w1[(size_t)warp * C + c];
      acc = fmaf(w, beta[c], acc);
      const float wf = w * gamma[c];
      w1f[(size_t)warp * C + c] = fmt == 1 ? __bfloat16_as_ushort(__float2bfloat16_rn(wf)) : __half_as_ushort(__float2half_rn(wf));
    }
    acc = warp_sum(acc);
    if (lane == 0) b1f[warp] = b1[warp] + acc;
  }
  const int n2 = C * hid;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += gridDim.x * blockDim.x)
    w2h[i] = fmt == 1 ? __bfloat16_as_ushort(__float2bfloat16_rn(0.5f * w2[i])) : __half_as_ushort(__float2half_rn(0.5f * w2[i]));
}

}  // namespace
}  // namespace tc
}  // namespace b200

using namespace b200;

/* debugging aid (not part of the public header): device buffer of 16*64 int64 receiving CTA 0's event clock stamps */
extern "C" B200_API void b200_debug_set_mlp_timeline(void* buf) { g_mlp_dbg = (long long*)buf; }

extern "C" B200_API int b200_swin_mlp_supported(int64_t rows, int32_t C, int32_t dtype) {
  return (dtype == B200_BF16 || dtype == B200_F16) && rows > 0 && rows < (1ll << 31) - 256 && C == tc::kC;
}

extern "C" B200_API int b200_swin_mlp_prep(const float* w1, const float* b1, const float* gamma, const float* beta, const float* w2,
                                           void* w1f, float* b1f, void* w2h, int32_t C, int32_t dtype, void* stream) {
  B200_REQUIRE(dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "swin_mlp_prep: 16-bit dtypes only (got %d)", dtype);
  B200_REQUIRE(C > 0 && w1 && b1 && gamma && beta && w2 && w1f && b1f && w2h, B200_ERR_SHAPE, "swin_mlp_prep: null pointer / bad C");
  const int hid = 4 * C;
  const int threads = 256, blocks = (hid * 32 + threads - 1) / threads;
  tc::swin_mlp_prep_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(w1, b1, gamma, beta, w2, (uint16_t*)w1f, b1f, (uint16_t*)w2h, C, hid,
                                                                         dtype == B200_BF16 ? 1 : 0);
  return check_launch("swin_mlp_prep");
}

extern "C" B200_API int b200_swin_mlp_fwd(const void* y1, const void* w1f, const float* b1f, const void* w2h, const float* b2, void* out,
                                          void* h2, int64_t rows, int32_t C, float eps, int32_t dtype, void* stream) {
  B200_REQUIRE(b200_swin_mlp_supported(rows, C, dtype), B200_ERR_UNSUPPORTED,
               "swin_mlp_fwd: unsupported problem rows=%lld C=%d dtype=%d (16-bit dtypes, C = 128)", (long long)rows, C, dtype);
  B200_REQUIRE(y1 && w1f && b1f && w2h && b2 && out, B200_ERR_SHAPE, "swin_mlp_fwd: null pointer");
  B200_REQUIRE((((uintptr_t)y1 | (uintptr_t)w1f | (uintptr_t)w2h | (uintptr_t)out) & 15) == 0, B200_ERR_ALIGN,
               "swin_mlp_fwd: 16-byte alignment required");
  using namespace b200::tc;
  const CUtensorMap* mY = tensor_map_2d(y1, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  const CUtensorMap* mO = tensor_map_2d(out, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  const CUtensorMap* mW1 = tensor_map_2d(w1f, kHid, kC, kC, 128, 64, dtype);
  const CUtensorMap* mW2 = tensor_map_2d(w2h, kC, kHid, kHid, 128, 64, dtype);
  const CUtensorMap* mH = h2 ? tensor_map_2d(h2, (uint64_t)rows, kHid, kHid, kTileM, 64, dtype) : mO;
  if (!mY || !mO || !mW1 || !mW2 || !mH) return B200_ERR_LAUNCH;
  B200_REQUIRE(((uintptr_t)h2 & 15) == 0, B200_ERR_ALIGN, "swin_mlp_fwd: 16-byte alignment required");
  MlpParams P;
  P.save_h = h2 != nullptr;
  P.b1f = b1f; P.b2 = b2; P.out = out; P.P = rows; P.dbg = g_mlp_dbg; P.n_tiles = (int)((rows + kTileM - 1) / kTileM); P.fmt = dtype == B200_BF16 ? 1 : 0; P.eps = eps;
  const int grid = P.n_tiles < sm_count() ? P.n_tiles : sm_count();
  auto kern = dtype == B200_BF16 ? swin_mlp_fwd_kernel<1> : swin_mlp_fwd_kernel<0>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, MlpSmem::TOTAL);
  kern<<<grid, kThreads, MlpSmem::TOTAL, (cudaStream_t)stream>>>(*mY, *mO, *mW1, *mW2, *mH, P);
  return check_launch("swin_mlp_fwd");
}

extern "C" B200_API int b200_swin_mlp_bwd(const void* gout, const void* y1, const void* w1f, const float* b1f, const void* w2h, void* gy1,
                                          void* xhat, void* ga, int64_t rows, int32_t C, float eps, int32_t dtype, void* stream) {
  B200_REQUIRE(b200_swin_mlp_supported(rows, C, dtype), B200_ERR_UNSUPPORTED,
               "swin_mlp_bwd: unsupported problem rows=%lld C=%d dtype=%d (16-bit dtypes, C = 128)", (long long)rows, C, dtype);
  B200_REQUIRE(gout && y1 && w1f && b1f && w2h && gy1 && xhat && ga, B200_ERR_SHAPE, "swin_mlp_bwd: null pointer");
  B200_REQUIRE((((uintptr_t)gout | (uintptr_t)y1 | (uintptr_t)w1f | (uintptr_t)w2h | (uintptr_t)gy1 | (uintptr_t)xhat | (uintptr_t)ga) & 15) == 0,
               B200_ERR_ALIGN, "swin_mlp_bwd: 16-byte alignment required");
  using namespace b200::tc;
  const CUtensorMap* mY = tensor_map_2d(y1, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  const CUtensorMap* mG = tensor_map_2d(gout, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  const CUtensorMap* mW1 = tensor_map_2d(w1f, kHid, kC, kC, 64, 64, dtype);
  const CUtensorMap* mW2 = tensor_map_2d(w2h, kC, kHid, kHid, 128, 64, dtype);
  const CUtensorMap* mX = tensor_map_2d(xhat, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  const CUtensorMap* mGa = tensor_map_2d(ga, (uint64_t)rows, kHid, kHid, kTileM, 64, dtype);
  const CUtensorMap* mGy = tensor_map_2d(gy1, (uint64_t)rows, kC, kC, kTileM, 64, dtype);
  if (!mY || !mG || !mW1 || !mW2 || !mX || !mGa || !mGy) return B200_ERR_LAUNCH;
  MlpBwdParams P;
  P.b1f = b1f; P.P = rows; P.dbg = g_mlp_dbg; P.n_tiles = (int)((rows + kTileM - 1) / kTileM); P.eps = eps;
  const int grid = P.n_tiles < sm_count() ? P.n_tiles : sm_count();
  auto kern = dtype == B200_BF16 ? swin_mlp_bwd_kernel<1> : swin_mlp_bwd_kernel<0>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, MlpBwdSmem::TOTAL);
  kern<<<grid, kThreads, MlpBwdSmem::TOTAL, (cudaStream_t)stream>>>(*mY, *mG, *mW1, *mW2, *mX, *mGa, *mGy, P);
  return check_launch("swin_mlp_bwd");
}
