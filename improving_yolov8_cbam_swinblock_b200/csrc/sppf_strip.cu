// SPPF pooling cascade (block.py:224-226) and its backward for the plane the model actually uses -- P5 = 20x20 at 640^2 -- with
// 16-bit activations: every strip (a row or a column of one 32-bit lane word = two channels) lives in the REGISTERS of one thread.
//
// The generic kernels (sppf_pool.cu) walk strips of run-time length through shared memory with a ring of K window slots; at
// [64,128,20,20] their backward issues 46 M warp instructions (ncu: issue-bound, 7 % of DRAM peak).  Here the side is a compile-time
// constant, so a whole strip is 20 registers, every window index, boundary and shared-memory offset is an immediate, and the passes
// are straight-line code:
//   * values: windowed maxima by doubling (p2 = max of 2 neighbours, p4 = max of two p2, ...): ~3 packed HMNMX2 per output word
//     for any K, on the raw 16-bit pairs (the tile is checked for NaN / -0.0 while it is loaded: exactly the two cases where the
//     hardware max differs from ATen's `v > best || isnan(v)` scan; such a tile takes the exact scalar passes of sppf_word.cuh);
//   * winners (backward only): first window position whose value equals the maximum -- one packed compare (HSET2.BM) + one LOP3
//     select per candidate, scanned right to left so the leftmost match survives = ATen's first-occurrence rule; kept as one byte
//     per word (4 + 4 bits, the format of the generic kernel) in shared memory;
//   * routing: a gather in registers: target t sums, in ascending source order, the <= K sources whose winner offset points at it
//     (fixed order, no atomics: deterministic), IN PLACE over the one f32 gradient plane, which itself overlays the two value planes.
// Nothing is staged: the y0 strip, the four concat-slice gradients and the result go straight between global memory and the
// registers of the thread that owns the strip (64 contiguous bytes per pixel and half-warp).
// CTA = (image, 32 channels): 320 threads = 20 strips x 16 words; eleven passes with a barrier between them.
#include <stdlib.h>

#include "common.cuh"
#include "sppf_word.cuh"

namespace b200 {
namespace {
using sppf::pass1d;
using sppf::Word;

constexpr int S = 20;           // plane side
constexpr int WP = S + 1;       // row pitch in pixels (odd: the two strips of a warp land 16 banks apart in both directions)
constexpr int CW = 16;          // lane words per pixel in a CTA's chunk (32 channels = 64 bytes)
constexpr int NT = S * CW;      // one strip per thread
constexpr int PW = S * WP * CW; // words (or bytes of the winner planes) per plane

template <typename T> struct Pair;
template <> struct Pair<__nv_bfloat16> {
  __device__ static __forceinline__ uint32_t eq(uint32_t a, uint32_t b) {
    return __heq2_mask(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
  }
  __device__ static __forceinline__ float lo(uint32_t w) { return __uint_as_float(w << 16); }
  __device__ static __forceinline__ float hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};
template <> struct Pair<__half> {
  __device__ static __forceinline__ uint32_t eq(uint32_t a, uint32_t b) {
    return __heq2_mask(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
  }
  __device__ static __forceinline__ float lo(uint32_t w) { return __low2float(*reinterpret_cast<const __half2*>(&w)); }
  __device__ static __forceinline__ float hi(uint32_t w) { return __high2float(*reinterpret_cast<const __half2*>(&w)); }
  __device__ static __forceinline__ uint32_t pack(float a, float b) {
    const __half2 p = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};

// m[i] = max of v over the window [i-R, i+R] clipped to the strip; ob[i] (WANT_OFF) = winner offsets of the two halves,
// (lo | hi << 4), offset = winner position - (i - R), first occurrence.
template <typename T, int K, bool WANT_OFF>
__device__ __forceinline__ void strip_max(const uint32_t (&v)[S], uint32_t (&m)[S], uint32_t (&ob)[S]) {
  using WD = Word<T>;
  constexpr int R = K / 2;
  uint32_t p2[S], p4[S], p8[S];   // p<L>[i] = max(v[i .. i+L-1]) where it exists
#pragma unroll
  for (int i = 0; i + 1 < S; ++i) p2[i] = WD::vmax(v[i], v[i + 1]);
#pragma unroll
  for (int i = 0; i + 3 < S; ++i) p4[i] = WD::vmax(p2[i], p2[i + 2]);
  if constexpr (K >= 8) {
#pragma unroll
    for (int i = 0; i + 7 < S; ++i) p8[i] = WD::vmax(p4[i], p4[i + 4]);
  }
#pragma unroll
  for (int i = 0; i < S; ++i) {
    const int lo = i - R < 0 ? 0 : i - R, hi = i + R > S - 1 ? S - 1 : i + R, len = hi - lo + 1;
    uint32_t mx;
    if (len >= 8 && K >= 8) mx = WD::vmax(p8[lo], p8[hi - 7]);
    else if (len >= 4) mx = WD::vmax(p4[lo], p4[hi - 3]);
    else if (len >= 2) mx = WD::vmax(p2[lo], p2[hi - 1]);
    else mx = v[lo];
    m[i] = mx;
    if (WANT_OFF) {
      uint32_t o = (uint32_t)(hi - (i - R)) * 0x00010001u;
#pragma unroll
      for (int d = K - 2; d >= 0; --d) {           // window slot d <-> position i - R + d, right to left: the leftmost match survives
        const int j = i - R + d;
        if (j >= lo && j < hi) {
          const uint32_t e = Pair<T>::eq(v[j], mx);
          o = (e & ((uint32_t)d * 0x00010001u)) | (~e & o);
        }
      }
      ob[i] = (o | (o >> 12)) & 0xffu;
    }
  }
}

// dst(t) = sum, in ascending source order, of the sources whose winner is t.  Source-major: source i is fetched (src(i), off(i)),
// tested against its K possible targets (one packed compare for both halves + two predicated adds, the predicates consumed at once -- the target-major form made
// the compiler park dozens of predicates in bit masks) and target i - R, now complete, leaves through dst: about 2K live
// accumulators instead of whole strips, and the walk may run IN PLACE (position t is written after source t + R was read).
template <int K, class SRC, class OFF, class DST>
__device__ __forceinline__ void strip_route(SRC src, OFF off, DST dst) {
  constexpr int R = K / 2;
  float a0[S], a1[S];
#pragma unroll
  for (int t = 0; t < S; ++t) { a0[t] = 0.f; a1[t] = 0.f; }
#pragma unroll
  for (int i = 0; i < S; ++i) {
    const float2 gi = src(i);
    const uint32_t ob = off(i);
    const uint32_t x = ((ob << 12) | ob) & 0x000f000fu;   // the two offsets as the halves of an f16x2 (tiny denormals: exact compare)
#pragma unroll
    for (int o = 0; o < K; ++o) {
      const int t = i - R + o;
      if (t >= 0 && t < S) {
        // one packed compare yields both predicates (HSETP2), consumed at once by the two conditional adds
        asm("{\n\t.reg .pred p, q;\n\t"
            "setp.eq.f16x2 p|q, %2, %3;\n\t"
            "@p add.f32 %0, %0, %4;\n\t"
            "@q add.f32 %1, %1, %5;\n\t}"
            : "+f"(a0[t]), "+f"(a1[t]) : "r"(x), "r"((uint32_t)o * 0x00010001u), "f"(gi.x), "f"(gi.y));
      }
    }
    if (i - R >= 0) dst(i - R, make_float2(a0[i - R], a1[i - R]));
  }
#pragma unroll
  for (int t = S - R; t < S; ++t) dst(t, make_float2(a0[t], a1[t]));
}

template <typename T, int K>
__global__ void __launch_bounds__(NT, 2) sppf_strip_bwd_kernel(const T* __restrict__ gcat, const T* __restrict__ y0, T* __restrict__ gy0,
                                                               int C) {
  using WD = Word<T>;
  using PR = Pair<T>;
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t* Bp = smem;                                   // word plane B | the f32 gradient plane overlays B and A once the
  uint32_t* A = smem + PW;                               // word plane A | cascade has been recomputed
  float2* G = reinterpret_cast<float2*>(smem);           // [S][WP][CW] float2
  uint8_t* O = reinterpret_cast<uint8_t*>(smem + 2 * PW);   // [6][S][WP][CW] winner bytes of the six forward passes

  const int w = threadIdx.x & (CW - 1), s = threadIdx.x / CW;
  const int chunks = C / (2 * CW);
  const int b = blockIdx.x / chunks, c0 = (blockIdx.x - b * chunks) * (2 * CW);
  const size_t cw = (size_t)C / 2;                       // words per pixel of y0 / gy0; the concat has 4 * cw
  const uint32_t* yin = reinterpret_cast<const uint32_t*>(y0) + (size_t)b * S * S * cw + c0 / 2 + w;
  const uint32_t* gin = reinterpret_cast<const uint32_t*>(gcat) + (size_t)b * S * S * 4 * cw + c0 / 2 + w;
  uint32_t* gout = reinterpret_cast<uint32_t*>(gy0) + (size_t)b * S * S * cw + c0 / 2 + w;
  // element e of row strip s = pixel (s, e); of column strip s = pixel (e, s)
  const int rbase = s * WP * CW + w, cbase = s * CW + w;
  constexpr int RS = CW, CS = WP * CW;

  uint32_t v[S], m[S], ob[S];
  uint32_t gw[S], gn[S];   // concat-slice gradient strips, fetched one phase before they are consumed
  auto fetch_g3 = [&]() {
#pragma unroll
    for (int e = 0; e < S; ++e) gw[e] = __ldg(gin + 3 * cw + (size_t)(e * S + s) * 4 * cw);       // column strip
  };
  auto fetch_row = [&](int slice) {
#pragma unroll
    for (int e = 0; e < S; ++e) gn[e] = __ldg(gin + (size_t)slice * cw + (size_t)(s * S + e) * 4 * cw);
  };
#pragma unroll
  for (int e = 0; e < S; ++e) v[e] = __ldg(yin + (size_t)(s * S + e) * cw);
  int special = 0;
#pragma unroll
  for (int e = 0; e < S; ++e) special |= WD::special(v[e]) ? 1 : 0;
  special = __syncthreads_or(special);

  if (!special) {
#pragma unroll 1
    for (int st = 0; st < 3; ++st) {
      if (st == 2) fetch_g3();
      if (st > 0) {
#pragma unroll
        for (int e = 0; e < S; ++e) v[e] = Bp[rbase + e * RS];
      }
      strip_max<T, K, true>(v, m, ob);
      uint8_t* orow = O + (size_t)(2 * st) * PW;
#pragma unroll
      for (int e = 0; e < S; ++e) { A[rbase + e * RS] = m[e]; orow[rbase + e * RS] = (uint8_t)ob[e]; }
      __syncthreads();
#pragma unroll
      for (int e = 0; e < S; ++e) v[e] = A[cbase + e * CS];
      if (st == 2) break;
      strip_max<T, K, true>(v, m, ob);
      uint8_t* ocol = O + (size_t)(2 * st + 1) * PW;
#pragma unroll
      for (int e = 0; e < S; ++e) { Bp[cbase + e * CS] = m[e]; ocol[cbase + e * CS] = (uint8_t)ob[e]; }
      __syncthreads();
    }
    __syncthreads();   // every thread holds its stage-3 column strip: the gradient plane may now overwrite A and B
    strip_max<T, K, true>(v, m, ob);
  } else {
    // exact scalar passes (ATen's update rule) through shared memory; same winner format
    fetch_g3();
#pragma unroll
    for (int e = 0; e < S; ++e) A[rbase + e * RS] = v[e];
    __syncthreads();
#pragma unroll 1
    for (int st = 0; st < 3; ++st) {
      pass1d<T, K>(A + rbase, RS, Bp + rbase, RS, S, O + (size_t)(2 * st) * PW + rbase, RS);
      __syncthreads();
      pass1d<T, K>(Bp + cbase, CS, A + cbase, CS, S, O + (size_t)(2 * st + 1) * PW + cbase, CS);
      __syncthreads();
    }
#pragma unroll
    for (int e = 0; e < S; ++e) ob[e] = O[(size_t)5 * PW + cbase + e * CS];
  }

  // stage-3 column pass backward on G3 = g3 (straight from global memory), the winners still in registers
  fetch_row(2);
  strip_route<K>([&](int i) { return make_float2(PR::lo(gw[i]), PR::hi(gw[i])); }, [&](int i) { return ob[i]; },
                 [&](int t_, float2 r) { G[cbase + t_ * CS] = r; });
  __syncthreads();
#pragma unroll 1
  for (int st = 2; st >= 0; --st) {
    if (st < 2) {   // column pass backward of stage st + 1, in place
      const uint8_t* ocol = O + (size_t)(2 * st + 1) * PW;
      strip_route<K>([&](int i) { return G[cbase + i * CS]; }, [&](int i) { return (uint32_t)ocol[cbase + i * CS]; },
                     [&](int t_, float2 r) { G[cbase + t_ * CS] = r; });
      __syncthreads();
    }
    // row pass backward, then + the concat-slice gradient g_st (block.py:226: slice st of the concat IS this stage's input)
#pragma unroll
    for (int e = 0; e < S; ++e) gw[e] = gn[e];
    if (st > 0) fetch_row(st - 1);
    const uint8_t* orow = O + (size_t)(2 * st) * PW;
    if (st > 0) {
      strip_route<K>([&](int i) { return G[rbase + i * RS]; }, [&](int i) { return (uint32_t)orow[rbase + i * RS]; },
                     [&](int t_, float2 r) { G[rbase + t_ * RS] = make_float2(r.x + PR::lo(gw[t_]), r.y + PR::hi(gw[t_])); });
      __syncthreads();
    } else {
      strip_route<K>([&](int i) { return G[rbase + i * RS]; }, [&](int i) { return (uint32_t)orow[rbase + i * RS]; },
                     [&](int t_, float2 r) { gout[(size_t)(s * S + t_) * cw] = PR::pack(r.x + PR::lo(gw[t_]), r.y + PR::hi(gw[t_])); });
    }
  }
}

template <typename T, int K>
__global__ void __launch_bounds__(NT, 3) sppf_strip_fwd_kernel(const T* __restrict__ y0, T* __restrict__ cat, int C) {
  using WD = Word<T>;
  extern __shared__ __align__(16) uint32_t smem[];
  uint32_t* Bp = smem;
  uint32_t* A = smem + PW;
  const int w = threadIdx.x & (CW - 1), s = threadIdx.x / CW;
  const int chunks = C / (2 * CW);
  const int b = blockIdx.x / chunks, c0 = (blockIdx.x - b * chunks) * (2 * CW);
  const size_t cw = (size_t)C / 2;
  const uint32_t* yin = reinterpret_cast<const uint32_t*>(y0) + (size_t)b * S * S * cw + c0 / 2 + w;
  uint32_t* out = reinterpret_cast<uint32_t*>(cat) + (size_t)b * S * S * 4 * cw + c0 / 2 + w;   // slice k at + k * cw
  const int rbase = s * WP * CW + w, cbase = s * CW + w;
  constexpr int RS = CW, CS = WP * CW;

  uint32_t v[S], m[S], ob[S];
#pragma unroll
  for (int e = 0; e < S; ++e) v[e] = __ldg(yin + (size_t)(s * S + e) * cw);
  int special = 0;
#pragma unroll
  for (int e = 0; e < S; ++e) {
    out[(size_t)(s * S + e) * 4 * cw] = v[e];            // concat slice 0 = y0
    special |= WD::special(v[e]) ? 1 : 0;
  }
  special = __syncthreads_or(special);
  if (!special) {
#pragma unroll 1
    for (int st = 0; st < 3; ++st) {
      if (st > 0) {
#pragma unroll
        for (int e = 0; e < S; ++e) v[e] = Bp[rbase + e * RS];
      }
      strip_max<T, K, false>(v, m, ob);
#pragma unroll
      for (int e = 0; e < S; ++e) A[rbase + e * RS] = m[e];
      __syncthreads();
#pragma unroll
      for (int e = 0; e < S; ++e) v[e] = A[cbase + e * CS];
      strip_max<T, K, false>(v, m, ob);
      uint32_t* os = out + (size_t)(st + 1) * cw;
#pragma unroll
      for (int e = 0; e < S; ++e) {
        if (st < 2) Bp[cbase + e * CS] = m[e];
        os[(size_t)(e * S + s) * 4 * cw] = m[e];
      }
      if (st < 2) __syncthreads();
    }
  } else {
#pragma unroll
    for (int e = 0; e < S; ++e) A[rbase + e * RS] = v[e];
    __syncthreads();
#pragma unroll 1
    for (int st = 0; st < 3; ++st) {
      pass1d<T, K>(A + rbase, RS, Bp + rbase, RS, S, nullptr, 0);
      __syncthreads();
      pass1d<T, K>(Bp + cbase, CS, A + cbase, CS, S, nullptr, 0);
      uint32_t* os = out + (size_t)(st + 1) * cw;
#pragma unroll
      for (int e = 0; e < S; ++e) os[(size_t)(e * S + s) * 4 * cw] = A[cbase + e * CS];   // own column strip: no barrier needed
      __syncthreads();
    }
  }
}

bool strip_shape(int C, int H, int W, int k, int dtype) {
  if (const char* off = getenv("B200_SPPF_NO_STRIP")) if (off[0] == '1') return false;   // A/B aid: force the generic kernels
  return H == S && W == S && C % (2 * CW) == 0 && (dtype == B200_BF16 || dtype == B200_F16) && k >= 3 && k <= 13 && (k & 1);
}

template <typename T, int K>
int launch_bwd(const void* gcat, const void* y0, void* gy0, int B, int C, cudaStream_t st) {
  constexpr int smem = PW * 8 + PW * 6;
  auto kern = sppf_strip_bwd_kernel<T, K>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  kern<<<B * (C / (2 * CW)), NT, smem, st>>>((const T*)gcat, (const T*)y0, (T*)gy0, C);
  return check_launch("sppf_pool_bwd(strip)");
}
template <typename T, int K>
int launch_fwd(const void* y0, void* cat, int B, int C, cudaStream_t st) {
  constexpr int smem = PW * 8;
  auto kern = sppf_strip_fwd_kernel<T, K>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  kern<<<B * (C / (2 * CW)), NT, smem, st>>>((const T*)y0, (T*)cat, C);
  return check_launch("sppf_pool_fwd(strip)");
}

#define B200_STRIP_K(k, ...)                                   \
  switch (k) {                                                 \
    case 3: { constexpr int K = 3; return __VA_ARGS__; }       \
    case 5: { constexpr int K = 5; return __VA_ARGS__; }       \
    case 7: { constexpr int K = 7; return __VA_ARGS__; }       \
    case 9: { constexpr int K = 9; return __VA_ARGS__; }       \
    case 11: { constexpr int K = 11; return __VA_ARGS__; }     \
    default: { constexpr int K = 13; return __VA_ARGS__; }     \
  }

}  // namespace

namespace sppf {
int strip_fwd(const void* y0, void* cat, int B, int C, int H, int W, int k, int dtype, cudaStream_t st) {
  if (!strip_shape(C, H, W, k, dtype)) return -1;
  if (dtype == B200_BF16) { B200_STRIP_K(k, launch_fwd<__nv_bfloat16, K>(y0, cat, B, C, st)) }
  B200_STRIP_K(k, launch_fwd<__half, K>(y0, cat, B, C, st))
}
int strip_bwd(const void* gcat, const void* y0, void* gy0, int B, int C, int H, int W, int k, int dtype, cudaStream_t st) {
  if (!strip_shape(C, H, W, k, dtype)) return -1;
  if (dtype == B200_BF16) { B200_STRIP_K(k, launch_bwd<__nv_bfloat16, K>(gcat, y0, gy0, B, C, st)) }
  B200_STRIP_K(k, launch_bwd<__half, K>(gcat, y0, gy0, B, C, st))
}
}  // namespace sppf
}  // namespace b200
