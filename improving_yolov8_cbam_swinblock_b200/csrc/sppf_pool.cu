// SPPF pooling cascade: three chained stride-1 "same" max-pools + the 4-way channel concat, computed from ONE
// shared-memory-staged tile per (image, channel chunk).  Replaces block.py:224-226 of the reference.
//
// Layout: NHWC.  A CTA owns image b, channels [c0, c0 + LP*EPL) over the WHOLE H x W plane (the reference only
// uses SPPF at P5 = 20x20; larger planes shrink LP so the plane still fits in shared memory).  One 32-bit word
// per lane = EPL elements (1 f32 / 2 bf16|f16), LP lanes per pixel, so a pixel's chunk is LP*4 contiguous bytes.
// Each max-pool is separable: a row pass (threads walk rows) into `tmp`, a column pass (threads walk columns)
// back into `cur` + straight to the concat slice in global memory.  Both passes use ATen's exact update rule
// "take iff (v > best) || isnan(v)", scanning left->right / top->bottom, which composes to the row-major
// first-occurrence argmax of max_pool2d_with_indices (and "last NaN wins").
//
// Backward: the per-stage winners (row offset, col offset: 4+4 bits) are recomputed from y0 with the same rule,
// then gradients are routed stage 3 -> 1 by two 1-D scatters per stage.  Every strip (row / column, channel)
// is owned by exactly one thread, so the scatter is race-free and summation order is fixed: deterministic.
#include "common.cuh"
#include "sppf_word.cuh"

namespace b200 {
namespace {
using sppf::Word;
using sppf::pass1d;

// Values-only 1-D max pass with packed hardware max (HMNMX2 / FMNMX).  Exact selection as long as the tile has no
// NaN and no -0.0 (the two cases where a hardware max differs from ATen's `v > best || isnan(v)` scan).
// Optionally also stores every output word to global memory (the concat slice) with stride gstride words.
template <typename T, int K>
__device__ __forceinline__ void pass1d_fast(const uint32_t* __restrict__ src, int sstride, uint32_t* __restrict__ dst,
                                            int dstride, int len, uint32_t* __restrict__ gdst, size_t gstride) {
  using WD = Word<T>;
  constexpr int R = K / 2;
  uint32_t win[K];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int p = j - R;
    win[j] = (p >= 0 && p < len) ? src[p * sstride] : WD::neg_inf();
  }
  for (int i = 0; i < len; ++i) {
    uint32_t o = win[0];
#pragma unroll
    for (int j = 1; j < K; ++j) o = WD::vmax(o, win[j]);
    dst[i * dstride] = o;
    if (gdst) gdst[(size_t)i * gstride] = o;
#pragma unroll
    for (int j = 0; j < K - 1; ++j) win[j] = win[j + 1];
    const int p = i + 1 + R;
    win[K - 1] = (p < len) ? src[p * sstride] : WD::neg_inf();
  }
}

// Winner-tracking 1-D pass for 16-bit types via packed integer keys: key = sortable16(value) << 16 | (0xFFFF - pos),
// so one unsigned max picks the larger value and, among equal values, the smaller position (first occurrence).
// Same validity condition as pass1d_fast (no NaN / -0.0 in the tile); out-of-range slots carry key 0 (never win).
// The tile is held in the SORTABLE domain (to_sortable2 applied once at load time): an order-preserving bijection, so the
// cascade's values never have to be decoded -- the backward only needs the winners.  The K-slot window is a ring buffer
// (max is commutative; the position lives in the key), the loop is unrolled K times so slot indices are static.
__device__ __forceinline__ uint32_t to_sortable2(uint32_t w) {     // per 16-bit half: negative -> ~v, else v ^ 0x8000
  return w ^ ((((w >> 15) & 0x00010001u) * 0x7fffu) | 0x80008000u);
}
__device__ __forceinline__ uint32_t from_sortable2(uint32_t k) {
  return k ^ ((((~k >> 15) & 0x00010001u) * 0x7fffu) | 0x80008000u);
}
template <typename T, int K>
__device__ __forceinline__ void pass1d_key(const uint32_t* __restrict__ src, int sstride, uint32_t* __restrict__ dst,
                                           int dstride, int len, uint8_t* __restrict__ win_out, int wstride, int i0, int i1) {
  static_assert(Word<T>::EPL == 2, "key path is for 16-bit types");
  constexpr int R = K / 2;
  uint32_t k0[K], k1[K];
  // slot (p - (i0 - R)) mod K holds source position p
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int p = i0 + j - R;
    if (p >= 0 && p < len) {
      const uint32_t w = src[p * sstride], pinv = 0xffffu - (uint32_t)p;
      k0[j] = (w << 16) | pinv;
      k1[j] = (w & 0xffff0000u) | pinv;
    } else { k0[j] = 0u; k1[j] = 0u; }
  }
  for (int ib = i0; ib < i1; ib += K) {
#pragma unroll
    for (int u = 0; u < K; ++u) {
      const int i = ib + u;
      if (i < i1) {
        uint32_t b0 = k0[0], b1 = k1[0];
#pragma unroll
        for (int j = 1; j < K; ++j) { b0 = max(b0, k0[j]); b1 = max(b1, k1[j]); }
        dst[i * dstride] = __byte_perm(b0, b1, 0x7632);            // (b0 >> 16) | (b1 & 0xffff0000)
        const uint32_t base = 0xffffu - (uint32_t)(i - R);          // offset in the window = pos - (i - R)
        win_out[i * wstride] = (uint8_t)((base - (b0 & 0xffffu)) | ((base - (b1 & 0xffffu)) << 4));
        const int p = i + 1 + R;                                    // replaces the oldest slot: position i - R = slot u
        if (p < len) {
          const uint32_t w = src[p * sstride], pinv = 0xffffu - (uint32_t)p;
          k0[u] = (w << 16) | pinv;
          k1[u] = (w & 0xffff0000u) | pinv;
        } else { k0[u] = 0u; k1[u] = 0u; }
      }
    }
  }
}
template <typename T, int K, bool IS16 = (Word<T>::EPL == 2)> struct KeyPass {
  __device__ static __forceinline__ void run(const uint32_t* src, int ss, uint32_t* dst, int ds, int len, uint8_t* w, int ws,
                                             int i0, int i1) {
    pass1d_key<T, K>(src, ss, dst, ds, len, w, ws, i0, i1);
  }
};
template <typename T, int K> struct KeyPass<T, K, false> {
  __device__ static __forceinline__ void run(const uint32_t* src, int ss, uint32_t* dst, int ds, int len, uint8_t* w, int ws,
                                             int i0, int i1) {
    pass1d<T, K>(src, ss, dst, ds, len, w, ws, i0, i1);
  }
};

// ---- cooperative, vectorised tile movers ------------------------------------------------------------------
// pixel index -> (y, x) without an integer division (exact for p < 2^22)
__device__ __forceinline__ void pix_yx(int p, int W, float invW, int* y, int* x) {
  int yy = __float2int_rz(((float)p + 0.5f) * invW);
  *y = yy; *x = p - yy * W;
}
// global words [H*W pixels][LP words] (pixel stride gstride words) -> smem [H][Wp][LP]; returns OR of Word::special
// (and mirrors the words to gcopy when non-null: concat slice 0).  16-byte path when everything is aligned.
template <typename T, int LP>
__device__ __forceinline__ int tile_load_words(uint32_t* __restrict__ sm, const uint32_t* __restrict__ gsrc, size_t gstride,
                                               uint32_t* __restrict__ gcopy, size_t cstride, int H, int W, int Wp,
                                               int valid_words, uint32_t fill) {
  using WD = Word<T>;
  int special = 0;
  const float invW = 1.f / (float)W;
  const bool vec = (LP % 4 == 0) && valid_words == LP && (gstride % 4 == 0) && ((reinterpret_cast<uintptr_t>(gsrc) & 15) == 0) &&
                   (!gcopy || ((cstride % 4 == 0) && (reinterpret_cast<uintptr_t>(gcopy) & 15) == 0));
  if (vec) {
    constexpr int VPP = LP / 4 > 0 ? LP / 4 : 1;
    const int items = H * W * VPP;
    for (int it0 = threadIdx.x; it0 < items; it0 += 4 * blockDim.x) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int it = it0 + u * blockDim.x;
        if (it < items) {
          const int p = it / VPP, q = it - p * VPP;
          v[u] = ldg_stream16(gsrc + (size_t)p * gstride + q * 4);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int it = it0 + u * blockDim.x;
        if (it < items) {
          const int p = it / VPP, q = it - p * VPP;
          int y, x;
          pix_yx(p, W, invW, &y, &x);
          *reinterpret_cast<uint4*>(sm + (size_t)(y * Wp + x) * LP + q * 4) = v[u];
          if (gcopy) *reinterpret_cast<uint4*>(gcopy + (size_t)p * cstride + q * 4) = v[u];
          special |= (WD::special(v[u].x) || WD::special(v[u].y) || WD::special(v[u].z) || WD::special(v[u].w)) ? 1 : 0;
        }
      }
    }
  } else {
    const int items = H * W * LP;
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
      const int p = it / LP, l = it - p * LP;
      int y, x;
      pix_yx(p, W, invW, &y, &x);
      uint32_t w = fill;
      if (l < valid_words) {
        w = gsrc[(size_t)p * gstride + l];
        if (gcopy) gcopy[(size_t)p * cstride + l] = w;
        special |= WD::special(w) ? 1 : 0;
      }
      sm[(size_t)(y * Wp + x) * LP + l] = w;
    }
  }
  return special;
}
// global words -> smem f32 [H][Wp][LP][EPL] (set or accumulate)
template <typename T, int LP, bool ACC>
__device__ __forceinline__ void tile_load_f32(float* __restrict__ sm, const uint32_t* __restrict__ gsrc, size_t gstride, int H,
                                              int W, int Wp, int valid_words) {
  using WD = Word<T>;
  constexpr int EPL = WD::EPL;
  const float invW = 1.f / (float)W;
  const bool vec = (LP % 4 == 0) && valid_words == LP && (gstride % 4 == 0) && ((reinterpret_cast<uintptr_t>(gsrc) & 15) == 0);
  if (vec) {
    constexpr int VPP = LP / 4 > 0 ? LP / 4 : 1;
    const int items = H * W * VPP;
    for (int it0 = threadIdx.x; it0 < items; it0 += 4 * blockDim.x) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int it = it0 + u * blockDim.x;
        if (it < items) {
          const int p = it / VPP, q = it - p * VPP;
          v[u] = ldg_stream16(gsrc + (size_t)p * gstride + q * 4);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int it = it0 + u * blockDim.x;
        if (it < items) {
          const int p = it / VPP, q = it - p * VPP;
          int y, x;
          pix_yx(p, W, invW, &y, &x);
          float* d = sm + ((size_t)(y * Wp + x) * LP + q * 4) * EPL;
          const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int e = 0; e < EPL; ++e) {
              const float f = WD::bits_to_f(WD::bits(w[k], e));
              d[k * EPL + e] = ACC ? d[k * EPL + e] + f : f;
            }
        }
      }
    }
  } else {
    const int items = H * W * LP;
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
      const int p = it / LP, l = it - p * LP;
      int y, x;
      pix_yx(p, W, invW, &y, &x);
      const uint32_t w = l < valid_words ? gsrc[(size_t)p * gstride + l] : 0u;
      float* d = sm + ((size_t)(y * Wp + x) * LP + l) * EPL;
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        const float f = l < valid_words ? WD::bits_to_f(WD::bits(w, e)) : 0.f;
        d[e] = ACC ? d[e] + f : f;
      }
    }
  }
}
// smem f32 [H][Wp][LP][EPL] -> global words
template <typename T, int LP>
__device__ __forceinline__ void tile_store_f32(const float* __restrict__ sm, uint32_t* __restrict__ gdst, size_t gstride, int H,
                                               int W, int Wp, int valid_words) {
  using WD = Word<T>;
  constexpr int EPL = WD::EPL;
  const float invW = 1.f / (float)W;
  const bool vec = (LP % 4 == 0) && valid_words == LP && (gstride % 4 == 0) && ((reinterpret_cast<uintptr_t>(gdst) & 15) == 0);
  const int items = vec ? H * W * (LP / 4) : H * W * LP;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    if (vec) {
      constexpr int VPP = LP / 4 > 0 ? LP / 4 : 1;
      const int p = it / VPP, q = it - p * VPP;
      int y, x;
      pix_yx(p, W, invW, &y, &x);
      const float* sp = sm + ((size_t)(y * Wp + x) * LP + q * 4) * EPL;
      uint32_t w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        w[k] = 0;
#pragma unroll
        for (int e = 0; e < EPL; ++e) w[k] = WD::put(w[k], e, WD::f_to_bits(sp[k * EPL + e]));
      }
      stg_stream16(gdst + (size_t)p * gstride + q * 4, make_uint4(w[0], w[1], w[2], w[3]));
    } else {
      const int p = it / LP, l = it - p * LP;
      if (l >= valid_words) continue;
      int y, x;
      pix_yx(p, W, invW, &y, &x);
      const float* sp = sm + ((size_t)(y * Wp + x) * LP + l) * EPL;
      uint32_t w = 0;
#pragma unroll
      for (int e = 0; e < EPL; ++e) w = WD::put(w, e, WD::f_to_bits(sp[e]));
      gdst[(size_t)p * gstride + l] = w;
    }
  }
}

struct PoolGeom {
  int B, C, H, W, Wp;  // Wp: padded pitch in pixels (odd -> consecutive rows land 16 banks apart for LP=16)
  int nseg;            // backward: segments per strip (threads = strips * nseg * lanes)
};

// ---------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------
template <typename T, int K, int LP, bool WITH_IDX>
__global__ void __launch_bounds__(512) sppf_pool_fwd_kernel(const T* __restrict__ y0, T* __restrict__ cat,
                                                            int32_t* __restrict__ idx, PoolGeom g) {
  using WD = Word<T>;
  constexpr int EPL = WD::EPL;
  constexpr int CC = LP * EPL;
  extern __shared__ __align__(16) uint32_t smem[];
  const int plane = g.H * g.Wp;
  uint32_t* cur = smem;               // [H][Wp][LP]
  uint32_t* tmp = smem + plane * LP;  // [H][Wp][LP]
  uint8_t* wrow = reinterpret_cast<uint8_t*>(smem + 2 * plane * LP);  // [H][Wp][LP] (WITH_IDX only)

  const int chunks = (g.C + CC - 1) / CC;
  const int b = blockIdx.x / chunks;
  const int c0 = (blockIdx.x % chunks) * CC;
  const int lane = threadIdx.x % LP;
  const int sid = threadIdx.x / LP;
  const int nstrips = blockDim.x / LP;
  const int c = c0 + lane * EPL;
  const bool cvalid = c < g.C;  // C % EPL == 0 is enforced on the host
  const size_t in_img = (size_t)b * g.H * g.W * g.C;
  const size_t out_img = (size_t)b * g.H * g.W * 4 * g.C;

  // stage the tile (word loads: LP*4 contiguous bytes per pixel) and emit concat slice 0
  const int valid_words = min(LP, (g.C - c0) / EPL);  // words of this chunk that exist (C bound)
  int special = tile_load_words<T, LP>(cur, reinterpret_cast<const uint32_t*>(y0 + in_img + c0), (size_t)g.C / EPL,
                                       reinterpret_cast<uint32_t*>(cat + out_img + c0), (size_t)4 * g.C / EPL, g.H, g.W, g.Wp,
                                       valid_words, WD::neg_inf());
  special = __syncthreads_or(special);

  if (!WITH_IDX && !special) {
    // fast path: packed hardware max, column pass stores straight into the concat slice
    uint32_t* gout = reinterpret_cast<uint32_t*>(cat + out_img + c);
    const size_t wstride = (size_t)4 * g.C * sizeof(T) / 4;   // words between vertically adjacent pixels' slices / W
    for (int st = 0; st < 3; ++st) {
      for (int y = sid; y < g.H; y += nstrips)
        pass1d_fast<T, K>(cur + (y * g.Wp) * LP + lane, LP, tmp + (y * g.Wp) * LP + lane, LP, g.W, nullptr, 0);
      __syncthreads();
      for (int x = sid; x < g.W; x += nstrips) {
        uint32_t* gd = cvalid ? gout + ((size_t)x * 4 * g.C + (size_t)(st + 1) * g.C) * sizeof(T) / 4 : nullptr;
        pass1d_fast<T, K>(tmp + x * LP + lane, g.Wp * LP, cur + x * LP + lane, g.Wp * LP, g.H, gd, wstride * g.W);
      }
      __syncthreads();
    }
    return;
  }

  for (int st = 0; st < 3; ++st) {
    // row pass: cur -> tmp
    for (int y = sid; y < g.H; y += nstrips)
      pass1d<T, K>(cur + (y * g.Wp) * LP + lane, LP, tmp + (y * g.Wp) * LP + lane, LP, g.W,
                   WITH_IDX ? wrow + (y * g.Wp) * LP + lane : nullptr, LP);
    __syncthreads();
    // column pass: tmp -> cur, and out to global
    for (int x = sid; x < g.W; x += nstrips) {
      if (!WITH_IDX) {
        pass1d<T, K>(tmp + x * LP + lane, g.Wp * LP, cur + x * LP + lane, g.Wp * LP, g.H, nullptr, 0);
      } else {
        // need the column winners too: reuse pass1d with a private winner strip in registers is awkward for
        // runtime H, so write winners into the (now free) low byte lanes of a second byte plane
        uint8_t* wcol = wrow + plane * LP;
        pass1d<T, K>(tmp + x * LP + lane, g.Wp * LP, cur + x * LP + lane, g.Wp * LP, g.H,
                     wcol + x * LP + lane, g.Wp * LP);
      }
    }
    __syncthreads();
    // emit slice st+1 (+ indices)
    for (int p = sid; p < g.H * g.W; p += nstrips) {
      const int y = p / g.W, x = p - y * g.W;
      if (!cvalid) continue;
      const int sp = (y * g.Wp + x) * LP + lane;
      *reinterpret_cast<uint32_t*>(cat + out_img + (size_t)p * 4 * g.C + (size_t)(st + 1) * g.C + c) = cur[sp];
      if (WITH_IDX) {
        const uint8_t* wcol = wrow + plane * LP;
        const uint32_t wc = wcol[sp];
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
          const int yy = y - K / 2 + (int)((wc >> (4 * e)) & 15u);
          const uint32_t wr = wrow[(yy * g.Wp + x) * LP + lane];
          const int xx = x - K / 2 + (int)((wr >> (4 * e)) & 15u);
          idx[(((size_t)st * g.B + b) * g.H * g.W + p) * g.C + c + e] = yy * g.W + xx;
        }
      }
    }
    if (WITH_IDX) __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------------
// scatter one strip of gradients through a 1-D max pass: dst[i + off(i) - R] += src[i]; strips are thread-private.
// Winners move monotonically along a strip, so contributions to one target are consecutive: accumulate them in a
// register and touch shared memory once per target (summation order = strip order: deterministic).
// A strip may be split over several threads by TARGET range [t0, t1): each scans the sources that can reach its range
// ([t0-R, t1+R)) and keeps those landing inside, so every target still has exactly one owner and one summation order.
template <int K, int EPL>
__device__ __forceinline__ void scatter1d(const float* __restrict__ src, int sstride, float* __restrict__ dst,
                                          int dstride, int len, const uint8_t* __restrict__ win, int wstride, int t0, int t1) {
  constexpr int R = K / 2;
  // Branch-free: every source adds straight into its (thread-private, pre-zeroed) target.  Sources are visited in strip
  // order, so each target still sums its contributions in the same fixed order; data-dependent run tracking in registers
  // made the lanes of a warp diverge on every element and cost 5x the instructions.
  const int ia = max(t0 - R, 0), ib = min(t1 + R, len);
#pragma unroll 2
  for (int i = ia; i < ib; ++i) {
    const uint32_t ws = win[i * wstride];
    float v[EPL];
    if (EPL == 2) {
      const float2 t2 = *reinterpret_cast<const float2*>(src + (size_t)i * sstride);
      v[0] = t2.x; v[EPL - 1] = t2.y;
    } else v[0] = src[(size_t)i * sstride];
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int t = i - R + (int)((ws >> (4 * e)) & 15u);
      if (t >= t0 && t < t1) dst[(size_t)t * dstride + e] += v[e];
    }
  }
}

template <typename T, int K, int LP>
__global__ void __launch_bounds__(512) sppf_pool_bwd_kernel(const T* __restrict__ gcat, const T* __restrict__ y0,
                                                            T* __restrict__ gy0, PoolGeom g) {
  using WD = Word<T>;
  constexpr int EPL = WD::EPL;
  constexpr int CC = LP * EPL;
  extern __shared__ __align__(16) uint32_t smem[];
  const int plane = g.H * g.Wp;
  // gradient ping-pong buffers (f32, EPL per lane) double as the value buffers of the recompute phase
  float* ga = reinterpret_cast<float*>(smem);                   // [plane][LP][EPL]
  float* gb = ga + (size_t)plane * LP * EPL;                    // [plane][LP][EPL]
  uint8_t* wrow = reinterpret_cast<uint8_t*>(gb + (size_t)plane * LP * EPL);  // [3][plane][LP]
  uint8_t* wcol = wrow + (size_t)3 * plane * LP;                // [3][plane][LP]
  uint32_t* cur = reinterpret_cast<uint32_t*>(ga);              // [plane][LP] words (fits: EPL*4 >= 4)
  uint32_t* tmp = reinterpret_cast<uint32_t*>(gb);

  const int chunks = (g.C + CC - 1) / CC;
  const int b = blockIdx.x / chunks;
  const int c0 = (blockIdx.x % chunks) * CC;
  const int lane = threadIdx.x % LP;
  const int sid = threadIdx.x / LP;
  const int nstrips = blockDim.x / LP;
  const int c = c0 + lane * EPL;
  const bool cvalid = c < g.C;
  const size_t in_img = (size_t)b * g.H * g.W * g.C;
  const size_t cat_img = (size_t)b * g.H * g.W * 4 * g.C;

  const int valid_words = min(LP, (g.C - c0) / EPL);
  int special = tile_load_words<T, LP>(cur, reinterpret_cast<const uint32_t*>(y0 + in_img + c0), (size_t)g.C / EPL, nullptr, 0,
                                       g.H, g.W, g.Wp, valid_words, WD::neg_inf());
  special = __syncthreads_or(special);
  if constexpr (EPL == 2) {
    if (!special) {   // packed-key path: move the tile into the sortable domain once (see pass1d_key)
      for (int i = threadIdx.x; i < plane * LP; i += blockDim.x) cur[i] = to_sortable2(cur[i]);
      __syncthreads();
    }
  }
  // Every strip (row or column of one lane word) is split into `nseg` segments walked by different threads: the smem
  // state (74 KB per CTA) bounds the strips in flight, so segmenting is what raises the number of resident warps.
  const int nseg = g.nseg;
  auto seg_lo = [&](int len, int sg) { return (len * sg) / nseg; };
  // recompute winners of the three stages (packed-key path unless the tile holds NaN / -0.0 or is f32)
  for (int st = 0; st < 3; ++st) {
    for (int u = sid; u < g.H * nseg; u += nstrips) {
      const int y = u / nseg, sg = u - y * nseg, i0 = seg_lo(g.W, sg), i1 = seg_lo(g.W, sg + 1);
      const uint32_t* sp = cur + (y * g.Wp) * LP + lane;
      uint32_t* dp = tmp + (y * g.Wp) * LP + lane;
      uint8_t* wp = wrow + ((size_t)st * plane + y * g.Wp) * LP + lane;
      if (special) pass1d<T, K>(sp, LP, dp, LP, g.W, wp, LP, i0, i1);
      else KeyPass<T, K>::run(sp, LP, dp, LP, g.W, wp, LP, i0, i1);
    }
    __syncthreads();
    for (int u = sid; u < g.W * nseg; u += nstrips) {
      const int x = u / nseg, sg = u - x * nseg, i0 = seg_lo(g.H, sg), i1 = seg_lo(g.H, sg + 1);
      const uint32_t* sp = tmp + x * LP + lane;
      uint32_t* dp = cur + x * LP + lane;
      uint8_t* wp = wcol + ((size_t)st * plane + x) * LP + lane;
      if (special) pass1d<T, K>(sp, g.Wp * LP, dp, g.Wp * LP, g.H, wp, g.Wp * LP, i0, i1);
      else KeyPass<T, K>::run(sp, g.Wp * LP, dp, g.Wp * LP, g.H, wp, g.Wp * LP, i0, i1);
    }
    __syncthreads();
  }
  // G3 = g3
  auto load_slice = [&](float* dstbuf, int slice, bool accumulate) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(gcat + cat_img + (size_t)slice * g.C + c0);
    if (accumulate) tile_load_f32<T, LP, true>(dstbuf, src, (size_t)4 * g.C / EPL, g.H, g.W, g.Wp, valid_words);
    else tile_load_f32<T, LP, false>(dstbuf, src, (size_t)4 * g.C / EPL, g.H, g.W, g.Wp, valid_words);
  };
  auto zero = [&](float* buf) {   // plane * LP * EPL floats: a multiple of 4 for every LP >= 4 (16-byte stores), scalar otherwise
    if constexpr ((LP * EPL) % 4 == 0) {
      uint4* b4 = reinterpret_cast<uint4*>(buf);
      for (int i = threadIdx.x; i < plane * LP * EPL / 4; i += blockDim.x) b4[i] = make_uint4(0u, 0u, 0u, 0u);
    } else {
      for (int i = threadIdx.x; i < plane * LP * EPL; i += blockDim.x) buf[i] = 0.f;
    }
  };
  load_slice(ga, 3, false);
  __syncthreads();
  for (int st = 2; st >= 0; --st) {
    // column-pass backward: ga (grad of stage output) -> gb (grad of row-pass output)
    zero(gb);
    __syncthreads();
    for (int u = sid; u < g.W * nseg; u += nstrips) {
      const int x = u / nseg, sg = u - x * nseg;
      scatter1d<K, EPL>(ga + ((size_t)x * LP + lane) * EPL, g.Wp * LP * EPL, gb + ((size_t)x * LP + lane) * EPL,
                        g.Wp * LP * EPL, g.H, wcol + ((size_t)st * plane + x) * LP + lane, g.Wp * LP, seg_lo(g.H, sg),
                        seg_lo(g.H, sg + 1));
    }
    __syncthreads();
    // row-pass backward: gb -> ga (grad of stage input).  ga starts from the concat slice gradient g_st instead of
    // zero + a separate accumulate pass: one sweep and one barrier fewer per stage (padding columns are never touched)
    load_slice(ga, st, false);
    __syncthreads();
    for (int u = sid; u < g.H * nseg; u += nstrips) {
      const int y = u / nseg, sg = u - y * nseg;
      scatter1d<K, EPL>(gb + ((size_t)(y * g.Wp) * LP + lane) * EPL, LP * EPL,
                        ga + ((size_t)(y * g.Wp) * LP + lane) * EPL, LP * EPL, g.W,
                        wrow + ((size_t)st * plane + y * g.Wp) * LP + lane, LP, seg_lo(g.W, sg), seg_lo(g.W, sg + 1));
    }
    __syncthreads();
  }
  tile_store_f32<T, LP>(ga, reinterpret_cast<uint32_t*>(gy0 + in_img + c0), (size_t)g.C / EPL, g.H, g.W, g.Wp, valid_words);
}

// ---- in-place variant (16-bit dtypes, two segments per strip) ---------------------------------------------------
// The routing pass is written as a GATHER: target t sums, in ascending source order, the sources i in [t-R, t+R] whose
// winner offset points at t (offset == t - i + R) -- the same values in the same order as scatter1d, so the results are
// bit-identical -- which lets it run IN PLACE: one f32 gradient buffer instead of two (47 KB instead of 74 KB of shared
// memory per CTA: 4 CTAs per SM = 592 slots, so the 512 work items of [64,128,20,20] are ONE wave instead of 1.15).
// Each strip is owned by two threads that both start at the middle and walk outwards (left one descending, right one
// ascending): everything a thread reads across the boundary is in its initial K-source window, loaded before the barrier
// that precedes the first write; afterwards it only reads sources further out than anything it or its partner has written.
// The window is a ring of K sources in registers; the walk is unrolled K times so ring slots are static.
template <int K> struct Ring {
  float2 v[K];
  uint32_t lo[K], hi[K];   // winner offsets of the two elements of the word (15 = no source)
};
template <int K>
__device__ __forceinline__ void ring_fetch(Ring<K>& rg, int slot, const float* __restrict__ buf, int stride,
                                           const uint8_t* __restrict__ win, int wstride, int p, int len) {
  if (p >= 0 && p < len) {
    rg.v[slot] = *reinterpret_cast<const float2*>(buf + (size_t)p * stride);
    const uint32_t w = win[p * wstride];
    rg.lo[slot] = w & 15u; rg.hi[slot] = w >> 4;
  } else {
    rg.v[slot] = make_float2(0.f, 0.f);
    rg.lo[slot] = 15u; rg.hi[slot] = 15u;
  }
}
// window of target k = 0: logical sources -R..R in slots 0..K-1 (position = start + dir * logical index)
template <int K>
__device__ __forceinline__ void ring_load(Ring<K>& rg, const float* buf, int stride, const uint8_t* win, int wstride, int start,
                                          int dir, int len) {
#pragma unroll
  for (int m = 0; m < K; ++m) ring_fetch<K>(rg, m, buf, stride, win, wstride, start + dir * (m - K / 2), len);
}
template <int K, int DIR>
__device__ __forceinline__ void ring_walk(Ring<K>& rg, float* buf, int stride, const uint8_t* win, int wstride, int start, int n,
                                          int len) {
  constexpr int R = K / 2;
  for (int k0 = 0; k0 < n; k0 += K) {
#pragma unroll
    for (int u = 0; u < K; ++u) {
      const int k = k0 + u;
      if (k < n) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int mm = 0; mm < K; ++mm) {
          const int m = DIR > 0 ? mm : K - 1 - mm;        // ascending source POSITION in both directions
          const int sl = (u + m) % K;                      // slot of window entry m at unrolled step u
          const uint32_t need = DIR > 0 ? K - 1 - m : m;   // offset that makes that source's winner this target
          if (rg.lo[sl] == need) a0 += rg.v[sl].x;
          if (rg.hi[sl] == need) a1 += rg.v[sl].y;
        }
        const int t = start + DIR * k;
        *reinterpret_cast<float2*>(buf + (size_t)t * stride) = make_float2(a0, a1);
        ring_fetch<K>(rg, u, buf, stride, win, wstride, start + DIR * (k + R + 1), len);   // replaces logical source k - R
      }
    }
  }
}

template <typename T, int K, int LP, int MAXT>   // MAXT 320: registers capped for 4 (K <= 5) / 3 CTAs per SM
__global__ void __launch_bounds__(MAXT, MAXT <= 320 ? (K <= 5 ? 4 : 3) : 1) sppf_pool_bwd_inplace_kernel(const T* __restrict__ gcat, const T* __restrict__ y0,
                                                                    T* __restrict__ gy0, PoolGeom g) {
  using WD = Word<T>;
  constexpr int EPL = WD::EPL;
  static_assert(EPL == 2, "in-place variant: 16-bit dtypes");
  constexpr int CC = LP * EPL;
  extern __shared__ __align__(16) uint32_t smem[];
  const int plane = g.H * g.Wp;
  float* ga = reinterpret_cast<float*>(smem);                                  // [plane][LP][2] f32 gradients
  uint8_t* wrow = reinterpret_cast<uint8_t*>(ga + (size_t)plane * LP * EPL);   // [3][plane][LP]
  uint8_t* wcol = wrow + (size_t)3 * plane * LP;                               // [3][plane][LP]
  uint32_t* cur = reinterpret_cast<uint32_t*>(ga);                             // recompute phase: two word planes inside ga
  uint32_t* tmp = cur + (size_t)plane * LP;

  const int chunks = (g.C + CC - 1) / CC;
  const int b = blockIdx.x / chunks;
  const int c0 = (blockIdx.x % chunks) * CC;
  const size_t in_img = (size_t)b * g.H * g.W * g.C;
  const size_t cat_img = (size_t)b * g.H * g.W * 4 * g.C;
  const int valid_words = min(LP, (g.C - c0) / EPL);
  int special = tile_load_words<T, LP>(cur, reinterpret_cast<const uint32_t*>(y0 + in_img + c0), (size_t)g.C / EPL, nullptr, 0,
                                       g.H, g.W, g.Wp, valid_words, WD::neg_inf());
  special = __syncthreads_or(special);
  if (!special) {
    for (int i = threadIdx.x; i < plane * LP; i += blockDim.x) cur[i] = to_sortable2(cur[i]);
    __syncthreads();
  }
  {  // winners of the three stages: strips split in two segments, interleaved over the threads
    const int lane = threadIdx.x % LP, sid = threadIdx.x / LP, nstrips = blockDim.x / LP;
    for (int st = 0; st < 3; ++st) {
      for (int u = sid; u < g.H * 2; u += nstrips) {
        const int y = u >> 1, sg = u & 1, i0 = sg ? g.W / 2 : 0, i1 = sg ? g.W : g.W / 2;
        const uint32_t* sp = cur + (y * g.Wp) * LP + lane;
        uint32_t* dp = tmp + (y * g.Wp) * LP + lane;
        uint8_t* wp = wrow + ((size_t)st * plane + y * g.Wp) * LP + lane;
        if (special) pass1d<T, K>(sp, LP, dp, LP, g.W, wp, LP, i0, i1);
        else pass1d_key<T, K>(sp, LP, dp, LP, g.W, wp, LP, i0, i1);
      }
      __syncthreads();
      for (int u = sid; u < g.W * 2; u += nstrips) {
        const int x = u >> 1, sg = u & 1, i0 = sg ? g.H / 2 : 0, i1 = sg ? g.H : g.H / 2;
        const uint32_t* sp = tmp + x * LP + lane;
        uint32_t* dp = cur + x * LP + lane;
        uint8_t* wp = wcol + ((size_t)st * plane + x) * LP + lane;
        if (special) pass1d<T, K>(sp, g.Wp * LP, dp, g.Wp * LP, g.H, wp, g.Wp * LP, i0, i1);
        else pass1d_key<T, K>(sp, g.Wp * LP, dp, g.Wp * LP, g.H, wp, g.Wp * LP, i0, i1);
      }
      __syncthreads();
    }
  }
  auto load_slice = [&](int slice, bool accumulate) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(gcat + cat_img + (size_t)slice * g.C + c0);
    if (accumulate) tile_load_f32<T, LP, true>(ga, src, (size_t)4 * g.C / EPL, g.H, g.W, g.Wp, valid_words);
    else tile_load_f32<T, LP, false>(ga, src, (size_t)4 * g.C / EPL, g.H, g.W, g.Wp, valid_words);
  };
  load_slice(3, false);
  __syncthreads();
  // routing: first half of the CTA's threads walks the left segments (descending), second half the right ones (warp-uniform)
  const int per = blockDim.x / 2;
  const int sg = threadIdx.x >= per ? 1 : 0;
  const int r_ = threadIdx.x - sg * per;
  const int lane = r_ % LP, sid = r_ / LP;
  Ring<K> rg;
  auto route = [&](float* buf, int stride, const uint8_t* win, int wstride, int len, bool act) {
    const int mid = len / 2;
    if (act) ring_load<K>(rg, buf, stride, win, wstride, sg ? mid : mid - 1, sg ? 1 : -1, len);
    __syncthreads();   // every thread holds its boundary window: the buffer may now be overwritten
    if (act) {
      if (sg) ring_walk<K, 1>(rg, buf, stride, win, wstride, mid, len - mid, len);
      else ring_walk<K, -1>(rg, buf, stride, win, wstride, mid - 1, mid, len);
    }
    __syncthreads();
  };
  for (int st = 2; st >= 0; --st) {
    // column-pass backward, then row-pass backward, both in place; then add the concat slice gradient g_st
    route(ga + ((size_t)sid * LP + lane) * EPL, g.Wp * LP * EPL, wcol + ((size_t)st * plane + sid) * LP + lane, g.Wp * LP, g.H,
          sid < g.W);
    route(ga + ((size_t)(sid * g.Wp) * LP + lane) * EPL, LP * EPL, wrow + ((size_t)st * plane + sid * g.Wp) * LP + lane, LP, g.W,
          sid < g.H);
    load_slice(st, true);
    __syncthreads();
  }
  tile_store_f32<T, LP>(ga, reinterpret_cast<uint32_t*>(gy0 + in_img + c0), (size_t)g.C / EPL, g.H, g.W, g.Wp, valid_words);
}

// ---------------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------------
template <typename T, int K, int LP>
int launch_fwd(const void* y0, void* cat, int32_t* idx, PoolGeom g, cudaStream_t st, bool* done) {
  constexpr int EPL = Word<T>::EPL;
  const size_t plane = (size_t)g.H * g.Wp;
  const size_t smem = plane * LP * 4 * 2 + (idx ? plane * LP * 2 : 0);
  if (smem > (size_t)max_smem_optin()) return B200_OK;  // try a smaller LP
  *done = true;
  const int chunks = (g.C + LP * EPL - 1) / (LP * EPL);
  int strips = g.H > g.W ? g.H : g.W;
  int threads = ((strips * LP + 31) / 32) * 32;
  if (threads > 512) threads = 512;
  if (threads < 64) threads = 64;
  dim3 grid(g.B * chunks);
  if (idx) {
    auto kern = sppf_pool_fwd_kernel<T, K, LP, true>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, threads, smem, st>>>((const T*)y0, (T*)cat, idx, g);
  } else {
    auto kern = sppf_pool_fwd_kernel<T, K, LP, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<grid, threads, smem, st>>>((const T*)y0, (T*)cat, idx, g);
  }
  return check_launch("sppf_pool_fwd");
}

template <typename T, int K, int LP>
int launch_bwd(const void* gcat, const void* y0, void* gy0, PoolGeom g, cudaStream_t st, bool* done) {
  constexpr int EPL = Word<T>::EPL;
  const size_t plane = (size_t)g.H * g.Wp;
  const size_t smem = plane * LP * EPL * 4 * 2 + plane * LP * 6;
  if (smem > (size_t)max_smem_optin()) return B200_OK;
  *done = true;
  const int chunks = (g.C + LP * EPL - 1) / (LP * EPL);
  int strips = g.H > g.W ? g.H : g.W;
  g.nseg = 1;
  // two segments per strip measured best (89 us vs 107 with one, 97 with three at 64x128x20x20): the kernel is bound by
  // instruction issue, and every extra segment re-scans K-1 sources
  while (g.nseg < 2 && strips * (g.nseg + 1) * LP <= 512 && (g.H < g.W ? g.H : g.W) / (g.nseg + 1) >= K) ++g.nseg;
  if constexpr (EPL == 2) {
    // 16-bit dtypes, two segments per strip, every strip covered in one sweep: in-place routing (one gradient buffer)
    const int per = ((strips * LP + 31) / 32) * 32;
    if (g.nseg == 2 && 2 * per <= 512 && g.H >= 2 && g.W >= 2) {
      const size_t smem_ip = plane * LP * EPL * 4 + plane * LP * 6;
      auto kip = 2 * per <= 320 ? sppf_pool_bwd_inplace_kernel<T, K, LP, 320> : sppf_pool_bwd_inplace_kernel<T, K, LP, 512>;
      cudaFuncSetAttribute(kip, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ip);
      kip<<<dim3(g.B * chunks), 2 * per, smem_ip, st>>>((const T*)gcat, (const T*)y0, (T*)gy0, g);
      return check_launch("sppf_pool_bwd");
    }
  }
  int threads = ((strips * g.nseg * LP + 31) / 32) * 32;
  if (threads > 512) threads = 512;
  if (threads < 64) threads = 64;
  auto kern = sppf_pool_bwd_kernel<T, K, LP>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<dim3(g.B * chunks), threads, smem, st>>>((const T*)gcat, (const T*)y0, (T*)gy0, g);
  return check_launch("sppf_pool_bwd");
}

template <typename T, int K>
int fwd_k(const void* y0, void* cat, int32_t* idx, PoolGeom g, cudaStream_t st) {
  bool done = false;
  int rc = launch_fwd<T, K, 16>(y0, cat, idx, g, st, &done);
  if (!done) rc = launch_fwd<T, K, 8>(y0, cat, idx, g, st, &done);
  if (!done) rc = launch_fwd<T, K, 4>(y0, cat, idx, g, st, &done);
  if (!done) rc = launch_fwd<T, K, 2>(y0, cat, idx, g, st, &done);
  if (!done) rc = launch_fwd<T, K, 1>(y0, cat, idx, g, st, &done);
  B200_REQUIRE(done, B200_ERR_UNSUPPORTED, "sppf_pool_fwd: %dx%d plane does not fit in shared memory", g.H, g.W);
  return rc;
}
template <typename T, int K>
int bwd_k(const void* gcat, const void* y0, void* gy0, PoolGeom g, cudaStream_t st) {
  bool done = false;
  int rc = launch_bwd<T, K, 8>(gcat, y0, gy0, g, st, &done);
  if (!done) rc = launch_bwd<T, K, 4>(gcat, y0, gy0, g, st, &done);
  if (!done) rc = launch_bwd<T, K, 2>(gcat, y0, gy0, g, st, &done);
  if (!done) rc = launch_bwd<T, K, 1>(gcat, y0, gy0, g, st, &done);
  B200_REQUIRE(done, B200_ERR_UNSUPPORTED, "sppf_pool_bwd: %dx%d plane does not fit in shared memory", g.H, g.W);
  return rc;
}

int check_args(const void* a, const void* b, int B, int C, int H, int W, int k, int dtype) {
  B200_REQUIRE(a && b, B200_ERR_SHAPE, "sppf_pool: null tensor pointer");
  B200_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, B200_ERR_SHAPE, "sppf_pool: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
  B200_REQUIRE(k >= 3 && k <= 13 && (k & 1), B200_ERR_SHAPE, "sppf_pool: k must be odd in [3,13], got %d", k);
  B200_REQUIRE(H < 4096 && W < 4096, B200_ERR_SHAPE, "sppf_pool: plane too large");
  if (dtype != B200_F32) B200_REQUIRE(C % 2 == 0, B200_ERR_ALIGN, "sppf_pool: C must be even for 16-bit dtypes (C=%d)", C);
  B200_REQUIRE(((uintptr_t)a & 3) == 0 && ((uintptr_t)b & 3) == 0, B200_ERR_ALIGN, "sppf_pool: pointers must be 4-byte aligned");
  return B200_OK;
}

#define B200_DISPATCH_K(k, ...)                                           \
  [&]() -> int {                                                          \
    switch (k) {                                                          \
      case 3: { constexpr int K = 3; return __VA_ARGS__(); }              \
      case 5: { constexpr int K = 5; return __VA_ARGS__(); }              \
      case 7: { constexpr int K = 7; return __VA_ARGS__(); }              \
      case 9: { constexpr int K = 9; return __VA_ARGS__(); }              \
      case 11: { constexpr int K = 11; return __VA_ARGS__(); }            \
      default: { constexpr int K = 13; return __VA_ARGS__(); }            \
    }                                                                     \
  }()

}  // namespace
}  // namespace b200

extern "C" B200_API int b200_sppf_pool_fwd(const void* y0, void* cat, int32_t* idx, int32_t B, int32_t C, int32_t H,
                                  int32_t W, int32_t k, int32_t dtype, void* stream) {
  using namespace b200;
  if (int rc = check_args(y0, cat, B, C, H, W, k, dtype)) return rc;
  PoolGeom g{B, C, H, W, (W & 1) ? W : W + 1};
  cudaStream_t st = (cudaStream_t)stream;
  if (!idx) {   // values only on the model's own plane: strips in registers (sppf_strip.cu)
    const int rc = sppf::strip_fwd(y0, cat, B, C, H, W, k, dtype, st);
    if (rc != -1) return rc;
  }
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    return B200_DISPATCH_K(k, [&]() -> int { return fwd_k<T, K>(y0, cat, idx, g, st); });
  });
}

extern "C" B200_API int b200_sppf_pool_bwd(const void* gcat, const void* y0, void* gy0, int32_t B, int32_t C, int32_t H,
                                  int32_t W, int32_t k, int32_t dtype, void* stream) {
  using namespace b200;
  if (int rc = check_args(gcat, y0, B, C, H, W, k, dtype)) return rc;
  B200_REQUIRE(gy0, B200_ERR_SHAPE, "sppf_pool_bwd: null output");
  PoolGeom g{B, C, H, W, (W & 1) ? W : W + 1};
  cudaStream_t st = (cudaStream_t)stream;
  {
    const int rc = sppf::strip_bwd(gcat, y0, gy0, B, C, H, W, k, dtype, st);
    if (rc != -1) return rc;
  }
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    return B200_DISPATCH_K(k, [&]() -> int { return bwd_k<T, K>(gcat, y0, gy0, g, st); });
  });
}
