// SwinBlock: the non-GEMM stages (window partition / reverse folded into the loads and stores, LayerNorm,
// residuals, GELU) forward and backward.  Replaces the data-movement and normalisation ops of
// swin_block.py:37-58 (F.pad, rearrange, window_partition, norm1, residual adds, norm2, GELU, window_reverse,
// crop) and their autograd backward (SURVEY.md App. A.3).
//
// Token order: t = ((b*nWh + wh)*nWw + ww)*L + r*ws + c  <->  pixel (y, x) = (wh*ws + r, ww*ws + c); tokens with
// y >= H or x >= W are the zero padding of swin_block.py:41-43 (they become norm1.bias after LN1 and still act
// as keys/values -- SURVEY D3).  Activations are NHWC so a token's C channels are contiguous on both sides:
// partition / reverse is pure address arithmetic in the kernels below, never a separate copy.
#include "common.cuh"

namespace b200 {
namespace {

// division by a run-time constant as multiply-high + shifts (Granlund-Montgomery / libdivide "branchfree" form),
// exact for every 32-bit numerator: the token -> pixel map needs four divisions per token and the plain 64-bit
// '/' and '%' cost more instructions than the LayerNorm itself.
struct FastDiv {
  uint32_t d, m, s1, s2;
  __host__ void init(uint32_t div) {
    d = div;
    uint32_t l = 0;
    while ((1ull << l) < div) ++l;
    m = (uint32_t)((((1ull << 32) * ((1ull << l) - div)) / div) + 1);
    s1 = l < 1 ? l : 1;
    s2 = l > 0 ? l - 1 : 0;
  }
  __device__ __forceinline__ uint32_t div(uint32_t n) const {
    const uint32_t t = __umulhi(m, n);
    return (t + ((n - t) >> s1)) >> s2;
  }
};

struct WinGeom {
  int B, C, H, W, ws, nWh, nWw, L, shift;
  long long T;  // padded token count (< 2^31, checked on the host)
  FastDiv dL, dWw, dWh, dws;
};

__device__ __forceinline__ long long token_pixel(const WinGeom& g, long long t64, bool* real) {
  const uint32_t t = (uint32_t)t64;
  const uint32_t win = g.dL.div(t), l = t - win * g.L;
  const uint32_t q = g.dWw.div(win), ww = win - q * g.nWw;
  const uint32_t b = g.dWh.div(q), wh = q - b * g.nWh;
  const uint32_t r = g.dws.div(l), c = l - r * g.ws;
  // window coordinates index the padded map AFTER the cyclic shift by (-shift, -shift): source pixel = (+shift) mod size
  int y = (int)(wh * g.ws + r) + g.shift, x = (int)(ww * g.ws + c) + g.shift;
  if (y >= g.nWh * g.ws) y -= g.nWh * g.ws;
  if (x >= g.nWw * g.ws) x -= g.nWw * g.ws;
  *real = (y < g.H) && (x < g.W);
  return ((long long)b * g.H + y) * g.W + x;
}

template <typename T> __device__ __forceinline__ float ldf(const T* p) { return DT<T>::to_f(*p); }

// ---- warp-per-token LayerNorm statistics over a register-resident row ------------------------------------------
// Each lane holds elements c = lane + 32*i (i < NPL).  Two-pass (mean, then centred variance) for fp32 parity.
template <int MAXPL>
__device__ __forceinline__ void row_stats(const float (&v)[MAXPL], int npl, int C, int lane, float* mean, float* rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXPL; ++i)
    if (i < npl && lane + 32 * i < C) s += v[i];
  s = warp_sum(s);
  const float mu = s / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXPL; ++i)
    if (i < npl && lane + 32 * i < C) { const float d = v[i] - mu; q += d * d; }
  q = warp_sum(q);
  *mean = mu;
  *rstd = rsqrtf(q / (float)C + 1e-5f);
}

constexpr int kMaxPL = 32;  // C <= 1024 (generic kernels)

// ---- sub-warp-per-token vector kernels ---------------------------------------------------------------------
// A token's C channels are spread over LPT lanes (a power of two <= 32), each lane holding NV 16-byte vectors at
// channel offsets (l + LPT*v)*VE, l = lane % LPT, VE = 16/sizeof(T).  A warp therefore normalises 32/LPT tokens at
// once: the per-token costs that dominated the warp-per-token version (token->pixel index arithmetic, two chains of
// shuffle reductions) are paid once per 32/LPT tokens and the shuffle trees are log2(LPT) deep.
template <typename T> struct VecOf { static constexpr int VE = 16 / (int)sizeof(T); };
template <typename T> struct alignas(16) Pack16 { T e[16 / sizeof(T)]; };

template <typename T, int LPT, int NV>
__device__ __forceinline__ void load_row(const T* __restrict__ row, int l, float (&v)[NV * VecOf<T>::VE]) {
  constexpr int VE = VecOf<T>::VE;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const Pack16<T> p = *reinterpret_cast<const Pack16<T>*>(row + (l + LPT * i) * VE);
#pragma unroll
    for (int e = 0; e < VE; ++e) v[i * VE + e] = DT<T>::to_f(p.e[e]);
  }
}
template <typename T, int LPT, int NV>
__device__ __forceinline__ void store_row(T* __restrict__ row, int l, const float (&v)[NV * VecOf<T>::VE]) {
  constexpr int VE = VecOf<T>::VE;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    Pack16<T> p;
#pragma unroll
    for (int e = 0; e < VE; ++e) p.e[e] = DT<T>::from_f(v[i * VE + e]);
    *reinterpret_cast<Pack16<T>*>(row + (l + LPT * i) * VE) = p;
  }
}
template <int VE, int LPT, int NV>
__device__ __forceinline__ void load_vecf(const float* __restrict__ p, int l, float (&v)[NV * VE]) {
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int e = 0; e < VE; ++e) v[i * VE + e] = p[(l + LPT * i) * VE + e];
}
template <int LPT> __device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPT / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int N, int LPT>
__device__ __forceinline__ void stats_full(const float (&v)[N], int C, float* mean, float* rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) s += v[i];
  const float mu = group_sum<LPT>(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) { const float d = v[i] - mu; q += d * d; }
  *mean = mu;
  *rstd = rsqrtf(group_sum<LPT>(q) / (float)C + 1e-5f);
}

// n1[t,:] = LN1(token t of x) (padded tokens: LN(0) = beta).  Saves mean / rstd per token for the backward.
template <typename T, int LPT, int NV>
__global__ void __launch_bounds__(256) swin_ln1_partition_vec_kernel(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta, T* __restrict__ n1,
                                                                    float* __restrict__ mean, float* __restrict__ rstd,
                                                                    WinGeom g) {
  constexpr int VE = VecOf<T>::VE, N = NV * VE, TPW = 32 / LPT;
  const int lane = threadIdx.x & 31, l = lane % LPT, grp = lane / LPT;
  float gm[N], bt[N];
  load_vecf<VE, LPT, NV>(gamma, l, gm);
  load_vecf<VE, LPT, NV>(beta, l, bt);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * TPW; t0 < g.T; t0 += nwarps * TPW) {
    const long long t = t0 + grp;
    const bool live = t < g.T;
    bool real = false;
    long long pix = 0;
    if (live) pix = token_pixel(g, t, &real);
    float v[N];
    if (real) load_row<T, LPT, NV>(x + pix * g.C, l, v);
    else {
#pragma unroll
      for (int i = 0; i < N; ++i) v[i] = 0.f;
    }
    float mu, rs;
    stats_full<N, LPT>(v, g.C, &mu, &rs);
    if (live) {
#pragma unroll
      for (int i = 0; i < N; ++i) v[i] = (v[i] - mu) * rs * gm[i] + bt[i];
      store_row<T, LPT, NV>(n1 + t * g.C, l, v);
      if (l == 0) { mean[t] = mu; rstd[t] = rs; }
    }
  }
}

template <typename T, int LPT, int NV>
__global__ void __launch_bounds__(256) swin_res_ln2_vec_kernel(const T* __restrict__ n1, const T* __restrict__ a,
                                                              const float* __restrict__ gamma, const float* __restrict__ beta,
                                                              T* __restrict__ y1, T* __restrict__ u, float* __restrict__ mean,
                                                              float* __restrict__ rstd, long long Ttok, int C) {
  constexpr int VE = VecOf<T>::VE, N = NV * VE, TPW = 32 / LPT;
  const int lane = threadIdx.x & 31, l = lane % LPT, grp = lane / LPT;
  float gm[N], bt[N];
  load_vecf<VE, LPT, NV>(gamma, l, gm);
  load_vecf<VE, LPT, NV>(beta, l, bt);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * TPW; t0 < Ttok; t0 += nwarps * TPW) {
    const bool live = t0 + grp < Ttok;
    const long long t = live ? t0 + grp : Ttok - 1;
    float v[N];
    load_row<T, LPT, NV>(n1 + t * C, l, v);
    if (a) {  // a == nullptr: `n1` already holds y1 (residual fused into the out_proj GEMM epilogue)
      float w[N];
      load_row<T, LPT, NV>(a + t * C, l, w);
#pragma unroll
      for (int i = 0; i < N; ++i) v[i] = DT<T>::to_f(DT<T>::from_f(v[i] + w[i]));  // LN2 sees exactly the stored y1
      if (live) store_row<T, LPT, NV>(y1 + t * C, l, v);
    }
    float mu, rs;
    stats_full<N, LPT>(v, C, &mu, &rs);
    if (live) {
#pragma unroll
      for (int i = 0; i < N; ++i) v[i] = (v[i] - mu) * rs * gm[i] + bt[i];
      store_row<T, LPT, NV>(u + t * C, l, v);
      if (l == 0) { mean[t] = mu; rstd[t] = rs; }
    }
  }
}

// out[b,y,x,:] = y1[t,:] + m[t,:] for real tokens (MODE 0)   /   tok[t,:] = src[b,y,x,:] or 0 (MODE 1), vectorised
template <typename T, int LPT, int NV, int MODE>
__global__ void __launch_bounds__(256) swin_move_vec_kernel(const T* __restrict__ a, const T* __restrict__ b2, T* __restrict__ out,
                                                           WinGeom g) {
  constexpr int VE = VecOf<T>::VE, N = NV * VE, TPW = 32 / LPT;
  const int lane = threadIdx.x & 31, l = lane % LPT, grp = lane / LPT;
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t0 = ((long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * TPW; t0 < g.T; t0 += nwarps * TPW) {
    const long long t = t0 + grp;
    if (t >= g.T) continue;
    bool real;
    const long long pix = token_pixel(g, t, &real);
    float v[N];
    if (MODE == 0) {
      if (!real) continue;
      float w[N];
      load_row<T, LPT, NV>(a + t * g.C, l, v);
      if (b2) {   // null: window_reverse + crop only
        load_row<T, LPT, NV>(b2 + t * g.C, l, w);
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] += w[i];
      }
      store_row<T, LPT, NV>(out + pix * g.C, l, v);
    } else {
      if (real) {
        load_row<T, LPT, NV>(a + pix * g.C, l, v);
        if (b2) {   // second addend in the same pixel layout (the residual gradient of the fused MLP backward)
          float w[N];
          load_row<T, LPT, NV>(b2 + pix * g.C, l, w);
#pragma unroll
          for (int i = 0; i < N; ++i) v[i] += w[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < N; ++i) v[i] = 0.f;
      }
      store_row<T, LPT, NV>(out + t * g.C, l, v);
    }
  }
}

// LayerNorm backward, vectorised (see swin_ln_bwd_kernel below for the maths / modes)
template <typename T, int LPT, int NV, int MODE>
__global__ void __launch_bounds__(256) swin_ln_bwd_vec_kernel(const T* __restrict__ gout, const T* __restrict__ xin,
                                                             const T* __restrict__ gres, const float* __restrict__ gamma,
                                                             const float* __restrict__ mean, const float* __restrict__ rstd,
                                                             T* __restrict__ gin, float* __restrict__ part, WinGeom g) {
  constexpr int VE = VecOf<T>::VE, N = NV * VE, TPW = 32 / LPT;
  extern __shared__ float sm[];  // [warps][2][C]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int l = lane % LPT, grp = lane / LPT;
  const int C = g.C;
  float gm[N], accg[N], accb[N];
  load_vecf<VE, LPT, NV>(gamma, l, gm);
#pragma unroll
  for (int i = 0; i < N; ++i) { accg[i] = 0.f; accb[i] = 0.f; }
  const long long nwarps = (long long)gridDim.x * nwarp;
  for (long long t0 = ((long long)blockIdx.x * nwarp + warp) * TPW; t0 < g.T; t0 += nwarps * TPW) {
    const long long t = t0 + grp;
    const bool live = t < g.T;
    bool real = true;
    long long src = live ? t : 0;
    if (live && MODE == 1) src = token_pixel(g, t, &real);
    float go[N], xh[N];
    float mu = 0.f, rs = 0.f;
    if (live) {
      mu = mean[t]; rs = rstd[t];
      load_row<T, LPT, NV>(gout + t * C, l, go);
      if (MODE == 1 && !real) {
#pragma unroll
        for (int i = 0; i < N; ++i) xh[i] = 0.f;
      } else load_row<T, LPT, NV>(xin + src * C, l, xh);
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) { go[i] = 0.f; xh[i] = 0.f; }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      xh[i] = (xh[i] - mu) * rs;
      accg[i] += go[i] * xh[i];
      accb[i] += go[i];
      go[i] *= gm[i];
      s1 += go[i];
      s2 += go[i] * xh[i];
    }
    s1 = group_sum<LPT>(s1) / (float)C;
    s2 = group_sum<LPT>(s2) / (float)C;
    if (live && (MODE == 0 || real)) {
      float r[N];
      if (MODE == 0) load_row<T, LPT, NV>(gres + t * C, l, r);
#pragma unroll
      for (int i = 0; i < N; ++i) r[i] = (go[i] - s1 - xh[i] * s2) * rs + (MODE == 0 ? r[i] : 0.f);
      store_row<T, LPT, NV>(gin + src * C, l, r);
    }
  }
  // fold the token groups of the warp (same channels live in lanes l, l+LPT, ...), then the warps of the CTA
#pragma unroll
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int o = LPT; o < 32; o <<= 1) {
      accg[i] += __shfl_xor_sync(0xffffffffu, accg[i], o);
      accb[i] += __shfl_xor_sync(0xffffffffu, accb[i], o);
    }
  }
  if (grp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
      for (int e = 0; e < VE; ++e) {
        const int c = (l + LPT * i) * VE + e;
        sm[(warp * 2 + 0) * C + c] = accg[i * VE + e];
        sm[(warp * 2 + 1) * C + c] = accb[i * VE + e];
      }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < nwarp; ++w) s += sm[w * 2 * C + i];
    part[(size_t)blockIdx.x * 2 * C + i] = s;
  }
}

// pick (LPT, NV) with C == LPT*NV*VE, preferring two vectors per lane; false when C has no instantiation
template <typename T>
inline bool pick_vec(int C, int* lpt, int* nv) {
  constexpr int VE = VecOf<T>::VE;
  for (int want : {2, 3, 1})
    for (int L : {8, 16, 32})
      if (C == L * want * VE) { *lpt = L; *nv = want; return true; }
  return false;
}
#define B200_VEC_CASE(L_, N_, ...) if (vec == L_ && iters == N_) { constexpr int VEC = L_; constexpr int ITERS = N_; __VA_ARGS__; }
#define B200_DISPATCH_VEC(...)                                                                              \
  do {                                                                                                      \
    B200_VEC_CASE(8, 1, __VA_ARGS__) B200_VEC_CASE(8, 2, __VA_ARGS__) B200_VEC_CASE(8, 3, __VA_ARGS__)       \
    B200_VEC_CASE(16, 1, __VA_ARGS__) B200_VEC_CASE(16, 2, __VA_ARGS__) B200_VEC_CASE(16, 3, __VA_ARGS__)    \
    B200_VEC_CASE(32, 1, __VA_ARGS__) B200_VEC_CASE(32, 2, __VA_ARGS__) B200_VEC_CASE(32, 3, __VA_ARGS__)    \
  } while (0)

// ---- generic (any C <= 1024) kernels ------------------------------------------------------------------------
// n1[t,:] = LN1(token t of x) (padded tokens: LN(0) = beta).  Saves mean / rstd per token for the backward.
template <typename T>
__global__ void __launch_bounds__(256) swin_ln1_partition_kernel(const T* __restrict__ x, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, T* __restrict__ n1,
                                                                float* __restrict__ mean, float* __restrict__ rstd,
                                                                WinGeom g) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= g.T) return;
  bool real;
  const long long pix = token_pixel(g, t, &real);
  const int npl = (g.C + 31) / 32;
  float v[kMaxPL];
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) {
    const int c = lane + 32 * i;
    v[i] = (i < npl && c < g.C && real) ? ldf(x + pix * g.C + c) : 0.f;
  }
  float mu, rs;
  row_stats<kMaxPL>(v, npl, g.C, lane, &mu, &rs);
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) {
    const int c = lane + 32 * i;
    if (i < npl && c < g.C) n1[t * g.C + c] = DT<T>::from_f((v[i] - mu) * rs * gamma[c] + beta[c]);
  }
  if (lane == 0) { mean[t] = mu; rstd[t] = rs; }
}

// y1 = n1 + a (a = out_proj output incl. bias);  u = LN2(y1).  Saves mean / rstd.
template <typename T>
__global__ void __launch_bounds__(256) swin_res_ln2_kernel(const T* __restrict__ n1, const T* __restrict__ a,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          T* __restrict__ y1, T* __restrict__ u, float* __restrict__ mean,
                                                          float* __restrict__ rstd, long long Ttok, int C) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= Ttok) return;
  const int npl = (C + 31) / 32;
  float v[kMaxPL];
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) {
    const int c = lane + 32 * i;
    if (i < npl && c < C) {
      // the residual sum is rounded to the activation dtype first: LN2 must see exactly the stored y1
      if (a) {
        const T s = DT<T>::from_f(ldf(n1 + t * C + c) + ldf(a + t * C + c));
        y1[t * C + c] = s;
        v[i] = DT<T>::to_f(s);
      } else v[i] = ldf(n1 + t * C + c);
    } else v[i] = 0.f;
  }
  float mu, rs;
  row_stats<kMaxPL>(v, npl, C, lane, &mu, &rs);
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) {
    const int c = lane + 32 * i;
    if (i < npl && c < C) u[t * C + c] = DT<T>::from_f((v[i] - mu) * rs * gamma[c] + beta[c]);
  }
  if (lane == 0) { mean[t] = mu; rstd[t] = rs; }
}

__device__ __forceinline__ float gelu_erf(float a) { return 0.5f * a * (1.f + erff(a * 0.70710678118654752440f)); }
__device__ __forceinline__ float gelu_erf_grad(float a) {
  const float cdf = 0.5f * (1.f + erff(a * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * a * a);
  return cdf + a * pdf;
}

// h = gelu(a)   /   ga = gh * gelu'(a)        (elementwise, 16-byte vectorised when aligned)
template <typename T, bool BWD>
__global__ void __launch_bounds__(256) swin_gelu_kernel(const T* __restrict__ a, const T* __restrict__ gh, T* __restrict__ out,
                                                       long long n) {
  constexpr int V = 16 / sizeof(T);
  const long long nv = n / V;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    uint4 av = *reinterpret_cast<const uint4*>(a + i * V);
    uint4 gv = BWD ? *reinterpret_cast<const uint4*>(gh + i * V) : make_uint4(0, 0, 0, 0);
    uint4 ov;
    const T* ap = reinterpret_cast<const T*>(&av);
    const T* gp = reinterpret_cast<const T*>(&gv);
    T* op = reinterpret_cast<T*>(&ov);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      const float f = DT<T>::to_f(ap[e]);
      op[e] = DT<T>::from_f(BWD ? DT<T>::to_f(gp[e]) * gelu_erf_grad(f) : gelu_erf(f));
    }
    *reinterpret_cast<uint4*>(out + i * V) = ov;
  }
  if (blockIdx.x == 0)
    for (long long i = nv * V + threadIdx.x; i < n; i += blockDim.x) {
      const float f = DT<T>::to_f(a[i]);
      out[i] = DT<T>::from_f(BWD ? DT<T>::to_f(gh[i]) * gelu_erf_grad(f) : gelu_erf(f));
    }
}

// out[b,y,x,:] = y1[t,:] + m[t,:] for real tokens (window_reverse + crop folded into the store address)
template <typename T>
__global__ void __launch_bounds__(256) swin_res_reverse_kernel(const T* __restrict__ y1, const T* __restrict__ m,
                                                              T* __restrict__ out, WinGeom g) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= g.T) return;
  bool real;
  const long long pix = token_pixel(g, t, &real);
  if (!real) return;
  for (int c = lane; c < g.C; c += 32) out[pix * g.C + c] = DT<T>::from_f(ldf(y1 + t * g.C + c) + (m ? ldf(m + t * g.C + c) : 0.f));
}

// gy2[t,:] = g[b,y,x,:] for real tokens, 0 for padded ones (they are cropped, swin_block.py:58)
template <typename T>
__global__ void __launch_bounds__(256) swin_partition_kernel(const T* __restrict__ gsrc, const T* __restrict__ gadd, T* __restrict__ gtok, WinGeom g) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= g.T) return;
  bool real;
  const long long pix = token_pixel(g, t, &real);
  for (int c = lane; c < g.C; c += 32) {
    float v = 0.f;
    if (real) v = ldf(gsrc + pix * g.C + c) + (gadd ? ldf(gadd + pix * g.C + c) : 0.f);
    gtok[t * g.C + c] = DT<T>::from_f(v);
  }
}

// LayerNorm backward for a block of tokens + column partials of gamma / beta gradients.
//   gin[t,:] = (ghat - mean(ghat) - xhat*mean(ghat*xhat)) * rstd (+ gres[t,:]),  ghat = gout*gamma
// MODE 0 (LN2): xin = y1 tokens, output token-major, adds the residual gradient gres (= g_y2).
// MODE 1 (LN1): xin = x in NHWC (gathered through the window map; padded tokens are all-zero rows), output is
//               scattered back to NHWC gx for real tokens only; gres = nullptr.
// gamma/beta partials: one row of [2][C] per CTA in `part` (folded by a second tiny kernel: deterministic).
template <typename T, int MODE>
__global__ void __launch_bounds__(256) swin_ln_bwd_kernel(const T* __restrict__ gout, const T* __restrict__ xin,
                                                         const T* __restrict__ gres, const float* __restrict__ gamma,
                                                         const float* __restrict__ mean, const float* __restrict__ rstd,
                                                         T* __restrict__ gin, float* __restrict__ part, WinGeom g,
                                                         int tokens_per_cta) {
  extern __shared__ float sm[];  // [warps][2][C]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int C = g.C, npl = (C + 31) / 32;
  float accg[kMaxPL], accb[kMaxPL];
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) { accg[i] = 0.f; accb[i] = 0.f; }
  const long long t0 = (long long)blockIdx.x * tokens_per_cta;
  for (int k = warp; k < tokens_per_cta; k += nwarp) {
    const long long t = t0 + k;
    if (t >= g.T) break;
    bool real = true;
    long long src = t;
    if (MODE == 1) src = token_pixel(g, t, &real);
    const float mu = mean[t], rs = rstd[t];
    float go[kMaxPL], xh[kMaxPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxPL; ++i) {
      const int c = lane + 32 * i;
      if (i < npl && c < C) {
        const float gv = ldf(gout + t * C + c);
        const float xv = (MODE == 1 && !real) ? 0.f : ldf(xin + src * C + c);
        xh[i] = (xv - mu) * rs;
        go[i] = gv * gamma[c];
        s1 += go[i];
        s2 += go[i] * xh[i];
        accg[i] += gv * xh[i];
        accb[i] += gv;
      } else { go[i] = 0.f; xh[i] = 0.f; }
    }
    s1 = warp_sum(s1) / (float)C;
    s2 = warp_sum(s2) / (float)C;
    if (MODE == 0 || real) {
#pragma unroll
      for (int i = 0; i < kMaxPL; ++i) {
        const int c = lane + 32 * i;
        if (i < npl && c < C) {
          float r = (go[i] - s1 - xh[i] * s2) * rs;
          if (MODE == 0) r += ldf(gres + t * C + c);
          gin[src * C + c] = DT<T>::from_f(r);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kMaxPL; ++i) {
    const int c = lane + 32 * i;
    if (i < npl && c < C) { sm[(warp * 2 + 0) * C + c] = accg[i]; sm[(warp * 2 + 1) * C + c] = accb[i]; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    float s = 0.f;
    for (int w = 0; w < nwarp; ++w) s += sm[w * 2 * C + i];
    part[(size_t)blockIdx.x * 2 * C + i] = s;
  }
}

// [rows][2][C] partials -> ggamma[C], gbeta[C]   (fixed order)
__global__ void __launch_bounds__(1024) fold_ln_kernel(const float* __restrict__ part, float* __restrict__ gg, float* __restrict__ gb,
                                                       int rows, int C) {
  // 32 columns per block: lane = column, the block's 32 warps split the rows, fixed-order smem fold
  __shared__ float sm[32][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (i < 2 * C)
    for (int r = warp; r < rows; r += 32) s += part[(size_t)r * 2 * C + i];
  sm[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && i < 2 * C) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 32; ++w) t += sm[w][lane];
    if (i < C) gg[i] = t; else gb[i - C] = t;
  }
}

// out[i] = sum_r part[r][i]   (fixed order)
__global__ void fold_rows_kernel(const float* __restrict__ part, float* __restrict__ out, int rows, int n) {
  __shared__ float sm[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (i < n)
    for (int r = warp; r < rows; r += 8) s += part[(size_t)r * n + i];
  sm[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && i < n) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += sm[w][lane];
    out[i] = t;
  }
}

template <typename T, int VEC> struct alignas(sizeof(T) * VEC) PackT { T e[VEC]; };

// column sums of a [rows, n] activation matrix -> f32 [n] (bias gradients); two-stage, deterministic
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T* __restrict__ a, float* __restrict__ part, long long rows,
                                                            int n, int rows_per_cta) {
  // blockIdx.x: 128-column strip (lane owns 4 columns), blockIdx.y: row slab; the 8 warps interleave the slab's rows
  __shared__ float sm[8][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + lane * 4;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  if (c + 3 < n) {
    for (long long r = r0 + warp; r < r1; r += 8) {
      const PackT<T, 4> p = *reinterpret_cast<const PackT<T, 4>*>(a + r * n + c);
#pragma unroll
      for (int e = 0; e < 4; ++e) s[e] += DT<T>::to_f(p.e[e]);
    }
  } else {
    for (long long r = r0 + warp; r < r1; r += 8)
      for (int e = 0; e < 4; ++e)
        if (c + e < n) s[e] += ldf(a + r * n + c + e);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) sm[warp][lane * 4 + e] = s[e];
  __syncthreads();
  if (threadIdx.x < 128 && blockIdx.x * 128 + threadIdx.x < n) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += sm[w][threadIdx.x];
    part[(size_t)blockIdx.y * n + blockIdx.x * 128 + threadIdx.x] = t;
  }
}

int make_geom(WinGeom* g, int B, int C, int H, int W, int ws, int shift = 0) {
  B200_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && ws > 0, B200_ERR_SHAPE, "swin: bad shape B=%d C=%d H=%d W=%d ws=%d", B, C, H, W, ws);
  B200_REQUIRE(shift >= 0 && shift < ws, B200_ERR_SHAPE, "swin: shift %d must lie in [0, window size %d)", shift, ws);
  g->shift = shift;
  B200_REQUIRE(C <= 32 * kMaxPL, B200_ERR_UNSUPPORTED, "swin: C=%d > %d unsupported", C, 32 * kMaxPL);
  g->B = B; g->C = C; g->H = H; g->W = W; g->ws = ws;
  g->nWh = (H + ws - 1) / ws; g->nWw = (W + ws - 1) / ws; g->L = ws * ws;
  g->T = (long long)B * g->nWh * g->nWw * g->L;
  B200_REQUIRE(g->T < (1ll << 31), B200_ERR_UNSUPPORTED, "swin: %lld tokens exceed the 32-bit token index", g->T);
  g->dL.init((uint32_t)g->L); g->dWw.init((uint32_t)g->nWw); g->dWh.init((uint32_t)g->nWh); g->dws.init((uint32_t)ws);
  return B200_OK;
}

inline unsigned warps_grid(long long tokens) { return (unsigned)((tokens + 7) / 8); }
// grid-stride kernels: enough CTAs to fill the chip a few times over, never more than the work
inline unsigned capped_grid(long long tokens, int tokens_per_warp = 1) {
  const long long need = (tokens + 8 * tokens_per_warp - 1) / (8 * tokens_per_warp), cap = (long long)sm_count() * 8;
  return (unsigned)(need < cap ? need : cap);
}
constexpr int kLnMaxCtas = 1024;
inline unsigned ln_bwd_ctas(long long tokens) {
  long long need = (tokens + 63) / 64, cap = (long long)sm_count() * 4;
  if (cap > kLnMaxCtas) cap = kLnMaxCtas;
  return (unsigned)(need < cap ? need : cap);
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API long long b200_swin_num_tokens(int32_t B, int32_t H, int32_t W, int32_t ws) {
  if (B <= 0 || H <= 0 || W <= 0 || ws <= 0) return 0;
  return (long long)B * ((H + ws - 1) / ws) * ((W + ws - 1) / ws) * ws * ws;
}

extern "C" B200_API int b200_swin_ln1_partition(const void* x, const float* gamma, const float* beta, void* n1, float* mean,
                                                float* rstd, int32_t B, int32_t C, int32_t H, int32_t W, int32_t ws,
                                                int32_t shift, int32_t dtype, void* stream) {
  WinGeom g;
  if (int rc = make_geom(&g, B, C, H, W, ws, shift)) return rc;
  B200_REQUIRE(x && gamma && beta && n1 && mean && rstd, B200_ERR_SHAPE, "swin_ln1_partition: null pointer");
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    int vec, iters;
    if (pick_vec<T>(C, &vec, &iters) && (((uintptr_t)x | (uintptr_t)n1) & 15) == 0) {
      const unsigned grid = capped_grid(g.T, 32 / vec);
      B200_DISPATCH_VEC({
        swin_ln1_partition_vec_kernel<T, VEC, ITERS><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)x, gamma, beta, (T*)n1, mean, rstd, g);
        return check_launch("swin_ln1_partition");
      });
    }
    swin_ln1_partition_kernel<T><<<warps_grid(g.T), 256, 0, (cudaStream_t)stream>>>((const T*)x, gamma, beta, (T*)n1, mean, rstd, g);
    return check_launch("swin_ln1_partition");
  });
}

extern "C" B200_API int b200_swin_res_ln2(const void* n1, const void* a, const float* gamma, const float* beta, void* y1,
                                          void* u, float* mean, float* rstd, int64_t tokens, int32_t C, int32_t dtype,
                                          void* stream) {
  B200_REQUIRE(n1 && gamma && beta && u && mean && rstd && (!a || y1), B200_ERR_SHAPE, "swin_res_ln2: null pointer");
  B200_REQUIRE(tokens > 0 && C > 0 && C <= 32 * kMaxPL, B200_ERR_SHAPE, "swin_res_ln2: bad shape");
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    int vec, iters;
    if (pick_vec<T>(C, &vec, &iters) && (((uintptr_t)n1 | (uintptr_t)a | (uintptr_t)y1 | (uintptr_t)u) & 15) == 0) {
      const unsigned grid = capped_grid(tokens, 32 / vec);
      B200_DISPATCH_VEC({
        swin_res_ln2_vec_kernel<T, VEC, ITERS><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)n1, (const T*)a, gamma, beta, (T*)y1,
                                                                                       (T*)u, mean, rstd, tokens, C);
        return check_launch("swin_res_ln2");
      });
    }
    swin_res_ln2_kernel<T><<<warps_grid(tokens), 256, 0, (cudaStream_t)stream>>>((const T*)n1, (const T*)a, gamma, beta, (T*)y1,
                                                                                 (T*)u, mean, rstd, tokens, C);
    return check_launch("swin_res_ln2");
  });
}

extern "C" B200_API int b200_swin_gelu(const void* a, const void* gh, void* out, int64_t n, int32_t dtype, int32_t backward,
                                       void* stream) {
  B200_REQUIRE(a && out && n > 0 && (!backward || gh), B200_ERR_SHAPE, "swin_gelu: bad arguments");
  B200_REQUIRE((((uintptr_t)a | (uintptr_t)out | (uintptr_t)gh) & 15) == 0, B200_ERR_ALIGN, "swin_gelu: pointers must be 16-byte aligned");
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    const long long nv = n / (16 / sizeof(T));
    unsigned grid = (unsigned)((nv + 255) / 256);
    const unsigned cap = (unsigned)sm_count() * 16;
    if (grid > cap) grid = cap;
    if (grid == 0) grid = 1;
    if (backward) swin_gelu_kernel<T, true><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)a, (const T*)gh, (T*)out, n);
    else swin_gelu_kernel<T, false><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)a, nullptr, (T*)out, n);
    return check_launch("swin_gelu");
  });
}

extern "C" B200_API int b200_swin_res_reverse(const void* y1, const void* m, void* out, int32_t B, int32_t C, int32_t H,
                                              int32_t W, int32_t ws, int32_t shift, int32_t dtype, void* stream) {
  WinGeom g;
  if (int rc = make_geom(&g, B, C, H, W, ws, shift)) return rc;
  B200_REQUIRE(y1 && out, B200_ERR_SHAPE, "swin_res_reverse: null pointer");   // m may be null: reverse + crop only
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    int vec, iters;
    if (pick_vec<T>(C, &vec, &iters) && (((uintptr_t)y1 | (uintptr_t)m | (uintptr_t)out) & 15) == 0) {
      const unsigned grid = capped_grid(g.T, 32 / vec);
      B200_DISPATCH_VEC({
        swin_move_vec_kernel<T, VEC, ITERS, 0><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)y1, (const T*)m, (T*)out, g);
        return check_launch("swin_res_reverse");
      });
    }
    swin_res_reverse_kernel<T><<<warps_grid(g.T), 256, 0, (cudaStream_t)stream>>>((const T*)y1, (const T*)m, (T*)out, g);
    return check_launch("swin_res_reverse");
  });
}

static int swin_partition_impl(const void* src, const void* add, void* tok, int32_t B, int32_t C, int32_t H, int32_t W, int32_t ws,
                               int32_t shift, int32_t dtype, void* stream) {
  WinGeom g;
  if (int rc = make_geom(&g, B, C, H, W, ws, shift)) return rc;
  B200_REQUIRE(src && tok, B200_ERR_SHAPE, "swin_partition: null pointer");
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    int vec, iters;
    if (pick_vec<T>(C, &vec, &iters) && (((uintptr_t)src | (uintptr_t)add | (uintptr_t)tok) & 15) == 0) {
      const unsigned grid = capped_grid(g.T, 32 / vec);
      B200_DISPATCH_VEC({
        swin_move_vec_kernel<T, VEC, ITERS, 1><<<grid, 256, 0, (cudaStream_t)stream>>>((const T*)src, (const T*)add, (T*)tok, g);
        return check_launch("swin_partition");
      });
    }
    swin_partition_kernel<T><<<warps_grid(g.T), 256, 0, (cudaStream_t)stream>>>((const T*)src, (const T*)add, (T*)tok, g);
    return check_launch("swin_partition");
  });
}

extern "C" B200_API int b200_swin_partition(const void* src, void* tok, int32_t B, int32_t C, int32_t H, int32_t W,
                                            int32_t ws, int32_t shift, int32_t dtype, void* stream) {
  return swin_partition_impl(src, nullptr, tok, B, C, H, W, ws, shift, dtype, stream);
}

/* tok[t,:] = src[pixel(t),:] + add[pixel(t),:] for real tokens, 0 for padded ones */
extern "C" B200_API int b200_swin_partition_add(const void* src, const void* add, void* tok, int32_t B, int32_t C, int32_t H, int32_t W,
                                                int32_t ws, int32_t shift, int32_t dtype, void* stream) {
  B200_REQUIRE(add, B200_ERR_SHAPE, "swin_partition_add: null pointer");
  return swin_partition_impl(src, add, tok, B, C, H, W, ws, shift, dtype, stream);
}

extern "C" B200_API size_t b200_swin_ln_bwd_workspace_bytes(int64_t tokens, int32_t C) {
  (void)tokens;
  return (size_t)kLnMaxCtas * 2 * C * sizeof(float);
}

// mode 0: LN2 backward (token-major in/out, + residual);  mode 1: LN1 backward (gathers x / scatters gx in NHWC)
extern "C" B200_API int b200_swin_ln_bwd(const void* gout, const void* xin, const void* gres, const float* gamma,
                                         const float* mean, const float* rstd, void* gin, float* ggamma, float* gbeta,
                                         void* workspace, size_t workspace_bytes, int32_t B, int32_t C, int32_t H,
                                         int32_t W, int32_t ws, int32_t shift, int32_t dtype, int32_t mode, void* stream) {
  WinGeom g;
  if (int rc = make_geom(&g, B, C, H, W, ws, shift)) return rc;
  B200_REQUIRE(gout && xin && gamma && mean && rstd && gin && ggamma && gbeta, B200_ERR_SHAPE, "swin_ln_bwd: null pointer");
  B200_REQUIRE(mode == 1 || gres, B200_ERR_SHAPE, "swin_ln_bwd: LN2 mode needs the residual gradient");
  const size_t need = b200_swin_ln_bwd_workspace_bytes(g.T, C);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "swin_ln_bwd: workspace %zu < %zu", workspace_bytes, need);
  const unsigned ctas = ln_bwd_ctas(g.T);
  const int kLnTokensPerCta = (int)((g.T + ctas - 1) / ctas);
  const size_t smem = (size_t)8 * 2 * C * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    int vec, iters;
    if (pick_vec<T>(C, &vec, &iters) && (((uintptr_t)gout | (uintptr_t)xin | (uintptr_t)gres | (uintptr_t)gin) & 15) == 0) {
      B200_DISPATCH_VEC({
        if (mode == 0) {
          auto k = swin_ln_bwd_vec_kernel<T, VEC, ITERS, 0>;
          cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
          k<<<ctas, 256, smem, st>>>((const T*)gout, (const T*)xin, (const T*)gres, gamma, mean, rstd, (T*)gin, (float*)workspace, g);
        } else {
          auto k = swin_ln_bwd_vec_kernel<T, VEC, ITERS, 1>;
          cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
          k<<<ctas, 256, smem, st>>>((const T*)gout, (const T*)xin, nullptr, gamma, mean, rstd, (T*)gin, (float*)workspace, g);
        }
        return check_launch("swin_ln_bwd");
      });
    }
    if (mode == 0) {
      auto k = swin_ln_bwd_kernel<T, 0>;
      cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      k<<<ctas, 256, smem, st>>>((const T*)gout, (const T*)xin, (const T*)gres, gamma, mean, rstd, (T*)gin, (float*)workspace, g, kLnTokensPerCta);
    } else {
      auto k = swin_ln_bwd_kernel<T, 1>;
      cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      k<<<ctas, 256, smem, st>>>((const T*)gout, (const T*)xin, nullptr, gamma, mean, rstd, (T*)gin, (float*)workspace, g, kLnTokensPerCta);
    }
    return check_launch("swin_ln_bwd");
  });
  if (rc) return rc;
  fold_ln_kernel<<<(2 * C + 31) / 32, 1024, 0, st>>>((const float*)workspace, ggamma, gbeta, (int)ctas, C);
  return check_launch("swin_ln_bwd_fold");
}

static const int kColsumMaxSlabs = 512;
static inline int colsum_slabs(int64_t rows, int n) {
  // ~4 CTAs per SM in total across the column strips
  const int strips = (n + 127) / 128;
  long long want = ((long long)b200::sm_count() * 4 + strips - 1) / strips;
  const long long maxs = (rows + 63) / 64;
  if (want > maxs) want = maxs;
  if (want > kColsumMaxSlabs) want = kColsumMaxSlabs;
  return want < 1 ? 1 : (int)want;
}

extern "C" B200_API size_t b200_colsum_workspace_bytes(int64_t rows, int32_t n) {
  (void)rows;
  return (size_t)kColsumMaxSlabs * n * sizeof(float);
}

// out[n] (f32) = column sums of a [rows, n] (bias gradients: attn.in_proj_bias, out_proj.bias, mlp.{0,2}.bias)
extern "C" B200_API int b200_colsum(const void* a, float* out, void* workspace, size_t workspace_bytes, int64_t rows,
                                    int32_t n, int32_t dtype, void* stream) {
  B200_REQUIRE(a && out && rows > 0 && n > 0, B200_ERR_SHAPE, "colsum: bad arguments");
  const size_t need = b200_colsum_workspace_bytes(rows, n);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "colsum: workspace %zu < %zu", workspace_bytes, need);
  const unsigned rblocks = (unsigned)colsum_slabs(rows, n);
  const int rows_per = (int)((rows + rblocks - 1) / rblocks);
  B200_REQUIRE(((uintptr_t)a & 7) == 0 && (n % 4 == 0 || true), B200_ERR_ALIGN, "colsum: input must be 8-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    if (n % 4 != 0 || (((uintptr_t)a) & (4 * sizeof(T) - 1)) != 0) {
      b200::set_error("colsum: n must be a multiple of 4 and the input %zu-byte aligned", 4 * sizeof(T));
      return B200_ERR_ALIGN;
    }
    colsum_partial_kernel<T><<<dim3((n + 127) / 128, rblocks), 256, 0, st>>>((const T*)a, (float*)workspace, rows, n, rows_per);
    return check_launch("colsum_partial");
  });
  if (rc) return rc;
  fold_rows_kernel<<<(n + 31) / 32, 256, 0, st>>>((const float*)workspace, out, (int)rblocks, n);
  return check_launch("colsum_fold");
}
