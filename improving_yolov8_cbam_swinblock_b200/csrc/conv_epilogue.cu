// Fused BatchNorm2d (+ SiLU) epilogue of the stock `Conv` block, forward and backward, NHWC.
// Replaces `self.act(self.bn(...))` of Conv.forward (ultralytics/nn/modules/conv.py:65-79: BatchNorm2d then SiLU) for
// the SPPF cv1/cv2 convolutions (block.py:218-219; SURVEY section 8(f)-1) and, through the same module, the other
// Conv callers either side of the hot path.  Training mode uses per-GPU batch statistics like the reference (no
// SyncBN) and updates running_mean / running_var exactly like torch (momentum, unbiased variance).
//
// The conv output x is a row-major [M = B*H*W, C] matrix.  A thread owns one 16-byte channel vector (8 bf16 / 4 f32)
// and walks rows; a CTA owns a contiguous block of rows:
//   fwd  stats : per-channel shifted sums (shift = first row of the block, so E[(x-k)^2] - E[x-k]^2 does not cancel)
//                -> per-CTA (mean, M2) partials
//        final : warp per channel: Chan-merge the partials in a fixed order -> mean, rstd, running stats,
//                scale = gamma*rstd, shift = beta - mean*scale
//        apply : z = act(x*scale + shift)                       (x read twice, z written once: 2R + 1W;
//                                                                torch: stats R, transform R+W, SiLU R+W)
//   bwd  reduce: gy = gz * act'(y) recomputed from x; per-channel sum(gy), sum(gy*xhat) partials
//        final : warp per channel -> g_gamma, g_beta
//        apply : gx = gamma*rstd*(gy - sum(gy)/M - xhat*sum(gy*xhat)/M)     (4R + 1W; torch: 6R + 2W)
// Nothing but x, mean and rstd is kept for the backward (torch keeps x, the BN output and mean/rstd).
// Deterministic: no atomics, fixed summation order.
#include <type_traits>

#include "common.cuh"

namespace b200 {
namespace {

constexpr int kT = 256;

struct BnGeo {
  long long M;      // rows
  int C, nch, tpr, ngrp, rpt, rpb, G;   // vectors/row, threads/row, row groups/CTA, rows/thread, rows/CTA, CTAs
  float invM;
};

template <typename T, int VW> struct alignas(sizeof(T) * VW) VP { T e[VW]; };
template <typename T, int VW>
__device__ __forceinline__ void unpack(const uint4& raw, float (&v)[VW]) {
  if constexpr (sizeof(T) == 4) {
    v[0] = __uint_as_float(raw.x); v[1] = __uint_as_float(raw.y); v[2] = __uint_as_float(raw.z); v[3] = __uint_as_float(raw.w);
  } else if constexpr (std::is_same<T, __nv_bfloat16>::value) {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u); }
  } else {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
  }
}
template <typename T, int VW>
__device__ __forceinline__ uint4 pack(const float (&v)[VW]) {
  uint4 r;
  if constexpr (sizeof(T) == 4) {
    r = make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  } else {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        const __nv_bfloat162 p = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&p);
      } else {
        const __half2 p = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&p);
      }
    }
    r = make_uint4(w[0], w[1], w[2], w[3]);
  }
  return r;
}

__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// sigmoid: exact-ish (ex2 + rcp) for f32 activations, one MUFU.TANH for 16-bit activations (error 2^-11 << 2^-8 of bf16)
template <bool FAST> __device__ __forceinline__ float sigmoid_t(float y) {
  if (FAST) return fmaf(0.5f, tanh_fast(0.5f * y), 0.5f);
  return __frcp_rn(1.f + __expf(-y));
}

constexpr int kFT = 256, kFW = 8;   // finalize kernels: threads per CTA, warps per channel (one channel per CTA; 16 warps measured no better)
constexpr int RB = 4;   // rows in flight per thread: RB independent 16-byte loads before any use

// per-CTA additive reduction of NV values per channel held by the row groups: red[ngrp][NV][C] -> out via f(c, v[NV])
template <int NV, typename F>
__device__ __forceinline__ void cta_fold(float* red, int C, int ngrp, F emit) {
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += kT) {
    float acc[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) acc[j] = 0.f;
    for (int g = 0; g < ngrp; ++g) {
#pragma unroll
      for (int j = 0; j < NV; ++j) acc[j] += red[((size_t)g * NV + j) * C + c];
    }
    emit(c, acc);
  }
}

// ---- forward statistics: per-CTA sums of (x-k), (x-k)^2 with ONE shift k[c] = x[0][c] for the whole tensor, so the
// partials of different CTAs simply add up and E[d^2] - E[d]^2 does not cancel (|mean - k| ~ one standard deviation)
template <typename T, int VW>
__global__ void __launch_bounds__(kT, 4) bn_stats_kernel(const T* __restrict__ x, float* __restrict__ part, const BnGeo G) {
  extern __shared__ __align__(16) float red[];   // [ngrp][2][C]
  const int C = G.C, tpr = G.tpr;
  const int rg = threadIdx.x / tpr, ch = threadIdx.x - rg * tpr;
  const long long r0 = (long long)blockIdx.x * G.rpb;
  const int nrows = (int)min((long long)G.rpb, G.M - r0);
  if (rg < G.ngrp) {
    float s[VW], q[VW], k[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) { s[e] = 0.f; q[e] = 0.f; }
    unpack<T, VW>(ldg_stream16(x + ch * VW), k);
    const T* base = x + (size_t)r0 * C + ch * VW;
    for (int r = rg; r < nrows; r += RB * G.ngrp) {
      uint4 raw[RB];
#pragma unroll
      for (int u = 0; u < RB; ++u)
        if (r + u * G.ngrp < nrows) raw[u] = ldg_stream16(base + (size_t)(r + u * G.ngrp) * C);
#pragma unroll
      for (int u = 0; u < RB; ++u)
        if (r + u * G.ngrp < nrows) {
          float v[VW];
          unpack<T, VW>(raw[u], v);
#pragma unroll
          for (int e = 0; e < VW; ++e) { const float d = v[e] - k[e]; s[e] += d; q[e] = fmaf(d, d, q[e]); }
        }
    }
    float* rs = red + (size_t)rg * 2 * C + ch * VW;
#pragma unroll
    for (int e = 0; e < VW; ++e) { rs[e] = s[e]; rs[C + e] = q[e]; }
  }
  float* dst = part + (size_t)blockIdx.x * 2 * C;
  cta_fold<2>(red, C, G.ngrp, [&](int c, const float (&a)[2]) { dst[c] = a[0]; dst[C + c] = a[1]; });
}

// ---- forward finalize: warp per channel sums the G partials (fixed order) -> mean, rstd, running stats, scale/shift
template <typename T>
__global__ void __launch_bounds__(kFT) bn_final_kernel(const T* __restrict__ x, const float* __restrict__ part,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      float* __restrict__ running_mean, float* __restrict__ running_var,
                                                      float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                      float* __restrict__ scsh, float eps, float momentum, int training,
                                                      long long* __restrict__ num_batches_tracked, const BnGeo G) {
  // kFW warps per channel: the G partial rows (up to 16 per SM) are summed by 256 lanes with 2 loads in flight each --
  // one warp per channel made this 8-CTA kernel a 10 us latency chain, 59 times per step (2982 -> 3123 img/s)
  __shared__ float fs[kFT / 32][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = warp % kFW, C = G.C;
  const int c = blockIdx.x * (kFT / 32 / kFW) + warp / kFW;
  const bool live = c < C;
  float mean, rstd;
  // nn.BatchNorm2d.forward's bookkeeping, folded in here instead of one more launch per layer (59 per step)
  if (training && num_batches_tracked && blockIdx.x == 0 && threadIdx.x == 0) *num_batches_tracked += 1;
  if (training) {
    float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
    if (live) {
      int g = sub * 32 + lane;
      for (; g + 32 * kFW < G.G; g += 64 * kFW) {
        s0 += part[(size_t)g * 2 * C + c]; q0 += part[(size_t)g * 2 * C + C + c];
        s1 += part[(size_t)(g + 32 * kFW) * 2 * C + c]; q1 += part[(size_t)(g + 32 * kFW) * 2 * C + C + c];
      }
      if (g < G.G) { s0 += part[(size_t)g * 2 * C + c]; q0 += part[(size_t)g * 2 * C + C + c]; }
    }
    const float Sw = warp_sum(s0 + s1), Qw = warp_sum(q0 + q1);
    if (lane == 0) { fs[warp][0] = Sw; fs[warp][1] = Qw; }
    __syncthreads();
    if (!live || sub != 0) return;
    float S = 0.f, Q = 0.f;
#pragma unroll
    for (int k = 0; k < kFW; ++k) { S += fs[warp + k][0]; Q += fs[warp + k][1]; }
    const float dm = S * G.invM;
    mean = DT<T>::to_f(x[c]) + dm;
    const float m2 = fmaxf(Q - S * dm, 0.f);
    const float var = m2 * G.invM;   // biased variance normalises (torch BatchNorm)
    rstd = rsqrtf(var + eps);
    if (lane == 0 && running_mean) {
      const float unb = G.M > 1 ? m2 / (float)(G.M - 1) : var;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * unb;
    }
  } else {
    if (!live || sub != 0) return;
    mean = running_mean[c];
    rstd = rsqrtf(running_var[c] + eps);
  }
  if (lane == 0) {
    if (mean_out) { mean_out[c] = mean; rstd_out[c] = rstd; }
    const float sc = gamma[c] * rstd;
    scsh[c] = sc;
    scsh[C + c] = beta[c] - mean * sc;
  }
}

// ---- forward apply: z = act(x*scale + shift) ---------------------------------------------------------------
template <typename T, int VW, int ACT>
__global__ void __launch_bounds__(kT, 4) bn_apply_kernel(const T* __restrict__ x, const float* __restrict__ scsh,
                                                      T* __restrict__ z, const BnGeo G) {
  constexpr bool FAST = sizeof(T) == 2;
  const int C = G.C, tpr = G.tpr;
  const int rg = threadIdx.x / tpr, ch = threadIdx.x - rg * tpr;
  if (rg >= G.ngrp) return;
  const long long r0 = (long long)blockIdx.x * G.rpb;
  const int nrows = (int)min((long long)G.rpb, G.M - r0);
  float sc[VW], sh[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) { sc[e] = scsh[ch * VW + e]; sh[e] = scsh[C + ch * VW + e]; }
  const T* xb = x + (size_t)r0 * C + ch * VW;
  T* zb = z + (size_t)r0 * C + ch * VW;
  for (int r = rg; r < nrows; r += RB * G.ngrp) {
    uint4 raw[RB];
#pragma unroll
    for (int u = 0; u < RB; ++u)
      if (r + u * G.ngrp < nrows) raw[u] = ldg_stream16(xb + (size_t)(r + u * G.ngrp) * C);
#pragma unroll
    for (int u = 0; u < RB; ++u)
      if (r + u * G.ngrp < nrows) {
        float v[VW];
        unpack<T, VW>(raw[u], v);
#pragma unroll
        for (int e = 0; e < VW; ++e) {
          const float y = fmaf(v[e], sc[e], sh[e]);
          v[e] = ACT ? y * sigmoid_t<FAST>(y) : y;
        }
        stg_stream16(zb + (size_t)(r + u * G.ngrp) * C, pack<T, VW>(v));
      }
  }
}

// gy = gz * act'(y), y = x*a + b
template <bool FAST, int ACT> __device__ __forceinline__ float grad_y(float g, float y) {
  if (!ACT) return g;
  const float sg = sigmoid_t<FAST>(y);
  return g * (sg * fmaf(y, 1.f - sg, 1.f));
}

// ---- backward reduce: per-CTA sum(gy), sum(gy*x) with gy recomputed from x (sum(gy*xhat) follows in the finalize) --
template <typename T, int VW, int ACT>
__global__ void __launch_bounds__(kT, 4) bn_bwd_reduce_kernel(const T* __restrict__ x, const T* __restrict__ gz,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           const float* __restrict__ mean, const float* __restrict__ rstd,
                                                           float* __restrict__ part, const long long gzs, const BnGeo G) {
  constexpr bool FAST = sizeof(T) == 2;   // gzs: row stride of gz in elements (the gradient of a concat slice is a strided view)
  extern __shared__ __align__(16) float red[];   // [ngrp][2][C]
  const int C = G.C, tpr = G.tpr;
  const int rg = threadIdx.x / tpr, ch = threadIdx.x - rg * tpr;
  const long long r0 = (long long)blockIdx.x * G.rpb;
  const int nrows = (int)min((long long)G.rpb, G.M - r0);
  if (rg < G.ngrp) {
    float a[VW], b[VW], a1[VW], a2[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) {
      const int c = ch * VW + e;
      a[e] = gamma[c] * rstd[c];
      b[e] = beta[c] - mean[c] * a[e];
      a1[e] = 0.f; a2[e] = 0.f;
    }
    const T* xb = x + (size_t)r0 * C + ch * VW;
    const T* gb = gz + (size_t)r0 * gzs + ch * VW;
    constexpr int RB2 = RB / 2;
    for (int r = rg; r < nrows; r += RB2 * G.ngrp) {
      uint4 rx[RB2], rgz[RB2];
#pragma unroll
      for (int u = 0; u < RB2; ++u)
        if (r + u * G.ngrp < nrows) {
          rx[u] = ldg_stream16(xb + (size_t)(r + u * G.ngrp) * C);
          rgz[u] = ldg_stream16(gb + (size_t)(r + u * G.ngrp) * gzs);
        }
#pragma unroll
      for (int u = 0; u < RB2; ++u)
        if (r + u * G.ngrp < nrows) {
          float v[VW], g[VW];
          unpack<T, VW>(rx[u], v);
          unpack<T, VW>(rgz[u], g);
#pragma unroll
          for (int e = 0; e < VW; ++e) {
            const float gy = grad_y<FAST, ACT>(g[e], fmaf(v[e], a[e], b[e]));
            a1[e] += gy;
            a2[e] = fmaf(gy, v[e], a2[e]);
          }
        }
    }
    float* rr = red + (size_t)rg * 2 * C + ch * VW;
#pragma unroll
    for (int e = 0; e < VW; ++e) { rr[e] = a1[e]; rr[C + e] = a2[e]; }
  }
  float* dst = part + (size_t)blockIdx.x * 2 * C;
  cta_fold<2>(red, C, G.ngrp, [&](int c, const float (&acc)[2]) { dst[c] = acc[0]; dst[C + c] = acc[1]; });
}

// ---- backward finalize: warp per channel -> g_beta = sum(gy), g_gamma = sum(gy*xhat) = rstd*(sum(gy*x) - mean*sum(gy)),
// and the three coefficients of g_x = A*gy + Bc*x + Cc  (coef[3][C]) --------------------------------------------------
__global__ void __launch_bounds__(kFT) bn_bwd_final_kernel(const float* __restrict__ part, const float* __restrict__ gamma,
                                                          const float* __restrict__ mean, const float* __restrict__ rstd,
                                                          float* __restrict__ ggamma, float* __restrict__ gbeta,
                                                          float* __restrict__ coef, int training, const BnGeo G) {
  __shared__ float fs[kFT / 32][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, sub = warp % kFW, C = G.C;
  const int c = blockIdx.x * (kFT / 32 / kFW) + warp / kFW;
  const bool live = c < C;
  float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
  if (live) {
    int g = sub * 32 + lane;
    for (; g + 32 * kFW < G.G; g += 64 * kFW) {
      s0 += part[(size_t)g * 2 * C + c]; q0 += part[(size_t)g * 2 * C + C + c];
      s1 += part[(size_t)(g + 32 * kFW) * 2 * C + c]; q1 += part[(size_t)(g + 32 * kFW) * 2 * C + C + c];
    }
    if (g < G.G) { s0 += part[(size_t)g * 2 * C + c]; q0 += part[(size_t)g * 2 * C + C + c]; }
  }
  const float Sw = warp_sum(s0 + s1), Qw = warp_sum(q0 + q1);
  if (lane == 0) { fs[warp][0] = Sw; fs[warp][1] = Qw; }
  __syncthreads();
  if (!live || sub != 0) return;
  float sgy = 0.f, sgyx = 0.f;
#pragma unroll
  for (int k = 0; k < kFW; ++k) { sgy += fs[warp + k][0]; sgyx += fs[warp + k][1]; }
  if (lane == 0) {
    const float mu = mean[c], rs = rstd[c], ga = gamma[c];
    const float gg = rs * (sgyx - mu * sgy);
    gbeta[c] = sgy;
    ggamma[c] = gg;
    // gx = ga*rs*(gy - sgy/M - xhat*gg/M), xhat = (x - mu)*rs   (eval mode: statistics are constants -> gx = ga*rs*gy)
    const float A = ga * rs, k1 = training ? sgy * G.invM : 0.f, k2 = training ? gg * G.invM : 0.f;
    coef[c] = A;
    coef[C + c] = -A * k2 * rs;
    coef[2 * C + c] = -A * k1 + A * k2 * rs * mu;
  }
}

// ---- backward apply: g_x = A*gy + Bc*x + Cc -----------------------------------------------------------------------
template <typename T, int VW, int ACT>
__global__ void __launch_bounds__(kT, 4) bn_bwd_apply_kernel(const T* __restrict__ x, const T* __restrict__ gz,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          const float* __restrict__ mean, const float* __restrict__ rstd,
                                                          const float* __restrict__ coef, T* __restrict__ gx, const long long gzs,
                                                          const BnGeo G) {
  constexpr bool FAST = sizeof(T) == 2;
  extern __shared__ __align__(16) float cs[];   // [5][C]: a, b (y = x*a + b), A, Bc, Cc
  const int C = G.C, tpr = G.tpr;
  for (int c = threadIdx.x; c < C; c += kT) {
    const float a = gamma[c] * rstd[c];
    cs[c] = a;
    cs[C + c] = beta[c] - mean[c] * a;
    cs[2 * C + c] = coef[c];
    cs[3 * C + c] = coef[C + c];
    cs[4 * C + c] = coef[2 * C + c];
  }
  __syncthreads();
  const int rg = threadIdx.x / tpr, ch = threadIdx.x - rg * tpr;
  if (rg >= G.ngrp) return;
  const long long r0 = (long long)blockIdx.x * G.rpb;
  const int nrows = (int)min((long long)G.rpb, G.M - r0);
  const T* xb = x + (size_t)r0 * C + ch * VW;
  const T* gb = gz + (size_t)r0 * gzs + ch * VW;
  T* ob = gx + (size_t)r0 * C + ch * VW;
  // The five per-channel constants of this thread's channel vector stay in shared memory and are re-read four channels at a
  // time (5 LDS.128 per half vector): holding all 5 x VW of them in registers cost 80 registers = 3 CTAs per SM
  const float* cv = cs + ch * VW;
  constexpr int RB2 = RB / 2;
  for (int r = rg; r < nrows; r += RB2 * G.ngrp) {
    uint4 rx[RB2], rgz[RB2];
#pragma unroll
    for (int u = 0; u < RB2; ++u)
      if (r + u * G.ngrp < nrows) {
        rx[u] = ldg_stream16(xb + (size_t)(r + u * G.ngrp) * C);
        rgz[u] = ldg_stream16(gb + (size_t)(r + u * G.ngrp) * gzs);
      }
    float v[RB2][VW], g[RB2][VW];
#pragma unroll
    for (int u = 0; u < RB2; ++u) {
      unpack<T, VW>(rx[u], v[u]);
      unpack<T, VW>(rgz[u], g[u]);
    }
#pragma unroll
    for (int q = 0; q < VW / 4; ++q) {
      const float4 t0 = *reinterpret_cast<const float4*>(cv + 4 * q);
      const float4 t1 = *reinterpret_cast<const float4*>(cv + C + 4 * q);
      const float4 t2 = *reinterpret_cast<const float4*>(cv + 2 * C + 4 * q);
      const float4 t3 = *reinterpret_cast<const float4*>(cv + 3 * C + 4 * q);
      const float4 t4 = *reinterpret_cast<const float4*>(cv + 4 * C + 4 * q);
      const float a[4] = {t0.x, t0.y, t0.z, t0.w}, b[4] = {t1.x, t1.y, t1.z, t1.w}, kA[4] = {t2.x, t2.y, t2.z, t2.w},
                  kB[4] = {t3.x, t3.y, t3.z, t3.w}, kC[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
      for (int u = 0; u < RB2; ++u)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float xe = v[u][4 * q + e];
          const float gy = grad_y<FAST, ACT>(g[u][4 * q + e], fmaf(xe, a[e], b[e]));
          v[u][4 * q + e] = fmaf(kA[e], gy, fmaf(kB[e], xe, kC[e]));
        }
    }
#pragma unroll
    for (int u = 0; u < RB2; ++u)
      if (r + u * G.ngrp < nrows) stg_stream16(ob + (size_t)(r + u * G.ngrp) * C, pack<T, VW>(v[u]));
  }
}

void fill_geo(BnGeo& G, long long M, int C, int vw) {
  G.M = M; G.C = C; G.nch = C / vw; G.tpr = G.nch; G.ngrp = kT / G.tpr;
  long long rpt = (M + (long long)592 * G.ngrp - 1) / ((long long)592 * G.ngrp);   // ~4 CTAs per SM ...
  if (rpt < 4) rpt = 4;
  while ((M + rpt * G.ngrp - 1) / (rpt * G.ngrp) > 2368) rpt *= 2;                  // ... and at most 16 per SM
  G.rpt = (int)rpt;
  G.rpb = G.rpt * G.ngrp;
  G.G = (int)((M + G.rpb - 1) / G.rpb);
  G.invM = 1.f / (float)M;
}

int make_geo(BnGeo& G, long long M, int C, int dtype, const void* p0, const void* p1, const void* p2) {
  const int vw = dtype == B200_F32 ? 4 : 8;
  B200_REQUIRE(M > 0 && C > 0, B200_ERR_SHAPE, "bn_silu: bad shape rows=%lld C=%d", M, C);
  B200_REQUIRE(dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "bn_silu: unsupported dtype code %d", dtype);
  B200_REQUIRE(C % vw == 0 && C / vw <= kT, B200_ERR_UNSUPPORTED, "bn_silu: C=%d must be a multiple of %d and <= %d", C, vw, vw * kT);
  B200_REQUIRE((((uintptr_t)p0 | (uintptr_t)p1 | (uintptr_t)p2) & 15) == 0, B200_ERR_ALIGN, "bn_silu: tensors must be 16-byte aligned");
  fill_geo(G, M, C, vw);
  return B200_OK;
}

inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace
}  // namespace b200

extern "C" B200_API int b200_bn_silu_supported(int64_t rows, int32_t C, int32_t dtype) {
  const int vw = dtype == B200_F32 ? 4 : 8;
  return rows > 0 && C > 0 && (dtype >= 0 && dtype <= 2) && C % vw == 0 && C / vw <= b200::kT;
}

extern "C" B200_API size_t b200_bn_silu_workspace_bytes(int64_t rows, int32_t C, int32_t dtype) {
  if (!b200_bn_silu_supported(rows, C, dtype)) return 0;
  b200::BnGeo G;
  b200::fill_geo(G, rows, C, dtype == B200_F32 ? 4 : 8);
  return b200::up256((size_t)G.G * 2 * C * 4) + b200::up256((size_t)3 * C * 4);   // per-CTA partials + scale/shift | bwd coefficients
}

extern "C" B200_API int b200_bn_silu_fwd_tracked(const void* x, const float* gamma, const float* beta, float* running_mean,
                                                 float* running_var, int64_t* num_batches_tracked, void* z, float* mean_out,
                                                 float* rstd_out, void* workspace, size_t workspace_bytes, int64_t rows, int32_t C,
                                                 float eps, float momentum, int32_t training, int32_t act, int32_t dtype,
                                                 void* stream);

extern "C" B200_API int b200_bn_silu_fwd(const void* x, const float* gamma, const float* beta, float* running_mean,
                                         float* running_var, void* z, float* mean_out, float* rstd_out, void* workspace,
                                         size_t workspace_bytes, int64_t rows, int32_t C, float eps, float momentum,
                                         int32_t training, int32_t act, int32_t dtype, void* stream) {
  return b200_bn_silu_fwd_tracked(x, gamma, beta, running_mean, running_var, nullptr, z, mean_out, rstd_out, workspace, workspace_bytes,
                                  rows, C, eps, momentum, training, act, dtype, stream);
}

extern "C" B200_API int b200_bn_silu_fwd_tracked(const void* x, const float* gamma, const float* beta, float* running_mean,
                                                 float* running_var, int64_t* num_batches_tracked, void* z, float* mean_out,
                                                 float* rstd_out, void* workspace, size_t workspace_bytes, int64_t rows, int32_t C,
                                                 float eps, float momentum, int32_t training, int32_t act, int32_t dtype,
                                                 void* stream) {
  using namespace b200;
  B200_REQUIRE(x && gamma && beta && z, B200_ERR_SHAPE, "bn_silu_fwd: null tensor pointer");
  B200_REQUIRE(training || (running_mean && running_var), B200_ERR_SHAPE, "bn_silu_fwd: eval mode needs running statistics");
  BnGeo G;
  if (int rc = make_geo(G, rows, C, dtype, x, z, nullptr)) return rc;
  const size_t need = up256((size_t)G.G * 2 * C * 4) + up256((size_t)3 * C * 4);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "bn_silu_fwd: workspace %zu < %zu bytes", workspace_bytes, need);
  float* part = (float*)workspace;
  float* scsh = (float*)((char*)workspace + up256((size_t)G.G * 2 * C * 4));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)G.ngrp * 2 * C * 4;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    constexpr int VW = 16 / (int)sizeof(T);
    if (training) bn_stats_kernel<T, VW><<<G.G, kT, smem, st>>>((const T*)x, part, G);
    bn_final_kernel<T><<<(C * kFW + kFT / 32 - 1) / (kFT / 32), kFT, 0, st>>>((const T*)x, part, gamma, beta, running_mean, running_var,
              mean_out, rstd_out, scsh, eps, momentum, training, (long long*)num_batches_tracked, G);
    if (act) bn_apply_kernel<T, VW, 1><<<G.G, kT, 0, st>>>((const T*)x, scsh, (T*)z, G);
    else bn_apply_kernel<T, VW, 0><<<G.G, kT, 0, st>>>((const T*)x, scsh, (T*)z, G);
    return check_launch("bn_silu_fwd");
  });
}

extern "C" B200_API int b200_bn_silu_bwd(const void* gz, int64_t gz_row_stride, const void* x, const float* gamma, const float* beta,
                                         const float* mean, const float* rstd, void* gx, float* ggamma, float* gbeta,
                                         void* workspace, size_t workspace_bytes, int64_t rows, int32_t C, int32_t training,
                                         int32_t act, int32_t dtype, void* stream) {
  using namespace b200;
  B200_REQUIRE(gz && x && gamma && beta && mean && rstd && gx && ggamma && gbeta, B200_ERR_SHAPE, "bn_silu_bwd: null tensor pointer");
  BnGeo G;
  if (int rc = make_geo(G, rows, C, dtype, x, gz, gx)) return rc;
  const long long gzs = gz_row_stride > 0 ? gz_row_stride : C;
  B200_REQUIRE(gzs >= C && (gzs * (dtype == B200_F32 ? 4 : 2)) % 16 == 0, B200_ERR_ALIGN,
               "bn_silu_bwd: gz row stride %lld must be >= C and a multiple of 16 bytes", gzs);
  const size_t need = up256((size_t)G.G * 2 * C * 4) + up256((size_t)3 * C * 4);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "bn_silu_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
  float* part = (float*)workspace;
  float* coef = (float*)((char*)workspace + up256((size_t)G.G * 2 * C * 4));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)G.ngrp * 2 * C * 4;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    constexpr int VW = 16 / (int)sizeof(T);
    if (act) bn_bwd_reduce_kernel<T, VW, 1><<<G.G, kT, smem, st>>>((const T*)x, (const T*)gz, gamma, beta, mean, rstd, part, gzs, G);
    else bn_bwd_reduce_kernel<T, VW, 0><<<G.G, kT, smem, st>>>((const T*)x, (const T*)gz, gamma, beta, mean, rstd, part, gzs, G);
    bn_bwd_final_kernel<<<(C * kFW + kFT / 32 - 1) / (kFT / 32), kFT, 0, st>>>(part, gamma, mean, rstd, ggamma, gbeta, coef, training, G);
    const size_t smc = (size_t)5 * C * 4;
    if (act) bn_bwd_apply_kernel<T, VW, 1><<<G.G, kT, smc, st>>>((const T*)x, (const T*)gz, gamma, beta, mean, rstd, coef, (T*)gx, gzs, G);
    else bn_bwd_apply_kernel<T, VW, 0><<<G.G, kT, smc, st>>>((const T*)x, (const T*)gz, gamma, beta, mean, rstd, coef, (T*)gx, gzs, G);
    return check_launch("bn_silu_bwd");
  });
}
