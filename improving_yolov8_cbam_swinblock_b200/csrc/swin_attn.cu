// SwinBlock window attention, forward and backward, fp32-accurate SIMT path (any activation dtype).
// Replaces the bmm / softmax / bmm core of nn.MultiheadAttention as called at swin_block.py:51
// (torch F.multi_head_attention_forward: q scaled by hd^-0.5, softmax over the L = ws*ws keys of the window, no
// mask, no dropout; head h = channels [h*hd, (h+1)*hd) of the packed q|k|v rows).
//
// One CTA per (window, head); one thread per query row, scores of the whole row live in registers (L <= 64), K and
// V rows are staged in shared memory as f32 and read as broadcast float4.  Used for f32 activations (parity
// rtol 1e-5) and as the reference-accurate path for 16-bit ones; the tcgen05 path (swin_attn_tc.cu) supersedes it
// for bf16/f16 when present.
//
//   qkv  [T, 3C]  packed rows (q | k | v) as produced by the in_proj GEMM (+bias)
//   o    [T, C]   heads concatenated
//   lse  [T, nh]  f32 log-sum-exp of the scaled scores (saved for the backward)
// BIAS (SwinBlockRPB): the dense relative-position bias [nh][64][64] (swin_rpb.cu) is added to the scores before the
// mask; the backward also writes each CTA's unscaled dS = p (dP - delta) to its own workspace slot [win][h][64][64].
#include "swin_rpb.cuh"

namespace b200 {
namespace {

constexpr int LMAX = 64;

template <typename T> __device__ __forceinline__ float ldf(const T* p) { return DT<T>::to_f(*p); }

template <typename T, bool BIAS>
__global__ void __launch_bounds__(LMAX) swin_attn_fwd_kernel(const T* __restrict__ qkv, T* __restrict__ o, float* __restrict__ lse,
                                                             int L, int C, int nh, const ShiftMask M, const float* __restrict__ bias) {
  extern __shared__ __align__(16) float sm[];
  const int hd = C / nh, hp = hd + 4;
  float* ks = sm;             // [L][hp]
  float* vs = sm + L * hp;    // [L][hp]
  const int win = blockIdx.x / nh, h = blockIdx.x % nh;
  const long long t0 = (long long)win * L;
  const T* base = qkv + t0 * 3 * C + h * hd;
  for (int i = threadIdx.x; i < L * hd; i += blockDim.x) {
    const int j = i / hd, d = i - j * hd;
    ks[j * hp + d] = ldf(base + (long long)j * 3 * C + C + d);
    vs[j * hp + d] = ldf(base + (long long)j * 3 * C + 2 * C + d);
  }
  __syncthreads();
  const int i = threadIdx.x;
  if (i >= L) return;
  const float scale = rsqrtf((float)hd);
  const T* qrow = base + (long long)i * 3 * C;
  float s[LMAX];
#pragma unroll
  for (int j = 0; j < LMAX; ++j) s[j] = 0.f;
  for (int d = 0; d < hd; d += 4) {
    const float q0 = ldf(qrow + d) * scale, q1 = ldf(qrow + d + 1) * scale, q2 = ldf(qrow + d + 2) * scale,
                q3 = ldf(qrow + d + 3) * scale;
#pragma unroll
    for (int j = 0; j < LMAX; ++j)
      if (j < L) {
        const float4 kv = *reinterpret_cast<const float4*>(ks + j * hp + d);
        s[j] += q0 * kv.x + q1 * kv.y + q2 * kv.z + q3 * kv.w;
      }
  }
  if constexpr (BIAS) {
    const float* brow = bias + ((size_t)h * 64 + i) * 64;
#pragma unroll
    for (int j = 0; j < LMAX; ++j)
      if (j < L) s[j] += brow[j];
  }
  const unsigned long long allowed = allowed_keys(M, win, i);   // shifted-window mask (all ones when shift == 0)
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < LMAX; ++j)
    if (j < L) {
      if (!((allowed >> j) & 1ull)) s[j] = -INFINITY;
      m = fmaxf(m, s[j]);
    }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < LMAX; ++j)
    if (j < L) { s[j] = expf(s[j] - m); sum += s[j]; }
  const float inv = 1.f / sum;
  if (lse) lse[(t0 + i) * nh + h] = m + logf(sum);
  T* orow = o + (t0 + i) * C + h * hd;
  for (int d = 0; d < hd; d += 4) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int j = 0; j < LMAX; ++j)
      if (j < L) {
        const float4 vv = *reinterpret_cast<const float4*>(vs + j * hp + d);
        a0 += s[j] * vv.x; a1 += s[j] * vv.y; a2 += s[j] * vv.z; a3 += s[j] * vv.w;
      }
    orow[d] = DT<T>::from_f(a0 * inv); orow[d + 1] = DT<T>::from_f(a1 * inv);
    orow[d + 2] = DT<T>::from_f(a2 * inv); orow[d + 3] = DT<T>::from_f(a3 * inv);
  }
}

// backward: gqkv [T,3C] from qkv, o, lse and go [T,C]   (SURVEY App. A.3 "Attention")
template <typename T, bool BIAS>
__global__ void __launch_bounds__(LMAX) swin_attn_bwd_kernel(const T* __restrict__ qkv, const T* __restrict__ o,
                                                             const float* __restrict__ lse, const T* __restrict__ go,
                                                             T* __restrict__ gqkv, int L, int C, int nh, const ShiftMask M,
                                                             const float* __restrict__ bias, float* __restrict__ dws) {
  extern __shared__ __align__(16) float sm[];
  const int hd = C / nh, hp = hd + 4, lp = L + 1;
  float* b0 = sm;               // phase 1: K rows     phase 2: dO rows
  float* b1 = sm + L * hp;      // phase 1: V rows     phase 2: Q rows
  float* ps = b1 + L * hp;      // [L][lp] probabilities
  float* ds = ps + L * lp;      // [L][lp] dS (already scaled by hd^-0.5)
  const int win = blockIdx.x / nh, h = blockIdx.x % nh;
  const long long t0 = (long long)win * L;
  const T* base = qkv + t0 * 3 * C + h * hd;
  const T* gobase = go + t0 * C + h * hd;
  T* gbase = gqkv + t0 * 3 * C + h * hd;
  for (int i = threadIdx.x; i < L * hd; i += blockDim.x) {
    const int j = i / hd, d = i - j * hd;
    b0[j * hp + d] = ldf(base + (long long)j * 3 * C + C + d);
    b1[j * hp + d] = ldf(base + (long long)j * 3 * C + 2 * C + d);
  }
  __syncthreads();
  const int i = threadIdx.x;
  const float scale = rsqrtf((float)hd);
  if (i < L) {
    const T* qrow = base + (long long)i * 3 * C;
    const T* gorow = gobase + (long long)i * C;
    const T* orow = o + (t0 + i) * C + h * hd;
    float s[LMAX], dp[LMAX];
#pragma unroll
    for (int j = 0; j < LMAX; ++j) { s[j] = 0.f; dp[j] = 0.f; }
    float delta = 0.f;
    for (int d = 0; d < hd; d += 4) {
      const float q0 = ldf(qrow + d) * scale, q1 = ldf(qrow + d + 1) * scale, q2 = ldf(qrow + d + 2) * scale,
                  q3 = ldf(qrow + d + 3) * scale;
      const float g0 = ldf(gorow + d), g1 = ldf(gorow + d + 1), g2 = ldf(gorow + d + 2), g3 = ldf(gorow + d + 3);
      delta += g0 * ldf(orow + d) + g1 * ldf(orow + d + 1) + g2 * ldf(orow + d + 2) + g3 * ldf(orow + d + 3);
#pragma unroll
      for (int j = 0; j < LMAX; ++j)
        if (j < L) {
          const float4 kv = *reinterpret_cast<const float4*>(b0 + j * hp + d);
          const float4 vv = *reinterpret_cast<const float4*>(b1 + j * hp + d);
          s[j] += q0 * kv.x + q1 * kv.y + q2 * kv.z + q3 * kv.w;
          dp[j] += g0 * vv.x + g1 * vv.y + g2 * vv.z + g3 * vv.w;
        }
    }
    const float l = lse[(t0 + i) * nh + h];
    const unsigned long long allowed = allowed_keys(M, win, i);
    if constexpr (BIAS) {
      const float* brow = bias + ((size_t)h * 64 + i) * 64;
#pragma unroll
      for (int j = 0; j < LMAX; ++j)
        if (j < L) s[j] += brow[j];
    }
#pragma unroll
    for (int j = 0; j < LMAX; ++j)
      if (j < L) {
        const float p = ((allowed >> j) & 1ull) ? expf(s[j] - l) : 0.f;
        const float dsj = p * (dp[j] - delta) * scale;
        ps[i * lp + j] = p;
        ds[i * lp + j] = dsj;
        if constexpr (BIAS) dws[((size_t)win * nh + h) * 4096 + i * 64 + j] = p * (dp[j] - delta);
        s[j] = dsj;
      }
    // dQ[i,:] = sum_j dS[i,j] K[j,:]
    T* gq = gbase + (long long)i * 3 * C;
    for (int d = 0; d < hd; d += 4) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int j = 0; j < LMAX; ++j)
        if (j < L) {
          const float4 kv = *reinterpret_cast<const float4*>(b0 + j * hp + d);
          a0 += s[j] * kv.x; a1 += s[j] * kv.y; a2 += s[j] * kv.z; a3 += s[j] * kv.w;
        }
      gq[d] = DT<T>::from_f(a0); gq[d + 1] = DT<T>::from_f(a1); gq[d + 2] = DT<T>::from_f(a2); gq[d + 3] = DT<T>::from_f(a3);
    }
  }
  __syncthreads();
  // phase 2: restage dO and Q; thread j owns key/value row j
  for (int k = threadIdx.x; k < L * hd; k += blockDim.x) {
    const int r = k / hd, d = k - r * hd;
    b0[r * hp + d] = ldf(gobase + (long long)r * C + d);
    b1[r * hp + d] = ldf(base + (long long)r * 3 * C + d);
  }
  __syncthreads();
  const int j = threadIdx.x;
  if (j >= L) return;
  float pc[LMAX], dc[LMAX];
#pragma unroll
  for (int r = 0; r < LMAX; ++r)
    if (r < L) { pc[r] = ps[r * lp + j]; dc[r] = ds[r * lp + j]; } else { pc[r] = 0.f; dc[r] = 0.f; }
  T* gk = gbase + (long long)j * 3 * C + C;
  T* gv = gbase + (long long)j * 3 * C + 2 * C;
  for (int d = 0; d < hd; d += 4) {
    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f, k0 = 0.f, k1 = 0.f, k2 = 0.f, k3 = 0.f;
#pragma unroll
    for (int r = 0; r < LMAX; ++r)
      if (r < L) {
        const float4 gg = *reinterpret_cast<const float4*>(b0 + r * hp + d);
        const float4 qq = *reinterpret_cast<const float4*>(b1 + r * hp + d);
        v0 += pc[r] * gg.x; v1 += pc[r] * gg.y; v2 += pc[r] * gg.z; v3 += pc[r] * gg.w;
        k0 += dc[r] * qq.x; k1 += dc[r] * qq.y; k2 += dc[r] * qq.z; k3 += dc[r] * qq.w;
      }
    gv[d] = DT<T>::from_f(v0); gv[d + 1] = DT<T>::from_f(v1); gv[d + 2] = DT<T>::from_f(v2); gv[d + 3] = DT<T>::from_f(v3);
    gk[d] = DT<T>::from_f(k0); gk[d + 1] = DT<T>::from_f(k1); gk[d + 2] = DT<T>::from_f(k2); gk[d + 3] = DT<T>::from_f(k3);
  }
}

int check_attn(int64_t tokens, int L, int C, int nh) {
  B200_REQUIRE(tokens > 0 && L > 0 && C > 0 && nh > 0, B200_ERR_SHAPE, "swin_attn: bad shape");
  B200_REQUIRE(L <= LMAX, B200_ERR_UNSUPPORTED, "swin_attn: window of %d tokens > %d unsupported", L, LMAX);
  B200_REQUIRE(tokens % L == 0, B200_ERR_SHAPE, "swin_attn: token count %lld not a multiple of window length %d", (long long)tokens, L);
  B200_REQUIRE(C % nh == 0 && (C / nh) % 4 == 0, B200_ERR_SHAPE, "swin_attn: head dim must be a multiple of 4 (C=%d heads=%d)", C, nh);
  return B200_OK;
}

template <bool BIAS>
int launch_attn_fwd(const void* qkv, const float* bias, void* o, float* lse, int64_t tokens, int L, int C, int nh, const ShiftMask& M,
                    int dtype, cudaStream_t st) {
  const int hd = C / nh;
  const size_t smem = (size_t)2 * L * (hd + 4) * sizeof(float);
  B200_REQUIRE(smem <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "swin_attn_fwd: head dim %d too large", hd);
  const unsigned grid = (unsigned)(tokens / L * nh);
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    auto k = swin_attn_fwd_kernel<T, BIAS>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k<<<grid, LMAX, smem, st>>>((const T*)qkv, (T*)o, lse, L, C, nh, M, bias);
    return check_launch("swin_attn_fwd");
  });
}

template <bool BIAS>
int launch_attn_bwd(const void* qkv, const void* o, const float* lse, const void* go, const float* bias, void* gqkv, float* dws,
                    int64_t tokens, int L, int C, int nh, const ShiftMask& M, int dtype, cudaStream_t st) {
  const int hd = C / nh;
  const size_t smem = ((size_t)2 * L * (hd + 4) + (size_t)2 * L * (L + 1)) * sizeof(float);
  B200_REQUIRE(smem <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "swin_attn_bwd: head dim %d too large", hd);
  const unsigned grid = (unsigned)(tokens / L * nh);
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    auto k = swin_attn_bwd_kernel<T, BIAS>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k<<<grid, LMAX, smem, st>>>((const T*)qkv, (const T*)o, lse, (const T*)go, (T*)gqkv, L, C, nh, M, bias, dws);
    return check_launch("swin_attn_bwd");
  });
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_swin_attn_fwd(const void* qkv, void* o, float* lse, int64_t tokens, int32_t L, int32_t C,
                                           int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                           void* stream) {
  if (int rc = check_attn(tokens, L, C, nh)) return rc;
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(qkv && o, B200_ERR_SHAPE, "swin_attn_fwd: null pointer");
  return launch_attn_fwd<false>(qkv, nullptr, o, lse, tokens, L, C, nh, M, dtype, (cudaStream_t)stream);
}

extern "C" B200_API int b200_swin_attn_bwd(const void* qkv, const void* o, const float* lse, const void* go, void* gqkv,
                                           int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws,
                                           int32_t shift, int32_t dtype, void* stream) {
  if (int rc = check_attn(tokens, L, C, nh)) return rc;
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(qkv && o && lse && go && gqkv, B200_ERR_SHAPE, "swin_attn_bwd: null pointer");
  return launch_attn_bwd<false>(qkv, o, lse, go, nullptr, gqkv, nullptr, tokens, L, C, nh, M, dtype, (cudaStream_t)stream);
}

extern "C" B200_API int b200_swin_attn_fwd_rpb(const void* qkv, const float* bias, void* o, float* lse, int64_t tokens, int32_t L,
                                               int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift,
                                               int32_t dtype, void* stream) {
  if (int rc = check_attn(tokens, L, C, nh)) return rc;
  if (int rc = check_rpb(L, ws)) return rc;
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(qkv && bias && o, B200_ERR_SHAPE, "swin_attn_fwd_rpb: null pointer");
  return launch_attn_fwd<true>(qkv, bias, o, lse, tokens, L, C, nh, M, dtype, (cudaStream_t)stream);
}

extern "C" B200_API int b200_swin_attn_bwd_rpb(const void* qkv, const void* o, const float* lse, const void* go, const float* bias,
                                               void* gqkv, float* gtable, int32_t table_rows, void* workspace, size_t workspace_bytes,
                                               int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws,
                                               int32_t shift, int32_t dtype, void* stream) {
  if (int rc = check_attn(tokens, L, C, nh)) return rc;
  if (int rc = check_rpb(L, ws)) return rc;
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(table_rows == (2 * ws - 1) * (2 * ws - 1), B200_ERR_SHAPE, "swin_attn_bwd_rpb: table has %d rows, ws %d needs %d",
               table_rows, ws, (2 * ws - 1) * (2 * ws - 1));
  B200_REQUIRE(qkv && o && lse && go && bias && gqkv && gtable && workspace, B200_ERR_SHAPE, "swin_attn_bwd_rpb: null pointer");
  const long long nslots = tokens / L;
  B200_REQUIRE(workspace_bytes >= rpb_workspace_bytes(nslots, nh), B200_ERR_WORKSPACE, "swin_attn_bwd_rpb: workspace %zu < %zu bytes",
               workspace_bytes, rpb_workspace_bytes(nslots, nh));
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = launch_attn_bwd<true>(qkv, o, lse, go, bias, gqkv, (float*)workspace, tokens, L, C, nh, M, dtype, st)) return rc;
  return rpb_fold((const float*)workspace, nslots, nh, ws, gtable, st);
}
