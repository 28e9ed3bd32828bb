// Classification term of the v8 detection loss (SURVEY 8(f)-4: the step either side of the model forward) as two streaming
// kernels over the Detect head's class maps.  Replaces, for the [B, 8400, nc] logits of ultralytics/utils/loss.py:207-213,235:
//   cat + permute + contiguous + .float() of the three levels, F.one_hot(target_labels) * norm (a dense [B, 8400, nc] f32 target),
//   BCEWithLogitsLoss(reduction="none").sum() and its backward (about a dozen passes over 43 M elements)
// by ONE read of the logits per direction.  The target of anchor (b, a) is described by (label, value): t[b,a,c] = value * [c == label]
// (label < 0: background), which is exactly what TaskAlignedAssigner produces (tal.py:98-107: one-hot of the assigned label,
// scaled by the normalised alignment metric).
//   forward :  sum_{b,a,c} softplus(x) - x * t          (per-CTA partials folded in a fixed order: deterministic)
//   backward:  g[b,a,c] = (sigmoid(x) - t) * scale[0]   written in the layout of the logits (channels_last class maps)
// Rows = anchors (b*A_l + a within a level), C = nc columns, 16-byte vectors; logits may be 16-bit or f32.
#include "common.cuh"

namespace b200 {
namespace {

constexpr int kMaxLevels = 4;
struct BceLevel {
  const void* x;          // logits [rows, C] (row stride = ld elements)
  void* g;                // gradient, same layout (backward only)
  long long rows, ld;     // rows = B * A_l
  int A, a0;              // anchors per image in this level, offset of the level in the concatenated anchor axis
};
struct BceParams {
  BceLevel lv[kMaxLevels];
  int n_levels, C, A_total;
  const int* label;       // [B, A_total]
  const float* value;     // [B, A_total]
  const float* scale;     // backward: device scalar
  float* part;            // forward: [grid] partial sums
  long long vec_total;    // total 16-byte vectors over all levels
};

// max(x,0) + log(1 + exp(-|x|)): the argument of the log lies in (1, 2], so the fast log has no cancellation problem
__device__ __forceinline__ float softplus_f(float x) { return fmaxf(x, 0.f) + __logf(1.f + __expf(-fabsf(x))); }

template <typename T, int VE, bool BWD>
__global__ void __launch_bounds__(256) bce_kernel(const BceParams P) {
  const int vpr = P.C / VE;   // vectors per row
  float acc = 0.f;
  const float sc = BWD ? P.scale[0] : 0.f;
  const uint32_t nvec = (uint32_t)P.vec_total;   // < 2^31 (checked on the host): 32-bit index arithmetic
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += gridDim.x * blockDim.x) {
    uint32_t r = v / (uint32_t)vpr;
    const int k = (int)(v - r * (uint32_t)vpr);
    int l = 0;
    while (l + 1 < P.n_levels && r >= (uint32_t)P.lv[l].rows) { r -= (uint32_t)P.lv[l].rows; ++l; }
    const BceLevel& L = P.lv[l];
    const uint32_t b = r / (uint32_t)L.A, a = r - b * (uint32_t)L.A;
    const long long t = (long long)b * P.A_total + L.a0 + a;
    const int lab = P.label[t] - k * VE;      // position of the positive class inside this vector (if any)
    const float val = P.value[t];
    float x[VE];
    const T* xp = reinterpret_cast<const T*>(L.x) + (long long)r * L.ld + k * VE;
    if (sizeof(T) == 2) {
      const uint4 w = ldg_stream16(xp);
      const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (DT<T>::code == B200_BF16) { x[2 * e] = __uint_as_float(ww[e] << 16); x[2 * e + 1] = __uint_as_float(ww[e] & 0xffff0000u); }
        else { const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&ww[e])); x[2 * e] = f.x; x[2 * e + 1] = f.y; }
      }
    } else {
      const uint4 w = ldg_stream16(xp);
      x[0] = __uint_as_float(w.x); x[1] = __uint_as_float(w.y); x[2] = __uint_as_float(w.z); x[3] = __uint_as_float(w.w);
    }
    if (!BWD) {
#pragma unroll
      for (int e = 0; e < VE; ++e) acc += softplus_f(x[e]) - (e == lab ? x[e] * val : 0.f);
    } else {
      float g[VE];
#pragma unroll
      for (int e = 0; e < VE; ++e) g[e] = (sigmoidf_(x[e]) - (e == lab ? val : 0.f)) * sc;
      T* gp = reinterpret_cast<T*>(L.g) + (long long)r * L.ld + k * VE;
      if (sizeof(T) == 2) {
        uint4 o;
        uint32_t* ow = &o.x;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (DT<T>::code == B200_BF16) { __nv_bfloat162 p = __floats2bfloat162_rn(g[2 * e], g[2 * e + 1]); ow[e] = *reinterpret_cast<uint32_t*>(&p); }
          else { __half2 p = __floats2half2_rn(g[2 * e], g[2 * e + 1]); ow[e] = *reinterpret_cast<uint32_t*>(&p); }
        }
        stg_stream16(gp, o);
      } else {
        stg_stream16(gp, make_uint4(__float_as_uint(g[0]), __float_as_uint(g[1]), __float_as_uint(g[2]), __float_as_uint(g[3])));
      }
    }
  }
  if (!BWD) {
    __shared__ float red[8];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float s = 0.f;
      for (int i = 0; i < 8; ++i) s += red[i];
      P.part[blockIdx.x] = s;
    }
  }
}

__global__ void __launch_bounds__(256) bce_fold_kernel(const float* __restrict__ part, int n, float* __restrict__ out) {
  __shared__ float red[8];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) s += part[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    out[0] = t;
  }
}

int fill(BceParams& P, const void* const* x, void* const* g, const int32_t* A, const int64_t* ld, int n_levels, int B, int C, int dtype,
         const int* label, const float* value) {
  B200_REQUIRE(n_levels >= 1 && n_levels <= kMaxLevels, B200_ERR_SHAPE, "bce: 1..%d levels (got %d)", kMaxLevels, n_levels);
  B200_REQUIRE(dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "bce: unsupported dtype %d", dtype);
  const int ve = dtype == B200_F32 ? 4 : 8;
  B200_REQUIRE(B > 0 && C > 0 && C % ve == 0, B200_ERR_ALIGN, "bce: the class count %d must be a multiple of %d (16-byte vectors)", C, ve);
  B200_REQUIRE(label && value, B200_ERR_SHAPE, "bce: null target");
  P.n_levels = n_levels; P.C = C; P.label = label; P.value = value; P.A_total = 0; P.vec_total = 0;
  for (int l = 0; l < n_levels; ++l) {
    B200_REQUIRE(x[l] && A[l] > 0 && ld[l] >= C && (ld[l] * (dtype == B200_F32 ? 4 : 2)) % 16 == 0 && ((uintptr_t)x[l] & 15) == 0 &&
                     (!g || (g[l] && ((uintptr_t)g[l] & 15) == 0)),
                 B200_ERR_ALIGN, "bce: level %d needs 16-byte aligned rows", l);
    P.lv[l].x = x[l]; P.lv[l].g = g ? g[l] : nullptr; P.lv[l].rows = (long long)B * A[l]; P.lv[l].ld = ld[l]; P.lv[l].A = A[l];
    P.lv[l].a0 = P.A_total;
    P.A_total += A[l];
    P.vec_total += P.lv[l].rows * (C / ve);
  }
  B200_REQUIRE(P.vec_total < (1ll << 31), B200_ERR_SHAPE, "bce: too many elements");
  return B200_OK;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API size_t b200_bce_logits_workspace_bytes(void) { return (size_t)(sm_count() * 8) * sizeof(float); }

extern "C" B200_API int b200_bce_logits_fwd(const void* const* logits, const int32_t* anchors, const int64_t* row_stride, int32_t n_levels,
                                            const int32_t* label, const float* value, float* loss_sum, void* workspace,
                                            size_t workspace_bytes, int32_t B, int32_t C, int32_t dtype, void* stream) {
  BceParams P{};
  if (int rc = fill(P, logits, nullptr, anchors, row_stride, n_levels, B, C, dtype, label, value)) return rc;
  B200_REQUIRE(loss_sum && workspace && workspace_bytes >= b200_bce_logits_workspace_bytes(), B200_ERR_WORKSPACE, "bce_fwd: workspace too small");
  const int grid = sm_count() * 8;
  P.part = (float*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_F32) bce_kernel<float, 4, false><<<grid, 256, 0, st>>>(P);
  else if (dtype == B200_BF16) bce_kernel<__nv_bfloat16, 8, false><<<grid, 256, 0, st>>>(P);
  else bce_kernel<__half, 8, false><<<grid, 256, 0, st>>>(P);
  if (int rc = check_launch("bce_logits_fwd")) return rc;
  bce_fold_kernel<<<1, 256, 0, st>>>(P.part, grid, loss_sum);
  return check_launch("bce_logits_fold");
}

extern "C" B200_API int b200_bce_logits_bwd(const void* const* logits, void* const* grads, const int32_t* anchors, const int64_t* row_stride,
                                            int32_t n_levels, const int32_t* label, const float* value, const float* scale, int32_t B,
                                            int32_t C, int32_t dtype, void* stream) {
  BceParams P{};
  B200_REQUIRE(grads && scale, B200_ERR_SHAPE, "bce_bwd: null pointer");
  if (int rc = fill(P, logits, grads, anchors, row_stride, n_levels, B, C, dtype, label, value)) return rc;
  P.scale = scale;
  const int grid = sm_count() * 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_F32) bce_kernel<float, 4, true><<<grid, 256, 0, st>>>(P);
  else if (dtype == B200_BF16) bce_kernel<__nv_bfloat16, 8, true><<<grid, 256, 0, st>>>(P);
  else bce_kernel<__half, 8, true><<<grid, 256, 0, st>>>(P);
  return check_launch("bce_logits_bwd");
}
