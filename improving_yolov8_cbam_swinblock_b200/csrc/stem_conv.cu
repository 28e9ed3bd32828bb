// The model's first convolution -- Conv(3, c2, k=3, s=2, p=1) on the 640x640 input (yaml backbone row 0; conv.py:37-91 `self.conv`,
// bias-free, BatchNorm follows) -- forward and weight gradient.  cuDNN has no tensor-op kernel for 3 input channels in 16-bit NHWC:
// it converts the 157 MB input to fp32, runs a TF32 fprop and converts the result back (652 us), and pads the channels and runs an
// sm80 legacy wgrad for the backward (808 us); the data movement alone is 367 MB = 56 us at the HBM roofline.  Here:
//   forward : CTA = 4 output rows of one image; the 9 input rows are staged ONCE in shared memory (16-byte copies) and every warp
//             computes 16 output pixels x c2 channels per step with mma.sync m16n8k16 (bf16/f16 in, f32 accumulate).  The
//             im2col operand is never materialised: for one kernel row ky the 9 values (kx, c) of an output pixel are
//             CONTIGUOUS in the NHWC row (elements 6*ox-3 .. 6*ox+5), so with K ordered as k = 10*ky + j, j = 0 a dummy slot whose
//             weight is zero (element 6*ox-4: it makes every (k, k+1) pair 4-byte aligned), the A fragment is eight 32-bit
//             shared-memory loads at immediate offsets.  K = 30 padded to 32.
//   wgrad   : dW[oc][k] = sum over pixels gy[p][oc] * patch[p][k]: M = c2, N = 32 (k as above), K = pixels.  gy tiles staged in
//             shared memory, A = gy^T through ldmatrix.trans, B gathered from the same staged input rows; per-warp f32
//             accumulators over a persistent CTA's tiles, per-CTA partial matrices folded in a fixed order (deterministic).
// Tensor-core work is negligible (5.7 GFLOP); both kernels are bound by the one pass over the input and the output / gradient.
#include "common.cuh"

namespace b200 {
namespace {

constexpr int kR = 4;            // output rows per tile, forward (9 input rows staged)
constexpr int kRW = 2;           // output rows per tile, weight gradient: smaller tiles, 5 CTAs per SM -- the staging of one CTA
                                 // runs under the MMAs of the others (there is no double buffering inside a CTA)
constexpr int kPad = 16;         // zero bytes in front of every staged input row (x = -1 and the dummy slot of ox = 0)

template <typename T> struct Mma;
template <> struct Mma<__nv_bfloat16> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};
template <> struct Mma<__half> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    const __half2 p = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};

// k in [0, 32) -> byte offset of the element inside the staged rows relative to (tile row 2*orow, pixel ox = 0, x = 0):
// ky * pitch + 2 * (j - 4); k >= 30 (padding of K) reads a valid finite element (its weight / its dW column is zero / unused)
__device__ __forceinline__ int k_offset(int k, int pitch) {
  if (k >= 30) k = 28;
  const int ky = k / 10, j = k - ky * 10;
  return ky * pitch + 2 * (j - 4);
}
// weight of slot k for output channel n (w: [OC][3][3][3] f32, OIHW); j = 0 and k >= 30 are zero slots; j - 1 = kx * 3 + c
__device__ __forceinline__ float k_weight(const float* __restrict__ w, int n, int k) {
  if (k >= 30) return 0.f;
  const int ky = k / 10, j = k - ky * 10;
  if (j == 0) return 0.f;
  const int kx = (j - 1) / 3, c = (j - 1) - kx * 3;
  return w[((n * 3 + c) * 3 + ky) * 3 + kx];
}

// stage the kIR input rows of tile (b, oy0) : row i <-> input row 2*oy0 - 1 + i (zero outside the image)
template <typename T, int IR>
__device__ __forceinline__ void stage_input(unsigned char* xs, const T* __restrict__ x, int b, int oy0, int H, int W, int pitch) {
  // asynchronous copies: the whole tile is requested at once (register-staged batches of four loads were four DRAM round trips per
  // tile and left the kernels latency-bound at a third of the HBM rate); the caller waits with cp_async_wait_all + __syncthreads
  const int vpr = W * 6 / 16 + 1;   // + 1: the zero pad in front of the row (v == 0)
  const unsigned char* xb = reinterpret_cast<const unsigned char*>(x);
#pragma unroll
  for (int i = 0; i < IR; ++i) {   // row by row: no integer division per copy
    const int iy = 2 * oy0 - 1 + i;
    const bool row_ok = iy >= 0 && iy < H;
    const unsigned char* rsrc = xb + ((size_t)(b * H + (row_ok ? iy : 0)) * W) * 6;
    unsigned char* rdst = xs + (size_t)i * pitch;
    for (int v = threadIdx.x; v < vpr; v += blockDim.x) {
      const bool ok = row_ok && v > 0;
      cp_async16(rdst + (size_t)v * 16, ok ? rsrc + (size_t)(v - 1) * 16 : xb, ok);
    }
  }
}

template <typename T, int OC>
__global__ void __launch_bounds__(256) stem_fwd_kernel(const T* __restrict__ x, const float* __restrict__ w, T* __restrict__ y, int H, int W,
                                                       int Ho, int Wo, int tiles_per_img, int pitch) {
  extern __shared__ __align__(16) unsigned char xs[];
  constexpr int NT = OC / 8;
  const int b = blockIdx.x / tiles_per_img, oy0 = (blockIdx.x - b * tiles_per_img) * kR;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, q = lane & 3, r = lane >> 2;
  uint32_t bw[2][NT][2];
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k = 16 * s + 2 * q + 8 * h, n = nt * 8 + r;
        bw[s][nt][h] = Mma<T>::pack(k_weight(w, n, k), k_weight(w, n, k + 1));
      }
  int koff[2][2];
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int h = 0; h < 2; ++h) koff[s][h] = k_offset(16 * s + 2 * q + 8 * h, pitch);
  stage_input<T, 2 * kR + 1>(xs, x, b, oy0, H, W, pitch);
  cp_async_wait_all();
  __syncthreads();
  const int gpr = Wo / 16;   // 16-pixel groups per output row
  const int rows = min(kR, Ho - oy0);
  for (int g = warp; g < rows * gpr; g += (int)(blockDim.x >> 5)) {
    const int orow = g / gpr, ox0 = (g - orow * gpr) * 16;
    const unsigned char* base = xs + (size_t)(2 * orow) * pitch + kPad + 12 * (ox0 + r);
    float d[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) { d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f; }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      uint32_t a[4];
      a[0] = *reinterpret_cast<const uint32_t*>(base + koff[s][0]);
      a[1] = *reinterpret_cast<const uint32_t*>(base + koff[s][0] + 12 * 8);
      a[2] = *reinterpret_cast<const uint32_t*>(base + koff[s][1]);
      a[3] = *reinterpret_cast<const uint32_t*>(base + koff[s][1] + 12 * 8);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) Mma<T>::run(d[nt], a, bw[s][nt][0], bw[s][nt][1]);
    }
    T* yo = y + ((size_t)(b * Ho + oy0 + orow) * Wo + ox0 + r) * OC + 2 * q;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      *reinterpret_cast<uint32_t*>(yo + nt * 8) = Mma<T>::pack(d[nt][0], d[nt][1]);
      *reinterpret_cast<uint32_t*>(yo + (size_t)8 * OC + nt * 8) = Mma<T>::pack(d[nt][2], d[nt][3]);
    }
  }
}

template <typename T, int OC>
__global__ void __launch_bounds__(256) stem_wgrad_kernel(const T* __restrict__ gy, const T* __restrict__ x, float* __restrict__ part, int H,
                                                         int W, int Ho, int Wo, int tiles_per_img, int n_tiles, int pitch) {
  extern __shared__ __align__(16) unsigned char smem[];
  constexpr int MT = OC / 16;
  unsigned char* xs = smem;                                  // 2 * kRW + 1 input rows
  unsigned char* gs = smem + (size_t)(2 * kRW + 1) * pitch;   // kRW rows of gy: [kRW][Wo][OC]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, q = lane & 3, r = lane >> 2;
  const int gpr = Wo / 16;
  float acc[MT][4][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = acc[mt][nt][2] = acc[mt][nt][3] = 0.f;
  int koff[4];   // element offset of this lane's B column n = nt * 8 + r
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) koff[nt] = k_offset(nt * 8 + r, pitch);
  // ldmatrix row address of this lane inside a 16-pixel x 16-channel block of gy: matrices (pix 0-7 | 8-15) x (oc 0-7 | 8-15)
  const int lm_pix = (lane & 7) + ((lane & 16) ? 8 : 0), lm_oc = (lane & 8) ? 8 : 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_img, oy0 = (tile - b * tiles_per_img) * kRW;
    const int rows = min(kRW, Ho - oy0);
    __syncthreads();   // previous tile fully consumed
    stage_input<T, 2 * kRW + 1>(xs, x, b, oy0, H, W, pitch);
    {
      const int vecs = rows * Wo * OC * 2 / 16;
      const unsigned char* src = reinterpret_cast<const unsigned char*>(gy) + ((size_t)(b * Ho + oy0) * Wo) * OC * 2;
      for (int v = threadIdx.x; v < vecs; v += blockDim.x) cp_async16(gs + (size_t)v * 16, src + (size_t)v * 16, true);
    }
    cp_async_wait_all();
    __syncthreads();
    for (int g = warp; g < rows * gpr; g += (int)(blockDim.x >> 5)) {
      const int orow = g / gpr, ox0 = (g - orow * gpr) * 16;
      uint32_t a[MT][4];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const uint32_t addr = smem_u32(gs + ((size_t)(orow * Wo + ox0 + lm_pix) * OC + mt * 16 + lm_oc) * 2);
        // transposed 8x8 blocks: a0 = (oc 0-7, pix 0-7), a1 = (oc 8-15, pix 0-7), a2 = (oc 0-7, pix 8-15), a3 = (oc 8-15, pix 8-15)
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(a[mt][0]), "=r"(a[mt][1]), "=r"(a[mt][2]), "=r"(a[mt][3]) : "r"(addr));
      }
      const unsigned char* base = xs + (size_t)(2 * orow) * pitch + kPad + 12 * ox0;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const unsigned char* p = base + koff[nt] + 12 * (2 * q);
        const uint32_t e0 = *reinterpret_cast<const unsigned short*>(p), e1 = *reinterpret_cast<const unsigned short*>(p + 12);
        const uint32_t e8 = *reinterpret_cast<const unsigned short*>(p + 12 * 8), e9 = *reinterpret_cast<const unsigned short*>(p + 12 * 9);
        const uint32_t b0 = e0 | (e1 << 16), b1 = e8 | (e9 << 16);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) Mma<T>::run(acc[mt][nt], a[mt], b0, b1);
      }
    }
  }
  // fold the warps' accumulators in a fixed order, one partial [OC][32] matrix per CTA
  __syncthreads();
  float* red = reinterpret_cast<float*>(smem);   // [8 warps][OC * 32]
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      float* o = red + (size_t)warp * OC * 32;
      o[(mt * 16 + r) * 32 + nt * 8 + 2 * q] = acc[mt][nt][0];
      o[(mt * 16 + r) * 32 + nt * 8 + 2 * q + 1] = acc[mt][nt][1];
      o[(mt * 16 + r + 8) * 32 + nt * 8 + 2 * q] = acc[mt][nt][2];
      o[(mt * 16 + r + 8) * 32 + nt * 8 + 2 * q + 1] = acc[mt][nt][3];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < OC * 32; i += blockDim.x) {
    float s = 0.f;
    for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) s += red[(size_t)wv * OC * 32 + i];
    part[(size_t)blockIdx.x * OC * 32 + i] = s;
  }
}

// dW[oc][c][ky][kx] = sum over CTAs of part[cta][oc][10 * ky + 1 + 3 * kx + c]: one warp per element, lanes stride over the CTAs
// (independent loads; one thread walking all partials was a 100 us chain of L2 latencies), fixed-order butterfly: deterministic
__global__ void __launch_bounds__(256) stem_wgrad_fold_kernel(const float* __restrict__ part, int n_part, int OC, float* __restrict__ gw) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= OC * 27) return;
  const int oc = i / 27, rem = i - oc * 27, c = rem / 9, ky = (rem - c * 9) / 3, kx = rem - c * 9 - ky * 3;
  const int col = 10 * ky + 1 + 3 * kx + c;
  float s = 0.f;
  for (int p = lane; p < n_part; p += 32) s += part[((size_t)p * OC + oc) * 32 + col];
  s = warp_sum(s);
  if (lane == 0) gw[i] = s;
}

int check_stem(int B, int H, int W, int OC, int dtype, const void* a, const void* b, const void* c) {
  B200_REQUIRE(a && b && c, B200_ERR_SHAPE, "stem_conv: null pointer");
  B200_REQUIRE(dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "stem_conv: 16-bit activations only (dtype %d)", dtype);
  B200_REQUIRE(OC == 16 || OC == 32 || OC == 48, B200_ERR_UNSUPPORTED, "stem_conv: c2 must be 16, 32 or 48 (got %d)", OC);
  B200_REQUIRE(B > 0 && H > 0 && W > 0 && H % 2 == 0 && W % 32 == 0, B200_ERR_SHAPE,
               "stem_conv: H even and W a multiple of 32 required (H=%d W=%d)", H, W);
  B200_REQUIRE((((uintptr_t)a | (uintptr_t)c) & 15) == 0, B200_ERR_ALIGN, "stem_conv: tensors must be 16-byte aligned");
  return B200_OK;
}
int stem_pitch(int W) { return kPad + W * 6; }   // W % 8 == 0: a multiple of 16 bytes

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_stem_conv_supported(int32_t H, int32_t W, int32_t c2, int32_t dtype) {
  return (dtype == B200_BF16 || dtype == B200_F16) && (c2 == 16 || c2 == 32 || c2 == 48) && H > 0 && W > 0 && H % 2 == 0 && W % 32 == 0 &&
         (size_t)(2 * kR + 1) * stem_pitch(W) <= (size_t)max_smem_optin();
}

extern "C" B200_API int b200_stem_conv_fwd(const void* x, const float* w, void* y, int32_t B, int32_t H, int32_t W, int32_t c2, int32_t dtype,
                                           void* stream) {
  if (int rc = check_stem(B, H, W, c2, dtype, x, w, y)) return rc;
  const int Ho = H / 2, Wo = W / 2, tpi = (Ho + kR - 1) / kR, pitch = stem_pitch(W);
  const size_t smem = (size_t)(2 * kR + 1) * pitch;
  B200_REQUIRE(smem <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "stem_conv_fwd: W=%d does not fit in shared memory", W);
  cudaStream_t st = (cudaStream_t)stream;
#define B200_STEM_FWD(TT, OCC)                                                                                 \
  {                                                                                                            \
    auto kern = stem_fwd_kernel<TT, OCC>;                                                                      \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                        \
    kern<<<B * tpi, 256, smem, st>>>((const TT*)x, w, (TT*)y, H, W, Ho, Wo, tpi, pitch);                       \
  }
  if (dtype == B200_BF16) {
    if (c2 == 16) B200_STEM_FWD(__nv_bfloat16, 16) else if (c2 == 32) B200_STEM_FWD(__nv_bfloat16, 32) else B200_STEM_FWD(__nv_bfloat16, 48)
  } else {
    if (c2 == 16) B200_STEM_FWD(__half, 16) else if (c2 == 32) B200_STEM_FWD(__half, 32) else B200_STEM_FWD(__half, 48)
  }
#undef B200_STEM_FWD
  return check_launch("stem_conv_fwd");
}

extern "C" B200_API size_t b200_stem_conv_wgrad_workspace_bytes(int32_t c2) { return (size_t)(sm_count() * 5) * c2 * 32 * sizeof(float); }

extern "C" B200_API int b200_stem_conv_wgrad(const void* gy, const void* x, float* gw, void* workspace, size_t workspace_bytes, int32_t B,
                                             int32_t H, int32_t W, int32_t c2, int32_t dtype, void* stream) {
  if (int rc = check_stem(B, H, W, c2, dtype, gy, gw, x)) return rc;
  B200_REQUIRE(workspace && workspace_bytes >= b200_stem_conv_wgrad_workspace_bytes(c2), B200_ERR_WORKSPACE, "stem_conv_wgrad: workspace too small");
  const int Ho = H / 2, Wo = W / 2, tpi = (Ho + kRW - 1) / kRW, pitch = stem_pitch(W), n_tiles = B * tpi;
  const size_t smem_in = (size_t)(2 * kRW + 1) * pitch + (size_t)kRW * Wo * c2 * 2, smem_red = (size_t)8 * c2 * 32 * 4;
  const size_t smem = smem_in > smem_red ? smem_in : smem_red;
  B200_REQUIRE(smem <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "stem_conv_wgrad: W=%d does not fit in shared memory", W);
  int grid = 0;
  float* part = (float*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  // persistent CTAs: exactly one resident wave (the occupancy query accounts for registers as well as shared memory)
#define B200_STEM_WG(TT, OCC)                                                                                  \
  {                                                                                                            \
    auto kern = stem_wgrad_kernel<TT, OCC>;                                                                    \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                        \
    int per_sm = 1;                                                                                            \
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);                                   \
    per_sm = per_sm < 1 ? 1 : per_sm > 5 ? 5 : per_sm;                                                         \
    grid = sm_count() * per_sm;                                                                                \
    if (grid > n_tiles) grid = n_tiles;                                                                        \
    kern<<<grid, 256, smem, st>>>((const TT*)gy, (const TT*)x, part, H, W, Ho, Wo, tpi, n_tiles, pitch);       \
  }
  if (dtype == B200_BF16) {
    if (c2 == 16) B200_STEM_WG(__nv_bfloat16, 16) else if (c2 == 32) B200_STEM_WG(__nv_bfloat16, 32) else B200_STEM_WG(__nv_bfloat16, 48)
  } else {
    if (c2 == 16) B200_STEM_WG(__half, 16) else if (c2 == 32) B200_STEM_WG(__half, 32) else B200_STEM_WG(__half, 48)
  }
#undef B200_STEM_WG
  if (int rc = check_launch("stem_conv_wgrad")) return rc;
  stem_wgrad_fold_kernel<<<(c2 * 27 * 32 + 255) / 256, 256, 0, st>>>(part, grid, c2, gw);
  return check_launch("stem_conv_wgrad_fold");
}
