// Channel concat of NHWC (channels_last) maps: the seam either side of the blocks (SURVEY 8(f)-2: `C2f` chunk/cat,
// `Concat`, the Detect head's cat -- block.py C2f.forward, conv.py Concat.forward, head.py:66-76).
//
// Every source is a row-strided view `[rows = B*H*W, C_i]` (row stride S_i >= C_i elements: a channel slice of a wider
// channels_last tensor qualifies, which is what `chunk(2, 1)` and the gradient of a concat hand over), the destination is
// dense `[rows, sum C_i]`.  One thread moves one 16-byte vector; four independent vectors in flight per thread.  ATen's
// CatArrayBatchedCopy treats channels_last inputs as generic strided tensors and reaches ~15 % of the copy roofline on
// these shapes; this is a plain vectorised copy.
#include "common.cuh"

namespace b200 {
namespace {

constexpr int kMaxSrc = 8;
constexpr int kT = 256;
constexpr int kInFlight = 4;

struct FastDiv {   // exact 32-bit division by a run-time constant (multiply-high + shifts)
  uint32_t d, m, s1, s2;
  void init(uint32_t div) {
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

struct CatParams {
  const unsigned char* src[kMaxSrc];
  long long stride[kMaxSrc];   // source row stride in bytes
  uint32_t first[kMaxSrc + 1]; // first unit (16-byte vector or element) of source i inside a destination row
  unsigned char* dst;
  uint32_t n, upr;             // sources, units per destination row
  uint32_t items;              // rows * upr
  FastDiv dupr;
};

template <typename V>   // V = uint4 (16-byte vectors) or a 2/4-byte scalar
__global__ void __launch_bounds__(kT) nhwc_concat_kernel(const __grid_constant__ CatParams P) {
  const uint32_t step = gridDim.x * kT;
  for (uint32_t i0 = blockIdx.x * kT + threadIdx.x; i0 < P.items; i0 += kInFlight * step) {
    V v[kInFlight];
#pragma unroll
    for (int u = 0; u < kInFlight; ++u) {
      const uint32_t i = i0 + u * step;
      if (i < P.items) {
        const uint32_t row = P.dupr.div(i), col = i - row * P.upr;
        uint32_t j = 0;
#pragma unroll
        for (int k = 1; k < kMaxSrc; ++k) j += (k < (int)P.n && col >= P.first[k]) ? 1u : 0u;
        v[u] = *reinterpret_cast<const V*>(P.src[j] + (long long)row * P.stride[j] + (size_t)(col - P.first[j]) * sizeof(V));
      }
    }
#pragma unroll
    for (int u = 0; u < kInFlight; ++u) {
      const uint32_t i = i0 + u * step;
      if (i < P.items) *reinterpret_cast<V*>(P.dst + (size_t)i * sizeof(V)) = v[u];
    }
  }
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_nhwc_concat(const void* const* srcs, const int32_t* src_channels, const int64_t* src_row_stride,
                                         int32_t n_src, void* dst, int64_t rows, int32_t dtype, void* stream) {
  B200_REQUIRE(srcs && src_channels && src_row_stride && dst, B200_ERR_SHAPE, "nhwc_concat: null pointer");
  B200_REQUIRE(n_src >= 1 && n_src <= kMaxSrc, B200_ERR_UNSUPPORTED, "nhwc_concat: %d sources (1..%d supported)", n_src, kMaxSrc);
  B200_REQUIRE(dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "nhwc_concat: unsupported dtype code %d", dtype);
  B200_REQUIRE(rows > 0, B200_ERR_SHAPE, "nhwc_concat: rows=%lld", (long long)rows);
  const int es = dtype == B200_F32 ? 4 : 2;
  long long ctot = 0;
  bool vec = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
  for (int i = 0; i < n_src; ++i) {
    B200_REQUIRE(srcs[i] && src_channels[i] > 0 && src_row_stride[i] >= src_channels[i], B200_ERR_SHAPE,
                 "nhwc_concat: source %d: channels=%d row stride=%lld", i, src_channels[i], (long long)src_row_stride[i]);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(srcs[i]) & (es - 1)) == 0, B200_ERR_ALIGN, "nhwc_concat: source %d is not element-aligned", i);
    ctot += src_channels[i];
    vec = vec && (reinterpret_cast<uintptr_t>(srcs[i]) & 15) == 0 && ((long long)src_channels[i] * es) % 16 == 0 &&
          ((long long)src_row_stride[i] * es) % 16 == 0;
  }
  const int unit = vec ? 16 : es;
  const long long upr = ctot * es / unit;
  B200_REQUIRE(rows * upr < (1ll << 31), B200_ERR_UNSUPPORTED, "nhwc_concat: %lld x %lld units exceed the 31-bit item range",
               (long long)rows, upr);
  CatParams P;
  uint32_t first = 0;
  for (int i = 0; i < kMaxSrc; ++i) {
    const int k = i < n_src ? i : n_src - 1;
    P.src[i] = static_cast<const unsigned char*>(srcs[k]);
    P.stride[i] = (long long)src_row_stride[k] * es;
    P.first[i] = first;
    if (i < n_src) first += (uint32_t)((long long)src_channels[i] * es / unit);
  }
  P.first[kMaxSrc] = first;
  P.dst = static_cast<unsigned char*>(dst);
  P.n = (uint32_t)n_src; P.upr = (uint32_t)upr; P.items = (uint32_t)(rows * upr);
  P.dupr.init((uint32_t)upr);
  long long blocks = ((long long)P.items + (long long)kT * kInFlight - 1) / ((long long)kT * kInFlight);
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cudaStream_t st = (cudaStream_t)stream;
  if (vec) nhwc_concat_kernel<uint4><<<(unsigned)blocks, kT, 0, st>>>(P);
  else if (es == 4) nhwc_concat_kernel<uint32_t><<<(unsigned)blocks, kT, 0, st>>>(P);
  else nhwc_concat_kernel<uint16_t><<<(unsigned)blocks, kT, 0, st>>>(P);
  return check_launch("nhwc_concat");
}

// ---------------------------------------------------------------------------------------------------------
// Gradient fan-in at the seams: a feature map with several consumers (a bottleneck output inside `C2f` feeds the next
// bottleneck AND the concat -- block.py C2f.forward `y.extend(m(y[-1]) for m in self.m)`; a saved layer `y[j]` of
// `_predict_once`, tasks.py:171-176, feeds the next layer AND a later `Concat`) receives one gradient per consumer and
// autograd sums them.  One of them is a channel slice of a concat's gradient (a row-strided view), which sends ATen's add
// down its generic strided path (one element per thread, ~2 TB/s).  Here: 2..4 row-strided `[rows, C]` sources of one
// dtype -> dense `[rows, C]`, 16-byte vectors, summed in f32 in source order and rounded once (for two sources that is
// exactly ATen's `a + b` on 16-bit tensors).
// ---------------------------------------------------------------------------------------------------------
namespace b200 {
namespace {

constexpr int kMaxAdd = 4;
struct AddParams {
  const unsigned char* src[kMaxAdd];
  long long stride[kMaxAdd];   // source row stride in bytes
  unsigned char* dst;
  uint32_t n, upr, items;      // sources, 16-byte vectors per row, rows * upr
  FastDiv dupr;
};

template <typename T> __device__ __forceinline__ void add_unpack(const uint4& r, float* v) {
  if constexpr (sizeof(T) == 4) {
    v[0] = __uint_as_float(r.x); v[1] = __uint_as_float(r.y); v[2] = __uint_as_float(r.z); v[3] = __uint_as_float(r.w);
  } else {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (sizeof(T) == 2 && DT<T>::code == B200_BF16) {
        v[2 * i] = __uint_as_float(w[i] << 16); v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
      } else {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
      }
    }
  }
}
template <typename T> __device__ __forceinline__ uint4 add_pack(const float* v) {
  if constexpr (sizeof(T) == 4) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  } else {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (DT<T>::code == B200_BF16) {
        const __nv_bfloat162 p = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&p);
      } else {
        const __half2 p = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        w[i] = *reinterpret_cast<const uint32_t*>(&p);
      }
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
}

template <typename T, int N>
__global__ void __launch_bounds__(kT) nhwc_add_kernel(const __grid_constant__ AddParams P) {
  constexpr int VW = 16 / (int)sizeof(T);
  constexpr int U = N <= 2 ? 4 : 2;   // vectors in flight per thread and source
  const uint32_t step = gridDim.x * kT;
  for (uint32_t i0 = blockIdx.x * kT + threadIdx.x; i0 < P.items; i0 += U * step) {
    uint4 raw[U][N];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t i = i0 + u * step;
      if (i < P.items) {
        const uint32_t row = P.dupr.div(i), col = i - row * P.upr;
#pragma unroll
        for (int k = 0; k < N; ++k) raw[u][k] = ldg_stream16(P.src[k] + (long long)row * P.stride[k] + (size_t)col * 16);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t i = i0 + u * step;
      if (i < P.items) {
        float acc[VW], v[VW];
        add_unpack<T>(raw[u][0], acc);
#pragma unroll
        for (int k = 1; k < N; ++k) {
          add_unpack<T>(raw[u][k], v);
#pragma unroll
          for (int e = 0; e < VW; ++e) acc[e] += v[e];
        }
        stg_stream16(P.dst + (size_t)i * 16, add_pack<T>(acc));
      }
    }
  }
}

}  // namespace
}  // namespace b200

extern "C" B200_API int b200_nhwc_add(const void* const* srcs, const int64_t* src_row_stride, int32_t n_src, void* dst, int64_t rows,
                                      int32_t cols, int32_t dtype, void* stream) {
  B200_REQUIRE(srcs && src_row_stride && dst, B200_ERR_SHAPE, "nhwc_add: null pointer");
  B200_REQUIRE(n_src >= 2 && n_src <= kMaxAdd, B200_ERR_UNSUPPORTED, "nhwc_add: %d sources (2..%d supported)", n_src, kMaxAdd);
  B200_REQUIRE(dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "nhwc_add: unsupported dtype code %d", dtype);
  B200_REQUIRE(rows > 0 && cols > 0, B200_ERR_SHAPE, "nhwc_add: rows=%lld cols=%d", (long long)rows, cols);
  const int es = dtype == B200_F32 ? 4 : 2;
  B200_REQUIRE(((long long)cols * es) % 16 == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0, B200_ERR_ALIGN,
               "nhwc_add: rows of %d elements / the destination are not 16-byte multiples", cols);
  AddParams P;
  for (int i = 0; i < kMaxAdd; ++i) {
    const int k = i < n_src ? i : n_src - 1;
    B200_REQUIRE(srcs[k] && src_row_stride[k] >= cols, B200_ERR_SHAPE, "nhwc_add: source %d: row stride %lld < %d", k,
                 (long long)src_row_stride[k], cols);
    B200_REQUIRE((reinterpret_cast<uintptr_t>(srcs[k]) & 15) == 0 && ((long long)src_row_stride[k] * es) % 16 == 0, B200_ERR_ALIGN,
                 "nhwc_add: source %d is not 16-byte aligned / strided", k);
    P.src[i] = static_cast<const unsigned char*>(srcs[k]);
    P.stride[i] = (long long)src_row_stride[k] * es;
  }
  const long long upr = (long long)cols * es / 16;
  B200_REQUIRE(rows * upr < (1ll << 31), B200_ERR_UNSUPPORTED, "nhwc_add: %lld x %lld vectors exceed the 31-bit item range",
               (long long)rows, upr);
  P.dst = static_cast<unsigned char*>(dst);
  P.n = (uint32_t)n_src; P.upr = (uint32_t)upr; P.items = (uint32_t)(rows * upr);
  P.dupr.init((uint32_t)upr);
  const int per = n_src <= 2 ? 4 : 2;
  long long blocks = ((long long)P.items + (long long)kT * per - 1) / ((long long)kT * per);
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  cudaStream_t st = (cudaStream_t)stream;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    if (n_src == 2) nhwc_add_kernel<T, 2><<<(unsigned)blocks, kT, 0, st>>>(P);
    else if (n_src == 3) nhwc_add_kernel<T, 3><<<(unsigned)blocks, kT, 0, st>>>(P);
    else nhwc_add_kernel<T, 4><<<(unsigned)blocks, kT, 0, st>>>(P);
    return check_launch("nhwc_add");
  });
}

// ---------------------------------------------------------------------------------------------------------
// Input seam: uint8 NCHW image batch -> scaled float NHWC in the compute dtype, one pass.  Replaces the trainer's
// `img.float() / 255` (detect/train.py:100) + channels_last conversion + autocast's cast of the first conv input
// (four full passes over a 315 MB fp32 tensor) by one read of the uint8 batch and one write of the 16-bit map.
// Bit-identical to that chain on the GPU: ATen's CUDA division by a host scalar multiplies by the f32 reciprocal
// (`a * (1 / b)`, BinaryDivTrueKernel.cu), so this does too, then one round-to-nearest-even conversion.
// ---------------------------------------------------------------------------------------------------------
namespace b200 {
namespace {

template <typename T, int CH>
__global__ void __launch_bounds__(256) u8_to_nhwc_kernel(const uint8_t* __restrict__ img, T* __restrict__ out, long long hw,
                                                         long long quads, float inv) {
  // thread = 4 consecutive pixels of one image: CH uchar4 loads (one per plane), 4*CH contiguous output elements
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += (long long)gridDim.x * blockDim.x) {
    const long long hq = hw / 4;
    const long long b = q / hq, p4 = q - b * hq;
    const uint8_t* src = img + (size_t)b * CH * hw + (size_t)p4 * 4;
    uchar4 v[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) v[c] = *reinterpret_cast<const uchar4*>(src + (size_t)c * hw);
    alignas(16) T o[4 * CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      o[0 * CH + c] = DT<T>::from_f((float)v[c].x * inv);
      o[1 * CH + c] = DT<T>::from_f((float)v[c].y * inv);
      o[2 * CH + c] = DT<T>::from_f((float)v[c].z * inv);
      o[3 * CH + c] = DT<T>::from_f((float)v[c].w * inv);
    }
    T* dst = out + ((size_t)b * hw + (size_t)p4 * 4) * CH;
    // 4*CH elements: 8-byte aligned for every CH when T is 16-bit (4*CH*2 bytes per thread), 16-byte for f32
    constexpr int WORDS = 4 * CH * (int)sizeof(T) / 8;
    const uint2* ow = reinterpret_cast<const uint2*>(o);
#pragma unroll
    for (int w = 0; w < WORDS; ++w) reinterpret_cast<uint2*>(dst)[w] = ow[w];
  }
}

template <typename T>
int launch_u8(const uint8_t* img, void* out, int B, int C, long long hw, float inv, cudaStream_t st) {
  const long long quads = (long long)B * hw / 4;
  long long blocks = (quads + 255) / 256;
  const long long cap = (long long)sm_count() * 32;
  if (blocks > cap) blocks = cap;
  switch (C) {
    case 1: u8_to_nhwc_kernel<T, 1><<<(unsigned)blocks, 256, 0, st>>>(img, (T*)out, hw, quads, inv); break;
    case 2: u8_to_nhwc_kernel<T, 2><<<(unsigned)blocks, 256, 0, st>>>(img, (T*)out, hw, quads, inv); break;
    case 3: u8_to_nhwc_kernel<T, 3><<<(unsigned)blocks, 256, 0, st>>>(img, (T*)out, hw, quads, inv); break;
    default: u8_to_nhwc_kernel<T, 4><<<(unsigned)blocks, 256, 0, st>>>(img, (T*)out, hw, quads, inv); break;
  }
  return check_launch("u8_to_nhwc");
}

}  // namespace
}  // namespace b200

extern "C" B200_API int b200_u8_to_nhwc(const void* img, void* out, int32_t B, int32_t C, int32_t H, int32_t W, float divisor,
                                        int32_t dtype, void* stream) {
  B200_REQUIRE(img && out, B200_ERR_SHAPE, "u8_to_nhwc: null pointer");
  B200_REQUIRE(B > 0 && C >= 1 && C <= 4 && H > 0 && W > 0, B200_ERR_SHAPE, "u8_to_nhwc: bad shape B=%d C=%d H=%d W=%d (1..4 channels)", B, C, H, W);
  const long long hw = (long long)H * W;
  B200_REQUIRE(hw % 4 == 0, B200_ERR_UNSUPPORTED, "u8_to_nhwc: H*W=%lld must be a multiple of 4", hw);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(img) & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, B200_ERR_ALIGN,
               "u8_to_nhwc: img must be 4-byte and out 16-byte aligned");
  B200_REQUIRE(divisor != 0.f, B200_ERR_SHAPE, "u8_to_nhwc: divisor is zero");
  cudaStream_t st = (cudaStream_t)stream;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int { return launch_u8<T>(static_cast<const uint8_t*>(img), out, B, C, hw, 1.0f / divisor, st); });
}

// ---------------------------------------------------------------------------------------------------------
// Nearest-neighbour up-sampling by integer factors on NHWC maps (the two `nn.Upsample(None, 2, "nearest")` rows of the
// yaml head) and its backward.  ATen's channels_last nearest kernels reach ~0.3 TB/s on these shapes; both directions
// are plain 16-byte vector moves (forward: one source vector feeds sh*sw outputs; backward: f32 sum of the sh*sw
// gradients of one input pixel, fixed order).  The backward reads a row-strided gradient (a concat slice) in place.
// ---------------------------------------------------------------------------------------------------------
namespace b200 {
namespace {

struct UpGeo {
  uint32_t vpp, OW, OH, W, H, sh, sw, items;
  long long gstride;   // backward: bytes between consecutive pixels of the incoming gradient
  FastDiv dvpp, dOW, dOH, dsh, dsw, dW, dH;
};

__global__ void __launch_bounds__(256) upsample_fwd_kernel(const uint4* __restrict__ x, uint4* __restrict__ out, const __grid_constant__ UpGeo G) {
  const uint32_t step = gridDim.x * 256;
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < G.items; i += step) {
    const uint32_t pix = G.dvpp.div(i), v = i - pix * G.vpp;
    const uint32_t t = G.dOW.div(pix), ox = pix - t * G.OW;
    const uint32_t b = G.dOH.div(t), oy = t - b * G.OH;
    const uint32_t iy = G.dsh.div(oy), ix = G.dsw.div(ox);
    out[i] = x[((size_t)(b * G.H + iy) * G.W + ix) * G.vpp + v];
  }
}

template <typename T>
__global__ void __launch_bounds__(256) upsample_bwd_kernel(const unsigned char* __restrict__ g, uint4* __restrict__ gin,
                                                           const __grid_constant__ UpGeo G) {
  constexpr int VW = 16 / (int)sizeof(T);
  const uint32_t step = gridDim.x * 256;
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < G.items; i += step) {
    const uint32_t pix = G.dvpp.div(i), v = i - pix * G.vpp;
    const uint32_t t = G.dW.div(pix), ix = pix - t * G.W;
    const uint32_t b = G.dH.div(t), iy = t - b * G.H;
    float acc[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) acc[e] = 0.f;
    for (uint32_t dy = 0; dy < G.sh; ++dy)
      for (uint32_t dx = 0; dx < G.sw; ++dx) {
        const size_t op = (size_t)(b * G.OH + iy * G.sh + dy) * G.OW + ix * G.sw + dx;
        const uint4 raw = *reinterpret_cast<const uint4*>(g + op * G.gstride + (size_t)v * 16);
        const T* e8 = reinterpret_cast<const T*>(&raw);
#pragma unroll
        for (int e = 0; e < VW; ++e) acc[e] += DT<T>::to_f(e8[e]);
      }
    alignas(16) T o[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) o[e] = DT<T>::from_f(acc[e]);
    gin[i] = *reinterpret_cast<const uint4*>(o);
  }
}

int up_geo(UpGeo& G, int B, int C, int H, int W, int sh, int sw, int dtype, bool backward, long long gstride_elems) {
  const int es = dtype == B200_F32 ? 4 : 2;
  B200_REQUIRE(dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16, B200_ERR_DTYPE, "nhwc_upsample: unsupported dtype code %d", dtype);
  B200_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && sh >= 1 && sw >= 1, B200_ERR_SHAPE, "nhwc_upsample: bad shape B=%d C=%d H=%d W=%d x%d x%d", B, C, H, W, sh, sw);
  B200_REQUIRE(((long long)C * es) % 16 == 0, B200_ERR_ALIGN, "nhwc_upsample: C=%d must span a multiple of 16 bytes", C);
  G.vpp = (uint32_t)((long long)C * es / 16);
  G.H = H; G.W = W; G.sh = sh; G.sw = sw; G.OH = H * sh; G.OW = W * sw;
  const long long items = (long long)B * (backward ? (long long)H * W : (long long)G.OH * G.OW) * G.vpp;
  B200_REQUIRE(items < (1ll << 31) && (long long)B * G.OH * G.OW * G.vpp < (1ll << 31), B200_ERR_UNSUPPORTED, "nhwc_upsample: tensor too large");
  G.items = (uint32_t)items;
  G.gstride = (gstride_elems > 0 ? gstride_elems : C) * es;
  B200_REQUIRE(G.gstride >= (long long)C * es && G.gstride % 16 == 0, B200_ERR_ALIGN, "nhwc_upsample: gradient row stride must be >= C and a multiple of 16 bytes");
  G.dvpp.init(G.vpp); G.dOW.init(G.OW); G.dOH.init(G.OH); G.dsh.init(sh); G.dsw.init(sw); G.dW.init(W); G.dH.init(H);
  return B200_OK;
}
unsigned up_blocks(uint32_t items) {
  long long blocks = ((long long)items + 255) / 256;
  const long long cap = (long long)sm_count() * 32;
  return (unsigned)(blocks > cap ? cap : blocks);
}

}  // namespace
}  // namespace b200

extern "C" B200_API int b200_nhwc_upsample_fwd(const void* x, void* out, int32_t B, int32_t C, int32_t H, int32_t W, int32_t sh,
                                               int32_t sw, int32_t dtype, void* stream) {
  B200_REQUIRE(x && out, B200_ERR_SHAPE, "nhwc_upsample_fwd: null pointer");
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0, B200_ERR_ALIGN, "nhwc_upsample_fwd: tensors must be 16-byte aligned");
  UpGeo G;
  if (int rc = up_geo(G, B, C, H, W, sh, sw, dtype, false, 0)) return rc;
  upsample_fwd_kernel<<<up_blocks(G.items), 256, 0, (cudaStream_t)stream>>>(static_cast<const uint4*>(x), static_cast<uint4*>(out), G);
  return check_launch("nhwc_upsample_fwd");
}

extern "C" B200_API int b200_nhwc_upsample_bwd(const void* gout, int64_t gout_row_stride, void* gin, int32_t B, int32_t C, int32_t H,
                                               int32_t W, int32_t sh, int32_t sw, int32_t dtype, void* stream) {
  B200_REQUIRE(gout && gin, B200_ERR_SHAPE, "nhwc_upsample_bwd: null pointer");
  B200_REQUIRE(((reinterpret_cast<uintptr_t>(gout) | reinterpret_cast<uintptr_t>(gin)) & 15) == 0, B200_ERR_ALIGN, "nhwc_upsample_bwd: tensors must be 16-byte aligned");
  UpGeo G;
  if (int rc = up_geo(G, B, C, H, W, sh, sw, dtype, true, gout_row_stride)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    upsample_bwd_kernel<T><<<up_blocks(G.items), 256, 0, st>>>(static_cast<const unsigned char*>(gout), static_cast<uint4*>(gin), G);
    return check_launch("nhwc_upsample_bwd");
  });
}
