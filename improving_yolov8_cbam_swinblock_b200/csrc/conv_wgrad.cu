// Weight gradient of the narrow 3x3 convolutions at the top of the model (yaml backbone rows 1-4: Conv / C2f bottlenecks with 16 or
// 32 input channels; conv.py:37-91 `self.conv`, autograd of F.conv2d w.r.t. the weight).  For these widths cuDNN falls back to sm80
// legacy wgrad kernels (launch list of round 2: 8 launches, 1.5 ms per step, 3-20 x their HBM time).  Here, per tap (ky, kx):
//   dW[oc][c][ky][kx] = sum over output pixels p of gy[p][oc] * x[s*p + (ky, kx) - 1][c]
// is an [OC x CIN x pixels] product on mma.sync m16n8k16 with BOTH operands read by ldmatrix.trans from tiles staged once per CTA
// in shared memory: gy rows [pixel][oc] transposed give A = gy^T, the NHWC input rows [pixel][c] (a zero pixel of padding on both
// sides, zero rows outside the image: no bounds checks) transposed give B; a stride-2 convolution only changes the row addresses.
// CTA = 9 warps, warp t owns tap t for every 16-pixel group of the tile, so its accumulators ARE the tap's [OC x CIN] matrix: no
// cross-warp reduction; persistent CTAs write one partial matrix per tap, folded in a fixed order (deterministic).
#include "common.cuh"

namespace b200 {
namespace {

template <typename T> struct MmaW;
template <> struct MmaW<__nv_bfloat16> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};
template <> struct MmaW<__half> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
};
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

template <int S> struct TileRows { static constexpr int R = S == 1 ? 4 : 2, IR = S * (R - 1) + 3; };
// Warp layout.  With 16 input channels a 16-pixel group is 2 MMAs per tap and 16 output channels: walking it once per tap (one tap
// per warp, the first version) cost ~70 instructions of loop / address work for 2 MMAs and ran at a tenth of the HBM rate.  A warp
// therefore keeps TPW taps' accumulators and reuses the A fragments: OC = 16: all 9 taps (72 accumulator registers), 8 warps split
// the pixel groups; OC = 32: one kernel row (3 taps, 48 registers), 3 x 3 warps.  Warps that share a tap set are folded at the end
// of the kernel in a fixed order through one shared-memory copy of the result.
template <int OC> struct WarpPlan { static constexpr int TPW = OC == 16 ? 9 : 3, TS = 9 / TPW, PS = OC == 16 ? 8 : 3, NW = TS * PS; };
constexpr int kCin = 16;

template <typename T, int OC, int S>
__global__ void __launch_bounds__(WarpPlan<OC>::NW * 32, 2) conv3_wgrad_kernel(const T* __restrict__ gy, const T* __restrict__ x,
                                                                                float* __restrict__ part, int H, int W, int Ho, int Wo,
                                                                                int tiles_per_img, int n_tiles) {
  using WP = WarpPlan<OC>;
  constexpr int R = TileRows<S>::R, IR = TileRows<S>::IR, MT = OC / 16, NT = kCin / 8, PB = kCin * 2, NTH = WP::NW * 32, TPW = WP::TPW;
  // shared-memory pixel pitches: 16 bytes of padding per pixel, so that the eight 16-byte rows of an ldmatrix tile (consecutive pixels,
  // or every second one at stride 2) fall into different banks -- at the dense pitches (32 / 64 bytes) every ldmatrix was a 2- to 4-way
  // bank conflict and ncu showed the kernel waiting on shared memory (short_scoreboard 5-8 warps per issue)
  constexpr int PBP = PB + 16, GP = OC * 2 + 16;
  extern __shared__ __align__(16) unsigned char smem[];
  const int pitch = (W + 2) * PBP;
  unsigned char* xs = smem;                          // IR input rows: [zero pixel | W pixels | zero pixel] x 16 channels
  unsigned char* gs = smem + (size_t)IR * pitch;     // R rows of gy: [R][Wo][GP bytes]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, q = lane & 3, r = lane >> 2;
  const int ts = warp % WP::TS, ps = warp / WP::TS;  // tap set, pixel-group split
  const int lm_pix = (lane & 7) + ((lane & 16) ? 8 : 0), lm_c = (lane & 8) ? 8 : 0;
  const int gpr = Wo / 16;
  float acc[TPW][MT][NT][4];
#pragma unroll
  for (int t = 0; t < TPW; ++t)
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) acc[t][mt][nt][0] = acc[t][mt][nt][1] = acc[t][mt][nt][2] = acc[t][mt][nt][3] = 0.f;
  const int vpr = (W + 2) * (PB / 16), vpp = PB / 16;   // 16-byte chunks of data per staged input row / per pixel
  const uint32_t xs_lane = smem_u32(xs) + (uint32_t)(S * lm_pix * PBP + lm_c * 2);
  const uint32_t gs_lane = smem_u32(gs) + (uint32_t)(lm_pix * GP + lm_c * 2);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_img, oy0 = (tile - b * tiles_per_img) * R;
    const int rows = min(R, Ho - oy0);
    __syncthreads();   // previous tile fully consumed
    {  // the whole tile as asynchronous 16-byte copies (zero-filled pads / rows outside the image), one wait
      const unsigned char* xb = reinterpret_cast<const unsigned char*>(x);
#pragma unroll
      for (int i = 0; i < IR; ++i) {   // row by row: no integer division per copy (it made the staging as many instructions as the MMAs)
        const int iy = S * oy0 - 1 + i;
        const bool row_ok = iy >= 0 && iy < H;
        const unsigned char* rsrc = xb + ((size_t)(b * H + (row_ok ? iy : 0)) * W) * PB;
        unsigned char* rdst = xs + (size_t)i * pitch;
        for (int v = threadIdx.x; v < vpr; v += NTH) {
          const bool ok = row_ok && v >= vpp && v < vpr - vpp;
          const int px = v / vpp, ch = v - px * vpp;   // vpp is a power of two (kCin = 16: 2)
          cp_async16(rdst + (size_t)px * PBP + ch * 16, ok ? rsrc + (size_t)(v - vpp) * 16 : xb, ok);
        }
      }
      const int vecs = rows * Wo * OC * 2 / 16;
      const unsigned char* src = reinterpret_cast<const unsigned char*>(gy) + ((size_t)(b * Ho + oy0) * Wo) * OC * 2;
      constexpr int cpp = OC * 2 / 16;   // 16-byte chunks per gy pixel
      for (int v = threadIdx.x; v < vecs; v += NTH) cp_async16(gs + (size_t)(v / cpp) * GP + (v % cpp) * 16, src + (size_t)v * 16, true);
      cp_async_wait_all();
    }
    __syncthreads();
    int orow = 0, og = ps;
    while (og >= gpr) { og -= gpr; ++orow; }
    while (orow < rows) {
      const int ox0 = og * 16;
      uint32_t a[MT][4];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)   // a0 = (oc 0-7, pix 0-7), a1 = (oc 8-15, pix 0-7), a2 = (oc 0-7, pix 8-15), a3 = (oc 8-15, pix 8-15)
        ldsm_x4_t(a[mt], gs_lane + (uint32_t)((orow * Wo + ox0) * GP + mt * 32));
      const uint32_t xg = xs_lane + (uint32_t)(S * orow * pitch + S * ox0 * PBP);
#pragma unroll
      for (int t = 0; t < TPW; ++t) {
        const int tap = ts * TPW + t, ky = tap / 3, kx = tap - ky * 3;
        uint32_t bb[4];   // b0(c 0-7), b0(c 8-15), b1(c 0-7), b1(c 8-15)
        ldsm_x4_t(bb, xg + (uint32_t)(ky * pitch + kx * PBP));
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          MmaW<T>::run(acc[t][mt][0], a[mt], bb[0], bb[2]);
          MmaW<T>::run(acc[t][mt][1], a[mt], bb[1], bb[3]);
        }
      }
      og += WP::PS;
      while (og >= gpr) { og -= gpr; ++orow; }
    }
  }
  // fold the pixel splits of every tap set in a fixed order (split 0 stores, 1 .. PS-1 add), then one partial per CTA
  __syncthreads();
  float* red = reinterpret_cast<float*>(smem);   // [9][OC][16]
  for (int turn = 0; turn < WP::PS; ++turn) {
    if (ps == turn) {
#pragma unroll
      for (int t = 0; t < TPW; ++t)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int nt = 0; nt < NT; ++nt) {
            float* o = red + ((size_t)(ts * TPW + t) * OC + mt * 16 + r) * kCin + nt * 8 + 2 * q;
            float2 lo = make_float2(acc[t][mt][nt][0], acc[t][mt][nt][1]), hi = make_float2(acc[t][mt][nt][2], acc[t][mt][nt][3]);
            if (turn) {
              const float2 l0 = *reinterpret_cast<float2*>(o), h0 = *reinterpret_cast<float2*>(o + 8 * kCin);
              lo.x += l0.x; lo.y += l0.y; hi.x += h0.x; hi.y += h0.y;
            }
            *reinterpret_cast<float2*>(o) = lo;
            *reinterpret_cast<float2*>(o + 8 * kCin) = hi;
          }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 9 * OC * kCin; i += NTH) part[(size_t)blockIdx.x * 9 * OC * kCin + i] = red[i];
}

// gw[oc][c][ky][kx] = sum over CTAs of part[cta][ky * 3 + kx][oc][c]; warp per element, fixed-order butterfly
__global__ void __launch_bounds__(256) conv3_wgrad_fold_kernel(const float* __restrict__ part, int n_part, int OC, int CIN, float* __restrict__ gw) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= OC * CIN * 9) return;
  const int oc = i / (CIN * 9), rem = i - oc * CIN * 9, c = rem / 9, tap = rem - c * 9;
  float s = 0.f;
  for (int p = lane; p < n_part; p += 32) s += part[(((size_t)p * 9 + tap) * OC + oc) * CIN + c];
  s = warp_sum(s);
  if (lane == 0) gw[i] = s;
}

bool wgrad_shape_ok(int H, int W, int cin, int oc, int stride, int dtype) {
  // 32 input channels and more: cuDNN's sm100 wgrad kernels are the faster ones (measured: 76 vs 99 us at [64,32,80,80]); they stay
  if (!(dtype == B200_BF16 || dtype == B200_F16) || cin != kCin || !(oc == 16 || oc == 32) || !(stride == 1 || stride == 2)) return false;
  if (H <= 0 || W <= 0 || (stride == 2 && ((H | W) & 1))) return false;
  const int Wo = W / stride;
  const int R = stride == 1 ? 4 : 2, IR = stride * (R - 1) + 3;
  const size_t smem = (size_t)IR * (W + 2) * (cin * 2 + 16) + (size_t)R * Wo * (oc * 2 + 16);
  return Wo % 16 == 0 && smem <= (size_t)max_smem_optin();
}

template <typename T, int OC, int S>
int launch_wgrad(const void* gy, const void* x, float* gw, float* part, int n_ctas_max, int B, int H, int W, cudaStream_t st) {
  constexpr int R = TileRows<S>::R, IR = TileRows<S>::IR, NTH = WarpPlan<OC>::NW * 32;
  const int Ho = H / S, Wo = W / S, tpi = (Ho + R - 1) / R, n_tiles = B * tpi;
  const size_t smem_tile = (size_t)IR * (W + 2) * (kCin * 2 + 16) + (size_t)R * Wo * (OC * 2 + 16), smem_red = (size_t)9 * OC * kCin * 4;
  const size_t smem = smem_tile > smem_red ? smem_tile : smem_red;
  auto kern = conv3_wgrad_kernel<T, OC, S>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  // persistent CTAs: exactly one resident wave (the occupancy query accounts for registers as well as shared memory)
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NTH, smem);
  per_sm = per_sm < 1 ? 1 : per_sm > 4 ? 4 : per_sm;
  int grid = sm_count() * per_sm;
  if (grid > n_tiles) grid = n_tiles;
  if (grid > n_ctas_max) grid = n_ctas_max;
  kern<<<grid, NTH, smem, st>>>((const T*)gy, (const T*)x, part, H, W, Ho, Wo, tpi, n_tiles);
  if (int rc = check_launch("conv3x3_wgrad")) return rc;
  conv3_wgrad_fold_kernel<<<(OC * kCin * 9 * 32 + 255) / 256, 256, 0, st>>>(part, grid, OC, kCin, gw);
  return check_launch("conv3x3_wgrad_fold");
}

template <typename T>
int launch_any(int oc, int stride, const void* gy, const void* x, float* gw, float* part, int nmax, int B, int H, int W, cudaStream_t st) {
  if (oc == 16) return stride == 1 ? launch_wgrad<T, 16, 1>(gy, x, gw, part, nmax, B, H, W, st) : launch_wgrad<T, 16, 2>(gy, x, gw, part, nmax, B, H, W, st);
  return stride == 1 ? launch_wgrad<T, 32, 1>(gy, x, gw, part, nmax, B, H, W, st) : launch_wgrad<T, 32, 2>(gy, x, gw, part, nmax, B, H, W, st);
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_conv3x3_wgrad_supported(int32_t H, int32_t W, int32_t cin, int32_t cout, int32_t stride, int32_t dtype) {
  return wgrad_shape_ok(H, W, cin, cout, stride, dtype) ? 1 : 0;
}
extern "C" B200_API size_t b200_conv3x3_wgrad_workspace_bytes(int32_t cin, int32_t cout) {
  return (size_t)(sm_count() * 4) * 9 * cin * cout * sizeof(float);
}
extern "C" B200_API int b200_conv3x3_wgrad(const void* gy, const void* x, float* gw, void* workspace, size_t workspace_bytes, int32_t B, int32_t H,
                                           int32_t W, int32_t cin, int32_t cout, int32_t stride, int32_t dtype, void* stream) {
  B200_REQUIRE(gy && x && gw && workspace, B200_ERR_SHAPE, "conv3x3_wgrad: null pointer");
  B200_REQUIRE(B > 0 && wgrad_shape_ok(H, W, cin, cout, stride, dtype), B200_ERR_UNSUPPORTED,
               "conv3x3_wgrad: unsupported shape H=%d W=%d cin=%d cout=%d stride=%d dtype=%d", H, W, cin, cout, stride, dtype);
  B200_REQUIRE((((uintptr_t)gy | (uintptr_t)x) & 15) == 0, B200_ERR_ALIGN, "conv3x3_wgrad: tensors must be 16-byte aligned");
  const size_t per = (size_t)9 * cin * cout * sizeof(float);
  B200_REQUIRE(workspace_bytes >= per, B200_ERR_WORKSPACE, "conv3x3_wgrad: workspace too small");
  const int nmax = (int)(workspace_bytes / per);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_BF16) return launch_any<__nv_bfloat16>(cout, stride, gy, x, gw, (float*)workspace, nmax, B, H, W, st);
  return launch_any<__half>(cout, stride, gy, x, gw, (float*)workspace, nmax, B, H, W, st);
}
