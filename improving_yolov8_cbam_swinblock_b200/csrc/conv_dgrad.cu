// Input gradient of the narrow stride-2 3x3 convolution at the top of the model (yaml backbone row 1 at scale n:
// nn.Conv2d(16, 32, 3, 2, 1, bias=False); conv.py:37-91 `self.conv`, autograd of F.conv2d w.r.t. the input).  cuDNN runs its
// generic strided-dgrad kernel there: 0.38 ms for 52 MB in / 210 MB out, 8x the HBM time, the slowest single launch of the step.
//
//   gx[b, iy, ix, ci] = sum over (ky, kx, oc) with iy = 2*oy - 1 + ky, ix = 2*ox - 1 + kx of gy[b, oy, ox, oc] * w[oc, ci, ky, kx]
//
// The parity of (iy, ix) decides which taps contribute: for iy = 2*py + dy, ix = 2*px + dx
//   dy = 0: ky = 1 (oy = py)              dy = 1: ky = 0 (oy = py + 1), ky = 2 (oy = py)        -- the same in x --
// so the four parity classes are four small implicit GEMMs with 1, 2, 2 and 4 taps: [16 pixels x 32 oc] x [32 oc x 16 ci] per tap
// on mma.sync m16n8k16.  A = gy rows as stored (pixel-major, oc contiguous) read by ldmatrix from a tile staged once per CTA with
// cp.async (rows py .. py + R, one zero pixel past the row end, zero rows past the map: no bounds checks); B = the weight
// re-laid as [tap][ci][oc] in shared memory.  A warp owns 16 consecutive px of one py row = a 2 x 32 block of input pixels: its
// four accumulator sets are interleaved through a per-warp staging tile and leave as 16-byte stores of whole pixel rows.
// No atomics, every output element written exactly once: deterministic.
//
// Measured (profiles/README.md): the first version of this kernel and of the forward kernel below took 103-105 us whatever the tile
// height, the CTAs per SM (2 or 3) or the staging (single- or double-buffered cp.async).  ncu named the limiter: the shared-memory
// pipe (stall reasons mio_throttle / short_scoreboard in front; HMMA at 26 % of its rate, DRAM at 30 %, 0.24 instructions issued per
// cycle and scheduler) -- 26 ldmatrix per 36 MMAs, 18 of them re-reading the weight fragments.  With the weights of 7 of the 9 taps
// resident in registers and one parity class accumulated at a time: 105 -> 86 us (forward: 6 taps resident, 102 -> 93 us).
#include <type_traits>

#include "common.cuh"

namespace b200 {
namespace {

constexpr int kCi = 16, kOc = 32, kR = 4, kWarps = 8, kThreads = kWarps * 32;
constexpr int kGP = 80;    // bytes per gy pixel in shared memory: 64 of data + 16 of padding (ldmatrix rows hit distinct banks)
constexpr int kWP = 80;    // bytes per (tap, ci) weight row: 32 oc + padding
constexpr int kSP = 48;    // bytes per staged output pixel: 32 of data + 16 of padding
constexpr int kStageWarp = 2 * 32 * kSP;
constexpr int kDBReg = 7;  // taps of the input-gradient kernel whose weight fragments stay in registers (8 registers each)

template <typename T> struct MmaD;
template <> struct MmaD<__nv_bfloat16> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    const __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};
template <> struct MmaD<__half> {
  __device__ static __forceinline__ void run(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
  __device__ static __forceinline__ uint32_t pack(float lo, float hi) {
    const __half2 p = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&p);
  }
};
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

// four 8x8 16-bit matrices from the accumulator fragment layout to shared memory in one instruction (lane l supplies the address of
// row l % 8 of matrix l / 8)
__device__ __forceinline__ void stsm_x4(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.shared.b16 [%0], {%1,%2,%3,%4};" :: "r"(addr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}

struct WStride { long long oc, ci, ky, kx; };
// L2 prefetch of a row segment the NEXT tile will stage (one 128-byte line per call): after the shared-memory work ncu showed these
// kernels waiting on the global loads of the tile staging (long_scoreboard / wait); a persistent CTA knows its next tile
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }

// tap -> (A tile: row offset a, pixel offset b) and parity class (dy * 2 + dx); see the header
struct Tap { int ky, kx, a, b, cls; };
__device__ constexpr Tap kTaps[9] = {{1, 1, 0, 0, 0}, {1, 0, 0, 1, 1}, {1, 2, 0, 0, 1}, {0, 1, 1, 0, 2}, {2, 1, 0, 0, 2},
                                     {0, 0, 1, 1, 3}, {0, 2, 1, 0, 3}, {2, 0, 0, 1, 3}, {2, 2, 0, 0, 3}};

template <typename T>
__global__ void __launch_bounds__(kThreads, 2) conv3_dgrad_s2_kernel(const T* __restrict__ gy, const T* __restrict__ w, const WStride ws,
                                                                      T* __restrict__ gx, int H, int W, int Ho, int Wo, int tiles_per_img,
                                                                      int n_tiles) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int RP = (Wo + 1) * kGP;                       // bytes per staged gy row
  unsigned char* gs = smem;                            // [kR + 1][Wo + 1][kGP]
  unsigned char* wsm = gs + (size_t)(kR + 1) * RP;     // [9][kCi][kWP]
  unsigned char* stage = wsm + 9 * kCi * kWP;          // [kWarps][2][32][kSP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, q = lane & 3, r = lane >> 2;
  // weight -> [tap][ci][oc] in the 16-bit dtype; the zero pixel past the end of every staged row
  for (int i = tid; i < 9 * kCi * kOc; i += kThreads) {
    const int tap = i / (kCi * kOc), rem = i - tap * kCi * kOc, ci = rem / kOc, oc = rem - ci * kOc;
    const int ky = tap / 3, kx = tap - ky * 3;
    *reinterpret_cast<T*>(wsm + (size_t)(tap * kCi + ci) * kWP + oc * 2) = w[oc * ws.oc + ci * ws.ci + ky * ws.ky + kx * ws.kx];
  }
  for (int i = tid; i < (kR + 1) * (kGP / 16); i += kThreads)
    *reinterpret_cast<uint4*>(gs + (size_t)(i / (kGP / 16)) * RP + (size_t)Wo * kGP + (i % (kGP / 16)) * 16) = make_uint4(0, 0, 0, 0);

  const uint32_t gs_u = smem_u32(gs), ws_u = smem_u32(wsm);
  const uint32_t a_lane = (uint32_t)(((lane & 7) + ((lane & 8) ? 8 : 0)) * kGP + ((lane & 16) ? 16 : 0));
  const uint32_t b_lane = (uint32_t)(((lane & 7) + ((lane & 16) ? 8 : 0)) * kWP + ((lane & 8) ? 16 : 0));
  unsigned char* st = stage + (size_t)warp * kStageWarp;
  const uint32_t st_u = smem_u32(st);
  const int gpr = Wo / 16;
  // The weight fragments of the first kDBReg taps (in kTaps order) stay in registers for the whole kernel: re-reading all 18 of
  // them per 16-pixel group kept the kernel on the shared-memory pipe (ncu: mio_throttle / short_scoreboard lead the stalls; HMMA
  // at 26 % of its rate, DRAM at 30 %)
  __syncthreads();
  uint32_t Bf[kDBReg][2][4];
#pragma unroll
  for (int t = 0; t < kDBReg; ++t)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
      ldsm_x4(Bf[t][ks], ws_u + (uint32_t)((kTaps[t].ky * 3 + kTaps[t].kx) * kCi * kWP + ks * 32) + b_lane);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_img, py0 = (tile - b * tiles_per_img) * kR;
    __syncthreads();   // previous tile consumed
    for (int i = 0; i <= kR; ++i) {
      const int oy = py0 + i;
      const bool ok = oy < Ho;
      const unsigned char* src = reinterpret_cast<const unsigned char*>(gy) + ((size_t)(b * Ho + (ok ? oy : 0)) * Wo) * (kOc * 2);
      unsigned char* dst = gs + (size_t)i * RP;
      for (int v = tid; v < Wo * 4; v += kThreads) cp_async16(dst + (size_t)(v >> 2) * kGP + (v & 3) * 16, src + (size_t)v * 16, ok);
    }
    cp_async_wait_all();
    __syncthreads();
    if (tile + (int)gridDim.x < n_tiles) {   // pull the next tile's gy rows into L2 while this one is multiplied
      const int nt_ = tile + gridDim.x, nb = nt_ / tiles_per_img, npy = (nt_ - nb * tiles_per_img) * kR;
      const int rows_n = min(kR + 1, Ho - npy), bytes = rows_n * Wo * (kOc * 2);   // the rows of a tile are contiguous in gy
      const unsigned char* src = reinterpret_cast<const unsigned char*>(gy) + ((size_t)(nb * Ho + npy) * Wo) * (kOc * 2);
      for (int o = tid * 128; o < bytes; o += kThreads * 128) prefetch_l2(src + o);
    }
    for (int g = warp; g < kR * gpr; g += kWarps) {
      const int pr = g / gpr, px0 = (g - pr * gpr) * 16;
      if (py0 + pr >= Ho) break;
      uint32_t A[2][2][2][4];   // [row offset a][pixel offset b][k step: oc 0-15 | 16-31]
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int bb = 0; bb < 2; ++bb)
#pragma unroll
          for (int ks = 0; ks < 2; ++ks)
            ldsm_x4(A[a][bb][ks], gs_u + (uint32_t)((pr + a) * RP + (px0 + bb) * kGP + ks * 32) + a_lane);
      // one parity class at a time (8 accumulator registers live instead of 32), staged pixel (dy, 2*m + dx), m = the warp's px index
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float acc[2][4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          if (kTaps[t].cls != c) continue;
          const Tap tp = kTaps[t];
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
            if (t < kDBReg) {
              MmaD<T>::run(acc[0], A[tp.a][tp.b][ks], Bf[t < kDBReg ? t : 0][ks][0], Bf[t < kDBReg ? t : 0][ks][1]);
              MmaD<T>::run(acc[1], A[tp.a][tp.b][ks], Bf[t < kDBReg ? t : 0][ks][2], Bf[t < kDBReg ? t : 0][ks][3]);
            } else {
              uint32_t B[4];   // b0 / b1 of ci 0-7, b0 / b1 of ci 8-15
              ldsm_x4(B, ws_u + (uint32_t)((tp.ky * 3 + tp.kx) * kCi * kWP + ks * 32) + b_lane);
              MmaD<T>::run(acc[0], A[tp.a][tp.b][ks], B[0], B[1]);
              MmaD<T>::run(acc[1], A[tp.a][tp.b][ks], B[2], B[3]);
            }
          }
        }
        // matrices (n-tile, pixel half): lane l addresses row l % 8 of matrix l / 8 = staged pixel 2 * (8 * half + row) + dx
        const int dy = c >> 1, dx = c & 1;
        stsm_x4(st_u + (uint32_t)(dy * (32 * kSP) + (2 * (8 * ((lane >> 3) & 1) + (lane & 7)) + dx) * kSP + (lane >> 4) * 16),
                MmaD<T>::pack(acc[0][0], acc[0][1]), MmaD<T>::pack(acc[0][2], acc[0][3]), MmaD<T>::pack(acc[1][0], acc[1][1]),
                MmaD<T>::pack(acc[1][2], acc[1][3]));
      }
      __syncwarp();
      unsigned char* orow = reinterpret_cast<unsigned char*>(gx) + (((size_t)b * H + 2 * (py0 + pr)) * W + 2 * px0) * (kCi * 2);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = lane + 32 * j, dy = c >> 6, rem = c & 63;   // 64 16-byte chunks = one row of 32 input pixels
        const uint4 v = *reinterpret_cast<const uint4*>(st + dy * (32 * kSP) + (rem >> 1) * kSP + (rem & 1) * 16);
        stg_stream16(orow + (size_t)dy * W * (kCi * 2) + (size_t)rem * 16, v);
      }
      __syncwarp();
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------------
// Forward of the same layer: y[b, oy, ox, oc] = sum over (ky, kx, ci) of x[b, 2*oy - 1 + ky, 2*ox - 1 + kx, ci] * w[oc, ci, ky, kx].
// cuDNN picks an sm80 legacy fprop here (0.14 ms for 210 MB in / 105 MB out: 3x the HBM time).  Implicit GEMM per 16 output pixels:
// M = 16, N = 32 oc, K = 9 taps x 16 ci = 36 MMAs.  The A fragment of tap (ky, kx) is ONE ldmatrix.x4 on the staged NHWC input
// row 2*orow + ky: matrix rows = the 16-byte halves of pixels 2*(ox0 + m) + kx (pixel 0 of a staged row is x = -1, a zero pixel).
// Rows 64 bytes apart would hit four banks eight times; the 16-byte chunks of every 128-byte line (4 pixels) are therefore XOR-
// swizzled with the line index (chunk ^= line & 3), which makes the eight rows of a matrix land in eight different chunks.
// ---------------------------------------------------------------------------------------------------------------------------
constexpr int kFR = 2, kFWarps = 10, kFThreads = kFWarps * 32;   // 2 output rows x 10 groups of 16 pixels at W/2 = 160: 2 groups per warp
constexpr int kFWP = 48;   // bytes per (tap, oc) weight row: 16 ci + padding
constexpr int kFSP = 80;   // bytes per staged output pixel: 32 oc + padding

__device__ __host__ __forceinline__ int fwd_phys(int p, int h) {   // byte offset of half h of pixel slot p inside a staged row
  return (p >> 2) * 128 + (((((p & 3) << 1) | h) ^ ((p >> 2) & 3)) << 4);
}

template <typename T>
__global__ void __launch_bounds__(kFThreads, 2) conv3_fwd_s2_kernel(const T* __restrict__ x, const T* __restrict__ w, const WStride ws,
                                                                     T* __restrict__ y, int H, int W, int Ho, int Wo, int tiles_per_img,
                                                                     int n_tiles) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int IR = 2 * kFR + 1;
  const int RPB = ((W + 1 + 3) / 4) * 128;             // bytes per staged input row: slot 0 = x = -1, slots 1..W, rounded up to a line
  unsigned char* xs = smem;                            // [IR][slots][32 B], swizzled
  unsigned char* wsm = xs + (size_t)IR * RPB;          // [9][kOc][kFWP]
  unsigned char* stage = wsm + 9 * kOc * kFWP;         // [kFWarps][16][kFSP]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, q = lane & 3, r = lane >> 2;
  for (int i = tid; i < 9 * kOc * kCi; i += kFThreads) {
    const int tap = i / (kOc * kCi), rem = i - tap * kOc * kCi, oc = rem / kCi, ci = rem - oc * kCi;
    const int ky = tap / 3, kx = tap - ky * 3;
    *reinterpret_cast<T*>(wsm + (size_t)(tap * kOc + oc) * kFWP + ci * 2) = w[oc * ws.oc + ci * ws.ci + ky * ws.ky + kx * ws.kx];
  }
  for (int i = tid; i < IR * 2; i += kFThreads)        // the zero pixel in front of every staged row
    *reinterpret_cast<uint4*>(xs + (size_t)(i >> 1) * RPB + fwd_phys(0, i & 1)) = make_uint4(0, 0, 0, 0);

  const uint32_t xs_u = smem_u32(xs), ws_u = smem_u32(wsm);
  const int m_l = (lane & 7) + ((lane & 8) ? 8 : 0), h_l = (lane & 16) ? 1 : 0;
  uint32_t a_off[3];
#pragma unroll
  for (int kx = 0; kx < 3; ++kx) a_off[kx] = (uint32_t)fwd_phys(2 * m_l + kx, h_l);   // + og * 1024 per group (16 pixels = 8 lines)
  const uint32_t b_lane = (uint32_t)(((lane & 7) + ((lane & 16) ? 8 : 0)) * kFWP + ((lane & 8) ? 16 : 0));
  unsigned char* st = stage + (size_t)warp * (16 * kFSP);
  const int gpr = Wo / 16;
  // The weight fragments live in registers for the whole kernel (9 taps x 2 x 4 registers): re-reading them per 16-pixel group
  // was 18 of the 27 ldmatrix per group, and ncu showed the kernel stalled on the shared-memory pipe (mio_throttle /
  // short_scoreboard), not on HMMA (26 % of its rate) or DRAM (30 %)
  __syncthreads();
  constexpr int kBReg = 6;   // taps whose fragments fit next to the accumulators under the 2-CTAs-per-SM register budget (102)
  uint32_t Bf[kBReg][2][4];
#pragma unroll
  for (int t = 0; t < kBReg; ++t) {
    ldsm_x4(Bf[t][0], ws_u + (uint32_t)((t * kOc) * kFWP) + b_lane);          // oc 0-15: b0/b1 of n-tiles 0, 1
    ldsm_x4(Bf[t][1], ws_u + (uint32_t)((t * kOc + 16) * kFWP) + b_lane);     // oc 16-31: n-tiles 2, 3
  }
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int b = tile / tiles_per_img, oy0 = (tile - b * tiles_per_img) * kFR;
    __syncthreads();   // previous tile consumed
#pragma unroll
    for (int i = 0; i < IR; ++i) {
      const int iy = 2 * oy0 - 1 + i;
      const bool ok = iy >= 0 && iy < H;
      const unsigned char* src = reinterpret_cast<const unsigned char*>(x) + ((size_t)(b * H + (ok ? iy : 0)) * W) * (kCi * 2);
      unsigned char* dst = xs + (size_t)i * RPB;
      for (int v = tid; v < W * 2; v += kFThreads) cp_async16(dst + fwd_phys((v >> 1) + 1, v & 1), src + (size_t)v * 16, ok);
    }
    cp_async_wait_all();
    __syncthreads();
    if (tile + (int)gridDim.x < n_tiles) {   // pull the next tile's input rows into L2 while this one is multiplied
      const int nt_ = tile + gridDim.x, nb = nt_ / tiles_per_img, noy = (nt_ - nb * tiles_per_img) * kFR;
      const int iy0 = max(2 * noy - 1, 0), iy1 = min(2 * noy - 1 + IR, H), bytes = (iy1 - iy0) * W * (kCi * 2);   // contiguous rows of x
      const unsigned char* src = reinterpret_cast<const unsigned char*>(x) + ((size_t)(nb * H + iy0) * W) * (kCi * 2);
      for (int o = tid * 128; o < bytes; o += kFThreads * 128) prefetch_l2(src + o);
    }
    for (int g = warp; g < kFR * gpr; g += kFWarps) {
      const int orow = g / gpr, og = g - orow * gpr;
      if (oy0 + orow >= Ho) break;
      float acc[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int ky = t / 3, kx = t - ky * 3;
        uint32_t A[4];
        ldsm_x4(A, xs_u + (uint32_t)((2 * orow + ky) * RPB + og * 1024) + a_off[kx]);
        if (t < kBReg) {
          MmaD<T>::run(acc[0], A, Bf[t < kBReg ? t : 0][0][0], Bf[t < kBReg ? t : 0][0][1]);
          MmaD<T>::run(acc[1], A, Bf[t < kBReg ? t : 0][0][2], Bf[t < kBReg ? t : 0][0][3]);
          MmaD<T>::run(acc[2], A, Bf[t < kBReg ? t : 0][1][0], Bf[t < kBReg ? t : 0][1][1]);
          MmaD<T>::run(acc[3], A, Bf[t < kBReg ? t : 0][1][2], Bf[t < kBReg ? t : 0][1][3]);
        } else {
          uint32_t B0[4], B1[4];
          ldsm_x4(B0, ws_u + (uint32_t)((t * kOc) * kFWP) + b_lane);
          ldsm_x4(B1, ws_u + (uint32_t)((t * kOc + 16) * kFWP) + b_lane);
          MmaD<T>::run(acc[0], A, B0[0], B0[1]);
          MmaD<T>::run(acc[1], A, B0[2], B0[3]);
          MmaD<T>::run(acc[2], A, B1[0], B1[1]);
          MmaD<T>::run(acc[3], A, B1[2], B1[3]);
        }
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        unsigned char* o = st + r * kFSP + (nt * 8 + 2 * q) * 2;
        *reinterpret_cast<uint32_t*>(o) = MmaD<T>::pack(acc[nt][0], acc[nt][1]);
        *reinterpret_cast<uint32_t*>(o + 8 * kFSP) = MmaD<T>::pack(acc[nt][2], acc[nt][3]);
      }
      __syncwarp();
      unsigned char* orow_g = reinterpret_cast<unsigned char*>(y) + (((size_t)b * Ho + oy0 + orow) * Wo + og * 16) * (kOc * 2);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int c = lane + 32 * j;   // 64 16-byte chunks = 16 pixels x 32 oc, contiguous in y
        stg_stream16(orow_g + (size_t)c * 16, *reinterpret_cast<const uint4*>(st + (c >> 2) * kFSP + (c & 3) * 16));
      }
      __syncwarp();
    }
  }
}

size_t fwd_smem_bytes(int W) { return (size_t)(2 * kFR + 1) * (((W + 1 + 3) / 4) * 128) + 9 * kOc * kFWP + kFWarps * 16 * kFSP; }

bool dgrad_shape_ok(int H, int W, int cin, int cout, int dtype) {
  if (!(dtype == B200_BF16 || dtype == B200_F16) || cin != kCi || cout != kOc) return false;
  if (H <= 0 || W <= 0 || ((H | W) & 1)) return false;
  const int Wo = W / 2;
  const size_t smem = (size_t)(kR + 1) * (Wo + 1) * kGP + 9 * kCi * kWP + kWarps * kStageWarp;
  return Wo % 16 == 0 && smem <= (size_t)max_smem_optin() && fwd_smem_bytes(W) <= (size_t)max_smem_optin();
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_conv3x3_dgrad_s2_supported(int32_t H, int32_t W, int32_t cin, int32_t cout, int32_t dtype) {
  return dgrad_shape_ok(H, W, cin, cout, dtype) ? 1 : 0;
}

extern "C" B200_API int b200_conv3x3_dgrad_s2(const void* gy, const void* w, const int64_t* w_stride, void* gx, int32_t B, int32_t H, int32_t W,
                                              int32_t cin, int32_t cout, int32_t dtype, void* stream) {
  B200_REQUIRE(gy && w && w_stride && gx, B200_ERR_SHAPE, "conv3x3_dgrad_s2: null pointer");
  B200_REQUIRE(B > 0 && dgrad_shape_ok(H, W, cin, cout, dtype), B200_ERR_UNSUPPORTED,
               "conv3x3_dgrad_s2: unsupported shape H=%d W=%d cin=%d cout=%d dtype=%d", H, W, cin, cout, dtype);
  B200_REQUIRE((((uintptr_t)gy | (uintptr_t)gx) & 15) == 0, B200_ERR_ALIGN, "conv3x3_dgrad_s2: tensors must be 16-byte aligned");
  const int Ho = H / 2, Wo = W / 2, tpi = (Ho + kR - 1) / kR, n_tiles = B * tpi;
  const size_t smem = (size_t)(kR + 1) * (Wo + 1) * kGP + 9 * kCi * kWP + kWarps * kStageWarp;
  const WStride ws{w_stride[0], w_stride[1], w_stride[2], w_stride[3]};
  cudaStream_t st = (cudaStream_t)stream;
  auto go = [&](auto kern, auto* tag) -> int {
    using T = typename std::remove_pointer<decltype(tag)>::type;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem);
    per_sm = per_sm < 1 ? 1 : per_sm > 4 ? 4 : per_sm;
    int grid = sm_count() * per_sm;   // persistent CTAs: one resident wave
    if (grid > n_tiles) grid = n_tiles;
    kern<<<grid, kThreads, smem, st>>>((const T*)gy, (const T*)w, ws, (T*)gx, H, W, Ho, Wo, tpi, n_tiles);
    return check_launch("conv3x3_dgrad_s2");
  };
  if (dtype == B200_BF16) return go(conv3_dgrad_s2_kernel<__nv_bfloat16>, (__nv_bfloat16*)nullptr);
  return go(conv3_dgrad_s2_kernel<__half>, (__half*)nullptr);
}

extern "C" B200_API int b200_conv3x3_fwd_s2(const void* x, const void* w, const int64_t* w_stride, void* y, int32_t B, int32_t H, int32_t W,
                                            int32_t cin, int32_t cout, int32_t dtype, void* stream) {
  B200_REQUIRE(x && w && w_stride && y, B200_ERR_SHAPE, "conv3x3_fwd_s2: null pointer");
  B200_REQUIRE(B > 0 && dgrad_shape_ok(H, W, cin, cout, dtype), B200_ERR_UNSUPPORTED,
               "conv3x3_fwd_s2: unsupported shape H=%d W=%d cin=%d cout=%d dtype=%d", H, W, cin, cout, dtype);
  B200_REQUIRE((((uintptr_t)x | (uintptr_t)y) & 15) == 0, B200_ERR_ALIGN, "conv3x3_fwd_s2: tensors must be 16-byte aligned");
  const int Ho = H / 2, Wo = W / 2, tpi = (Ho + kFR - 1) / kFR, n_tiles = B * tpi;
  const size_t smem = fwd_smem_bytes(W);
  const WStride ws{w_stride[0], w_stride[1], w_stride[2], w_stride[3]};
  cudaStream_t st = (cudaStream_t)stream;
  auto go = [&](auto kern, auto* tag) -> int {
    using T = typename std::remove_pointer<decltype(tag)>::type;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kFThreads, smem);
    per_sm = per_sm < 1 ? 1 : per_sm > 4 ? 4 : per_sm;
    int grid = sm_count() * per_sm;   // persistent CTAs: one resident wave
    if (grid > n_tiles) grid = n_tiles;
    kern<<<grid, kFThreads, smem, st>>>((const T*)x, (const T*)w, ws, (T*)y, H, W, Ho, Wo, tpi, n_tiles);
    return check_launch("conv3x3_fwd_s2");
  };
  if (dtype == B200_BF16) return go(conv3_fwd_s2_kernel<__nv_bfloat16>, (__nv_bfloat16*)nullptr);
  return go(conv3_fwd_s2_kernel<__half>, (__half*)nullptr);
}
