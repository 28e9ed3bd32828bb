// CBAM (channel attention -> spatial attention -> gate), forward and backward.
// Replaces cbam.py:29-38 / :48-53 / :62-71 of the reference (and their autograd backward).
//
// The block is a chain of lean streaming kernels; the feature map x (NHWC) is read from HBM by the first one and
// re-read from the 126 MB L2 by the later ones (13-52 MB at the model's shapes), written once:
//   fwd  pool : per-channel sum / max (/ first argmax pixel) over a pixel slice; thread = one 16-byte channel
//               vector, looping over pixels                                  -> partials [B][S][3][C]
//        mlp  : per image: fold the S partials, shared MLP + sigmoid (cbam.py:24-38)      -> ca [B][C]
//        map  : per-pixel mean_c / max_c (/ argmax_c) of x*ca, sub-warp per pixel         -> maps [B][3][HW]
//        gate : zero-padded 2-D tile of the maps in smem, 7x7 conv + sigmoid (4 lanes per pixel), out = x*ca*sa
//               with packed 16-bit multiplies and 16-byte stores
//   bwd  gz   : g_z = (sum_c g x ca) sa (1-sa) per pixel
//        mid  : conv^T(g_z) -> g_s per pixel, conv weight-gradient partials, g_ca partials  (SA mode: writes g_x)
//        mlp  : per image: MLP backward, weight-gradient partials, g_pavg / g_pmax per channel
//        fin  : g_x = (g sa + g_s0 + [c==argmax_c] g_s1) ca + g_pavg/HW (+ g_pmax at the pooled-max pixel)
//        fold : weight-gradient partials -> gradients, fixed order (deterministic, no atomics anywhere)
// The forward stashes its small by-products (pooled avg/max, both argmax maps, the 2-channel map) so the backward
// recomputes nothing.  A 3x3 spatial-attention kernel (cbam.py:43) runs as a 7x7 kernel embedded in zeros.
// (An earlier one-launch design -- one thread-block cluster per image with the chunk resident in shared memory and
// DSMEM reductions -- had the minimal 1R+1W HBM traffic but was bound by its per-CTA dependency chain at these
// sizes: 31 us at the model's shape against 10 us for a plain copy; see profiles/README.md.)
//
// NaN note: the channel/pixel maxima use the hardware max (which drops NaN) because every output they can reach is
// already NaN through the sum/mean computed over the same elements (a NaN in x makes the pooled average, hence the
// whole ca vector, NaN; a NaN in x*ca makes the channel mean at that pixel NaN, and the mean and max maps feed the
// same conv window) -- the result is NaN in exactly the positions where the reference's is.
#include "cbam.cuh"


namespace b200 {
namespace {
using namespace cbam;

// =====================================================================================================
// forward
// =====================================================================================================
// ---- pool: per-channel sum / max (+ first argmax pixel when IDX) over the CTA's pixel slice ---------------------
template <typename T, int VW, bool IDX>
__global__ void __launch_bounds__(kT) cbam_pool_kernel(const T* __restrict__ x, float* __restrict__ part, const Geo G) {
  extern __shared__ __align__(16) float red[];   // [groups][3][C]
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nw = G.nch, groups = G.groups;
  const int p0 = s * G.np, npix = min(G.np, G.HW - p0);
  const T* xc = x + ((size_t)b * G.HW + p0) * C;
  const int tpg = nw < kT ? nw : kT;   // threads per pixel group
  const int pg = threadIdx.x / tpg, tw = threadIdx.x - pg * tpg;
  for (int w = tw; w < nw; w += kT) {
    float sm[VW], m[VW];
    int mi[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) { sm[e] = 0.f; m[e] = -INFINITY; mi[e] = p0; }
    if (pg < groups) {
      const T* src = xc + w * VW;
#pragma unroll 4
      for (int p = pg; p < npix; p += groups) {
        float v[VW];
        Vec<T, VW>::load(src + (size_t)p * C, v);
#pragma unroll
        for (int e = 0; e < VW; ++e) {
          sm[e] += v[e];
          if (IDX) {
            if (v[e] > m[e]) { m[e] = v[e]; mi[e] = p0 + p; }
          } else {
            m[e] = fmaxf(m[e], v[e]);
          }
        }
      }
      float* rs = red + (size_t)pg * C * 3;
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        rs[w * VW + e] = sm[e];
        rs[C + w * VW + e] = m[e];
        if (IDX) reinterpret_cast<int*>(rs)[2 * C + w * VW + e] = mi[e];
      }
    }
  }
  __syncthreads();
  float* dst = part + ((size_t)b * G.S + s) * 3 * C;
  for (int c = threadIdx.x; c < C; c += kT) {
    float sm = 0.f, m = -INFINITY;
    int mi = p0;
    for (int gi = 0; gi < groups; ++gi) {  // groups interleave pixels: combine by (value, then smaller index)
      const float* rs = red + (size_t)gi * C * 3;
      sm += rs[c];
      const float v = rs[C + c];
      if (IDX) {
        const int vi = reinterpret_cast<const int*>(rs)[2 * C + c];
        if (v > m || (v == m && vi < mi && v != -INFINITY)) { m = v; mi = vi; }
      } else {
        m = fmaxf(m, v);
      }
    }
    dst[c] = sm; dst[C + c] = m;
    if (IDX) reinterpret_cast<int*>(dst)[2 * C + c] = mi;
  }
}

// ---- mlp: fold the slice partials of one image, shared MLP + sigmoid (cbam.py:24-38) ---------------------------
__global__ void __launch_bounds__(kT) cbam_mlp_kernel(const float* __restrict__ part, const float* __restrict__ w1,
                                                      const float* __restrict__ w2, float* __restrict__ ca_out,
                                                      float* __restrict__ pooled, int* __restrict__ amx, const Geo G) {
  extern __shared__ __align__(16) float sm[];   // pav[C] | pmx[C] | hid[2r]
  const int b = blockIdx.x, C = G.C, r = G.r, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* pav = sm;
  float* pmx = sm + C;
  float* hid = sm + 2 * C;
  const float* src = part + (size_t)b * G.S * 3 * C;
  for (int c = tid; c < C; c += kT) {
    float s = 0.f, m = -INFINITY;
    int mi = 0;
    for (int k = 0; k < G.S; ++k) {          // slices ascend in pixel order, strict >: first occurrence
      s += src[(size_t)k * 3 * C + c];
      const float v = src[(size_t)k * 3 * C + C + c];
      if (v > m || k == 0) { m = v; if (amx) mi = reinterpret_cast<const int*>(src)[(size_t)k * 3 * C + 2 * C + c]; }
    }
    const float a = s * G.invHW, mm = (s != s) ? s : m;   // a NaN anywhere in the channel makes the pooled max NaN too
    pav[c] = a; pmx[c] = mm;
    if (pooled) { pooled[(size_t)b * 2 * C + c] = a; pooled[(size_t)b * 2 * C + C + c] = mm; }
    if (amx) amx[(size_t)b * C + c] = mi;
  }
  __syncthreads();
  for (int j = warp; j < 2 * r; j += kWarps) {  // hidden = relu(W1 pooled); j < r: avg branch, j >= r: max branch
    const float* wrow = w1 + (size_t)(j < r ? j : j - r) * C;
    const float* pv = j < r ? pav : pmx;
    float acc = 0.f;
#pragma unroll 4
    for (int c = lane; c < C; c += 32) acc += wrow[c] * pv[c];
    acc = warp_sum(acc);
    if (lane == 0) hid[j] = relu_nan(acc);
  }
  __syncthreads();
  for (int c = tid; c < C; c += kT) {
    const float* wrow = w2 + (size_t)c * r;
    float z = 0.f;
#pragma unroll 4
    for (int j = 0; j < r; ++j) z += wrow[j] * (hid[j] + hid[r + j]);
    ca_out[(size_t)b * C + c] = sigmoidf_(z);
  }
}

// ---- map: per-pixel channel mean / max (/ first argmax channel) of x*ca; sub-warp of LPP lanes per pixel -------
template <typename T, int VW, bool IDX>
__global__ void __launch_bounds__(kT) cbam_map_kernel(const T* __restrict__ x, const float* __restrict__ ca,
                                                      float* __restrict__ maps, const Geo G) {
  extern __shared__ __align__(16) float cas[];   // [C] when a lane owns more than one channel vector
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nch = G.nch, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = s * G.np, npix = min(G.np, G.HW - p0);
  const int LPP = G.lpp, PPW = 32 / LPP, sub = lane / LPP, sl = lane & (LPP - 1);
  const bool one = G.one != 0;
  float car[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) car[e] = 1.f;
  if (ca) {
    if (one) {
      if (sl < nch) {
#pragma unroll
        for (int e = 0; e < VW; ++e) car[e] = ca[(size_t)b * C + sl * VW + e];
      }
    } else {
      for (int c = tid; c < C; c += kT) cas[c] = ca[(size_t)b * C + c];
      __syncthreads();
    }
  }
  const T* xc = x + ((size_t)b * G.HW + p0) * C;
  float* mp = maps + (size_t)b * 3 * G.HW + p0;
  constexpr int U = 2;   // pixels in flight per sub-warp
  for (int k = warp * PPW; k < npix; k += U * kWarps * PPW) {
    float sum[U], mx[U];
    int mi[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = k + u * kWarps * PPW + sub;
      sum[u] = 0.f; mx[u] = -INFINITY; mi[u] = 0x7fffffff;
      if (p < npix) {
        for (int w = sl; w < nch; w += LPP) {
          float v[VW];
          Vec<T, VW>::load(xc + (size_t)p * C + w * VW, v);
          if (!one && ca) {
#pragma unroll
            for (int e = 0; e < VW; ++e) car[e] = cas[w * VW + e];
          }
#pragma unroll
          for (int e = 0; e < VW; ++e) {
            const float t = v[e] * car[e];
            sum[u] += t;
            if (IDX) {
              if (t > mx[u]) { mx[u] = t; mi[u] = w * VW + e; }
            } else {
              mx[u] = fmaxf(mx[u], t);
            }
          }
        }
      }
    }
    for (int o = LPP >> 1; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        sum[u] += __shfl_xor_sync(0xffffffffu, sum[u], o);
        const float tm = __shfl_xor_sync(0xffffffffu, mx[u], o);
        if (IDX) {
          const int ti = __shfl_xor_sync(0xffffffffu, mi[u], o);
          if (tm > mx[u] || (tm == mx[u] && ti < mi[u])) { mx[u] = tm; mi[u] = ti; }  // larger, then first channel
        } else {
          mx[u] = fmaxf(mx[u], tm);
        }
      }
    }
    if (sl == 0) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int p = k + u * kWarps * PPW + sub;
        if (p < npix) {
          mp[p] = sum[u] * G.invC;
          mp[G.HW + p] = mx[u];
          if (IDX) reinterpret_cast<int*>(mp)[2 * G.HW + p] = mi[u] == 0x7fffffff ? 0 : mi[u];
        }
      }
    }
  }
}

// zero-padded [nrow][tw] tile (rows ya-3 .., columns -3 .. W+3) of a per-pixel map of image b
template <typename F>
__device__ __forceinline__ void build_tile(float* tile, int ya, int nrow, const Geo& G, F value_at) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int ty = warp; ty < nrow; ty += kWarps) {
    const int y = ya - PADK + ty;
    float* dst = tile + (size_t)ty * G.tw;
    for (int tx = lane; tx < G.tw; tx += 32) {
      const int xx = tx - PADK;
      dst[tx] = (y >= 0 && y < G.H && xx >= 0 && xx < G.W) ? value_at(y * G.W + xx) : 0.f;
    }
  }
}

// ---- gate: 7x7 conv + sigmoid on the map tile, out = x*ca*sa -------------------------------------------------
template <typename T, int VW>
__global__ void __launch_bounds__(kT) cbam_gate_kernel(const T* __restrict__ x, const float* __restrict__ ca,
                                                       const float* __restrict__ maps, const float* __restrict__ wsa,
                                                       T* __restrict__ out, float* __restrict__ sa_out, const Geo G) {
  extern __shared__ __align__(16) float sm[];   // wsas[112] | tile[2][th][tw] | sas[np] | cas[C]
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nch = G.nch, W = G.W, tw = G.tw;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = s * G.np, npix = min(G.np, G.HW - p0);
  float* wsas = sm;
  float* tile = sm + NTAPS;
  float* sas = tile + 2 * G.th * tw;
  float* cas = sas + ((G.np + 3) & ~3);
  load_taps(wsas, wsa, G.ksa);
  const int ya = p0 / W, nrow = (p0 + npix - 1) / W - ya + 1 + 2 * PADK;
  const float* mp = maps + (size_t)b * 3 * G.HW;
  build_tile(tile, ya, nrow, G, [&](int q) { return mp[q]; });
  build_tile(tile + G.th * tw, ya, nrow, G, [&](int q) { return mp[G.HW + q]; });
  const int LPP = G.lpp, PPW = 32 / LPP, sub = lane / LPP, sl = lane & (LPP - 1);
  const bool one = G.one != 0;
  float car[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) car[e] = 1.f;
  if (ca && out) {
    if (one) {
      if (sl < nch) {
#pragma unroll
        for (int e = 0; e < VW; ++e) car[e] = ca[(size_t)b * C + sl * VW + e];
      }
    } else {
      for (int c = tid; c < C; c += kT) cas[c] = ca[(size_t)b * C + c];
    }
  }
  __syncthreads();
  // 4 lanes per pixel split the 14 tap rows, taps broadcast as float4
  for (int base = warp * 32; base < npix * 4; base += kT) {
    const int i = base + lane, p = i >> 2, part = i & 3;
    float z = 0.f;
    if (p < npix) {
      const int q = p0 + p, y = q / W, xx = q - y * W;
      const float* t0 = tile + (size_t)(y - ya) * tw + xx;
      for (int rr = part; rr < 2 * KS; rr += 4) {       // rr = ch*7 + u
        const int ch = rr >= KS ? 1 : 0, u = rr - ch * KS;
        const float4 wa = *reinterpret_cast<const float4*>(wsas + rr * KROW);
        const float4 wb = *reinterpret_cast<const float4*>(wsas + rr * KROW + 4);
        const float* tr = t0 + (size_t)(ch * G.th + u) * tw;
        z += wa.x * tr[0] + wa.y * tr[1] + wa.z * tr[2] + wa.w * tr[3] + wb.x * tr[4] + wb.y * tr[5] + wb.z * tr[6];
      }
    }
    z += __shfl_xor_sync(0xffffffffu, z, 1);
    z += __shfl_xor_sync(0xffffffffu, z, 2);
    if (part == 0 && p < npix) {
      const float a = sigmoidf_(z);
      sas[p] = a;
      if (sa_out) sa_out[(size_t)b * G.HW + p0 + p] = a;
    }
  }
  if (!out) return;
  __syncthreads();
  const T* xc = x + ((size_t)b * G.HW + p0) * C;
  T* og = out + ((size_t)b * G.HW + p0) * C;
  if constexpr (sizeof(T) == 2 && VW == 8) {
    // packed 16-bit gate: out = (x*ca)*sa, rounded after each product exactly like the 16-bit reference ops
    using P2 = typename Pair2<T>::type;
    P2 ca2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) ca2[i] = make_pair(T(), car[2 * i], car[2 * i + 1]);
#pragma unroll 2
    for (int k = warp * PPW; k < npix; k += kWarps * PPW) {
      const int p = k + sub;
      if (p >= npix) continue;
      const float sp = sas[p];
      const P2 sp2 = make_pair(T(), sp, sp);
      for (int w = sl; w < nch; w += LPP) {
        uint4 raw = ldg_stream16(xc + (size_t)p * C + w * VW);
        P2* rp = reinterpret_cast<P2*>(&raw);
        if (!one) {
#pragma unroll
          for (int i = 0; i < 4; ++i) ca2[i] = make_pair(T(), cas[w * VW + 2 * i], cas[w * VW + 2 * i + 1]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) rp[i] = __hmul2(__hmul2(rp[i], ca2[i]), sp2);
        stg_stream16(og + (size_t)p * C + w * VW, raw);
      }
    }
  } else {
    for (int k = warp * PPW; k < npix; k += kWarps * PPW) {
      const int p = k + sub;
      if (p >= npix) continue;
      const float sp = sas[p];
      for (int w = sl; w < nch; w += LPP) {
        float v[VW];
        Vec<T, VW>::load(xc + (size_t)p * C + w * VW, v);
#pragma unroll
        for (int e = 0; e < VW; ++e) v[e] = v[e] * (one ? car[e] : cas[w * VW + e]) * sp;
        Vec<T, VW>::store(og + (size_t)p * C + w * VW, v);
      }
    }
  }
}

// =====================================================================================================
// backward (SURVEY App. A.1)
// =====================================================================================================
// ---- gz: g_z[p] = (sum_c g x ca) sa (1-sa) ----------------------------------------------------------------
template <typename T, int VW>
__global__ void __launch_bounds__(kT) cbam_bwd_gz_kernel(const T* __restrict__ x, const T* __restrict__ g,
                                                         const float* __restrict__ ca, const float* __restrict__ sa,
                                                         float* __restrict__ gz, const Geo G) {
  extern __shared__ __align__(16) float cas[];
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nch = G.nch, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = s * G.np, npix = min(G.np, G.HW - p0);
  const int LPP = G.lpp, PPW = 32 / LPP, sub = lane / LPP, sl = lane & (LPP - 1);
  const bool one = G.one != 0;
  float car[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) car[e] = 1.f;
  if (ca) {
    if (one) {
      if (sl < nch) {
#pragma unroll
        for (int e = 0; e < VW; ++e) car[e] = ca[(size_t)b * C + sl * VW + e];
      }
    } else {
      for (int c = tid; c < C; c += kT) cas[c] = ca[(size_t)b * C + c];
      __syncthreads();
    }
  }
  const T* xc = x + ((size_t)b * G.HW + p0) * C;
  const T* gc = g + ((size_t)b * G.HW + p0) * C;
  constexpr int U = 2;
  for (int k = warp * PPW; k < npix; k += U * kWarps * PPW) {
    float acc[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = k + u * kWarps * PPW + sub;
      acc[u] = 0.f;
      if (p < npix) {
        for (int w = sl; w < nch; w += LPP) {
          float v[VW], gv[VW];
          Vec<T, VW>::load(xc + (size_t)p * C + w * VW, v);
          Vec<T, VW>::load(gc + (size_t)p * C + w * VW, gv);
          if (!one && ca) {
#pragma unroll
            for (int e = 0; e < VW; ++e) car[e] = cas[w * VW + e];
          }
#pragma unroll
          for (int e = 0; e < VW; ++e) acc[u] += gv[e] * (v[e] * car[e]);
        }
      }
    }
    for (int o = LPP >> 1; o > 0; o >>= 1) {
#pragma unroll
      for (int u = 0; u < U; ++u) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], o);
    }
    if (sl == 0) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int p = k + u * kWarps * PPW + sub;
        if (p < npix) {
          const float a = sa[(size_t)b * G.HW + p0 + p];
          gz[(size_t)b * G.HW + p0 + p] = acc[u] * a * (1.f - a);
        }
      }
    }
  }
}

// ---- mid: conv^T(g_z) -> per-pixel {sa, g_s0/C, g_s1, argmax_c}; conv weight-gradient partials; g_ca partials --
// FULL: gzin = g_z map;  SA: gzin = dL/dsa (g_z formed on the fly) and g_x is written here.
template <typename T, int VW>
__global__ void __launch_bounds__(kT) cbam_bwd_mid_kernel(const T* __restrict__ x, const T* __restrict__ g,
                                                          const float* __restrict__ gzin, const float* __restrict__ sa,
                                                          const float* __restrict__ maps, const float* __restrict__ wsa,
                                                          float4* __restrict__ pixg, float* __restrict__ cpart,
                                                          float* __restrict__ gpart, T* __restrict__ gx_sa, const Geo G) {
  extern __shared__ __align__(16) float sm[];   // wsas[112] | tile[3][th][tw] | pix float4[np] | gzs[np] | poff[np] | red
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nch = G.nch, W = G.W, tw = G.tw, HW = G.HW;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = s * G.np, npix = min(G.np, HW - p0), npad = (G.np + 3) & ~3;
  float* wsas = sm;
  float* tile = sm + NTAPS;
  float4* pix = reinterpret_cast<float4*>(tile + ((3 * G.th * tw + 3) & ~3));
  float* gzs = reinterpret_cast<float*>(pix + npad);
  int* poff = reinterpret_cast<int*>(gzs + npad);
  float* red = reinterpret_cast<float*>(poff + npad);
  load_taps(wsas, wsa, G.ksa);
  const int ya = p0 / W, nrow = (p0 + npix - 1) / W - ya + 1 + 2 * PADK;
  const float* mp = maps + (size_t)b * 3 * HW;
  const float* sab = sa + (size_t)b * HW;
  const float* gzb = gzin + (size_t)b * HW;
  const bool sa_mode = G.mode == B200_CBAM_SA;
  if (sa_mode) build_tile(tile, ya, nrow, G, [&](int q) { const float a = sab[q]; return gzb[q] * a * (1.f - a); });
  else build_tile(tile, ya, nrow, G, [&](int q) { return gzb[q]; });
  build_tile(tile + G.th * tw, ya, nrow, G, [&](int q) { return mp[q]; });
  build_tile(tile + 2 * G.th * tw, ya, nrow, G, [&](int q) { return mp[HW + q]; });
  for (int p = tid; p < npix; p += kT) {
    const int q = p0 + p, y = q / W;
    poff[p] = (y - ya) * tw + (q - y * W);
  }
  __syncthreads();
  // g_s = conv^T(g_z): g_s[j][y][x] = sum_{u,v} w[j][u][v] * g_z[y-(u-3)][x-(v-3)]; 4 lanes per pixel split the rows u
  for (int base = warp * 32; base < npix * 4; base += kT) {
    const int i = base + lane, p = i >> 2, part = i & 3;
    float g0 = 0.f, g1 = 0.f;
    if (p < npix) {
      const float* t0 = tile + poff[p];
      for (int u = part; u < KS; u += 4) {
        const float* tr = t0 + (KS - 1 - u) * tw;
        const float* w0 = wsas + u * KROW;
        const float* w1 = wsas + (KS + u) * KROW;
#pragma unroll
        for (int v = 0; v < KS; ++v) {
          const float z = tr[KS - 1 - v];
          g0 += w0[v] * z;
          g1 += w1[v] * z;
        }
      }
    }
    g0 += __shfl_xor_sync(0xffffffffu, g0, 1);
    g1 += __shfl_xor_sync(0xffffffffu, g1, 1);
    g0 += __shfl_xor_sync(0xffffffffu, g0, 2);
    g1 += __shfl_xor_sync(0xffffffffu, g1, 2);
    if (part == 0 && p < npix) {
      const int q = p0 + p;
      // {sa, broadcast share of the channel mean, share routed to the argmax channel, argmax channel}
      const float4 pp = make_float4(sab[q], g0 * G.invC, g1, mp[2 * HW + q]);
      pix[p] = pp;
      gzs[p] = tile[poff[p] + PADK * tw + PADK];
      if (pixg) pixg[(size_t)b * HW + q] = pp;
    }
  }
  __syncthreads();
  // g_Wsa[j,u,v] = sum_p g_z[p] * s[j, p + (u-3, v-3)]: warp per tap over this CTA's pixels -> per-CTA partial,
  // folded over images and slices in a fixed order by fold_partials_kernel
  float* cp = cpart + ((size_t)b * G.S + s) * NT7;
  for (int t = warp; t < NT7; t += kWarps) {
    const int j = t / (KS * KS), u = (t / KS) % KS, v = t % KS;
    const float* tj = tile + (size_t)((1 + j) * G.th + u) * tw + v;
    float acc = 0.f;
    for (int p = lane; p < npix; p += 32) acc += gzs[p] * tj[poff[p]];
    acc = warp_sum(acc);
    if (lane == 0) cp[t] = acc;
  }
  if (sa_mode) {   // gx = g_s0 + [c == argmax_c] g_s1, no channel attention involved
    T* og = gx_sa + ((size_t)b * HW + p0) * C;
    for (int i = tid; i < npix * nch; i += kT) {
      const int p = i / nch, w = i - p * nch;
      const float4 pp = pix[p];
      const int am = __float_as_int(pp.w);
      float o[VW];
#pragma unroll
      for (int e = 0; e < VW; ++e) o[e] = pp.y + ((w * VW + e) == am ? pp.z : 0.f);
      Vec<T, VW>::store(og + (size_t)p * C + w * VW, o);
    }
    return;
  }
  // g_x1 = g*sa + g_s0 + [c==argmax_c] g_s1 ;  g_ca[c] = sum_p g_x1 * x  (per-CTA partial)
  const T* xc = x + ((size_t)b * HW + p0) * C;
  const T* gc = g + ((size_t)b * HW + p0) * C;
  const int groups = G.groups;
  const int tpg = nch < kT ? nch : kT;
  const int pg = tid / tpg, twi = tid - pg * tpg;
  for (int w = twi; w < nch; w += kT) {
    float acc[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) acc[e] = 0.f;
    if (pg < groups) {
#pragma unroll 2
      for (int p = pg; p < npix; p += groups) {
        float v[VW], gv[VW];
        Vec<T, VW>::load(xc + (size_t)p * C + w * VW, v);
        Vec<T, VW>::load(gc + (size_t)p * C + w * VW, gv);
        const float4 pp = pix[p];
        const unsigned d = (unsigned)(__float_as_int(pp.w) - w * VW);
#pragma unroll
        for (int e = 0; e < VW; ++e) acc[e] += (gv[e] * pp.x + pp.y) * v[e];
        if (d < (unsigned)VW) {   // the argmax channel of this pixel lies in this thread's vector (1 lane per pixel)
#pragma unroll
          for (int e = 0; e < VW; ++e) acc[e] += (d == (unsigned)e) ? pp.z * v[e] : 0.f;
        }
      }
#pragma unroll
      for (int e = 0; e < VW; ++e) red[(size_t)pg * C + w * VW + e] = acc[e];
    }
  }
  __syncthreads();
  float* gp = gpart + ((size_t)b * G.S + s) * C;
  for (int c = tid; c < C; c += kT) {
    float a = 0.f;
    for (int gi = 0; gi < groups; ++gi) a += red[(size_t)gi * C + c];
    gp[c] = a;
  }
}

// ---- mlp backward per image: g_ca -> weight-gradient partials, g_pavg/HW and g_pmax per channel ---------------
__global__ void __launch_bounds__(kT) cbam_mlp_bwd_kernel(const float* __restrict__ gpart, const float* __restrict__ gca_in,
                                                          const float* __restrict__ ca, const float* __restrict__ pooled,
                                                          const float* __restrict__ w1, const float* __restrict__ w2,
                                                          float* __restrict__ part, float* __restrict__ vec, const Geo G) {
  extern __shared__ __align__(16) float sm[];   // pav[C] | pmx[C] | ga[C] | hid[3r]
  const int b = blockIdx.x, C = G.C, r = G.r, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* pav = sm;
  float* pmx = sm + C;
  float* ga = sm + 2 * C;
  float* hid = sm + 3 * C;   // [0,2r): pre-activations, [2r,3r): u = W2^T g_a
  for (int c = tid; c < C; c += kT) {
    float gs = 0.f;
    if (gca_in) gs = gca_in[(size_t)b * C + c];
    else
      for (int k = 0; k < G.S; ++k) gs += gpart[((size_t)b * G.S + k) * C + c];
    const float a = ca[(size_t)b * C + c];
    ga[c] = gs * a * (1.f - a);
    pav[c] = pooled[(size_t)b * 2 * C + c];
    pmx[c] = pooled[(size_t)b * 2 * C + C + c];
  }
  __syncthreads();
  for (int j = warp; j < 3 * r; j += kWarps) {
    float acc = 0.f;
    if (j < 2 * r) {
      const float* wrow = w1 + (size_t)(j < r ? j : j - r) * C;
      const float* pv = j < r ? pav : pmx;
#pragma unroll 4
      for (int c = lane; c < C; c += 32) acc += wrow[c] * pv[c];
    } else {
      const float* wcol = w2 + (j - 2 * r);
#pragma unroll 4
      for (int c = lane; c < C; c += 32) acc += wcol[(size_t)c * r] * ga[c];
    }
    acc = warp_sum(acc);
    if (lane == 0) hid[j] = acc;
  }
  __syncthreads();
  float* gw = part + (size_t)b * 2 * r * C;   // per-image partials [r*C | C*r]
  for (int c = tid; c < C; c += kT) {
    const float gac = ga[c];
    float gpa = 0.f, gpm = 0.f;
    for (int j = 0; j < r; ++j) {
      const float ha = hid[j], hm = hid[r + j], u = hid[2 * r + j];
      const float gha = ha > 0.f ? u : 0.f, ghm = hm > 0.f ? u : 0.f;
      gw[(size_t)r * C + (size_t)c * r + j] = gac * (fmaxf(ha, 0.f) + fmaxf(hm, 0.f));  // g_W2[c,j]
      gw[(size_t)j * C + c] = gha * pav[c] + ghm * pmx[c];                              // g_W1[j,c]
      const float w = w1[(size_t)j * C + c];
      gpa += w * gha;
      gpm += w * ghm;
    }
    vec[(size_t)b * 2 * C + c] = gpa * G.invHW;
    vec[(size_t)b * 2 * C + C + c] = gpm;
  }
}

// ---- fin: g_x = (g sa + g_s0 + [c==argmax_c] g_s1) ca + g_pavg/HW (+ g_pmax at the pooled-max pixel) --------
// CA mode: g == nullptr -> g_x = g_pavg/HW (+ g_pmax).
template <typename T, int VW>
__global__ void __launch_bounds__(kT) cbam_bwd_fin_kernel(const T* __restrict__ g, const float* __restrict__ ca,
                                                          const float4* __restrict__ pixg, const float* __restrict__ vec,
                                                          const int* __restrict__ amx, T* __restrict__ gx, const Geo G) {
  extern __shared__ __align__(16) float sm[];   // cas[C] | gav[C]   (when a lane owns more than one channel vector)
  const int s = blockIdx.x, b = blockIdx.y, C = G.C, nch = G.nch, HW = G.HW;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int p0 = s * G.np, npix = min(G.np, HW - p0);
  const int LPP = G.lpp, PPW = 32 / LPP, sub = lane / LPP, sl = lane & (LPP - 1);
  const bool one = G.one != 0, full = g != nullptr;
  float* cas = sm;
  float* gavs = sm + C;
  float car[VW], gav[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) { car[e] = 0.f; gav[e] = 0.f; }
  if (one) {
    if (sl < nch) {
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        car[e] = ca[(size_t)b * C + sl * VW + e];
        gav[e] = vec[(size_t)b * 2 * C + sl * VW + e];
      }
    }
  } else {
    for (int c = tid; c < C; c += kT) { cas[c] = ca[(size_t)b * C + c]; gavs[c] = vec[(size_t)b * 2 * C + c]; }
    __syncthreads();
  }
  const T* gc = full ? g + ((size_t)b * HW + p0) * C : nullptr;
  T* og = gx + ((size_t)b * HW + p0) * C;
  const float4* pg = pixg + (size_t)b * HW + p0;
#pragma unroll 2
  for (int k = warp * PPW; k < npix; k += kWarps * PPW) {
    const int p = k + sub;
    if (p >= npix) continue;
    float4 pp = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
    if (full) pp = pg[p];
    const int am = __float_as_int(pp.w);
    for (int w = sl; w < nch; w += LPP) {
      float gv[VW], o[VW];
      if (full) Vec<T, VW>::load(gc + (size_t)p * C + w * VW, gv);
      if (!one) {
#pragma unroll
        for (int e = 0; e < VW; ++e) { car[e] = cas[w * VW + e]; gav[e] = gavs[w * VW + e]; }
      }
      const unsigned d = (unsigned)(am - w * VW);
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        float gx1 = 0.f;
        if (full) gx1 = gv[e] * pp.x + pp.y;
        o[e] = gx1 * car[e] + gav[e];
      }
      if (full && d < (unsigned)VW) {
#pragma unroll
        for (int e = 0; e < VW; ++e) o[e] += (d == (unsigned)e) ? pp.z * car[e] : 0.f;
      }
      Vec<T, VW>::store(og + (size_t)p * C + w * VW, o);
    }
  }
  __syncthreads();
  // the pooled-max pixel of each channel receives g_pmax on top (adaptive_max_pool2d backward, first occurrence)
  for (int c = tid; c < C; c += kT) {
    const int pm = amx[(size_t)b * C + c] - p0;
    if (pm >= 0 && pm < npix) {
      T* dst = og + (size_t)pm * C + c;
      *dst = DT<T>::from_f(DT<T>::to_f(*dst) + vec[(size_t)b * 2 * C + C + c]);
    }
  }
}

// fold the weight-gradient partials in a fixed order (deterministic): warp per output element, lanes over the
// partials (images for the MLP weights [B][n12], image slices for the conv taps [B*S][98]), shuffle tree
__global__ void __launch_bounds__(256) fold_partials_kernel(const float* __restrict__ part, const float* __restrict__ cpart,
                                                            float* gw1, float* gw2, float* gwsa, int B, int BS, int n1,
                                                            int n2, int ks) {
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int n = n1 + n2;
  if (i < n) {
    float acc = 0.f;
    for (int b = lane; b < B; b += 32) acc += part[(size_t)b * n + i];
    acc = warp_sum(acc);
    if (lane == 0) { if (i < n1) gw1[i] = acc; else gw2[i - n1] = acc; }
    return;
  }
  const int t = i - n;
  if (t >= 2 * ks * ks || !gwsa) return;
  const int j = t / (ks * ks), uu = (t / ks) % ks, vv = t % ks, o = (KS - ks) / 2;
  const int slot = (j * KS + uu + o) * KS + vv + o;
  float acc = 0.f;
  for (int k = lane; k < BS; k += 32) acc += cpart[(size_t)k * NT7 + slot];
  acc = warp_sum(acc);
  if (lane == 0) gwsa[t] = acc;
}

int check_common(const void* x, int B, int C, int H, int W, int r, int ksa, int dtype, int mode) {
  B200_REQUIRE(x, B200_ERR_SHAPE, "cbam: null input");
  B200_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, B200_ERR_SHAPE, "cbam: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
  B200_REQUIRE(B <= 65535, B200_ERR_SHAPE, "cbam: batch %d > 65535", B);
  B200_REQUIRE(mode >= 0 && mode <= 2, B200_ERR_SHAPE, "cbam: bad mode %d", mode);
  if (mode != B200_CBAM_SA) B200_REQUIRE(r > 0, B200_ERR_SHAPE, "cbam: hidden width r must be > 0");
  if (mode != B200_CBAM_CA) B200_REQUIRE(ksa == 3 || ksa == 7, B200_ERR_SHAPE, "cbam: kernel size must be 3 or 7 (cbam.py:43), got %d", ksa);
  if (dtype != B200_F32) B200_REQUIRE(C % 2 == 0, B200_ERR_ALIGN, "cbam: C must be even for 16-bit dtypes");
  B200_REQUIRE(((uintptr_t)x & 3) == 0, B200_ERR_ALIGN, "cbam: input must be 4-byte aligned");
  return B200_OK;
}

// pixel slices per image: ~24 KB of the feature map per CTA, at least 32 pixels
int splits(int C, int HW, size_t esize) {
  const int np = std::min(HW, std::max(32, (int)(24576 / ((size_t)C * esize))));
  return (HW + np - 1) / np;
}

void make_geo(Geo& G, int B, int C, int H, int W, int r, int ksa, int mode, int vw, size_t esize) {
  G.B = B; G.C = C; G.H = H; G.W = W; G.HW = H * W; G.r = r; G.ksa = ksa; G.mode = mode;
  G.nch = C / vw;
  G.lpp = 1;
  while (G.lpp < G.nch && G.lpp < 32) G.lpp <<= 1;
  G.one = G.nch <= G.lpp;
  G.S = splits(C, G.HW, esize);
  G.np = (G.HW + G.S - 1) / G.S;
  G.S = (G.HW + G.np - 1) / G.np;
  G.groups = G.nch >= kT ? 1 : kT / G.nch;
  G.tw = W + 2 * PADK;
  G.th = (G.np - 1) / W + 2 + 2 * PADK;
  G.invC = 1.f / (float)C;
  G.invHW = 1.f / (float)G.HW;
}

// forward workspace: slice partials [B][S][3][C] | ca [B][C] | maps [B][3][HW]
struct FwdWs { float* part; float* ca; float* maps; size_t bytes; };
FwdWs carve_fwd(void* base, int B, int C, int HW, int S) {
  char* p = (char*)base;
  FwdWs w;
  w.part = (float*)p; p += up256((size_t)B * S * 3 * C * 4);
  w.ca = (float*)p; p += up256((size_t)B * C * 4);
  w.maps = (float*)p; p += up256((size_t)B * 3 * HW * 4);
  w.bytes = (size_t)(p - (char*)base);
  return w;
}
// backward workspace: gz [B][HW] | pixg [B][HW] float4 | gpart [B][S][C] | vec [B][2][C] | part [B][2rC] | cpart [B][S][98]
struct BwdWs { float* gz; float4* pixg; float* gpart; float* vec; float* part; float* cpart; size_t bytes; };
BwdWs carve_bwd(void* base, int B, int C, int HW, int S, int r) {
  char* p = (char*)base;
  BwdWs w;
  w.gz = (float*)p; p += up256((size_t)B * HW * 4);
  w.pixg = (float4*)p; p += up256((size_t)B * HW * 16);
  w.gpart = (float*)p; p += up256((size_t)B * S * C * 4);
  w.vec = (float*)p; p += up256((size_t)B * 2 * C * 4);
  w.part = (float*)p; p += up256((size_t)B * 2 * r * C * 4);
  w.cpart = (float*)p; p += up256((size_t)B * S * NT7 * 4);
  w.bytes = (size_t)(p - (char*)base);
  return w;
}

template <typename K>
int ensure_smem(K kern, size_t bytes, const char* what) {
  if (bytes > 48 * 1024) {
    B200_REQUIRE(bytes <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "%s: shape needs %zu B of shared memory", what, bytes);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  }
  return B200_OK;
}

template <typename T, int VW>
int run_fwd(const void* x, const float* w1, const float* w2, const float* wsa, void* out, float* ca_out, float* sa_out,
            void* stash, void* workspace, const Geo& G, cudaStream_t st) {
  const FwdWs ws = carve_fwd(workspace, G.B, G.C, G.HW, G.S);
  Stash sh{nullptr, nullptr, ws.maps, 0};
  if (stash) sh = carve_stash(stash, G.B, G.C, G.HW);
  float* ca = ca_out ? ca_out : ws.ca;
  const dim3 grid(G.S, G.B);
  const T* xt = (const T*)x;
  if (G.mode != B200_CBAM_SA) {
    const size_t sm1 = (size_t)G.groups * G.C * 12;
    if (stash) {
      if (int rc = ensure_smem(cbam_pool_kernel<T, VW, true>, sm1, "cbam_fwd")) return rc;
      cbam_pool_kernel<T, VW, true><<<grid, kT, sm1, st>>>(xt, ws.part, G);
    } else {
      if (int rc = ensure_smem(cbam_pool_kernel<T, VW, false>, sm1, "cbam_fwd")) return rc;
      cbam_pool_kernel<T, VW, false><<<grid, kT, sm1, st>>>(xt, ws.part, G);
    }
    cbam_mlp_kernel<<<G.B, kT, (size_t)(2 * G.C + 2 * G.r) * 4, st>>>(ws.part, w1, w2, ca, sh.pooled, sh.amx, G);
    if (G.mode == B200_CBAM_CA) return check_launch("cbam_fwd");
  }
  const float* cap = G.mode == B200_CBAM_SA ? nullptr : ca;
  const size_t sm2 = G.one ? 0 : (size_t)G.C * 4;
  if (stash) cbam_map_kernel<T, VW, true><<<grid, kT, sm2, st>>>(xt, cap, sh.maps, G);
  else cbam_map_kernel<T, VW, false><<<grid, kT, sm2, st>>>(xt, cap, sh.maps, G);
  const size_t sm3 = (size_t)(NTAPS + 2 * G.th * G.tw + ((G.np + 3) & ~3) + (G.one ? 0 : G.C)) * 4;
  if (int rc = ensure_smem(cbam_gate_kernel<T, VW>, sm3, "cbam_fwd")) return rc;
  cbam_gate_kernel<T, VW><<<grid, kT, sm3, st>>>(xt, cap, sh.maps, wsa, G.mode == B200_CBAM_FULL ? (T*)out : nullptr, sa_out, G);
  return check_launch("cbam_fwd");
}

template <typename T, int VW>
int run_bwd(const void* g, const void* x, const float* w1, const float* w2, const float* wsa, const float* ca,
            const float* sa, void* stash, void* gx, float* gw1, float* gw2, float* gwsa, void* workspace, const Geo& G,
            cudaStream_t st) {
  const BwdWs ws = carve_bwd(workspace, G.B, G.C, G.HW, G.S, G.r);
  const Stash sh = carve_stash(stash, G.B, G.C, G.HW);
  const dim3 grid(G.S, G.B);
  const T* xt = (const T*)x;
  const size_t smc = G.one ? 0 : (size_t)G.C * 4;
  const int npad = (G.np + 3) & ~3;
  if (G.mode != B200_CBAM_CA) {
    const float* gzin = (const float*)g;   // SA mode: dL/dsa
    if (G.mode == B200_CBAM_FULL) {
      cbam_bwd_gz_kernel<T, VW><<<grid, kT, smc, st>>>(xt, (const T*)g, ca, sa, ws.gz, G);
      gzin = ws.gz;
    }
    const size_t smm = (size_t)(NTAPS + ((3 * G.th * G.tw + 3) & ~3) + npad * 4 + npad + npad + G.groups * G.C) * 4;
    if (int rc = ensure_smem(cbam_bwd_mid_kernel<T, VW>, smm, "cbam_bwd")) return rc;
    cbam_bwd_mid_kernel<T, VW><<<grid, kT, smm, st>>>(xt, G.mode == B200_CBAM_FULL ? (const T*)g : nullptr, gzin, sa, sh.maps,
                                                      wsa, G.mode == B200_CBAM_FULL ? ws.pixg : nullptr, ws.cpart, ws.gpart,
                                                      (T*)gx, G);
  }
  if (G.mode != B200_CBAM_SA) {
    cbam_mlp_bwd_kernel<<<G.B, kT, (size_t)(3 * G.C + 3 * G.r) * 4, st>>>(ws.gpart, G.mode == B200_CBAM_CA ? (const float*)g : nullptr, ca, sh.pooled, w1, w2, ws.part, ws.vec, G);
    cbam_bwd_fin_kernel<T, VW><<<grid, kT, 2 * smc, st>>>(G.mode == B200_CBAM_FULL ? (const T*)g : nullptr, ca, ws.pixg, ws.vec,
                                                          sh.amx, (T*)gx, G);
  }
  const int n1 = G.mode != B200_CBAM_SA ? G.r * G.C : 0, n2 = n1;
  const int outs = n1 + n2 + (G.mode != B200_CBAM_CA ? 2 * G.ksa * G.ksa : 0);
  fold_partials_kernel<<<(outs + 7) / 8, 256, 0, st>>>(ws.part, ws.cpart, gw1, gw2, G.mode != B200_CBAM_CA ? gwsa : nullptr, G.B,
                                                       G.B * G.S, n1, n2, G.ksa);
  return check_launch("cbam_bwd");
}

}  // namespace
}  // namespace b200

extern "C" B200_API size_t b200_cbam_stash_bytes(int32_t B, int32_t C, int32_t H, int32_t W) {
  return b200::carve_stash(nullptr, B, C, H * W).bytes;
}

extern "C" B200_API size_t b200_cbam_fwd_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W, int32_t dtype) {
  const size_t esize = dtype == B200_F32 ? 4 : 2;
  return b200::carve_fwd(nullptr, B, C, H * W, b200::splits(C, H * W, esize)).bytes;
}

extern "C" B200_API int b200_cbam_fwd(const void* x, const float* w1, const float* w2, const float* wsa, void* out,
                             float* ca_out, float* sa_out, void* stash, void* workspace, size_t workspace_bytes,
                             int32_t B, int32_t C, int32_t H, int32_t W, int32_t r, int32_t ksa, int32_t dtype,
                             int32_t mode, void* stream) {
  using namespace b200;
  if (mode == B200_CBAM_CA) ksa = 3;
  if (mode == B200_CBAM_SA) r = 1;
  if (int rc = check_common(x, B, C, H, W, r, ksa, dtype, mode)) return rc;
  if (mode != B200_CBAM_SA) B200_REQUIRE(w1 && w2, B200_ERR_SHAPE, "cbam_fwd: null MLP weights");
  if (mode != B200_CBAM_CA) B200_REQUIRE(wsa, B200_ERR_SHAPE, "cbam_fwd: null conv weight");
  if (mode == B200_CBAM_FULL) B200_REQUIRE(out, B200_ERR_SHAPE, "cbam_fwd: null output");
  if (mode == B200_CBAM_CA) B200_REQUIRE(ca_out, B200_ERR_SHAPE, "cbam_fwd: null ca output");
  if (mode == B200_CBAM_SA) B200_REQUIRE(sa_out, B200_ERR_SHAPE, "cbam_fwd: null sa output");
  const size_t need = b200_cbam_fwd_workspace_bytes(B, C, H, W, dtype);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "cbam_fwd: workspace %zu < %zu bytes", workspace_bytes, need);
  const size_t esize = dtype == B200_F32 ? 4 : 2;
  const int ve = 16 / (int)esize, ew = 4 / (int)esize;
  const bool vec16 = C % ve == 0 && ((uintptr_t)x & 15) == 0 && (mode != B200_CBAM_FULL || ((uintptr_t)out & 15) == 0);
  Geo G;
  make_geo(G, B, C, H, W, r, ksa, mode, vec16 ? ve : ew, esize);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec16) {   // one-launch resident cluster kernel when the image fits in cluster shared memory (cbam_cluster.cu)
    Stash sh{};
    if (stash) sh = carve_stash(stash, B, C, H * W);
    const int rc = cluster_fwd(x, w1, w2, wsa, out, ca_out, sa_out, stash ? &sh : nullptr, B, C, H, W, r, ksa, dtype, mode, ve, st);
    if (rc >= 0) return rc;
  }
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    constexpr int VE = Words<T>::VE, EW = Words<T>::EPL;
    if (vec16) return run_fwd<T, VE>(x, w1, w2, wsa, out, ca_out, sa_out, stash, workspace, G, st);
    return run_fwd<T, EW>(x, w1, w2, wsa, out, ca_out, sa_out, stash, workspace, G, st);
  });
}

extern "C" B200_API size_t b200_cbam_bwd_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W, int32_t r, int32_t dtype) {
  const size_t esize = dtype == B200_F32 ? 4 : 2;
  return b200::carve_bwd(nullptr, B, C, H * W, b200::splits(C, H * W, esize), r > 0 ? r : 1).bytes;
}

extern "C" B200_API int b200_cbam_bwd(const void* g, const void* x, const float* w1, const float* w2, const float* wsa,
                             const float* ca, const float* sa, const void* stash, void* gx, float* gw1, float* gw2,
                             float* gwsa, void* workspace, size_t workspace_bytes, int32_t B, int32_t C, int32_t H,
                             int32_t W, int32_t r, int32_t ksa, int32_t dtype, int32_t mode, void* stream) {
  using namespace b200;
  if (mode == B200_CBAM_CA) ksa = 3;
  if (mode == B200_CBAM_SA) r = 1;
  if (int rc = check_common(x, B, C, H, W, r, ksa, dtype, mode)) return rc;
  B200_REQUIRE(g && gx && stash, B200_ERR_SHAPE, "cbam_bwd: null gradient / stash pointer");
  if (mode != B200_CBAM_SA) B200_REQUIRE(w1 && w2 && ca && gw1 && gw2, B200_ERR_SHAPE, "cbam_bwd: null MLP weights / ca map / gradients");
  if (mode != B200_CBAM_CA) B200_REQUIRE(wsa && sa && gwsa, B200_ERR_SHAPE, "cbam_bwd: null conv weight / sa map / gradient");
  const size_t need = b200_cbam_bwd_workspace_bytes(B, C, H, W, r, dtype);
  B200_REQUIRE(workspace && workspace_bytes >= need, B200_ERR_WORKSPACE, "cbam_bwd: workspace %zu < %zu bytes", workspace_bytes, need);
  const size_t esize = dtype == B200_F32 ? 4 : 2;
  const int ve = 16 / (int)esize, ew = 4 / (int)esize;
  const bool vec16 = C % ve == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)gx & 15) == 0 &&
                     (mode != B200_CBAM_FULL || ((uintptr_t)g & 15) == 0);
  Geo G;
  make_geo(G, B, C, H, W, r, ksa, mode, vec16 ? ve : ew, esize);
  cudaStream_t st = (cudaStream_t)stream;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    constexpr int VE = Words<T>::VE, EW = Words<T>::EPL;
    if (vec16) return run_bwd<T, VE>(g, x, w1, w2, wsa, ca, sa, const_cast<void*>(stash), gx, gw1, gw2, gwsa, workspace, G, st);
    return run_bwd<T, EW>(g, x, w1, w2, wsa, ca, sa, const_cast<void*>(stash), gx, gw1, gw2, gwsa, workspace, G, st);
  });
}
