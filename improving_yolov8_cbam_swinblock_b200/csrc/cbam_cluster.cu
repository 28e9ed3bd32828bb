// CBAM forward, one launch: one thread-block CLUSTER per image with the image resident in shared memory.
// Replaces cbam.py:29-38 / :48-53 / :62-71 of the reference.  Used when the image fits in the shared memory of an
// 8- or 16-CTA cluster (the model's P5 use: 204 KB per image); other shapes run the streaming chain of cbam.cu.
//
// grid = CS x B, cluster = CS x 1.  The image (NHWC, so a pixel range is one contiguous byte range) is split into CS
// contiguous pixel chunks, one per CTA, and each chunk is pulled into shared memory ONCE by a 1-D bulk TMA copy
// (cp.async.bulk -> UBLKCP); everything else happens on chip, so HBM sees the algorithmic 1 read + 1 write:
//   A  per-channel sum / max (/ first argmax pixel) over the chunk; thread = one 16-byte channel vector
//      [cluster.sync]  rank k folds the partials of channel slice S_k over all ranks (DSMEM) and multiplies with
//                      W1[:, S_k]                          -> partial hidden activations
//      [cluster.sync]  all ranks sum the partial hiddens, rank k computes ca for S_k with W2[S_k, :]
//      [cluster.sync]  all ranks gather the full ca vector (DSMEM)
//   B  per-pixel mean_c / max_c (/ argmax_c) of x*ca, sub-warp per pixel, two pixels in flight -> map chunk in smem
//      [cluster.sync]  gather a zero-padded 2-D tile (rows of the chunk +-3, columns -3..W+3) of the map from the
//                      neighbouring ranks (DSMEM): the 7x7 taps then need no bounds checks
//   C  7x7 conv + sigmoid -> sa (4 lanes per pixel); out = x*ca*sa with packed 16-bit multiplies, 16-byte stores.
// All shape-dependent constants (chunking, lane mapping, shared-memory offsets) come from the host (`Plan`): a CTA
// owns ~50 pixels at the model's shape, so scalar set-up code is what the kernel's latency is made of.
// With a stash the kernel also writes the by-products the (streaming) backward of cbam.cu consumes.
#include <cooperative_groups.h>

#include <map>
#include <mutex>
#include <tuple>

#include "cbam.cuh"

namespace cg = cooperative_groups;

namespace b200 {
namespace cbam {
namespace {

struct Plan {
  int B, C, H, W, HW, r, ksa, mode;
  int cs, pchunk, nch, lpp, groups, th, tw, cper;
  float invC, invHW;
  // shared-memory byte offsets
  int xs, psum, pmax, pidx, pav, pmx, hpart, hid, ca, smap, tile, sas, wsa, red, bar, total;
};

struct Params {
  const void* x;
  void* out;
  const float* w1;
  const float* w2;
  const float* wsa;
  float* ca;      // [B][C] (nullable)
  float* sa;      // [B][HW] (nullable)
  float* pooled;  // stash (nullable as a group)
  int* amx;
  float* maps;
  Plan pl;
};

template <typename T, int VW, bool IDX>
__device__ __forceinline__ void channel_partials(const T* xc, int np, int p0, int C, int nw, int groups, float* psum,
                                                 float* pmax, int* pidx, float* red) {
  const int tpg = nw < kT ? nw : kT;   // threads per pixel group
  const int pg = threadIdx.x / tpg, tw = threadIdx.x - pg * tpg;
  for (int w = tw; w < nw; w += kT) {
    float s[VW], m[VW];
    int mi[VW];
#pragma unroll
    for (int e = 0; e < VW; ++e) { s[e] = 0.f; m[e] = -INFINITY; mi[e] = p0; }
    if (pg < groups) {
      const T* src = xc + w * VW;
#pragma unroll 2
      for (int p = pg; p < np; p += groups) {
        const VPack<T, VW> k = *reinterpret_cast<const VPack<T, VW>*>(src + (size_t)p * C);
#pragma unroll
        for (int e = 0; e < VW; ++e) {
          const float v = DT<T>::to_f(k.e[e]);
          s[e] += v;
          if (IDX) {
            if (v > m[e]) { m[e] = v; mi[e] = p0 + p; }
          } else {
            m[e] = fmaxf(m[e], v);
          }
        }
      }
      float* rs = red + (size_t)pg * C * 3;
#pragma unroll
      for (int e = 0; e < VW; ++e) {
        rs[w * VW + e] = s[e];
        rs[C + w * VW + e] = m[e];
        if (IDX) reinterpret_cast<int*>(rs)[2 * C + w * VW + e] = mi[e];
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += kT) {
    float s = 0.f, m = -INFINITY;
    int mi = p0;
    for (int gi = 0; gi < groups; ++gi) {  // groups interleave pixels: combine by (value, then smaller index)
      const float* rs = red + (size_t)gi * C * 3;
      s += rs[c];
      const float v = rs[C + c];
      if (IDX) {
        const int vi = reinterpret_cast<const int*>(rs)[2 * C + c];
        if (v > m || (v == m && vi < mi && v != -INFINITY)) { m = v; mi = vi; }
      } else {
        m = fmaxf(m, v);
      }
    }
    psum[c] = s; pmax[c] = m;
    if (IDX) pidx[c] = mi;
  }
}

template <typename T, int VW, bool IDX>
__global__ void __launch_bounds__(kT) cbam_cluster_fwd_kernel(const __grid_constant__ Params P) {
  cg::cluster_group cluster = cg::this_cluster();
  const Plan& L = P.pl;
  const int CS = L.cs, rank = blockIdx.x, b = blockIdx.y;
  const int C = L.C, HW = L.HW, W = L.W, r = L.r, nch = L.nch, pc = L.pchunk;
  const int p0 = min(rank * pc, HW), p1 = min(p0 + pc, HW), np = p1 - p0;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  T* xs = reinterpret_cast<T*>(smem_raw + L.xs);
  float* psum = reinterpret_cast<float*>(smem_raw + L.psum);
  float* pmax = reinterpret_cast<float*>(smem_raw + L.pmax);
  int* pidx = reinterpret_cast<int*>(smem_raw + L.pidx);
  float* pav = reinterpret_cast<float*>(smem_raw + L.pav);     // slice-owner: pooled avg of the slice
  float* pmx = reinterpret_cast<float*>(smem_raw + L.pmx);
  float* hpart = reinterpret_cast<float*>(smem_raw + L.hpart); // this rank's partial hidden pre-activations [2][r]
  float* hid = reinterpret_cast<float*>(smem_raw + L.hid);
  float* ca = reinterpret_cast<float*>(smem_raw + L.ca);
  float* smap = reinterpret_cast<float*>(smem_raw + L.smap);
  float* tile = reinterpret_cast<float*>(smem_raw + L.tile);
  float* sas = reinterpret_cast<float*>(smem_raw + L.sas);
  float* wsas = reinterpret_cast<float*>(smem_raw + L.wsa);
  float* red = reinterpret_cast<float*>(smem_raw + L.red);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + L.bar);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const T* xg = reinterpret_cast<const T*>(P.x) + ((size_t)b * HW + p0) * C;
  {
    const uint32_t bytes = (uint32_t)((size_t)np * C * sizeof(T));   // host guarantees 16-byte multiples / alignment
    if (tid == 0) {
      mbar_init(bar, 1);
      fence_mbar_init();
      if (bytes) {
        mbar_expect_tx(bar, bytes);
        for (uint32_t off = 0; off < bytes; off += 32768)
          bulk_g2s(reinterpret_cast<char*>(xs) + off, reinterpret_cast<const char*>(xg) + off,
                   (bytes - off) > 32768 ? 32768 : (bytes - off), bar);
      }
    }
    load_taps(wsas, P.wsa, L.ksa);   // overlaps the bulk copy
    __syncthreads();                 // mbarrier init + taps visible
    if (bytes) mbar_wait(bar, 0);
  }
  const T* xc = xs;
  const int cper = L.cper, cs0 = min(rank * cper, C), cs1 = min(cs0 + cper, C);

  if (L.mode != B200_CBAM_SA) {
    channel_partials<T, VW, IDX>(xc, np, p0, C, nch, L.groups, psum, pmax, pidx, red);
    cluster.sync();  // (1) partials visible cluster-wide
    // slice owner: fold the slice over the ranks -> pooled avg / max (cbam.py:8-9), partial hidden = W1[:, S] . pooled[S]
    for (int c = cs0 + tid; c < cs1; c += kT) {
      float s = 0.f, m = -INFINITY;
      int mi = 0;
      for (int k2 = 0; k2 < CS; ++k2) {        // ranks ascend in pixel order, strict >: first occurrence
        s += cluster.map_shared_rank(psum, k2)[c];
        const float v = cluster.map_shared_rank(pmax, k2)[c];
        if (v > m || k2 == 0) { m = v; if (IDX) mi = cluster.map_shared_rank(pidx, k2)[c]; }
      }
      const float a = s * L.invHW, mm = (s != s) ? s : m;   // a NaN anywhere in the channel makes the pooled max NaN too
      pav[c - cs0] = a;
      pmx[c - cs0] = mm;
      if (IDX) {
        P.pooled[(size_t)b * 2 * C + c] = a;
        P.pooled[(size_t)b * 2 * C + C + c] = mm;
        P.amx[(size_t)b * C + c] = mi;
      }
    }
    __syncthreads();
    for (int j = warp; j < 2 * r; j += kWarps) {  // j < r: avg branch, j >= r: max branch
      const float* wrow = P.w1 + (size_t)(j < r ? j : j - r) * C;
      const float* src = j < r ? pav : pmx;
      float acc = 0.f;
      for (int c = cs0 + lane; c < cs1; c += 32) acc += wrow[c] * src[c - cs0];
      acc = warp_sum(acc);
      if (lane == 0) hpart[j] = acc;
    }
    cluster.sync();  // (2) partial hiddens visible
    for (int j = tid; j < 2 * r; j += kT) {
      float acc = 0.f;
      for (int k2 = 0; k2 < CS; ++k2) acc += cluster.map_shared_rank(hpart, k2)[j];
      hid[j] = relu_nan(acc);  // ReLU (cbam.py:25)
    }
    __syncthreads();
    for (int c = cs0 + tid; c < cs1; c += kT) {
      const float* wrow = P.w2 + (size_t)c * r;
      float z = 0.f;
#pragma unroll 4
      for (int j = 0; j < r; ++j) z += wrow[j] * (hid[j] + hid[r + j]);
      const float a = sigmoidf_(z);
      ca[c] = a;  // own slice goes straight to its final place; peers read it from `ca` of this rank
      if (P.ca) P.ca[(size_t)b * C + c] = a;
    }
    cluster.sync();  // (3) every rank's ca slice visible
    for (int c = tid; c < C; c += kT) {
      const int owner = min(c / cper, CS - 1);
      if (owner != rank) ca[c] = cluster.map_shared_rank(ca, owner)[c];
    }
    __syncthreads();
    if (L.mode == B200_CBAM_CA) { cluster.sync(); return; }
  } else {
    for (int c = tid; c < C; c += kT) ca[c] = 1.f;
    __syncthreads();
  }

  // ---- phase B: per-pixel channel mean / max of x*ca (sub-warp of LPP lanes per pixel, 2 pixels in flight) ------
  const int LPP = L.lpp, PPW = 32 / LPP, sub = lane / LPP, sl = lane & (LPP - 1);
  const bool one = nch <= LPP;   // one chunk per lane: its ca values stay in registers
  float car[VW];
#pragma unroll
  for (int e = 0; e < VW; ++e) car[e] = (one && sl < nch) ? ca[sl * VW + e] : 0.f;
  {
    constexpr int U = 2;
    float* mg = IDX ? P.maps + (size_t)b * 3 * HW + p0 : nullptr;
    for (int k = warp * PPW; k < np; k += U * kWarps * PPW) {
      float sum[U], mx[U];
      int mi[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int p = k + u * kWarps * PPW + sub;
        sum[u] = 0.f; mx[u] = -INFINITY; mi[u] = 0x7fffffff;
        if (p < np) {
          for (int w = sl; w < nch; w += LPP) {
            const VPack<T, VW> kk = *reinterpret_cast<const VPack<T, VW>*>(xc + (size_t)p * C + w * VW);
            if (!one) {
#pragma unroll
              for (int e = 0; e < VW; ++e) car[e] = ca[w * VW + e];
            }
#pragma unroll
            for (int e = 0; e < VW; ++e) {
              const float t = DT<T>::to_f(kk.e[e]) * car[e];
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
      // lmx = this lane's own maximum.  The lanes hold ascending channel ranges, so the FIRST lane whose own maximum equals
      // the reduced one owns the first arg-max channel: one ballot instead of an index butterfly
      float lmx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) lmx[u] = mx[u];
      for (int o = LPP >> 1; o > 0; o >>= 1) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          sum[u] += __shfl_xor_sync(0xffffffffu, sum[u], o);
          mx[u] = fmaxf(mx[u], __shfl_xor_sync(0xffffffffu, mx[u], o));
        }
      }
      if (IDX) {
        const unsigned submask = (LPP == 32 ? 0xffffffffu : ((1u << LPP) - 1u)) << (sub * LPP);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const unsigned hit = __ballot_sync(0xffffffffu, lmx[u] == mx[u]) & submask;
          mi[u] = __shfl_sync(0xffffffffu, mi[u], hit ? __ffs(hit) - 1 : (int)(sub * LPP));
        }
      }
      if (sl == 0) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int p = k + u * kWarps * PPW + sub;
          if (p < np) {
            const float mean = sum[u] * L.invC;
            smap[p] = mean;
            smap[pc + p] = mx[u];
            if (IDX) {
              mg[p] = mean;
              mg[HW + p] = mx[u];
              reinterpret_cast<int*>(mg)[2 * HW + p] = mi[u] == 0x7fffffff ? 0 : mi[u];
            }
          }
        }
      }
    }
  }
  cluster.sync();  // (4) map chunks visible
  const int ya = p0 / W, tw = L.tw;
  const int nrow = (np > 0 ? (p1 - 1) / W - ya + 1 : 0) + 2 * PADK;
  for (int row = warp; row < 2 * nrow; row += kWarps) {   // zero-padded tiles of both maps, gathered over DSMEM
    const int j = row >= nrow ? 1 : 0, ty = row - j * nrow, y = ya - PADK + ty;
    float* dst = tile + (size_t)(j * L.th + ty) * tw;
    for (int tx = lane; tx < tw; tx += 32) {
      const int xx = tx - PADK;
      float v = 0.f;
      if (y >= 0 && y < L.H && xx >= 0 && xx < W) {
        const int q = y * W + xx;
        const int owner = min(q / pc, CS - 1);
        v = cluster.map_shared_rank(smap, owner)[j * pc + (q - owner * pc)];
      }
      dst[tx] = v;
    }
  }
  __syncthreads();
  // ---- phase C: 7x7 conv + sigmoid; 4 lanes per pixel split the 14 tap rows, taps broadcast as float4 ------------
  for (int base = warp * 32; base < np * 4; base += kT) {
    const int i = base + lane, p = i >> 2, part = i & 3;
    float z = 0.f;
    if (p < np) {
      const int q = p0 + p, y = q / W, xx = q - y * W;
      const float* t0 = tile + (size_t)(y - ya) * tw + xx;
      for (int rr = part; rr < 2 * KS; rr += 4) {       // rr = ch*7 + u
        const int ch = rr >= KS ? 1 : 0, u = rr - ch * KS;
        const float4 wa = *reinterpret_cast<const float4*>(wsas + rr * KROW);
        const float4 wb = *reinterpret_cast<const float4*>(wsas + rr * KROW + 4);
        const float* tr = t0 + (size_t)(ch * L.th + u) * tw;
        z += wa.x * tr[0] + wa.y * tr[1] + wa.z * tr[2] + wa.w * tr[3] + wb.x * tr[4] + wb.y * tr[5] + wb.z * tr[6];
      }
    }
    z += __shfl_xor_sync(0xffffffffu, z, 1);
    z += __shfl_xor_sync(0xffffffffu, z, 2);
    if (part == 0 && p < np) {
      const float a = sigmoidf_(z);
      sas[p] = a;
      if (P.sa) P.sa[(size_t)b * HW + p0 + p] = a;
    }
  }
  __syncthreads();
  if (L.mode == B200_CBAM_FULL) {
    T* og = reinterpret_cast<T*>(P.out) + ((size_t)b * HW + p0) * C;
    if constexpr (sizeof(T) == 2 && VW == 8) {
      // packed 16-bit gate: out = (x*ca)*sa, rounded after each product exactly like the 16-bit reference ops
      using P2 = typename Pair2<T>::type;
      P2 ca2[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) ca2[i] = make_pair(T(), car[2 * i], car[2 * i + 1]);
#pragma unroll 2
      for (int k = warp * PPW; k < np; k += kWarps * PPW) {
        const int p = k + sub;
        if (p >= np) continue;
        const float sp = sas[p];
        const P2 sp2 = make_pair(T(), sp, sp);
        for (int w = sl; w < nch; w += LPP) {
          uint4 raw = *reinterpret_cast<const uint4*>(xc + (size_t)p * C + w * VW);
          P2* rp = reinterpret_cast<P2*>(&raw);
          if (!one) {
#pragma unroll
            for (int i = 0; i < 4; ++i) ca2[i] = make_pair(T(), ca[w * VW + 2 * i], ca[w * VW + 2 * i + 1]);
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) rp[i] = __hmul2(__hmul2(rp[i], ca2[i]), sp2);
          stg_stream16(og + (size_t)p * C + w * VW, raw);
        }
      }
    } else {
      for (int k = warp * PPW; k < np; k += kWarps * PPW) {
        const int p = k + sub;
        if (p >= np) continue;
        const float sp = sas[p];
        for (int w = sl; w < nch; w += LPP) {
          const VPack<T, VW> kk = *reinterpret_cast<const VPack<T, VW>*>(xc + (size_t)p * C + w * VW);
          float v[VW];
#pragma unroll
          for (int e = 0; e < VW; ++e) v[e] = DT<T>::to_f(kk.e[e]) * (one ? car[e] : ca[w * VW + e]) * sp;
          Vec<T, VW>::store(og + (size_t)p * C + w * VW, v);
        }
      }
    }
  }
  cluster.sync();  // keep smem alive until every peer finished its DSMEM reads
}

void layout(Plan& L, size_t esize) {
  const int C = L.C, r = L.r, pc = L.pchunk;
  L.tw = L.W + 2 * PADK;
  L.th = (pc - 1) / L.W + 2 + 2 * PADK;
  size_t o = 0;
  auto take = [&](size_t bytes) { const int at = (int)o; o += (bytes + 15) & ~(size_t)15; return at; };
  L.xs = take((size_t)pc * C * esize);
  L.psum = take((size_t)C * 4);
  L.pmax = take((size_t)C * 4);
  L.pidx = take((size_t)C * 4);
  L.pav = take((size_t)L.cper * 4);
  L.pmx = take((size_t)L.cper * 4);
  L.hpart = take((size_t)2 * r * 4);
  L.hid = take((size_t)2 * r * 4);
  L.ca = take((size_t)C * 4);
  L.smap = take((size_t)pc * 4 * 2);
  L.tile = take((size_t)L.th * L.tw * 4 * 2);
  L.sas = take((size_t)pc * 4);
  L.wsa = take((size_t)NTAPS * 4);
  L.red = take((size_t)L.groups * C * 12);
  L.bar = take(16);
  L.total = (int)o;
}

template <typename K>
int launch(K kern, const Params& P, cudaStream_t st) {
  const Plan& L = P.pl;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total);
  if (L.cs > 8) cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(L.cs, L.B);
  cfg.blockDim = dim3(kT);
  cfg.dynamicSmemBytes = L.total;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = L.cs;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  // can this device co-schedule one such cluster at all (MIG slices, small GPCs, 16-CTA non-portable clusters)?  Asked once
  // per (kernel, cluster size, smem); 0 or a failed launch -> -1 = "not taken", the caller runs the streaming chain (cbam.cu)
  static std::mutex mu;
  static std::map<std::tuple<const void*, int, int, int>, int> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  int nclusters = 0;
  {
    std::lock_guard<std::mutex> lk(mu);
    auto key = std::make_tuple((const void*)kern, L.cs, L.total, dev);
    auto it = cache.find(key);
    if (it == cache.end()) {
      if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg) != cudaSuccess) { nclusters = 0; cudaGetLastError(); }
      cache.emplace(key, nclusters);
    } else {
      nclusters = it->second;
    }
  }
  if (nclusters <= 0) return -1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, P);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return check_launch("cbam_fwd");
}

}  // namespace

int cluster_fwd(const void* x, const float* w1, const float* w2, const float* wsa, void* out, float* ca_out, float* sa_out,
                const Stash* stash, int B, int C, int H, int W, int r, int ksa, int dtype, int mode, int vw, cudaStream_t st) {
  const size_t esize = dtype == B200_F32 ? 4 : 2;
  if ((size_t)vw * esize != 16) return -1;   // the resident kernel is the 16-byte-vector path only
  Params P{x, out, w1, w2, wsa, ca_out, sa_out, stash ? stash->pooled : nullptr, stash ? stash->amx : nullptr,
           stash ? stash->maps : nullptr, {}};
  Plan& L = P.pl;
  L.B = B; L.C = C; L.H = H; L.W = W; L.HW = H * W; L.r = r; L.ksa = ksa; L.mode = mode;
  L.nch = C / vw;
  L.lpp = 1;
  while (L.lpp < L.nch && L.lpp < 32) L.lpp <<= 1;
  L.groups = L.nch >= kT ? 1 : std::min(kT / L.nch, std::max(1, 13312 / (C * 12)));   // keeps 4 CTAs per SM at C=256
  L.invC = 1.f / (float)C;
  L.invHW = 1.f / (float)L.HW;
  // whole image in the shared memory of one cluster, at least two CTAs per SM so the phases of different clusters
  // overlap; bulk copies need 16-byte chunk sizes
  bool ok = false;
  for (int c : {8, 16}) {
    L.cs = c; L.pchunk = (L.HW + c - 1) / c; L.cper = (C + c - 1) / c;
    if (((size_t)L.pchunk * C * esize) % 16) continue;
    layout(L, esize);
    if (L.total <= 100 * 1024) { ok = true; break; }
  }
  if (!ok) return -1;
  return B200_DISPATCH_DTYPE(dtype, [&]() -> int {
    constexpr int VE = Words<T>::VE;
    return stash ? launch(cbam_cluster_fwd_kernel<T, VE, true>, P, st) : launch(cbam_cluster_fwd_kernel<T, VE, false>, P, st);
  });
}

}  // namespace cbam
}  // namespace b200
