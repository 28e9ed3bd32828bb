// Fused attention half of the SwinBlock on tcgen05 tensor cores (bf16 / f16, C = 128, 2 heads of 64, L = ws*ws <= 64, no shift):
//     y1 = n1 + out_proj(MHSA(n1)),   n1 = LayerNorm1(window tokens of zero-padded x)            (swin_block.py:41-52)
// One kernel replaces F.pad + rearrange + window_partition + norm1 + nn.MultiheadAttention (packed in_proj, two bmm, softmax,
// out_proj) + the residual add + window_reverse + the crop for this half: q / k / v / the scores / the attention output never
// leave the SM, and y1 is written straight in pixel order (what the fused MLP kernel, csrc/swin_mlp.cu, consumes).
//
// Work unit = a PAIR of windows stacked in one 128-row UMMA tile (rows [0,L) = window 2p, rows [64,64+L) = window 2p+1; the other
// rows stay zero for the whole kernel).  Per tile:
//   TMA    the two windows of x arrive as 4-D boxes [1, ws, ws, 64 ch] of the NHWC map: ws*ws consecutive 128-byte rows = the
//          K-major A operand; out-of-bounds pixels are zero-filled by the TMA unit = the reference's zero padding BEFORE LayerNorm
//   LN     row threads: statistics -> n1 (16 bit, in place)
//   MMA    QKV[128 x 384] = n1 * W_in^T      (W_in / W_out streamed through a 4-stage TMA ring of [128 x 64] blocks, L2 resident)
//   SIMT   + b_in -> 16 bit -> six K-major tiles Q_h, K_h, V_h [128 x 64]
//   MMA    S_h = Q_h K_h^T (both heads; only the two diagonal 64x64 blocks are meaningful)
//   SIMT   thread = (row, head): scale, mask keys >= L, exp2 softmax in registers, un-normalised P_h (16 bit, block diagonal) over
//          the dead Q_h / K_h tiles
//   MMA    O_h = P_h V_h                     (V_h tile as written, MN-major descriptor)
//   SIMT   O_h / rowsum -> 16 bit over the dead V_h tiles = the K-major A operand of
//   MMA    Y = O * W_out^T
//   SIMT   Y + b_out + n1 (residual, re-read from the A tile) -> 16 bit, in place -> TMA 4-D box stores into y1 (NHWC): pixels
//          outside the map are clipped by the TMA unit = the reference's crop
// In training the by-products the (unfused) backward consumes also leave through TMA stores: n1, qkv, o in token order, plus
// lse / mean / rstd.  TMEM: QKV 384 columns (S aliases q|k, O aliases v) + Y 128 columns.
#include "tc.cuh"

namespace b200 {
namespace tc {
namespace {

constexpr int kC = 128, kHD = 64;
constexpr int kLnWarps = 4, kFinWarps = 4, kWorkWarps = 16;
constexpr int kFirstLnWarp = 3, kFirstFinWarp = kFirstLnWarp + kLnWarps, kFirstWorkWarp = kFirstFinWarp + kFinWarps;
constexpr int kThreads = 32 * (kFirstWorkWarp + kWorkWarps);   // 864
constexpr int kRing = 4;
constexpr int kBlk = 128 * 128;                                // 16 KB: one [128 rows][128 B] operand block
constexpr int kTile = 2 * kBlk;                                // 32 KB: [2 K-blocks][128 rows][128 B]

struct ABSmem {
  static constexpr int OFF_A = 0;                  // 2 x 32 KB: x windows -> n1 (A of QKV) -> y1 staging
  static constexpr int OFF_T = OFF_A + 2 * kTile;  // 6 x 16 KB: Q0 Q1 K0 K1 V0 V1 (P_h over Q_h|K_h, O_h over V_h)
  static constexpr int OFF_W = OFF_T + 6 * kBlk;   // kRing x 16 KB weight blocks
  static constexpr int OFF_BI = OFF_W + kRing * kBlk;   // b_in [384] f32
  static constexpr int OFF_BO = OFF_BI + 3 * kC * 4;    // b_out [128] f32
  static constexpr int OFF_BAR = OFF_BO + kC * 4;
  static constexpr int TOTAL = OFF_BAR + 256;
};
static_assert(ABSmem::TOTAL <= 232448, "shared memory budget");

struct ABParams {
  const float *gamma, *beta, *b_in, *b_out;
  float *lse, *mean, *rstd;     // training by-products (null: inference)
  long long* dbg;               // optional timeline of CTA 0 (profiles/attn_block_timeline.py)
  int nwin, n_tiles, L, ws, nWh, nWw, train;
  float scale_log2, eps;
};

// debug timeline (CTA 0 only, dbg != nullptr): event e in [0,16), tile index i < 16
__device__ __forceinline__ void stamp(const ABParams& P, int e, int i) {
  if (P.dbg != nullptr && blockIdx.x == 0 && i < 16) {
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t));
    P.dbg[e * 16 + i] = t;
  }
}

template <int FMT> __device__ __forceinline__ uint32_t pack2h(float lo, float hi) {
  if (FMT == 1) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
  }
  __half2 p = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}
template <int FMT> __device__ __forceinline__ float up_lo(uint32_t w) {
  return FMT == 1 ? __uint_as_float(w << 16) : __half2float(__ushort_as_half((unsigned short)(w & 0xffff)));
}
template <int FMT> __device__ __forceinline__ float up_hi(uint32_t w) {
  return FMT == 1 ? __uint_as_float(w & 0xffff0000u) : __half2float(__ushort_as_half((unsigned short)(w >> 16)));
}
// 16-byte chunk c (0..15) of row `row` of a [2 K-blocks][128 rows][128 B] swizzled tile
__device__ __forceinline__ uint4* row_chunk(unsigned char* tile, int row, int c) {
  return reinterpret_cast<uint4*>(tile + (c >> 3) * kBlk + sw128_offset(row, c & 7));
}

template <int FMT>
__global__ void __launch_bounds__(kThreads, 1)
swin_attn_block_fwd_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
                           const __grid_constant__ CUtensorMap tmWin, const __grid_constant__ CUtensorMap tmWo,
                           const __grid_constant__ CUtensorMap tmN1, const __grid_constant__ CUtensorMap tmQKV,
                           const __grid_constant__ CUtensorMap tmO, ABParams P) {
  using S = ABSmem;
  extern __shared__ __align__(1024) unsigned char smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  float* sbi = reinterpret_cast<float*>(smem + S::OFF_BI);
  float* sbo = reinterpret_cast<float*>(smem + S::OFF_BO);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BAR);
  uint64_t* x_full = bars;              // [2] x windows landed (TMA)
  uint64_t* n1_ready = bars + 2;        // [2] n1 written (128 LayerNorm threads)
  uint64_t* a_free = bars + 4;          // [2] A buffer reusable (y1 stores have read it)
  uint64_t* n1_stored = bars + 6;       // [2] the n1 by-product stores have read the A buffer: it may become the y1 staging tile
  uint64_t* w_full = bars + 8;          // [kRing]
  uint64_t* w_empty = w_full + kRing;
  uint64_t* qkv_full = w_empty + kRing; // QKV accumulator complete (commit)
  uint64_t* qk_ready = qkv_full + 1;    // Q/K/V tiles written (512 worker threads)
  uint64_t* s_full = qkv_full + 2;      // S accumulators complete (commit)
  uint64_t* p_ready = qkv_full + 3;     // P tiles written (256 softmax threads)
  uint64_t* o_full = qkv_full + 4;      // O accumulators complete (commit)
  uint64_t* o_ready = qkv_full + 5;     // O tiles written (256 threads)
  uint64_t* y_full = qkv_full + 6;      // Y accumulator complete (commit): also "out_proj has read the O tiles"
  uint64_t* y_free = qkv_full + 7;      // Y accumulator read back (128 final threads)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(qkv_full + 8);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_local = (int)blockIdx.x < P.n_tiles ? (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int L = P.L;
  auto abuf = [&](int b) { return smem + S::OFF_A + b * kTile; };
  auto tbuf = [&](int i) { return smem + S::OFF_T + i * kBlk; };   // 0,1 = Q_h; 2,3 = K_h; 4,5 = V_h
  // window `win` -> (image, first pixel row, first pixel column)
  auto win_origin = [&](int win, int* b, int* y0, int* x0) {
    const int ww = win % P.nWw, q = win / P.nWw;
    *b = q / P.nWh; *y0 = (q % P.nWh) * P.ws; *x0 = ww * P.ws;
  };

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmX); prefetch_tmap(&tmY); prefetch_tmap(&tmWin); prefetch_tmap(&tmWo);
    if (P.train) { prefetch_tmap(&tmN1); prefetch_tmap(&tmQKV); prefetch_tmap(&tmO); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&x_full[i], 1); mbar_init(&n1_ready[i], 32 * kLnWarps); mbar_init(&a_free[i], 1); mbar_init(&n1_stored[i], 1);
    }
    for (int i = 0; i < kRing; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    mbar_init(qkv_full, 1); mbar_init(qk_ready, 32 * kWorkWarps); mbar_init(s_full, 1); mbar_init(p_ready, 16 * kWorkWarps);
    mbar_init(o_full, 1); mbar_init(o_ready, 16 * kWorkWarps); mbar_init(y_full, 1); mbar_init(y_free, 32 * kFinWarps);
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  // rows L..63 of each half of the A tiles are never written: zero once (zero rows -> zero Q/K/V rows before the bias)
  for (int i = threadIdx.x; i < 2 * kTile / 16; i += kThreads) reinterpret_cast<uint4*>(smem + S::OFF_A)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 3 * kC; i += kThreads) sbi[i] = P.b_in[i];
  for (int i = threadIdx.x; i < kC; i += kThreads) sbo[i] = P.b_out[i];
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tQKV = tmem_base, tS = tmem_base, tO = tmem_base + 256, tY = tmem_base + 384;

  if (warp == 0) {
    // ===================== weight producer: per tile Wq, Wk, Wv (rows 0/128/256 of W_in) then W_out, two K blocks each =====================
    if (elect_one()) {
      int st = 0; uint32_t ph = 0;
      for (int n = 0; n < n_local; ++n)
        for (int c = 0; c < 8; ++c) {
          mbar_wait(&w_empty[st], ph ^ 1);
          mbar_expect_tx(&w_full[st], kBlk);
          if (c < 6) tma_load_2d(smem + S::OFF_W + st * kBlk, &tmWin, &w_full[st], (c & 1) * 64, (c >> 1) * 128);
          else tma_load_2d(smem + S::OFF_W + st * kBlk, &tmWo, &w_full[st], (c & 1) * 64, 0);
          if (++st == kRing) { st = 0; ph ^= 1; }
        }
    }
  } else if (warp == 2) {
    // ===================== x window loader =====================
    if (elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int b = n & 1;
        const int tile = blockIdx.x + n * gridDim.x;
        mbar_wait(&a_free[b], ((n >> 1) & 1) ^ 1);
        const int nw = (2 * tile + 1 < P.nwin) ? 2 : 1;
        mbar_expect_tx(&x_full[b], (uint32_t)(nw * 2 * L * 128));
        for (int w = 0; w < nw; ++w) {
          int bi, y0, x0;
          win_origin(2 * tile + w, &bi, &y0, &x0);
          tma_load_4d(abuf(b) + w * 64 * 128, &tmX, &x_full[b], 0, x0, y0, bi);
          tma_load_4d(abuf(b) + kBlk + w * 64 * 128, &tmX, &x_full[b], 64, x0, y0, bi);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      const uint32_t id128 = idesc_f16(128, 128, FMT), id_pv = idesc_f16(128, 64, FMT, 0, 1);
      int st = 0; uint32_t ph = 0;
      for (int n = 0; n < n_local; ++n) {
        const int b = n & 1;
        const uint32_t tp = n & 1;       // parity of the once-per-tile barriers
        // ---- QKV = n1 * W_in^T ----
        mbar_wait(&n1_ready[b], (n >> 1) & 1);
        fence_after_sync();
        stamp(P, 0, n);
        for (int c = 0; c < 6; ++c) {
          mbar_wait(&w_full[st], ph);
          fence_after_sync();
          const uint64_t da = smem_desc_k_sw128(abuf(b) + (c & 1) * kBlk), db = smem_desc_k_sw128(smem + S::OFF_W + st * kBlk);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tQKV + (c >> 1) * 128, da + 2 * k, db + 2 * k, id128, ((c & 1) | k) ? 1u : 0u);
          umma_commit(&w_empty[st]);
          if (++st == kRing) { st = 0; ph ^= 1; }
        }
        umma_commit(qkv_full);
        stamp(P, 1, n);
        // ---- S_h = Q_h K_h^T ----
        mbar_wait(qk_ready, tp);
        fence_after_sync();
        stamp(P, 2, n);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint64_t da = smem_desc_k_sw128(tbuf(h)), db = smem_desc_k_sw128(tbuf(2 + h));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tS + h * 128, da + 2 * k, db + 2 * k, id128, k ? 1u : 0u);
        }
        umma_commit(s_full);
        // ---- O_h = P_h V_h : P_h = [K-block 0 over Q_h | K-block 1 over K_h], V_h [128 keys x 64] MN-major ----
        mbar_wait(p_ready, tp);
        fence_after_sync();
        stamp(P, 3, n);
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            const uint64_t da = smem_desc_k_sw128(tbuf(kb * 2 + h));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16(tO + h * 64, da + 2 * k, smem_desc_mn_sw128(tbuf(4 + h) + kb * (64 * 128) + k * 2048, kBlk), id_pv, (kb | k) ? 1u : 0u);
          }
        umma_commit(o_full);
        // ---- Y = O * W_out^T : O = [K-block 0 over V_0 | K-block 1 over V_1] ----
        mbar_wait(o_ready, tp);
        mbar_wait(y_free, tp ^ 1);
        fence_after_sync();
        stamp(P, 4, n);
        for (int kb = 0; kb < 2; ++kb) {
          mbar_wait(&w_full[st], ph);
          fence_after_sync();
          const uint64_t da = smem_desc_k_sw128(tbuf(4 + kb)), db = smem_desc_k_sw128(smem + S::OFF_W + st * kBlk);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tY, da + 2 * k, db + 2 * k, id128, (kb | k) ? 1u : 0u);
          umma_commit(&w_empty[st]);
          if (++st == kRing) { st = 0; ph ^= 1; }
        }
        umma_commit(y_full);
        stamp(P, 5, n);
      }
    }
  } else if (warp >= kFirstLnWarp && warp < kFirstFinWarp) {
    // ===================== LayerNorm warps (thread = tile row) =====================
    const int row = (warp & 3) * 32 + lane;
    const int w = row >> 6, i = row & 63;
    const bool leader = (warp == kFirstLnWarp && lane == 0);
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      const int win = 2 * tile + w;
      const bool live = i < L && win < P.nwin;
      unsigned char* u = abuf(b);
      if (row == 0) stamp(P, 6, n);
      mbar_wait(&x_full[b], (n >> 1) & 1);
      if (row == 0) stamp(P, 7, n);
      if (live) {
        const float x0 = up_lo<FMT>(row_chunk(u, row, 0)->x);
        float s = 0.f, ss = 0.f;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const uint4 v = *row_chunk(u, row, c);
          const float d0 = up_lo<FMT>(v.x) - x0, d1 = up_hi<FMT>(v.x) - x0, d2 = up_lo<FMT>(v.y) - x0, d3 = up_hi<FMT>(v.y) - x0;
          const float d4 = up_lo<FMT>(v.z) - x0, d5 = up_hi<FMT>(v.z) - x0, d6 = up_lo<FMT>(v.w) - x0, d7 = up_hi<FMT>(v.w) - x0;
          s += ((d0 + d1) + (d2 + d3)) + ((d4 + d5) + (d6 + d7));
          ss += fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3) + (fmaf(d4, d4, d5 * d5) + fmaf(d6, d6, d7 * d7));
        }
        const float md = s * (1.f / kC);
        const float mean = x0 + md;
        const float rstd = rsqrtf(fmaxf(ss * (1.f / kC) - md * md, 0.f) + P.eps);
        if (P.train) {
          const long long t = (long long)win * L + i;
          P.mean[t] = mean; P.rstd[t] = rstd;
        }
#pragma unroll 4
        for (int c = 0; c < 16; ++c) {
          uint4* p = row_chunk(u, row, c);
          const uint4 v = *p;
          const float4 g0 = __ldg(reinterpret_cast<const float4*>(P.gamma) + 2 * c), g1 = __ldg(reinterpret_cast<const float4*>(P.gamma) + 2 * c + 1);
          const float4 e0 = __ldg(reinterpret_cast<const float4*>(P.beta) + 2 * c), e1 = __ldg(reinterpret_cast<const float4*>(P.beta) + 2 * c + 1);
          uint4 o;
          o.x = pack2h<FMT>(fmaf((up_lo<FMT>(v.x) - mean) * rstd, g0.x, e0.x), fmaf((up_hi<FMT>(v.x) - mean) * rstd, g0.y, e0.y));
          o.y = pack2h<FMT>(fmaf((up_lo<FMT>(v.y) - mean) * rstd, g0.z, e0.z), fmaf((up_hi<FMT>(v.y) - mean) * rstd, g0.w, e0.w));
          o.z = pack2h<FMT>(fmaf((up_lo<FMT>(v.z) - mean) * rstd, g1.x, e1.x), fmaf((up_hi<FMT>(v.z) - mean) * rstd, g1.y, e1.y));
          o.w = pack2h<FMT>(fmaf((up_lo<FMT>(v.w) - mean) * rstd, g1.z, e1.z), fmaf((up_hi<FMT>(v.w) - mean) * rstd, g1.w, e1.w));
          *p = o;
        }
      }
      fence_proxy_async();
      mbar_arrive(&n1_ready[b]);
      if (row == 0) stamp(P, 8, n);
      if (P.train) {              // n1 in token order for the backward: boxes [L rows x 64 columns] straight from the A tile
        named_bar_sync(1, 32 * kLnWarps);
        if (leader) {
          for (int ww = 0; ww < 2; ++ww)
            if (2 * tile + ww < P.nwin) {
              tma_store_2d(&tmN1, u + ww * 64 * 128, 0, (2 * tile + ww) * L);
              tma_store_2d(&tmN1, u + kBlk + ww * 64 * 128, 64, (2 * tile + ww) * L);
            }
          bulk_commit();
          bulk_wait_read_all();
          mbar_arrive(&n1_stored[b]);
        }
      } else if (leader) {
        mbar_arrive(&n1_stored[b]);
      }
    }
    if (leader) bulk_wait_all();
  } else if (warp >= kFirstFinWarp && warp < kFirstWorkWarp) {
    // ===================== final warps: Y + b_out + n1 -> y1 rows, in place over n1, TMA box stores (thread = tile row) =====================
    const int q = warp & 3, row = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const int i = row & 63;
    const bool leader = (warp == kFirstFinWarp && lane == 0);
    for (int n = 0; n < n_local; ++n) {
      const int b = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      unsigned char* u = abuf(b);
      mbar_wait(y_full, n & 1);
      fence_after_sync();
      if (row == 0) stamp(P, 9, n);
      mbar_wait(&n1_stored[b], (n >> 1) & 1);
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t v[32];
        tmem_ld32(tY + lane_sel + ch * 32, v);
        tmem_ld_wait();
        if (ch == 3) { fence_before_sync(); mbar_arrive(y_free); }
        if (i < L) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint4* p = row_chunk(u, row, ch * 4 + c);
            const uint4 r = *p;
            const float* bp = sbo + ch * 32 + c * 8;
            const float4 ba = *reinterpret_cast<const float4*>(bp), bb = *reinterpret_cast<const float4*>(bp + 4);
            uint4 o;
            o.x = pack2h<FMT>(__uint_as_float(v[c * 8 + 0]) + ba.x + up_lo<FMT>(r.x), __uint_as_float(v[c * 8 + 1]) + ba.y + up_hi<FMT>(r.x));
            o.y = pack2h<FMT>(__uint_as_float(v[c * 8 + 2]) + ba.z + up_lo<FMT>(r.y), __uint_as_float(v[c * 8 + 3]) + ba.w + up_hi<FMT>(r.y));
            o.z = pack2h<FMT>(__uint_as_float(v[c * 8 + 4]) + bb.x + up_lo<FMT>(r.z), __uint_as_float(v[c * 8 + 5]) + bb.y + up_hi<FMT>(r.z));
            o.w = pack2h<FMT>(__uint_as_float(v[c * 8 + 6]) + bb.z + up_lo<FMT>(r.w), __uint_as_float(v[c * 8 + 7]) + bb.w + up_hi<FMT>(r.w));
            *p = o;
          }
        }
      }
      fence_proxy_async();
      named_bar_sync(2, 32 * kFinWarps);
      if (leader) {
        for (int w = 0; w < 2; ++w)
          if (2 * tile + w < P.nwin) {
            int bi, y0, x0;
            win_origin(2 * tile + w, &bi, &y0, &x0);
            tma_store_4d(&tmY, u + w * 64 * 128, 0, x0, y0, bi);
            tma_store_4d(&tmY, u + kBlk + w * 64 * 128, 64, x0, y0, bi);
          }
        bulk_commit();
        bulk_wait_read_all();
        mbar_arrive(&a_free[b]);
        stamp(P, 10, n);
      }
    }
    if (leader) bulk_wait_all();
  } else if (warp >= kFirstWorkWarp) {
    // ===================== worker warps =====================
    const int ww_ = warp - kFirstWorkWarp;
    const int q = warp & 3, cg = ww_ >> 2;             // TMEM lane quadrant; column group 0..3
    const int row = q * 32 + lane;
    const int w = row >> 6, i = row & 63;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool leader = (ww_ == 0 && lane == 0);       // issues the qkv / o by-product stores
    const bool smax = cg < 2;                           // softmax / O threads: (row, head = cg)
    for (int n = 0; n < n_local; ++n) {
      const uint32_t tp = n & 1;
      const int tile = blockIdx.x + n * gridDim.x;
      const int win = 2 * tile + w;
      // ---- QKV accumulator -> + b_in -> 16 bit -> Q/K/V tiles: this thread's 96 columns = 3 x 32 ----
      mbar_wait(qkv_full, tp);
      fence_after_sync();
      if (leader) stamp(P, 11, n);
      if (n > 0) {
        mbar_wait(y_full, tp ^ 1);                     // out_proj of the previous tile has read the O (= V) tiles
        if (P.train) {                                 // ... and the previous tile's o stores have read them too
          if (leader) bulk_wait_read_all();
          named_bar_sync(3, 32 * kWorkWarps);
        }
      }
#pragma unroll 1
      for (int r3 = 0; r3 < 3; ++r3) {
        const int col = cg * 96 + r3 * 32;             // first of 32 QKV columns
        uint32_t v[32];
        tmem_ld32(tQKV + lane_sel + col, v);
        tmem_ld_wait();
        unsigned char* t = tbuf(col >> 6);             // (q|k|v, head) tile
        const int c16 = (col & 63) >> 3;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float* bp = sbi + col + c * 8;
          const float4 ba = *reinterpret_cast<const float4*>(bp), bb = *reinterpret_cast<const float4*>(bp + 4);
          uint4 o;
          o.x = pack2h<FMT>(__uint_as_float(v[c * 8 + 0]) + ba.x, __uint_as_float(v[c * 8 + 1]) + ba.y);
          o.y = pack2h<FMT>(__uint_as_float(v[c * 8 + 2]) + ba.z, __uint_as_float(v[c * 8 + 3]) + ba.w);
          o.z = pack2h<FMT>(__uint_as_float(v[c * 8 + 4]) + bb.x, __uint_as_float(v[c * 8 + 5]) + bb.y);
          o.w = pack2h<FMT>(__uint_as_float(v[c * 8 + 6]) + bb.z, __uint_as_float(v[c * 8 + 7]) + bb.w);
          *reinterpret_cast<uint4*>(t + sw128_offset(row, c16 + c)) = o;
        }
      }
      fence_before_sync();
      fence_proxy_async();
      mbar_arrive(qk_ready);
      if (leader) stamp(P, 12, n);
      if (P.train) {             // qkv rows in token order: six [L x 64] boxes per window
        named_bar_sync(3, 32 * kWorkWarps);
        if (leader) {
          for (int wv = 0; wv < 2; ++wv)
            if (2 * tile + wv < P.nwin)
              for (int ti = 0; ti < 6; ++ti) tma_store_2d(&tmQKV, tbuf(ti) + wv * 64 * 128, ti * 64, (2 * tile + wv) * L);
          bulk_commit();
        }
      }
      if (smax) {
        // ---- softmax: thread = (row, head): 64 scores of its own window ----
        const int h = cg;
        mbar_wait(s_full, tp);
        fence_after_sync();
        if (leader) stamp(P, 13, n);
        uint32_t sa[32], sb[32];
        tmem_ld32(tS + lane_sel + h * 128 + w * 64, sa);
        tmem_ld32(tS + lane_sel + h * 128 + w * 64 + 32, sb);
        tmem_ld_wait();
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float a = j < L ? __uint_as_float(sa[j]) * P.scale_log2 : -INFINITY;
          const float c = j + 32 < L ? __uint_as_float(sb[j]) * P.scale_log2 : -INFINITY;
          sa[j] = __float_as_uint(a); sb[j] = __float_as_uint(c);
          m = fmaxf(m, fmaxf(a, c));
        }
        float sum = 0.f;
        uint32_t pk[32];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          pk[j] = pack2h<FMT>(exp2f(__uint_as_float(sa[2 * j]) - m), exp2f(__uint_as_float(sa[2 * j + 1]) - m));
          pk[16 + j] = pack2h<FMT>(exp2f(__uint_as_float(sb[2 * j]) - m), exp2f(__uint_as_float(sb[2 * j + 1]) - m));
          // the row sum is taken from the ROUNDED probabilities: exactly what the PV MMA consumes
          sum += up_lo<FMT>(pk[j]) + up_hi<FMT>(pk[j]) + up_lo<FMT>(pk[16 + j]) + up_hi<FMT>(pk[16 + j]);
        }
        if (P.train) {                                 // the qkv stores must have read the Q / K tiles before P overwrites them
          if (leader) bulk_wait_read_all();
          named_bar_sync(4, 16 * kWorkWarps);
        }
        // P_h row: K-block w (own window's keys) = probabilities, K-block 1-w = zeros; K-block kb lives over tile (kb*2 + h)
        unsigned char* pw = tbuf(w * 2 + h);
        unsigned char* pz = tbuf((1 - w) * 2 + h);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          *reinterpret_cast<uint4*>(pw + sw128_offset(row, c)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
          *reinterpret_cast<uint4*>(pz + sw128_offset(row, c)) = make_uint4(0, 0, 0, 0);
        }
        fence_before_sync();
        fence_proxy_async();
        mbar_arrive(p_ready);
        if (leader) stamp(P, 14, n);
        const bool live = i < L && win < P.nwin;
        if (P.train && live) P.lse[((long long)win * L + i) * 2 + h] = (m + log2f(sum)) * 0.69314718055994530942f;
        const float inv = 1.f / sum;
        // ---- O_h / rowsum -> 16 bit -> over the V_h tile ----
        mbar_wait(o_full, tp);
        fence_after_sync();
        uint32_t oa[32], ob[32];
        tmem_ld32(tO + lane_sel + h * 64, oa);
        tmem_ld32(tO + lane_sel + h * 64 + 32, ob);
        tmem_ld_wait();
        unsigned char* ot = tbuf(4 + h);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 o;
          o.x = pack2h<FMT>(__uint_as_float(oa[c * 8 + 0]) * inv, __uint_as_float(oa[c * 8 + 1]) * inv);
          o.y = pack2h<FMT>(__uint_as_float(oa[c * 8 + 2]) * inv, __uint_as_float(oa[c * 8 + 3]) * inv);
          o.z = pack2h<FMT>(__uint_as_float(oa[c * 8 + 4]) * inv, __uint_as_float(oa[c * 8 + 5]) * inv);
          o.w = pack2h<FMT>(__uint_as_float(oa[c * 8 + 6]) * inv, __uint_as_float(oa[c * 8 + 7]) * inv);
          *reinterpret_cast<uint4*>(ot + sw128_offset(row, c)) = o;
          uint4 o2;
          o2.x = pack2h<FMT>(__uint_as_float(ob[c * 8 + 0]) * inv, __uint_as_float(ob[c * 8 + 1]) * inv);
          o2.y = pack2h<FMT>(__uint_as_float(ob[c * 8 + 2]) * inv, __uint_as_float(ob[c * 8 + 3]) * inv);
          o2.z = pack2h<FMT>(__uint_as_float(ob[c * 8 + 4]) * inv, __uint_as_float(ob[c * 8 + 5]) * inv);
          o2.w = pack2h<FMT>(__uint_as_float(ob[c * 8 + 6]) * inv, __uint_as_float(ob[c * 8 + 7]) * inv);
          *reinterpret_cast<uint4*>(ot + sw128_offset(row, 4 + c)) = o2;
        }
        fence_before_sync();
        fence_proxy_async();
        mbar_arrive(o_ready);
        if (leader) stamp(P, 15, n);
        if (P.train) {           // o rows in token order: [L x 64] boxes per (window, head)
          named_bar_sync(4, 16 * kWorkWarps);
          if (leader) {
            for (int wv = 0; wv < 2; ++wv)
              if (2 * tile + wv < P.nwin)
                for (int hh = 0; hh < 2; ++hh) tma_store_2d(&tmO, tbuf(4 + hh) + wv * 64 * 128, hh * 64, (2 * tile + wv) * L);
            bulk_commit();
          }
        }
      }
    }
    if (leader) bulk_wait_all();
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 1) { fence_after_sync(); tmem_dealloc(tmem_base, 512); }
}

}  // namespace
}  // namespace tc
}  // namespace b200

using namespace b200;

static long long* g_ab_dbg = nullptr;
/* debugging aid (not part of the public header): device buffer of 16*16 int64 receiving CTA 0's event clock stamps */
extern "C" B200_API void b200_debug_set_attn_block_timeline(void* buf) { g_ab_dbg = (long long*)buf; }

extern "C" B200_API int b200_swin_attn_block_supported(int32_t B, int32_t C, int32_t H, int32_t W, int32_t heads, int32_t ws, int32_t shift,
                                                       int32_t dtype) {
  if (dtype != B200_BF16 && dtype != B200_F16) return 0;
  if (B <= 0 || H <= 0 || W <= 0 || C != tc::kC || heads != 2 || shift != 0 || ws < 2 || ws > 8) return 0;
  const long long T = (long long)B * ((H + ws - 1) / ws) * ((W + ws - 1) / ws) * ws * ws;
  return T < (1ll << 31) - 256;
}

extern "C" B200_API int b200_swin_attn_block_fwd(const void* x, const float* gamma, const float* beta, const void* w_in, const float* b_in,
                                                 const void* w_out, const float* b_out, void* y1, void* n1, void* qkv, void* o, float* lse,
                                                 float* mean, float* rstd, int32_t B, int32_t C, int32_t H, int32_t W, int32_t heads,
                                                 int32_t ws, float eps, int32_t dtype, void* stream) {
  B200_REQUIRE(b200_swin_attn_block_supported(B, C, H, W, heads, ws, 0, dtype), B200_ERR_UNSUPPORTED,
               "swin_attn_block_fwd: unsupported problem (16-bit dtypes, C = 128, 2 heads, window <= 8, no shift)");
  B200_REQUIRE(x && gamma && beta && w_in && b_in && w_out && b_out && y1, B200_ERR_SHAPE, "swin_attn_block_fwd: null pointer");
  const bool train = n1 != nullptr;
  B200_REQUIRE(!train || (qkv && o && lse && mean && rstd), B200_ERR_SHAPE, "swin_attn_block_fwd: training needs all by-product buffers");
  B200_REQUIRE((((uintptr_t)x | (uintptr_t)w_in | (uintptr_t)w_out | (uintptr_t)y1 | (uintptr_t)n1 | (uintptr_t)qkv | (uintptr_t)o) & 15) == 0,
               B200_ERR_ALIGN, "swin_attn_block_fwd: 16-byte alignment required");
  using namespace b200::tc;
  const int nWh = (H + ws - 1) / ws, nWw = (W + ws - 1) / ws, L = ws * ws;
  const long long nwin = (long long)B * nWh * nWw, T = nwin * L;
  const CUtensorMap* mX = tensor_map_nhwc(x, B, H, W, C, ws, ws, dtype);
  const CUtensorMap* mY = tensor_map_nhwc(y1, B, H, W, C, ws, ws, dtype);
  const CUtensorMap* mWi = tensor_map_2d(w_in, 3 * kC, kC, kC, 128, 64, dtype);
  const CUtensorMap* mWo = tensor_map_2d(w_out, kC, kC, kC, 128, 64, dtype);
  const CUtensorMap* mN1 = train ? tensor_map_2d(n1, (uint64_t)T, kC, kC, (uint32_t)L, 64, dtype) : mWo;
  const CUtensorMap* mQ = train ? tensor_map_2d(qkv, (uint64_t)T, 3 * kC, 3 * kC, (uint32_t)L, 64, dtype) : mWo;
  const CUtensorMap* mO = train ? tensor_map_2d(o, (uint64_t)T, kC, kC, (uint32_t)L, 64, dtype) : mWo;
  if (!mX || !mY || !mWi || !mWo || !mN1 || !mQ || !mO) return B200_ERR_LAUNCH;
  ABParams P;
  P.gamma = gamma; P.beta = beta; P.b_in = b_in; P.b_out = b_out; P.lse = lse; P.mean = mean; P.rstd = rstd;
  P.nwin = (int)nwin; P.n_tiles = (int)((nwin + 1) / 2); P.L = L; P.ws = ws; P.nWh = nWh; P.nWw = nWw; P.train = train ? 1 : 0;
  P.scale_log2 = 1.4426950408889634f / sqrtf((float)kHD); P.eps = eps; P.dbg = g_ab_dbg;
  const int grid = P.n_tiles < sm_count() ? P.n_tiles : sm_count();
  auto kern = dtype == B200_BF16 ? swin_attn_block_fwd_kernel<1> : swin_attn_block_fwd_kernel<0>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ABSmem::TOTAL);
  kern<<<grid, kThreads, ABSmem::TOTAL, (cudaStream_t)stream>>>(*mX, *mY, *mWi, *mWo, *mN1, *mQ, *mO, P);
  return check_launch("swin_attn_block_fwd");
}
