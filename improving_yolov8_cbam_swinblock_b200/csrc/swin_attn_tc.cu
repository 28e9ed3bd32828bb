// SwinBlock window attention on tcgen05 tensor cores (bf16 / f16 activations), forward.
// Replaces the bmm / softmax / bmm core of nn.MultiheadAttention at swin_block.py:51 for 16-bit activations.
//
// Work unit = a PAIR of (window, head) items stacked in one M = 128 UMMA tile: rows [0,64) belong to item 0, rows
// [64,128) to item 1 (L = ws*ws <= 64 real rows each).  Per pair:
//   TMA   Q, K, V boxes [64 tokens][64 channels] straight out of the packed qkv[T,3C] rows (128-byte swizzle)
//   MMA   S[128x128] = Q K^T            (A, B K-major)  -> TMEM; only the two diagonal 64x64 blocks are meaningful
//   warps thread = row: tcgen05.ld its 64 scores, scale, mask j >= L, exp2 softmax in registers, write the
//         un-normalised probabilities as bf16 into a K-major A tile in shared memory (off-diagonal blocks stay 0)
//   MMA   O[128xHD] = P V               (A K-major from smem, B = the V tile as loaded, MN-major descriptor)
//   warps tcgen05.ld O, multiply by 1/rowsum, store the L real rows to o[T,C]; lse saved for the backward
// Persistent CTAs (one per SM), 6 warps: 0-3 softmax/epilogue (TMEM lane quadrant = warp), 4 TMA producer, 5 MMA
// issuer.  With HD = 64 everything is double-buffered so S(k+1) is computed while softmax(k) runs.
#include "tc.cuh"

namespace b200 {
namespace tc {
namespace {

constexpr int kThreads10 = 320;   // 8 softmax/epilogue warps + TMA warp + MMA warp

struct AttnParams {
  void* o;
  float* lse;
  long long T;
  int L, C, nh, n_items, n_pairs, fmt;
  float scale_log2;
  ShiftMask mask;
};

template <int HD> struct ACfg {
  static constexpr int KB = HD / 64;                 // 64-wide channel blocks per head
  static constexpr int STAGES = HD == 64 ? 2 : 1;
  static constexpr int Q_BYTES = KB * 128 * 128;     // [KB][128 rows][128 B]
  static constexpr int P_BYTES = 2 * 128 * 128;      // [2 key blocks][128 rows][128 B]
  static constexpr int STAGE_BYTES = 3 * Q_BYTES + P_BYTES;
  static constexpr int OFF_BAR = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = OFF_BAR + 256 + 1024;
  static constexpr int TMEM_COLS = (STAGES * (128 + HD)) <= 256 ? 256 : 512;
};

__device__ __forceinline__ uint32_t pack2f(float lo, float hi, int fmt) {
  if (fmt == 1) {
    __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
  }
  __half2 p = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

template <int HD>
__global__ void __launch_bounds__(kThreads10, 1) swin_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmO, AttnParams P) {
  using Cfg = ACfg<HD>;
  constexpr int KB = Cfg::KB, STAGES = Cfg::STAGES;
  extern __shared__ unsigned char smem_raw_[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw_) + 1023) & ~(uintptr_t)1023);
  // per stage: Q/K landed, V landed (TMA); S done + Q/K reusable, O done + V/P reusable (tcgen05.commit); P written (128 threads)
  uint64_t* qk_full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* v_full = qk_full + STAGES;
  uint64_t* s_full = v_full + STAGES;
  uint64_t* qk_free = s_full + STAGES;
  uint64_t* p_full = qk_free + STAGES;
  uint64_t* o_full = p_full + STAGES;
  uint64_t* v_free = o_full + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(v_free + STAGES);
  const int n_local = blockIdx.x < P.n_pairs ? (P.n_pairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  auto sQ = [&](int s) { return smem + s * Cfg::STAGE_BYTES; };
  auto sK = [&](int s) { return smem + s * Cfg::STAGE_BYTES + Cfg::Q_BYTES; };
  auto sV = [&](int s) { return smem + s * Cfg::STAGE_BYTES + 2 * Cfg::Q_BYTES; };
  auto sP = [&](int s) { return smem + s * Cfg::STAGE_BYTES + 3 * Cfg::Q_BYTES; };

  if (warp == 8 && elect_one()) {
    prefetch_tmap(&tmQKV); prefetch_tmap(&tmO);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&qk_full[s], 1); mbar_init(&v_full[s], 1); mbar_init(&s_full[s], 1); mbar_init(&qk_free[s], 1);
      mbar_init(&p_full[s], 128); mbar_init(&o_full[s], 1); mbar_init(&v_free[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 9) { tmem_alloc(tmem_slot, Cfg::TMEM_COLS); tmem_relinquish(); }
  if (warp < 4) {
    // off-diagonal P blocks are never written again: zero them once (zero is swizzle-invariant)
    const int row = warp * 32 + lane, r = row >> 6;
    for (int s = 0; s < STAGES; ++s) {
      uint4* z = reinterpret_cast<uint4*>(sP(s) + (1 - r) * (128 * 128) + row * 128);
#pragma unroll
      for (int i = 0; i < 8; ++i) z[i] = make_uint4(0, 0, 0, 0);
    }
  }
  // The TMA boxes carry exactly L token rows per item, so rows L..63 of every Q / K / V tile keep these zeros for the whole
  // kernel: a non-finite value in a NEIGHBOURING window (which a 64-row box would pull in) can never meet a zero
  // probability in the PV MMA (0 x Inf = NaN).
  for (int s = 0; s < STAGES; ++s)
    for (int i = threadIdx.x; i < 3 * Cfg::Q_BYTES / 16; i += kThreads10) reinterpret_cast<uint4*>(sQ(s))[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  auto tS = [&](int s) { return tmem_base + s * 128; };
  auto tO = [&](int s) { return tmem_base + STAGES * 128 + s * HD; };

  if (warp == 8) {
    // ===================== TMA producer =====================
    // Q/K of a stage are reloaded as soon as the S MMAs that read them have completed, V once the PV MMAs have: the loads of
    // pair n+STAGES are in flight while pair n is still in its softmax / epilogue
    if (elect_one()) {
      const uint32_t box_bytes = 2u * KB * (uint32_t)P.L * 128u;   // one operand tile: 2 items x KB boxes of [L rows][128 B]
      for (int n = 0; n < n_local; ++n) {
        const int pair = blockIdx.x + n * gridDim.x;
        const int s = n % STAGES;
        const uint32_t ph = (n / STAGES) & 1;
        int t0[2], col[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          int it = 2 * pair + r;
          if (it >= P.n_items) it = P.n_items - 1;
          const int win = it / P.nh, h = it - win * P.nh;
          t0[r] = win * P.L; col[r] = h * HD;
        }
        mbar_wait(&qk_free[s], ph ^ 1);
        mbar_expect_tx(&qk_full[s], 2 * box_bytes);
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            tma_load_2d(sQ(s) + kb * 16384 + r * 8192, &tmQKV, &qk_full[s], col[r] + kb * 64, t0[r]);
            tma_load_2d(sK(s) + kb * 16384 + r * 8192, &tmQKV, &qk_full[s], P.C + col[r] + kb * 64, t0[r]);
          }
        mbar_wait(&v_free[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], box_bytes);
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(sV(s) + kb * 16384 + r * 8192, &tmQKV, &v_full[s], 2 * P.C + col[r] + kb * 64, t0[r]);
      }
    }
  } else if (warp == 9) {
    // ===================== MMA issuer =====================
    // S of pair a and PV of pair b are issued in whichever order their inputs become ready (a < b + STAGES: S(a) overwrites
    // the TMEM columns softmax(a-STAGES) read, which p_full(a-STAGES) -- waited on before PV(a-STAGES) -- covers)
    if (elect_one()) {
      const uint32_t idesc_s = idesc_f16(128, 128, P.fmt, 0, 0);
      const uint32_t idesc_o = idesc_f16(128, HD, P.fmt, 0, 1);
      int a = 0, b = 0;
      while (b < n_local) {
        bool did = false;
        if (a < n_local && a < b + STAGES) {
          const int s = a % STAGES;
          if (mbar_test(&qk_full[s], (a / STAGES) & 1)) {
            fence_after_sync();
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16(tS(s), smem_desc_k_sw128(sQ(s) + kb * 16384 + k * 32), smem_desc_k_sw128(sK(s) + kb * 16384 + k * 32),
                         idesc_s, (kb | k) != 0);
            umma_commit(&s_full[s]);
            umma_commit(&qk_free[s]);
            ++a; did = true;
          }
        }
        if (!did) {
          const int s = b % STAGES;
          const uint32_t ph = (b / STAGES) & 1;
          if (mbar_test(&p_full[s], ph)) {
            mbar_wait(&v_full[s], ph);
            fence_after_sync();
#pragma unroll
            for (int kb = 0; kb < 2; ++kb)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16(tO(s), smem_desc_k_sw128(sP(s) + kb * 16384 + k * 32),
                         smem_desc_mn_sw128(sV(s) + kb * 8192 + k * 2048, 16384), idesc_o, (kb | k) != 0);
            umma_commit(&o_full[s]);
            umma_commit(&v_free[s]);
            ++b;
          }
        }
      }
    }
  } else if ((warp >> 2) < STAGES) {
    // ===================== softmax + epilogue: warp group g = warp >> 2 owns stage g (thread = row) =====================
    // the two groups work on alternate pairs, so one group's softmax overlaps the other's PV MMA + epilogue
    const int g = warp >> 2, q = warp & 3;
    const int row = q * 32 + lane, r = row >> 6, i = row & 63;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const int s = g;
    const uint32_t bar_id = 1 + g * 2 + r;      // named barrier of the 64 threads (2 warps) that own one item of the pair
    bool stores_pending = false;
    for (int n = g; n < n_local; n += STAGES) {
      const int pair = blockIdx.x + n * gridDim.x;
      const uint32_t ph = (n / STAGES) & 1;
      const int it = 2 * pair + r;
      const bool valid = it < P.n_items && i < P.L;
      const int itc = it < P.n_items ? it : P.n_items - 1;
      const int win = itc / P.nh, h = itc - win * P.nh;
      const long long tok = (long long)win * P.L + i;
      const unsigned long long allowed = allowed_keys(P.mask, win, i);   // shifted-window mask (all ones when shift == 0)
      mbar_wait(&s_full[s], ph);
      fence_after_sync();
      uint32_t v[32], w[32];
      tmem_ld32(tS(s) + lane_sel + r * 64, v);
      tmem_ld32(tS(s) + lane_sel + r * 64 + 32, w);
      tmem_ld_wait();
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float a = (j < P.L && ((allowed >> j) & 1ull)) ? __uint_as_float(v[j]) * P.scale_log2 : -INFINITY;
        const float b = (j + 32 < P.L && ((allowed >> (j + 32)) & 1ull)) ? __uint_as_float(w[j]) * P.scale_log2 : -INFINITY;
        v[j] = __float_as_uint(a); w[j] = __float_as_uint(b);
        m = fmaxf(m, fmaxf(a, b));
      }
      float sum = 0.f;
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float e0 = exp2f(__uint_as_float(v[2 * j]) - m), e1 = exp2f(__uint_as_float(v[2 * j + 1]) - m);
        const float f0 = exp2f(__uint_as_float(w[2 * j]) - m), f1 = exp2f(__uint_as_float(w[2 * j + 1]) - m);
        pk[j] = pack2f(e0, e1, P.fmt);
        pk[16 + j] = pack2f(f0, f1, P.fmt);
        // accumulate the row sum from the ROUNDED probabilities, i.e. exactly what the PV MMA will consume
        if (P.fmt == 1) {
          sum += __uint_as_float(pk[j] << 16) + __uint_as_float(pk[j] & 0xffff0000u) + __uint_as_float(pk[16 + j] << 16) +
                 __uint_as_float(pk[16 + j] & 0xffff0000u);
        } else {
          const float2 a2 = __half22float2(*reinterpret_cast<__half2*>(&pk[j]));
          const float2 b2 = __half22float2(*reinterpret_cast<__half2*>(&pk[16 + j]));
          sum += a2.x + a2.y + b2.x + b2.y;
        }
      }
      unsigned char* prow = sP(s) + r * (128 * 128);
      if (stores_pending) {                      // the previous pair's O store reads the rows written next
        if (i == 0) bulk_wait_read_all();
        named_bar_sync(bar_id, 64);
      }
#pragma unroll
      for (int c = 0; c < 8; ++c)
        *reinterpret_cast<uint4*>(prow + sw128_offset(row, c)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
      fence_proxy_async();
      fence_before_sync();
      mbar_arrive(&p_full[s]);
      if (valid && P.lse) P.lse[tok * P.nh + h] = (m + log2f(sum)) * 0.69314718055994530942f;
      const float inv = 1.f / sum;
      // ---- O ----
      mbar_wait(&o_full[s], ph);
      fence_after_sync();
      if constexpr (HD == 64) {
        // the normalised row is staged in this thread's own (consumed) P row, 128-byte swizzled, and leaves as one TMA tensor
        // store of [L rows x 64 columns] per item: full-line writes instead of 16-byte row fragments
        uint32_t ok[32];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
          uint32_t ov[32];
          tmem_ld32(tO(s) + lane_sel + ch * 32, ov);
          tmem_ld_wait();
#pragma unroll
          for (int e = 0; e < 16; ++e) ok[ch * 16 + e] = pack2f(__uint_as_float(ov[2 * e]) * inv, __uint_as_float(ov[2 * e + 1]) * inv, P.fmt);
        }
#pragma unroll
        for (int c = 0; c < 8; ++c)
          *reinterpret_cast<uint4*>(prow + sw128_offset(row, c)) = make_uint4(ok[4 * c], ok[4 * c + 1], ok[4 * c + 2], ok[4 * c + 3]);
        fence_proxy_async();
        named_bar_sync(bar_id, 64);
        if (i == 0 && it < P.n_items) {
          tma_store_2d(&tmO, prow + r * (64 * 128), h * HD, win * P.L);
          bulk_commit();
        }
        stores_pending = true;
      } else {
        uint16_t* orow = reinterpret_cast<uint16_t*>(P.o) + tok * P.C + h * HD;
#pragma unroll
        for (int ch = 0; ch < HD / 32; ++ch) {
          uint32_t ov[32];
          tmem_ld32(tO(s) + lane_sel + ch * 32, ov);
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              uint4 st;
              st.x = pack2f(__uint_as_float(ov[8 * c + 0]) * inv, __uint_as_float(ov[8 * c + 1]) * inv, P.fmt);
              st.y = pack2f(__uint_as_float(ov[8 * c + 2]) * inv, __uint_as_float(ov[8 * c + 3]) * inv, P.fmt);
              st.z = pack2f(__uint_as_float(ov[8 * c + 4]) * inv, __uint_as_float(ov[8 * c + 5]) * inv, P.fmt);
              st.w = pack2f(__uint_as_float(ov[8 * c + 6]) * inv, __uint_as_float(ov[8 * c + 7]) * inv, P.fmt);
              *reinterpret_cast<uint4*>(orow + ch * 32 + c * 8) = st;
            }
          }
        }
      }
    }
  }
  bulk_wait_all();                              // outstanding O stores (no-op for threads that issued none)
  fence_before_sync();
  __syncthreads();
  if (warp == 9) { fence_after_sync(); tmem_dealloc(tmem_base, Cfg::TMEM_COLS); }
}

template <int HD>
int launch_fwd(const void* qkv, void* o, float* lse, long long T, int L, int C, int nh, const ShiftMask& M, int dtype, cudaStream_t st) {
  using Cfg = ACfg<HD>;
  const CUtensorMap* m = tensor_map_2d(qkv, (uint64_t)T, (uint64_t)3 * C, (uint64_t)3 * C, (uint32_t)L, 64, dtype);
  const CUtensorMap* mo = tensor_map_2d(o, (uint64_t)T, (uint64_t)C, (uint64_t)C, (uint32_t)L, 64, dtype);
  if (!m || !mo) return B200_ERR_LAUNCH;
  AttnParams P;
  P.o = o; P.lse = lse; P.T = T; P.L = L; P.C = C; P.nh = nh; P.mask = M;
  P.n_items = (int)(T / L) * nh;
  P.n_pairs = (P.n_items + 1) / 2;
  P.fmt = dtype == B200_BF16 ? 1 : 0;
  P.scale_log2 = 1.4426950408889634f / sqrtf((float)HD);
  auto k = swin_attn_fwd_tc_kernel<HD>;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::TOTAL);
  int grid = P.n_pairs < sm_count() ? P.n_pairs : sm_count();
  k<<<grid, kThreads10, Cfg::TOTAL, st>>>(*m, *mo, P);
  return check_launch("swin_attn_fwd_tc");
}


// =====================================================================================================
// backward:  gqkv[T,3C] from qkv, lse and go[T,C]   (SURVEY App. A.3 "Attention"; flash-style recompute)
//   S  = Q K^T,  dP = dO V^T                      (K-major operands)            -> TMEM
//   threads: P = exp2(S*c - lse), delta = sum_j P dP, dS = P (dP - delta) * hd^-0.5 -> bf16 tiles P, dS in smem
//   dQ = dS K      (A = dS K-major,  B = K tile MN-major)
//   dV = P^T dO    (A = P  MN-major, B = dO tile MN-major)
//   dK = dS^T Q    (A = dS MN-major, B = Q tile MN-major)        -> TMEM (dQ/dK alias the S/dP columns) -> global
// =====================================================================================================
struct AttnBwdParams {
  void* gqkv;
  const float* lse;
  long long T;
  int L, C, nh, n_items, n_pairs, fmt;
  float scale_log2, scale;
  ShiftMask mask;
};

template <int HD> struct BCfg {
  static constexpr int KB = HD / 64;
  static constexpr int T_BYTES = KB * 128 * 128;   // one operand tile [KB][128 rows][128 B]
  // P / dS of a window pair are block diagonal ([item 0 | 0 ; 0 | item 1]).  Stored as [item 0 rows: 8 KB][64 zero rows: 8 KB]
  // [item 1 rows: 8 KB]: key block 0 = bytes 0..16K, key block 1 = bytes 8K..24K -- the zero rows are shared by both.
  static constexpr int P_BYTES = 3 * 64 * 128;
  static constexpr int KB_STRIDE = 64 * 128;       // byte distance between the two key blocks of P / dS
  static constexpr int STAGES = HD == 64 ? 2 : 1;  // a stage = operand tiles + P/dS + TMEM columns of one pair in flight
  // HD 192: four 48 KB operand tiles leave no room for P / dS (2 x 24 KB): they overlay the V tile, which is dead once the
  // dP MMAs have completed (exactly 48 KB).  The overlay's zero rows are re-zeroed for every pair; rows L..63 of the V tile stay
  // zero because the rows of P / dS that fall there belong to padded query rows, which write zeros.
  static constexpr bool OVERLAY = HD == 192;
  static constexpr int OFF_Q = 0, OFF_K = T_BYTES, OFF_DO = 2 * T_BYTES, OFF_V = 3 * T_BYTES;
  static constexpr int OFF_P = OVERLAY ? OFF_V : 4 * T_BYTES, OFF_DS = OFF_P + P_BYTES;
  static constexpr int STAGE_BYTES = OVERLAY ? 4 * T_BYTES : OFF_DS + P_BYTES;
  static constexpr int OFF_BAR = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = OFF_BAR + 256 + 1024;
  static_assert(TOTAL <= 232448, "shared memory budget");
  // HD 64: per stage S 128 (dQ aliases columns 0..63, dV columns 64..127) | dP 128 (dK aliases 0..63)  -> 2 x 256
  // HD 128: S 128 (= dQ) | dP 128 (= dK) | dV 128
  // HD 192: S 128 | dP 128 during the first half; then dQ 0..191 | dK 192..383 | dV[:, 0:128] 384..511, and dV[:, 128:192] in
  //         columns 0..63 in a third round once dQ has been read back (3 x 192 fp32 columns do not fit in 512)
  static constexpr int TMEM_STAGE = 256;
  static constexpr int TMEM_COLS = 512;
};

template <int HD>
__global__ void __launch_bounds__(kThreads10, 1)
swin_attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmGO,
                        const __grid_constant__ CUtensorMap tmOut, AttnBwdParams P) {
  using Cfg = BCfg<HD>;
  constexpr int KB = Cfg::KB, STAGES = Cfg::STAGES, KBS = Cfg::KB_STRIDE;
  extern __shared__ unsigned char smem_raw_[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw_) + 1023) & ~(uintptr_t)1023);
  // per stage: operands landed (TMA) | operands reusable (commit) | S, dP done (commit) | P, dS written (128 threads) |
  // dQ, dK, dV done (commit) | TMEM columns read back (128 threads)
  uint64_t* in_full = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* smem_free = in_full + 2;
  uint64_t* sdp_full = in_full + 4;
  uint64_t* pds_full = in_full + 6;
  uint64_t* out_full = in_full + 8;
  uint64_t* tmem_free = in_full + 10;
  uint64_t* dq_read = in_full + 12;     // HD 192: dQ read back (128 threads) -> its columns may take the last third of dV
  uint64_t* out2_full = in_full + 13;   // HD 192: that third is complete (commit)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_full + 14);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_local = blockIdx.x < P.n_pairs ? (P.n_pairs - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  auto stage = [&](int s) { return smem + s * Cfg::STAGE_BYTES; };

  if (warp == 8 && elect_one()) {
    prefetch_tmap(&tmQKV); prefetch_tmap(&tmGO); prefetch_tmap(&tmOut);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&in_full[s], 1); mbar_init(&smem_free[s], 1); mbar_init(&sdp_full[s], 1); mbar_init(&pds_full[s], 128);
      mbar_init(&out_full[s], 1); mbar_init(&tmem_free[s], 128);
    }
    mbar_init(dq_read, 128); mbar_init(out2_full, 1);
    fence_mbar_init();
  }
  if (warp == 9) { tmem_alloc(tmem_slot, Cfg::TMEM_COLS); tmem_relinquish(); }
  if (warp < 4) {
    // the shared zero rows of P / dS are never written again (zero is swizzle-invariant)
    const int t = warp * 32 + lane;            // 128 threads x 64 B = 8 KB per matrix
    for (int s = 0; s < STAGES; ++s) {
      uint4* z0 = reinterpret_cast<uint4*>(stage(s) + Cfg::OFF_P + KBS + t * 64);
      uint4* z1 = reinterpret_cast<uint4*>(stage(s) + Cfg::OFF_DS + KBS + t * 64);
#pragma unroll
      for (int i = 0; i < 4; ++i) { z0[i] = make_uint4(0, 0, 0, 0); z1[i] = make_uint4(0, 0, 0, 0); }
    }
  }
  // operand tiles: rows L..63 of every item stay zero (the TMA boxes carry exactly L rows; see the forward kernel)
  for (int s = 0; s < STAGES; ++s)
    for (int i = threadIdx.x; i < 4 * Cfg::T_BYTES / 16; i += kThreads10) reinterpret_cast<uint4*>(stage(s))[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  auto tS = [&](int s) { return tmem_base + s * Cfg::TMEM_STAGE; };
  auto tDP = [&](int s) { return tmem_base + s * Cfg::TMEM_STAGE + 128; };
  auto tDQ = [&](int s) { return tS(s); };
  auto tDK = [&](int s) { return HD == 192 ? tmem_base + 192 : tDP(s); };
  auto tDV = [&](int s) { return HD == 64 ? tS(s) + 64 : (HD == 192 ? tmem_base + 384 : tmem_base + 256); };

  if (warp == 8) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      for (int n = 0; n < n_local; ++n) {
        const int pair = blockIdx.x + n * gridDim.x;
        const int s = n % STAGES;
        unsigned char* sQ = stage(s) + Cfg::OFF_Q;
        unsigned char* sK = stage(s) + Cfg::OFF_K;
        unsigned char* sV = stage(s) + Cfg::OFF_V;
        unsigned char* sDO = stage(s) + Cfg::OFF_DO;
        mbar_wait(&smem_free[s], ((n / STAGES) & 1) ^ 1);
        mbar_expect_tx(&in_full[s], 4u * 2u * KB * (uint32_t)P.L * 128u);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          int it = 2 * pair + r;
          if (it >= P.n_items) it = P.n_items - 1;
          const int win = it / P.nh, h = it - win * P.nh;
          const int t0 = win * P.L;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            const int col = h * HD + kb * 64;
            tma_load_2d(sQ + kb * 16384 + r * 8192, &tmQKV, &in_full[s], col, t0);
            tma_load_2d(sK + kb * 16384 + r * 8192, &tmQKV, &in_full[s], P.C + col, t0);
            tma_load_2d(sV + kb * 16384 + r * 8192, &tmQKV, &in_full[s], 2 * P.C + col, t0);
            tma_load_2d(sDO + kb * 16384 + r * 8192, &tmGO, &in_full[s], col, t0);
          }
        }
      }
    }
  } else if (warp == 9) {
    // ===================== MMA issuer =====================
    // first half of pair a (S, dP) and second half of pair b (dQ, dV, dK) are issued in whichever order their inputs become
    // ready, so one warp group's softmax overlaps the other group's MMAs and read-back
    if (elect_one()) {
      const uint32_t id_kk = idesc_f16(128, 128, P.fmt, 0, 0);   // S, dP
      const uint32_t id_kmn = idesc_f16(128, HD, P.fmt, 0, 1);   // dQ
      const uint32_t id_mnmn = idesc_f16(128, HD, P.fmt, 1, 1);  // dV, dK
      int a = 0, b = 0;
      while (b < n_local) {
        bool did = false;
        if (a < n_local && a < b + STAGES) {
          const int s = a % STAGES;
          const uint32_t ph = (a / STAGES) & 1;
          if (mbar_test(&in_full[s], ph) && mbar_test(&tmem_free[s], ph ^ 1)) {
            unsigned char* sQ = stage(s) + Cfg::OFF_Q;
            unsigned char* sK = stage(s) + Cfg::OFF_K;
            unsigned char* sV = stage(s) + Cfg::OFF_V;
            unsigned char* sDO = stage(s) + Cfg::OFF_DO;
            fence_after_sync();
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                umma_f16(tS(s), smem_desc_k_sw128(sQ + kb * 16384 + k * 32), smem_desc_k_sw128(sK + kb * 16384 + k * 32), id_kk,
                         (kb | k) != 0);
                umma_f16(tDP(s), smem_desc_k_sw128(sDO + kb * 16384 + k * 32), smem_desc_k_sw128(sV + kb * 16384 + k * 32), id_kk,
                         (kb | k) != 0);
              }
            umma_commit(&sdp_full[s]);
            ++a; did = true;
          }
        }
        if (!did) {
          const int s = b % STAGES;
          if (mbar_test(&pds_full[s], (b / STAGES) & 1)) {
            unsigned char* sQ = stage(s) + Cfg::OFF_Q;
            unsigned char* sK = stage(s) + Cfg::OFF_K;
            unsigned char* sDO = stage(s) + Cfg::OFF_DO;
            unsigned char* sP = stage(s) + Cfg::OFF_P;
            unsigned char* sDS = stage(s) + Cfg::OFF_DS;
            fence_after_sync();
            // dQ = dS K : reduction over the 128 key slots (2 key blocks x 4 k-steps of 16)
#pragma unroll
            for (int kb = 0; kb < 2; ++kb)
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_f16(tDQ(s), smem_desc_k_sw128(sDS + kb * KBS + k * 32), smem_desc_mn_sw128(sK + kb * 8192 + k * 2048, 16384),
                         id_kmn, (kb | k) != 0);
            // dV = P^T dO, dK = dS^T Q : reduction over the 128 query rows (8 k-steps of 16 rows)
            if constexpr (HD == 192) {
              const uint32_t id_v128 = idesc_f16(128, 128, P.fmt, 1, 1), id_v64 = idesc_f16(128, 64, P.fmt, 1, 1);
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                umma_f16(tDV(s), smem_desc_mn_sw128(sP + k * 2048, KBS), smem_desc_mn_sw128(sDO + k * 2048, 16384), id_v128, k != 0);
                umma_f16(tDK(s), smem_desc_mn_sw128(sDS + k * 2048, KBS), smem_desc_mn_sw128(sQ + k * 2048, 16384), id_mnmn, k != 0);
              }
              umma_commit(&out_full[s]);
              mbar_wait(dq_read, b & 1);          // third round: dV[:, 128:192] over the columns dQ occupied
              fence_after_sync();
#pragma unroll
              for (int k = 0; k < 8; ++k)
                umma_f16(tmem_base, smem_desc_mn_sw128(sP + k * 2048, KBS), smem_desc_mn_sw128(sDO + 2 * 16384 + k * 2048, 16384),
                         id_v64, k != 0);
              umma_commit(&smem_free[s]);
              umma_commit(out2_full);
            } else {
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                umma_f16(tDV(s), smem_desc_mn_sw128(sP + k * 2048, KBS), smem_desc_mn_sw128(sDO + k * 2048, 16384), id_mnmn, k != 0);
                umma_f16(tDK(s), smem_desc_mn_sw128(sDS + k * 2048, KBS), smem_desc_mn_sw128(sQ + k * 2048, 16384), id_mnmn, k != 0);
              }
              umma_commit(&smem_free[s]);
              umma_commit(&out_full[s]);
            }
            ++b;
          }
        }
      }
    }
  } else if ((warp >> 2) < STAGES) {
    // ===================== softmax + read-back: warp group g = warp >> 2 owns stage g (thread = row) =====================
    const int g = warp >> 2, q = warp & 3;
    const int row = q * 32 + lane, r = row >> 6, i = row & 63;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const int s = g;
    unsigned char* prow = stage(s) + Cfg::OFF_P + r * (2 * KBS);     // item 1's rows 64..127 live in key block 1 = +8 KB
    unsigned char* drow = stage(s) + Cfg::OFF_DS + r * (2 * KBS);
    const uint32_t bar_id = 1 + g * 2 + r;      // named barrier of the 64 threads (2 warps) that own one item of the pair
    bool stores_pending = false;
    for (int n = g; n < n_local; n += STAGES) {
      const int pair = blockIdx.x + n * gridDim.x;
      const uint32_t ph = (n / STAGES) & 1;
      const int it = 2 * pair + r;
      const bool valid = it < P.n_items && i < P.L;
      const int itc = it < P.n_items ? it : P.n_items - 1;
      const int win = itc / P.nh, h = itc - win * P.nh;
      const long long tok = (long long)win * P.L + i;
      const unsigned long long allowed = allowed_keys(P.mask, win, i);   // shifted-window mask (all ones when shift == 0)
      const float lraw = valid ? P.lse[tok * P.nh + h] : 0.f;   // consumed after the wait below: the load latency hides behind it
      mbar_wait(&sdp_full[s], ph);
      fence_after_sync();
      const float l2 = lraw * 1.4426950408889634f;
      uint32_t sv[64];
      float delta = 0.f;
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t (&sh)[32] = *reinterpret_cast<uint32_t (*)[32]>(&sv[hf * 32]);
        uint32_t dv[32];
        tmem_ld32(tS(s) + lane_sel + r * 64 + hf * 32, sh);
        tmem_ld32(tDP(s) + lane_sel + r * 64 + hf * 32, dv);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) {
          const int j = hf * 32 + jj;
          const float p = (j < P.L && valid && ((allowed >> j) & 1ull)) ? exp2f(__uint_as_float(sh[jj]) * P.scale_log2 - l2) : 0.f;
          sh[jj] = __float_as_uint(p);
          delta += p * __uint_as_float(dv[jj]);
        }
      }
      if (stores_pending) {                      // the previous pair's output stores read the P / dS rows written next
        if (i == 0) bulk_wait_read_all();
        named_bar_sync(bar_id, 64);
      }
      if constexpr (Cfg::OVERLAY) {               // the shared zero rows were overwritten by this pair's V tile
        uint4* z0 = reinterpret_cast<uint4*>(stage(s) + Cfg::OFF_P + KBS + row * 64);
        uint4* z1 = reinterpret_cast<uint4*>(stage(s) + Cfg::OFF_DS + KBS + row * 64);
#pragma unroll
        for (int e = 0; e < 4; ++e) { z0[e] = make_uint4(0, 0, 0, 0); z1[e] = make_uint4(0, 0, 0, 0); }
      }
      // second pass re-reads dP from TMEM (cheaper than keeping 64 more registers live)
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t dv[32];
        tmem_ld32(tDP(s) + lane_sel + r * 64 + hf * 32, dv);
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c = hf * 4 + cc;
          uint32_t pw[4], dw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int jj = cc * 8 + 2 * e;
            const float p0 = __uint_as_float(sv[hf * 32 + jj]), p1 = __uint_as_float(sv[hf * 32 + jj + 1]);
            pw[e] = pack2f(p0, p1, P.fmt);
            // padded rows write exact zeros (their dP may be 0 x Inf = NaN): with the overlay these bytes are rows L..63 of
            // the next pair's V tile
            dw[e] = valid ? pack2f(p0 * (__uint_as_float(dv[jj]) - delta) * P.scale, p1 * (__uint_as_float(dv[jj + 1]) - delta) * P.scale, P.fmt)
                          : 0u;
          }
          *reinterpret_cast<uint4*>(prow + sw128_offset(i, c)) = make_uint4(pw[0], pw[1], pw[2], pw[3]);
          *reinterpret_cast<uint4*>(drow + sw128_offset(i, c)) = make_uint4(dw[0], dw[1], dw[2], dw[3]);
        }
      }
      fence_proxy_async();
      fence_before_sync();
      mbar_arrive(&pds_full[s]);
      // ---- outputs: this thread owns token `tok` as query (dQ) and as key/value (dK, dV) ----
      mbar_wait(&out_full[s], ph);
      fence_after_sync();
      if constexpr (HD == 64) {
        // rows are staged in this thread's own (now consumed) P / dS rows in the 128-byte-swizzled layout and leave as one
        // TMA tensor store of [L rows x 64 columns] per item and output: full-line writes instead of 16-byte row fragments
        auto stage_rows = [&](uint32_t tsrc, unsigned char* blk, bool pre_wait) {
          uint32_t pk[32];
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            uint32_t ov[32];
            tmem_ld32(tsrc + lane_sel + ch * 32, ov);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 16; ++e) pk[ch * 16 + e] = pack2f(__uint_as_float(ov[2 * e]), __uint_as_float(ov[2 * e + 1]), P.fmt);
          }
          if (pre_wait) {                     // the rows still hold an output whose store may be reading them
            if (i == 0) bulk_wait_read_all();
            named_bar_sync(bar_id, 64);
          }
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<uint4*>(blk + sw128_offset(i, c)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        };
        stage_rows(tDQ(s), prow, false);
        stage_rows(tDK(s), drow, false);
        fence_proxy_async();
        named_bar_sync(bar_id, 64);
        if (i == 0 && it < P.n_items) {
          tma_store_2d(&tmOut, prow, h * HD, win * P.L);
          tma_store_2d(&tmOut, drow, P.C + h * HD, win * P.L);
          bulk_commit();
        }
        stage_rows(tDV(s), prow, true);
        fence_before_sync();
        mbar_arrive(&tmem_free[s]);           // all TMEM columns of the stage are read back
        fence_proxy_async();
        named_bar_sync(bar_id, 64);
        if (i == 0 && it < P.n_items) {
          tma_store_2d(&tmOut, prow, 2 * P.C + h * HD, win * P.L);
          bulk_commit();
        }
        stores_pending = true;
      } else {
        uint16_t* grow = reinterpret_cast<uint16_t*>(P.gqkv) + tok * 3 * P.C + h * HD;
#pragma unroll
        for (int which = 0; which < 3; ++which) {
          const uint32_t tsrc = which == 0 ? tDQ(s) : (which == 1 ? tDK(s) : tDV(s));
#pragma unroll
          for (int ch = 0; ch < HD / 32; ++ch) {
            uint32_t ov[32];
            uint32_t taddr = tsrc + lane_sel + ch * 32;
            if constexpr (HD == 192) {
              if (which == 1 && ch == 0) {          // dQ is out of TMEM: release its columns for the last third of dV
                fence_before_sync();
                mbar_arrive(dq_read);
              }
              if (which == 2 && ch == 4) {
                mbar_wait(out2_full, (n / STAGES) & 1);
                fence_after_sync();
              }
              if (which == 2 && ch >= 4) taddr = tmem_base + lane_sel + (ch - 4) * 32;
            }
            tmem_ld32(taddr, ov);
            tmem_ld_wait();
            if (valid) {
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                uint4 st;
                st.x = pack2f(__uint_as_float(ov[8 * c + 0]), __uint_as_float(ov[8 * c + 1]), P.fmt);
                st.y = pack2f(__uint_as_float(ov[8 * c + 2]), __uint_as_float(ov[8 * c + 3]), P.fmt);
                st.z = pack2f(__uint_as_float(ov[8 * c + 4]), __uint_as_float(ov[8 * c + 5]), P.fmt);
                st.w = pack2f(__uint_as_float(ov[8 * c + 6]), __uint_as_float(ov[8 * c + 7]), P.fmt);
                *reinterpret_cast<uint4*>(grow + which * P.C + ch * 32 + c * 8) = st;
              }
            }
          }
        }
        fence_before_sync();
        mbar_arrive(&tmem_free[s]);
      }
    }
  }
  bulk_wait_all();                              // outstanding output stores (no-op for threads that issued none)
  fence_before_sync();
  __syncthreads();
  if (warp == 9) { fence_after_sync(); tmem_dealloc(tmem_base, Cfg::TMEM_COLS); }
}

template <int HD>
int launch_bwd(const void* qkv, const float* lse, const void* go, void* gqkv, long long T, int L, int C, int nh, const ShiftMask& M, int dtype,
               cudaStream_t st) {
  using Cfg = BCfg<HD>;
  const CUtensorMap* m = tensor_map_2d(qkv, (uint64_t)T, (uint64_t)3 * C, (uint64_t)3 * C, (uint32_t)L, 64, dtype);
  const CUtensorMap* mg = tensor_map_2d(go, (uint64_t)T, (uint64_t)C, (uint64_t)C, (uint32_t)L, 64, dtype);
  const CUtensorMap* mo = tensor_map_2d(gqkv, (uint64_t)T, (uint64_t)3 * C, (uint64_t)3 * C, (uint32_t)L, 64, dtype);
  if (!m || !mg || !mo) return B200_ERR_LAUNCH;
  AttnBwdParams P;
  P.gqkv = gqkv; P.lse = lse; P.T = T; P.L = L; P.C = C; P.nh = nh; P.mask = M;
  P.n_items = (int)(T / L) * nh;
  P.n_pairs = (P.n_items + 1) / 2;
  P.fmt = dtype == B200_BF16 ? 1 : 0;
  P.scale = 1.f / sqrtf((float)HD);
  P.scale_log2 = 1.4426950408889634f * P.scale;
  auto k = swin_attn_bwd_tc_kernel<HD>;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::TOTAL);
  int grid = P.n_pairs < sm_count() ? P.n_pairs : sm_count();
  k<<<grid, kThreads10, Cfg::TOTAL, st>>>(*m, *mg, *mo, P);
  return check_launch("swin_attn_bwd_tc");
}

}  // namespace
}  // namespace tc
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_swin_attn_tc_supported(int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t dtype) {
  if (dtype != B200_BF16 && dtype != B200_F16) return 0;
  if (tokens <= 0 || L <= 0 || L > 64 || tokens % L != 0 || nh <= 0 || C % nh != 0) return 0;
  const int hd = C / nh;
  return (hd == 64 || hd == 128 || hd == 192) && (3 * C) % 8 == 0;
}

extern "C" B200_API int b200_swin_attn_fwd_tc(const void* qkv, void* o, float* lse, int64_t tokens, int32_t L, int32_t C,
                                              int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                              void* stream) {
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(b200_swin_attn_tc_supported(tokens, L, C, nh, dtype), B200_ERR_UNSUPPORTED,
               "swin_attn_fwd_tc: unsupported problem (16-bit dtype, L<=64, head dim 64, 128 or 192)");
  B200_REQUIRE(qkv && o, B200_ERR_SHAPE, "swin_attn_fwd_tc: null pointer");
  B200_REQUIRE((((uintptr_t)qkv | (uintptr_t)o) & 15) == 0, B200_ERR_ALIGN, "swin_attn_fwd_tc: 16-byte alignment required");
  cudaStream_t st = (cudaStream_t)stream;
  if (C / nh == 64) return tc::launch_fwd<64>(qkv, o, lse, tokens, L, C, nh, M, dtype, st);
  if (C / nh == 192) return tc::launch_fwd<192>(qkv, o, lse, tokens, L, C, nh, M, dtype, st);
  return tc::launch_fwd<128>(qkv, o, lse, tokens, L, C, nh, M, dtype, st);
}

extern "C" B200_API int b200_swin_attn_bwd_tc(const void* qkv, const float* lse, const void* go, void* gqkv, int64_t tokens,
                                              int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws,
                                              int32_t shift, int32_t dtype, void* stream) {
  if (int rc = check_shift(tokens, L, nWh, nWw, ws, shift)) return rc;
  const ShiftMask M = make_shift_mask(nWh, nWw, ws, shift);
  B200_REQUIRE(b200_swin_attn_tc_supported(tokens, L, C, nh, dtype), B200_ERR_UNSUPPORTED,
               "swin_attn_bwd_tc: unsupported problem (16-bit dtype, L<=64, head dim 64, 128 or 192)");
  B200_REQUIRE(qkv && lse && go && gqkv, B200_ERR_SHAPE, "swin_attn_bwd_tc: null pointer");
  B200_REQUIRE((((uintptr_t)qkv | (uintptr_t)go | (uintptr_t)gqkv) & 15) == 0, B200_ERR_ALIGN, "swin_attn_bwd_tc: 16-byte alignment required");
  cudaStream_t st = (cudaStream_t)stream;
  if (C / nh == 64) return tc::launch_bwd<64>(qkv, lse, go, gqkv, tokens, L, C, nh, M, dtype, st);
  if (C / nh == 192) return tc::launch_bwd<192>(qkv, lse, go, gqkv, tokens, L, C, nh, M, dtype, st);
  return tc::launch_bwd<128>(qkv, lse, go, gqkv, tokens, L, C, nh, M, dtype, st);
}
