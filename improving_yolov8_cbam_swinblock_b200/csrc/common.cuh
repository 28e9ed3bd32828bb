// Shared device/host helpers for the sm_100a kernels (CBAM / SPPF pool / SwinBlock).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200_yolo_blocks.h"

namespace b200 {

// ---- error plumbing (C-ABI: return codes + b200_last_error(), never throw) -------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define B200_REQUIRE(cond, code, ...)  \
  do {                                 \
    if (!(cond)) {                     \
      b200::set_error(__VA_ARGS__);    \
      return (code);                   \
    }                                  \
  } while (0)

int sm_count();
int max_smem_optin();

// ---- dtype helpers ------------------------------------------------------------------------------------
template <typename T> struct DT;
template <> struct DT<float> {
  static constexpr int code = B200_F32;
  __device__ static __forceinline__ float to_f(float v) { return v; }
  __device__ static __forceinline__ float from_f(float v) { return v; }
};
template <> struct DT<__nv_bfloat16> {
  static constexpr int code = B200_BF16;
  __device__ static __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
  __device__ static __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct DT<__half> {
  static constexpr int code = B200_F16;
  __device__ static __forceinline__ float to_f(__half v) { return __half2float(v); }
  __device__ static __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

#define B200_DISPATCH_DTYPE(dtype, ...)                                         \
  [&]() -> int {                                                                \
    switch (dtype) {                                                            \
      case B200_F32: { using T = float; return __VA_ARGS__(); }                 \
      case B200_BF16: { using T = __nv_bfloat16; return __VA_ARGS__(); }        \
      case B200_F16: { using T = __half; return __VA_ARGS__(); }                \
      default: b200::set_error("unsupported dtype code %d", (int)(dtype));      \
               return B200_ERR_DTYPE;                                           \
    }                                                                           \
  }()

// ---- small device utilities -----------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sigmoidf_(float z) { return 1.0f / (1.0f + __expf(-z)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// 16-byte streaming global accesses (read-once / write-once data: keep it out of L1)
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream16(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// 16-byte asynchronous global -> shared copy (LDGSTS, L1 bypassed); !valid zero-fills the destination (src-size 0: nothing is read).
// A thread can have any number in flight -- no staging registers -- which is what lets a CTA request a whole tile at once.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- shifted-window mask (SwinBlock extension; the reference block is unshifted: shift == 0 disables it) ----------
// After the cyclic shift by `shift` only the windows of the last window row / column mix image regions; inside them a
// query attends to the keys on its own side of the seam (row/col index >= ws-shift or not).  ra / ca: bit j = key j
// lies past the seam in the row / column direction (window length L <= 64).
struct ShiftMask {
  int nWh, nWw, shift;
  unsigned long long ra, ca;
};
inline ShiftMask make_shift_mask(int nWh, int nWw, int ws, int shift) {
  ShiftMask m{nWh, nWw, shift, 0ull, 0ull};
  if (shift > 0)
    for (int j = 0; j < ws * ws && j < 64; ++j) {
      if (j / ws >= ws - shift) m.ra |= 1ull << j;
      if (j % ws >= ws - shift) m.ca |= 1ull << j;
    }
  return m;
}
__device__ __forceinline__ unsigned long long allowed_keys(const ShiftMask& M, int win, int i) {
  unsigned long long a = ~0ull;
  if (M.shift) {
    const int ww = win % M.nWw, wh = (win / M.nWw) % M.nWh;
    if (wh == M.nWh - 1) a &= ~(M.ra ^ (((M.ra >> (i & 63)) & 1ull) ? ~0ull : 0ull));
    if (ww == M.nWw - 1) a &= ~(M.ca ^ (((M.ca >> (i & 63)) & 1ull) ? ~0ull : 0ull));
  }
  return a;
}
int check_shift(int64_t tokens, int L, int nWh, int nWw, int ws, int shift);

// ---- mbarrier + 1-D bulk TMA (cp.async.bulk: SASS UBLKCP) -------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// With a suspend-time hint the hardware may park the waiting thread until the phase completes (the hint is an upper bound).  Half of
// the executed instructions of the fused SwinBlock kernels are such try_wait + branch spins of idle roles; the hint was measured to
// change neither that count's effect nor the kernel times (the working warps are latency-, not issue-bound) -- kept as the idiom.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}"
      :: "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u) : "memory");
}
// non-blocking probe (may suspend for the hardware's try_wait time limit): true once the phase with `parity` has completed
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// truly non-blocking probe (mbarrier.test_wait never suspends): for issue loops that choose between several ready queues
__device__ __forceinline__ bool mbar_poll(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// global -> shared bulk copy, completion signalled on an mbarrier. bytes % 16 == 0, 16-B aligned both sides.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// shared -> global bulk store (bulk async-group completion)
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               :: "l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }

}  // namespace b200
