// C-ABI plumbing: version, thread-local error string, launch accounting, device queries.
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

namespace b200 {
namespace {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e));
    return B200_ERR_LAUNCH;
  }
  return B200_OK;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
    cached_dev = dev;
  }
  return cached > 0 ? cached : 148;
}

int max_smem_optin() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    if (cudaDeviceGetAttribute(&cached, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) cached = 0;
    cached_dev = dev;
    cudaGetLastError();
  }
  return cached > 0 ? cached : 232448;  // 227 KB on sm_100
}
int check_shift(int64_t tokens, int L, int nWh, int nWw, int ws, int shift) {
  if (shift == 0) return B200_OK;
  B200_REQUIRE(ws > 0 && shift > 0 && shift < ws, B200_ERR_SHAPE, "swin: shift %d must lie in [0, window size %d)", shift, ws);
  B200_REQUIRE(L == ws * ws && L <= 64, B200_ERR_UNSUPPORTED, "swin: shifted windows need L = ws*ws <= 64 (L=%d ws=%d)", L, ws);
  B200_REQUIRE(nWh > 0 && nWw > 0 && (tokens / L) % ((int64_t)nWh * nWw) == 0, B200_ERR_SHAPE,
               "swin: %lld windows are not a multiple of the %dx%d window grid", (long long)(tokens / L), nWh, nWw);
  return B200_OK;
}
}  // namespace b200

extern "C" B200_API int b200_abi_version(void) { return B200_ABI_VERSION; }
extern "C" B200_API const char* b200_last_error(void) { return b200::g_err; }
extern "C" B200_API uint64_t b200_launch_count(void) { return b200::g_launches.load(std::memory_order_relaxed); }
