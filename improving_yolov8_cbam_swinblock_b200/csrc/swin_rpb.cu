// Learned relative-position bias of Swin window attention (Liu et al. 2021, "Swin Transformer: Hierarchical Vision
// Transformer using Shifted Windows", eq. 4): S[h,i,j] = q_i.k_j * hd^-0.5 + table[idx(i,j), h] with
//   idx(i,j) = (y_i - y_j + ws - 1) * (2ws - 1) + (x_i - x_j + ws - 1),   (y, x) = row / column of a token in its window.
//
//   expand : table [(2ws-1)^2, nh] -> dense bias [nh][64][64], rows / columns >= L = ws*ws set to zero, so every
//            (row < 64, head) a softmax thread can form reads in bounds
//   fold   : the attention backward's per-slot dS [nslots][nh][64][64] -> gtable [(2ws-1)^2, nh], summed in a fixed order
//            (run-to-run bit-identical, no atomics); gtable is overwritten
#include "swin_rpb.cuh"

namespace b200 {
namespace {

constexpr int kFoldRows = 16;   // slot groups per element in the fold's first stage

__global__ void rpb_expand_kernel(const float* __restrict__ table, float* __restrict__ bias, int ws, int nh) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;   // (h, i, j) of [nh][64][64]
  if (e >= nh * 4096) return;
  const int h = e >> 12, i = (e >> 6) & 63, j = e & 63, L = ws * ws;
  float v = 0.f;
  if (i < L && j < L) v = table[((i / ws - j / ws + ws - 1) * (2 * ws - 1) + (i % ws - j % ws + ws - 1)) * nh + h];
  bias[e] = v;
}

// dense[h][i][j] (i, j < L) = sum over all slots: thread (x, y) sums slots y, y + 16, ... of element x, then row y = 0 adds
// the 16 partial sums in order
__global__ void __launch_bounds__(32 * kFoldRows) rpb_fold_slots_kernel(const float* __restrict__ ws, long long nslots, int nh, int L,
                                                                       float* __restrict__ dense) {
  __shared__ float part[kFoldRows][33];
  const int LL = L * L;
  const int e = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (e < nh * LL) {
    const int h = e / LL, r = e - h * LL, i = r / L, j = r - i * L;
    const float* src = ws + (size_t)h * 4096 + i * 64 + j;
    for (long long s = threadIdx.y; s < nslots; s += kFoldRows) acc += src[s * nh * 4096];
  }
  part[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && e < nh * LL) {
    float t = part[0][threadIdx.x];
#pragma unroll
    for (int k = 1; k < kFoldRows; ++k) t += part[k][threadIdx.x];
    dense[e] = t;
  }
}

// gtable[idx, h] = sum of dense[h][i][j] over the (i, j) with idx(i, j) = idx: one warp per entry, lane k takes the k-th,
// (k+32)-th ... pair in query-row order, then a fixed butterfly
__global__ void rpb_fold_scatter_kernel(const float* __restrict__ dense, int nh, int ws, float* __restrict__ gtable) {
  const int D = 2 * ws - 1, L = ws * ws;
  const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (e >= D * D * nh) return;
  const int idx = e / nh, h = e - idx * nh;
  const int dy = idx / D - (ws - 1), dx = idx % D - (ws - 1);
  const int y0 = max(0, dy), x0 = max(0, dx), ny = ws - abs(dy), nx = ws - abs(dx);
  float acc = 0.f;
  for (int k = lane; k < ny * nx; k += 32) {
    const int yi = y0 + k / nx, xi = x0 + k % nx;
    acc += dense[(size_t)h * L * L + (yi * ws + xi) * L + (yi - dy) * ws + (xi - dx)];
  }
  acc = warp_sum(acc);
  if (lane == 0) gtable[e] = acc;
}

}  // namespace

int check_rpb(int L, int ws) {
  B200_REQUIRE(ws > 0 && ws <= kRpbMaxWs, B200_ERR_UNSUPPORTED, "swin_rpb: window size %d unsupported (1..%d)", ws, kRpbMaxWs);
  B200_REQUIRE(L == ws * ws, B200_ERR_SHAPE, "swin_rpb: window length %d != ws*ws (ws=%d)", L, ws);
  return B200_OK;
}

size_t rpb_workspace_bytes(long long nslots, int nh) {
  return ((size_t)nslots + 1) * (size_t)nh * 4096 * sizeof(float);   // the slots + the dense slot sum
}

int rpb_fold(const float* workspace, long long nslots, int nh, int ws, float* gtable, cudaStream_t st) {
  const int L = ws * ws;
  float* dense = const_cast<float*>(workspace) + (size_t)nslots * nh * 4096;
  rpb_fold_slots_kernel<<<(nh * L * L + 31) / 32, dim3(32, kFoldRows), 0, st>>>(workspace, nslots, nh, L, dense);
  if (int rc = check_launch("swin_rpb_fold_slots")) return rc;
  const int n = (2 * ws - 1) * (2 * ws - 1) * nh;
  rpb_fold_scatter_kernel<<<(n + 7) / 8, 256, 0, st>>>(dense, nh, ws, gtable);
  return check_launch("swin_rpb_fold_scatter");
}

}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_swin_rpb_expand(const float* table, int32_t table_rows, float* bias, int32_t ws, int32_t nh, void* stream) {
  if (int rc = check_rpb(ws * ws, ws)) return rc;
  B200_REQUIRE(nh > 0, B200_ERR_SHAPE, "swin_rpb_expand: bad head count %d", nh);
  B200_REQUIRE(table_rows == (2 * ws - 1) * (2 * ws - 1), B200_ERR_SHAPE, "swin_rpb_expand: table has %d rows, ws %d needs %d",
               table_rows, ws, (2 * ws - 1) * (2 * ws - 1));
  B200_REQUIRE(table && bias, B200_ERR_SHAPE, "swin_rpb_expand: null pointer");
  rpb_expand_kernel<<<(nh * 4096 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(table, bias, ws, nh);
  return check_launch("swin_rpb_expand");
}

extern "C" B200_API size_t b200_swin_rpb_workspace_bytes(int64_t tokens, int32_t L, int32_t nh, int32_t tc) {
  if (tokens <= 0 || L <= 0 || L > 64 || nh <= 0 || tokens % L != 0) return 0;
  const long long items = tokens / L * nh;
  const long long pairs = (items + 1) / 2;
  const long long slots = tc ? 4 * (pairs < kRpbTcCtas ? pairs : kRpbTcCtas) : tokens / L;
  return rpb_workspace_bytes(slots, nh);
}
