// Task-aligned assigner + box / DFL terms of the v8 detection loss as kernels over the Detect head's un-concatenated maps
// (SURVEY 8(f)-4).  Replaces, per training step, ultralytics/utils/loss.py:207-255 (`v8DetectionLoss.__call__`: bbox_decode, the
// assigner call, `BboxLoss.forward` = CIoU + DFL) and ultralytics/utils/tal.py:41-327 (`TaskAlignedAssigner.forward`,
// `get_pos_mask`, `get_box_metrics`, `select_topk_candidates`, `select_highest_overlaps`, `get_targets`) -- about 150 small ATen
// launches over [B, nmax, 8400] / [B, 8400, 4, 16] tensors -- by six launches:
//   det_decode   : per anchor: softmax-expectation of the 4 x 16 DFL logits -> predicted box (grid units); sigmoid of the class
//                  logit of every ground-truth box's own class (the only class scores the assigner reads)
//   tal_topk     : CTA per (image, GT): in-box test, CIoU overlap, alignment metric score^alpha * overlap^beta over all anchors
//                  (kept in shared memory), the top-k anchors by repeated block-wide arg-max (value, then lower anchor index)
//   tal_resolve  : per anchor: which GTs selected it; an anchor claimed by several GTs goes to the GT with the largest overlap
//                  (tal.py select_highest_overlaps); per-GT maxima of alignment / overlap over its positives (order-free atomicMax)
//   tal_finish   : per anchor: target label, normalised target value align * max_ovl / (max_align + eps), target box / stride
//   box_dfl_fwd  : sum over positives of (1 - CIoU) * weight and of the DFL cross-entropy * weight (per-CTA partials, fixed-order fold)
//   box_dfl_bwd  : gradient of both terms w.r.t. the DFL logits, written in the layout of the box maps (dense NHWC)
// The metric arithmetic mirrors the PyTorch restatement (harness/loss.py) operation by operation in f32 with explicitly rounded
// multiplies / adds (no FMA contraction), so the selected anchors are the same wherever the inputs are.
#include <math.h>

#include "common.cuh"

namespace b200 {
namespace {

inline size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }
constexpr int kMaxLevels = 4;
constexpr int kReg = 16;   // DFL bins per side (reg_max)
struct DetLevel {
  const void* box;   // [B * A, 64] DFL logits (dense NHWC box map)
  const void* cls;   // [B * A, nc] class logits
  void* gbox;        // gradient of the box map (backward)
  int H, W, A, a0;   // a0: offset of the level in the concatenated anchor axis
  float stride;
  long long rows;    // B * A
};
struct DetParams {
  DetLevel lv[kMaxLevels];
  int n_levels, B, A_total, nc, nmax, topk;
  long long rows_total;
  const float* gt;   // [B, nmax, 5]: class, x1, y1, x2, y2 (pixels); all-zero box = padding
  float* pred;       // [B, A_total, 4] predicted boxes, grid units
  float* scores;     // [B, nmax, A_total]
  int* sel_idx;      // [B, nmax, topk]
  float* sel_align;  // [B, nmax, topk]
  float* sel_ovl;    // [B, nmax, topk]
  unsigned* pos_align;   // [B, nmax] float bits (values >= 0: integer order = float order)
  unsigned* pos_ovl;     // [B, nmax]
  int* asg_j;        // [B, A_total] assigned GT (-1: background)
  float* asg_align;  // [B, A_total]
  int* tlabel;       // [B, A_total]
  float* tvalue;     // [B, A_total]
  float* tbox;       // [B, A_total, 4] target box, grid units
  float alpha, beta, eps;
  const float* gscale;   // backward: [2] upstream gradients of the two sums
  float* part;       // forward: [grid][2] partial sums
};

__device__ __forceinline__ int find_level(const DetParams& P, long long& r) {
  int l = 0;
  while (l + 1 < P.n_levels && r >= P.lv[l].rows) { r -= P.lv[l].rows; ++l; }
  return l;
}
__device__ __forceinline__ int level_of_anchor(const DetParams& P, int a) {
  int l = 0;
  while (l + 1 < P.n_levels && a >= P.lv[l].a0 + P.lv[l].A) ++l;
  return l;
}

template <typename T> __device__ __forceinline__ void load16(const T* p, float (&x)[kReg]);
template <> __device__ __forceinline__ void load16<float>(const float* p, float (&x)[kReg]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(p + 4 * q);
    x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
  }
}
template <> __device__ __forceinline__ void load16<__nv_bfloat16>(const __nv_bfloat16* p, float (&x)[kReg]) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const uint4 v = *reinterpret_cast<const uint4*>(p + 8 * q);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) { x[8 * q + 2 * e] = __uint_as_float(w[e] << 16); x[8 * q + 2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u); }
  }
}
template <> __device__ __forceinline__ void load16<__half>(const __half* p, float (&x)[kReg]) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const uint4 v = *reinterpret_cast<const uint4*>(p + 8 * q);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
      x[8 * q + 2 * e] = f.x; x[8 * q + 2 * e + 1] = f.y;
    }
  }
}
template <typename T> __device__ __forceinline__ void store16(T* p, const float (&g)[kReg]);
template <> __device__ __forceinline__ void store16<float>(float* p, const float (&g)[kReg]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) *reinterpret_cast<float4*>(p + 4 * q) = make_float4(g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]);
}
template <> __device__ __forceinline__ void store16<__nv_bfloat16>(__nv_bfloat16* p, const float (&g)[kReg]) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(g[8 * q + 2 * e], g[8 * q + 2 * e + 1]);
      w[e] = *reinterpret_cast<const uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p + 8 * q) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}
template <> __device__ __forceinline__ void store16<__half>(__half* p, const float (&g)[kReg]) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __half2 h = __floats2half2_rn(g[8 * q + 2 * e], g[8 * q + 2 * e + 1]);
      w[e] = *reinterpret_cast<const uint32_t*>(&h);
    }
    *reinterpret_cast<uint4*>(p + 8 * q) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// softmax of 16 logits (exp(x - max) / sum, as ATen's softmax) and its expectation over the bin index
__device__ __forceinline__ float softmax16(const float (&x)[kReg], float (&p)[kReg], float* lse = nullptr) {
  float m = x[0];
#pragma unroll
  for (int k = 1; k < kReg; ++k) m = fmaxf(m, x[k]);
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < kReg; ++k) { p[k] = expf(x[k] - m); s += p[k]; }
  if (lse) *lse = m + logf(s);   // log_softmax(x)[k] = x[k] - lse (finite where log(p[k]) would underflow)
  const float inv = 1.f / s;
  float d = 0.f;
#pragma unroll
  for (int k = 0; k < kReg; ++k) { p[k] *= inv; d += p[k] * (float)k; }
  return d;
}

// CIoU of b1 against b2 (xyxy), utils/metrics.py bbox_iou(xywh=False, CIoU=True) as restated in harness/loss.py:_ciou, operation by
// operation in f32 (explicitly rounded: the compiler must not contract a*b+c, ATen evaluates every op separately)
struct Box { float x1, y1, x2, y2; };
__device__ __forceinline__ float ciou_exact(const Box a, const Box b) {
  const float eps = 1e-7f;
  const float w1 = __fsub_rn(a.x2, a.x1), h1 = __fadd_rn(__fsub_rn(a.y2, a.y1), eps);
  const float w2 = __fsub_rn(b.x2, b.x1), h2 = __fadd_rn(__fsub_rn(b.y2, b.y1), eps);
  const float iw = fmaxf(__fsub_rn(fminf(a.x2, b.x2), fmaxf(a.x1, b.x1)), 0.f);
  const float ih = fmaxf(__fsub_rn(fminf(a.y2, b.y2), fmaxf(a.y1, b.y1)), 0.f);
  const float inter = __fmul_rn(iw, ih);
  const float uni = __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(w1, h1), __fmul_rn(w2, h2)), inter), eps);
  const float iou = __fdiv_rn(inter, uni);
  const float cw = __fsub_rn(fmaxf(a.x2, b.x2), fminf(a.x1, b.x1));
  const float ch = __fsub_rn(fmaxf(a.y2, b.y2), fminf(a.y1, b.y1));
  const float c2 = __fadd_rn(__fadd_rn(__fmul_rn(cw, cw), __fmul_rn(ch, ch)), eps);
  const float dx = __fsub_rn(__fsub_rn(__fadd_rn(b.x1, b.x2), a.x1), a.x2);
  const float dy = __fsub_rn(__fsub_rn(__fadd_rn(b.y1, b.y2), a.y1), a.y2);
  const float rho2 = __fdiv_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), 4.f);
  const float at = __fsub_rn(atanf(__fdiv_rn(w2, h2)), atanf(__fdiv_rn(w1, h1)));
  const float v = __fmul_rn((float)(4.0 / (M_PI * M_PI)), __fmul_rn(at, at));
  const float alpha = __fdiv_rn(v, __fadd_rn(__fsub_rn(v, iou), (float)(1.0 + 1e-7)));
  return __fsub_rn(iou, __fadd_rn(__fdiv_rn(rho2, c2), __fmul_rn(v, alpha)));
}

__device__ __forceinline__ Box gt_box(const DetParams& P, int b, int j) {
  const float* g = P.gt + ((size_t)b * P.nmax + j) * 5;
  return Box{g[1], g[2], g[3], g[4]};
}
__device__ __forceinline__ bool gt_valid(const Box g) { return __fadd_rn(__fadd_rn(__fadd_rn(g.x1, g.y1), g.x2), g.y2) > 0.f; }
// anchor centre in pixels and predicted box in pixels
__device__ __forceinline__ void anchor_geom(const DetParams& P, int b, int a, float* px, float* py, Box* pb) {
  const int l = level_of_anchor(P, a);
  const DetLevel& L = P.lv[l];
  const int al = a - L.a0, y = al / L.W, x = al - y * L.W;
  *px = ((float)x + 0.5f) * L.stride;
  *py = ((float)y + 0.5f) * L.stride;
  const float4 q = *reinterpret_cast<const float4*>(P.pred + ((size_t)b * P.A_total + a) * 4);
  *pb = Box{__fmul_rn(q.x, L.stride), __fmul_rn(q.y, L.stride), __fmul_rn(q.z, L.stride), __fmul_rn(q.w, L.stride)};
}
// tal.py select_candidates_in_gts: min(anchor - lt, rb - anchor) > eps (1e-9)
__device__ __forceinline__ bool in_box(const Box g, float px, float py) {
  const float d = fminf(fminf(__fsub_rn(px, g.x1), __fsub_rn(py, g.y1)), fminf(__fsub_rn(g.x2, px), __fsub_rn(g.y2, py)));
  return d > 1e-9f;
}
__device__ __forceinline__ float align_metric(const DetParams& P, float score, float ovl) {
  const float sa = P.alpha == 0.5f ? sqrtf(score) : powf(score, P.alpha);   // ATen's pow special-cases 0.5 as sqrt
  return __fmul_rn(sa, powf(ovl, P.beta));
}

// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) det_decode_kernel(const DetParams P) {
  const long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long r = gi >> 2;
  const int side = (int)(gi & 3);
  const bool live = r < P.rows_total;
  if (!live) r = P.rows_total - 1;   // keep the quad together for the shuffles
  const int l = find_level(P, r);
  const DetLevel& L = P.lv[l];
  const int b = (int)(r / L.A), al = (int)(r - (long long)b * L.A);
  float x[kReg], p[kReg];
  load16<T>(reinterpret_cast<const T*>(L.box) + r * (4 * kReg) + side * kReg, x);
  const float d = softmax16(x, p);
  const int base = (threadIdx.x & 31) & ~3;
  const float d0 = __shfl_sync(0xffffffffu, d, base), d1 = __shfl_sync(0xffffffffu, d, base + 1);
  const float d2 = __shfl_sync(0xffffffffu, d, base + 2), d3 = __shfl_sync(0xffffffffu, d, base + 3);
  if (!live) return;
  const int a = L.a0 + al;
  if (side == 0) {
    const int y = al / L.W, xx = al - y * L.W;
    const float ax = (float)xx + 0.5f, ay = (float)y + 0.5f;
    *reinterpret_cast<float4*>(P.pred + ((size_t)b * P.A_total + a) * 4) = make_float4(ax - d0, ay - d1, ax + d2, ay + d3);
  }
  const T* crow = reinterpret_cast<const T*>(L.cls) + r * P.nc;
  for (int j = side; j < P.nmax; j += 4) {
    int lab = (int)P.gt[((size_t)b * P.nmax + j) * 5];
    lab = min(max(lab, 0), P.nc - 1);
    const float z = DT<T>::to_f(crow[lab]);
    P.scores[((size_t)b * P.nmax + j) * P.A_total + a] = 1.f / (1.f + expf(-z));
  }
}

__global__ void __launch_bounds__(256) tal_topk_kernel(const DetParams P) {
  extern __shared__ float sm[];
  float* s_align = sm;                 // [A_total]
  float* s_ovl = sm + P.A_total;       // [A_total]
  __shared__ unsigned long long red[8];
  __shared__ unsigned long long winner;
  const int b = blockIdx.x / P.nmax, j = blockIdx.x - b * P.nmax;
  const Box g = gt_box(P, b, j);
  const size_t so = ((size_t)b * P.nmax + j) * P.topk;
  if (threadIdx.x == 0) { P.pos_align[b * P.nmax + j] = 0u; P.pos_ovl[b * P.nmax + j] = 0u; }
  if (!gt_valid(g)) {
    for (int k = threadIdx.x; k < P.topk; k += blockDim.x) { P.sel_idx[so + k] = -1; P.sel_align[so + k] = 0.f; P.sel_ovl[so + k] = 0.f; }
    return;
  }
  const float* sc = P.scores + ((size_t)b * P.nmax + j) * P.A_total;
  for (int a = threadIdx.x; a < P.A_total; a += blockDim.x) {
    float px, py;
    Box pb;
    anchor_geom(P, b, a, &px, &py, &pb);
    float al = 0.f, ov = 0.f;
    if (in_box(g, px, py)) {
      ov = fmaxf(ciou_exact(g, pb), 0.f);
      al = align_metric(P, sc[a], ov);
    }
    s_align[a] = al;
    s_ovl[a] = ov;
  }
  __syncthreads();
  for (int k = 0; k < P.topk; ++k) {
    unsigned long long best = 0ull;
    for (int a = threadIdx.x; a < P.A_total; a += blockDim.x) {
      const float v = s_align[a];
      if (v > 0.f) {
        const unsigned long long key = ((unsigned long long)__float_as_uint(v) << 32) | (unsigned long long)(0xffffffffu - (unsigned)a);
        best = key > best ? key : best;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
      best = other > best ? other : best;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long w = 0ull;
      for (int i = 0; i < (int)(blockDim.x >> 5); ++i) w = red[i] > w ? red[i] : w;
      winner = w;
      if (w) {
        const int a = (int)(0xffffffffu - (unsigned)(w & 0xffffffffull));
        P.sel_idx[so + k] = a; P.sel_align[so + k] = s_align[a]; P.sel_ovl[so + k] = s_ovl[a];
        s_align[a] = -1.f;
      } else {
        P.sel_idx[so + k] = -1; P.sel_align[so + k] = 0.f; P.sel_ovl[so + k] = 0.f;
      }
    }
    __syncthreads();
    if (!winner) {   // no positive candidate left: the remaining slots stay empty
      for (int k2 = k + 1 + threadIdx.x; k2 < P.topk; k2 += blockDim.x) { P.sel_idx[so + k2] = -1; P.sel_align[so + k2] = 0.f; P.sel_ovl[so + k2] = 0.f; }
      return;
    }
  }
}

__global__ void __launch_bounds__(256) tal_resolve_kernel(const DetParams P) {
  extern __shared__ int s_sel[];   // [nmax * topk] selected anchors of this image
  const int b = blockIdx.y, n = P.nmax * P.topk;
  for (int e = threadIdx.x; e < n; e += blockDim.x) s_sel[e] = P.sel_idx[(size_t)b * n + e];
  __syncthreads();
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= P.A_total) return;
  int count = 0, first = -1;
  for (int e = 0; e < n; ++e)
    if (s_sel[e] == a) { if (!count) first = e; ++count; }
  int j = -1;
  float al = 0.f, ov = 0.f;
  if (count == 1) {
    j = first / P.topk;
    al = P.sel_align[(size_t)b * n + first];
    ov = P.sel_ovl[(size_t)b * n + first];
  } else if (count > 1) {
    // claimed by several GTs: the GT with the largest (masked) overlap takes it (first maximum), whether or not it selected it
    float px, py;
    Box pb;
    anchor_geom(P, b, a, &px, &py, &pb);
    float best = -1.f;
    for (int q = 0; q < P.nmax; ++q) {
      const Box g = gt_box(P, b, q);
      float o = 0.f;
      if (gt_valid(g) && in_box(g, px, py)) o = fmaxf(ciou_exact(g, pb), 0.f);
      if (o > best) { best = o; j = q; }
    }
    ov = best;
    al = align_metric(P, P.scores[((size_t)b * P.nmax + j) * P.A_total + a], ov);
  }
  P.asg_j[(size_t)b * P.A_total + a] = j;
  P.asg_align[(size_t)b * P.A_total + a] = al;
  if (j >= 0) {
    atomicMax(P.pos_align + b * P.nmax + j, __float_as_uint(al));
    atomicMax(P.pos_ovl + b * P.nmax + j, __float_as_uint(ov));
  }
}

__global__ void __launch_bounds__(256) tal_finish_kernel(const DetParams P) {
  const int b = blockIdx.y;
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= P.A_total) return;
  const size_t i = (size_t)b * P.A_total + a;
  const int j = P.asg_j[i];
  int lab = -1;
  float val = 0.f;
  float4 tb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (j >= 0) {
    const float pa = __uint_as_float(P.pos_align[b * P.nmax + j]), po = __uint_as_float(P.pos_ovl[b * P.nmax + j]);
    val = __fdiv_rn(__fmul_rn(P.asg_align[i], po), __fadd_rn(pa, P.eps));
    const float* g = P.gt + ((size_t)b * P.nmax + j) * 5;
    lab = max((int)g[0], 0);
    const float st = P.lv[level_of_anchor(P, a)].stride;
    tb = make_float4(__fdiv_rn(g[1], st), __fdiv_rn(g[2], st), __fdiv_rn(g[3], st), __fdiv_rn(g[4], st));
  }
  P.tlabel[i] = lab;
  P.tvalue[i] = val;
  *reinterpret_cast<float4*>(P.tbox + i * 4) = tb;
}

// ---- box (CIoU) + DFL terms -------------------------------------------------------------------------------------
struct CiouGrad { float l, gx1, gy1, gx2, gy2; };   // l = 1 - ciou(pred, target); gradient of l w.r.t. the predicted box
__device__ __forceinline__ float d_max(float a, float b) { return a > b ? 1.f : (a == b ? 0.5f : 0.f); }   // d max(a,b) / d a (ATen splits ties)
__device__ __forceinline__ float d_min(float a, float b) { return a < b ? 1.f : (a == b ? 0.5f : 0.f); }
__device__ __forceinline__ CiouGrad ciou_loss_grad(const Box a, const Box t, bool want_grad) {
  const float eps = 1e-7f, kv = (float)(4.0 / (M_PI * M_PI));
  const float w1 = a.x2 - a.x1, h1 = a.y2 - a.y1 + eps, w2 = t.x2 - t.x1, h2 = t.y2 - t.y1 + eps;
  const float ix = fminf(a.x2, t.x2) - fmaxf(a.x1, t.x1), iy = fminf(a.y2, t.y2) - fmaxf(a.y1, t.y1);
  const float iw = fmaxf(ix, 0.f), ih = fmaxf(iy, 0.f), inter = iw * ih;
  const float uni = w1 * h1 + w2 * h2 - inter + eps, iou = inter / uni;
  const float cw = fmaxf(a.x2, t.x2) - fminf(a.x1, t.x1), ch = fmaxf(a.y2, t.y2) - fminf(a.y1, t.y1);
  const float c2 = cw * cw + ch * ch + eps;
  const float dx = t.x1 + t.x2 - a.x1 - a.x2, dy = t.y1 + t.y2 - a.y1 - a.y2;
  const float rho2 = (dx * dx + dy * dy) * 0.25f;
  const float u = w1 / h1, at = atanf(w2 / h2) - atanf(u), v = kv * at * at;
  const float alpha = v / (v - iou + (float)(1.0 + 1e-7));
  CiouGrad r;
  r.l = 1.f - (iou - (rho2 / c2 + v * alpha));
  if (want_grad) {
    const float iu2 = 1.f / (uni * uni);
    const float dinter = -(1.f / uni + inter * iu2);
    const float dat = alpha * 2.f * kv * at / (1.f + u * u);
    const float dw1 = inter * h1 * iu2 - dat / h1;
    const float dh1 = inter * w1 * iu2 + dat * w1 / (h1 * h1);
    const float dix = ix >= 0.f ? dinter * ih : 0.f, diy = iy >= 0.f ? dinter * iw : 0.f;
    const float dc2 = -rho2 / (c2 * c2), dcw = dc2 * 2.f * cw, dch = dc2 * 2.f * ch;
    const float hx = dx / (2.f * c2), hy = dy / (2.f * c2);
    r.gx1 = -dw1 - dix * d_max(a.x1, t.x1) - dcw * d_min(a.x1, t.x1) - hx;
    r.gx2 = dw1 + dix * d_min(a.x2, t.x2) + dcw * d_max(a.x2, t.x2) - hx;
    r.gy1 = -dh1 - diy * d_max(a.y1, t.y1) - dch * d_min(a.y1, t.y1) - hy;
    r.gy2 = dh1 + diy * d_min(a.y2, t.y2) + dch * d_max(a.y2, t.y2) - hy;
  }
  return r;
}
// DFL target of one side (loss.py:96-107 as restated): distance clamped to [0, reg_max - 1 - 0.01], left bin + weights
__device__ __forceinline__ void dfl_target(float dist, int* tl, float* wl) {
  const float d = fminf(fmaxf(dist, 0.f), (float)(kReg - 1) - 0.01f);
  *tl = (int)d;
  *wl = (float)(*tl + 1) - d;
}

template <typename T>
__global__ void __launch_bounds__(256) box_dfl_fwd_kernel(const DetParams P) {
  float acc_box = 0.f, acc_dfl = 0.f;
  for (long long r0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; r0 < P.rows_total; r0 += (long long)gridDim.x * blockDim.x) {
    long long r = r0;
    const int l = find_level(P, r);
    const DetLevel& L = P.lv[l];
    const int b = (int)(r / L.A), al = (int)(r - (long long)b * L.A);
    const size_t i = (size_t)b * P.A_total + L.a0 + al;
    const float wgt = P.tvalue[i];
    if (!(wgt > 0.f)) continue;
    const int y = al / L.W, xx = al - y * L.W;
    const float ax = (float)xx + 0.5f, ay = (float)y + 0.5f;
    const float4 tb = *reinterpret_cast<const float4*>(P.tbox + i * 4);
    const float tdist[4] = {ax - tb.x, ay - tb.y, tb.z - ax, tb.w - ay};
    float d[4], ce = 0.f;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      float x[kReg], p[kReg];
      load16<T>(reinterpret_cast<const T*>(L.box) + r * (4 * kReg) + s * kReg, x);
      float lse;
      d[s] = softmax16(x, p, &lse);
      int tl;
      float wl;
      dfl_target(tdist[s], &tl, &wl);
      float xl = 0.f, xr = 0.f;
#pragma unroll
      for (int k = 0; k < kReg; ++k) { xl = k == tl ? x[k] : xl; xr = k == tl + 1 ? x[k] : xr; }
      ce += (lse - xl) * wl + (lse - xr) * (1.f - wl);
    }
    const CiouGrad cg = ciou_loss_grad(Box{ax - d[0], ay - d[1], ax + d[2], ay + d[3]}, Box{tb.x, tb.y, tb.z, tb.w}, false);
    acc_box += cg.l * wgt;
    acc_dfl += ce * 0.25f * wgt;
  }
  __shared__ float red[8][2];
  acc_box = warp_sum(acc_box);
  acc_dfl = warp_sum(acc_dfl);
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = acc_box; red[threadIdx.x >> 5][1] = acc_dfl; }
  __syncthreads();
  if (threadIdx.x < 2) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
    P.part[blockIdx.x * 2 + threadIdx.x] = s;
  }
}
__global__ void __launch_bounds__(256) fold2_kernel(const float* __restrict__ part, int n, float* __restrict__ out) {
  __shared__ float red[8][2];
  float s0 = 0.f, s1 = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) { s0 += part[2 * i]; s1 += part[2 * i + 1]; }
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; }
  __syncthreads();
  if (threadIdx.x < 2) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    out[threadIdx.x] = t;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) box_dfl_bwd_kernel(const DetParams P) {
  const float g_box = P.gscale[0], g_dfl = P.gscale[1];
  const long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long r = gi >> 2;
  const int side = (int)(gi & 3);
  const bool live = r < P.rows_total;
  if (!live) r = P.rows_total - 1;
  const int l = find_level(P, r);
  const DetLevel& L = P.lv[l];
  const int b = (int)(r / L.A), al = (int)(r - (long long)b * L.A);
  const size_t i = (size_t)b * P.A_total + L.a0 + al;
  const float wgt = P.tvalue[i];
  float g[kReg];
#pragma unroll
  for (int k = 0; k < kReg; ++k) g[k] = 0.f;
  // a quad shares the anchor, hence the branch: no divergence inside a shuffle group
  if (wgt > 0.f) {
    float x[kReg], p[kReg];
    load16<T>(reinterpret_cast<const T*>(L.box) + r * (4 * kReg) + side * kReg, x);
    const float d = softmax16(x, p);
    const int base = (threadIdx.x & 31) & ~3;
    const unsigned qm = 0xfu << base;
    const float d0 = __shfl_sync(qm, d, base), d1 = __shfl_sync(qm, d, base + 1);
    const float d2 = __shfl_sync(qm, d, base + 2), d3 = __shfl_sync(qm, d, base + 3);
    const int y = al / L.W, xx = al - y * L.W;
    const float ax = (float)xx + 0.5f, ay = (float)y + 0.5f;
    const float4 tb = *reinterpret_cast<const float4*>(P.tbox + i * 4);
    const CiouGrad cg = ciou_loss_grad(Box{ax - d0, ay - d1, ax + d2, ay + d3}, Box{tb.x, tb.y, tb.z, tb.w}, true);
    // box = (ax - d0, ay - d1, ax + d2, ay + d3): d l / d d_side
    const float gd = side == 0 ? -cg.gx1 : side == 1 ? -cg.gy1 : side == 2 ? cg.gx2 : cg.gy2;
    const float tdist = side == 0 ? ax - tb.x : side == 1 ? ay - tb.y : side == 2 ? tb.z - ax : tb.w - ay;
    int tl;
    float wl;
    dfl_target(tdist, &tl, &wl);
    const float cb = g_box * wgt * gd, cd = g_dfl * wgt * 0.25f;
#pragma unroll
    for (int k = 0; k < kReg; ++k) {
      const float onehot = k == tl ? wl : (k == tl + 1 ? 1.f - wl : 0.f);
      g[k] = cb * p[k] * ((float)k - d) + cd * (p[k] - onehot);
    }
  }
  if (live) store16<T>(reinterpret_cast<T*>(L.gbox) + r * (4 * kReg) + side * kReg, g);
}

int fill_levels(DetParams& P, const void* const* box, const void* const* cls, void* const* gbox, const int32_t* H, const int32_t* W,
                const float* strides, int n_levels, int B) {
  B200_REQUIRE(n_levels >= 1 && n_levels <= kMaxLevels, B200_ERR_SHAPE, "det: 1..%d levels (got %d)", kMaxLevels, n_levels);
  B200_REQUIRE(B > 0, B200_ERR_SHAPE, "det: empty batch");
  P.n_levels = n_levels; P.B = B; P.A_total = 0; P.rows_total = 0;
  for (int l = 0; l < n_levels; ++l) {
    B200_REQUIRE(H[l] > 0 && W[l] > 0 && strides[l] > 0.f, B200_ERR_SHAPE, "det: bad level %d geometry", l);
    B200_REQUIRE((!box || (box[l] && ((uintptr_t)box[l] & 15) == 0)) && (!gbox || (gbox[l] && ((uintptr_t)gbox[l] & 15) == 0)) &&
                     (!cls || cls[l]), B200_ERR_ALIGN, "det: level %d needs 16-byte aligned maps", l);
    DetLevel& L = P.lv[l];
    L.box = box ? box[l] : nullptr; L.cls = cls ? cls[l] : nullptr; L.gbox = gbox ? gbox[l] : nullptr;
    L.H = H[l]; L.W = W[l]; L.A = H[l] * W[l]; L.a0 = P.A_total; L.stride = strides[l]; L.rows = (long long)B * L.A;
    P.A_total += L.A;
    P.rows_total += L.rows;
  }
  B200_REQUIRE(P.rows_total * 4 < (1ll << 31), B200_ERR_SHAPE, "det: too many anchors");
  return B200_OK;
}
bool dtype_ok(int dtype) { return dtype == B200_F32 || dtype == B200_BF16 || dtype == B200_F16; }

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" B200_API int b200_det_decode(const void* const* box_maps, const void* const* cls_maps, const int32_t* H, const int32_t* W,
                                        const float* strides, int32_t n_levels, const float* gt, float* pred_boxes, float* scores,
                                        int32_t B, int32_t nc, int32_t nmax, int32_t dtype, void* stream) {
  DetParams P{};
  B200_REQUIRE(box_maps && cls_maps && gt && pred_boxes && scores, B200_ERR_SHAPE, "det_decode: null pointer");
  B200_REQUIRE(dtype_ok(dtype), B200_ERR_DTYPE, "det_decode: unsupported dtype %d", dtype);
  B200_REQUIRE(nc > 0 && nmax > 0, B200_ERR_SHAPE, "det_decode: nc / nmax must be positive");
  if (int rc = fill_levels(P, box_maps, cls_maps, nullptr, H, W, strides, n_levels, B)) return rc;
  P.nc = nc; P.nmax = nmax; P.gt = gt; P.pred = pred_boxes; P.scores = scores;
  const long long threads = P.rows_total * 4;
  const int grid = (int)((threads + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_F32) det_decode_kernel<float><<<grid, 256, 0, st>>>(P);
  else if (dtype == B200_BF16) det_decode_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(P);
  else det_decode_kernel<__half><<<grid, 256, 0, st>>>(P);
  return check_launch("det_decode");
}

extern "C" B200_API size_t b200_tal_workspace_bytes(int32_t B, int32_t nmax, int32_t A_total, int32_t topk) {
  const size_t sel = up256((size_t)B * nmax * topk * 4);
  return 3 * sel + 2 * up256((size_t)B * nmax * 4) + 2 * up256((size_t)B * A_total * 4);
}

extern "C" B200_API int b200_tal_assign(const float* pred_boxes, const float* scores, const float* gt, const int32_t* H, const int32_t* W,
                                        const float* strides, int32_t n_levels, int32_t* target_label, float* target_value,
                                        float* target_box, void* workspace, size_t workspace_bytes, int32_t B, int32_t nmax, int32_t topk,
                                        float alpha, float beta, float eps, void* stream) {
  DetParams P{};
  B200_REQUIRE(pred_boxes && scores && gt && target_label && target_value && target_box, B200_ERR_SHAPE, "tal_assign: null pointer");
  B200_REQUIRE(nmax > 0 && topk > 0 && topk <= 64, B200_ERR_SHAPE, "tal_assign: nmax > 0 and 0 < topk <= 64 required");
  if (int rc = fill_levels(P, nullptr, nullptr, nullptr, H, W, strides, n_levels, B)) return rc;
  B200_REQUIRE(workspace && workspace_bytes >= b200_tal_workspace_bytes(B, nmax, P.A_total, topk), B200_ERR_WORKSPACE,
               "tal_assign: workspace too small");
  P.nmax = nmax; P.topk = topk; P.gt = gt; P.pred = const_cast<float*>(pred_boxes); P.scores = const_cast<float*>(scores);
  P.alpha = alpha; P.beta = beta; P.eps = eps;
  P.tlabel = target_label; P.tvalue = target_value; P.tbox = target_box;
  char* w = (char*)workspace;
  const size_t sel = up256((size_t)B * nmax * topk * 4), pg = up256((size_t)B * nmax * 4), pa = up256((size_t)B * P.A_total * 4);
  P.sel_idx = (int*)w; w += sel;
  P.sel_align = (float*)w; w += sel;
  P.sel_ovl = (float*)w; w += sel;
  P.pos_align = (unsigned*)w; w += pg;
  P.pos_ovl = (unsigned*)w; w += pg;
  P.asg_j = (int*)w; w += pa;
  P.asg_align = (float*)w;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem_topk = (size_t)P.A_total * 8;
  B200_REQUIRE(smem_topk <= (size_t)max_smem_optin(), B200_ERR_UNSUPPORTED, "tal_assign: %d anchors do not fit in shared memory", P.A_total);
  cudaFuncSetAttribute(tal_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_topk);
  tal_topk_kernel<<<B * nmax, 256, smem_topk, st>>>(P);
  if (int rc = check_launch("tal_topk")) return rc;
  const dim3 grid((P.A_total + 255) / 256, B);
  const size_t smem_sel = (size_t)nmax * topk * 4;
  B200_REQUIRE(smem_sel <= 48 * 1024, B200_ERR_UNSUPPORTED, "tal_assign: nmax * topk = %d too large", nmax * topk);
  tal_resolve_kernel<<<grid, 256, smem_sel, st>>>(P);
  if (int rc = check_launch("tal_resolve")) return rc;
  tal_finish_kernel<<<grid, 256, 0, st>>>(P);
  return check_launch("tal_finish");
}

extern "C" B200_API size_t b200_box_dfl_workspace_bytes(void) { return (size_t)(sm_count() * 4) * 2 * sizeof(float); }

extern "C" B200_API int b200_box_dfl_fwd(const void* const* box_maps, const int32_t* H, const int32_t* W, int32_t n_levels,
                                         const float* target_box, const float* weight, float* sums, void* workspace,
                                         size_t workspace_bytes, int32_t B, int32_t dtype, void* stream) {
  DetParams P{};
  B200_REQUIRE(box_maps && target_box && weight && sums, B200_ERR_SHAPE, "box_dfl_fwd: null pointer");
  B200_REQUIRE(dtype_ok(dtype), B200_ERR_DTYPE, "box_dfl_fwd: unsupported dtype %d", dtype);
  B200_REQUIRE(workspace && workspace_bytes >= b200_box_dfl_workspace_bytes(), B200_ERR_WORKSPACE, "box_dfl_fwd: workspace too small");
  const float ones[kMaxLevels] = {1.f, 1.f, 1.f, 1.f};
  if (int rc = fill_levels(P, box_maps, nullptr, nullptr, H, W, ones, n_levels, B)) return rc;
  P.tbox = const_cast<float*>(target_box); P.tvalue = const_cast<float*>(weight); P.part = (float*)workspace;
  const int grid = sm_count() * 4;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_F32) box_dfl_fwd_kernel<float><<<grid, 256, 0, st>>>(P);
  else if (dtype == B200_BF16) box_dfl_fwd_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(P);
  else box_dfl_fwd_kernel<__half><<<grid, 256, 0, st>>>(P);
  if (int rc = check_launch("box_dfl_fwd")) return rc;
  fold2_kernel<<<1, 256, 0, st>>>(P.part, grid, sums);
  return check_launch("box_dfl_fold");
}

extern "C" B200_API int b200_box_dfl_bwd(const void* const* box_maps, void* const* grad_maps, const int32_t* H, const int32_t* W,
                                         int32_t n_levels, const float* target_box, const float* weight, const float* grad_sums, int32_t B,
                                         int32_t dtype, void* stream) {
  DetParams P{};
  B200_REQUIRE(box_maps && grad_maps && target_box && weight && grad_sums, B200_ERR_SHAPE, "box_dfl_bwd: null pointer");
  B200_REQUIRE(dtype_ok(dtype), B200_ERR_DTYPE, "box_dfl_bwd: unsupported dtype %d", dtype);
  const float ones[kMaxLevels] = {1.f, 1.f, 1.f, 1.f};
  if (int rc = fill_levels(P, box_maps, nullptr, grad_maps, H, W, ones, n_levels, B)) return rc;
  P.tbox = const_cast<float*>(target_box); P.tvalue = const_cast<float*>(weight); P.gscale = grad_sums;
  const long long threads = P.rows_total * 4;
  const int grid = (int)((threads + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B200_F32) box_dfl_bwd_kernel<float><<<grid, 256, 0, st>>>(P);
  else if (dtype == B200_BF16) box_dfl_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(P);
  else box_dfl_bwd_kernel<__half><<<grid, 256, 0, st>>>(P);
  return check_launch("box_dfl_bwd");
}
