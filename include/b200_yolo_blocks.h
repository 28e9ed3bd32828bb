/*
 * b200_yolo_blocks.h -- C-ABI of the B200 (sm_100a) kernels behind the CBAM / SwinBlock / SPPF drop-ins.
 *
 * The reference (mazouziwissem/improving_yolov8_CBAM_SwinBlock, an Ultralytics 8.3.108 fork) is pure Python:
 * its "operator interface" for this path is the nn.Module.forward of three classes that parse_model binds by
 * name (ultralytics/nn/tasks.py:1438).  Each entry point below replaces the ATen op sequence of one of those
 * forwards (or of its autograd backward) and is what a ctypes / cffi stub on the reference side binds
 * (INTEGRATION.md shows the stub).  Conventions (SURVEY.md section 8b):
 *
 *   - plain pointers + sizes only; device pointers unless stated; no torch types.
 *   - activations are NHWC-dense ("channels_last"): element (b,c,h,w) lives at ((b*H+h)*W+w)*C+c.
 *   - dtype codes: 0=f32, 1=bf16, 2=f16 for activations; parameters and parameter gradients are always f32.
 *   - every call only ENQUEUES work on `stream` (a cudaStream_t passed as void*) of the current device;
 *     no hidden synchronisation, no allocation: scratch memory is passed in as `workspace`.
 *   - return 0 on success, a B200_ERR_* code otherwise (message via b200_last_error(), thread-local);
 *     nothing throws or exits across the ABI.  Stateless and re-entrant.
 */
#ifndef B200_YOLO_BLOCKS_H_
#define B200_YOLO_BLOCKS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 3
#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

enum { B200_F32 = 0, B200_BF16 = 1, B200_F16 = 2 };
enum {
  B200_OK = 0,
  B200_ERR_SHAPE = 1,
  B200_ERR_DTYPE = 2,
  B200_ERR_ALIGN = 3,
  B200_ERR_LAUNCH = 4,
  B200_ERR_WORKSPACE = 5,
  B200_ERR_UNSUPPORTED = 6
};

B200_API int b200_abi_version(void);
B200_API const char* b200_last_error(void);
/* number of kernel launches enqueued through this library by the calling process so far (bench bookkeeping) */
B200_API uint64_t b200_launch_count(void);

/* ------------------------------------------------------------------------------------------------------
 * SPPF pooling cascade -- replaces `y = [cv1(x)]; y.extend(self.m(y[-1]) for _ in range(3)); torch.cat(y, 1)`
 * (ultralytics/nn/modules/block.py:224-226; self.m = MaxPool2d(k, 1, k//2), block.py:220).
 *   y0  [B,H,W,C]   in
 *   cat [B,H,W,4C]  out: channel slices [y0 | m(y0) | m(m(y0)) | m(m(m(y0)))]
 *   idx [3,B,H,W,C] optional (NULL to skip): per-stage argmax as torch's flat h*W+w index into the previous
 *                   stage's plane, with ATen's rule (row-major window scan, replace iff val>max or isnan(val)).
 * k odd, 3 <= k <= 13.  Values are exact selections: bit-exact in every dtype.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_sppf_pool_fwd(const void* y0, void* cat, int32_t* idx, int32_t B, int32_t C, int32_t H, int32_t W,
                       int32_t k, int32_t dtype, void* stream);
/* backward of the cascade + concat w.r.t. y0 (autograd of block.py:224-226):
 *   gcat [B,H,W,4C] in, y0 [B,H,W,C] in (argmax maps are recomputed from it with the same rule),
 *   gy0 [B,H,W,C] out.  Deterministic (no atomics); accumulation in f32. */
B200_API int b200_sppf_pool_bwd(const void* gcat, const void* y0, void* gy0, int32_t B, int32_t C, int32_t H, int32_t W,
                       int32_t k, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * CBAM -- replaces CBAM.forward / ChannelAttention.forward / SpatialAttention.forward
 * (ultralytics/nn/modules/cbam.py:62-71, :29-38, :48-53).
 *   mode B200_CBAM_FULL : out[B,H,W,C] = x * ca * sa        (cbam.py:62-71)
 *   mode B200_CBAM_CA   : ca_out[B,C]  = sigmoid(MLP(avg)+MLP(max))   only (cbam.py:29-38), `out` unused
 *   mode B200_CBAM_SA   : sa_out[B,H*W] = sigmoid(conv(cat[mean_c x, max_c x])) only (cbam.py:48-53)
 *   w1 [r,C], w2 [C,r]  shared_MLP.{0,2}.weight (no bias, cbam.py:24-26); wsa [2,ksa,ksa] sa.conv.weight,
 *   ksa in {3,7} (cbam.py:43).  ca_out / sa_out (f32) may be NULL in FULL mode when no backward is needed.
 *   stash (nullable): b200_cbam_stash_bytes(...) bytes that receive the forward's small by-products for the
 *   backward (pooled avg/max [B,2,C], first-argmax pixel per channel [B,C], mean_c / max_c / argmax_c maps [B,3,HW]).
 *   workspace: b200_cbam_fwd_workspace_bytes(...) bytes of device scratch.
 * ------------------------------------------------------------------------------------------------------ */
enum { B200_CBAM_FULL = 0, B200_CBAM_CA = 1, B200_CBAM_SA = 2 };
B200_API size_t b200_cbam_stash_bytes(int32_t B, int32_t C, int32_t H, int32_t W);
B200_API size_t b200_cbam_fwd_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W, int32_t dtype);
B200_API int b200_cbam_fwd(const void* x, const float* w1, const float* w2, const float* wsa, void* out, float* ca_out,
                  float* sa_out, void* stash, void* workspace, size_t workspace_bytes, int32_t B, int32_t C,
                  int32_t H, int32_t W, int32_t r, int32_t ksa, int32_t dtype, int32_t mode, void* stream);
/* backward (autograd of the same forwards; SURVEY.md App. A.1).
 *   FULL: g = dL/dout [B,H,W,C];  CA: g = dL/dca [B,C] (f32);  SA: g = dL/dsa [B,H*W] (f32).
 *   ca/sa: the maps written by the forward (f32); stash: the forward's stash.  gx [B,H,W,C] out (activation dtype).
 *   gw1 [r,C], gw2 [C,r], gwsa [2,ksa,ksa]: f32, OVERWRITTEN (not accumulated).
 *   workspace: b200_cbam_bwd_workspace_bytes(...) bytes of device scratch (per-pixel maps and per-image / per-slice
 *   weight-gradient partials, folded in a fixed order: deterministic, no atomics). */
B200_API size_t b200_cbam_bwd_workspace_bytes(int32_t B, int32_t C, int32_t H, int32_t W, int32_t r, int32_t dtype);
B200_API int b200_cbam_bwd(const void* g, const void* x, const float* w1, const float* w2, const float* wsa,
                  const float* ca, const float* sa, const void* stash, void* gx, float* gw1, float* gw2,
                  float* gwsa, void* workspace, size_t workspace_bytes, int32_t B, int32_t C, int32_t H, int32_t W,
                  int32_t r, int32_t ksa, int32_t dtype, int32_t mode, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * SwinBlock stages -- replace SwinBlock.forward (ultralytics/nn/modules/swin_block.py:37-58) and its autograd
 * backward.  x is NHWC [B,H,W,C]; "tokens" are the zero-padded, window-partitioned rows
 *   t = ((b*nWh + wh)*nWw + ww)*L + r*ws + c,   L = ws*ws,  nWh = ceil(H/ws), nWw = ceil(W/ws)
 * (swin_block.py:8-13,41-47).  T = b200_swin_num_tokens(...).
 * EXTENSION (not in the reference, whose block is unshifted -- SURVEY D1): `shift` in [0, ws) cyclically shifts the padded
 * map by (-shift, -shift) before partitioning (folded into the token -> pixel addressing of every stage) and the
 * attention entry points then mask, in registers before the softmax, the keys that lie across the wrap-around seam
 * (windows of the last window row / column; `nWh, nWw, ws` describe the window grid).  shift == 0 is the reference block
 * and ignores nWh / nWw / ws.  The dense contractions between the stages
 * (in_proj / out_proj / mlp.0 / mlp.2, torch F.linear in the reference) are b200_gemm_* below.
 * ------------------------------------------------------------------------------------------------------ */
B200_API long long b200_swin_num_tokens(int32_t B, int32_t H, int32_t W, int32_t ws);
/* n1[T,C] = LayerNorm_1(partition(pad(x)))  (swin_block.py:41-50); mean/rstd [T] f32 saved for the backward */
B200_API int b200_swin_ln1_partition(const void* x, const float* gamma, const float* beta, void* n1, float* mean,
                                     float* rstd, int32_t B, int32_t C, int32_t H, int32_t W, int32_t ws,
                                     int32_t shift, int32_t dtype, void* stream);
/* windowed multi-head attention on packed rows qkv[T,3C] (q|k|v) -> o[T,C]; lse[T,nh] f32 (swin_block.py:51,
 * torch F.multi_head_attention_forward: q*hd^-0.5, softmax over the window's L keys, heads concatenated) */
B200_API int b200_swin_attn_fwd(const void* qkv, void* o, float* lse, int64_t tokens, int32_t L, int32_t C,
                                int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                void* stream);
B200_API int b200_swin_attn_bwd(const void* qkv, const void* o, const float* lse, const void* go, void* gqkv,
                                int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw,
                                int32_t ws, int32_t shift, int32_t dtype, void* stream);
/* y1 = n1 + a (post-norm residual, swin_block.py:52, SURVEY D2);  u = LayerNorm_2(y1) (swin_block.py:53).
 * a == NULL: `n1` already holds y1 (residual fused into the out_proj GEMM) and y1 is not written. */
B200_API int b200_swin_res_ln2(const void* n1, const void* a, const float* gamma, const float* beta, void* y1,
                               void* u, float* mean, float* rstd, int64_t tokens, int32_t C, int32_t dtype,
                               void* stream);
/* GELU(erf) forward (backward=0: out = gelu(a)) / backward (backward=1: out = gh * gelu'(a)), swin_block.py:33 */
B200_API int b200_swin_gelu(const void* a, const void* gh, void* out, int64_t n, int32_t dtype, int32_t backward,
                            void* stream);
/* out[B,H,W,C] = reverse(crop(y1 + m))  (swin_block.py:53-58) */
B200_API int b200_swin_res_reverse(const void* y1, const void* m, void* out, int32_t B, int32_t C, int32_t H,
                                   int32_t W, int32_t ws, int32_t shift, int32_t dtype, void* stream);
/* tok[T,C] = partition(pad(src)) without normalisation (used for the upstream gradient) */
B200_API int b200_swin_partition(const void* src, void* tok, int32_t B, int32_t C, int32_t H, int32_t W,
                                 int32_t ws, int32_t shift, int32_t dtype, void* stream);
/* the same with a second addend in pixel layout: tok = partition(src + add) -- used to add the residual gradient g_out to the
 * LayerNorm-backward term that b200_swin_mlp_bwd leaves in g_y1 */
B200_API int b200_swin_partition_add(const void* src, const void* add, void* tok, int32_t B, int32_t C, int32_t H, int32_t W,
                                     int32_t ws, int32_t shift, int32_t dtype, void* stream);
/* LayerNorm backward.  mode 0 (LN2): token-major, gin = LN^T(gout) + gres.  mode 1 (LN1): xin = x (NHWC, gathered
 * through the window map), gin = gx scattered back to NHWC; ggamma/gbeta [C] f32 overwritten; norm1.bias receives
 * gradient from padded tokens too (SURVEY App. A.3). */
B200_API size_t b200_swin_ln_bwd_workspace_bytes(int64_t tokens, int32_t C);
B200_API int b200_swin_ln_bwd(const void* gout, const void* xin, const void* gres, const float* gamma,
                              const float* mean, const float* rstd, void* gin, float* ggamma, float* gbeta,
                              void* workspace, size_t workspace_bytes, int32_t B, int32_t C, int32_t H,
                              int32_t W, int32_t ws, int32_t shift, int32_t dtype, int32_t mode, void* stream);
/* out[n] f32 = column sums of a[rows,n]  (bias gradients) */
B200_API size_t b200_colsum_workspace_bytes(int64_t rows, int32_t n);
B200_API int b200_colsum(const void* a, float* out, void* workspace, size_t workspace_bytes, int64_t rows,
                         int32_t n, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Channel concat of channels_last maps: the seams around the blocks (SURVEY 8(f)-2) -- `torch.cat(y, 1)` of
 * C2f.forward (block.py), Concat.forward (conv.py), the Detect head (head.py:66-76), and the backward of
 * `chunk(2, 1)`.  Source i is a row-strided view [rows, src_channels[i]] with row stride src_row_stride[i]
 * elements (>= channels: a channel slice of a wider NHWC tensor qualifies); dst is dense [rows, sum channels].
 * 1..8 sources; 16-byte vectors when every pointer / width / stride allows, element copies otherwise.
 * srcs / src_channels / src_row_stride are HOST arrays.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_nhwc_concat(const void* const* srcs, const int32_t* src_channels, const int64_t* src_row_stride,
                              int32_t n_src, void* dst, int64_t rows, int32_t dtype, void* stream);
/* Gradient fan-in at the seams: dst[rows, cols] (dense) = sum of 2..4 row-strided sources [rows, cols] of one dtype
 * (row stride src_row_stride[i] >= cols elements), summed in f32 in source order and rounded once.  Replaces the adds
 * autograd issues where a map has several consumers -- a bottleneck output inside C2f (block.py C2f.forward:
 * `y.extend(m(y[-1]) for m in self.m)` feeds the next bottleneck AND the concat) and the saved layers `y[j]` of
 * `_predict_once` (tasks.py:171-176) -- one operand there is a channel slice of a concat's gradient, which ATen adds
 * through its generic strided kernel.  Rows, pointers and strides must be 16-byte multiples.  HOST arrays. */
B200_API int b200_nhwc_add(const void* const* srcs, const int64_t* src_row_stride, int32_t n_src, void* dst, int64_t rows,
                           int32_t cols, int32_t dtype, void* stream);
/* Input seam: uint8 NCHW image batch -> `img.float() / divisor` in `dtype`, NHWC, one pass (detect/train.py:100 +
 * the channels_last conversion + autocast's cast of the first conv input).  Bit-identical to ATen's CUDA division by a
 * host scalar (multiply by the f32 reciprocal) followed by one round-to-nearest conversion.  1..4 channels, H*W % 4 == 0. */
B200_API int b200_u8_to_nhwc(const void* img, void* out, int32_t B, int32_t C, int32_t H, int32_t W, float divisor,
                             int32_t dtype, void* stream);
/* Nearest-neighbour up-sampling by integer factors (sh, sw) on NHWC maps -- the `nn.Upsample(None, 2, "nearest")` rows
 * of the yaml head -- and its backward (f32 sum of the sh*sw gradients of one input pixel, fixed order).  H, W are the
 * INPUT sizes; C must span a multiple of 16 bytes.  gout_row_stride: elements between consecutive pixels of gout
 * (0 = dense = C; a concat-slice gradient is read in place). */
B200_API int b200_nhwc_upsample_fwd(const void* x, void* out, int32_t B, int32_t C, int32_t H, int32_t W, int32_t sh,
                                    int32_t sw, int32_t dtype, void* stream);
B200_API int b200_nhwc_upsample_bwd(const void* gout, int64_t gout_row_stride, void* gin, int32_t B, int32_t C, int32_t H,
                                    int32_t W, int32_t sh, int32_t sw, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * tcgen05 GEMM for the SwinBlock's dense contractions (torch F.linear at swin_block.py:51,53):
 *   D[M,N] = epi(A[M,K] * B[N,K]^T + bias[N]),  A/B/D/D2/R in the 16-bit activation dtype (bf16 | f16), f32 accumulate.
 *   epi 0: bias;  epi 1: D = gelu_erf(a), D2 (nullable) = a = pre-activation;  epi 2: D = a + R[M,N] (residual);
 *   epi 3: D = a * gelu_erf'(R[M,N])  (GELU backward fused into the mlp.2 data-gradient GEMM).
 * b200_gemm_nt_supported() tells whether the problem is one the kernel tiles.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_gemm_nt_supported(int64_t M, int32_t N, int32_t K, int32_t dtype);
B200_API int b200_gemm_nt(const void* A, const void* B, const float* bias, void* D, void* D2, const void* R,
                          int64_t M, int32_t N, int32_t K, int32_t dtype, int32_t epi, void* stream);

/* Split-K tcgen05 GEMM with selectable operand majorness, f32 output (weight gradients dW = dY^T X, autograd of
 * F.linear at swin_block.py:51,53, are the a_mn=b_mn=1 form with K = tokens):
 *   D[M,N] (f32) = sum_k A(m,k) * B(n,k);  a_mn=0: A is [M,K] row-major, a_mn=1: A is [K,M] row-major; same for B/N.
 * colsum (nullable, f32 [M]) = sum_k A(m,k): the bias gradient sum_t dY[t,:] falls out of the same pass as one extra
 * N=16 MMA against a tile of ones.  Deterministic: per-split f32 partials in `workspace` folded in a fixed order. */
B200_API size_t b200_gemm_splitk_workspace_bytes(int32_t M, int32_t N, int64_t K);
B200_API int b200_gemm_splitk(const void* A, const void* B, float* D, float* colsum, void* workspace,
                              size_t workspace_bytes, int32_t M, int32_t N, int64_t K, int32_t a_mn, int32_t b_mn,
                              int32_t dtype, void* stream);

/* Window attention on tcgen05 tensor cores (bf16 | f16, L <= 64, head dim 64 or 128): same contract as
 * b200_swin_attn_fwd / _bwd.  b200_swin_attn_tc_supported() says whether the problem qualifies. */
B200_API int b200_swin_attn_tc_supported(int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t dtype);
B200_API int b200_swin_attn_fwd_tc(const void* qkv, void* o, float* lse, int64_t tokens, int32_t L, int32_t C,
                                   int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                   void* stream);
B200_API int b200_swin_attn_bwd_tc(const void* qkv, const float* lse, const void* go, void* gqkv, int64_t tokens,
                                   int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws,
                                   int32_t shift, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Learned relative-position bias of window attention (SwinBlockRPB; EXTENSION: the reference block has none, SURVEY D1).
 * Liu et al. 2021, "Swin Transformer: Hierarchical Vision Transformer using Shifted Windows", eq. 4:
 *   S[h,i,j] = (q_i . k_j) * hd^-0.5 + table[idx(i,j), h]   (+ the shift mask when shift > 0)
 *   idx(i,j) = (y_i - y_j + ws - 1) * (2ws - 1) + (x_i - x_j + ws - 1),  (y, x) = row / column of a token in its window
 * table [(2ws-1)^2, nh] f32 (table_rows = (2ws-1)^2), 1 <= ws <= 8, L = ws*ws.  Padded and shifted windows use the same
 * index by window position, as in Swin.  lse is that of the biased scores.
 *   b200_swin_rpb_expand : table -> dense bias [nh][64][64] f32, rows / columns >= L zero (what the attention entries read)
 *   *_fwd_rpb / *_fwd_tc_rpb : b200_swin_attn_fwd / _fwd_tc with the dense bias added to the scores before the softmax
 *   *_bwd_rpb / *_bwd_tc_rpb : b200_swin_attn_bwd / _bwd_tc plus gtable [(2ws-1)^2, nh] f32 = dL/dtable, OVERWRITTEN and
 *       run-to-run bit-identical (per-slot dS in `workspace`, folded in a fixed order; no atomics).  workspace:
 *       b200_swin_rpb_workspace_bytes(tokens, L, nh, tc) bytes, tc = 1 for the _tc entry, 0 for the SIMT one.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_swin_rpb_expand(const float* table, int32_t table_rows, float* bias, int32_t ws, int32_t nh, void* stream);
B200_API size_t b200_swin_rpb_workspace_bytes(int64_t tokens, int32_t L, int32_t nh, int32_t tc);
B200_API int b200_swin_attn_fwd_rpb(const void* qkv, const float* bias, void* o, float* lse, int64_t tokens, int32_t L,
                                    int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                    void* stream);
B200_API int b200_swin_attn_bwd_rpb(const void* qkv, const void* o, const float* lse, const void* go, const float* bias,
                                    void* gqkv, float* gtable, int32_t table_rows, void* workspace, size_t workspace_bytes,
                                    int64_t tokens, int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws,
                                    int32_t shift, int32_t dtype, void* stream);
B200_API int b200_swin_attn_fwd_tc_rpb(const void* qkv, const float* bias, void* o, float* lse, int64_t tokens, int32_t L,
                                       int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift, int32_t dtype,
                                       void* stream);
B200_API int b200_swin_attn_bwd_tc_rpb(const void* qkv, const float* lse, const void* go, const float* bias, void* gqkv,
                                       float* gtable, int32_t table_rows, void* workspace, size_t workspace_bytes, int64_t tokens,
                                       int32_t L, int32_t C, int32_t nh, int32_t nWh, int32_t nWw, int32_t ws, int32_t shift,
                                       int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Conv epilogue -- replaces `self.act(self.bn(y))` of Conv.forward (ultralytics/nn/modules/conv.py:65-79:
 * BatchNorm2d then SiLU) on the conv output y, for SPPF's cv1/cv2 (block.py:218-219; SURVEY section 8(f)-1) and the
 * other Conv callers either side of the path.  x/z/gz/gx: NHWC viewed as [rows = B*H*W, C] in the activation dtype;
 * gamma, beta, running_mean, running_var, mean, rstd, ggamma, gbeta: f32 [C].
 *   training != 0: batch statistics of THIS GPU (no SyncBN, like the reference), running_mean/var updated in place
 *                  as torch does (momentum; unbiased variance); mean_out/rstd_out (nullable) saved for the backward.
 *   training == 0: running statistics.   act: 1 = SiLU, 0 = identity.
 * b200_bn_silu_supported(): C a multiple of 16 bytes of elements, C <= 256 vectors.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_bn_silu_supported(int64_t rows, int32_t C, int32_t dtype);
B200_API size_t b200_bn_silu_workspace_bytes(int64_t rows, int32_t C, int32_t dtype);
B200_API int b200_bn_silu_fwd(const void* x, const float* gamma, const float* beta, float* running_mean,
                              float* running_var, void* z, float* mean_out, float* rstd_out, void* workspace,
                              size_t workspace_bytes, int64_t rows, int32_t C, float eps, float momentum,
                              int32_t training, int32_t act, int32_t dtype, void* stream);
/* Same, plus nn.BatchNorm2d.forward's bookkeeping (torch/nn/modules/batchnorm.py: `self.num_batches_tracked.add_(1)` in training
 * mode) folded into the finalize kernel: `num_batches_tracked` is the module's int64 device scalar (NULL: not touched). */
B200_API int b200_bn_silu_fwd_tracked(const void* x, const float* gamma, const float* beta, float* running_mean,
                                      float* running_var, int64_t* num_batches_tracked, void* z, float* mean_out, float* rstd_out,
                                      void* workspace, size_t workspace_bytes, int64_t rows, int32_t C, float eps, float momentum,
                                      int32_t training, int32_t act, int32_t dtype, void* stream);
/* backward: gx = dL/dx, ggamma / gbeta OVERWRITTEN; mean/rstd = the statistics the forward normalised with
 * (training == 0: pass running_mean and 1/sqrt(running_var + eps)).  Deterministic (no atomics).
 * gz_row_stride: elements between consecutive rows of gz (0 = dense = C); the gradient that reaches a Conv feeding a
 * concat is a channel slice of the concat's gradient, read in place instead of being copied first. */
B200_API int b200_bn_silu_bwd(const void* gz, int64_t gz_row_stride, const void* x, const float* gamma, const float* beta, const float* mean,
                              const float* rstd, void* gx, float* ggamma, float* gbeta, void* workspace,
                              size_t workspace_bytes, int64_t rows, int32_t C, int32_t training, int32_t act,
                              int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Fused MLP half of the SwinBlock -- replaces `x_windows + self.mlp(self.norm2(x_windows))`, `window_reverse` and the
 * crop (ultralytics/nn/modules/swin_block.py:53-58) for 16-bit activations with C = 128, in ONE tcgen05 kernel per
 * direction: LayerNorm2 -> mlp.0 -> GELU -> mlp.2 -> + residual with the [rows, 4C] hidden activation kept on chip
 * (TMEM / shared memory).  Rows are the real tokens in pixel order (y1 [rows = B*H*W, C], NHWC-dense).
 *   b200_swin_mlp_prep : w1f = mlp.0.weight * norm2.weight (16-bit), b1f = mlp.0.bias + mlp.0.weight @ norm2.bias (f32),
 *                        w2h = mlp.2.weight / 2 (16-bit; the kernels form 2 * gelu) -- LayerNorm's affine part folded
 *                        into the first GEMM.
 *   b200_swin_mlp_fwd  : out = y1 + mlp.2(gelu(xhat @ w1f^T + b1f)) + b2,  xhat = (y1 - mean) * rstd per row; in training
 *                        the 16-bit tiles 2*gelu(a) that feed the second GEMM are also stored (h2) for the backward.
 *   b200_swin_mlp_bwd  : from g_out [rows, C] and y1 recomputes xhat / the hidden pre-activation and writes
 *                        g_y1 [rows, C] (the LayerNorm2-backward term; the residual "+ g_out" is added by the consumer,
 *                        b200_swin_partition_add) plus the operands of the weight-gradient contractions it owns:
 *                        xhat [rows, C] and g_a [rows, 4C]   (d mlp.0.weight = g_a^T xhat * gamma + ...,
 *                        d mlp.2.weight = g_out^T h2 / 2 with the forward's h2: b200_gemm_splitk).
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_swin_mlp_supported(int64_t rows, int32_t C, int32_t dtype);
B200_API int b200_swin_mlp_prep(const float* w1, const float* b1, const float* gamma, const float* beta, const float* w2,
                                void* w1f, float* b1f, void* w2h, int32_t C, int32_t dtype, void* stream);
B200_API int b200_swin_mlp_fwd(const void* y1, const void* w1f, const float* b1f, const void* w2h, const float* b2, void* out,
                               void* h2 /* optional [rows, 4C]: 2*gelu(a), saved for the backward */, int64_t rows, int32_t C,
                               float eps, int32_t dtype, void* stream);
B200_API int b200_swin_mlp_bwd(const void* gout, const void* y1, const void* w1f, const float* b1f, const void* w2h, void* gy1,
                               void* xhat, void* ga, int64_t rows, int32_t C, float eps, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Fused attention half of the SwinBlock -- replaces F.pad, rearrange, window_partition, norm1, nn.MultiheadAttention and the
 * first residual add (ultralytics/nn/modules/swin_block.py:41-52) plus window_reverse / crop for that half (:55-58), for
 * 16-bit activations with C = 128, 2 heads, window <= 8 and no shift, in ONE tcgen05 kernel:
 *     y1 [B,H,W,C] (pixel order) = n1 + out_proj(MHSA(n1)),  n1 = LayerNorm1(window tokens of the zero-padded x).
 * w_in [3C,C] / w_out [C,C] are the 16-bit copies of attn.in_proj_weight / attn.out_proj.weight; biases and LayerNorm
 * parameters f32.  Training (n1 != NULL): the by-products the backward consumes are written too, in window-token order
 * (T = b200_swin_num_tokens rows): n1 [T,C], qkv [T,3C], o [T,C], lse [T,2], mean / rstd [T].
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_swin_attn_block_supported(int32_t B, int32_t C, int32_t H, int32_t W, int32_t heads, int32_t ws, int32_t shift,
                                            int32_t dtype);
B200_API int b200_swin_attn_block_fwd(const void* x, const float* gamma, const float* beta, const void* w_in, const float* b_in,
                                      const void* w_out, const float* b_out, void* y1, void* n1, void* qkv, void* o, float* lse,
                                      float* mean, float* rstd, int32_t B, int32_t C, int32_t H, int32_t W, int32_t heads,
                                      int32_t ws, float eps, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Classification term of the v8 detection loss (SURVEY 8(f)-4) -- replaces, for the class logits of
 * ultralytics/utils/loss.py:207-213,235 (`self.bce(pred_scores, target_scores.to(dtype)).sum()`), the cat / permute /
 * contiguous / float copies of the three Detect levels, the dense one-hot target of TaskAlignedAssigner (tal.py:98-107)
 * and BCEWithLogits forward + backward, by one streaming read of the logits per direction.
 *   logits[l]  : class map of level l, NHWC-dense (or row-strided) [B * anchors[l], C] with row stride row_stride[l] elements
 *   label,value: [B, sum(anchors)] target of each anchor: t[b,a,c] = value * (c == label); label < 0 = background
 *   fwd: loss_sum[0] = sum softplus(x) - x*t (f32, deterministic).   bwd: grads[l] = (sigmoid(x) - t) * scale[0], same layout.
 * ------------------------------------------------------------------------------------------------------ */
B200_API size_t b200_bce_logits_workspace_bytes(void);
B200_API int b200_bce_logits_fwd(const void* const* logits, const int32_t* anchors, const int64_t* row_stride, int32_t n_levels,
                                 const int32_t* label, const float* value, float* loss_sum, void* workspace, size_t workspace_bytes,
                                 int32_t B, int32_t C, int32_t dtype, void* stream);
B200_API int b200_bce_logits_bwd(const void* const* logits, void* const* grads, const int32_t* anchors, const int64_t* row_stride,
                                 int32_t n_levels, const int32_t* label, const float* value, const float* scale, int32_t B, int32_t C,
                                 int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Task-aligned assigner + box / DFL terms of the v8 detection loss (SURVEY 8(f)-4) on the Detect head's un-concatenated maps.
 * Replaces ultralytics/utils/loss.py:207-255 (`v8DetectionLoss.__call__`: `bbox_decode` :199, the assigner call :224-232,
 * `BboxLoss.forward` :84-107 = CIoU + DFL) and ultralytics/utils/tal.py:41-327 (`TaskAlignedAssigner.forward`, `get_pos_mask`,
 * `get_box_metrics`, `select_topk_candidates`, `select_highest_overlaps`, `get_targets`).
 *   box_maps[l] : DFL logits of level l, NHWC-dense [B * H[l] * W[l], 64] (4 sides x reg_max 16); cls_maps[l]: [B * H*W, nc]
 *   gt          : [B, nmax, 5] f32 rows (class, x1, y1, x2, y2 in pixels); an all-zero box is padding (loss.py:175-190)
 *   anchors of all levels are concatenated level-major: A = sum H[l] * W[l]; anchor centre = (x + 0.5, y + 0.5) grid units
 * b200_det_decode : pred_boxes [B, A, 4] f32 = anchor -/+ softmax-expectation of the DFL logits (grid units);
 *                   scores [B, nmax, A] f32 = sigmoid(class logit of GT j's own class) -- all the assigner reads of the class maps
 * b200_tal_assign : target_label [B, A] (int32, -1 = background), target_value [B, A] (the normalised alignment metric =
 *                   the value of the one-hot target_scores row), target_box [B, A, 4] (grid units).  top-k ties: lower anchor
 *                   index; anchors with a zero metric are never selected (they carry a zero target either way)
 * b200_box_dfl_fwd: sums[0] = sum_a (1 - CIoU(pred_a, target_a)) * weight_a, sums[1] = sum_a DFL(a) * weight_a  (weight = target_value)
 * b200_box_dfl_bwd: grad_maps[l] = grad_sums[0] * d sums[0] / d logits + grad_sums[1] * d sums[1] / d logits, layout of box_maps
 * No atomics on floating-point sums (per-GT maxima use an order-free integer atomicMax): deterministic.
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_det_decode(const void* const* box_maps, const void* const* cls_maps, const int32_t* H, const int32_t* W,
                             const float* strides, int32_t n_levels, const float* gt, float* pred_boxes, float* scores, int32_t B,
                             int32_t nc, int32_t nmax, int32_t dtype, void* stream);
B200_API size_t b200_tal_workspace_bytes(int32_t B, int32_t nmax, int32_t A_total, int32_t topk);
B200_API int b200_tal_assign(const float* pred_boxes, const float* scores, const float* gt, const int32_t* H, const int32_t* W,
                             const float* strides, int32_t n_levels, int32_t* target_label, float* target_value, float* target_box,
                             void* workspace, size_t workspace_bytes, int32_t B, int32_t nmax, int32_t topk, float alpha, float beta,
                             float eps, void* stream);
B200_API size_t b200_box_dfl_workspace_bytes(void);
B200_API int b200_box_dfl_fwd(const void* const* box_maps, const int32_t* H, const int32_t* W, int32_t n_levels, const float* target_box,
                              const float* weight, float* sums, void* workspace, size_t workspace_bytes, int32_t B, int32_t dtype,
                              void* stream);
B200_API int b200_box_dfl_bwd(const void* const* box_maps, void* const* grad_maps, const int32_t* H, const int32_t* W, int32_t n_levels,
                              const float* target_box, const float* weight, const float* grad_sums, int32_t B, int32_t dtype,
                              void* stream);

/* ------------------------------------------------------------------------------------------------------
 * The model's first convolution: Conv(3, c2, k=3, s=2, p=1), bias-free (yaml backbone row 0: `[-1, 1, Conv, [64, 3, 2]]` scaled;
 * ultralytics/nn/modules/conv.py:37-91 `self.conv`), on a 16-bit NHWC image x [B, H, W, 3] -> y [B, H/2, W/2, c2], and its weight
 * gradient (the input needs none).  w / gw: [c2, 3, 3, 3] f32 (OIHW, as nn.Conv2d.weight).  H even, W % 32 == 0, c2 in {16, 32, 48}.
 * Deterministic (per-CTA partial matrices folded in a fixed order).
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_stem_conv_supported(int32_t H, int32_t W, int32_t c2, int32_t dtype);
B200_API int b200_stem_conv_fwd(const void* x, const float* w, void* y, int32_t B, int32_t H, int32_t W, int32_t c2, int32_t dtype,
                                void* stream);
B200_API size_t b200_stem_conv_wgrad_workspace_bytes(int32_t c2);
B200_API int b200_stem_conv_wgrad(const void* gy, const void* x, float* gw, void* workspace, size_t workspace_bytes, int32_t B, int32_t H,
                                  int32_t W, int32_t c2, int32_t dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Weight gradient of the narrow 3x3 convolutions at the top of the model (yaml backbone rows 1-2 at scale n: the 16 -> 32 stride-2
 * Conv and the 16 -> 16 C2f bottleneck convolutions: nn.Conv2d(16, cout, 3, stride, 1, bias=False), cout in {16, 32}, stride 1 or 2;
 * conv.py:37-91 `self.conv`; wider layers stay on cuDNN, whose sm100 kernels are faster there): gw [cout, cin, 3, 3] f32 = d loss / d weight from x [B, H, W, cin] and gy [B, H/stride, W/stride, cout] (16-bit NHWC).
 * (W / stride) % 16 == 0.  Deterministic.  The forward and the input gradient stay the caller's (cuDNN).
 * ------------------------------------------------------------------------------------------------------ */
B200_API int b200_conv3x3_wgrad_supported(int32_t H, int32_t W, int32_t cin, int32_t cout, int32_t stride, int32_t dtype);
B200_API size_t b200_conv3x3_wgrad_workspace_bytes(int32_t cin, int32_t cout);
B200_API int b200_conv3x3_wgrad(const void* gy, const void* x, float* gw, void* workspace, size_t workspace_bytes, int32_t B, int32_t H,
                                int32_t W, int32_t cin, int32_t cout, int32_t stride, int32_t dtype, void* stream);

/* Input gradient of the stride-2 member of that family (yaml backbone row 1 at scale n: nn.Conv2d(16, 32, 3, 2, 1, bias=False);
 * autograd of F.conv2d w.r.t. the input, conv.py:37-91 `self.conv`): gx [B, H, W, 16] from gy [B, H/2, W/2, 32] (16-bit NHWC) and
 * the weight w [32, 16, 3, 3] in the same 16-bit dtype, read through its element strides (w_stride = {oc, ci, ky, kx}: the
 * parameter is channels_last in the harness).  cuDNN runs its generic strided-dgrad kernel there (0.38 ms, 8x its HBM time);
 * here each of the four input-pixel parities is its own small implicit GEMM (1, 2, 2 and 4 taps) on mma.sync.
 * H, W even, (W / 2) % 16 == 0, cin == 16, cout == 32. */
B200_API int b200_conv3x3_dgrad_s2_supported(int32_t H, int32_t W, int32_t cin, int32_t cout, int32_t dtype);
B200_API int b200_conv3x3_dgrad_s2(const void* gy, const void* w, const int64_t* w_stride, void* gx, int32_t B, int32_t H, int32_t W,
                                   int32_t cin, int32_t cout, int32_t dtype, void* stream);
/* Forward of the same layer (nn.Conv2d(16, 32, 3, 2, 1, bias=False) on 16-bit NHWC maps): y [B, H/2, W/2, 32] from x [B, H, W, 16]
 * and w [32, 16, 3, 3] (16-bit, element strides as for the input gradient).  cuDNN picks an sm80 legacy fprop there (0.14 ms, 3x the HBM time).
 * Implicit GEMM on mma.sync: M = 16 output pixels, N = 32, K = 9 taps x 16 channels, the A operand read by ldmatrix straight from
 * the staged NHWC input rows (stride-2 pixel addresses, XOR-swizzled 16-byte chunks).  Same shape limits as the input gradient
 * (b200_conv3x3_dgrad_s2_supported answers for both). */
B200_API int b200_conv3x3_fwd_s2(const void* x, const void* w, const int64_t* w_stride, void* y, int32_t B, int32_t H, int32_t W,
                                 int32_t cin, int32_t cout, int32_t dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_YOLO_BLOCKS_H_ */
