"""torch.autograd.Function wrappers over the C-ABI kernels (include/b200_yolo_blocks.h).

PyTorch is plumbing here: it owns device memory, streams and the autograd graph; every number on the CBAM /
SwinBlock / SPPF path is produced by ``libb200yolo.so``.  Tensors are logical NCHW (what the callers in
``ultralytics/nn/tasks.py:171`` pass) held in channels_last memory = the NHWC layout the kernels address; an
NCHW-contiguous input is converted once on entry (run the model ``channels_last`` to avoid that copy).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import call, dtype_code, lib, ptr, stream_ptr

_I64, _I32, _VP, _SZ = C.c_int64, C.c_int32, C.c_void_p, C.c_size_t
_lib.register("b200_swin_num_tokens", C.c_longlong, [_I32] * 4)
_lib.register("b200_swin_ln1_partition", C.c_int, [_VP] * 6 + [_I32] * 7 + [_VP])
_lib.register("b200_swin_attn_fwd", C.c_int, [_VP] * 3 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_bwd", C.c_int, [_VP] * 5 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_tc_supported", C.c_int, [_I64] + [_I32] * 4)
_lib.register("b200_swin_attn_fwd_tc", C.c_int, [_VP] * 3 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_bwd_tc", C.c_int, [_VP] * 4 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_rpb_expand", C.c_int, [_VP, _I32, _VP, _I32, _I32, _VP])
_lib.register("b200_swin_rpb_workspace_bytes", _SZ, [_I64, _I32, _I32, _I32])
_lib.register("b200_swin_attn_fwd_rpb", C.c_int, [_VP] * 4 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_bwd_rpb", C.c_int, [_VP] * 7 + [_I32, _VP, _SZ, _I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_fwd_tc_rpb", C.c_int, [_VP] * 4 + [_I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_attn_bwd_tc_rpb", C.c_int, [_VP] * 6 + [_I32, _VP, _SZ, _I64] + [_I32] * 8 + [_VP])
_lib.register("b200_swin_res_ln2", C.c_int, [_VP] * 8 + [_I64] + [_I32] * 2 + [_VP])
_lib.register("b200_swin_gelu", C.c_int, [_VP] * 3 + [_I64] + [_I32] * 2 + [_VP])
_lib.register("b200_swin_res_reverse", C.c_int, [_VP] * 3 + [_I32] * 7 + [_VP])
_lib.register("b200_swin_partition", C.c_int, [_VP] * 2 + [_I32] * 7 + [_VP])
_lib.register("b200_swin_partition_add", C.c_int, [_VP] * 3 + [_I32] * 7 + [_VP])
_lib.register("b200_swin_ln_bwd_workspace_bytes", _SZ, [_I64, _I32])
_lib.register("b200_swin_ln_bwd", C.c_int, [_VP] * 10 + [_SZ] + [_I32] * 8 + [_VP])
_lib.register("b200_colsum_workspace_bytes", _SZ, [_I64, _I32])
_lib.register("b200_colsum", C.c_int, [_VP] * 3 + [_SZ] + [_I64] + [_I32] * 2 + [_VP])
_lib.register("b200_bn_silu_supported", C.c_int, [_I64, _I32, _I32])
_lib.register("b200_bn_silu_workspace_bytes", _SZ, [_I64, _I32, _I32])
_lib.register("b200_bn_silu_fwd", C.c_int, [_VP] * 9 + [_SZ, _I64, _I32, C.c_float, C.c_float, _I32, _I32, _I32, _VP])
_lib.register("b200_bn_silu_fwd_tracked", C.c_int, [_VP] * 10 + [_SZ, _I64, _I32, C.c_float, C.c_float, _I32, _I32, _I32, _VP])
_lib.register("b200_bn_silu_bwd", C.c_int, [_VP, _I64] + [_VP] * 9 + [_SZ, _I64, _I32, _I32, _I32, _I32, _VP])
_lib.register("b200_det_decode", C.c_int, [_VP] * 5 + [_I32] + [_VP] * 3 + [_I32] * 4 + [_VP])
_lib.register("b200_tal_workspace_bytes", _SZ, [_I32] * 4)
_lib.register("b200_tal_assign", C.c_int, [_VP] * 6 + [_I32] + [_VP] * 4 + [_SZ] + [_I32] * 3 + [C.c_float] * 3 + [_VP])
_lib.register("b200_box_dfl_workspace_bytes", _SZ, [])
_lib.register("b200_box_dfl_fwd", C.c_int, [_VP] * 3 + [_I32] + [_VP] * 4 + [_SZ, _I32, _I32, _VP])
_lib.register("b200_box_dfl_bwd", C.c_int, [_VP] * 4 + [_I32] + [_VP] * 3 + [_I32, _I32, _VP])
_lib.register("b200_stem_conv_supported", C.c_int, [_I32] * 4)
_lib.register("b200_stem_conv_fwd", C.c_int, [_VP] * 3 + [_I32] * 5 + [_VP])
_lib.register("b200_stem_conv_wgrad_workspace_bytes", _SZ, [_I32])
_lib.register("b200_stem_conv_wgrad", C.c_int, [_VP] * 4 + [_SZ] + [_I32] * 5 + [_VP])
_lib.register("b200_conv3x3_wgrad_supported", C.c_int, [_I32] * 6)
_lib.register("b200_conv3x3_wgrad_workspace_bytes", _SZ, [_I32] * 2)
_lib.register("b200_conv3x3_wgrad", C.c_int, [_VP] * 4 + [_SZ] + [_I32] * 7 + [_VP])
_lib.register("b200_conv3x3_dgrad_s2_supported", C.c_int, [_I32] * 5)
_lib.register("b200_conv3x3_dgrad_s2", C.c_int, [_VP, _VP, _VP, _VP] + [_I32] * 6 + [_VP])
_lib.register("b200_conv3x3_fwd_s2", C.c_int, [_VP, _VP, _VP, _VP] + [_I32] * 6 + [_VP])
_lib.register("b200_nhwc_concat", C.c_int, [_VP, _VP, _VP, _I32, _VP, _I64, _I32, _VP])
_lib.register("b200_nhwc_add", C.c_int, [_VP, _VP, _I32, _VP, _I64, _I32, _I32, _VP])
_lib.register("b200_u8_to_nhwc", C.c_int, [_VP, _VP] + [_I32] * 4 + [C.c_float, _I32, _VP])
_lib.register("b200_nhwc_upsample_fwd", C.c_int, [_VP, _VP] + [_I32] * 7 + [_VP])
_lib.register("b200_nhwc_upsample_bwd", C.c_int, [_VP, _I64, _VP] + [_I32] * 7 + [_VP])
_lib.register("b200_bce_logits_workspace_bytes", _SZ, [])
_lib.register("b200_bce_logits_fwd", C.c_int, [_VP, _VP, _VP, _I32, _VP, _VP, _VP, _VP, _SZ, _I32, _I32, _I32, _VP])
_lib.register("b200_bce_logits_bwd", C.c_int, [_VP, _VP, _VP, _VP, _I32, _VP, _VP, _VP, _I32, _I32, _I32, _VP])
_lib.register("b200_swin_attn_block_supported", C.c_int, [_I32] * 8)
_lib.register("b200_swin_attn_block_fwd", C.c_int, [_VP] * 14 + [_I32] * 6 + [C.c_float, _I32, _VP])
_lib.register("b200_swin_mlp_supported", C.c_int, [_I64, _I32, _I32])
_lib.register("b200_swin_mlp_prep", C.c_int, [_VP] * 8 + [_I32, _I32, _VP])
_lib.register("b200_swin_mlp_fwd", C.c_int, [_VP] * 7 + [_I64, _I32, C.c_float, _I32, _VP])
_lib.register("b200_swin_mlp_bwd", C.c_int, [_VP] * 8 + [_I64, _I32, C.c_float, _I32, _VP])


def _nhwc(x: torch.Tensor) -> torch.Tensor:
    """Return x (logical [B,C,H,W]) in dense channels_last memory."""
    if x.dim() != 4:
        raise RuntimeError(f"expected a 4-D [B,C,H,W] tensor, got shape {tuple(x.shape)}")
    if not x.is_cuda:
        raise RuntimeError("B200 kernels need a CUDA tensor (there is no CPU compute path in this package)")
    return x.contiguous(memory_format=torch.channels_last)


def _empty_nhwc(B, Cc, H, W, dtype, device):
    return torch.empty((B, Cc, H, W), dtype=dtype, device=device, memory_format=torch.channels_last)


def _f32(w: torch.Tensor) -> torch.Tensor:
    return w.detach().to(torch.float32).contiguous()


# --------------------------------------------------------------------------------------------------
# channel concat / chunk of channels_last maps (the seams around the blocks: C2f, Concat, Detect head)
# --------------------------------------------------------------------------------------------------
def _row_strided(t: torch.Tensor):
    """Row stride S (elements) if t [B,C,H,W] is a channel slice of a dense channels_last map, else None."""
    B, Cc, H, W = t.shape
    S = t.stride(3) if W > 1 else (t.stride(2) if H > 1 else (t.stride(0) if B > 1 else Cc))
    if S < Cc or (Cc > 1 and t.stride(1) != 1):
        return None
    if (W > 1 and t.stride(3) != S) or (H > 1 and t.stride(2) != W * S) or (B > 1 and t.stride(0) != H * W * S):
        return None
    return S


def nhwc_concat_raw(tensors) -> torch.Tensor:
    """cat(tensors, 1) into a dense channels_last tensor with one vectorised copy kernel; sources may be channel slices."""
    t0 = tensors[0]
    B, _, H, W = t0.shape
    strides = [_row_strided(t) for t in tensors]
    if any(st is None for st in strides):   # an NCHW-dense operand: convert that one, as the kernels' callers always do
        tensors = [t if st is not None else _nhwc(t) for t, st in zip(tensors, strides)]
        strides = [_row_strided(t) for t in tensors]
    chans = [int(t.shape[1]) for t in tensors]
    out = _empty_nhwc(B, sum(chans), H, W, t0.dtype, t0.device)
    n = len(tensors)
    srcs = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
    cc = (C.c_int32 * n)(*chans)
    ss = (C.c_int64 * n)(*[int(v) for v in strides])
    with torch.cuda.device(t0.device):
        call("b200_nhwc_concat", C.addressof(srcs), C.addressof(cc), C.addressof(ss), n, ptr(out), B * H * W, dtype_code(t0.dtype),
             stream_ptr(t0.device), tag=f"b200_nhwc_concat[{B * H * W}x{sum(chans)}]")
    return out


def _concat_ok(tensors) -> bool:
    t0 = tensors[0]
    return (t0.is_cuda and t0.dim() == 4 and 1 <= len(tensors) <= 8 and t0.dtype in (torch.float32, torch.bfloat16, torch.float16)
            and all(t.is_cuda and t.device == t0.device and t.dim() == 4 and t.dtype == t0.dtype and t.shape[0] == t0.shape[0]
                    and t.shape[2:] == t0.shape[2:] for t in tensors))


class NhwcConcatFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, *tensors):
        ctx.chans = [int(t.shape[1]) for t in tensors]
        return nhwc_concat_raw(tensors)

    @staticmethod
    def backward(ctx, g):
        outs, off = [], 0
        for i, c in enumerate(ctx.chans):   # channel slices of g (views, like aten's cat backward)
            outs.append(g.narrow(1, off, c) if ctx.needs_input_grad[i] else None)
            off += c
        return tuple(outs)


class NhwcChunkFn(torch.autograd.Function):
    """x.chunk(n, 1) whose backward is ONE concat kernel (aten: SplitBackward -> generic strided cat)."""

    @staticmethod
    def forward(ctx, x, n):
        parts = x.chunk(n, 1)
        ctx.meta = (x.shape, x.dtype, x.device, [int(p.shape[1]) for p in parts])
        return parts

    @staticmethod
    def backward(ctx, *gs):
        shape, dtype, device, chans = ctx.meta
        B, _, H, W = shape
        gs = [g if g is not None else torch.zeros((B, c, H, W), dtype=dtype, device=device).contiguous(memory_format=torch.channels_last)
              for g, c in zip(gs, chans)]
        return nhwc_concat_raw(gs), None


def nhwc_concat(tensors) -> torch.Tensor:
    """Drop-in for ``torch.cat(tensors, 1)`` on 4-D CUDA maps (result in channels_last memory); anything else -> torch.cat."""
    tensors = list(tensors)
    if not _concat_ok(tensors):
        return torch.cat(tensors, 1)
    return NhwcConcatFn.apply(*tensors)


def u8_to_nhwc(img: torch.Tensor, dtype: torch.dtype = torch.float32, divisor: float = 255.0) -> torch.Tensor:
    """uint8 NCHW image batch -> ``img.float() / divisor`` in ``dtype`` and channels_last memory, one kernel (the trainer's
    input seam, detect/train.py:100).  Bit-identical to ATen's CUDA ``img.float() / divisor`` (a multiply by the f32 reciprocal)
    followed by one cast to ``dtype``."""
    if not (img.is_cuda and img.dtype == torch.uint8 and img.dim() == 4 and img.is_contiguous()):
        raise RuntimeError("u8_to_nhwc: expected a contiguous uint8 CUDA tensor [B,C,H,W]")
    B, Cc, H, W = img.shape
    out = _empty_nhwc(B, Cc, H, W, dtype, img.device)
    with torch.cuda.device(img.device):
        call("b200_u8_to_nhwc", ptr(img), ptr(out), B, Cc, H, W, float(divisor), dtype_code(dtype), stream_ptr(img.device))
    return out


class NhwcUpsampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, sh, sw):
        x = _nhwc(x)
        B, Cc, H, W = x.shape
        ctx.cfg = (B, Cc, H, W, sh, sw)
        out = _empty_nhwc(B, Cc, H * sh, W * sw, x.dtype, x.device)
        with torch.cuda.device(x.device):
            call("b200_nhwc_upsample_fwd", ptr(x), ptr(out), B, Cc, H, W, sh, sw, dtype_code(x.dtype), stream_ptr(x.device))
        return out

    @staticmethod
    def backward(ctx, g):
        B, Cc, H, W, sh, sw = ctx.cfg
        gs = _row_strided(g)   # a channel slice of the following Concat's gradient is read in place
        if gs is None or (gs * g.element_size()) % 16 or g.data_ptr() % 16:
            g, gs = _nhwc(g), Cc
        gin = _empty_nhwc(B, Cc, H, W, g.dtype, g.device)
        with torch.cuda.device(g.device):
            call("b200_nhwc_upsample_bwd", ptr(g), gs, ptr(gin), B, Cc, H, W, sh, sw, dtype_code(g.dtype), stream_ptr(g.device))
        return gin, None, None


def nhwc_upsample_nearest(x: torch.Tensor, sh: int, sw: int) -> torch.Tensor:
    """``F.interpolate(x, scale_factor=(sh, sw), mode="nearest")`` for integer factors on a CUDA map, channels_last result."""
    if not (x.is_cuda and x.dim() == 4 and x.dtype in (torch.float32, torch.bfloat16, torch.float16)
            and (x.shape[1] * x.element_size()) % 16 == 0):
        return torch.nn.functional.interpolate(x, scale_factor=(float(sh), float(sw)), mode="nearest")
    return NhwcUpsampleFn.apply(x, int(sh), int(sw))


def nhwc_chunk(x: torch.Tensor, n: int):
    """Drop-in for ``x.chunk(n, 1)`` (views of x) with the concat kernel as its backward."""
    if not (x.is_cuda and x.dim() == 4 and x.dtype in (torch.float32, torch.bfloat16, torch.float16) and _row_strided(x) is not None):
        return x.chunk(n, 1)
    return NhwcChunkFn.apply(x, n)


# --------------------------------------------------------------------------------------------------
# gradient fan-in: a map with several consumers (C2f bottleneck outputs, the saved layers of `_predict_once`)
# --------------------------------------------------------------------------------------------------
def _add_ok(gs) -> bool:
    g0 = gs[0]
    es = g0.element_size()
    if not (g0.is_cuda and g0.dim() == 4 and 2 <= len(gs) <= 4 and g0.dtype in (torch.float32, torch.bfloat16, torch.float16)
            and (g0.shape[1] * es) % 16 == 0):
        return False
    for g in gs:
        if not (g.is_cuda and g.device == g0.device and g.dtype == g0.dtype and g.shape == g0.shape):
            return False
        S = _row_strided(g)
        if S is None or (S * es) % 16 or g.data_ptr() % 16:
            return False
    return True


def nhwc_add(gs) -> torch.Tensor:
    """Sum of 2..4 same-shape maps (dense channels_last or channel slices of one) in ONE vectorised kernel: f32 sum in list
    order, one rounding (two operands: bit-identical to ``a + b``).  Anything else -> torch adds."""
    gs = list(gs)
    if not _add_ok(gs):
        out = gs[0]
        for g in gs[1:]:
            out = out + g
        return out
    g0 = gs[0]
    B, Cc, H, W = g0.shape
    out = _empty_nhwc(B, Cc, H, W, g0.dtype, g0.device)
    n = len(gs)
    srcs = (C.c_void_p * n)(*[g.data_ptr() for g in gs])
    ss = (C.c_int64 * n)(*[int(_row_strided(g)) for g in gs])
    with torch.cuda.device(g0.device):
        call("b200_nhwc_add", C.addressof(srcs), C.addressof(ss), n, ptr(out), B * H * W, Cc, dtype_code(g0.dtype),
             stream_ptr(g0.device), tag=f"b200_nhwc_add[{B * H * W}x{Cc}x{n}]")
    return out


class NhwcForkFn(torch.autograd.Function):
    """x -> n aliases of x, one per consumer.  Backward: ONE fan-in kernel over the consumers' gradients (a concat-slice
    gradient is read in place as a row-strided view) instead of autograd's pairwise accumulation, which runs ATen's generic
    strided add as soon as one operand is such a slice."""

    @staticmethod
    def forward(ctx, x, n):
        return tuple(x.view_as(x) for _ in range(n))

    @staticmethod
    def backward(ctx, *gs):
        gs = [g for g in gs if g is not None]
        if not gs:
            return None, None
        return (gs[0] if len(gs) == 1 else nhwc_add(gs)), None


def nhwc_fork(x: torch.Tensor, n: int = 2):
    """n aliases of ``x`` for n consumers (see NhwcForkFn); plain repetition when no gradient will flow."""
    if n <= 1 or not (x.is_cuda and x.requires_grad and torch.is_grad_enabled()):
        return (x,) * max(n, 1)
    return NhwcForkFn.apply(x, n)


# --------------------------------------------------------------------------------------------------
# classification term of the detection loss   (utils/loss.py:235 + the dense one-hot target of tal.py:98-107)
# --------------------------------------------------------------------------------------------------
def _level_args(maps):
    n = len(maps)
    ptrs = (C.c_void_p * n)(*[m.data_ptr() for m in maps])
    anchors = (C.c_int32 * n)(*[int(m.shape[2] * m.shape[3]) for m in maps])
    strides = (C.c_int64 * n)(*[int(m.shape[1]) for m in maps])
    return n, ptrs, anchors, strides


class ClsLossFn(torch.autograd.Function):
    """sum_{b,a,c} BCEWithLogits(x, t) with t[b,a,c] = value[b,a] * (c == label[b,a]) over the Detect class maps
    (one [B,nc,H,W] channels_last map per level), read in place: no cat / permute / float copies, no dense target."""

    @staticmethod
    def forward(ctx, label, value, *maps):
        maps = tuple(_nhwc(m) for m in maps)
        m0 = maps[0]
        B, nc = m0.shape[0], m0.shape[1]
        dev, code = m0.device, dtype_code(m0.dtype)
        label = label.to(torch.int32).contiguous()
        value = value.to(torch.float32).contiguous()
        n, ptrs, anchors, strides = _level_args(maps)
        nbytes = lib().b200_bce_logits_workspace_bytes()
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            call("b200_bce_logits_fwd", C.addressof(ptrs), C.addressof(anchors), C.addressof(strides), n, ptr(label), ptr(value), ptr(out),
                 ptr(ws), nbytes, B, nc, code, stream_ptr(dev), tag=f"b200_bce_logits_fwd[{B * sum(anchors)}x{nc}]")
        ctx.save_for_backward(label, value, *maps)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        label, value, *maps = ctx.saved_tensors
        m0 = maps[0]
        B, nc = m0.shape[0], m0.shape[1]
        dev, code = m0.device, dtype_code(m0.dtype)
        grads = [torch.empty_like(m) for m in maps]   # channels_last, like the maps
        n, ptrs, anchors, strides = _level_args(maps)
        gptrs = (C.c_void_p * n)(*[t.data_ptr() for t in grads])
        scale = g.detach().to(torch.float32).reshape(1).contiguous()
        with torch.cuda.device(dev):
            call("b200_bce_logits_bwd", C.addressof(ptrs), C.addressof(gptrs), C.addressof(anchors), C.addressof(strides), n, ptr(label),
                 ptr(value), ptr(scale), B, nc, code, stream_ptr(dev), tag=f"b200_bce_logits_bwd[{B * sum(anchors)}x{nc}]")
        return (None, None, *grads)


def cls_bce_sum(maps, label, value):
    """BCEWithLogits(reduction='sum') of the class maps against the (label, value) targets of the task-aligned assigner."""
    return ClsLossFn.apply(label, value, *maps)


# --------------------------------------------------------------------------------------------------
# task-aligned assigner + box / DFL terms of the detection loss   (utils/loss.py:199-255, utils/tal.py:41-327)
# --------------------------------------------------------------------------------------------------
def _geom_args(maps, strides):
    n = len(maps)
    Hs = (C.c_int32 * n)(*[int(m.shape[2]) for m in maps])
    Ws = (C.c_int32 * n)(*[int(m.shape[3]) for m in maps])
    st = (C.c_float * n)(*[float(s) for s in strides])
    return n, Hs, Ws, st


def _box_maps_ok(maps, reg_max=16):
    m0 = maps[0]
    return all(m.is_cuda and m.dim() == 4 and m.shape[1] == 4 * reg_max and m.dtype == m0.dtype and m.device == m0.device
               for m in maps) and m0.dtype in (torch.float32, torch.bfloat16, torch.float16)


def det_decode(box_maps, cls_maps, strides, gt):
    """pred_boxes [B, A, 4] (grid units) and scores [B, nmax, A] = sigmoid of every GT's own class logit (no autograd)."""
    box_maps = [_nhwc(m.detach()) for m in box_maps]
    cls_maps = [_nhwc(m.detach()) for m in cls_maps]
    m0 = box_maps[0]
    B, nc, nmax, dev = m0.shape[0], cls_maps[0].shape[1], gt.shape[1], m0.device
    A = sum(int(m.shape[2] * m.shape[3]) for m in box_maps)
    gt = gt.detach().to(torch.float32).contiguous()
    pred = torch.empty((B, A, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((B, nmax, A), dtype=torch.float32, device=dev)
    n, Hs, Ws, st = _geom_args(box_maps, strides)
    bp = (C.c_void_p * n)(*[m.data_ptr() for m in box_maps])
    cp = (C.c_void_p * n)(*[m.data_ptr() for m in cls_maps])
    with torch.cuda.device(dev):
        call("b200_det_decode", C.addressof(bp), C.addressof(cp), C.addressof(Hs), C.addressof(Ws), C.addressof(st), n, ptr(gt),
             ptr(pred), ptr(scores), B, nc, nmax, dtype_code(m0.dtype), stream_ptr(dev), tag=f"b200_det_decode[{B * A}x{4 * 16}]")
    return pred, scores


def tal_assign(pred, scores, gt, shapes, strides, topk=10, alpha=0.5, beta=6.0, eps=1e-9):
    """TaskAlignedAssigner on the decoded boxes: (target_label [B,A] int32, target_value [B,A], target_box [B,A,4] grid units)."""
    B, A, _ = pred.shape
    nmax, dev = gt.shape[1], pred.device
    gt = gt.detach().to(torch.float32).contiguous()
    n = len(shapes)
    Hs = (C.c_int32 * n)(*[int(s[0]) for s in shapes])
    Ws = (C.c_int32 * n)(*[int(s[1]) for s in shapes])
    st = (C.c_float * n)(*[float(s) for s in strides])
    tlabel = torch.empty((B, A), dtype=torch.int32, device=dev)
    tvalue = torch.empty((B, A), dtype=torch.float32, device=dev)
    tbox = torch.empty((B, A, 4), dtype=torch.float32, device=dev)
    nbytes = lib().b200_tal_workspace_bytes(B, nmax, A, int(topk))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        call("b200_tal_assign", ptr(pred), ptr(scores), ptr(gt), C.addressof(Hs), C.addressof(Ws), C.addressof(st), n, ptr(tlabel),
             ptr(tvalue), ptr(tbox), ptr(ws), nbytes, B, nmax, int(topk), float(alpha), float(beta), float(eps), stream_ptr(dev),
             tag=f"b200_tal_assign[{B}x{nmax}x{A}]")
    return tlabel, tvalue, tbox


class BoxDflLossFn(torch.autograd.Function):
    """(sum (1 - CIoU) * weight, sum DFL * weight) over the positive anchors, straight from the Detect box maps
    (one [B, 64, H, W] channels_last map per level); gradient written in the layout of the maps."""

    @staticmethod
    def forward(ctx, tbox, weight, *maps):
        maps = tuple(_nhwc(m) for m in maps)
        m0 = maps[0]
        B, dev, code = m0.shape[0], m0.device, dtype_code(m0.dtype)
        tbox = tbox.detach().to(torch.float32).contiguous()
        weight = weight.detach().to(torch.float32).contiguous()
        n, Hs, Ws, _ = _geom_args(maps, [1.0] * len(maps))
        bp = (C.c_void_p * n)(*[m.data_ptr() for m in maps])
        nbytes = lib().b200_box_dfl_workspace_bytes()
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        rows = B * sum(int(m.shape[2] * m.shape[3]) for m in maps)
        with torch.cuda.device(dev):
            call("b200_box_dfl_fwd", C.addressof(bp), C.addressof(Hs), C.addressof(Ws), n, ptr(tbox), ptr(weight), ptr(out), ptr(ws),
                 nbytes, B, code, stream_ptr(dev), tag=f"b200_box_dfl_fwd[{rows}x64]")
        ctx.save_for_backward(tbox, weight, *maps)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        tbox, weight, *maps = ctx.saved_tensors
        m0 = maps[0]
        B, dev, code = m0.shape[0], m0.device, dtype_code(m0.dtype)
        grads = [torch.empty_like(m) for m in maps]
        n, Hs, Ws, _ = _geom_args(maps, [1.0] * len(maps))
        bp = (C.c_void_p * n)(*[m.data_ptr() for m in maps])
        gp = (C.c_void_p * n)(*[t.data_ptr() for t in grads])
        gs = g.detach().to(torch.float32).reshape(2).contiguous()
        rows = B * sum(int(m.shape[2] * m.shape[3]) for m in maps)
        with torch.cuda.device(dev):
            call("b200_box_dfl_bwd", C.addressof(bp), C.addressof(gp), C.addressof(Hs), C.addressof(Ws), n, ptr(tbox), ptr(weight),
                 ptr(gs), B, code, stream_ptr(dev), tag=f"b200_box_dfl_bwd[{rows}x64]")
        return (None, None, *grads)


def box_dfl_sums(maps, tbox, weight):
    return BoxDflLossFn.apply(tbox, weight, *maps)


class DetLossKernels:
    """What harness/loss.py:DetectionLoss calls when the fused path is on (BLOCKS["det_loss"])."""
    supported = staticmethod(_box_maps_ok)
    decode = staticmethod(det_decode)
    assign = staticmethod(tal_assign)
    box_dfl = staticmethod(box_dfl_sums)


# --------------------------------------------------------------------------------------------------
# SPPF pooling cascade + concat   (block.py:224-226)
# --------------------------------------------------------------------------------------------------
def sppf_pool_forward_raw(y0: torch.Tensor, k: int, want_idx: bool = False):
    y0 = _nhwc(y0)
    B, Cc, H, W = y0.shape
    cat = _empty_nhwc(B, 4 * Cc, H, W, y0.dtype, y0.device)
    idx = torch.empty((3, B, H, W, Cc), dtype=torch.int32, device=y0.device) if want_idx else None
    with torch.cuda.device(y0.device):
        call("b200_sppf_pool_fwd", ptr(y0), ptr(cat), ptr(idx), B, Cc, H, W, int(k), dtype_code(y0.dtype),
                                       stream_ptr(y0.device))
    return cat, idx


class SPPFPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y0, k):
        y0 = _nhwc(y0)
        cat, _ = sppf_pool_forward_raw(y0, k)
        ctx.save_for_backward(y0)
        ctx.k = int(k)
        return cat

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gcat):
        (y0,) = ctx.saved_tensors
        B, Cc, H, W = y0.shape
        gcat = _nhwc(gcat.to(y0.dtype))
        gy0 = _empty_nhwc(B, Cc, H, W, y0.dtype, y0.device)
        with torch.cuda.device(y0.device):
            call("b200_sppf_pool_bwd", ptr(gcat), ptr(y0), ptr(gy0), B, Cc, H, W, ctx.k, dtype_code(y0.dtype),
                                           stream_ptr(y0.device))
        return gy0, None


class Conv1x1Fn(torch.autograd.Function):
    """1x1 stride-1 convolution (SPPF's cv1 / cv2, block.py:218-219: no bias; the Detect head's last convolutions, head.py:45-62:
    with bias) as a plain GEMM over the NHWC rows on the hand-written tcgen05 kernels: y[rows, c2] = x[rows, c1] @ W^T + b
    (b200_gemm_nt, bias in the epilogue); backward: dX = dY @ W (b200_gemm_nt), dW = dY^T X and db = column sums of dY in the same
    pass (b200_gemm_splitk: split-K over the rows, both operands MN-major, f32)."""

    @staticmethod
    def forward(ctx, x, w, bias=None):
        from . import gemm_tc as tc

        x = _nhwc(x)
        B, c1, H, W = x.shape
        c2 = w.shape[0]
        a = x.permute(0, 2, 3, 1).reshape(B * H * W, c1)       # NHWC-dense memory as [rows, c1]: a view
        wt = w.detach().reshape(c2, c1)
        with torch.cuda.device(x.device):
            y = tc.gemm_nt(a, wt, bias, tc.EPI_BIAS)
        ctx.save_for_backward(a, wt)
        ctx.meta = (B, c1, c2, H, W, w.shape, w.stride(), w.dtype, None if bias is None else bias.dtype)
        return y.view(B, H, W, c2).permute(0, 3, 1, 2)         # logical NCHW over NHWC memory = channels_last

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        from . import gemm_tc as tc

        a, wt = ctx.saved_tensors
        B, c1, c2, H, W, wshape, wstride, wdtype, bdtype = ctx.meta
        g = _nhwc(gy.to(a.dtype)).permute(0, 2, 3, 1).reshape(B * H * W, c2)
        gb = None
        with torch.cuda.device(a.device):
            gx = tc.gemm_nt(g, wt.t().contiguous(), None, tc.EPI_BIAS) if ctx.needs_input_grad[0] else None
            if bdtype is not None:
                gw, gb = tc.gemm_splitk(g, a, True, True, want_colsum=True)   # [c2, c1] f32 = sum_rows g(r, :)^T a(r, :); [c2]
                gb = gb.to(bdtype)
            else:
                gw = tc.gemm_splitk(g, a, True, True)
        if gx is not None:
            gx = gx.view(B, H, W, c1).permute(0, 3, 1, 2)
        return gx, gw.to(wdtype).as_strided(wshape, wstride), gb


def conv1x1_supported(x: torch.Tensor, conv, allow_bias: bool = False) -> bool:
    """True for a 1x1 / stride 1 / ungrouped nn.Conv2d on a 16-bit CUDA map whose widths the tcgen05 GEMM tiles."""
    if not (x.is_cuda and x.dim() == 4 and x.dtype in (torch.bfloat16, torch.float16) and type(conv) is torch.nn.Conv2d):
        return False
    if conv.kernel_size != (1, 1) or conv.stride != (1, 1) or conv.padding != (0, 0) or conv.groups != 1:
        return False
    if conv.bias is not None and not allow_bias:
        return False
    c2, c1 = conv.weight.shape[:2]
    rows = x.shape[0] * x.shape[2] * x.shape[3]
    ok = (c1 % 64 == 0 and c2 % 64 == 0) or (allow_bias and c1 % 8 == 0 and c2 % 8 == 0 and c1 >= 16 and c2 >= 16)
    return ok and rows % 8 == 0 and x.shape[1] == c1


def conv1x1(x: torch.Tensor, conv) -> torch.Tensor:
    return Conv1x1Fn.apply(x, conv.weight, conv.bias)


def head_conv(conv, x: torch.Tensor) -> torch.Tensor:
    """The Detect head's last 1x1 convolution of a branch (head.py:45-62: ``nn.Conv2d(c, 4*reg_max | nc, 1)`` with bias) on the
    tcgen05 GEMM with the bias in its epilogue and the bias gradient out of the weight-gradient pass; the module's own forward
    for anything the kernel does not tile (f32, CPU, odd widths)."""
    if x.is_cuda and torch.is_autocast_enabled("cuda") and x.dtype == torch.float32:
        x = x.to(torch.get_autocast_dtype("cuda"))
    if conv1x1_supported(x, conv, allow_bias=True):
        return conv1x1(x, conv)
    return conv(x)


class StemConvFn(torch.autograd.Function):
    """The model's first convolution Conv2d(3, c2, 3, 2, 1, bias=False) on a 16-bit channels_last image (hand-written mma kernels,
    csrc/stem_conv.cu): y = conv(x, w); backward: the weight gradient only -- the image needs none (an input gradient, if ever
    asked for, comes from ATen)."""

    @staticmethod
    def forward(ctx, x, w):
        x = _nhwc(x)
        B, _, H, W = x.shape
        c2 = w.shape[0]
        wf = _f32(w.detach())
        y = _empty_nhwc(B, c2, H // 2, W // 2, x.dtype, x.device)
        with torch.cuda.device(x.device):
            call("b200_stem_conv_fwd", ptr(x), ptr(wf), ptr(y), B, H, W, c2, dtype_code(x.dtype), stream_ptr(x.device),
                 tag=f"b200_stem_conv_fwd[{B}x{H}x{W}x3->{c2}]")
        ctx.save_for_backward(x, w)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        B, _, H, W = x.shape
        c2 = w.shape[0]
        gy = _nhwc(gy.to(x.dtype))
        gw = torch.empty(w.shape, dtype=torch.float32, device=x.device)
        nbytes = lib().b200_stem_conv_wgrad_workspace_bytes(c2)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            call("b200_stem_conv_wgrad", ptr(gy), ptr(x), ptr(gw), ptr(ws), nbytes, B, H, W, c2, dtype_code(x.dtype),
                 stream_ptr(x.device), tag=f"b200_stem_conv_wgrad[{B}x{H}x{W}x3->{c2}]")
        gx = None
        if ctx.needs_input_grad[0]:
            gx = torch.nn.grad.conv2d_input(x.shape, w.to(x.dtype), gy, stride=2, padding=1)
        return gx, gw.to(w.dtype)


def stem_conv(conv, x: torch.Tensor) -> torch.Tensor:
    """``conv(x)`` for the first layer's nn.Conv2d: the hand-written kernels when it is Conv2d(3, c2, 3, 2, 1, bias=False) on a
    16-bit CUDA image they tile, the module's own forward otherwise."""
    if x.is_cuda and x.dim() == 4 and torch.is_autocast_enabled("cuda") and x.dtype == torch.float32:
        x = x.to(torch.get_autocast_dtype("cuda"))
    if (x.is_cuda and x.dim() == 4 and x.dtype in (torch.bfloat16, torch.float16) and type(conv) is torch.nn.Conv2d
            and conv.in_channels == 3 and x.shape[1] == 3 and conv.kernel_size == (3, 3) and conv.stride == (2, 2)
            and conv.padding == (1, 1) and conv.dilation == (1, 1) and conv.groups == 1 and conv.bias is None
            and conv.padding_mode == "zeros"
            and lib().b200_stem_conv_supported(int(x.shape[2]), int(x.shape[3]), int(conv.out_channels), dtype_code(x.dtype))):
        return StemConvFn.apply(x, conv.weight)
    return conv(x)


FWD_S2 = [True]     # the same switch for the forward of that layer
DGRAD_S2 = [True]   # process-wide switch (tests / A-B timing): False = ATen's (cuDNN) input gradient for the stride-2 layer


class Conv3x3WgradFn(torch.autograd.Function):
    """A narrow 3x3 nn.Conv2d (bias-free, padding 1, stride 1 or 2) whose WEIGHT GRADIENT runs on the hand-written mma kernel
    (csrc/conv_wgrad.cu); the forward and the input gradient stay ATen's (cuDNN) -- for 16 / 32 input channels cuDNN's wgrad
    falls back to sm80 legacy kernels (1.5 ms per step in the round-2 launch list)."""

    @staticmethod
    def forward(ctx, x, w, stride):
        x = _nhwc(x)
        wl = w.detach().to(x.dtype)
        B, cin, H, W = x.shape
        cout, code = int(wl.shape[0]), dtype_code(x.dtype)
        if stride == 2 and FWD_S2[0] and lib().b200_conv3x3_dgrad_s2_supported(H, W, cin, cout, code):
            # the 16 -> 32 stride-2 layer: cuDNN picks an sm80 legacy fprop there (csrc/conv_dgrad.cu: conv3_fwd_s2_kernel)
            y = _empty_nhwc(B, cout, H // 2, W // 2, x.dtype, x.device)
            wst = (C.c_int64 * 4)(*[int(v) for v in wl.stride()])
            with torch.cuda.device(x.device):
                call("b200_conv3x3_fwd_s2", ptr(x), ptr(wl), C.addressof(wst), ptr(y), B, H, W, cin, cout, code,
                     stream_ptr(x.device), tag=f"b200_conv3x3_fwd_s2[{B}x{H}x{W}x{cin}->{cout}]")
        else:
            y = torch.nn.functional.conv2d(x, wl, None, stride, 1)
        ctx.save_for_backward(x, wl)
        ctx.meta = (int(stride), w.dtype)
        return y

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy):
        x, wl = ctx.saved_tensors
        stride, wdtype = ctx.meta
        B, cin, H, W = x.shape
        cout = wl.shape[0]
        gy = _nhwc(gy.to(x.dtype))
        gx = None
        if ctx.needs_input_grad[0]:
            code = dtype_code(x.dtype)
            if stride == 2 and DGRAD_S2[0] and lib().b200_conv3x3_dgrad_s2_supported(H, W, cin, cout, code):
                # the 16 -> 32 stride-2 layer: cuDNN's generic strided dgrad takes 0.38 ms there (csrc/conv_dgrad.cu)
                gx = torch.empty_like(x)
                wst = (C.c_int64 * 4)(*[int(v) for v in wl.stride()])
                with torch.cuda.device(x.device):
                    call("b200_conv3x3_dgrad_s2", ptr(gy), ptr(wl), C.addressof(wst), ptr(gx), B, H, W, cin, cout, code,
                         stream_ptr(x.device), tag=f"b200_conv3x3_dgrad_s2[{B}x{H}x{W}x{cin}<-{cout}]")
            else:
                gx = torch.ops.aten.convolution_backward(gy, x, wl, None, [stride, stride], [1, 1], [1, 1], False, [0, 0], 1,
                                                         [True, False, False])[0]
        gw = torch.empty(wl.shape, dtype=torch.float32, device=x.device)
        nbytes = lib().b200_conv3x3_wgrad_workspace_bytes(cin, cout)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            call("b200_conv3x3_wgrad", ptr(gy), ptr(x), ptr(gw), ptr(ws), nbytes, B, H, W, cin, cout, stride, dtype_code(x.dtype),
                 stream_ptr(x.device), tag=f"b200_conv3x3_wgrad[{B}x{H}x{W}x{cin}->{cout},s{stride}]")
        return gx, gw.to(wdtype), None


def conv3x3(conv, x: torch.Tensor) -> torch.Tensor:
    """``conv(x)`` with the weight gradient of a narrow 3x3 convolution on the hand-written kernel when the layer qualifies
    (training, 16-bit CUDA map, cin = 16, cout in {16, 32}); the module's own forward otherwise."""
    if x.is_cuda and x.dim() == 4 and torch.is_autocast_enabled("cuda") and x.dtype == torch.float32:
        x = x.to(torch.get_autocast_dtype("cuda"))
    if (x.is_cuda and x.dim() == 4 and torch.is_grad_enabled() and conv.weight.requires_grad and x.dtype in (torch.bfloat16, torch.float16)
            and type(conv) is torch.nn.Conv2d and conv.kernel_size == (3, 3) and conv.stride in ((1, 1), (2, 2))
            and conv.padding == (1, 1) and conv.dilation == (1, 1) and conv.groups == 1 and conv.bias is None
            and conv.padding_mode == "zeros" and x.shape[1] == conv.in_channels
            and lib().b200_conv3x3_wgrad_supported(int(x.shape[2]), int(x.shape[3]), int(conv.in_channels), int(conv.out_channels),
                                                   int(conv.stride[0]), dtype_code(x.dtype))):
        return Conv3x3WgradFn.apply(x, conv.weight, int(conv.stride[0]))
    return conv(x)


def sppf_pool(y0: torch.Tensor, k: int) -> torch.Tensor:
    """[B,c,H,W] -> [B,4c,H,W] = cat[y0, m(y0), m(m(y0)), m(m(m(y0)))], m = MaxPool2d(k,1,k//2)."""
    return SPPFPoolFn.apply(y0, k)


# --------------------------------------------------------------------------------------------------
# Conv epilogue: BatchNorm2d (+ SiLU) fused   (conv.py:65-79; SPPF cv1/cv2, block.py:218-219)
# --------------------------------------------------------------------------------------------------
class BnActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, training, momentum, eps, act, tracked=None):
        x = _nhwc(x)
        B, Cc, H, W = x.shape
        rows, dev, code = B * H * W, x.device, dtype_code(x.dtype)
        z = torch.empty_like(x)
        need_grad = any(ctx.needs_input_grad)
        mean = torch.empty(Cc, dtype=torch.float32, device=dev) if need_grad else None
        rstd = torch.empty(Cc, dtype=torch.float32, device=dev) if need_grad else None
        nbytes = lib().b200_bn_silu_workspace_bytes(rows, Cc, code)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        wf, bf = _f32(weight), _f32(bias)
        with torch.cuda.device(dev):
            call("b200_bn_silu_fwd_tracked", ptr(x), ptr(wf), ptr(bf), ptr(running_mean), ptr(running_var), ptr(tracked), ptr(z),
                 ptr(mean), ptr(rstd), ptr(ws), nbytes, rows, Cc, float(eps), float(momentum), int(training), int(act), code,
                 stream_ptr(dev), tag=f"b200_bn_silu_fwd[{rows}x{Cc}]")
        ctx.save_for_backward(x, wf, bf, mean, rstd)
        ctx.cfg = (rows, Cc, int(training), int(act), weight.dtype, bias.dtype)
        return z

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gz):
        x, wf, bf, mean, rstd = ctx.saved_tensors
        rows, Cc, training, act, wdt, bdt = ctx.cfg
        dev, code = x.device, dtype_code(x.dtype)
        gz = gz.to(x.dtype)
        gzs = _row_strided(gz)   # a channel slice of a concat's gradient is read in place (row stride > C)
        if gzs is None or (gzs * gz.element_size()) % 16 or gz.data_ptr() % 16:
            gz, gzs = _nhwc(gz), Cc
        gx = torch.empty_like(x)
        gg = torch.empty(Cc, dtype=torch.float32, device=dev)
        gb = torch.empty(Cc, dtype=torch.float32, device=dev)
        nbytes = lib().b200_bn_silu_workspace_bytes(rows, Cc, code)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            call("b200_bn_silu_bwd", ptr(gz), gzs, ptr(x), ptr(wf), ptr(bf), ptr(mean), ptr(rstd), ptr(gx), ptr(gg), ptr(gb),
                                     ptr(ws), nbytes, rows, Cc, training, act, code, stream_ptr(dev),
                                     tag=f"b200_bn_silu_bwd[{rows}x{Cc}]")
        return gx, gg.to(wdt), gb.to(bdt), None, None, None, None, None, None, None


def bn_act_supported(x: torch.Tensor, bn) -> bool:
    """True when the fused epilogue kernel tiles this BatchNorm2d input (16-byte channel vectors, affine, tracked)."""
    if not (x.is_cuda and x.dim() == 4 and type(bn) is torch.nn.BatchNorm2d and bn.affine and bn.track_running_stats):
        return False
    if bn.momentum is None or x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        return False
    if bn.training and bn.running_mean.dtype != torch.float32:
        return False   # a .half()-ed module in training mode: the in-place running-stat update needs f32 buffers
    B, Cc, H, W = x.shape
    return bool(lib().b200_bn_silu_supported(B * H * W, Cc, dtype_code(x.dtype)))


def bn_act(x: torch.Tensor, bn, silu: bool) -> torch.Tensor:
    """act(bn(x)) for the conv output x [B,C,H,W] with `bn` an nn.BatchNorm2d (conv.py:65-79); batch statistics and
    the running-stat update in training mode, running statistics in eval mode."""
    rm, rv = bn.running_mean, bn.running_var
    if rm.dtype != torch.float32:   # eval mode of a .half()-ed module (validator.py:147-149): read-only f32 copies
        rm, rv = rm.float(), rv.float()
    # nn.BatchNorm2d.forward's `num_batches_tracked.add_(1)` (state_dict parity) happens inside the finalize kernel
    nbt = bn.num_batches_tracked if bn.training and bn.num_batches_tracked is not None else None
    if nbt is not None and not (nbt.is_cuda and nbt.dtype == torch.int64):
        nbt.add_(1)
        nbt = None
    return BnActFn.apply(x, bn.weight, bn.bias, rm, rv, bn.training, bn.momentum, bn.eps, silu, nbt)


# --------------------------------------------------------------------------------------------------
# CBAM   (cbam.py:29-38, :48-53, :62-71)
# --------------------------------------------------------------------------------------------------
class CBAMFn(torch.autograd.Function):
    """mode 0: x*ca*sa;  mode 1: ca map [B,C,1,1];  mode 2: sa map [B,1,H,W]."""

    @staticmethod
    def forward(ctx, x, w1, w2, wsa, mode):
        x = _nhwc(x)
        B, Cc, H, W = x.shape
        dev = x.device
        code = dtype_code(x.dtype)
        r = w1.shape[0] if w1 is not None else 1
        ksa = wsa.shape[-1] if wsa is not None else 3
        w1f = _f32(w1).view(r, Cc) if w1 is not None else None
        w2f = _f32(w2).view(Cc, r) if w2 is not None else None
        wsf = _f32(wsa).view(2, ksa, ksa) if wsa is not None else None
        need_grad = any(ctx.needs_input_grad)
        L = lib()
        ca = torch.empty((B, Cc), dtype=torch.float32, device=dev) if mode != 2 else None
        sa = torch.empty((B, H * W), dtype=torch.float32, device=dev) if (mode == 2 or (need_grad and mode == 0)) else None
        out = _empty_nhwc(B, Cc, H, W, x.dtype, dev) if mode == 0 else None
        # small by-products (pooled avg/max, argmax maps, the 2-channel map) kept for the backward
        stash = torch.empty(L.b200_cbam_stash_bytes(B, Cc, H, W), dtype=torch.uint8, device=dev) if need_grad else None
        nbytes = L.b200_cbam_fwd_workspace_bytes(B, Cc, H, W, code)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            call("b200_cbam_fwd", ptr(x), ptr(w1f), ptr(w2f), ptr(wsf), ptr(out), ptr(ca), ptr(sa), ptr(stash), ptr(ws),
                                  nbytes, B, Cc, H, W, r, ksa, code, mode, stream_ptr(dev))
        ctx.mode, ctx.dims = mode, (B, Cc, H, W, r, ksa)
        ctx.wshapes = tuple(None if w is None else (w.shape, w.dtype, w.stride()) for w in (w1, w2, wsa))
        ctx.save_for_backward(x, w1f, w2f, wsf, ca, sa, stash)
        if mode == 0:
            return out
        if mode == 1:
            return ca.view(B, Cc, 1, 1).to(x.dtype)
        return sa.view(B, 1, H, W).to(x.dtype)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, w1f, w2f, wsf, ca, sa, stash = ctx.saved_tensors
        B, Cc, H, W, r, ksa = ctx.dims
        dev, mode = x.device, ctx.mode
        code = dtype_code(x.dtype)
        if mode == 0:
            g = _nhwc(g.to(x.dtype))
        else:
            g = g.to(torch.float32).contiguous().view(B, -1)
        gx = _empty_nhwc(B, Cc, H, W, x.dtype, dev)
        gw1 = torch.empty((r, Cc), dtype=torch.float32, device=dev) if mode != 2 else None
        gw2 = torch.empty((Cc, r), dtype=torch.float32, device=dev) if mode != 2 else None
        gws = torch.empty((2, ksa, ksa), dtype=torch.float32, device=dev) if mode != 1 else None
        L = lib()
        nbytes = L.b200_cbam_bwd_workspace_bytes(B, Cc, H, W, r, code)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            call("b200_cbam_bwd", ptr(g), ptr(x), ptr(w1f), ptr(w2f), ptr(wsf), ptr(ca), ptr(sa), ptr(stash), ptr(gx),
                                  ptr(gw1), ptr(gw2), ptr(gws), ptr(ws), nbytes, B, Cc, H, W, r, ksa, code, mode,
                                  stream_ptr(dev))
        outs = []
        for gw, meta in zip((gw1, gw2, gws), ctx.wshapes):
            # same memory order as the parameter (size-1 dims may carry channels_last strides): DDP bucket views match
            outs.append(None if (gw is None or meta is None) else gw.to(meta[1]).as_strided(meta[0], meta[2]))
        return gx, outs[0], outs[1], outs[2], None


def cbam(x, w1, w2, wsa):
    return CBAMFn.apply(x, w1, w2, wsa, _lib.CBAM_FULL)


def cbam_channel_attention(x, w1, w2):
    return CBAMFn.apply(x, w1, w2, None, _lib.CBAM_CA)


def cbam_spatial_attention(x, wsa):
    return CBAMFn.apply(x, None, None, wsa, _lib.CBAM_SA)


# --------------------------------------------------------------------------------------------------
# SwinBlock   (swin_block.py:37-58)
# --------------------------------------------------------------------------------------------------
def _gemm_nt(a: torch.Tensor, w: torch.Tensor, bias: torch.Tensor | None) -> torch.Tensor:
    """a[M,K] @ w[N,K]^T (+ bias) -> [M,N] in a's dtype."""
    from . import gemm

    return gemm.linear(a, w, bias)


def _colsum(a: torch.Tensor) -> torch.Tensor:
    rows, n = a.shape
    L = lib()
    nbytes = L.b200_colsum_workspace_bytes(rows, n)
    ws = torch.empty(max(nbytes, 4), dtype=torch.uint8, device=a.device)
    out = torch.empty(n, dtype=torch.float32, device=a.device)
    call("b200_colsum", ptr(a), ptr(out), ptr(ws), nbytes, rows, n, dtype_code(a.dtype), stream_ptr(a.device))
    return out


USE_TC_ATTENTION = True  # tests flip this to compare against the SIMT attention kernels


def attn_forward(qkv, T, Lw, Cc, nh, grid=(0, 0, 0, 0), bias=None):
    """windowed MHSA on packed qkv[T,3C] -> (o[T,C], lse[T,nh]).  grid = (nWh, nWw, ws, shift): shifted-window mask
    (extension; shift 0 = the reference's unmasked attention).  bias: dense relative-position bias [nh,64,64] f32 from
    rpb_expand (SwinBlockRPB), added to the scores before the softmax; grid must then carry ws."""
    dev, code = qkv.device, dtype_code(qkv.dtype)
    o = torch.empty((T, Cc), dtype=qkv.dtype, device=dev)
    lse = torch.empty((T, nh), dtype=torch.float32, device=dev)
    tc = USE_TC_ATTENTION and lib().b200_swin_attn_tc_supported(T, Lw, Cc, nh, code)
    if bias is not None:
        call("b200_swin_attn_fwd_tc_rpb" if tc else "b200_swin_attn_fwd_rpb", ptr(qkv), ptr(bias), ptr(o), ptr(lse), T, Lw, Cc, nh, *grid,
             code, stream_ptr(dev))
    elif tc:
        call("b200_swin_attn_fwd_tc", ptr(qkv), ptr(o), ptr(lse), T, Lw, Cc, nh, *grid, code, stream_ptr(dev))
    else:
        call("b200_swin_attn_fwd", ptr(qkv), ptr(o), ptr(lse), T, Lw, Cc, nh, *grid, code, stream_ptr(dev))
    return o, lse


def attn_backward(qkv, o, lse, go, T, Lw, Cc, nh, grid=(0, 0, 0, 0), bias=None):
    """gradient of attn_forward w.r.t. the packed qkv rows; with ``bias`` -> (gqkv, gtable [(2ws-1)^2, nh] f32), the
    gradient of the relative-position bias table that ``bias`` was expanded from."""
    dev, code = qkv.device, dtype_code(qkv.dtype)
    gqkv = torch.empty_like(qkv)
    tc = USE_TC_ATTENTION and lib().b200_swin_attn_tc_supported(T, Lw, Cc, nh, code)
    if bias is not None:
        ws = grid[2]
        rows = (2 * ws - 1) ** 2
        gtable = torch.empty((rows, nh), dtype=torch.float32, device=dev)
        nbytes = lib().b200_swin_rpb_workspace_bytes(T, Lw, nh, int(tc))
        wsb = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        if tc:
            call("b200_swin_attn_bwd_tc_rpb", ptr(qkv), ptr(lse), ptr(go), ptr(bias), ptr(gqkv), ptr(gtable), rows, ptr(wsb), nbytes, T, Lw,
                 Cc, nh, *grid, code, stream_ptr(dev))
        else:
            call("b200_swin_attn_bwd_rpb", ptr(qkv), ptr(o), ptr(lse), ptr(go), ptr(bias), ptr(gqkv), ptr(gtable), rows, ptr(wsb), nbytes,
                 T, Lw, Cc, nh, *grid, code, stream_ptr(dev))
        return gqkv, gtable
    if tc:
        call("b200_swin_attn_bwd_tc", ptr(qkv), ptr(lse), ptr(go), ptr(gqkv), T, Lw, Cc, nh, *grid, code, stream_ptr(dev))
    else:
        call("b200_swin_attn_bwd", ptr(qkv), ptr(o), ptr(lse), ptr(go), ptr(gqkv), T, Lw, Cc, nh, *grid, code, stream_ptr(dev))
    return gqkv


def rpb_expand(table: torch.Tensor, ws: int) -> torch.Tensor:
    """relative_position_bias_table [(2ws-1)^2, nh] (any float dtype) -> dense f32 bias [nh, 64, 64] (rows / columns >= ws*ws
    zero), the form the attention kernels read."""
    t = _f32(table)
    rows, nh = t.shape
    bias = torch.empty((nh, 64, 64), dtype=torch.float32, device=t.device)
    call("b200_swin_rpb_expand", ptr(t), rows, ptr(bias), ws, nh, stream_ptr(t.device))
    return bias


USE_FUSED_ATTN = True  # tests flip this to compare the fused tcgen05 attention half with the unfused stage-by-stage path


def fused_attn_supported(B, Cc, H, W, heads, ws, shift, dtype) -> bool:
    return (USE_FUSED_ATTN and dtype in (torch.bfloat16, torch.float16)
            and bool(lib().b200_swin_attn_block_supported(B, Cc, H, W, heads, ws, shift, dtype_code(dtype))))


def swin_attn_block_forward_raw(x, g1, b1, win, bin_, wo, bo, heads, ws, train=False, eps=1e-5):
    """y1 [B,C,H,W] (channels_last) = n1 + out_proj(MHSA(n1)), n1 = LN1(window tokens of zero-padded x), in one kernel.
    train: also returns (n1 [T,C], qkv [T,3C], o [T,C], lse [T,heads], mean [T], rstd [T]) in window-token order."""
    x = _nhwc(x)
    B, Cc, H, W = x.shape
    dev, dt = x.device, x.dtype
    y1 = _empty_nhwc(B, Cc, H, W, dt, dev)
    extra = None
    if train:
        T = int(lib().b200_swin_num_tokens(B, H, W, ws))
        f32 = dict(dtype=torch.float32, device=dev)
        extra = (torch.empty((T, Cc), dtype=dt, device=dev), torch.empty((T, 3 * Cc), dtype=dt, device=dev),
                 torch.empty((T, Cc), dtype=dt, device=dev), torch.empty((T, heads), **f32), torch.empty(T, **f32), torch.empty(T, **f32))
    e = extra or (None,) * 6
    wi, wod = win.detach().to(dt).contiguous(), wo.detach().to(dt).contiguous()
    with torch.cuda.device(dev):
        call("b200_swin_attn_block_fwd", ptr(x), ptr(_f32(g1)), ptr(_f32(b1)), ptr(wi), ptr(_f32(bin_)), ptr(wod), ptr(_f32(bo)), ptr(y1),
             ptr(e[0]), ptr(e[1]), ptr(e[2]), ptr(e[3]), ptr(e[4]), ptr(e[5]), B, Cc, H, W, heads, ws, float(eps), dtype_code(dt),
             stream_ptr(dev), tag=f"b200_swin_attn_block_fwd[{B}x{Cc}x{H}x{W},ws{ws}]")
    return (y1, *extra) if train else y1


USE_FUSED_MLP = True  # tests flip this to compare the fused tcgen05 MLP half with the unfused stage-by-stage path


def fused_mlp_supported(rows: int, Cc: int, dtype) -> bool:
    return USE_FUSED_MLP and dtype in (torch.bfloat16, torch.float16) and bool(lib().b200_swin_mlp_supported(rows, Cc, dtype_code(dtype)))


def swin_mlp_prep(g2, b2n, w1, bb1, w2, dtype):
    """(w1f, b1f, w2h): LayerNorm2's affine part folded into mlp.0, weights in the activation dtype (one small launch)."""
    Cc = w1.shape[1]
    dev = w1.device
    w1f = torch.empty((4 * Cc, Cc), dtype=dtype, device=dev)
    w2h = torch.empty((Cc, 4 * Cc), dtype=dtype, device=dev)
    b1f = torch.empty(4 * Cc, dtype=torch.float32, device=dev)
    call("b200_swin_mlp_prep", ptr(_f32(w1)), ptr(_f32(bb1)), ptr(_f32(g2)), ptr(_f32(b2n)), ptr(_f32(w2)), ptr(w1f), ptr(b1f), ptr(w2h),
         Cc, dtype_code(dtype), stream_ptr(dev))
    return w1f, b1f, w2h


def swin_mlp_forward_raw(y1p, w1f, b1f, w2h, bb2, eps=1e-5, save_h=False):
    """out[rows, C] = y1 + mlp.2(gelu(mlp.0(LN2(y1)))) on dense rows (pixel order), hidden activation kept on chip.
    save_h: also return h2 = 2*gelu(a) [rows, 4C] (the 16-bit tiles the second GEMM consumed) for the backward."""
    rows, Cc = y1p.shape
    out = torch.empty_like(y1p)
    h2 = torch.empty((rows, 4 * Cc), dtype=y1p.dtype, device=y1p.device) if save_h else None
    call("b200_swin_mlp_fwd", ptr(y1p), ptr(w1f), ptr(b1f), ptr(w2h), ptr(_f32(bb2)), ptr(out), ptr(h2), rows, Cc, float(eps),
         dtype_code(y1p.dtype), stream_ptr(y1p.device), tag=f"b200_swin_mlp_fwd[{rows}x{Cc}]")
    return (out, h2) if save_h else out


def swin_mlp_backward_raw(gout, y1p, w1f, b1f, w2h, eps=1e-5):
    """-> (g_y1' [rows,C], xhat [rows,C], g_a [rows,4C]): the LayerNorm2-backward term of the data gradient of the fused
    MLP half (the full gradient is g_y1' + gout: the residual is added by the consumer, b200_swin_partition_add) and the
    operands of the mlp.0 weight-gradient contraction (mlp.2's uses the forward's saved h2)."""
    rows, Cc = y1p.shape
    dev, dt = y1p.device, y1p.dtype
    gy1, xhat = torch.empty_like(y1p), torch.empty_like(y1p)
    ga = torch.empty((rows, 4 * Cc), dtype=dt, device=dev)
    call("b200_swin_mlp_bwd", ptr(gout), ptr(y1p), ptr(w1f), ptr(b1f), ptr(w2h), ptr(gy1), ptr(xhat), ptr(ga), rows, Cc, float(eps),
         dtype_code(dt), stream_ptr(dev), tag=f"b200_swin_mlp_bwd[{rows}x{Cc}]")
    return gy1, xhat, ga


class SwinBlockFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, *args):
        with torch.autocast("cuda", enabled=False):  # dtype is decided by the caller (swin_block), not by autocast
            return SwinBlockFn._forward(ctx, *args)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        with torch.autocast("cuda", enabled=False):
            return SwinBlockFn._backward(ctx, gout)

    @staticmethod
    def _forward(ctx, x, g1, b1, win, bin_, wo, bo, g2, b2, w1, bb1, w2, bb2, num_heads, ws, shift, rpb=None):
        from . import gemm

        x = _nhwc(x)
        B, Cc, H, W = x.shape
        dev, dt = x.device, x.dtype
        code = dtype_code(dt)
        L = lib()
        T = int(L.b200_swin_num_tokens(B, H, W, ws))
        Lw = ws * ws
        st = stream_ptr(dev)
        f32 = dict(dtype=torch.float32, device=dev)
        g1f, b1f, g2f, b2f = _f32(g1), _f32(b1), _f32(g2), _f32(b2)
        need_grad = any(ctx.needs_input_grad)
        with torch.cuda.device(dev):
            grid = (-(-H // ws), -(-W // ws), ws, shift)
            # the fused attention half takes no relative-position bias: with a table the attention half runs stage by stage
            fused_attn = (rpb is None and fused_attn_supported(B, Cc, H, W, num_heads, ws, shift, dt)
                          and fused_mlp_supported(B * H * W, Cc, dt))
            bias = rpb_expand(rpb, ws) if rpb is not None else None
            if fused_attn:
                # attention half in one tcgen05 kernel: x -> y1 in pixel order (+ the backward's by-products when training)
                if need_grad:
                    y1p, n1, qkv, o, lse, mean1, rstd1 = swin_attn_block_forward_raw(x, g1, b1, win, bin_, wo, bo, num_heads, ws, train=True)
                else:
                    y1p = swin_attn_block_forward_raw(x, g1, b1, win, bin_, wo, bo, num_heads, ws, train=False)
                    n1 = qkv = o = lse = mean1 = rstd1 = None
                y1 = None
            else:
                n1 = torch.empty((T, Cc), dtype=dt, device=dev)
                mean1, rstd1 = torch.empty(T, **f32), torch.empty(T, **f32)
                call("b200_swin_ln1_partition", ptr(x), ptr(g1f), ptr(b1f), ptr(n1), ptr(mean1), ptr(rstd1), B, Cc, H, W, ws,
                                                shift, code, st)
                qkv = gemm.linear(n1, win, bin_)
                o, lse = attn_forward(qkv, T, Lw, Cc, num_heads, grid, bias)
                y1 = gemm.linear_res(o, wo, bo, n1)  # post-norm residual fused into the out_proj epilogue
            fused = fused_mlp_supported(B * H * W, Cc, dt)
            if fused:
                # MLP half in one tcgen05 kernel on the real tokens in pixel order (window_reverse + crop = the row order)
                if not fused_attn:
                    y1p = _empty_nhwc(B, Cc, H, W, dt, dev)
                    call("b200_swin_res_reverse", ptr(y1), None, ptr(y1p), B, Cc, H, W, ws, shift, code, st)
                w1f, b1f, w2h = swin_mlp_prep(g2, b2, w1, bb1, w2, dt)
                out = _empty_nhwc(B, Cc, H, W, dt, dev)
                h2 = torch.empty((B * H * W, 4 * Cc), dtype=dt, device=dev) if need_grad else None   # 2*gelu(a), for d mlp.2.weight
                call("b200_swin_mlp_fwd", ptr(y1p), ptr(w1f), ptr(b1f), ptr(w2h), ptr(_f32(bb2)), ptr(out), ptr(h2), B * H * W, Cc, 1e-5,
                     code, st, tag=f"b200_swin_mlp_fwd[{B * H * W}x{Cc}]")
                ctx.save_for_backward(x, g1f, g2f, b2f, win, wo, w1, n1, mean1, rstd1, qkv, o, lse, y1p, w1f, b1f, w2h, h2)
            else:
                u = torch.empty_like(n1)
                mean2, rstd2 = torch.empty(T, **f32), torch.empty(T, **f32)
                call("b200_swin_res_ln2", ptr(y1), None, ptr(g2f), ptr(b2f), None, ptr(u), ptr(mean2), ptr(rstd2), T, Cc,
                                          code, st)
                h, hpre = gemm.linear_gelu(u, w1, bb1)
                m = gemm.linear(h, w2, bb2)
                out = _empty_nhwc(B, Cc, H, W, dt, dev)
                call("b200_swin_res_reverse", ptr(y1), ptr(m), ptr(out), B, Cc, H, W, ws, shift, code, st)
                ctx.save_for_backward(x, g1f, g2f, win, wo, w1, w2, n1, mean1, rstd1, qkv, o, lse, y1, u, mean2, rstd2, hpre, h)
        ctx.fused_mlp = fused
        ctx.bias = bias
        ctx.cfg = (B, Cc, H, W, ws, num_heads, T, shift)
        ctx.pdtypes = tuple(p.dtype for p in (g1, b1, win, bin_, wo, bo, g2, b2, w1, bb1, w2, bb2) + ((rpb,) if rpb is not None else ()))
        return out

    @staticmethod
    def _backward(ctx, gout):
        from . import gemm

        B, Cc, H, W, ws, nh, T, shift = ctx.cfg
        grid = (-(-H // ws), -(-W // ws), ws, shift)
        dev, dt = gout.device, ctx.saved_tensors[0].dtype
        code = dtype_code(dt)
        L = lib()
        st = stream_ptr(dev)
        Lw = ws * ws
        with torch.cuda.device(dev):
            gout = _nhwc(gout.to(dt))
            nbytes = L.b200_swin_ln_bwd_workspace_bytes(T, Cc)
            wsb = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            if ctx.fused_mlp:
                (x, g1f, g2f, b2f, win, wo, w1, n1, mean1, rstd1, qkv, o, lse, y1p, w1f, b1f, w2h, h2) = ctx.saved_tensors
                rows = B * H * W
                g2d = gout.permute(0, 2, 3, 1).reshape(rows, Cc)          # NHWC-dense memory viewed as [rows, C]: no copy
                gy1p, xhat, ga = swin_mlp_backward_raw(g2d, y1p.permute(0, 2, 3, 1).reshape(rows, Cc), w1f, b1f, w2h)
                gw2, gb2 = gemm.matmul_tn(g2d, h2)                         # 2 * [C, 4C] = g_out^T (2 gelu(a)),  [C] = sum g_out
                gw2 = gw2.mul_(0.5)
                G, gb1 = gemm.matmul_tn(ga, xhat)                          # [4C, C] = g_a^T xhat,       [4C] = sum g_a
                del ga, xhat
                # LayerNorm2's affine part was folded into mlp.0 (u = xhat * gamma + beta): unfold the three gradients
                w1d = w1.detach().float()
                gw1 = torch.addcmul(gb1[:, None] * b2f[None, :], G, g2f[None, :])
                gg2 = (w1d * G).sum(0)
                gbt2 = w1d.t() @ gb1
                gy1 = torch.empty((T, Cc), dtype=dt, device=dev)
                call("b200_swin_partition_add", ptr(gy1p), ptr(gout), ptr(gy1), B, Cc, H, W, ws, shift, code, st)   # + residual
                del gy1p
            else:
                (x, g1f, g2f, win, wo, w1, w2, n1, mean1, rstd1, qkv, o, lse, y1, u, mean2, rstd2, hpre, h) = ctx.saved_tensors
                gy2 = torch.empty((T, Cc), dtype=dt, device=dev)
                call("b200_swin_partition", ptr(gout), ptr(gy2), B, Cc, H, W, ws, shift, code, st)
                # MLP
                gw2, gb2 = gemm.matmul_tn(gy2, h)     # [C, 4C] = gy2^T h,  [C] = sum_t gy2
                ga = gemm.matmul_nn_gelu_bwd(gy2, w2, hpre)  # [T, 4C] = (gy2 W2) * gelu'(hpre)
                gw1, gb1 = gemm.matmul_tn(ga, u)      # [4C, C], [4C]
                gu = gemm.matmul_nn(ga, w1)           # [T, C]
                del ga
                # LN2 + residual
                gy1 = torch.empty_like(gy2)
                gg2 = torch.empty(Cc, dtype=torch.float32, device=dev)
                gbt2 = torch.empty(Cc, dtype=torch.float32, device=dev)
                call("b200_swin_ln_bwd", ptr(gu), ptr(y1), ptr(gy2), ptr(g2f), ptr(mean2), ptr(rstd2), ptr(gy1), ptr(gg2),
                                         ptr(gbt2), ptr(wsb), nbytes, B, Cc, H, W, ws, shift, code, 0, st)
                del gu, gy2
            # attention
            gwo, gbo = gemm.matmul_tn(gy1, o)     # [C, C], [C]
            go = gemm.matmul_nn(gy1, wo)          # [T, C]
            gtable = None
            if ctx.bias is None:
                gqkv = attn_backward(qkv, o, lse, go.contiguous(), T, Lw, Cc, nh, grid)
            else:
                gqkv, gtable = attn_backward(qkv, o, lse, go.contiguous(), T, Lw, Cc, nh, grid, ctx.bias)
            del go
            gwin, gbin = gemm.matmul_tn(gqkv, n1)  # [3C, C], [3C]
            gn1 = gemm.matmul_nn(gqkv, win, add=gy1)  # [T, C] = gy1 + gqkv Win
            del gqkv, gy1
            # LN1 + un-partition
            gx = _empty_nhwc(B, Cc, H, W, dt, dev)
            gg1 = torch.empty(Cc, dtype=torch.float32, device=dev)
            gbt1 = torch.empty(Cc, dtype=torch.float32, device=dev)
            call("b200_swin_ln_bwd", ptr(gn1), ptr(x), None, ptr(g1f), ptr(mean1), ptr(rstd1), ptr(gx), ptr(gg1),
                                     ptr(gbt1), ptr(wsb), nbytes, B, Cc, H, W, ws, shift, code, 1, st)
        grads = [gg1, gbt1, gwin, gbin, gwo, gbo, gg2, gbt2, gw1, gb1, gw2, gb2] + ([gtable] if gtable is not None else [])
        grads = [g.to(d) for g, d in zip(grads, ctx.pdtypes)]
        return (gx, *grads[:12], None, None, None, grads[12] if gtable is not None else None)


def swin_block(x, p: dict, num_heads: int, ws: int, shift: int = 0, rpb: torch.Tensor | None = None):
    """p: parameters keyed like the reference state_dict (norm1.weight, attn.in_proj_weight, ...).
    shift > 0: shifted-window extension (cyclic shift folded into the token addressing, seam mask applied in registers
    before the softmax); 0 = the reference block (swin_block.py has no shift, SURVEY D1).
    rpb: relative_position_bias_table [(2ws-1)^2, num_heads] of SwinBlockRPB (extension, Swin's learned bias; ws <= 8), or
    None (the reference block).  With a table the attention half runs stage by stage (the fused attention half takes no bias).

    Compute dtype = the autocast dtype when autocast is on (the reference runs its GEMMs there; trainer.py:383),
    else x.dtype."""
    if torch.is_autocast_enabled("cuda") and x.dtype == torch.float32:
        x = x.to(torch.get_autocast_dtype("cuda"))
    return SwinBlockFn.apply(
        x, p["norm1.weight"], p["norm1.bias"], p["attn.in_proj_weight"], p["attn.in_proj_bias"],
        p["attn.out_proj.weight"], p["attn.out_proj.bias"], p["norm2.weight"], p["norm2.bias"],
        p["mlp.0.weight"], p["mlp.0.bias"], p["mlp.2.weight"], p["mlp.2.bias"], num_heads, ws, int(shift), rpb)
