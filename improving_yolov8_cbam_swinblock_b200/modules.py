"""Drop-in nn.Modules: same class names, constructor arguments, sub-module names and state_dict keys as the
reference's ``ChannelAttention`` / ``SpatialAttention`` / ``CBAM`` (ultralytics/nn/modules/cbam.py:5-71),
``SwinBlock`` (ultralytics/nn/modules/swin_block.py:23-58) and ``SPPF`` (ultralytics/nn/modules/block.py:201-226),
with ``forward`` routed to the sm_100a kernels of ``libb200yolo.so``.

Modules hold only Parameters / ints (no library handles), so ``deepcopy``, whole-module pickling, ``.half()``,
``.to()`` and ``fuse()`` behave like the reference's (SURVEY.md section 8b).

CPU tensors: the callers run ONE CPU forward on ``zeros(1, ch, 256, 256)`` while constructing the model
(``DetectionModel.__init__`` stride pass, ultralytics/nn/tasks.py:350-364; CBAM creates its lazy MLP there,
cbam.py:31-33).  For a non-CUDA input the blocks therefore act as a *shape probe*: they create lazy parameters
and return zeros of the right shape and dtype, computing nothing.  That is not a compute fallback -- a CPU input
carrying real data raises, and on CUDA a missing ``libb200yolo.so`` raises.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import functional as Fb


def _shape_probe(x: torch.Tensor, what: str, channels: int | None = None) -> torch.Tensor:
    if x.is_cuda:
        raise AssertionError("shape probe called on a CUDA tensor")
    if x.numel() and bool(x.detach().ne(0).any()) and not _PROBE_ALLOWED[0]:
        raise RuntimeError(
            f"{what}: got a CPU tensor carrying data. This package computes on B200 GPUs only (no CPU path); "
            "CPU inputs are accepted solely as all-zero shape probes during model construction.")
    B, C, H, W = x.shape
    return x.new_zeros((B, C if channels is None else channels, H, W))


_PROBE_ALLOWED = [False]


class shape_probe_mode:
    """Context manager: allow non-zero CPU tensors to be treated as shape probes (e.g. thop FLOP counting)."""

    def __enter__(self):
        self.prev, _PROBE_ALLOWED[0] = _PROBE_ALLOWED[0], True

    def __exit__(self, *a):
        _PROBE_ALLOWED[0] = self.prev


class ChannelAttention(nn.Module):
    """cbam.py:5-38: returns the attention MAP sigmoid(MLP(avg)+MLP(max)) [B,C,1,1] (not x*map)."""

    def __init__(self, in_planes=None, ratio=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)  # kept for attribute parity; parameter-free
        self.max_pool = nn.AdaptiveMaxPool2d(1)
        self.in_planes = in_planes
        self.ratio = ratio
        if in_planes is not None:
            self.create_mlp(in_planes)
        else:
            self.shared_MLP = None

    def create_mlp(self, in_planes):
        reduced = max(1, in_planes // self.ratio)
        self.shared_MLP = nn.Sequential(
            nn.Conv2d(in_planes, reduced, 1, bias=False), nn.ReLU(), nn.Conv2d(reduced, in_planes, 1, bias=False))

    def _weights(self, x):
        if self.shared_MLP is None:  # lazy creation on first forward (CPU stride pass), cbam.py:31-33
            self.create_mlp(x.shape[1])
            self.shared_MLP.to(x.device)
        return self.shared_MLP[0].weight, self.shared_MLP[2].weight

    def forward(self, x):
        w1, w2 = self._weights(x)
        if not x.is_cuda:
            return _shape_probe(x, "ChannelAttention")[:, :, :1, :1]
        return Fb.cbam_channel_attention(x, w1, w2)


class SpatialAttention(nn.Module):
    """cbam.py:40-53: returns the attention MAP [B,1,H,W]."""

    def __init__(self, kernel_size=7):
        super().__init__()
        assert kernel_size in (3, 7), "kernel size must be 3 or 7"
        padding = 3 if kernel_size == 7 else 1
        self.conv = nn.Conv2d(2, 1, kernel_size, padding=padding, bias=False)

    def forward(self, x):
        if not x.is_cuda:
            return _shape_probe(x, "SpatialAttention", channels=1)
        return Fb.cbam_spatial_attention(x, self.conv.weight)


class CBAM(nn.Module):
    """cbam.py:55-71: x * ca(x) then * sa(x*ca) -- one fused cluster kernel each way."""

    def __init__(self, channels=None):
        super().__init__()
        self.ca = ChannelAttention(channels, ratio=8 if channels and channels < 128 else 16)
        self.sa = SpatialAttention(kernel_size=7)

    def forward(self, x):
        w1, w2 = self.ca._weights(x)
        if not x.is_cuda:
            return _shape_probe(x, "CBAM")
        return Fb.cbam(x, w1, w2, self.sa.conv.weight)


class SwinBlock(nn.Module):
    """swin_block.py:23-58.  ``attn`` is a real nn.MultiheadAttention used purely as the parameter container, so
    initialisation (xavier in_proj, zero biases), state_dict keys and optimizer grouping match the reference.

    ``shift_size`` (trailing optional yaml arg, default 0 = the reference block) is an EXTENSION: shifted windows with
    the seam mask, as in Swin; it adds no parameters, so state_dicts stay interchangeable."""

    def __init__(self, dim, num_heads=2, window_size=7, shift_size=0):
        super().__init__()
        if not 0 <= shift_size < window_size:
            raise ValueError(f"shift_size {shift_size} must lie in [0, window_size {window_size})")
        self.dim = dim
        self.num_heads = num_heads
        self.window_size = window_size
        self.shift_size = shift_size
        self.norm1 = nn.LayerNorm(dim)
        self.attn = nn.MultiheadAttention(embed_dim=dim, num_heads=num_heads, batch_first=True)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = nn.Sequential(nn.Linear(dim, dim * 4), nn.GELU(), nn.Linear(dim * 4, dim))

    def forward(self, x):
        if not x.is_cuda:
            return _shape_probe(x, "SwinBlock")
        if x.shape[1] != self.dim:
            raise RuntimeError(f"Given normalized_shape=[{self.dim}], expected input with {self.dim} channels, "
                               f"got {tuple(x.shape)}")
        # num_heads / shift come from state the reference class also has: a module pickled by the reference and unpickled
        # after plugin.install() (tasks.py:1222) never ran this __init__, so it has no `num_heads` / `shift_size` attribute
        return Fb.swin_block(x, _swin_params(self), self.attn.num_heads, self.window_size, getattr(self, "shift_size", 0))


def _swin_params(m: SwinBlock) -> dict:
    """A SwinBlock's parameters keyed like the reference state_dict (what functional.swin_block takes)."""
    return {
        "norm1.weight": m.norm1.weight, "norm1.bias": m.norm1.bias,
        "attn.in_proj_weight": m.attn.in_proj_weight, "attn.in_proj_bias": m.attn.in_proj_bias,
        "attn.out_proj.weight": m.attn.out_proj.weight, "attn.out_proj.bias": m.attn.out_proj.bias,
        "norm2.weight": m.norm2.weight, "norm2.bias": m.norm2.bias,
        "mlp.0.weight": m.mlp[0].weight, "mlp.0.bias": m.mlp[0].bias,
        "mlp.2.weight": m.mlp[2].weight, "mlp.2.bias": m.mlp[2].bias,
    }


class SwinBlockRPB(SwinBlock):
    """SwinBlock with Swin's learned relative-position bias (Liu et al. 2021, eq. 4) added to the attention scores:
    S[h,i,j] = q_i.k_j / sqrt(hd) + table[idx(i,j), h], idx = Swin's relative_position_index of the two tokens' positions in
    their window (computed, not stored).  EXTENSION, opt-in: the reference block has no bias (SURVEY D1).

    One parameter beyond SwinBlock's, ``relative_position_bias_table`` [(2ws-1)^2, num_heads] f32, trunc_normal(std=0.02)
    as in Swin; its name contains "bias", so the optimizer grouping (trainer.py:818-827) puts it in the no-decay group, as
    Swin does.  A SwinBlock state_dict loads with strict=False (only the table is missing).  Windows up to 8x8."""

    def __init__(self, dim, num_heads=2, window_size=7, shift_size=0):
        if not 1 <= window_size <= 8:
            raise ValueError(f"SwinBlockRPB supports window_size 1..8, got {window_size}")
        super().__init__(dim, num_heads, window_size, shift_size)
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * window_size - 1) ** 2, num_heads))
        nn.init.trunc_normal_(self.relative_position_bias_table, std=0.02)

    def forward(self, x):
        if not x.is_cuda:
            return _shape_probe(x, "SwinBlockRPB")
        if x.shape[1] != self.dim:
            raise RuntimeError(f"Given normalized_shape=[{self.dim}], expected input with {self.dim} channels, "
                               f"got {tuple(x.shape)}")
        return Fb.swin_block(x, _swin_params(self), self.attn.num_heads, self.window_size, getattr(self, "shift_size", 0),
                             self.relative_position_bias_table)


FUSE_CONV_EPILOGUE = [True]  # process-wide switch (tests / A-B timing); False = the caller's stock BatchNorm2d + SiLU


def conv_epilogue(conv_module, y):
    """``act(bn(y))`` of the reference ``Conv.forward`` (conv.py:65-79) on the conv output ``y``: one fused B200
    epilogue (batch statistics + affine + SiLU; csrc/conv_epilogue.cu) when the layer is BatchNorm2d + SiLU/Identity on
    a CUDA tensor the kernel tiles, else the module's own stock ops."""
    bn, act = conv_module.bn, conv_module.act
    if FUSE_CONV_EPILOGUE[0] and y.is_cuda and type(act) in (nn.SiLU, nn.Identity) and Fb.bn_act_supported(y, bn):
        return Fb.bn_act(y, bn, type(act) is nn.SiLU)
    return act(bn(y))


def make_conv(conv_cls, name="Conv", module=None):
    """Subclass of the caller's ``Conv`` (conv.py:37-91) whose un-fused forward runs the B200 BN+SiLU epilogue.
    Still a ``Conv`` instance with the same sub-modules / state_dict, so ``BaseModel.fuse`` (tasks.py:219-225) keeps
    folding its BN and swapping in ``forward_fuse``."""

    class Conv(conv_cls):
        def forward(self, x):
            return conv_epilogue(self, self.conv(x))

    Conv.__name__ = Conv.__qualname__ = name
    if module is not None:
        Conv.__module__ = module
    return Conv


GEMM_1X1 = [True]  # SPPF's cv1 / cv2 (1x1 convolutions = GEMMs over the NHWC rows) on the hand-written tcgen05 GEMM (SURVEY 8(f)-1)


def conv_block(conv_module, x):
    """``Conv.forward`` (conv.py:65-79) of a 1x1 Conv: the convolution itself as ``b200_gemm_nt`` when the layer is a plain
    1x1 GEMM the kernel tiles (16-bit activations under autocast, widths multiples of 64), followed by the fused BN + SiLU
    epilogue; anything else (f32, fused-BN ``forward_fuse`` after ``fuse()``, odd widths, CPU) takes the module's own forward."""
    if GEMM_1X1[0] and hasattr(conv_module, "bn") and x.is_cuda and torch.is_autocast_enabled("cuda") and x.dtype == torch.float32:
        x = x.to(torch.get_autocast_dtype("cuda"))
    if GEMM_1X1[0] and hasattr(conv_module, "bn") and Fb.conv1x1_supported(x, conv_module.conv):
        return conv_epilogue(conv_module, Fb.conv1x1(x, conv_module.conv))
    return conv_module(x)


def make_sppf(conv_cls, name="SPPF", module=None):
    """SPPF bound to the caller's stock ``Conv`` (cv1/cv2 stay Conv instances so ``BaseModel.fuse`` keeps folding
    their BN, tasks.py:219-225); only the pooling cascade + concat (block.py:224-226) runs in our kernel."""

    class SPPF(nn.Module):
        def __init__(self, c1, c2, k=5):
            super().__init__()
            c_ = c1 // 2
            self.cv1 = conv_cls(c1, c_, 1, 1)
            self.cv2 = conv_cls(c_ * 4, c2, 1, 1)
            self.m = nn.MaxPool2d(kernel_size=k, stride=1, padding=k // 2)  # attribute parity; parameter-free
            self.k = k

        def forward(self, x):
            if not x.is_cuda:
                y0 = self.cv1(x)
                B, c_, H, W = y0.shape
                return self.cv2(y0.new_zeros((B, 4 * c_, H, W)))
            y0 = conv_block(self.cv1, x)
            k = self.m.kernel_size   # not self.k: reference pickles loaded under the plugin never ran this __init__
            return conv_block(self.cv2, Fb.sppf_pool(y0, int(k[0] if isinstance(k, (tuple, list)) else k)))

    SPPF.__name__ = SPPF.__qualname__ = name
    if module is not None:
        SPPF.__module__ = module
    return SPPF


def _harness_sppf():
    from .harness.graph import Conv

    return make_sppf(Conv, module=__name__)


SPPF = _harness_sppf()
BLOCKS = {"CBAM": CBAM, "SwinBlock": SwinBlock, "SPPF": SPPF, "conv_epilogue": conv_epilogue,
          "concat": Fb.nhwc_concat, "chunk": Fb.nhwc_chunk, "input_prep": Fb.u8_to_nhwc, "cls_loss": Fb.cls_bce_sum,
          "upsample": Fb.nhwc_upsample_nearest, "head_conv": Fb.head_conv, "det_loss": Fb.DetLossKernels, "stem_conv": Fb.stem_conv, "conv3x3": Fb.conv3x3,
          "fork": Fb.nhwc_fork}
