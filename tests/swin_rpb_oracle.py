"""fp64 restatement of SwinBlockRPB shared by tests/test_swin_rpb_host.py (CPU) and tests/test_gpu_swin_rpb.py (GPU).

The block is ``oracle/blocks.swin_forward`` (the SwinBlock restatement pinned by the reference-generated fixtures) with Swin's
learned relative-position bias (Liu et al. 2021, eq. 4) added to the scaled scores before the shift mask.  It is written from the
same primitives as ``swin_forward`` (``oracle/blocks.py`` is left as it is), and its index is built the way Swin's code builds its
``relative_position_index`` buffer -- not from the closed form the kernels use -- so that the tests pin the kernels' arithmetic.
With an all-zero table it equals ``swin_forward`` exactly (checked in tests/test_swin_rpb_host.py).
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import blocks as ob


def relative_position_index(ws):
    """[L, L] int64 index into the bias table, as microsoft/Swin-Transformer's WindowAttention.__init__ builds it: meshgrid of
    the window's coordinates, flatten, pairwise difference, shift to start from 0, multiply the row offset by 2*ws-1, sum."""
    coords = torch.stack(torch.meshgrid(torch.arange(ws), torch.arange(ws), indexing="ij"))  # [2, ws, ws]
    coords_flatten = torch.flatten(coords, 1)  # [2, L]
    relative_coords = coords_flatten[:, :, None] - coords_flatten[:, None, :]  # [2, L, L]
    relative_coords = relative_coords.permute(1, 2, 0).contiguous()  # [L, L, 2]
    relative_coords[:, :, 0] += ws - 1
    relative_coords[:, :, 1] += ws - 1
    relative_coords[:, :, 0] *= 2 * ws - 1
    return relative_coords.sum(-1)


def swin_rpb_forward(x, p, num_heads, ws, shift, rpb):
    """SwinBlockRPB.forward: ``ob.swin_forward(x, p, num_heads, ws, shift)`` with ``rpb[idx(i, j), h]`` added to the scaled
    scores of every window (padded and shifted ones alike, by window position).  rpb: [(2ws-1)^2, num_heads]."""
    B, C, H, W = x.shape
    pad_h = (ws - H % ws) % ws
    pad_w = (ws - W % ws) % ws
    xp = F.pad(x, (0, pad_w, 0, pad_h))
    Hp, Wp = H + pad_h, W + pad_w
    if shift:
        xp = torch.roll(xp, shifts=(-shift, -shift), dims=(2, 3))
    t = ob.window_partition(xp.permute(0, 2, 3, 1), ws)  # [nWB, L, C]
    n1 = ob.layer_norm(t, p["norm1.weight"], p["norm1.bias"])
    nWB, L, _ = n1.shape
    hd = C // num_heads
    qkv = n1 @ p["attn.in_proj_weight"].t() + p["attn.in_proj_bias"]
    q, k, v = qkv.split(C, dim=-1)

    def heads(z):  # [nWB, L, C] -> [nWB, nh, L, hd]; head h = channels [h*hd, (h+1)*hd)
        return z.reshape(nWB, L, num_heads, hd).permute(0, 2, 1, 3)

    q, k, v = heads(q) * (1.0 / math.sqrt(hd)), heads(k), heads(v)
    s = q @ k.transpose(-1, -2)
    idx = relative_position_index(ws).to(rpb.device)
    s = s + rpb[idx.reshape(-1)].reshape(L, L, num_heads).permute(2, 0, 1)[None]
    if shift:
        m = ob.shift_attention_mask(Hp, Wp, ws, shift, s.dtype, s.device)  # [nW, L, L], windows ordered (wh, ww)
        s = (s.reshape(B, -1, num_heads, L, L) + m[None, :, None]).reshape(nWB, num_heads, L, L)
    s = s - s.max(dim=-1, keepdim=True).values
    e = torch.exp(s)
    pr = e / e.sum(dim=-1, keepdim=True)
    o = (pr @ v).permute(0, 2, 1, 3).reshape(nWB, L, C)
    a = o @ p["attn.out_proj.weight"].t() + p["attn.out_proj.bias"]
    y1 = n1 + a
    u = ob.layer_norm(y1, p["norm2.weight"], p["norm2.bias"])
    hmid = ob.gelu_erf(u @ p["mlp.0.weight"].t() + p["mlp.0.bias"])
    y2 = y1 + hmid @ p["mlp.2.weight"].t() + p["mlp.2.bias"]
    out = ob.window_reverse(y2, ws, Hp, Wp).permute(0, 3, 1, 2)
    if shift:
        out = torch.roll(out, shifts=(shift, shift), dims=(2, 3))
    return out[:, :, :H, :W]
