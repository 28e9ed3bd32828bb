"""B200-native (sm_100a) CBAM / SwinBlock / SPPF blocks for the YOLOv8-CBAM-Swin fork -- drop-in modules over a
C-ABI CUDA library.  See DESIGN.md / INTEGRATION.md at the repository root."""
from .modules import BLOCKS, CBAM, SPPF, ChannelAttention, SpatialAttention, SwinBlock, SwinBlockRPB  # noqa: F401

__all__ = ["CBAM", "ChannelAttention", "SpatialAttention", "SwinBlock", "SwinBlockRPB", "SPPF", "BLOCKS"]
