"""Upsampling layer (absent in the reference; PyTorch's nn.Upsample for integer factors)."""
from .module import Module
from .. import functional as F


class Upsample(Module):
    """F.interpolate as a layer: nearest or bilinear (align_corners=False) upsampling by an integer factor 1..8 that is the
    same for height and width, given as `scale_factor` or as the output `size`."""

    def __init__(self, size=None, scale_factor=None, mode: str = "nearest", align_corners=None) -> None:
        super().__init__()
        self.size, self.scale_factor, self.mode, self.align_corners = size, scale_factor, mode, align_corners

    def forward(self, x):
        return F.interpolate(x, self.size, self.scale_factor, self.mode, self.align_corners)

    def __repr__(self) -> str:
        return "Upsample(size={}, scale_factor={}, mode={!r})".format(self.size, self.scale_factor, self.mode)
