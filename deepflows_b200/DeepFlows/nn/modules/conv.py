"""Convolution layers (reference: DeepFlows/nn/modules/conv.py:13-124)."""
import math

from .module import Module
from ..parameter import Parameter
from .. import functional as F
from .. import init
from ... import tensor
from ... import backend_api


class _ConvNd(Module):
    def _make_params(self, weight_shape, bias_shape, bias, device, dtype):
        kwargs = {"device": backend_api.Device(device), "dtype": dtype}
        self.weight = Parameter(tensor.empty(weight_shape, **kwargs))
        self.bias = Parameter(tensor.empty(bias_shape, **kwargs)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        # Kaiming-uniform(a=sqrt(5)) weights, U(-1/sqrt(fan_in), 1/sqrt(fan_in)) bias [conv.py:96-102]
        init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            fan_in, _ = init._calculate_fan_in_and_fan_out(self.weight)
            if fan_in != 0:
                bound = 1 / math.sqrt(fan_in)
                init.uniform_(self.bias, -bound, bound)

    def __repr__(self) -> str:
        return "{}(in_channels={}, out_channels={}, kernel_size={}, padding={}, stride={}, bias={})".format(
            type(self).__name__, self.in_channels, self.out_channels, self.kernel_size, self.padding, self.stride,
            self.bias is not None)

    def move(self, device):
        self.device = device
        self.weight = self.weight.to(device)
        if self.bias is not None:
            self.bias = self.bias.to(device)


class Conv1d(_ConvNd):
    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, padding: int = 0, stride: int = 1,
                 bias: bool = True, device="cuda", dtype=None) -> None:
        super().__init__()
        self.in_channels, self.out_channels, self.kernel_size = in_channels, out_channels, kernel_size
        self.padding, self.stride = padding, stride
        self._make_params((out_channels, in_channels, kernel_size), (1, out_channels, 1), bias, device, dtype)

    def forward(self, x):
        out = F.conv1d(x, self.weight, self.padding, self.stride)
        return out + self.bias if self.bias is not None else out


class Conv2d(_ConvNd):
    """weight (out_channels, in_channels, k, k), bias (1, out_channels, 1, 1) [conv.py:69-108]."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, padding: int = 0, stride: int = 1,
                 bias: bool = True, device="cuda", dtype=None) -> None:
        super().__init__()
        self.in_channels, self.out_channels, self.kernel_size = in_channels, out_channels, kernel_size
        self.padding, self.stride = padding, stride
        self._make_params((out_channels, in_channels, kernel_size, kernel_size), (1, out_channels, 1, 1), bias,
                          device, dtype)

    def forward(self, x):
        # a bias-free convolution in training mode is (in every script) followed by BatchNorm: its epilogue also emits the
        # per-channel statistics of the output, which BatchNorm then does not have to compute (F.batch_norm)
        out = F.conv2d(x, self.weight, self.padding, self.stride, want_stats=self.bias is None and self.training)
        return out + self.bias if self.bias is not None else out


class ConvTranspose2d(_ConvNd):
    """Transposed convolution, weight (in_channels, out_channels, k, k) as in PyTorch's ConvTranspose2d, bias
    (1, out_channels, 1, 1); output size (H - 1) * stride - 2 * padding + k + output_padding, 0 <= output_padding < stride.
    The positional order is this package's Conv2d order - padding before stride, then output_padding - not PyTorch's
    (stride, padding, output_padding): pass them by keyword when porting a model. Initialisation is Conv2d's; fan_in is
    read from shape[1] = out_channels * k * k, as PyTorch does for this layer. See F.conv_transpose2d for the kernels."""

    def __init__(self, in_channels: int, out_channels: int, kernel_size: int, padding: int = 0, stride: int = 1,
                 output_padding: int = 0, bias: bool = True, device="cuda", dtype=None) -> None:
        super().__init__()
        F.check_conv_transpose2d_args(padding, stride, output_padding)
        self.in_channels, self.out_channels, self.kernel_size = in_channels, out_channels, kernel_size
        self.padding, self.stride, self.output_padding = padding, stride, output_padding
        self._make_params((in_channels, out_channels, kernel_size, kernel_size), (1, out_channels, 1, 1), bias,
                          device, dtype)

    def forward(self, x):
        out = F.conv_transpose2d(x, self.weight, self.padding, self.stride, self.output_padding)
        return out + self.bias if self.bias is not None else out
