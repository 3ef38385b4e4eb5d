"""nn.functional: same function names and argument meaning as the reference's
`DeepFlows/nn/functional.py`, with each op that the reference composes from many tensor ops
implemented as ONE graph node over the device's fused (L1) entry points.

    conv2d          reference: __pad2d + __im2col2d (k*k strided setitems) + permute/compact + naive matmul
                    [functional.py:249-344]  ->  implicit-GEMM fprop / dgrad / wgrad kernels
    max_pool2d      reference: pad + im2col + row max, equality-mask backward [347-374, tensor.py:779-791]
                    ->  one forward kernel, one backward kernel with the same tie semantics
    avg_pool2d      reference raises AttributeError [377-404] (SURVEY Q4)  ->  implemented
    conv_transpose2d  absent in the reference  ->  the convolution's dgrad / fprop / wgrad kernels with roles swapped
    interpolate     absent in the reference  ->  nearest / bilinear upsampling kernels, forward and backward
    cross_entropy   reference: 10 tensor ops [104-115]  ->  fused softmax-CE forward / backward
    batch_norm      reference: 16 tensor ops inside BatchNorm2d.forward [modules/batchnorm.py:30-55]
    relu            reference: maximum(x, 0) [15-16]  ->  same forward kernel, one-kernel backward

Activations flow between these ops as logical (N,C,H,W) views over channels-last memory, which is
also the physical order the reference's conv output has before its final transpose [343-344].
"""
import os
from typing import Optional

from .. import tensor
from ..tensor import Tensor, FusedOperator, UnaryOperator, BinaryOperator
from .. import backend_api
from ..backend.backend_tensor import (BackendTensor, PendingTensor, BnApply, precision_mode, get_dgrad_mode, get_fusion)

LAYOUT_NCHW, LAYOUT_NHWC = 0, 1
WLAYOUT_KCRS, WLAYOUT_KRSC = 0, 1


def _nhwc_view(handle, n, c, h, w, device):
    return BackendTensor.make((n, c, h, w), (h * w * c, 1, w * c, c), device, handle)


# ------------------------------------------------------------------------------------------------
# linear / activations
# ------------------------------------------------------------------------------------------------
_LINEAR_SMALL = os.environ.get("DEEPFLOWS_LINEAR_SMALL", "1") != "0"   # 0: the classifier through matmul + add again


class _linear_small(FusedOperator):
    """x @ W + b for a layer with at most 16 outputs (the classifier of every network) as ONE launch, and its backward
    (dx, dW, db) as one more - through the general path they are a split-K GEMM, its reduction and a row-vector add, and a
    column-sum kernel, two GEMMs and another reduction: eight launches of a few microseconds each for 0.66 MFLOP."""

    def __init__(self, x: Tensor, weight: Tensor, bias: Optional[Tensor]):
        self._has_bias = bias is not None
        super().__init__(*((x, weight, bias) if bias is not None else (x, weight)))

    def forward(self, x, weight, bias=None):
        xd, wd = x.data, weight.data
        xd = xd if xd.is_compact() and xd._offset == 0 else xd.compact()
        wd = wd if wd.is_compact() and wd._offset == 0 else wd.compact()
        m, k = xd.shape
        n = wd.shape[1]
        dev = xd.device
        y = BackendTensor.make((m, n), device=dev)
        b = None
        if bias is not None:
            b = bias.data if bias.data.is_compact() and bias.data._offset == 0 else bias.data.compact()
        dev.linear_small_fwd(xd._handle, wd._handle, b._handle if b is not None else None, y._handle, m, k, n)
        self._x, self._w, self._mkn = xd, wd, (m, k, n)
        return y

    def backward_all(self, grad, needs):
        m, k, n = self._mkn
        dev = self._x.device
        g = grad if grad.is_compact() and grad._offset == 0 else grad.compact()
        dx = BackendTensor.make((m, k), device=dev) if needs[0] else None
        dw = BackendTensor.make((k, n), device=dev) if needs[1] else None
        db = BackendTensor.make(self.inputs[2].shape, device=dev) if self._has_bias and needs[2] else None
        dev.linear_small_bwd(self._x._handle, self._w._handle, g._handle, dx._handle if dx is not None else None,
                             dw._handle if dw is not None else None, db._handle if db is not None else None, m, k, n)
        return (dx, dw, db) if self._has_bias else (dx, dw)

    def release(self):
        self._x = self._w = None


def linear(input: Tensor, weight: Tensor, bias: Optional[Tensor] = None):
    """x @ W + b with W stored (in_features, out_features) like the reference [8-12]."""
    if (_LINEAR_SMALL and get_fusion() and isinstance(input, Tensor) and input.ndim == 2 and weight.ndim == 2 and weight.shape[1] <= 16
            and input.shape[1] == weight.shape[0] and input.device.has("linear_small_fwd")
            and (bias is None or (isinstance(bias, Tensor) and bias.data.size == weight.shape[1]))):
        return _linear_small(input, weight, bias)
    out = input @ weight
    return out + bias if bias is not None else out


class _relu(UnaryOperator):
    def forward(self, x: Tensor):
        self._expr = None
        xd = x.data
        if isinstance(xd, PendingTensor) and xd.pending and xd.device.has("relu_bwd_bn"):
            fused = xd.with_relu()  # relu(bn(..) [+ ..]) written by the BatchNorm's own pass
            if fused is not None:
                self._expr, self._x = fused, None
                return fused
        src = xd if xd.is_dense() else xd.compact()
        self._x = src
        out = src._like()
        src.device.scalar_maximum(src._handle, 0.0, out._handle)
        return out

    def grad_fn(self, x: Tensor, grad):
        if self._expr is not None:
            aux = getattr(grad, "_aux", None)
            if aux is not None and aux[0] == "bn_sums" and len(aux) > 3 and aux[3] == id(self._expr):
                return grad   # the convolution that produced this gradient applied the mask in its epilogue
            # the pre-activation was never stored: the backward kernel recomputes it exactly as the forward pass did
            e = self._expr
            n, c, h, w = e.shape
            dev = e.device
            gy = grad.channels_last()
            dx = dev.Array(n * c * h * w)
            dev.relu_bwd_bn(e.sides[0].bwd_tuple(), e.sides[1].bwd_tuple() if len(e.sides) > 1 else None,
                            e.residual._handle if e.residual is not None else None, gy._handle, dx, n * h * w, c)
            return _nhwc_view(dx, n, c, h, w, dev)
        src = self._x
        dev = src.device
        if not dev.has("relu_bwd"):
            return (self.data == src) * grad
        if grad.shape != src.shape or grad.strides != src.strides or not grad.is_dense():
            # bring both to the plain compact layout
            src, grad = src.compact(), grad.compact()
        out = src._like()
        dev.relu_bwd(src._handle, grad._handle, out._handle, src._handle.size)
        return out


def relu(input: Tensor) -> Tensor:
    return _relu(input)


class sigmoid(UnaryOperator):
    """1/(1+exp(-x)), evaluated as 0.5*tanh(x/2)+0.5 (no overflow for large |x|). The reference version
    relies on boolean-mask indexing that BackendTensor does not implement [19-27]."""

    def forward(self, input: Tensor):
        return (input.data * 0.5).tanh() * 0.5 + 0.5

    def grad_fn(self, input: Tensor, grad):
        return self.data * (1 - self.data) * grad


class tanh(UnaryOperator):
    def forward(self, input: Tensor):
        return backend_api.tanh(input.data)

    def grad_fn(self, input: Tensor, grad):
        return (1 - self.data ** 2) * grad


def leaky_relu(input: Tensor, negative_slope: float):
    return tensor.maximum(input, input * negative_slope)


def softmax(input: Tensor, dim=None, keepdims=False):
    dim = 1 if dim is None else dim
    shifted = input - tensor.max(input, dim, True)
    e = tensor.exp(shifted)
    return e / tensor.sum(e, dim, True)


def log_softmax(input: Tensor, dim=None, keepdims=False):
    dim = 1 if dim is None else dim
    shifted = input - tensor.max(input, dim, True)
    return shifted - tensor.log(tensor.sum(tensor.exp(shifted), dim, True))


# ------------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------------
def _reduce_loss(per_elem: Tensor, reduction: str):
    if reduction == "mean":
        return tensor.mean(per_elem)
    if reduction == "sum":
        return tensor.sum(per_elem)
    assert 0, "reduction must be mean or sum."


def l1_loss(input: Tensor, target: Tensor, reduction: str = "mean"):
    diff = input - target
    return _reduce_loss(tensor.maximum(diff, diff * -1), reduction)


def nll_loss(input: Tensor, target: Tensor, reduction: str = "mean"):
    return _reduce_loss(-input * target, reduction)


def mse_loss(input: Tensor, target: Tensor, reduction: str = "mean"):
    return _reduce_loss(tensor.square(input - target), reduction)


def binary_cross_entropy(input: Tensor, target: Tensor, reduction: str = "mean"):
    raise NotImplementedError("binary_cross_entropy is a stub in the reference as well (functional.py:100-101)")


class _softmax_cross_entropy(FusedOperator):
    """loss = scale * sum_i sum_j -(x_ij - max_i - logsumexp_i) * t_ij, shape (1,)."""

    def __init__(self, logits: Tensor, target: Tensor, scale: float):
        self.scale = float(scale)
        super().__init__(logits, target)

    def forward(self, logits, target):
        x, t = logits.data.compact(), target.data.compact()
        self._x, self._t = x, t
        out = BackendTensor.make((1,), device=x.device)
        x.device.softmax_ce_fwd(x._handle, t._handle, out._handle, x.shape[0], x.shape[1], self.scale)
        return out

    def backward_all(self, grad, needs):
        x, t = self._x, self._t
        dx = None
        if needs[0]:
            dx = BackendTensor.make(x.shape, device=x.device)
            x.device.softmax_ce_bwd(x._handle, t._handle, grad.compact()._handle, dx._handle, x.shape[0], x.shape[1],
                                    self.scale)
        dt = None
        if needs[1]:  # d/dt = -scale * log_softmax(x); rare (targets are constants)
            ls = x - x.max(axis=1, keepdims=True).broadcast_to(x.shape)
            ls = ls - ls.exp().sum(axis=1, keepdims=True).log().broadcast_to(x.shape)
            dt = ls * (-self.scale) * grad.broadcast_to(x.shape)
        return dx, dt

    def release(self):
        self._x = self._t = None


def cross_entropy(input: Tensor, target: Tensor, reduction: str = "mean", dim: int = 1):
    """Stable log-softmax cross entropy against dense (one-hot or smoothed) target rows [104-115]."""
    assert reduction in ("mean", "sum"), "reduction must be mean or sum."
    target = target if isinstance(target, Tensor) else Tensor(target, device=input.device)
    if input.ndim == 2 and dim in (1, -1) and input.device.has("softmax_ce_fwd"):
        return _softmax_cross_entropy(input, target, 1.0 / input.shape[0] if reduction == "mean" else 1.0)
    shifted = input - tensor.max(input, dim, True)
    lse = tensor.log(tensor.sum(tensor.exp(shifted), dim, True))
    nll = -(shifted - lse) * target
    if reduction == "mean":
        return tensor.sum(tensor.sum(nll, dim, True)) * (1.0 / input.shape[0])
    return tensor.sum(nll)


# ------------------------------------------------------------------------------------------------
# convolution
# ------------------------------------------------------------------------------------------------
_SIDE_STREAM = os.environ.get("DEEPFLOWS_SIDE", "1") != "0"   # 0: weight gradients stay on the compute stream (measurements)
_SIDE_LAG = int(os.environ.get("DEEPFLOWS_SIDE_LAG", "2"))      # 0: join the weight gradient right behind its dgrad (round 1)


def _lazy(dev):
    """Trailing `lazy` argument of conv2d_fprop_stats / conv2d_dgrad_fused on a device that has statistic slots
    (include/dfb200.h: dfb_conv2d_fprop_stats_lazy): the statistics go ONLY to the BatchNorm kernels - here: to the BnApply
    record of the BatchNorm behind the convolution, and to `bn_bwd_apply` of the BatchNorm(s) that receive the gradient."""
    return (True,) if dev.has("STATS_LAZY") else ()


def _conv_weight(kernel: Tensor, dev):
    """(weight data, WLAYOUT_*) of a (K,C,R,R) convolution weight as the convolution kernels take it.
    Weights live channels-last (K,R,R,C) on the B200 device - the layout the tensor-core kernels read
    in place, for fprop and (as the transposed operand) for dgrad. A Parameter that arrives compact
    (fresh from init / load_state_dict / a checkpoint) is re-laid out once, here; its logical shape,
    `.numpy()` and every other consumer are unaffected (strides carry the layout)."""
    wd = kernel.data
    if wd.ndim == 4 and wd.is_channels_last():
        return wd, WLAYOUT_KRSC
    if (wd.ndim == 4 and dev.name == "cuda" and dev.has("WLAYOUT_KRSC")
            and not isinstance(kernel, (UnaryOperator, BinaryOperator, FusedOperator))):  # a stored tensor, not an op result
        kernel.data = wd = wd.channels_last()
        return wd, WLAYOUT_KRSC
    return wd.compact(), WLAYOUT_KCRS


def _workspace(dev, geom):
    n_floats = dev.conv2d_workspace_floats(*geom)
    return (dev.Array(n_floats), n_floats) if n_floats else (None, 0)


def _wgrad_beside_dgrad(dev, needs, weight: Tensor, wgrad, dgrad):
    """Runs the weight gradient `wgrad()` (when needs[1]) and returns the input gradient `dgrad()` (when needs[0], else
    None) of a convolution-like op. The two only share their inputs: when both are needed the weight gradient goes to the
    side stream and the two kernels (neither fills 148 SMs on the small layers) run concurrently."""
    both = needs[0] and needs[1] and dev.has("side_begin") and _SIDE_STREAM
    # The weight gradient is read by nobody before the end of backward() (Tensor.backward joins the side stream there;
    # DeepFlows.dist joins before it packs a bucket), so the compute stream only waits for the weight gradient of
    # _SIDE_LAG layers ago: wgrad overlaps the next layers' dgrad / BatchNorm chain instead of sitting on it. Not when
    # the weight already holds a gradient (shared weights, accumulation): the sum would read dw right away.
    lazy_join = both and _SIDE_LAG > 0 and dev.has("side_join_lag") and weight.grad is None
    if needs[1]:
        if both:
            dev.side_begin()
        try:
            wgrad()
        finally:
            if both:
                dev.side_end()
    dx = dgrad() if needs[0] else None
    if both:
        if lazy_join:
            dev.side_join_lag(_SIDE_LAG)
        else:
            dev.side_join()
    return dx


class _conv2d(FusedOperator):
    def __init__(self, x: Tensor, kernel: Tensor, padding: int, stride: int, want_stats: bool = False):
        self.padding, self.stride = int(padding), int(stride)
        self._want_stats = bool(want_stats)
        super().__init__(x, kernel)

    def forward(self, x, kernel):
        xd = x.data
        dev = xd.device
        wd, w_layout = _conv_weight(kernel, dev)
        n, c, h, w = xd.shape
        k, c2, r, r2 = wd.shape
        assert c == c2 and r == r2, "conv2d: kernel %s does not match input %s" % (wd.shape, xd.shape)
        mode = precision_mode()
        if xd.is_channels_last():
            layout = LAYOUT_NHWC
        elif xd.is_compact() and (mode == 3 or c <= 4):
            layout = LAYOUT_NCHW  # the FFMA / first-layer kernels gather straight from NCHW (network input)
        else:
            xd, layout = xd.channels_last(), LAYOUT_NHWC
        p, s = self.padding, self.stride
        oh, ow = (h + 2 * p - r) // s + 1, (w + 2 * p - r) // s + 1
        self._geom = (n, c, h, w, k, r, p, s)
        self._x, self._layout, self._w, self._mode = xd, layout, wd, mode
        self._wl = (w_layout,) if w_layout else ()  # trailing argument only when it is not the default
        self._col = None
        y = dev.Array(n * oh * ow * k)
        if (c <= 4 and c * r * r <= 32 and k % 4 == 0 and mode == 1 and n * oh * ow >= 16384 and self._want_stats and get_fusion()
                and w_layout == WLAYOUT_KRSC and dev.has("stem_cols") and tensor.is_grad_enable()):
            # First layer (image input) at training batch sizes in TF32 mode (fp32 mode keeps the exact FFMA first-layer kernels): the receptive fields are written once as a
            # [pixels x 32] column matrix; the convolution is its 1x1 convolution with the padded weights on the tensor
            # pipe (statistics for the BatchNorm included), and the matrix is kept for the weight gradient.
            cols = c * r * r
            col, wp, mean_var = dev.Array(n * oh * ow * 32), dev.Array(k * 32), dev.Array(2 * k)
            dev.stem_cols(xd._handle, layout, col, n, c, h, w, r, p, s, w_layout)
            dev.stem_pad_weights(wd._handle, wp, k, cols)
            # (in the fp32-accurate three-term mode 0: 27-75 taps of an HBM-bound layer cost nothing extra, and the network's
            # input layer keeps its precision in TF32 mode as it did on the FFMA first-layer kernels - with TF32 operands
            # here the BatchNorm behind it turns a 5e-4 output error into a 1e-1 error of this layer's weight gradient)
            dev.conv2d_fprop_stats(col, LAYOUT_NHWC, wp, WLAYOUT_KRSC, y, n, 32, oh, ow, k, 1, 0, 1, 0, mean_var, *_lazy(dev))
            self._col = (col, oh, ow, cols)
            out = _nhwc_view(y, n, k, oh, ow, dev)
            out._aux = ("colstats", mean_var)
            return out
        if self._want_stats and get_fusion() and dev.has("conv2d_fprop_stats") and tensor.is_grad_enable():
            # the BatchNorm that follows gets the per-channel mean / variance of y from this kernel's epilogue
            mean_var = dev.Array(2 * k)
            dev.conv2d_fprop_stats(xd._handle, layout, wd._handle, w_layout, y, n, c, h, w, k, r, p, s, mode, mean_var, *_lazy(dev))
            out = _nhwc_view(y, n, k, oh, ow, dev)
            out._aux = ("colstats", mean_var)
            return out
        ws, ws_n = _workspace(dev, self._geom)
        dev.conv2d_fprop(xd._handle, layout, wd._handle, y, n, c, h, w, k, r, p, s, mode, ws, ws_n, *self._wl)
        return _nhwc_view(y, n, k, oh, ow, dev)

    def backward_all(self, grad, needs):
        n, c, h, w, k, r, p, s = self._geom
        dev = self._x.device
        gy = grad.channels_last()
        ws, ws_n = _workspace(dev, self._geom)
        dw = None
        if needs[1]:
            # the weight gradient is produced in the weight's own layout, so optimizer and all-reduce walk
            # the two buffers side by side
            dw = _nhwc_view(dev.Array(k * c * r * r), k, c, r, r, dev) if self._wl else BackendTensor.make((k, c, r, r), device=dev)

        def wgrad():
            if self._col is not None:   # first layer: the column matrix of the forward pass is still there
                col, oh, ow, cols = self._col
                dev.conv2d_wgrad_cols(col, gy._handle, dw._handle, self._wl[0] if self._wl else WLAYOUT_KCRS, n, oh, ow, k, cols,
                                      self._mode)
            else:
                dev.conv2d_wgrad(self._x._handle, self._layout, gy._handle, dw._handle, n, c, h, w, k, r, p, s,
                                 self._mode, ws, ws_n, *self._wl)

        def dgrad():
            buf = dev.Array(n * h * w * c)
            dmode = 0 if get_dgrad_mode() == "reference" else 1
            fuse = self._dgrad_fusion(dev, n, c, h, w) if (dmode == 1 and get_fusion() and dev.has("conv2d_dgrad_fused")) else None
            if fuse is not None:
                addend, recs, sums, relu_expr = fuse
                res = relu_expr.residual if relu_expr is not None else None
                dev.conv2d_dgrad_fused(gy._handle, self._w._handle, self._wl[0] if self._wl else WLAYOUT_KCRS, buf, n, c, h, w, k, r, p,
                                       s, self._mode, dmode, addend._handle if addend is not None else None,
                                       recs[0].bwd_tuple() if len(recs) > 0 else None, recs[1].bwd_tuple() if len(recs) > 1 else None,
                                       sums, relu_expr is not None, res._handle if res is not None else None, *_lazy(dev))
                dx = _nhwc_view(buf, n, c, h, w, dev)
                if recs:
                    # (the 4th entry tells the ReLU node between this convolution and the BatchNorm(s) that its mask is applied)
                    dx._aux = ("bn_sums", sums, {id(rec): 1 + i for i, rec in enumerate(recs)}, id(relu_expr) if relu_expr is not None else None)
                if addend is not None:
                    dx = tensor.ReplacesGrad(dx)   # already holds (existing gradient of x) + dgrad
            else:
                dev.conv2d_dgrad(gy._handle, self._w._handle, buf, n, c, h, w, k, r, p, s, self._mode, dmode, ws, ws_n,
                                 *self._wl)
                dx = _nhwc_view(buf, n, c, h, w, dev)
            return dx

        return _wgrad_beside_dgrad(dev, needs, self.inputs[1], wgrad, dgrad), dw

    def _dgrad_fusion(self, dev, n, c, h, w):
        """What the dgrad epilogue can take over for the input tensor x of this convolution:
          * the sum with the gradient x already holds (the other branch of a residual block, processed earlier);
          * when this contribution COMPLETES x's gradient: the two reductions of BatchNorm backward for the BatchNorm(s)
            that will receive exactly this gradient - x itself (conv -> bn -> conv), or the two terms of the residual sum
            x = bn2(..) + bn_ds(..) / bn2(..) + identity (`add` hands its gradient to both parents unchanged).
        Returns (addend BackendTensor | None, [BnApply records], sums Array | None) or None."""
        x = self.inputs[0]
        addend = None
        if x.grad is not None:
            g = x.grad.data if isinstance(x.grad, Tensor) else x.grad
            if g.shape == (n, c, h, w) and g.is_channels_last():
                addend = g
            else:
                return None
        recs, relu_expr = [], None
        if x._ngrads + 1 == len(x.children):   # nothing else will arrive after this
            node = x
            if isinstance(node, _relu) and node._expr is not None and len(node.parents) == 1 and dev.has("relu_bwd_bn"):
                # x = relu(expression of BatchNorms): the epilogue applies the ReLU's backward too, if the node under the
                # ReLU feeds nothing else (its gradient is then exactly the masked one)
                below = node.parents[0]
                if isinstance(below, Tensor) and len(below.children) == 1 and below._ngrads == 0:
                    relu_expr, node = node._expr, below
            cand = []
            if isinstance(node, _batch_norm_train):
                cand = [node]
            elif isinstance(node, tensor.add) and all(isinstance(q, Tensor) for q in node.parents):
                cand = [q for q in node.parents if isinstance(q, _batch_norm_train) and len(q.children) == 1 and q._ngrads == 0]
            for bn in cand:
                rec = getattr(bn, "_rec", None)
                if rec is not None and rec.applied and rec.x.shape == (n, c, h, w):
                    recs.append(rec)
            if relu_expr is not None:
                # the mask needs every term of the pre-activation: all BatchNorms of the expression must be the ones found
                if [id(r_) for r_ in relu_expr.sides] != [id(r_) for r_ in recs]:
                    recs, relu_expr = [], None
        if addend is None and not recs:
            return None
        return addend, recs[:2], (dev.Array(3 * c) if recs else None), relu_expr

    def release(self):
        self._x = self._w = self._col = None


def conv2d(x: Tensor, kernel: Tensor, padding: int = 0, stride: int = 1, want_stats: bool = False):
    """2-d convolution, x (N,C,H,W), kernel (K,C,R,R); square kernel, symmetric zero padding, scalar
    stride, no dilation/groups - the reference's contract [316-335]. `want_stats` (new, optional): also produce the
    per-channel statistics of the output for a BatchNorm that follows (Conv2d sets it for bias-free convolutions)."""
    if not isinstance(x, Tensor):
        x = Tensor(x, device=kernel.device)
    return _conv2d(x, kernel, padding, stride, want_stats)


def check_conv_transpose2d_args(padding: int, stride: int, output_padding: int):
    """ValueError unless stride >= 1, padding >= 0 and 0 <= output_padding < stride - under that condition a convolution
    with the same kernel size, stride and padding maps the transposed convolution's output size back to its input size."""
    if stride < 1 or padding < 0:
        raise ValueError("conv_transpose2d: stride must be >= 1 and padding >= 0 (got stride=%d, padding=%d)" % (stride, padding))
    if not 0 <= output_padding < stride:
        raise ValueError("conv_transpose2d: output_padding must satisfy 0 <= output_padding < stride (got %d, stride %d)"
                         % (output_padding, stride))


def conv_transpose2d_size(h_in: int, kernel_size: int, padding: int, stride: int, output_padding: int) -> int:
    """Output height (or width) of a transposed convolution: (h_in - 1) * stride - 2 * padding + kernel_size + output_padding
    (arguments checked by check_conv_transpose2d_args; ValueError for an empty output)."""
    check_conv_transpose2d_args(padding, stride, output_padding)
    h = (h_in - 1) * stride - 2 * padding + kernel_size + output_padding
    if h < 1:
        raise ValueError("conv_transpose2d: input size %d, kernel %d, padding %d, stride %d give an empty output"
                         % (h_in, kernel_size, padding, stride))
    return h


class _conv_transpose2d(FusedOperator):
    """The transposed convolution of x (N,in,H,W) with weight (in,out,k,k) is the input gradient of the convolution
    conv2d(., weight, padding, stride) - K = in, C = out in the notation of the convolution entry points - so every pass
    runs on that convolution's kernels:
        forward        y  = conv2d_dgrad(x, w)              (always DGRAD_EXACT: the transposed convolution itself)
        d/dx           dx = conv2d_fprop(dy, w)
        d/dw           dw = conv2d_wgrad(x = dy, dy = x)    (in the weight's own layout, on the side stream)"""

    def __init__(self, x: Tensor, kernel: Tensor, padding: int, stride: int, output_padding: int):
        self.padding, self.stride, self.output_padding = int(padding), int(stride), int(output_padding)
        super().__init__(x, kernel)

    def forward(self, x, kernel):
        xd = x.data.channels_last()
        dev = xd.device
        wd, w_layout = _conv_weight(kernel, dev)
        n, k, hi, wi = xd.shape
        k2, c, r, r2 = wd.shape
        assert k == k2 and r == r2, "conv_transpose2d: weight %s does not match input %s" % (wd.shape, xd.shape)
        p, s, op = self.padding, self.stride, self.output_padding
        h, w = conv_transpose2d_size(hi, r, p, s, op), conv_transpose2d_size(wi, r, p, s, op)
        self._geom = (n, c, h, w, k, r, p, s)
        self._x, self._w, self._mode = xd, wd, precision_mode()
        self._wl = (w_layout,) if w_layout else ()
        ws, ws_n = _workspace(dev, self._geom)
        y = dev.Array(n * h * w * c)
        dev.conv2d_dgrad(xd._handle, wd._handle, y, n, c, h, w, k, r, p, s, self._mode, 1, ws, ws_n, *self._wl)
        return _nhwc_view(y, n, c, h, w, dev)

    def backward_all(self, grad, needs):
        n, c, h, w, k, r, p, s = self._geom
        dev = self._x.device
        hi, wi = self._x.shape[2:]
        gy = grad.channels_last()
        ws, ws_n = _workspace(dev, self._geom)
        dw = None
        if needs[1]:
            dw = _nhwc_view(dev.Array(k * c * r * r), k, c, r, r, dev) if self._wl else BackendTensor.make((k, c, r, r), device=dev)

        def wgrad():
            dev.conv2d_wgrad(gy._handle, LAYOUT_NHWC, self._x._handle, dw._handle, n, c, h, w, k, r, p, s, self._mode, ws, ws_n,
                             *self._wl)

        def dgrad():
            buf = dev.Array(n * hi * wi * k)
            dev.conv2d_fprop(gy._handle, LAYOUT_NHWC, self._w._handle, buf, n, c, h, w, k, r, p, s, self._mode, ws, ws_n, *self._wl)
            return _nhwc_view(buf, n, k, hi, wi, dev)

        return _wgrad_beside_dgrad(dev, needs, self.inputs[1], wgrad, dgrad), dw

    def release(self):
        self._x = self._w = None


def conv_transpose2d(x: Tensor, weight: Tensor, padding: int = 0, stride: int = 1, output_padding: int = 0):
    """2-d transposed convolution, x (N,in,H,W), weight (in,out,k,k) as in PyTorch -> (N,out,H_out,W_out) with
    H_out = (H - 1) * stride - 2 * padding + k + output_padding, 0 <= output_padding < stride. Square kernel, no
    dilation / groups. The positional order is this package's conv2d order - padding before stride - which a positional
    call written for torch.nn.functional.conv_transpose2d (stride, padding, output_padding) would misread.

    It is the input gradient of conv2d with the same weight, padding and stride, and runs on that convolution's kernels:
      * forward on the tensor pipe (tcgen05) in TF32 and fp32 mode when in % 4 == 0, out % 4 == 0, stride 1 or 2, and for
        stride 2 an even output size (k = 4 / p = 1, k = 2 / p = 0, k = 3 / p = 1 / output_padding = 1); odd stride-2 outputs
        (k = 3, p = 1, output_padding = 0), channel counts that are not multiples of 4 and stride >= 3 run on the exact FFMA
        kernels;
      * backward with respect to x: conv2d_fprop(dy, weight), and with respect to the weight: conv2d_wgrad with x and dy
        swapped - for an image-producing layer (out <= 4, out * k * k <= 80, in a multiple of 16 up to 64) both through the
        exact direct kernels of conv_direct.cu that serve the first layer of a convolutional network.
    The exact transposed convolution is computed whatever `set_dgrad_mode` says (that switch selects the reference's
    last-writer-wins quirk for Conv2d's backward only)."""
    if not isinstance(x, Tensor):
        x = Tensor(x, device=weight.device)
    return _conv_transpose2d(x, weight, padding, stride, output_padding)


# ------------------------------------------------------------------------------------------------
# pooling
# ------------------------------------------------------------------------------------------------
class _pool2d(FusedOperator):
    def __init__(self, x: Tensor, kernel_size: int, is_max: bool):
        self.k, self.is_max = int(kernel_size), is_max
        super().__init__(x)

    def forward(self, x):
        xd = x.data.channels_last()
        n, c, h, w = xd.shape
        k = self.k
        oh, ow = (h - k) // k + 1, (w - k) // k + 1
        dev = xd.device
        y = dev.Array(n * oh * ow * c)
        if self.is_max:
            dev.maxpool2d_fwd(xd._handle, y, None, n, h, w, c, k)
        else:
            dev.avgpool2d_fwd(xd._handle, y, n, h, w, c, k)
        out = _nhwc_view(y, n, c, oh, ow, dev)
        self._x, self._y = xd, out
        return out

    def backward_all(self, grad, needs):
        xd = self._x
        n, c, h, w = xd.shape
        dev = xd.device
        gy = grad.channels_last()
        dx = dev.Array(n * h * w * c)
        fused = self._bn_relu_below(dev, n, c, h, w) if self.is_max else None
        if fused is not None:
            # conv -> BatchNorm -> ReLU -> MaxPool (the first stage of the ResNet, every VGG stage): pool backward, the ReLU's
            # mask and the BatchNorm's two reductions in ONE pass over the BatchNorm's input instead of three
            rec, relu_expr = fused
            sums = dev.Array(3 * c)
            dev.maxpool_relu_bn_bwd(rec.bwd_tuple(), self._y._handle, gy._handle, dx, sums, n, h, w, c, self.k)
            out = _nhwc_view(dx, n, c, h, w, dev)
            out._aux = ("bn_sums", sums, {id(rec): 1}, id(relu_expr))   # (the ReLU node passes it through, the BatchNorm applies)
            return (out,)
        if self.is_max:  # every tied maximum receives the gradient (reference semantics, SURVEY Q2)
            dev.maxpool2d_bwd(xd._handle, self._y._handle, gy._handle, dx, n, h, w, c, self.k)
        else:
            dev.avgpool2d_bwd(gy._handle, dx, n, h, w, c, self.k)
        return (_nhwc_view(dx, n, c, h, w, dev),)

    def _bn_relu_below(self, dev, n, c, h, w):
        """(BnApply record, fused ReLU expression) when this pool's input is relu(bn(x)) written by ONE dfb_bn_fwd_apply
        launch, this gradient is everything the ReLU will receive, and the BatchNorm feeds nothing but the ReLU."""
        if not (get_fusion() and dev.has("maxpool_relu_bn_bwd") and dev.has("bn_bwd_apply")):
            return None
        x = self.inputs[0]
        if not (isinstance(x, _relu) and x._expr is not None and len(x.parents) == 1):
            return None
        if len(x.children) != 1:
            return None
        below = x.parents[0]
        if not (isinstance(below, _batch_norm_train) and len(below.children) == 1 and below._ngrads == 0):
            return None
        rec, expr = getattr(below, "_rec", None), x._expr
        if rec is None or not rec.applied or rec.x.shape != (n, c, h, w):
            return None
        if [id(r_) for r_ in expr.sides] != [id(rec)] or expr.residual is not None:
            return None
        return rec, expr

    def release(self):
        self._x = self._y = None


UPSAMPLE_NEAREST, UPSAMPLE_BILINEAR = 0, 1   # include/dfb200.h: DFB_UPSAMPLE_*
_UPSAMPLE_MODES = {"nearest": UPSAMPLE_NEAREST, "bilinear": UPSAMPLE_BILINEAR}
_UPSAMPLE_MAX_SCALE = 8


class _upsample2d(FusedOperator):
    """(N,C,H,W) -> (N,C,H*s,W*s) by an integer factor s, one channels-last kernel each way (dfb_upsample2d_fwd / _bwd)."""

    def __init__(self, x: Tensor, scale: int, mode: int):
        self.scale, self.mode = int(scale), int(mode)
        super().__init__(x)

    def forward(self, x):
        xd = x.data.channels_last()
        n, c, h, w = xd.shape
        dev = xd.device
        s = self.scale
        y = dev.Array(n * h * s * w * s * c)
        dev.upsample2d_fwd(xd._handle, y, n, h, w, c, s, self.mode)
        self._shape, self._dev = (n, c, h, w), dev
        return _nhwc_view(y, n, c, h * s, w * s, dev)

    def backward_all(self, grad, needs):
        n, c, h, w = self._shape
        dev = self._dev
        gy = grad.channels_last()
        dx = dev.Array(n * h * w * c)
        dev.upsample2d_bwd(gy._handle, dx, n, h, w, c, self.scale, self.mode)
        return (_nhwc_view(dx, n, c, h, w, dev),)

    def release(self):
        self._dev = None


def _integer_scale(v, what):
    """An integer upsampling factor from a number or a pair of equal numbers, else NotImplementedError."""
    if isinstance(v, (tuple, list)):
        if len(v) != 2 or v[0] != v[1]:
            raise NotImplementedError("interpolate: %s %r: only the same factor for height and width is supported" % (what, v))
        v = v[0]
    if isinstance(v, bool) or not isinstance(v, (int, float)) or v != int(v) or not 1 <= int(v) <= _UPSAMPLE_MAX_SCALE:
        raise NotImplementedError("interpolate: %s %r: only integer factors from 1 to %d are supported"
                                  % (what, v, _UPSAMPLE_MAX_SCALE))
    return int(v)


def interpolate(input: Tensor, size=None, scale_factor=None, mode: str = "nearest", align_corners=None):
    """Upsampling of an (N,C,H,W) tensor by an integer factor s (1..8, the same for H and W), torch.nn.functional.interpolate's
    arguments: `scale_factor` = s, or `size` = (H*s, W*s) (an int for both axes). Modes "nearest" (a copy of the source pixel
    (oh // s, ow // s)) and "bilinear" with align_corners=False (PyTorch's half-pixel rule, edges clamped). Other modes,
    align_corners=True and non-integer or per-axis factors raise NotImplementedError; malformed arguments ValueError."""
    if mode not in _UPSAMPLE_MODES:
        raise NotImplementedError("interpolate: mode %r is not supported (nearest, bilinear)" % (mode,))
    if align_corners is not None and mode == "nearest":
        raise ValueError("interpolate: align_corners can only be set with the interpolating mode 'bilinear'")
    if align_corners:
        raise NotImplementedError("interpolate: align_corners=True is not supported (align_corners=False / None is)")
    if input.ndim != 4:
        raise ValueError("interpolate: expected an (N,C,H,W) input, got shape %s" % (input.shape,))
    if (size is None) == (scale_factor is None):
        raise ValueError("interpolate: give exactly one of size and scale_factor")
    h, w = input.shape[2:]
    if scale_factor is not None:
        s = _integer_scale(scale_factor, "scale_factor")
    else:
        oh, ow = (size, size) if isinstance(size, int) else tuple(size)
        if oh % h or ow % w or oh // h != ow // w:
            raise NotImplementedError("interpolate: size %r is not the same integer multiple of the input size (%d, %d)"
                                      % (size, h, w))
        s = _integer_scale(oh // h, "size / input size")
    return _upsample2d(input, s, _UPSAMPLE_MODES[mode])


class _pad_spatial(UnaryOperator):
    """Zero padding of the trailing spatial axes (reference: __pad1d / __pad2d, functional.py:153-164,297-313)."""

    def __init__(self, x: Tensor, p: int):
        self.p = int(p)
        super().__init__(x)

    def forward(self, x: Tensor):
        if self.p == 0:
            return x.data
        return x.data.compact().pad([(0, 0), (0, 0)] + [(self.p, self.p)] * (x.ndim - 2))

    def grad_fn(self, x: Tensor, grad):
        if self.p == 0:
            return grad
        p = self.p
        return grad[(slice(None), slice(None)) + (slice(p, -p),) * (x.ndim - 2)].compact()


class _im2col(UnaryOperator):
    """Sliding windows as an explicit tensor, built from k (1-d) or k*k (2-d) strided slice copies like the reference's
    __im2col1d / __im2col2d (functional.py:118-145,249-294): (N,C,L) -> (N,C,k,Lo), (N,C,H,W) -> (N,C,k,k,OH,OW).
    Only the shapes the fused kernels do not take come through here (pooling with stride != kernel or padding, 1-d ops).
    Backward scatters the windows back: summed where windows overlap (`exact`), or - 2-d, dgrad mode `reference` - the
    reference's last-writer-wins assignment (SURVEY Q1)."""

    def __init__(self, x: Tensor, kernel_size: int, stride: int):
        self.k, self.s = int(kernel_size), int(stride)
        super().__init__(x)

    def _windows(self, shape):
        k, s = self.k, self.s
        if len(shape) == 3:
            lo = (shape[2] - k) // s + 1
            return [((i,), (slice(i, i + lo * s, s),)) for i in range(k)], (lo,)
        oh, ow = (shape[2] - k) // s + 1, (shape[3] - k) // s + 1
        return [((i, j), (slice(i, i + oh * s, s), slice(j, j + ow * s, s))) for i in range(k) for j in range(k)], (oh, ow)

    def forward(self, x: Tensor):
        xd = x.data.compact()
        n, c = xd.shape[:2]
        wins, out_sp = self._windows(xd.shape)
        col = backend_api.zeros((n, c) + (self.k,) * len(out_sp) + out_sp, device=xd.device)
        both, tail = (slice(None), slice(None)), (slice(None),) * len(out_sp)
        for pos, sl in wins:
            col[both + pos + tail] = xd[both + sl]
        return col

    def grad_fn(self, x: Tensor, grad):
        g = grad.compact()
        n, c = x.shape[:2]
        wins, out_sp = self._windows(x.shape)
        gx = backend_api.zeros(x.shape, device=x.device)
        both, tail = (slice(None), slice(None)), (slice(None),) * len(out_sp)
        overwrite = len(out_sp) == 2 and get_dgrad_mode() == "reference"
        for pos, sl in wins:
            piece = g[both + pos + tail].compact().reshape((n, c) + out_sp)
            if not overwrite:
                piece = gx[both + sl].compact() + piece
            gx[both + sl] = piece
        return gx


def _pool2d_general(x: Tensor, kernel_size: int, stride: int, padding: int, is_max: bool):
    """Pooling for any stride / zero padding, composed like the reference composes it [347-374]: pad with ZEROS (not
    -inf), windows, row maximum with the equality-mask gradient (every tied maximum receives it) / row average."""
    n, c = x.shape[:2]
    col = _im2col(_pad_spatial(x, padding), kernel_size, stride)
    oh, ow = col.shape[-2:]
    rows = col.transpose(0, 4, 5, 1, 2, 3).reshape(-1, kernel_size * kernel_size)
    # (keepdims: the reference's non-keepdims sum back-propagates by left-aligned broadcasting, SURVEY Q12)
    out = tensor.max(rows, 1, True) if is_max else tensor.sum(rows, 1, True) * (1.0 / (kernel_size * kernel_size))
    return out.reshape(n, oh, ow, c).transpose(0, 3, 1, 2)


def max_pool2d(x: Tensor, kernel_size: int, stride: int, padding=0):
    stride = kernel_size if not stride else stride
    if stride == kernel_size and padding == 0:
        return _pool2d(x, kernel_size, True)      # the fused kernels: every configuration of the scripts
    return _pool2d_general(x, kernel_size, stride, padding, True)


def avg_pool2d(x: Tensor, kernel_size: int, stride: int, padding=0):
    stride = kernel_size if not stride else stride
    if stride == kernel_size and padding == 0:
        return _pool2d(x, kernel_size, False)
    return _pool2d_general(x, kernel_size, stride, padding, False)


# ------------------------------------------------------------------------------------------------
# batch normalisation
# ------------------------------------------------------------------------------------------------
class _batch_norm_train(FusedOperator):
    def __init__(self, x, weight, bias, running_mean, running_var, momentum, eps):
        self._rm, self._rv = running_mean, running_var
        self.momentum, self.eps = float(momentum), float(eps)
        self._affine = weight is not None
        self._rec = None
        super().__init__(*([x, weight, bias] if self._affine else [x]))

    def forward(self, x, weight=None, bias=None):
        xd = x.data.channels_last()
        n, c, h, w = xd.shape
        dev = xd.device
        rows = n * h * w
        g = weight.data.compact() if weight is not None else None
        b = bias.data.compact() if bias is not None else None
        rm = self._rm.data.compact() if self._rm is not None else None
        rv = self._rv.data.compact() if self._rv is not None else None
        if rm is not None and rm is not self._rm.data:  # running stats were non-compact views: write back
            self._rm.data, self._rv.data = rm, rv
        self._x, self._g = xd, g
        self._rm = self._rv = None
        aux = getattr(xd, "_aux", None)
        if aux is not None and aux[0] == "colstats" and get_fusion() and dev.has("bn_fwd_apply"):
            # statistics came with the convolution's output: the BatchNorm is one elementwise pass, launched when its
            # output is first needed - by then `+ identity` / a second BatchNorm / ReLU may have joined the expression
            self._rec = BnApply(xd, aux[1], g, b, rm, rv, self.momentum, self.eps)
            self._mean, self._invstd = self._rec.save_mean, self._rec.save_invstd
            return PendingTensor.defer((n, c, h, w), (h * w * c, 1, w * c, c), dev, [self._rec])
        y = dev.Array(rows * c)
        self._mean, self._invstd = dev.Array(c), dev.Array(c)
        dev.bn_fwd_train(xd._handle, g._handle if g is not None else None, b._handle if b is not None else None, y,
                         self._mean, self._invstd, rm._handle if rm is not None else None,
                         rv._handle if rv is not None else None, self.momentum, self.eps, rows, c)
        return _nhwc_view(y, n, c, h, w, dev)

    def backward_all(self, grad, needs):
        xd = self._x
        n, c, h, w = xd.shape
        dev = xd.device
        gy = grad.channels_last()
        rows = n * h * w
        dx = dev.Array(rows * c) if needs[0] else None
        gh = self._g._handle if self._g is not None else None
        aux = getattr(gy, "_aux", None)
        if (aux is not None and aux[0] == "bn_sums" and self._rec is not None and id(self._rec) in aux[2]
                and dev.has("bn_bwd_apply")):
            # the convolution that produced this gradient also reduced it: sum(dy) and sum(dy * x_hat) are there
            sums, row = aux[1], aux[2][id(self._rec)]
            db = BackendTensor.make((1, c, 1, 1), None, dev, sums, 0)
            dg = BackendTensor.make((1, c, 1, 1), None, dev, sums, row * c)
            if dx is None and dev.has("STATS_LAZY"):
                dx = dev.Array(rows * c)   # lazily delivered sums become dbeta / dgamma in this kernel: it has to run
            if dx is not None:
                dev.bn_bwd_apply(xd._handle, gy._handle, gh, self._mean, self._invstd, (sums, 0), (sums, row * c), dx, rows, c)
            out = [_nhwc_view(dx, n, c, h, w, dev) if needs[0] else None]
            if self._affine:
                out += [dg if needs[1] else None, db if needs[2] else None]
            return out
        dg = BackendTensor.make((1, c, 1, 1), device=dev) if self._affine and needs[1] else None
        db = BackendTensor.make((1, c, 1, 1), device=dev) if self._affine and needs[2] else None
        dev.bn_bwd(xd._handle, gy._handle, gh, self._mean, self._invstd,
                   dx, dg._handle if dg is not None else None, db._handle if db is not None else None, rows, c)
        out = [_nhwc_view(dx, n, c, h, w, dev) if dx is not None else None]
        if self._affine:
            out += [dg, db]
        return out

    def release(self):
        self._x = self._g = self._mean = self._invstd = self._rec = None


def batch_norm(x: Tensor, weight, bias, running_mean, running_var, training: bool, momentum: float, eps: float):
    """BatchNorm2d forward. Training: batch mean / biased variance over (N,H,W), running statistics
    updated in place with the biased variance (reference quirk Q7). Evaluation: running statistics."""
    if training:
        return _batch_norm_train(x, weight, bias, running_mean, running_var, momentum, eps)
    if running_mean is None:
        x_hat = x
    elif not tensor.is_grad_enable() and x.device.has("bn_fwd_eval"):
        xd = x.data.channels_last()
        n, c, h, w = xd.shape
        dev = xd.device
        y = dev.Array(n * h * w * c)
        dev.bn_fwd_eval(xd._handle, weight.data.compact()._handle if weight is not None else None,
                        bias.data.compact()._handle if bias is not None else None,
                        running_mean.data.compact()._handle, running_var.data.compact()._handle, y, eps, n * h * w, c)
        return Tensor(_nhwc_view(y, n, c, h, w, dev))
    else:
        x_hat = (x - running_mean) / (running_var + eps) ** 0.5
    if weight is not None:
        return x_hat * weight + bias
    return x_hat


# ------------------------------------------------------------------------------------------------
# 1-d ops (composed from tensor ops; not on the accelerated path)
# ------------------------------------------------------------------------------------------------
def conv1d(input: Tensor, kernel: Tensor, padding: int = 0, stride: int = 1):
    """1-d convolution, input (N,C,L), kernel (K,C,k) -> (N,K,Lo). The reference's version cannot run (it indexes the
    window tensor with too few axes and calls a non-existent `.swapaxes`, functional.py:118-191); this is the operation
    it documents, composed the way it intended: pad, windows, one matmul."""
    k_out, c, k = kernel.shape
    n = input.shape[0]
    col = _im2col(_pad_spatial(input, padding), k, stride)             # (N, C, k, Lo)
    lo = col.shape[-1]
    rows = col.transpose(0, 3, 1, 2).reshape(n * lo, c * k)            # (N*Lo, C*k)
    out = rows @ kernel.reshape(k_out, c * k).transpose(1, 0)          # (N*Lo, K)
    return out.reshape(n, lo, k_out).transpose(0, 2, 1)


def max_pool1d(x: Tensor, kernel_size: int, stride: int, padding: int = 0):
    """(N,C,L) -> (N,C,Lo): zero padding, window maximum, equality-mask gradient [193-218]."""
    n, c = x.shape[:2]
    col = _im2col(_pad_spatial(x, padding), kernel_size, stride)       # (N, C, k, Lo)
    lo = col.shape[-1]
    return tensor.max(col.transpose(0, 1, 3, 2).reshape(n * c * lo, kernel_size), 1, True).reshape(n, c, lo)


def avg_pool1d(x: Tensor, kernel_size: int, stride: int, padding: int = 0):
    """(N,C,L) -> (N,C,Lo): zero padding, window average (padding zeros count, like the 2-d version) [221-246]."""
    n, c = x.shape[:2]
    col = _im2col(_pad_spatial(x, padding), kernel_size, stride)
    lo = col.shape[-1]
    return (tensor.sum(col.transpose(0, 1, 3, 2).reshape(n * c * lo, kernel_size), 1, True) * (1.0 / kernel_size)).reshape(n, c, lo)
