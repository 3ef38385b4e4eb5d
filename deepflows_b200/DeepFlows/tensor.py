"""Tensor + tape autograd, API-compatible with the reference's `DeepFlows/tensor.py`.

What is kept (reference file:line in brackets): the process-global `Graph.node_list` tape in creation
order and its `free_graph` / `free_graph_all` [9-53]; `Tensor(array, dtype, device, name,
requires_grad)` with `.data` / `.grad` as BackendTensors, `.children` / `.parents`, `.is_leaf`,
`.dispose()` [59-235]; operator overloads and the op classes `add sub mul div pow matmul sum mean max
exp log maximum Reshape transpose get_slice` with the `forward` / `grad_fn` extension protocol of
`UnaryOperator` / `BinaryOperator` [545-974]; `backward()` on a 1-d scalar walking the tape in
reverse [421-499]; creation helpers [1068-1112].

What is different: gradients that were broadcast in the forward pass are reduced on the device
(the reference round-trips them through numpy, [462-483]); gradient buffers are created when the first
gradient arrives instead of a zero-fill per node [134]; `FusedOperator` lets one node (conv2d,
batch-norm, pooling, cross-entropy in nn/functional.py) return the gradients of all its inputs from a
single fused backward kernel; `cat` (absent in the reference) is such a node.
"""
import builtins
from typing import Any, List, Optional, Tuple, Type, Union  # noqa: F401  (re-exported: the scripts star-import this module)

import numpy  # noqa: F401
import numpy as np

from .autograd import is_grad_enable, no_grad
from .backend_selection import Device, backend_api, BackendTensor, default_device

__all__ = [
    "Graph", "Tensor", "UnaryOperator", "BinaryOperator", "FusedOperator", "add", "sub", "mul", "div", "pow",
    "matmul", "sum", "mean", "max", "exp", "log", "maximum", "sqrt", "square", "Reshape", "transpose",
    "get_slice", "cat", "empty", "zeros", "ones", "randn", "rand", "uniform",
    # what `from DeepFlows.tensor import *` also brings into a script with the reference (it defines no __all__)
    "np", "numpy", "is_grad_enable", "no_grad", "Device", "backend_api", "BackendTensor", "default_device",
    "Any", "List", "Optional", "Tuple", "Type", "Union",
]


class Graph:
    """The dynamic computation graph: every tensor that requires grad, in creation order."""
    node_list: list = []

    @classmethod
    def add(cls, node):
        cls.node_list.append(node)

    @classmethod
    def clear(cls):
        cls.node_list.clear()

    @classmethod
    def free_graph(cls):
        """Drop intermediate nodes, keep leaves (parameters) with their edges cut [24-46]."""
        survivors = []
        for node in cls.node_list:
            leaf = node.is_leaf  # decide before the edges disappear
            node.children.clear()
            node.parents.clear()
            if leaf:
                survivors.append(node)
        Graph.node_list = survivors

    @classmethod
    def free_graph_all(cls):
        for node in cls.node_list:
            node.children.clear()
            node.parents.clear()
        Graph.node_list = []


_tensor_count = 0


class ReplacesGrad:
    """Returned by a fused backward (conv dgrad with the `addend` epilogue) instead of a plain gradient: `value`
    already contains the gradient its input had accumulated so far PLUS this contribution - it replaces the input's
    gradient instead of being added to it."""
    __slots__ = ("value",)

    def __init__(self, value):
        self.value = value


def _reduce_broadcast_grad(g: BackendTensor, shape) -> BackendTensor:
    """Sum `g` down to `shape` (the inverse of the forward broadcast) on the device."""
    shape = tuple(shape)
    dev = g.device
    if dev.has("colsum"):
        if g.ndim == 4 and shape == (1, g.shape[1], 1, 1):
            gl = g.channels_last()
            out = BackendTensor.make(shape, device=dev)
            n, c, h, w = g.shape
            dev.colsum(gl._handle, out._handle, n * h * w, c)
            return out
        if g.ndim == 2 and shape == (1, g.shape[1]):
            gc = g.compact()
            out = BackendTensor.make(shape, device=dev)
            dev.colsum(gc._handle, out._handle, g.shape[0], g.shape[1])
            return out
    while g.ndim > len(shape):  # leading axes added by the broadcast
        g = g.sum(axis=0)
    for ax, (have, want) in enumerate(zip(g.shape, shape)):
        if have != want:
            g = g.sum(axis=ax, keepdims=True)
    return g


class Tensor:
    def __init__(self, array, dtype="float32", device: Optional[Device] = None, name: Optional[str] = None,
                 requires_grad: bool = False) -> None:
        global _tensor_count
        _tensor_count += 1
        self.unique_id = _tensor_count
        self.name = name if name is not None else str(self.unique_id)

        if isinstance(array, BackendTensor):
            self.data = array
        elif isinstance(array, Tensor):
            if device is None or device == array.device:
                self.data = array.data
            else:
                self.data = backend_api.Btensor(array.numpy(), dtype=dtype, device=device)
        else:
            self.data = backend_api.Btensor(np.asarray(array), dtype=dtype,
                                            device=device if device else default_device())

        self.requires_grad = bool(requires_grad) and is_grad_enable()
        self.grad = None  # BackendTensor once a gradient has arrived
        self._ngrads = 0  # gradient contributions received in the current backward pass
        self.children = []
        self.parents = []
        if self.requires_grad:
            Graph.add(self)

    @staticmethod
    def _from_numpy(numpy_array, device, dtype):
        return backend_api.Btensor(numpy_array, dtype=dtype, device=device)

    @staticmethod
    def make_const(self_Tensor, requires_grad=False):
        return Tensor(self_Tensor, requires_grad=False)

    # ---- properties ---------------------------------------------------------------------------------
    @property
    def is_leaf(self) -> bool:
        return self.requires_grad and len(self.parents) == 0

    @property
    def shape(self) -> Tuple[int]:
        return self.data.shape

    @property
    def ndim(self):
        return self.data.ndim

    @property
    def dtype(self):
        return self.data.dtype

    @property
    def size(self):
        return self.data.size

    @property
    def device(self):
        return self.data.device

    def numpy(self):
        return self.data.numpy()

    def detach(self):
        return Tensor.make_const(self)

    def dispose(self):
        """Cut this tensor out of the tape [227-235]."""
        if self.grad is not None and not self.is_leaf:
            self.grad = None
        self.children.clear()
        self.parents.clear()
        nodes = Graph.node_list
        for i in range(len(nodes) - 1, -1, -1):
            if nodes[i] is self:
                del nodes[i]
                break

    @property
    def T(self):
        return self.transpose()

    def reshape(self, *new_shape):
        return Reshape(self, new_shape)

    def transpose(self, *axes):
        return transpose(self, axes if len(axes) != 0 else None)

    def max(self, axis=None, keepdims: bool = False):
        return max(self, axis, keepdims)

    def sum(self, axis=None, keepdims: bool = False):
        return sum(self, axis, keepdims)

    def build_edge(self, node):
        self.children.append(node)
        node.parents.append(self)

    # ---- operators ------------------------------------------------------------------------------------
    def __add__(self, x):
        return add(self, x)

    def __radd__(self, x):
        return add(x, self)

    def __sub__(self, x):
        return sub(self, x)

    def __rsub__(self, x):
        return sub(x, self)

    def __mul__(self, x):
        return mul(self, x)

    def __rmul__(self, x):
        return mul(x, self)

    def __matmul__(self, x):
        return matmul(self, x)

    def __rmatmul__(self, x):
        return matmul(x, self)

    def __truediv__(self, x):
        return div(self, x)

    def __rtruediv__(self, x):
        return div(x, self)

    def __pow__(self, x):
        return pow(self, x)

    def __rpow__(self, x):
        return pow(x, self)

    def __len__(self) -> int:
        return len(self.data)

    def __pos__(self):
        return self * 1

    def __neg__(self):
        return self * -1

    def __getitem__(self, key):
        return get_slice(self, key)

    def __setitem__(self, key, value):
        assert not self.requires_grad, "In-place operation is forbidden in node requires grad."
        if isinstance(key, Tensor):
            key = key.data
        self.data[key] = value.data if isinstance(value, Tensor) else value

    def _inplace(self, other, fn):
        assert not self.requires_grad, "In-place operation is forbidden in node requires grad."
        self.data = fn(self.data, other.data if isinstance(other, Tensor) else other)
        return self

    def __iadd__(self, other):
        return self._inplace(other, lambda a, b: a + b)

    def __isub__(self, other):
        return self._inplace(other, lambda a, b: a - b)

    def __imul__(self, other):
        return self._inplace(other, lambda a, b: a * b)

    def __itruediv__(self, other):
        return self._inplace(other, lambda a, b: a / b)

    def __imatmul__(self, other):
        return self._inplace(other, lambda a, b: a @ b)

    @staticmethod
    def _raw(other):
        return other.data if isinstance(other, Tensor) else other

    @no_grad()
    def __lt__(self, other):
        return Tensor(self.data < Tensor._raw(other))

    @no_grad()
    def __le__(self, other):
        return Tensor(self.data <= Tensor._raw(other))

    @no_grad()
    def eq(self, other):
        return Tensor(self.data == Tensor._raw(other))

    @no_grad()
    def ne(self, other):
        return Tensor(self.data != Tensor._raw(other))

    @no_grad()
    def __gt__(self, other):
        return Tensor(self.data > Tensor._raw(other))

    @no_grad()
    def __ge__(self, other):
        return Tensor(self.data >= Tensor._raw(other))

    # ---- reverse pass ---------------------------------------------------------------------------------
    def _accumulate_grad(self, g):
        if isinstance(g, ReplacesGrad):
            self.grad = g.value  # the producing kernel already added what was there
        else:
            if isinstance(g, Tensor):
                g = g.data
            if g.shape != self.data.shape:
                g = _reduce_broadcast_grad(g, self.data.shape)
            self.grad = g if self.grad is None else self.grad + g
        self._ngrads += 1
        hook = Tensor._grad_ready_hook
        if hook is not None and not self.parents:
            hook(self)

    def backward(self, retain_graph: bool = False):
        nodes = Graph.node_list
        start = -1
        for i in range(len(nodes) - 1, -1, -1):
            if nodes[i] is self:
                start = i
                break
        if start < 0:
            return
        if self.data.ndim != 1:
            raise ValueError("backward should be called only on a scalar.")

        with no_grad():
            self.grad = backend_api.ones_like(self.data)
            for node in nodes[start::-1]:
                g = node.grad
                if g is None:
                    continue
                if isinstance(g, Tensor):
                    g = g.data
                if node.parents:
                    fused = getattr(node, "backward_all", None)
                    if fused is not None:
                        inputs = node.inputs
                        for parent, pg in zip(inputs, fused(g, [p.requires_grad for p in inputs])):
                            if parent.requires_grad and pg is not None:
                                parent._accumulate_grad(pg)
                    else:
                        for parent in node.parents:
                            if parent.requires_grad:
                                parent._accumulate_grad(node.grad_fn(parent, g))
                node._ngrads = 0
                if not node.is_leaf:
                    node.grad = None
            dev = self.data.device
            if dev.has("side_join"):
                dev.side_join()   # weight gradients still on the side stream (nn/functional.py: _conv2d.backward_all)
        hook = Tensor._post_backward_hook
        if hook is not None:
            hook()
            if dev.has("side_join"):
                dev.side_join()   # buckets flushed by the hook were packed as side tasks (DeepFlows.dist)
        if not retain_graph:
            Graph.free_graph()

    _post_backward_hook = None  # set by DeepFlows.dist to launch bucketed all-reduces
    _grad_ready_hook = None     # set by DeepFlows.dist: called for a leaf every time a gradient contribution arrives

    def zero_grad(self):
        self.grad = None
        self._ngrads = 0

    def to(self, device):
        name = device if isinstance(device, str) else device.name
        if self.device.name == name:
            return self
        return Tensor(self.data.numpy(), dtype=self.dtype, device=backend_api.Device(name))

    def cpu(self):
        return self.to("cpu")

    def cuda(self):
        return self.to("cuda")

    def __repr__(self) -> str:
        return "Tensor({}, requires_grad={}, device={})".format(self.data, self.requires_grad, self.device)

    def __str__(self):
        return str(self.data)


# ------------------------------------------------------------------------------------------------
# operator base classes
# ------------------------------------------------------------------------------------------------
def _as_tensor(x, device=None):
    return x if isinstance(x, Tensor) else Tensor(x, device=device)


class UnaryOperator(Tensor):
    """y = forward(x); grad_fn(x, grad) returns dL/dx given dL/dy (both BackendTensors)."""

    def __init__(self, x: Tensor) -> None:
        x = _as_tensor(x)
        super().__init__(self.forward(x), device=x.device, requires_grad=is_grad_enable() and x.requires_grad)
        if self.requires_grad:
            x.build_edge(self)

    def forward(self, x: Tensor):
        raise NotImplementedError

    def grad_fn(self, x: Tensor, grad):
        raise NotImplementedError

    def __repr__(self) -> str:
        return "Tensor({}, op={})".format(self.data, self.__class__.__name__)


class BinaryOperator(Tensor):
    """z = forward(x.data, y.data-or-scalar). A Python scalar operand is kept as a float32 scalar for
    the kernel and wrapped in a 1-element tensor for the graph [581-619]."""

    def __init__(self, x, y) -> None:
        if isinstance(x, Tensor) and isinstance(y, Tensor):
            assert x.device == y.device
            self.x, self.y = x.data, y.data
        elif isinstance(x, Tensor) and isinstance(y, BackendTensor):
            assert x.device == y.device
            self.x, self.y = x.data, y
            y = Tensor(y)
        elif isinstance(x, Tensor):
            self.x, self.y = x.data, np.float32(y)
            y = _ScalarOperand(self.y, x.device)
        else:  # scalar (op) tensor
            y = _as_tensor(y)
            x = Tensor(backend_api.full(y.shape, float(x), device=y.device))
            self.x, self.y = x.data, y.data
        super().__init__(self.forward(self.x, self.y), device=x.device,
                         requires_grad=is_grad_enable() and (x.requires_grad or y.requires_grad))
        if self.requires_grad:
            x.build_edge(self)
            y.build_edge(self)

    def forward(self, x, y):
        raise NotImplementedError

    def grad_fn(self, node, grad):
        raise NotImplementedError

    def __repr__(self) -> str:
        return "Tensor({}, op={})".format(self.data, self.__class__.__name__)


class _ScalarOperand:
    """Graph stand-in for a Python scalar operand: never requires grad, materialises its 1-element
    device tensor only if a grad_fn actually reads `.data`."""
    requires_grad = False
    ndim = 1
    shape = (1,)

    def __init__(self, value, device):
        self.value = value
        self.device = device
        self.children = []
        self.parents = []
        self._data = None

    @property
    def data(self):
        if self._data is None:
            self._data = backend_api.Btensor(np.array([self.value], dtype=np.float32), device=self.device)
        return self._data

    def build_edge(self, node):
        self.children.append(node)
        node.parents.append(self)


class FusedOperator(Tensor):
    """A node with any number of inputs whose backward produces all input gradients at once.

    Subclasses implement `forward(*inputs) -> BackendTensor` and
    `backward_all(grad, needs) -> sequence of BackendTensor | None`, aligned with `self.inputs`."""

    def __init__(self, *inputs) -> None:
        self.inputs = [t for t in inputs]
        device = self.inputs[0].device
        needs = is_grad_enable() and any(t.requires_grad for t in self.inputs)
        super().__init__(self.forward(*self.inputs), device=device, requires_grad=needs)
        if self.requires_grad:
            for t in self.inputs:
                t.build_edge(self)
        else:
            self.release()

    def forward(self, *inputs):
        raise NotImplementedError

    def backward_all(self, grad, needs):
        raise NotImplementedError

    def release(self):
        """Drop whatever forward saved for backward (called when no gradient will be needed)."""

    def __repr__(self) -> str:
        return "Tensor({}, op={})".format(self.data, self.__class__.__name__)


# ------------------------------------------------------------------------------------------------
# arithmetic
# ------------------------------------------------------------------------------------------------
class add(BinaryOperator):
    def forward(self, x, y):
        return x + y

    def grad_fn(self, node, grad):
        return grad


class sub(BinaryOperator):
    def forward(self, x, y):
        return x - y

    def grad_fn(self, node, grad):
        return grad if node is self.parents[0] else -grad


class mul(BinaryOperator):
    def forward(self, x, y):
        return x * y

    def grad_fn(self, node, grad):
        other = self.parents[1] if node is self.parents[0] else self.parents[0]
        if isinstance(other, _ScalarOperand):
            return grad * other.value
        return grad * other.data


class div(BinaryOperator):
    def forward(self, x, y):
        return x / y

    def grad_fn(self, node, grad):
        den = self.parents[1]
        q = grad / (den.value if isinstance(den, _ScalarOperand) else den.data)
        return q if node is self.parents[0] else -self.data * q


class pow(BinaryOperator):  # noqa: A001 - reference name
    def forward(self, x, y):
        return x ** y

    def grad_fn(self, node, grad):
        if node is self.parents[0]:
            e = self.parents[1]
            e = e.value if isinstance(e, _ScalarOperand) else e.data
            return (self.data * e / node.data) * grad
        return self.data * backend_api.log(self.parents[0].data) * grad


class matmul(BinaryOperator):
    def forward(self, x, y):
        return x @ y

    def grad_fn(self, node, grad):
        a, b = self.parents
        if node is a:
            return grad @ b.data.transpose()       # dA = dC . B^T (B read transposed in place)
        return a.data.transpose() @ grad           # dB = A^T . dC


class sum(UnaryOperator):  # noqa: A001 - reference name
    def __init__(self, x: Tensor, axes=None, keepdims=False) -> None:
        self.axes = axes
        self.keepdims = keepdims
        super().__init__(x)

    def forward(self, x: Tensor):
        a = x.data
        if isinstance(self.axes, (list, tuple)) and len(self.axes) > 1:
            for axis in sorted(self.axes, reverse=True):
                a = a.sum(axis=axis)
            return a
        return backend_api.summation(a, axis=self.axes, keepdims=self.keepdims)

    def grad_fn(self, x: Tensor, grad):
        # the upstream gradient broadcasts (left-aligned padding) against x's shape, as in the reference
        # [747-750] whose expand_dims for the non-keepdims case is dead code (SURVEY Q12)
        if grad.shape == x.shape:
            return grad
        return grad.broadcast_to(x.shape).compact()


class mean(UnaryOperator):
    def __init__(self, x: Tensor, axis=None, keepdims=False) -> None:
        self.axis = axis
        self.keepdims = keepdims
        super().__init__(x)

    def forward(self, x: Tensor):
        return backend_api.mean(x.data, axis=self.axis, keepdims=self.keepdims)

    def grad_fn(self, x: Tensor, grad):
        if not (self.axis is None or self.keepdims):
            grad = backend_api.expand_dims(grad, axis=self.axis)
        # ones(x.shape) * grad * (out.size / x.size)  [763-766]
        scale = self.data.size / x.data.size
        dev = grad.device
        if dev.has("compact_scale") and grad.ndim <= 8:
            # the same products, written once: scalar_mul + compact of the broadcast view in one pass (dfb_compact_scale)
            view = grad.broadcast_to(x.shape)
            xd = x.data
            if view.ndim == 4 and xd.is_channels_last() and not xd.is_compact():
                # the input is an activation in channels-last memory order: its gradient is written in that order too (what
                # the BatchNorm / convolution backward kernels it goes to read), not compact and then copied over
                n, c, h, w = view._shape
                nhwc = view.permute((0, 2, 3, 1))
                out = BackendTensor.make((n, c, h, w), (h * w * c, 1, w * c, c), dev, dev.Array(n * c * h * w))
                dev.compact_scale(nhwc._handle, out._handle, nhwc._shape, nhwc._strides, nhwc._offset, float(scale))
                return out
            out = backend_api.empty(x.shape, device=dev)
            dev.compact_scale(view._handle, out._handle, view._shape, view._strides, view._offset, float(scale))
            return out
        return (grad * scale).broadcast_to(x.shape).compact()


class max(UnaryOperator):  # noqa: A001 - reference name
    def __init__(self, x: Tensor, axis=None, keepdims=False) -> None:
        self.axis = axis
        self.keepdims = keepdims
        super().__init__(x)

    def forward(self, x: Tensor):
        return backend_api.max(x.data, axis=self.axis, keepdims=self.keepdims)

    def grad_fn(self, x: Tensor, grad):
        y = self.data
        if not (self.keepdims or self.axis is None):
            y = backend_api.expand_dims(y, axis=self.axis)
            grad = backend_api.expand_dims(grad, axis=self.axis)
        # every element equal to the maximum receives the gradient [779-791] (SURVEY Q2)
        return (y.broadcast_to(x.data.shape) == x.data) * grad


class exp(UnaryOperator):
    def forward(self, x: Tensor):
        return backend_api.exp(x.data)

    def grad_fn(self, x: Tensor, grad):
        return self.data * grad


class log(UnaryOperator):
    def forward(self, x: Tensor):
        return backend_api.log(x.data)

    def grad_fn(self, x: Tensor, grad):
        return grad / x.data


class maximum(BinaryOperator):
    def forward(self, x, y):
        return backend_api.maximum(x, y)

    def grad_fn(self, x, grad):
        if isinstance(x, _ScalarOperand):
            return (self.data == x.value) * grad
        return (self.data == x.data) * grad


def sqrt(x: Tensor):
    return x ** 0.5


def square(x: Tensor):
    return x * x


class Reshape(UnaryOperator):
    def __init__(self, x: Tensor, new_shape):
        if len(new_shape) == 1 and isinstance(new_shape[0], (tuple, list)):
            new_shape = tuple(new_shape[0])
        self.new_shape = tuple(new_shape)
        super().__init__(x)

    def forward(self, x: Tensor):
        return x.data.compact().reshape(self.new_shape)

    def grad_fn(self, x: Tensor, grad):
        return grad.compact().reshape(x.shape)


class transpose(UnaryOperator):
    def __init__(self, x: Tensor, axes: Optional[tuple] = None):
        self.axes = axes
        super().__init__(x)

    def forward(self, x: Tensor):
        return x.data.transpose(self.axes)

    def grad_fn(self, x: Tensor, grad):
        if self.axes is None:
            return grad.transpose()
        return grad.transpose(tuple(int(i) for i in np.argsort(self.axes)))


class get_slice(UnaryOperator):
    def __init__(self, x: Tensor, key):
        self.key = key.data if isinstance(key, Tensor) else key
        super().__init__(x)

    def forward(self, x: Tensor):
        return x.data[self.key]

    def grad_fn(self, x: Tensor, grad):
        full = backend_api.zeros(x.shape, device=x.device)
        full[self.key] = grad
        return full


_CONCAT_MAX_SOURCES = 8   # include/dfb200.h: DFB_CONCAT_MAX_SOURCES


def _nhwc(handle, n, c, h, w, device):
    return BackendTensor.make((n, c, h, w), (h * w * c, 1, w * c, c), device, handle)


class _cat(FusedOperator):
    """Concatenation along `dim` as one graph node. 4-d inputs along dim 1 (at most 8 of them, on a device with
    concat_channels_fwd) take one channels-last kernel each way: the output is channels-last, and so is every input
    gradient - the layout a convolution's dgrad epilogue needs to add the gradient its input already holds. Everything else
    writes a compact output with one strided setitem per input and slices the gradient back out."""

    def __init__(self, tensors, dim):
        self.dim = dim
        x = tensors[0]
        self._fused = (x.ndim == 4 and dim == 1 and len(tensors) <= _CONCAT_MAX_SOURCES
                       and x.device.has("concat_channels_fwd"))
        super().__init__(*tensors)

    def forward(self, *inputs):
        datas = [t.data for t in inputs]
        dev = datas[0].device
        self._sizes = [d.shape[self.dim] for d in datas]
        self._ndim = datas[0].ndim
        shape = list(datas[0].shape)
        shape[self.dim] = builtins.sum(self._sizes)
        if self._fused:
            xs = [d.channels_last() for d in datas]   # a pending relu(bn(..)) is written here, once
            n, c, h, w = shape
            y = dev.Array(n * h * w * c)
            dev.concat_channels_fwd([x._handle for x in xs], self._sizes, y, n * h * w)
            return _nhwc(y, n, c, h, w, dev)
        out = BackendTensor.make(shape, device=dev)
        for key, d in zip(self._slices(), datas):
            out[key] = d
        return out

    def _slices(self):
        start = 0
        for size in self._sizes:
            yield tuple(slice(start, start + size) if a == self.dim else slice(None) for a in range(self._ndim))
            start += size

    def backward_all(self, grad, needs):
        if not self._fused:
            return [grad[key].compact() if need else None for key, need in zip(self._slices(), needs)]
        n, _, h, w = grad.shape
        dev = grad.device
        gy = grad.channels_last()
        outs = [dev.Array(n * h * w * c) if need else None for c, need in zip(self._sizes, needs)]
        dev.concat_channels_bwd(gy._handle, outs, self._sizes, n * h * w)
        return [_nhwc(o, n, c, h, w, dev) if o is not None else None for o, c in zip(outs, self._sizes)]


def cat(tensors, dim=0):
    """Concatenation of a non-empty sequence of tensors along `dim`, torch.cat's contract: the tensors live on one device,
    have the same number of axes and the same size on every axis but `dim` (negative `dim` counts from the end).
    ValueError for an empty sequence or mismatched tensors, IndexError for `dim` out of range. One graph node: a tensor
    listed twice receives the sum of both slices' gradients."""
    tensors = list(tensors)
    if not tensors:
        raise ValueError("cat: expected a non-empty sequence of tensors")
    if not all(isinstance(t, Tensor) for t in tensors):
        raise TypeError("cat: expected a sequence of Tensors")
    first = tensors[0]
    nd = first.ndim
    if not -nd <= dim < nd:
        raise IndexError("cat: dim %d is out of range for %d-d tensors" % (dim, nd))
    dim %= nd
    for i, t in enumerate(tensors):
        if t.ndim != nd:
            raise ValueError("cat: tensor %d has %d dimensions, tensor 0 has %d" % (i, t.ndim, nd))
        if t.device != first.device:
            raise ValueError("cat: tensor %d is on %s, tensor 0 on %s" % (i, t.device, first.device))
        if any(a != b for ax, (a, b) in enumerate(zip(t.shape, first.shape)) if ax != dim):
            raise ValueError("cat: tensor %d has shape %s, tensor 0 has %s: sizes must match except along dim %d"
                             % (i, t.shape, first.shape, dim))
    return _cat(tensors, dim)


# ------------------------------------------------------------------------------------------------
# creation helpers [1068-1112]
# ------------------------------------------------------------------------------------------------
def empty(shape, dtype=None, device=None, requires_grad=False):
    device = device if device else default_device()
    return Tensor(device.empty(tuple(shape) if not isinstance(shape, int) else (shape,)), dtype=dtype, device=device,
                  requires_grad=requires_grad)


def zeros(shape, dtype=None, device=None, requires_grad=False):
    device = device if device else default_device()
    return Tensor(device.full(tuple(shape) if not isinstance(shape, int) else (shape,), 0.0), dtype=dtype, device=device,
                  requires_grad=requires_grad)


def ones(shape, dtype=None, device=None, requires_grad=False):
    device = device if device else default_device()
    return Tensor(device.full(tuple(shape) if not isinstance(shape, int) else (shape,), 1.0), dtype=dtype, device=device,
                  requires_grad=requires_grad)


def randn(*shape, dtype=None, device=None, requires_grad=False):
    return Tensor(np.random.randn(*shape), dtype=dtype, device=device, requires_grad=requires_grad)


def rand(*shape, dtype=None, device=None, requires_grad=False):
    return Tensor(np.random.rand(*shape), dtype=dtype, device=device, requires_grad=requires_grad)


def uniform(low: float, high: float, shape=None, dtype=None, device=None, requires_grad=False):
    return Tensor(np.random.uniform(low, high, size=shape), dtype=dtype, device=device, requires_grad=requires_grad)
