"""tensor.cat on the B200 against the numpy device of concat_ref.py (whose kernel path and general path are checked against
torch.cat in test_concat_cpu.py): the copy kernels bit-exact, their inputs as the host layer hands them over, a skip tensor
feeding a convolution and a cat, and the unet workload trained on both devices and replayed from a CUDA graph."""
import numpy as np
import pytest

import concat_ref
import parity
import workloads
from conftest import rel_err

pytestmark = pytest.mark.gpu
F32 = np.float32


@pytest.fixture
def ref_device(cuda_device):
    from oracle import numpy_device
    from DeepFlows import backend_api
    dev = backend_api.register_numpy_device(concat_ref.device)
    yield dev
    backend_api.register_numpy_device(numpy_device)
    backend_api.set_precision("fp32")


def _cat_step(arrays, dim, gy, dev, channels_last=False):
    """y and the input gradients of sum(cat(xs, dim) * gy)."""
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.backend.backend_tensor import BackendTensor
    tensor.Graph.free_graph_all()
    xs = []
    for a in arrays:
        d = BackendTensor(a, device=dev)
        xs.append(Tensor(d.channels_last() if channels_last else d, requires_grad=True))
    y = tensor.cat(xs, dim=dim)
    tensor.sum(y * Tensor(gy, device=dev)).backward()
    return y.numpy(), [x.grad.numpy() for x in xs]


def _assert_same(got, want):
    assert np.array_equal(got[0], want[0])
    assert len(got[1]) == len(want[1])
    for a, b in zip(got[1], want[1]):
        assert np.array_equal(a, b)


# widths: multiples of 4 take the float4 kernels, the others the scalar ones
@pytest.mark.parametrize("widths", [(8, 16), (16, 32, 8), (3, 5), (5, 3, 8), (8,) * 8, (3, 4, 5, 6, 7, 9, 1, 2)])
def test_kernel_matches_reference(cuda_device, ref_device, widths):
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.backend.backend_tensor import BackendTensor
    rng = np.random.RandomState(sum(widths))
    n, h, w = 3, 5, 7   # 105 rows: no width fills the last block of the grid-stride loop
    arrays = [rng.randn(n, c, h, w).astype(F32) for c in widths]
    gy = rng.randn(n, sum(widths), h, w).astype(F32)
    want = _cat_step(arrays, 1, gy, ref_device)
    _assert_same(_cat_step(arrays, 1, gy, cuda_device, channels_last=True), want)
    _assert_same(_cat_step(arrays, 1, gy, cuda_device), want)   # NCHW-compact inputs: copied to channels-last first
    # one launch each way for channels-last inputs
    xs = [Tensor(BackendTensor(a, device=cuda_device).channels_last(), requires_grad=True) for a in arrays]
    g = BackendTensor(gy, device=cuda_device).channels_last()
    l0 = cuda_device.launch_count()
    y = tensor.cat(xs, dim=1)
    l1 = cuda_device.launch_count()
    grads = y.backward_all(g, [True] * len(xs))
    assert (l1 - l0, cuda_device.launch_count() - l1) == (1, 1)
    assert y.data.is_channels_last() and all(d.is_channels_last() for d in grads)
    for d, a in zip(grads, want[1]):
        assert np.array_equal(d.numpy(), a)
    tensor.Graph.free_graph_all()


@pytest.mark.parametrize("dim", [0, 2, 3])
def test_general_path_matches_reference(cuda_device, ref_device, dim):
    rng = np.random.RandomState(dim)
    shapes = [[2, 3, 4, 5] for _ in range(3)]
    for i, s in enumerate(shapes):
        s[dim] += i
    arrays = [rng.randn(*s).astype(F32) for s in shapes]
    out = list(shapes[0])
    out[dim] = sum(s[dim] for s in shapes)
    gy = rng.randn(*out).astype(F32)
    _assert_same(_cat_step(arrays, dim, gy, cuda_device), _cat_step(arrays, dim, gy, ref_device))


def _skip_net(dev, order, seed=0):
    """h = relu(bn(conv1(x))) feeds conv2(h) and cat([u, h]) (the consumers created in `order`); returns the loss and the
    gradients of x, u and every parameter."""
    from DeepFlows import backend_api, nn, tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.backend.backend_tensor import PendingTensor
    tensor.Graph.free_graph_all()
    np.random.seed(seed)
    conv1 = nn.Conv2d(4, 8, 3, padding=1, bias=False, device=dev)
    bn = nn.BatchNorm2d(8, device=dev)
    conv2 = nn.Conv2d(8, 8, 3, padding=1, bias=False, device=dev)
    rng = np.random.RandomState(seed + 1)
    d = backend_api.Device(dev)
    x = Tensor(rng.randn(4, 4, 8, 8).astype(F32), device=d, requires_grad=True)
    u = Tensor(rng.randn(4, 6, 8, 8).astype(F32), device=d, requires_grad=True)
    g1, g2 = Tensor(rng.randn(4, 8, 8, 8).astype(F32), device=d), Tensor(rng.randn(4, 14, 8, 8).astype(F32), device=d)
    h = nn.ReLU()(bn(conv1(x)))
    if dev == "cuda":
        assert isinstance(h.data, PendingTensor) and h.data.pending   # written by whichever consumer comes first
    if order == "conv_first":
        a = conv2(h)
        b = tensor.cat([u, h], dim=1)
    else:
        b = tensor.cat([u, h], dim=1)
        a = conv2(h)
    loss = tensor.sum(a * g1) + tensor.sum(b * g2)
    loss.backward()
    params = [conv1.weight, bn.weight, bn.bias, conv2.weight]
    return [loss.numpy(), x.grad.numpy(), u.grad.numpy()] + [p.grad.numpy() for p in params]


@pytest.mark.parametrize("order", ["conv_first", "cat_first"])
def test_skip_tensor_feeding_conv_and_cat(cuda_device, ref_device, order, monkeypatch):
    from DeepFlows import backend_api
    from DeepFlows.nn import functional as F
    backend_api.set_precision("fp32")
    want = _skip_net("cpu", order)
    fusions = []
    real = F._conv2d._dgrad_fusion

    def spy(self, *args):
        out = real(self, *args)
        fusions.append(out)
        return out
    monkeypatch.setattr(F._conv2d, "_dgrad_fusion", spy)
    got = _skip_net("cuda", order)
    for a, b in zip(got, want):
        assert rel_err(a, b) <= 1e-5
    if order == "conv_first":
        # the cat's backward runs first (reverse creation order) and leaves a channels-last gradient on h: conv2's dgrad
        # epilogue adds it instead of a separate sum
        assert any(f is not None and f[0] is not None for f in fusions)


def _unet_run(df, dev, steps, graph=False):
    from DeepFlows import backend_api, nn, tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.cuda_graph import CapturedStep
    tensor.Graph.free_graph_all()
    np.random.seed(21)
    model = workloads.unet(df, dev, widths=(8, 16, 32))
    rng = np.random.RandomState(22)
    xs = [rng.randn(4, 3, 16, 16).astype(F32) for _ in range(steps)]
    target = np.tanh(rng.randn(4, 3, 16, 16)).astype(F32)
    opt = df.optim.Adam(model.parameters(), lr=1e-3)
    crit = nn.MSELoss()
    d = backend_api.Device(dev)
    x = Tensor(backend_api.Btensor(xs[0], device=d))
    t = Tensor(backend_api.Btensor(target, device=d))

    def step_fn():
        loss = crit(model(x), t)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    step = CapturedStep(step_fn, device=d, warmup=1) if graph else step_fn
    losses = []
    for xb in xs:
        d.from_numpy(xb, x.data._handle)
        losses.append(step().data.numpy().copy())
    if graph:
        assert step.captured
        step.destroy()
    return losses, [p.data.numpy().copy() for _, p in workloads.all_parameters(model)]


def test_unet_adam_steps_match_reference(cuda_device, ref_device):
    from DeepFlows import backend_api
    df = parity.df_namespace()
    backend_api.set_precision("fp32")
    want = _unet_run(df, "cpu", 2)
    got = _unet_run(df, "cuda", 2)
    for a, b in zip(got[0], want[0]):
        assert abs(a.item() - b.item()) <= 1e-4 * max(1.0, abs(b.item()))
    assert len(got[1]) == len(want[1]) == 34
    for a, b in zip(got[1], want[1]):
        assert rel_err(a, b) <= 1e-4


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_unet_graph_replay_is_bit_identical(cuda_device, precision):
    from DeepFlows import backend_api
    df = parity.df_namespace()
    backend_api.set_precision(precision)
    try:
        eager = _unet_run(df, "cuda", 4)
        graph = _unet_run(df, "cuda", 4, graph=True)
    finally:
        backend_api.set_precision("fp32")
    for a, b in zip(eager[0], graph[0]):
        assert np.array_equal(a, b)
    for a, b in zip(eager[1], graph[1]):
        assert np.array_equal(a, b)
