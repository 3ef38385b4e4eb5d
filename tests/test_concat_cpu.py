"""tensor.cat and the U-Net workload without a GPU: the general path on the numpy device and the channels-last kernel path
on the numpy device of concat_ref.py, both against torch.cat (test-only dependency), argument checking, and the unet
workload trained for two steps."""
import numpy as np
import pytest

import concat_ref
import workloads

F32 = np.float32


@pytest.fixture
def ref_device(cpu_device):
    """The numpy device with the concat entry points, registered as `cpu` for one test."""
    from oracle import numpy_device
    from DeepFlows import backend_api
    yield backend_api.register_numpy_device(concat_ref.device)
    backend_api.register_numpy_device(numpy_device)


def _cat_step(arrays, grads, dim, gy, dev):
    """y and the input gradients (None where requires_grad is False) of sum(cat(xs, dim) * gy)."""
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    xs = [Tensor(a.astype(F32), device=dev, requires_grad=g) for a, g in zip(arrays, grads)]
    y = tensor.cat(xs, dim=dim)
    tensor.sum(y * Tensor(gy.astype(F32), device=dev)).backward()
    return y.numpy(), [x.grad.numpy() if x.grad is not None else None for x in xs]


def _torch_cat(torch, arrays, grads, dim, gy):
    ts = [torch.tensor(a.astype(F32), dtype=torch.float64, requires_grad=g) for a, g in zip(arrays, grads)]
    y = torch.cat(ts, dim=dim)
    (y * torch.tensor(gy.astype(F32), dtype=torch.float64)).sum().backward()
    return y.detach().numpy(), [t.grad.numpy() if g else None for t, g in zip(ts, grads)]


def _check_against_torch(arrays, grads, dim, dev, seed=0):
    torch = pytest.importorskip("torch")
    want_y, want_g = _torch_cat(torch, arrays, grads, dim, _gy(arrays, dim, seed))
    y, g = _cat_step(arrays, grads, dim, _gy(arrays, dim, seed), dev)
    assert y.shape == want_y.shape and np.array_equal(y, want_y)
    for a, b in zip(g, want_g):
        assert (a is None) == (b is None)
        if a is not None:
            assert np.array_equal(a, b)


def _gy(arrays, dim, seed):
    shape = list(arrays[0].shape)
    shape[dim] = sum(a.shape[dim] for a in arrays)
    return np.random.RandomState(seed + 100).randn(*shape)


SHAPES = {1: (5,), 2: (3, 4), 3: (2, 3, 4), 4: (2, 3, 4, 5)}


@pytest.mark.parametrize("rank", [1, 2, 3, 4])
@pytest.mark.parametrize("count", [1, 2, 3])
def test_general_path_matches_torch(cpu_device, rank, count):
    rng = np.random.RandomState(rank * 10 + count)
    for dim in range(-rank, rank):
        arrays = []
        for i in range(count):
            shape = list(SHAPES[rank])
            shape[dim] = i + 1 + (dim % rank)
            arrays.append(rng.randn(*shape))
        grads = [i != 1 for i in range(count)]   # the second input needs no gradient
        _check_against_torch(arrays, grads, dim, cpu_device, seed=rank + dim)


@pytest.mark.parametrize("widths", [(3, 5), (4, 8), (1, 2, 7), (8, 8, 8, 8, 8, 8, 8, 8), (3,) * 9, (6,)])
def test_kernel_path_matches_torch(ref_device, widths):
    from oracle import numpy_device
    rng = np.random.RandomState(len(widths))
    arrays = [rng.randn(2, w, 3, 5) for w in widths]
    grads = [True] * len(widths)
    before = numpy_device.counters.get("concat_channels_fwd", 0), numpy_device.counters.get("concat_channels_bwd", 0)
    _check_against_torch(arrays, grads, 1, ref_device)
    after = numpy_device.counters.get("concat_channels_fwd", 0), numpy_device.counters.get("concat_channels_bwd", 0)
    kernel = len(widths) <= concat_ref.MAX_SOURCES
    assert after == ((before[0] + 1, before[1] + 1) if kernel else before)


def test_kernel_path_negative_dim_and_channels_last_output(ref_device):
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    rng = np.random.RandomState(5)
    a, b = rng.randn(2, 3, 4, 5).astype(F32), rng.randn(2, 6, 4, 5).astype(F32)
    y = tensor.cat([Tensor(a, device=ref_device), Tensor(b, device=ref_device)], dim=-3)
    assert y.data.is_channels_last()
    assert np.array_equal(y.numpy(), np.concatenate([a, b], axis=1))


def test_same_tensor_twice_gets_both_slices(ref_device, cpu_device):
    torch = pytest.importorskip("torch")
    from DeepFlows import tensor, backend_api
    from DeepFlows.tensor import Tensor
    rng = np.random.RandomState(7)
    a, b = rng.randn(2, 3, 4, 4), rng.randn(2, 5, 4, 4)
    gy = rng.randn(2, 11, 4, 4)
    ta, tb = torch.tensor(a.astype(F32), dtype=torch.float64, requires_grad=True), torch.tensor(b.astype(F32), dtype=torch.float64)
    (torch.cat([ta, tb, ta], dim=1) * torch.tensor(gy.astype(F32), dtype=torch.float64)).sum().backward()
    from oracle import numpy_device
    for mod in (concat_ref.device, numpy_device):   # the kernel path, then the general path
        dev = backend_api.register_numpy_device(mod)
        x = Tensor(a.astype(F32), device=dev, requires_grad=True)
        y = tensor.cat([x, Tensor(b.astype(F32), device=dev), x], dim=1)
        tensor.sum(y * Tensor(gy.astype(F32), device=dev)).backward()
        assert np.allclose(x.grad.numpy(), ta.grad.numpy(), rtol=1e-6, atol=1e-6)


def test_input_without_grad_gets_no_buffer(ref_device, monkeypatch):
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    seen = []
    real = concat_ref.device.concat_channels_bwd

    def spy(dy, dsrcs, widths, rows):
        seen.append(list(dsrcs))
        real(dy, dsrcs, widths, rows)
    monkeypatch.setattr(concat_ref.device, "concat_channels_bwd", spy)
    rng = np.random.RandomState(9)
    xs = [Tensor(rng.randn(1, c, 2, 3).astype(F32), device=ref_device, requires_grad=g) for c, g in ((4, True), (3, False), (2, True))]
    tensor.sum(tensor.cat(xs, dim=1)).backward()
    assert len(seen) == 1 and seen[0][1] is None and seen[0][0] is not None and seen[0][2] is not None
    assert xs[1].grad is None and np.array_equal(xs[2].grad.numpy(), np.ones((1, 2, 2, 3), F32))


def test_rejected_arguments(ref_device):
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    a = Tensor(np.zeros((2, 3, 4, 4), F32), device=ref_device)
    with pytest.raises(ValueError):
        tensor.cat([])
    with pytest.raises(ValueError):
        tensor.cat([a, Tensor(np.zeros((2, 3, 4), F32), device=ref_device)], dim=1)
    with pytest.raises(ValueError):
        tensor.cat([a, Tensor(np.zeros((2, 3, 4, 5), F32), device=ref_device)], dim=1)
    for dim in (4, -5):
        with pytest.raises(IndexError):
            tensor.cat([a, a], dim=dim)
    assert tensor.cat([a, a], dim=-1).shape == (2, 3, 4, 8)
    with pytest.raises(ValueError):   # the library's limits, as the numpy device enforces them
        concat_ref.device.concat_channels_fwd([], [], None, 4)


def _unet_param_count(cin, cout, widths):
    def double(a, b):
        return 9 * a * b + 9 * b * b + 4 * b   # two bias-free 3x3 convs, two BatchNorms (gamma, beta)
    n = sum(double(a, b) for a, b in zip((cin,) + tuple(widths[:-1]), widths))
    n += sum(4 * widths[i + 1] * widths[i] + double(2 * widths[i], widths[i]) for i in range(len(widths) - 1))
    return n + widths[0] * cout + cout


def test_unet_trains_on_numpy_device(ref_device):
    import DeepFlows
    from DeepFlows import nn, tensor
    from DeepFlows.tensor import Tensor
    df = workloads.namespace(DeepFlows)
    np.random.seed(3)
    widths = (4, 8, 16)
    model = workloads.unet(df, "cpu", in_channels=3, out_channels=2, widths=widths)
    params = workloads.all_parameters(model)
    assert sum(p.data.size for _, p in params) == _unet_param_count(3, 2, widths)
    assert len(list(model.parameters())) == len(params)   # every layer is registered
    rng = np.random.RandomState(4)
    x = Tensor(rng.randn(2, 3, 8, 8).astype(F32), device=ref_device)
    t = Tensor(rng.randn(2, 2, 8, 8).astype(F32), device=ref_device)
    opt = df.optim.Adam(model.parameters(), lr=1e-3)
    losses = []
    for _ in range(2):
        y = model(x)
        assert y.shape == (2, 2, 8, 8)
        loss = nn.MSELoss()(y, t)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(loss.numpy().item())
    assert np.isfinite(losses).all()
    assert all(np.isfinite(p.data.numpy()).all() for _, p in params)
    with pytest.raises(ValueError, match="divisible"):
        model(Tensor(rng.randn(1, 3, 6, 6).astype(F32), device=ref_device))
    tensor.Graph.free_graph_all()
