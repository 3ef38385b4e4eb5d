"""ConvTranspose2d and Upsample on the B200 against the same layers on the numpy device (whose upsample functions and
transposed convolution are checked against PyTorch in test_decoder_cpu.py), and the generator workload trained on both."""
import numpy as np
import pytest

import decoder_ref
import parity
import workloads
from conftest import rel_err

pytestmark = pytest.mark.gpu
F32 = np.float32
TOL = {"fp32": 1e-5, "tf32": 2e-2}


@pytest.fixture
def ref_device(cuda_device):
    from oracle import numpy_device
    from DeepFlows import backend_api
    dev = backend_api.register_numpy_device(decoder_ref.device)
    yield dev
    backend_api.register_numpy_device(numpy_device)
    backend_api.set_precision("fp32")


def _layer_step(layer, x, gy, dev):
    """y, dx and the parameter gradients of sum(layer(x) * gy)."""
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    tensor.Graph.free_graph_all()
    tx = Tensor(x, device=dev, requires_grad=True)
    y = layer(tx)
    tensor.sum(y * Tensor(gy, device=dev)).backward()
    grads = {k: p.grad.numpy() for k, p in layer.named_parameters()}
    for _, p in layer.named_parameters():
        p.grad = None
    return y.numpy(), tx.grad.numpy(), grads


def _conv_transpose(cin, cout, k, p, s, op, dev, wt, b):
    from DeepFlows import nn, backend_api
    layer = nn.ConvTranspose2d(cin, cout, k, padding=p, stride=s, output_padding=op, device=dev)
    layer.weight.data = backend_api.Btensor(wt, device=dev)
    layer.bias.data = backend_api.Btensor(b, device=dev)
    return layer


# (in, out, k, padding, stride, output_padding, batch, input size, whether conv_tc_ok takes the forward pass)
GEOMS = {
    "k3s1p1": (16, 8, 3, 1, 1, 0, 4, 9, True),
    "k3s2p1op1": (16, 8, 3, 1, 2, 1, 4, 8, True),      # even output
    "k3s2p1op0": (16, 8, 3, 1, 2, 0, 4, 8, False),     # odd output: FFMA kernels
    "k4s2p1": (32, 16, 4, 1, 2, 0, 4, 8, True),
    "k2s2p0": (16, 16, 2, 0, 2, 0, 4, 8, True),
    "stride3": (8, 8, 3, 1, 3, 2, 2, 5, False),
    "out3_in5": (5, 3, 4, 1, 2, 0, 2, 8, False),
    "out3_in16": (16, 3, 4, 1, 2, 0, 4, 8, False),     # image-producing layer: direct kernels in its backward
    "partial_tiles": (64, 32, 4, 1, 2, 0, 3, 7, True),
}


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("name", sorted(GEOMS))
def test_conv_transpose2d_matches_reference(cuda_device, ref_device, name, precision):
    from DeepFlows import backend_api
    cin, cout, k, p, s, op, n, h, tc = GEOMS[name]
    rng = np.random.RandomState(sum(map(ord, name)))
    wt = (rng.randn(cin, cout, k, k) / np.sqrt(cin * k * k)).astype(F32)
    b = rng.randn(1, cout, 1, 1).astype(F32)
    x = rng.randn(n, cin, h, h + 1).astype(F32)
    ho, wo = (h - 1) * s - 2 * p + k + op, h * s - 2 * p + k + op
    gy = rng.randn(n, cout, ho, wo).astype(F32)
    want = _layer_step(_conv_transpose(cin, cout, k, p, s, op, ref_device, wt, b), x, gy, ref_device)
    backend_api.set_precision(precision)
    layer = _conv_transpose(cin, cout, k, p, s, op, cuda_device, wt, b)
    tc0 = cuda_device.tc_launch_count()
    got = _layer_step(layer, x, gy, cuda_device)
    if tc:
        assert cuda_device.tc_launch_count() > tc0, "the tensor pipe did not run"
    tol = TOL[precision]
    assert got[0].shape == (n, cout, ho, wo)
    assert rel_err(got[0], want[0]) <= tol
    assert rel_err(got[1], want[1]) <= tol
    assert rel_err(got[2]["weight"], want[2]["weight"]) <= tol
    assert rel_err(got[2]["bias"], want[2]["bias"]) <= tol


@pytest.mark.parametrize("name", ["k3s2p1op1", "k4s2p1", "stride3"])
def test_conv_transpose2d_ignores_dgrad_mode(cuda_device, name):
    from DeepFlows import backend_api, tensor
    from DeepFlows.tensor import Tensor
    cin, cout, k, p, s, op, n, h, _ = GEOMS[name]
    rng = np.random.RandomState(3)
    layer = _conv_transpose(cin, cout, k, p, s, op, cuda_device, rng.randn(cin, cout, k, k).astype(F32),
                            rng.randn(1, cout, 1, 1).astype(F32))
    x = Tensor(rng.randn(n, cin, h, h).astype(F32), device=cuda_device)
    with tensor.no_grad():
        exact = layer(x).numpy()
        backend_api.set_dgrad_mode("reference")
        quirk = layer(x).numpy()
    assert np.array_equal(exact, quirk)


@pytest.mark.parametrize("mode", ["nearest", "bilinear"])
@pytest.mark.parametrize("s", [2, 3, 4])
@pytest.mark.parametrize("c", [8, 6])
def test_upsample_matches_reference(cuda_device, ref_device, mode, s, c):
    from DeepFlows import nn
    rng = np.random.RandomState(s * c)
    x = rng.randn(3, c, 5, 7).astype(F32)
    gy = rng.randn(3, c, 5 * s, 7 * s).astype(F32)
    want = _layer_step(nn.Upsample(scale_factor=s, mode=mode), x, gy, ref_device)
    got = _layer_step(nn.Upsample(scale_factor=s, mode=mode), x, gy, cuda_device)
    if mode == "nearest":
        assert np.array_equal(got[0], want[0])
    else:
        assert rel_err(got[0], want[0]) <= 1e-6
    assert rel_err(got[1], want[1]) <= 1e-6


def _generator_run(df, dev, steps, graph=False):
    from DeepFlows import backend_api, nn, tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.cuda_graph import CapturedStep
    tensor.Graph.free_graph_all()
    np.random.seed(11)
    model = workloads.dcgan_generator(df, dev, nz=16, widths=(32, 16, 8, 8))
    rng = np.random.RandomState(12)
    zs = [rng.randn(4, 16).astype(F32) for _ in range(steps)]
    target = np.tanh(rng.randn(4, 3, 64, 64)).astype(F32)
    opt = df.optim.Adam(model.parameters(), lr=1e-3)
    crit = nn.MSELoss()
    d = backend_api.Device(dev)
    z = Tensor(backend_api.Btensor(zs[0], device=d))
    t = Tensor(backend_api.Btensor(target, device=d))

    def step_fn():
        loss = crit(model(z), t)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    step = CapturedStep(step_fn, device=d, warmup=1) if graph else step_fn
    losses = []
    for zb in zs:
        d.from_numpy(zb, z.data._handle)
        losses.append(step().data.numpy().copy())
    if graph:
        assert step.captured
        step.destroy()
    return losses, [p.data.numpy().copy() for _, p in workloads.all_parameters(model)]


def test_generator_adam_steps_match_reference(cuda_device, ref_device):
    from DeepFlows import backend_api
    df = parity.df_namespace()
    backend_api.set_precision("fp32")
    want = _generator_run(df, "cpu", 2)
    got = _generator_run(df, "cuda", 2)
    for a, b in zip(got[0], want[0]):
        assert abs(float(a) - float(b)) <= 1e-4 * max(1.0, abs(float(b)))
    assert len(got[1]) == len(want[1]) == 13
    for a, b in zip(got[1], want[1]):
        assert rel_err(a, b) <= 1e-4


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_generator_graph_replay_is_bit_identical(cuda_device, precision):
    from DeepFlows import backend_api
    df = parity.df_namespace()
    backend_api.set_precision(precision)
    try:
        eager = _generator_run(df, "cuda", 4)
        graph = _generator_run(df, "cuda", 4, graph=True)
    finally:
        backend_api.set_precision("fp32")
    for a, b in zip(eager[0], graph[0]):
        assert np.array_equal(a, b)
    for a, b in zip(eager[1], graph[1]):
        assert np.array_equal(a, b)
