"""ConvTranspose2d and Upsample without a GPU: the float64 references against PyTorch (test-only dependency), the host
layer on the numpy device against torch autograd, and argument checking."""
import numpy as np
import pytest

import decoder_ref as ref

F32 = np.float32


def _tensor_grads(torch, module_fn, x, gy):
    """torch forward / backward: (y, dx, {name: grad})."""
    tx = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    mod = module_fn()
    y = mod(tx)
    y.backward(torch.tensor(gy, dtype=torch.float64))
    params = mod.named_parameters() if hasattr(mod, "named_parameters") else []
    return y.detach().numpy(), tx.grad.numpy(), {k: p.grad.numpy() for k, p in params}


def _close(got, want, tol):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    err = np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)
    assert err <= tol, err


@pytest.mark.parametrize("s", [1, 2, 3, 4])
@pytest.mark.parametrize("shape", [(2, 3, 5, 4), (1, 4, 1, 3)])
def test_upsample_references_match_torch(s, shape):
    torch = pytest.importorskip("torch")
    rng = np.random.RandomState(s)
    x = rng.randn(*shape)
    gy = rng.randn(shape[0], shape[1], shape[2] * s, shape[3] * s)
    for mode, fwd, bwd in (("nearest", ref.upsample_nearest_fwd, ref.upsample_nearest_bwd),
                           ("bilinear", ref.upsample_bilinear_fwd, ref.upsample_bilinear_bwd)):
        kw = {"align_corners": False} if mode == "bilinear" else {}
        y, dx, _ = _tensor_grads(torch, lambda: (lambda t: torch.nn.functional.interpolate(t, scale_factor=s, mode=mode, **kw)), x, gy)
        _close(fwd(x, s), y, 1e-6)
        _close(bwd(gy, s), dx, 1e-6)


@pytest.mark.parametrize("k,s,p,op", [(3, 1, 1, 0), (3, 2, 1, 1), (3, 2, 1, 0), (4, 2, 1, 0), (2, 2, 0, 0), (3, 3, 1, 2)])
def test_conv_transpose_reference_matches_torch(k, s, p, op):
    torch = pytest.importorskip("torch")
    rng = np.random.RandomState(k * 10 + s)
    x, w = rng.randn(2, 5, 4, 3), rng.randn(5, 3, k, k)
    want = torch.nn.functional.conv_transpose2d(torch.tensor(x), torch.tensor(w), stride=s, padding=p, output_padding=op).numpy()
    _close(ref.conv_transpose2d(x, w, p, s, op), want, 1e-6)


@pytest.fixture
def ref_device(cpu_device):
    """The numpy device with the upsample entry points, registered as `cpu` for one test."""
    from oracle import numpy_device
    from DeepFlows import backend_api
    yield backend_api.register_numpy_device(ref.device)
    backend_api.register_numpy_device(numpy_device)


def _run_layer(layer, x, gy, dev):
    from DeepFlows import tensor
    from DeepFlows.tensor import Tensor
    tx = Tensor(x.astype(F32), device=dev, requires_grad=True)
    y = layer(tx)
    tensor.sum(y * Tensor(gy.astype(F32), device=dev)).backward()
    return y.numpy(), tx.grad.numpy()


@pytest.mark.parametrize("k,s,p,op,cin,cout", [(3, 1, 1, 0, 4, 8), (3, 2, 1, 1, 8, 4), (3, 2, 1, 0, 6, 5), (4, 2, 1, 0, 8, 8),
                                               (2, 2, 0, 0, 4, 4), (3, 3, 1, 2, 4, 4), (4, 2, 1, 0, 5, 3)])
def test_conv_transpose2d_layer_on_numpy_device(ref_device, k, s, p, op, cin, cout):
    torch = pytest.importorskip("torch")
    from DeepFlows import nn, backend_api
    rng = np.random.RandomState(k + 7 * s + cin)
    n, h, w = 3, 5, 4
    layer = nn.ConvTranspose2d(cin, cout, k, padding=p, stride=s, output_padding=op, device="cpu")
    assert layer.weight.shape == (cin, cout, k, k) and layer.bias.shape == (1, cout, 1, 1)
    wt, b = rng.randn(cin, cout, k, k).astype(F32) * 0.3, rng.randn(1, cout, 1, 1).astype(F32)
    layer.weight.data = backend_api.Btensor(wt, device=ref_device)
    layer.bias.data = backend_api.Btensor(b, device=ref_device)
    x = rng.randn(n, cin, h, w)
    ho, wo = (h - 1) * s - 2 * p + k + op, (w - 1) * s - 2 * p + k + op
    gy = rng.randn(n, cout, ho, wo)
    y, dx = _run_layer(layer, x, gy, ref_device)

    def torch_layer():
        m = torch.nn.ConvTranspose2d(cin, cout, k, stride=s, padding=p, output_padding=op).double()
        with torch.no_grad():
            m.weight.copy_(torch.tensor(wt))
            m.bias.copy_(torch.tensor(b.reshape(-1)))
        return m
    ty, tdx, tg = _tensor_grads(torch, torch_layer, x, gy)
    _close(y, ty, 1e-5)
    _close(dx, tdx, 1e-5)
    _close(layer.weight.grad.numpy(), tg["weight"], 1e-5)
    _close(layer.bias.grad.numpy().reshape(-1), tg["bias"], 1e-5)


@pytest.mark.parametrize("mode", ["nearest", "bilinear"])
@pytest.mark.parametrize("s,c", [(2, 4), (3, 3), (4, 5)])
def test_upsample_layer_on_numpy_device(ref_device, mode, s, c):
    torch = pytest.importorskip("torch")
    from DeepFlows import nn
    rng = np.random.RandomState(s * c)
    x = rng.randn(2, c, 3, 4)
    gy = rng.randn(2, c, 3 * s, 4 * s)
    y, dx = _run_layer(nn.Upsample(scale_factor=s, mode=mode), x, gy, ref_device)
    kw = {"align_corners": False} if mode == "bilinear" else {}
    ty, tdx, _ = _tensor_grads(torch, lambda: (lambda t: torch.nn.functional.interpolate(t, scale_factor=s, mode=mode, **kw)), x, gy)
    _close(y, ty, 1e-6)
    _close(dx, tdx, 1e-6)
    # `size` names the same layer
    y2, _ = _run_layer(nn.Upsample(size=(3 * s, 4 * s), mode=mode), x, gy, ref_device)
    assert np.array_equal(y, y2)


def test_output_size_formula():
    from DeepFlows.nn import functional as F
    for h, k, p, s, op in [(4, 4, 1, 2, 0), (5, 3, 1, 2, 1), (5, 3, 1, 2, 0), (7, 2, 0, 2, 0), (3, 3, 1, 3, 2), (6, 3, 1, 1, 0)]:
        ho = F.conv_transpose2d_size(h, k, p, s, op)
        assert ho == (h - 1) * s - 2 * p + k + op
        assert (ho + 2 * p - k) // s + 1 == h   # the convolution with the same geometry maps it back


def test_rejected_arguments(ref_device):
    from DeepFlows import nn
    from DeepFlows.nn import functional as F
    from DeepFlows.tensor import Tensor
    for s, op in [(1, 1), (2, 2), (2, 3), (3, -1)]:
        with pytest.raises(ValueError, match="output_padding"):
            nn.ConvTranspose2d(4, 4, 3, padding=1, stride=s, output_padding=op, device="cpu")
        with pytest.raises(ValueError, match="output_padding"):
            F.conv_transpose2d_size(4, 3, 1, s, op)
    x = Tensor(np.zeros((1, 2, 3, 3), F32), device=ref_device)
    for kw in [dict(scale_factor=1.5), dict(scale_factor=(2, 3)), dict(scale_factor=9), dict(scale_factor=0), dict(size=(7, 7)),
               dict(size=(6, 9)), dict(scale_factor=2, mode="bicubic"), dict(scale_factor=2, mode="bilinear", align_corners=True)]:
        with pytest.raises(NotImplementedError):
            F.interpolate(x, **kw)
    for kw in [dict(), dict(size=6, scale_factor=2), dict(scale_factor=2, mode="nearest", align_corners=False)]:
        with pytest.raises(ValueError):
            F.interpolate(x, **kw)
    with pytest.raises(NotImplementedError):
        nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)(x)
    assert F.interpolate(x, size=6).shape == F.interpolate(x, scale_factor=2.0).shape == (1, 2, 6, 6)
