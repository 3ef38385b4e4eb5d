"""Float64 references for the decoder layers, written as their direct definitions, and the numpy device with the upsample
entry points added (test infrastructure, like oracle/numpy_device.py, which it extends without changing).

    conv_transpose2d   y[n, o, ih*s - p + a, iw*s - p + b] += x[n, i, ih, iw] * w[i, o, a, b]   (scatter form)
    upsample nearest   y[oh, ow] = x[oh // s, ow // s]
    upsample bilinear  align_corners=False: src = max(0, (o + 0.5)/s - 0.5), i0 = floor(src), i1 = min(i0 + 1, n - 1),
                       weights 1 - (src - i0) and src - i0 per axis; the backward scatters dy with the same weights
"""
import types

import numpy as np

from oracle import numpy_device

NEAREST, BILINEAR = 0, 1


def conv_transpose2d(x, w, padding, stride, output_padding):
    x, w = np.asarray(x, np.float64), np.asarray(w, np.float64)
    n, cin, hi, wi = x.shape
    cin2, cout, k, k2 = w.shape
    assert cin == cin2 and k == k2
    s, p = stride, padding
    ho, wo = (hi - 1) * s - 2 * p + k + output_padding, (wi - 1) * s - 2 * p + k + output_padding
    full = np.zeros((n, cout, (hi - 1) * s + k + output_padding, (wi - 1) * s + k + output_padding))
    for a in range(k):
        for b in range(k):
            full[:, :, a:a + (hi - 1) * s + 1:s, b:b + (wi - 1) * s + 1:s] += np.einsum("nihw,io->nohw", x, w[:, :, a, b])
    return full[:, :, p:p + ho, p:p + wo]


def _lerp(n_out, n_in, s):
    """(i0, i1, l0, l1) arrays over the output indices of one axis."""
    src = np.maximum(0.0, (np.arange(n_out) + 0.5) / s - 0.5)
    i0 = np.floor(src).astype(np.int64)
    i1 = np.minimum(i0 + 1, n_in - 1)
    l1 = src - i0
    return i0, i1, 1.0 - l1, l1


def upsample_nearest_fwd(x, s):
    x = np.asarray(x, np.float64)
    n, c, h, w = x.shape
    y = np.zeros((n, c, h * s, w * s))
    for oh in range(h * s):
        for ow in range(w * s):
            y[:, :, oh, ow] = x[:, :, oh // s, ow // s]
    return y


def upsample_nearest_bwd(dy, s):
    dy = np.asarray(dy, np.float64)
    n, c, oh_, ow_ = dy.shape
    dx = np.zeros((n, c, oh_ // s, ow_ // s))
    for oh in range(oh_):
        for ow in range(ow_):
            dx[:, :, oh // s, ow // s] += dy[:, :, oh, ow]
    return dx


def upsample_bilinear_fwd(x, s):
    x = np.asarray(x, np.float64)
    n, c, h, w = x.shape
    ri0, ri1, rl0, rl1 = _lerp(h * s, h, s)
    ci0, ci1, cl0, cl1 = _lerp(w * s, w, s)
    y = np.zeros((n, c, h * s, w * s))
    for oh in range(h * s):
        for ow in range(w * s):
            y[:, :, oh, ow] = (rl0[oh] * (cl0[ow] * x[:, :, ri0[oh], ci0[ow]] + cl1[ow] * x[:, :, ri0[oh], ci1[ow]])
                               + rl1[oh] * (cl0[ow] * x[:, :, ri1[oh], ci0[ow]] + cl1[ow] * x[:, :, ri1[oh], ci1[ow]]))
    return y


def upsample_bilinear_bwd(dy, s):
    dy = np.asarray(dy, np.float64)
    n, c, oh_, ow_ = dy.shape
    h, w = oh_ // s, ow_ // s
    ri0, ri1, rl0, rl1 = _lerp(oh_, h, s)
    ci0, ci1, cl0, cl1 = _lerp(ow_, w, s)
    dx = np.zeros((n, c, h, w))
    for oh in range(oh_):
        for ow in range(ow_):
            g = dy[:, :, oh, ow]
            dx[:, :, ri0[oh], ci0[ow]] += rl0[oh] * cl0[ow] * g
            dx[:, :, ri0[oh], ci1[ow]] += rl0[oh] * cl1[ow] * g
            dx[:, :, ri1[oh], ci0[ow]] += rl1[oh] * cl0[ow] * g
            dx[:, :, ri1[oh], ci1[ow]] += rl1[oh] * cl1[ow] * g
    return dx


# ---- the numpy device's dfb_upsample2d_fwd / _bwd (include/dfb200.h) ---------------------------------------------------
def upsample2d_fwd(x, y, N, H, W, C, scale, mode):
    fn = upsample_nearest_fwd if mode == NEAREST else upsample_bilinear_fwd
    out = fn(numpy_device._nchw(numpy_device._flat(x), N, C, H, W), scale).astype(np.float32)
    numpy_device._store_nhwc(numpy_device._flat(y), out)


def upsample2d_bwd(dy, dx, N, H, W, C, scale, mode):
    fn = upsample_nearest_bwd if mode == NEAREST else upsample_bilinear_bwd
    out = fn(numpy_device._nchw(numpy_device._flat(dy), N, C, H * scale, W * scale), scale).astype(np.float32)
    numpy_device._store_nhwc(numpy_device._flat(dx), out)


class _Device(types.ModuleType):
    """oracle.numpy_device plus the two functions above."""

    def __getattr__(self, name):
        return getattr(numpy_device, name)


device = _Device("decoder_numpy_device")
device.upsample2d_fwd = upsample2d_fwd
device.upsample2d_bwd = upsample2d_bwd
