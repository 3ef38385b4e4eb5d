"""The numpy device with the channel-concatenation entry points added (test infrastructure, like oracle/numpy_device.py,
which it extends without changing; the upsample functions of decoder_ref.py are there too, so the U-Net and the decoder
layers run on one device).

    concat_channels_fwd   y[:, off_i : off_i + widths[i]] = srcs[i]        (each a [rows, width] matrix, y [rows, C])
    concat_channels_bwd   dsrcs[i] = dy[:, off_i : off_i + widths[i]]      (None entries skipped)

The argument checks are the library's (include/dfb200.h: dfb_concat_channels_fwd / _bwd), so a host-side caller that
passes what the library would refuse fails here too.
"""
import types

import numpy as np

import decoder_ref
from oracle import numpy_device

MAX_SOURCES = 8


def _check(name, parts, widths, rows):
    if not 1 <= len(widths) <= MAX_SOURCES or len(parts) != len(widths):
        raise ValueError("%s: %d sources (1 to %d)" % (name, len(widths), MAX_SOURCES))
    if rows <= 0 or any(w <= 0 for w in widths) or sum(widths) >= 2 ** 31:
        raise ValueError("%s: bad geometry rows=%d widths=%s" % (name, rows, list(widths)))
    return np.cumsum([0] + list(widths)), int(sum(widths))


def concat_channels_fwd(srcs, widths, y, rows):
    off, c = _check("concat_channels_fwd", srcs, widths, rows)
    if any(s is None for s in srcs) or y is None:
        raise ValueError("concat_channels_fwd: null pointer")
    numpy_device._count("concat_channels_fwd")
    out = numpy_device._flat(y)[:rows * c].reshape(rows, c)
    for i, (s, w) in enumerate(zip(srcs, widths)):
        out[:, off[i]:off[i] + w] = numpy_device._flat(s)[:rows * w].reshape(rows, w)


def concat_channels_bwd(dy, dsrcs, widths, rows):
    off, c = _check("concat_channels_bwd", dsrcs, widths, rows)
    if dy is None:
        raise ValueError("concat_channels_bwd: null pointer")
    if all(d is None for d in dsrcs):
        return
    numpy_device._count("concat_channels_bwd")
    g = numpy_device._flat(dy)[:rows * c].reshape(rows, c)
    for i, (d, w) in enumerate(zip(dsrcs, widths)):
        if d is not None:
            numpy_device._flat(d)[:rows * w] = g[:, off[i]:off[i] + w].reshape(-1)


class _Device(types.ModuleType):
    """oracle.numpy_device plus the functions above and decoder_ref's upsample functions."""

    def __getattr__(self, name):
        return getattr(numpy_device, name)


device = _Device("concat_numpy_device")
device.upsample2d_fwd = decoder_ref.upsample2d_fwd
device.upsample2d_bwd = decoder_ref.upsample2d_bwd
device.concat_channels_fwd = concat_channels_fwd
device.concat_channels_bwd = concat_channels_bwd
