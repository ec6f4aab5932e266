"""numpy restatement of the gradient of the correction path with respect to the transfer kernel (test infrastructure).

The reference has no gradient, so this is not part of oracle/cpu_oracle.py, which restates reference code line for line
and is pinned to it.  It is built from the same steps as ``oracle.apply_transform``.
"""
from __future__ import annotations

import numpy as np
import scipy.fft

from oracle import cpu_oracle as oracle


def transfer_kernel_gradient(image, grad, coordinates, size, pad_mode="symmetric"):
    """d<apply_transform(image), grad>/dK in PyTorch's convention (dL/dRe + i dL/dIm), without saturation.

    ``image`` and ``grad`` are (H, W) or (B, H, W); the result is the (N, size, size) complex128 sum over the frames of
    ``conj(X) * G / size**2`` per patch, with X the FFT2 of the apodized patch of the padded image (the stack
    ``apply_transform`` transforms) and G that of the zero-extended ``grad``.  Patches that do not touch the frame get
    an exact 0: no output pixel depends on their kernel.
    """
    image, grad = np.asarray(image, dtype=float), np.asarray(grad, dtype=float)
    if image.ndim == 2:
        image, grad = image[np.newaxis], grad[np.newaxis]
    p0 = p1 = size
    h, w = image.shape[1:]

    def window_of(corner):
        return (slice(corner[0] + 2 * p0, corner[0] + 3 * p0),
                slice(corner[1] + 2 * p1, corner[1] + 3 * p1))

    window = np.broadcast_to(oracle.apodization((p0, p1)), (len(coordinates), p0, p1))
    out = np.zeros((len(coordinates), p0, p1), dtype=np.complex128)
    for frame, g in zip(image, grad, strict=True):
        padded = np.pad(frame, ((2 * p0, 2 * p0), (2 * p1, 2 * p1)), mode=pad_mode)
        extended = np.zeros_like(padded)
        extended[2 * p0:2 * p0 + h, 2 * p1:2 * p1 + w] = g
        xs = scipy.fft.fft2(window * np.stack([padded[window_of(c)] for c in coordinates]))
        gs = scipy.fft.fft2(window * np.stack([extended[window_of(c)] for c in coordinates]))
        out += np.conj(xs) * gs / (p0 * p1)
    for i, c in enumerate(coordinates):
        if max(c[0], 0) >= min(c[0] + p0, h) or max(c[1], 0) >= min(c[1] + p1, w):
            out[i] = 0
    return out
