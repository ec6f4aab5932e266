"""numpy restatement of the transpose of the correction path (test infrastructure, like oracle/).

The reference has no transpose, so this is not part of oracle/cpu_oracle.py, which restates reference code line for
line and is pinned to it.  It is built from the same steps as ``oracle.apply_transform``.
"""
from __future__ import annotations

import numpy as np
import scipy.fft

from oracle import cpu_oracle as oracle


def apply_transform_adjoint(grad, coordinates, kernel_values, pad_mode="symmetric"):
    """The transpose of ``apply_transform`` without saturation (not reference code: the reference has no adjoint).

    ``grad`` is an (H, W) frame of output gradients.  The same loop as ``apply_transform`` on the zero-extended frame,
    with the conjugate kernel (the transpose of ``Re ifft2(K fft2(.))``), then ``padᵀ``: every padded position is
    added onto the frame pixel ``np.pad`` copied it from, found by padding the index ranges themselves (constant mode:
    -1, dropped).  float64.
    """
    p0, p1 = kernel_values.shape[1], kernel_values.shape[2]
    h, w = grad.shape
    padded = np.zeros((h + 4 * p0, w + 4 * p1))
    padded[2 * p0:2 * p0 + h, 2 * p1:2 * p1 + w] = grad                   # zero_extend

    def window_of(corner):
        return (slice(corner[0] + 2 * p0, corner[0] + 3 * p0),
                slice(corner[1] + 2 * p1, corner[1] + 3 * p1))

    window = np.broadcast_to(oracle.apodization((p0, p1)), (len(coordinates), p0, p1))
    stack = np.stack([padded[window_of(c)[0], window_of(c)[1]] for c in coordinates])
    stack = scipy.fft.fft2(window * stack)
    stack = np.real(scipy.fft.ifft2(stack * np.conj(kernel_values)))
    stack = stack * window

    canvas = np.zeros_like(padded)
    for corner, patch in zip(coordinates, stack, strict=True):
        canvas[window_of(corner)[0], window_of(corner)[1]] += patch

    def source_index(n, p):
        extra = {"constant_values": -1} if pad_mode == "constant" else {}
        return np.pad(np.arange(n), (2 * p, 2 * p), mode=pad_mode, **extra)

    rows, cols = source_index(h, p0), source_index(w, p1)
    folded_rows = np.zeros((h, canvas.shape[1]))
    np.add.at(folded_rows, rows[rows >= 0], canvas[rows >= 0])
    out = np.zeros((h, w))
    np.add.at(out.T, cols[cols >= 0], folded_rows[:, cols >= 0].T)
    return out
