"""numpy restatement of apply with a caller-given bad-pixel mask, its transpose and its kernel gradient (test
infrastructure, like oracle/).

The reference has no mask argument, so this is not part of oracle/cpu_oracle.py, which restates reference code line for
line and is pinned to it.  ``apply_masked`` is built from the steps of ``oracle.apply_transform``: the caller's mask,
padded like the image (``constant``: an unmasked margin), is ORed into the dilated saturation mask and the saturation
branch runs unchanged.  With an infinite threshold the map is linear in the image for images that are finite outside the
mask; ``apply_masked_linear`` is that map with the fill's contributors decided by the mask alone, and
``apply_masked_adjoint`` its explicit transpose (the fill run backwards).
"""
from __future__ import annotations

import math
import warnings

import numpy as np
import scipy.fft
from scipy.ndimage import binary_dilation

from oracle import cpu_oracle as oracle


def pad_mask(mask, size, pad_mode):
    """The caller's (H, W) mask padded by 2 * size per side with the image's pad mode (``constant``: unmasked)."""
    return np.pad(np.asarray(mask, dtype=bool), 2 * size, mode=pad_mode)


def _window(i, j, half):
    return slice(i - half, i + half), slice(j - half, j + half)


def _patch_canvas(padded, coordinates, kernel_values):
    """The patch path of ``oracle.apply_transform`` (transform.py:141-169) on a padded frame: the canvas before the
    restore and the crop."""
    p0, p1 = kernel_values.shape[1], kernel_values.shape[2]

    def window_of(corner):
        return (slice(corner[0] + 2 * p0, corner[0] + 3 * p0),
                slice(corner[1] + 2 * p1, corner[1] + 3 * p1))

    window = np.broadcast_to(oracle.apodization((p0, p1)), (len(coordinates), p0, p1))
    stack = np.stack([padded[window_of(c)[0], window_of(c)[1]] for c in coordinates])
    stack = scipy.fft.fft2(window * stack)
    stack = np.real(scipy.fft.ifft2(stack * kernel_values))
    stack = stack * window
    canvas = np.zeros_like(padded)
    for corner, patch in zip(coordinates, stack, strict=True):
        canvas[window_of(corner)[0], window_of(corner)[1]] += patch
    return canvas


def apply_masked(image, coordinates, kernel_values, mask, pad_mode="symmetric", saturation_threshold=math.inf,
                 saturation_dilation=1, neighborhood_width=7):
    """``apply(image, mask=mask, ...)`` for one (H, W) frame, float64: transform.py:116-177 with the padded caller's
    mask ORed into the dilated saturation mask (it is not dilated itself)."""
    p0, p1 = kernel_values.shape[1], kernel_values.shape[2]
    frame = image.copy().astype(float)
    padded = np.pad(frame, ((2 * p0, 2 * p0), (2 * p1, 2 * p1)), mode=pad_mode)
    raw = padded.copy()
    full = padded > saturation_threshold
    if np.any(full):
        full = binary_dilation(full, iterations=saturation_dilation)
    full = full | pad_mask(mask, p0, pad_mode)
    if np.any(full):
        padded[full] = np.nan
        half = neighborhood_width // 2
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)          # nanmean of an empty or all-NaN window: NaN
            for i, j in zip(*np.where(full)):
                padded[i, j] = np.nanmean(padded[_window(i, j, half)])
    canvas = _patch_canvas(padded, coordinates, kernel_values)
    canvas[full] = raw[full]
    return canvas[2 * p0:frame.shape[0] + 2 * p0, 2 * p1:frame.shape[1] + 2 * p1]


def fill_counts(full, half):
    """Contributor count of every masked pixel of the padded mask ``full`` when the unmasked pixels are finite (0: a
    structural NaN, a pixel whose window holds no unmasked pixel and no earlier fill that is finite)."""
    counts = np.zeros(full.shape, dtype=np.int64)
    finite = ~full
    for i, j in zip(*np.where(full)):
        n = 0 if half <= 0 or i < half or j < half else int(finite[_window(i, j, half)].sum())
        counts[i, j] = n
        finite[i, j] = n > 0
    return counts


def fill_linear(padded, full, counts, half):
    """F_M: the raster-ordered fill as a linear map (a structural NaN reads as 0 and contributes nothing)."""
    out = padded.astype(float).copy()
    out[full] = 0.0
    valid = ~full
    for i, j in zip(*np.where(full)):
        if counts[i, j]:
            w = _window(i, j, half)
            out[i, j] = out[w][valid[w]].sum() / counts[i, j]
            valid[i, j] = True
    return out


def fill_adjoint(v, full, counts, half):
    """F_Mᵀ, the fill run backwards: every masked pixel, last first, passes its accumulated gradient divided by its
    count to each contributor of its window.  Masked pixels come back 0 (the fill ignores their input)."""
    acc = v.astype(float).copy()
    out = acc.copy()
    out[full] = 0.0
    wp = full.shape[1]
    rows, cols = np.where(full)
    for i, j in zip(rows[::-1], cols[::-1]):
        if not counts[i, j]:
            continue
        share = acc[i, j] / counts[i, j]
        w = _window(i, j, half)
        rr, cc = np.meshgrid(np.arange(full.shape[0])[w[0]], np.arange(wp)[w[1]], indexing="ij")
        earlier = rr * wp + cc < i * wp + j
        out[w] += share * ~full[w]
        acc[w] += share * (full[w] & earlier & (counts[w] > 0))
    return out


def apply_masked_linear(image, coordinates, kernel_values, mask, pad_mode="symmetric", neighborhood_width=7):
    """L_M x = crop(pad(M) pad(x) + (1 - pad(M)) A_K(F_M pad(x))): ``apply_masked`` with an infinite threshold, for a
    frame finite outside the mask and without structural NaNs."""
    p = kernel_values.shape[1]
    h, w = image.shape
    padded = np.pad(np.asarray(image, dtype=float), 2 * p, mode=pad_mode)
    full = pad_mask(mask, p, pad_mode)
    half = neighborhood_width // 2
    canvas = _patch_canvas(fill_linear(padded, full, fill_counts(full, half), half), coordinates, kernel_values)
    canvas[full] = padded[full]
    return canvas[2 * p:2 * p + h, 2 * p:2 * p + w]


def apply_masked_adjoint(grad, coordinates, kernel_values, mask, pad_mode="symmetric", neighborhood_width=7):
    """L_Mᵀ g = padᵀ(pad(M) g_ext + (1 - pad(M)) F_Mᵀ A_Kᵀ((1 - M) g)), g_ext the zero-extended ``grad``."""
    p = kernel_values.shape[1]
    h, w = grad.shape
    full = pad_mask(mask, p, pad_mode)
    half = neighborhood_width // 2
    extended = np.zeros(full.shape)
    extended[2 * p:2 * p + h, 2 * p:2 * p + w] = grad
    kept = np.where(full, 0.0, extended)
    v = _patch_canvas(kept, coordinates, np.conj(kernel_values))
    combined = np.where(full, extended, fill_adjoint(v, full, fill_counts(full, half), half))

    def source_index(n):
        extra = {"constant_values": -1} if pad_mode == "constant" else {}
        return np.pad(np.arange(n), (2 * p, 2 * p), mode=pad_mode, **extra)

    rows, cols = source_index(h), source_index(w)
    folded_rows = np.zeros((h, combined.shape[1]))
    np.add.at(folded_rows, rows[rows >= 0], combined[rows >= 0])
    out = np.zeros((h, w))
    np.add.at(out.T, cols[cols >= 0], folded_rows[:, cols >= 0].T)
    return out


def masked_kernel_gradient(image, grad, coordinates, size, mask, pad_mode="symmetric", neighborhood_width=7):
    """d<apply_masked_linear(image), grad>/dK (PyTorch's convention), summed over the frames: conj(X) G / size**2 per
    patch with X the FFT2 of the apodized patch of F_M pad(image) and G that of the zero-extended (1 - M) grad.
    ``mask`` is (H, W) or (B, H, W).  Patches that do not touch the frame get 0."""
    image, grad = np.asarray(image, dtype=float), np.asarray(grad, dtype=float)
    if image.ndim == 2:
        image, grad = image[np.newaxis], grad[np.newaxis]
    masks = np.broadcast_to(np.asarray(mask, dtype=bool), image.shape)
    p = size
    h, w = image.shape[1:]
    half = neighborhood_width // 2

    def window_of(corner):
        return slice(corner[0] + 2 * p, corner[0] + 3 * p), slice(corner[1] + 2 * p, corner[1] + 3 * p)

    window = np.broadcast_to(oracle.apodization((p, p)), (len(coordinates), p, p))
    out = np.zeros((len(coordinates), p, p), dtype=np.complex128)
    for frame, g, m in zip(image, grad, masks, strict=True):
        full = pad_mask(m, p, pad_mode)
        filled = fill_linear(np.pad(frame, 2 * p, mode=pad_mode), full, fill_counts(full, half), half)
        extended = np.zeros_like(filled)
        extended[2 * p:2 * p + h, 2 * p:2 * p + w] = np.where(m, 0.0, g)
        xs = scipy.fft.fft2(window * np.stack([filled[window_of(c)] for c in coordinates]))
        gs = scipy.fft.fft2(window * np.stack([extended[window_of(c)] for c in coordinates]))
        out += np.conj(xs) * gs / (p * p)
    for i, c in enumerate(coordinates):
        if max(c[0], 0) >= min(c[0] + p, h) or max(c[1], 0) >= min(c[1] + p, w):
            out[i] = 0
    return out
