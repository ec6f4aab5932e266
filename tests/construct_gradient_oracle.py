"""numpy restatement of the gradient of ``ArrayPSFTransform.construct`` and of the PSF FFT cube (test infrastructure).

The reference has no gradient, so this is not part of oracle/cpu_oracle.py, which restates reference code line for line
and is pinned to it.  It evaluates the closed forms of DESIGN.md section 6 literally, in float64, and then applies the
special-bin policy:

- a bin with G = 0 contributes exact zeros to all four outputs;
- where K is finite and G != 0, the terms that are 0 * inf in the closed form (at |S| = 0, |T| = 0 or eps |T| = 0) take
  their limit, 0;
- where K is not finite and G != 0, the bin's source and target gradients are NaN, and so are grad_alpha and grad_eps.

Gradients use PyTorch's convention for complex numbers: dL/dRe + i dL/dIm.
"""
from __future__ import annotations

import numpy as np
import scipy.fft

from oracle import cpu_oracle as oracle


def construct_vjp(source_fft, target_fft, kernel_grad, alpha, epsilon):
    """(grad_source, grad_target, grad_alpha, grad_epsilon) of ``<K, G>`` for K = transfer_kernel(S, T, alpha, epsilon).

    ``source_fft``, ``target_fft`` and ``kernel_grad`` are complex arrays of one shape; the cubes come back complex128
    and the two scalars as Python floats.
    """
    s = np.asarray(source_fft, dtype=np.complex128)
    t = np.asarray(target_fft, dtype=np.complex128)
    g = np.asarray(kernel_grad, dtype=np.complex128)
    alpha, epsilon = float(alpha), float(epsilon)
    with np.errstate(all="ignore"):
        k = oracle.transfer_kernel(s, t, alpha, epsilon)
        a, b = np.abs(s), np.abs(t)
        c = epsilon * b
        p = alpha + 1
        d = a ** p + c ** p
        f = a ** (alpha - 1) / d
        w = np.real(g * s * np.conj(t))
        s_term = w * a ** (alpha - 3) * ((alpha - 1) * c ** p - 2 * a ** p) / d ** 2 * s
        t_term = w * (alpha + 1) * epsilon ** p * a ** (alpha - 1) * b ** (alpha - 1) / d ** 2 * t
        alpha_term = w * a ** (alpha - 1) * c ** p * np.log(a / c) / d ** 2
        eps_term = -w * (alpha + 1) * epsilon ** alpha * a ** (alpha - 1) * b ** p / d ** 2
        # limits of the 0 * inf products where K is finite
        s_term = np.where(a == 0, 0, s_term)
        t_term = np.where(b == 0, 0, t_term)
        alpha_term = np.where((a == 0) | (c == 0), 0, alpha_term)
        eps_term = np.where((a == 0) | (epsilon == 0), 0, eps_term)
        grad_s = f * np.conj(g) * t + s_term
        grad_t = f * g * s - t_term
    zero = (g == 0)
    bad = ~zero & ~np.isfinite(k)
    nan = complex(np.nan, np.nan)
    grad_s = np.where(zero, 0, np.where(bad, nan, grad_s))
    grad_t = np.where(zero, 0, np.where(bad, nan, grad_t))
    alpha_term = np.where(zero, 0, np.where(bad, np.nan, alpha_term))
    eps_term = np.where(zero, 0, np.where(bad, np.nan, eps_term))
    return grad_s, grad_t, float(np.sum(alpha_term)), float(np.sum(eps_term))


def psf_fft_vjp(spectrum_grad):
    """The gradient of ``<psf_fft(x), G>`` with respect to the real (N, P, P) values x: Re(fft2(conj(G)))."""
    return np.real(scipy.fft.fft2(np.conj(np.asarray(spectrum_grad, dtype=np.complex128))))
