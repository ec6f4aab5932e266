"""The numpy construct / PSF-FFT gradients (tests/construct_gradient_oracle.py) against finite differences of the
reference-pinned ``oracle.transfer_kernel`` and ``oracle.psf_fft``."""
import numpy as np
import pytest

from oracle import cpu_oracle as oracle
from tests.construct_gradient_oracle import construct_vjp, psf_fft_vjp


def _loss(s, t, g, alpha, epsilon):
    """<K, G> = Re sum conj(G) K: its gradient with respect to K is G in PyTorch's convention."""
    return float(np.sum(np.real(np.conj(g) * oracle.transfer_kernel(s, t, alpha, epsilon))))


def _complex(rng, n):
    return rng.normal(size=n) + 1j * rng.normal(size=n)


def _fd_cube(s, t, g, alpha, epsilon, which, index, h, one_sided=False):
    """d loss / d Re + i d loss / d Im of element `index` of S (which = 0) or T (which = 1)."""
    out = []
    for unit in (1.0, 1j):
        def at(step):
            args = [s.copy(), t.copy()]
            args[which][index] += unit * step
            return _loss(args[0], args[1], g, alpha, epsilon)
        out.append((at(h) - at(0.0)) / h if one_sided else (at(h) - at(-h)) / (2 * h))
    return complex(out[0], out[1])


@pytest.mark.parametrize("epsilon", [0.05, 0.2, 1.0])
@pytest.mark.parametrize("alpha", [0.5, 1.0, 1.5, 2.0, 3.0])
def test_construct_vjp_matches_central_differences(alpha, epsilon):
    rng = np.random.default_rng(int(alpha * 10) + int(epsilon * 100))
    n = 16
    s, t, g = _complex(rng, n), _complex(rng, n), _complex(rng, n)
    grad_s, grad_t, grad_a, grad_e = construct_vjp(s, t, g, alpha, epsilon)
    h = 1e-6
    fd_s = np.array([_fd_cube(s, t, g, alpha, epsilon, 0, i, h) for i in range(n)])
    fd_t = np.array([_fd_cube(s, t, g, alpha, epsilon, 1, i, h) for i in range(n)])
    fd_a = (_loss(s, t, g, alpha + h, epsilon) - _loss(s, t, g, alpha - h, epsilon)) / (2 * h)
    fd_e = (_loss(s, t, g, alpha, epsilon + h) - _loss(s, t, g, alpha, epsilon - h)) / (2 * h)
    scale = max(np.abs(grad_s).max(), np.abs(grad_t).max(), abs(grad_a), abs(grad_e))
    np.testing.assert_allclose(grad_s, fd_s, rtol=0, atol=1e-7 * scale)
    np.testing.assert_allclose(grad_t, fd_t, rtol=0, atol=1e-7 * scale)
    assert abs(grad_a - fd_a) <= 1e-7 * scale
    assert abs(grad_e - fd_e) <= 1e-7 * scale


@pytest.mark.parametrize("alpha", [1.0, 1.5])
def test_source_zero_bin_takes_the_limit(alpha):
    """S = 0 where K is finite (alpha >= 1): the second term of grad_S and the grad_alpha term vanish."""
    rng = np.random.default_rng(3)
    n = 6
    s, t, g = _complex(rng, n), _complex(rng, n), _complex(rng, n)
    s[2] = 0
    epsilon = 0.3
    grad_s, grad_t, grad_a, grad_e = construct_vjp(s, t, g, alpha, epsilon)
    assert np.all(np.isfinite(grad_s)) and np.all(np.isfinite(grad_t)) and np.isfinite(grad_a) and np.isfinite(grad_e)
    c = epsilon * abs(t[2])
    if alpha == 1.0:
        assert grad_s[2] == pytest.approx(np.conj(g[2]) * t[2] / c ** 2, rel=1e-14)
    else:
        assert grad_s[2] == 0
    # one-sided differences on that bin alone (the loss of the others would drown the step in rounding); for alpha > 1
    # the quotient falls like h^(alpha - 1)
    one = slice(2, 3)
    for h in (1e-8, 1e-12):
        fd = _fd_cube(s[one], t[one], g[one], alpha, epsilon, 0, 0, h, one_sided=True)
        bound = 1e-6 * abs(grad_s[2]) if alpha == 1.0 else 10 * h ** (alpha - 1) * abs(g[2] * t[2]) / c ** (alpha + 1)
        assert abs(fd - grad_s[2]) <= bound, (h, fd, grad_s[2])
    # the other derivatives at the same point still match central differences
    h = 1e-6
    fd_t = _fd_cube(s, t, g, alpha, epsilon, 1, 2, h)
    assert abs(fd_t - grad_t[2]) <= 1e-7 * np.abs(grad_t).max()
    # below alpha = 1 the S = 0 bin is 0/0: a one-sided difference in alpha
    fd_a = (_loss(s, t, g, alpha + h, epsilon) - _loss(s, t, g, alpha, epsilon)) / h
    fd_e = (_loss(s, t, g, alpha, epsilon + h) - _loss(s, t, g, alpha, epsilon - h)) / (2 * h)
    assert abs(fd_a - grad_a) <= 1e-5 * max(1.0, abs(grad_a))
    assert abs(fd_e - grad_e) <= 1e-7 * max(1.0, abs(grad_e))


@pytest.mark.parametrize("alpha", [0.5, 1.0, 2.0])
def test_target_zero_bin_takes_the_limit(alpha):
    rng = np.random.default_rng(5)
    n = 6
    s, t, g = _complex(rng, n), _complex(rng, n), _complex(rng, n)
    t[4] = 0
    grad_s, grad_t, grad_a, grad_e = construct_vjp(s, t, g, alpha, 0.2)
    assert np.all(np.isfinite(grad_t)) and np.isfinite(grad_a) and np.isfinite(grad_e)
    assert grad_s[4] == 0                                           # K = 0 for every S there
    fd = _fd_cube(s, t, g, alpha, 0.2, 1, 4, 1e-8, one_sided=True)
    assert abs(fd - grad_t[4]) <= 1e-6 * np.abs(grad_t).max()


@pytest.mark.parametrize("alpha", [1.0, 1.5, 2.0])
def test_epsilon_zero_takes_the_limit(alpha):
    rng = np.random.default_rng(7)
    n = 8
    s, t, g = _complex(rng, n), _complex(rng, n), _complex(rng, n)
    grad_s, grad_t, grad_a, grad_e = construct_vjp(s, t, g, alpha, 0.0)
    assert grad_a == 0 and grad_e == 0                              # K = conj(S) T / |S|^2: no alpha, no epsilon
    h = 1e-9
    fd_e = (_loss(s, t, g, alpha, h) - _loss(s, t, g, alpha, 0.0)) / h
    assert abs(fd_e) <= 1e-4 * np.abs(grad_s).max()
    h = 1e-6
    fd_s = np.array([_fd_cube(s, t, g, alpha, 0.0, 0, i, h) for i in range(n)])
    fd_t = np.array([_fd_cube(s, t, g, alpha, 0.0, 1, i, h) for i in range(n)])
    np.testing.assert_allclose(grad_s, fd_s, rtol=0, atol=1e-7 * np.abs(grad_s).max())
    np.testing.assert_allclose(grad_t, fd_t, rtol=0, atol=1e-7 * np.abs(grad_t).max())


def test_zero_gradient_bins_give_exact_zeros_and_nonfinite_kernel_bins_give_nan():
    s = np.array([0, 0, 1 + 1j, np.nan, 2 - 1j, 0], dtype=np.complex128)
    t = np.array([0, 1j, np.inf, 1, 1 + 0.5j, 0], dtype=np.complex128)
    g = np.array([0, 0, 0, 0, 1 - 2j, 1 + 1j], dtype=np.complex128)
    k = oracle.transfer_kernel(s, t, 1.0, 0.2)
    assert not np.isfinite(k[0]) and not np.isfinite(k[5])           # 0/0 at S = T = 0
    grad_s, grad_t, grad_a, grad_e = construct_vjp(s, t, g, 1.0, 0.2)
    assert np.all(grad_s[:4] == 0) and np.all(grad_t[:4] == 0)     # G = 0: exact zeros, whatever S and T hold
    assert np.isfinite(grad_s[4]) and np.isfinite(grad_t[4])
    assert np.isnan(grad_s[5].real) and np.isnan(grad_s[5].imag) and np.isnan(grad_t[5].real)
    assert np.isnan(grad_a) and np.isnan(grad_e)
    # without the non-finite bin, the sums are finite: the G = 0 bins cannot poison them
    _, _, grad_a, grad_e = construct_vjp(s[:5], t[:5], g[:5], 1.0, 0.2)
    assert np.isfinite(grad_a) and np.isfinite(grad_e)


def test_source_zero_below_alpha_one_is_a_nonfinite_kernel_bin():
    s = np.array([0, 1 + 1j], dtype=np.complex128)
    t = np.array([1 + 1j, 1], dtype=np.complex128)
    g = np.ones(2, dtype=np.complex128)
    assert np.isnan(oracle.transfer_kernel(s, t, 0.5, 0.2)[0])
    grad_s, grad_t, grad_a, _ = construct_vjp(s, t, g, 0.5, 0.2)
    assert np.isnan(grad_s[0]) and np.isnan(grad_t[0]) and np.isnan(grad_a)
    assert np.isfinite(grad_s[1])


@pytest.mark.parametrize("size", [16, 21])
def test_psf_fft_vjp_matches_differences_and_the_inner_product_identity(size):
    rng = np.random.default_rng(size)
    x = rng.normal(size=(2, size, size))
    g = rng.normal(size=(2, size, size)) + 1j * rng.normal(size=(2, size, size))
    vjp = psf_fft_vjp(g)
    assert vjp.dtype == np.float64 and vjp.shape == x.shape
    lhs = float(np.real(np.vdot(g, oracle.psf_fft(x))))            # <fft2 x, G> = Re sum conj(G) fft2(x)
    assert lhs == pytest.approx(float(np.sum(x * vjp)), rel=1e-12)
    h = 1e-6
    for index in [(0, 0, 0), (1, 3, 7), (0, size - 1, 2)]:
        e = np.zeros_like(x)
        e[index] = h
        fd = (np.real(np.vdot(g, oracle.psf_fft(x + e))) - np.real(np.vdot(g, oracle.psf_fft(x - e)))) / (2 * h)
        assert fd == pytest.approx(vjp[index], abs=1e-7 * np.abs(vjp).max())
