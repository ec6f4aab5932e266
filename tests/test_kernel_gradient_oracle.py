"""The numpy kernel gradient (tests/kernel_gradient_oracle.py) against the linearity of apply in the transfer kernel."""
import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from tests.helpers import load_golden
from tests.kernel_gradient_oracle import transfer_kernel_gradient

PAD_MODES = ["symmetric", "reflect", "edge", "wrap", "constant"]


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in oracle.covering(shape, size)]


def _irregular():
    g = load_golden("p16_irregular_coords")
    return g["image"].shape, int(g["size"]), [tuple(int(v) for v in c) for c in g["coords"]]


CASES = {
    "covering_64x48_p16": ((64, 48), 16, _covering((64, 48), 16)),
    "covering_odd_37x29_p8": ((37, 29), 8, _covering((37, 29), 8)),
    "frame_below_p_12x10_p16": ((12, 10), 16, _covering((12, 10), 16)),
    "irregular_64x64_p16": _irregular(),
}


def identity_error(shape, size, coords, pad_mode, batch, seed=0):
    """|sum_b <A_D x_b, g_b> - Re sum conj(grad) D| / (|A_D x| |g|) for a random complex cube D: apply is linear in K."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(len(coords), size, size)) + 1j * rng.normal(size=(len(coords), size, size))
    x, g = rng.normal(size=(batch,) + tuple(shape)), rng.normal(size=(batch,) + tuple(shape))
    ax = np.stack([oracle.apply_transform(f, coords, d, pad_mode=pad_mode) for f in x])
    grad = transfer_kernel_gradient(x, g, coords, size, pad_mode)
    assert grad.shape == d.shape and grad.dtype == np.complex128
    lhs = float(np.vdot(ax, g))
    rhs = float(np.real(np.sum(np.conj(grad) * d)))
    return abs(lhs - rhs) / (np.linalg.norm(ax) * np.linalg.norm(g))


@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_kernel_gradient_satisfies_linearity(case, pad_mode, batch):
    shape, size, coords = CASES[case]
    assert identity_error(shape, size, coords, pad_mode, batch) <= 1e-12


def test_oracle_kernel_gradient_is_hermitian_and_zero_off_the_frame():
    shape, size = (40, 36), 16
    coords = _covering(shape, size) + [(-20, 0), (0, 40)]            # two patches that never touch the frame
    rng = np.random.default_rng(4)
    grad = transfer_kernel_gradient(rng.normal(size=shape), rng.normal(size=shape), coords, size, "reflect")
    mirror = np.conj(np.roll(grad[:, ::-1, ::-1], 1, axis=(1, 2)))     # conj G[-k]
    np.testing.assert_allclose(grad, mirror, rtol=0, atol=1e-12 * np.abs(grad).max())
    assert not np.any(grad[-2:])


def test_transfer_kernel_gradient_rejects_unsupported_cases_without_a_gpu():
    t = rp.ArrayPSFTransform(rp.IndexedCube([(0, 0)], np.ones((1, 32, 32), dtype=np.complex64)))
    with pytest.raises(NotImplementedError):
        t.transfer_kernel_gradient(np.zeros((32, 32)), np.zeros((32, 32)), pad_mode="mean")
    embedded = rp.ArrayPSFTransform(rp.IndexedCube([(0, 0)], np.ones((1, 21, 21), dtype=np.complex64)))
    with pytest.raises(NotImplementedError):
        embedded.transfer_kernel_gradient(np.zeros((32, 32)), np.zeros((32, 32)))
