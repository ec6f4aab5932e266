"""The numpy masked apply, its transpose and its kernel gradient (tests/masked_apply_oracle.py), and the no-GPU
behaviour of apply(mask=)."""
import numpy as np
import pytest
from scipy.ndimage import binary_dilation

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from tests import masked_apply_oracle as mo

PAD_MODES = ["symmetric", "reflect", "edge", "wrap", "constant"]
SHAPE, SIZE = (64, 48), 16


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in oracle.covering(shape, size)]


def _masks(shape, seed=0):
    """Masks that touch the frame border, hold a run longer than 256 px (a whole column of a tall frame is built in
    test_long_runs) and a fully masked block whose inner windows hold masked pixels only."""
    rng = np.random.default_rng(seed)
    random = rng.random(shape) < 0.03
    border = np.zeros(shape, bool)
    border[0, :] = border[:, -1] = True
    border[5, 0] = True
    block = np.zeros(shape, bool)
    block[20:40, 10:30] = True
    return {"random": random, "border": border, "block": block}


def _kernel(n, size, seed=1):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(n, size, size)) + 1j * rng.normal(size=(n, size, size))


def dot_error(shape, size, mask, pad_mode, width, seed=2):
    coords = _covering(shape, size)
    kernel = _kernel(len(coords), size)
    rng = np.random.default_rng(seed)
    x, y = rng.normal(size=shape), rng.normal(size=shape)
    lx = mo.apply_masked_linear(x, coords, kernel, mask, pad_mode, width)
    lty = mo.apply_masked_adjoint(y, coords, kernel, mask, pad_mode, width)
    assert np.all(np.isfinite(lx)) and np.all(np.isfinite(lty))
    return abs(np.vdot(lx, y) - np.vdot(x, lty)) / (np.linalg.norm(lx) * np.linalg.norm(y))


def test_all_false_mask_reproduces_the_oracle():
    coords = _covering(SHAPE, SIZE)
    kernel = _kernel(len(coords), SIZE)
    x = oracle.starfield(SHAPE, seed=3).astype(float)
    for pad_mode in PAD_MODES:
        want = oracle.apply_transform(x, coords, kernel, pad_mode=pad_mode)
        got = mo.apply_masked(x, coords, kernel, np.zeros(SHAPE, bool), pad_mode)
        assert np.array_equal(want, got)


@pytest.mark.parametrize("dilation", [1, 2])
def test_the_dilated_saturation_mask_reproduces_the_saturation_oracle(dilation):
    coords = _covering(SHAPE, SIZE)
    kernel = _kernel(len(coords), SIZE)
    x = np.random.default_rng(4).normal(100.0, 5.0, SHAPE)
    x[[20, 21, 40, 12], [15, 15, 30, 33]] = 1e4
    threshold = 1e3
    want = oracle.apply_transform(x, coords, kernel, saturation_threshold=threshold, saturation_dilation=dilation)
    # masked pixels stay 2 * dilation px inside the frame, so that the padded masks agree
    sat = binary_dilation(x > threshold, iterations=dilation)
    assert not (sat[:4].any() or sat[-4:].any() or sat[:, :4].any() or sat[:, -4:].any())
    got = mo.apply_masked(x, coords, kernel, sat)
    assert np.array_equal(want, got)


def test_a_nan_under_the_mask_stays_at_its_pixel():
    coords = _covering(SHAPE, SIZE)
    kernel = _kernel(len(coords), SIZE)
    x = oracle.starfield(SHAPE, seed=5).astype(float)
    mask = np.zeros(SHAPE, bool)
    mask[30:34, 20:24] = True
    x[mask] = np.nan
    assert np.all(np.isnan(oracle.apply_transform(x, coords, kernel)[30:34, 20:24]))
    got = mo.apply_masked(x, coords, kernel, mask)
    assert np.array_equal(np.isnan(got), mask)
    x0 = np.where(mask, 0.0, x)
    np.testing.assert_allclose(got[~mask], mo.apply_masked_linear(x0, coords, kernel, mask)[~mask], rtol=0,
                               atol=1e-9 * np.abs(x0).max())


@pytest.mark.parametrize("width", [2, 7, 8])
@pytest.mark.parametrize("kind", ["random", "border", "block"])
def test_linear_map_is_the_masked_apply(kind, width):
    coords = _covering(SHAPE, SIZE)
    kernel = _kernel(len(coords), SIZE)
    x = np.random.default_rng(6).normal(size=SHAPE)
    mask = _masks(SHAPE)[kind]
    want = mo.apply_masked(x, coords, kernel, mask, neighborhood_width=width)
    got = mo.apply_masked_linear(x, coords, kernel, mask, neighborhood_width=width)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12 * np.abs(want).max())


@pytest.mark.parametrize("width", [0, 1, 2, 7, 8])
@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("kind", ["random", "border", "block"])
def test_oracle_masked_adjoint_is_the_transpose(kind, pad_mode, width):
    assert dot_error(SHAPE, SIZE, _masks(SHAPE)[kind], pad_mode, width) <= 1e-12


def test_long_runs_and_an_explicit_matrix():
    # a masked column longer than 256 px
    shape = (300, 24)
    mask = np.zeros(shape, bool)
    mask[:, 11] = True
    assert dot_error(shape, 8, mask, "symmetric", 7) <= 1e-12
    # tiny enough to build L_M column by column: L_Mᵀ must be its transpose entry for entry
    shape, size = (7, 6), 4
    coords = _covering(shape, size)
    kernel = _kernel(len(coords), size)
    mask = np.zeros(shape, bool)
    mask[0, 0] = mask[3, 2] = mask[3, 3] = mask[6, 5] = True
    basis = np.eye(shape[0] * shape[1]).reshape(-1, *shape)
    for pad_mode in PAD_MODES:
        a = np.stack([mo.apply_masked_linear(e, coords, kernel, mask, pad_mode, 3).ravel() for e in basis], 1)
        at = np.stack([mo.apply_masked_adjoint(e, coords, kernel, mask, pad_mode, 3).ravel() for e in basis], 1)
        np.testing.assert_allclose(at, a.T, rtol=0, atol=1e-13 * np.abs(a).max())


@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("batch", [1, 3])
def test_oracle_masked_kernel_gradient_satisfies_linearity(pad_mode, batch):
    coords = _covering(SHAPE, SIZE)
    rng = np.random.default_rng(7)
    d = _kernel(len(coords), SIZE, seed=8)
    x, g = rng.normal(size=(batch,) + SHAPE), rng.normal(size=(batch,) + SHAPE)
    masks = np.stack([_masks(SHAPE, seed=b)["random"] | _masks(SHAPE)["block"] for b in range(batch)])
    # the part of apply_masked_linear that depends on the kernel: the restored pixels do not
    lx = np.stack([mo.apply_masked_linear(f, coords, d, m, pad_mode) - np.where(m, f, 0.0)
                   for f, m in zip(x, masks, strict=True)])
    grad = mo.masked_kernel_gradient(x, g, coords, SIZE, masks, pad_mode)
    lhs = float(np.vdot(lx, g))
    rhs = float(np.real(np.sum(np.conj(grad) * d)))
    assert abs(lhs - rhs) / (np.linalg.norm(lx) * np.linalg.norm(g)) <= 1e-12


def test_masked_calls_reject_unsupported_cases_without_a_gpu():
    t = rp.ArrayPSFTransform(rp.IndexedCube([(0, 0)], np.ones((1, 32, 32), dtype=np.complex64)))
    mask = np.zeros((32, 32), bool)
    with pytest.raises(NotImplementedError):
        t.apply(np.zeros((32, 32)), pad_mode="mean", mask=mask)
    sharded = rp.ArrayPSFTransform.sharded(rp.IndexedCube([(0, 0)], np.ones((1, 32, 32), dtype=np.complex64)),
                                           [(0, 0), (0, 16)], [True, False])
    with pytest.raises(NotImplementedError):
        sharded.apply(np.zeros((32, 32)), mask=mask)
