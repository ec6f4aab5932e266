"""The numpy transpose of apply (tests/adjoint_oracle.py) and the no-GPU behaviour of apply_adjoint."""
import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from tests.adjoint_oracle import apply_transform_adjoint
from regularizepsf_b200.exceptions import NativeLibraryError
from tests.helpers import load_golden

PAD_MODES = ["symmetric", "reflect", "edge", "wrap", "constant"]


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in oracle.covering(shape, size)]


def _irregular():
    g = load_golden("p16_irregular_coords")
    return g["image"].shape, g["size"], g["coords"]


CASES = {
    "covering_64x48_p16": ((64, 48), 16, _covering((64, 48), 16)),
    "covering_odd_37x29_p8": ((37, 29), 8, _covering((37, 29), 8)),
    "frame_below_p_12x10_p16": ((12, 10), 16, _covering((12, 10), 16)),
    "irregular_64x64_p16": _irregular(),
    "covering_p12_50x40": ((50, 40), 12, _covering((50, 40), 12)),
}


def dot_identity_error(shape, size, coords, pad_mode, seed=0):
    """|<A x, y> - <x, Aᵀ y>| / (|A x| |y|) for a random, non-Hermitian complex kernel cube."""
    rng = np.random.default_rng(seed)
    kernel = rng.normal(size=(len(coords), size, size)) + 1j * rng.normal(size=(len(coords), size, size))
    x, y = rng.normal(size=shape), rng.normal(size=shape)
    ax = oracle.apply_transform(x, coords, kernel, pad_mode=pad_mode)
    aty = apply_transform_adjoint(y, coords, kernel, pad_mode)
    assert aty.shape == shape and aty.dtype == np.float64
    return abs(np.vdot(ax, y) - np.vdot(x, aty)) / (np.linalg.norm(ax) * np.linalg.norm(y))


@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_adjoint_is_the_transpose(case, pad_mode):
    shape, size, coords = CASES[case]
    assert dot_identity_error(shape, size, coords, pad_mode) <= 1e-12


def test_oracle_adjoint_fold_matches_explicit_matrix():
    # tiny enough to build A column by column: Aᵀ must be its transpose entry for entry
    shape, size = (6, 5), 4
    coords = _covering(shape, size)
    kernel = np.random.default_rng(3).normal(size=(len(coords), size, size)) * (1 + 0.5j)
    for pad_mode in PAD_MODES:
        basis = np.eye(shape[0] * shape[1]).reshape(-1, *shape)
        a = np.stack([oracle.apply_transform(e, coords, kernel, pad_mode=pad_mode).ravel() for e in basis], 1)
        at = np.stack([apply_transform_adjoint(e, coords, kernel, pad_mode).ravel() for e in basis], 1)
        np.testing.assert_allclose(at, a.T, rtol=0, atol=1e-13 * np.abs(a).max())


def test_apply_adjoint_has_no_cpu_fallback_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    t = rp.ArrayPSFTransform(rp.IndexedCube([(0, 0)], np.ones((1, 32, 32), dtype=np.complex64)))
    with pytest.raises(NativeLibraryError):
        t.apply_adjoint(np.zeros((32, 32)))


def test_apply_adjoint_rejects_pad_modes_without_an_index_map():
    t = rp.ArrayPSFTransform(rp.IndexedCube([(0, 0)], np.ones((1, 32, 32), dtype=np.complex64)))
    with pytest.raises(NotImplementedError):
        t.apply_adjoint(np.zeros((32, 32)), pad_mode="mean")
