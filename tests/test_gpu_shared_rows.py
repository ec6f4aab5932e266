"""Patches of one corner column share their row spectra (rpsf_bands.cuh): sharing must be exact.

The column pass of the full transform leaves, for every patch, the same spectrum bytes as a transform that holds only
that patch (np.array_equal), and the kernel gradient of the full transform equals the single-patch ones slot by slot.
"""
import ctypes

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


def _kernel(coords, size, shape):
    src = oracle.coma_psf_cube(coords, size, shape, core_sigma=min(2.5, size / 8), tail_scale=min(6.0, size / 6))
    tgt = oracle.gaussian_psf_cube(len(coords), size, min(3.0, size / 6))
    with np.errstate(all="ignore"):
        kernel = oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 1.0, 0.1)
    assert np.all(np.isfinite(kernel))
    return kernel


def _patch_spectra(coords, kernel, image, pad_mode, dtype, rows):
    """Spectrum workspace after the column pass: {corner: (P, P/2) complex} for the plan's active patches."""
    import torch
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    nt = t._native_transform(dtype)
    H, W = image.shape
    plan = nt.plan(H, W, _native.PAD_MODES[pad_mode], rows[0], rows[1], 1)
    n = nt.plan_info(plan)["active_patches"]
    real = torch.float32 if dtype == "float32" else torch.float64
    cdt = np.complex64 if dtype == "float32" else np.complex128
    img = torch.from_numpy(image).to(real).cuda()
    out = torch.zeros((H, W), dtype=real, device="cuda")
    torch.cuda.synchronize()
    _native.check(nt.lib.rpsf_apply_stages(plan, img.data_ptr(), W, H * W, 0, H, out.data_ptr(), W, H * W, 0, 1, 2, 0))
    ptr, nbytes = ctypes.c_void_p(), ctypes.c_int64()
    _native.check(nt.lib.rpsf_plan_workspace(plan, ctypes.byref(ptr), ctypes.byref(nbytes)))
    P = kernel.shape[-1]
    M = P if P & (P - 1) == 0 and P >= 16 else 1 << int(np.ceil(np.log2(2 * P - 1)))     # FFT length (embedded sizes)
    per_patch = M * (M // 2)
    host = np.empty(n * per_patch, dtype=cdt)
    assert nbytes.value >= host.nbytes
    _native.check(nt.lib.rpsf_copy_to_host(host.ctypes.data, ptr, host.nbytes, 0))
    # the plan's active patches: those touching the owned rows, in (corner row, corner column) order
    active = sorted((c for c in coords if max(c[0], rows[0]) < min(c[0] + P, rows[1]) and max(c[1], 0) < min(c[1] + P, W)),
                    key=lambda c: (c[0], c[1]))
    assert len(active) == n
    return {c: host[a * per_patch:(a + 1) * per_patch] for a, c in enumerate(active)}


CASES = {
    # name: (shape, patch size, coords or None for calculate_covering, pad mode, dtype, owned rows or None)
    "covering_symmetric_f32": ((320, 288), 64, None, "symmetric", "float32", None),
    "covering_constant_f64": ((320, 288), 64, None, "constant", "float64", None),
    "covering_reflect_f32_p32": ((160, 144), 32, None, "reflect", "float32", None),
    "covering_wrap_f64_p128": ((384, 320), 128, None, "wrap", "float64", None),
    "covering_p256_f32": ((640, 512), 256, None, "symmetric", "float32", None),
    "row_slab_f32": ((320, 288), 64, None, "reflect", "float32", (96, 200)),
    "irregular_mixed_parity": ((100, 90), 32, [(-5, 0), (0, 0), (3, 0), (10, 0), (17, 0), (40, 0), (41, 20),
                                               (-20, 70), (80, 70), (33, -10)], "symmetric", "float32", None),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_shared_rows_equal_a_patch_of_its_own(name):
    shape, size, coords, pad_mode, dtype, rows = CASES[name]
    if coords is None:
        coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]
    rows = rows or (0, shape[0])
    kernel = _kernel(coords, size, shape)
    image = oracle.starfield(shape, seed=11).astype(np.float64)
    full = _patch_spectra(coords, kernel, image, pad_mode, dtype, rows)
    # sampled patches: every frame edge, the corners, an interior one, and all of them for the irregular list
    keys = sorted(full, key=lambda c: (c[0], c[1]))
    if name.startswith("irregular"):
        picks = keys
    else:
        rows_of = sorted({c[0] for c in keys})
        cols_of = sorted({c[1] for c in keys})
        want = [(rows_of[0], cols_of[0]), (rows_of[0], cols_of[-1]), (rows_of[-1], cols_of[0]), (rows_of[-1], cols_of[-1]),
                (rows_of[len(rows_of) // 2], cols_of[len(cols_of) // 2]), (rows_of[1], cols_of[1]),
                (rows_of[-2], cols_of[-2])]
        picks = [c for c in dict.fromkeys(want) if c in full]
    assert picks
    index = {c: i for i, c in enumerate(coords)}
    for c in picks:
        i = index[c]
        own = _patch_spectra([c], kernel[i:i + 1], image, pad_mode, dtype, rows)
        assert np.array_equal(own[c], full[c]), (name, c)


@pytest.mark.parametrize("pad_mode,dtype", [("symmetric", "float32"), ("constant", "float64"), ("wrap", "float32")])
def test_kernel_gradient_equals_single_patch_transforms(pad_mode, dtype):
    import torch
    shape, size = (320, 288), 64
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]
    kernel = _kernel(coords, size, shape)
    rng = np.random.default_rng(3)
    real = torch.float32 if dtype == "float32" else torch.float64
    x = torch.from_numpy(rng.normal(size=(2,) + shape)).to(real).cuda()
    g = torch.from_numpy(rng.normal(size=(2,) + shape)).to(real).cuda()
    full = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel)).transfer_kernel_gradient(x, g, pad_mode=pad_mode,
                                                                                          dtype=dtype).cpu().numpy()
    for i in (0, 1, len(coords) // 2, len(coords) - 2, len(coords) - 1):
        one = rp.ArrayPSFTransform(rp.IndexedCube([coords[i]], kernel[i:i + 1])).transfer_kernel_gradient(
            x, g, pad_mode=pad_mode, dtype=dtype).cpu().numpy()
        assert np.array_equal(one[0], full[i]), (pad_mode, dtype, coords[i])
