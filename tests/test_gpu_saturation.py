"""The saturation branch of apply (transform.py:125-138,171-172) against the oracle, at full frame sizes and at its edges.

The device turns the reference's sequential raster-order fill into a parallel pipeline (mask, dilation, row count,
row scan, ordered scatter, and a fill whose CTAs claim 256-pixel chunks of the masked list and poll the state of
earlier pixels).  The scenes here are built to exercise every stage where it can go wrong: masked rows in every
1024-row chunk of the scan, a masked run wider than one fill chunk, mirrored blobs in the pad that are filled in a
different order, and transfer kernels that carry filled values onto unmasked output pixels with O(1) weights.

Bars: identical NaN pattern; max |diff| <= 1e-5 x max|image| in float32 mode, <= 1e-10 in float64 mode; masked output
pixels equal to the raw input (bit for bit when the input dtype is exact in the compute dtype, else within half a
float32 ulp); repeated calls, fresh plans, device and host paths and stitched row bands bit-identical.
"""
import functools
import math
import warnings

import numpy as np
import pytest
from scipy.ndimage import binary_dilation

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-10}
THR = 50000.0


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


# ------------------------------------------------------------------ kernels, scenes, the oracle
def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]


def _kernel(size, n, fwhm=None, shift=(0, 0)):
    """One spectrum for every patch: a circular shift by ``shift`` px, after a Gaussian blur of ``fwhm`` px if given.
    A shift carries each filled value onto the pixel ``shift`` away with weight 1 (times the windows)."""
    k = np.arange(size)
    spec = np.exp(-2j * np.pi * (k[:, None] * shift[0] + k[None, :] * shift[1]) / size)
    if fwhm is not None:
        r = np.minimum(k, size - k).astype(np.float64)
        g = np.exp(-4 * np.log(2) * (r[:, None] ** 2 + r[None, :] ** 2) / fwhm ** 2)
        spec = spec * np.fft.fft2(g / g.sum())
    return np.repeat(spec[np.newaxis].astype(np.complex128), n, axis=0)


def _blob(image, r, c, amp, sigma=1.2, half=4):
    h, w = image.shape
    rr, cc = np.mgrid[max(0, r - half):min(h, r + half + 1), max(0, c - half):min(w, c + half + 1)]
    image[rr, cc] = np.maximum(image[rr, cc], amp * np.exp(-((rr - r) ** 2 + (cc - c) ** 2) / (2 * sigma ** 2)))


def _full_scene(shape, seed, n_stars=800, rect=True):
    """A starfield with ``n_stars`` saturated stars over all rows, bleed columns a few hundred rows long, blobs on the
    four edges and corners, and (``rect``) one solid saturated rectangle 300 px wide and 30 rows tall."""
    rng = np.random.default_rng(seed)
    image = oracle.starfield(shape, seed=seed).astype(np.float32)
    h, w = shape
    for r, c in zip(rng.integers(0, h, n_stars), rng.integers(0, w, n_stars)):
        _blob(image, int(r), int(c), float(rng.uniform(55000.0, 300000.0)))
    for _ in range(6):
        col, top = int(rng.integers(2, w - 2)), int(rng.integers(0, h // 2))
        image[top:top + int(rng.integers(200, 400)), col:col + int(rng.integers(1, 3))] = 65535.0
    edges = [(0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (0, w // 3), (h - 1, 2 * w // 3), (h // 3, 0),
             (2 * h // 3, w - 1), (1, w // 2), (h // 2, 1), (h - 2, w // 5), (h // 5, w - 2)]
    for r, c in edges:
        _blob(image, r, c, 200000.0, sigma=2.0, half=6)
    if rect:
        r0, c0 = int(rng.integers(h // 4, h // 2)), int(rng.integers(10, w - 320))
        image[r0:r0 + 30, c0:c0 + 300] = 65535.0 + rng.uniform(0, 100, (30, 300)).astype(np.float32)
    return image


def _padded_mask(image, size, threshold, dilation, pad_mode="symmetric"):
    """The dilated mask of the padded frame, as the reference computes it (transform.py:125-131)."""
    pad = 2 * size
    padded = np.pad(np.asarray(image, dtype=np.float64), ((pad, pad), (pad, pad)), mode=pad_mode)
    with np.errstate(invalid="ignore"):
        mask = padded > threshold
    if mask.any():
        mask = binary_dilation(mask, iterations=dilation)
    return mask


def _frame_mask(image, size, threshold, dilation, pad_mode="symmetric"):
    pad = 2 * size
    h, w = np.shape(image)[-2:]
    return _padded_mask(image, size, threshold, dilation, pad_mode)[pad:pad + h, pad:pad + w]


def _assert_covers_scan_and_fill(image, size, dilation):
    """The scene reaches the parts of the pipeline it is meant for: masked pixels in every 1024-row chunk of the
    padded frame (the row scan's carry) and a masked run longer than one 256-pixel fill chunk."""
    mask = _padded_mask(image, size, THR, dilation)
    rows = mask.any(axis=1)
    for c in range(0, mask.shape[0], 1024):
        assert rows[c:c + 1024].any(), f"no masked pixel in padded rows [{c}, {c + 1024})"
    edges = np.diff(np.pad(mask.astype(np.int8), ((0, 0), (1, 1))), axis=1)
    starts, ends = np.nonzero(edges == 1), np.nonzero(edges == -1)
    assert int(np.max(ends[1] - starts[1])) > 256, "no masked run longer than a fill chunk"


def _oracle(image, coords, kernel, **kwargs):
    with warnings.catch_warnings(), np.errstate(invalid="ignore"):
        warnings.simplefilter("ignore", RuntimeWarning)         # nanmean of an empty or all-NaN window
        return oracle.apply_transform(np.asarray(image), coords, kernel, workers=-1, **kwargs)


def _sat(threshold=THR, dilation=1, width=7):
    return {"saturation_threshold": threshold, "saturation_dilation": dilation, "neighborhood_width": width}


def _check(got, want, image, mask, dtype, exact=True):
    """The bars of this module: NaN pattern, values, and the restored (masked) pixels."""
    got = np.asarray(got, dtype=np.float64)
    raw = np.asarray(image, dtype=np.float64)
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern differs from the oracle"
    finite = ~np.isnan(want)
    scale = float(np.nanmax(np.abs(raw)))
    if finite.any():
        err = float(np.max(np.abs(got[finite] - want[finite]))) / scale
        assert err <= TOL[dtype], f"max |device - oracle| = {err:.3e} x max|image| ({dtype})"
    if exact:
        assert np.array_equal(got[mask], raw[mask], equal_nan=True), "masked pixels are not the raw input"
    else:
        half_ulp = np.spacing(np.abs(raw[mask]).astype(np.float32)).astype(np.float64) / 2
        assert np.all(np.abs(got[mask] - raw[mask]) <= half_ulp), "masked pixels are not the raw input"


# (frame side, patch size, dilation, neighbourhood width): config 2's geometry, 1024^2 / 128 px, and one 2048^2 frame
# at 512 px (padded height 4096, the single-stage column pass)
FULL = [(2048, 256, 1, 7), (1024, 128, 2, 3), (2048, 512, 3, 9)]


@functools.lru_cache(maxsize=None)
def _full_case(side, size, dilation, width):
    shape = (side, side)
    coords = _covering(shape, size)
    kernel = _kernel(size, len(coords), fwhm=2.5, shift=(5, 3))
    image = _full_scene(shape, seed=side + size)
    _assert_covers_scan_and_fill(image, size, dilation)
    want = _oracle(image, coords, kernel, **_sat(THR, dilation, width))
    return coords, kernel, image, want


@functools.lru_cache(maxsize=None)
def _transform(coords, size, fwhm=2.5, shift=(5, 3)):
    """One transform per geometry and kernel, shared by the tests (its plans are cached across calls)."""
    return rp.ArrayPSFTransform(rp.IndexedCube(list(coords), _kernel(size, len(coords), fwhm, shift)))


# ------------------------------------------------------------------ 1. full-size scenes
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("side,size,dilation,width", FULL)
def test_full_size_scene_against_oracle(side, size, dilation, width, dtype):
    coords, kernel, image, want = _full_case(side, size, dilation, width)
    t = _transform(tuple(coords), size)
    got = t.apply(image, dtype=dtype, **_sat(THR, dilation, width))
    _check(got, want, image, _frame_mask(image, size, THR, dilation), dtype)
    # bit-stable although the fill is resolved by polling, on a fresh transform too
    assert np.array_equal(got, t.apply(image, dtype=dtype, **_sat(THR, dilation, width)))
    fresh = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    assert np.array_equal(got, fresh.apply(image, dtype=dtype, **_sat(THR, dilation, width)))


# ------------------------------------------------------------------ 2. a kernel that makes the fill visible
@functools.lru_cache(maxsize=None)
def _shift_case(dilation, width):
    shape, size = (1024, 1024), 128
    coords = _covering(shape, size)
    image = _full_scene(shape, seed=77)
    _assert_covers_scan_and_fill(image, size, dilation)
    kernel = _kernel(size, len(coords), shift=(size // 8, size // 16))
    return coords, kernel, image, _oracle(image, coords, kernel, **_sat(THR, dilation, width))


@pytest.mark.parametrize("dtype,dilation,width", [("float32", 1, 7), ("float64", 1, 7), ("float64", 2, 9)])
def test_shift_kernel_carries_the_fill_onto_unmasked_pixels(dtype, dilation, width):
    """With a pure shift by (P/8, P/16) every filled value lands on an unmasked output pixel with an O(1) weight, so
    the value bar checks the fill itself rather than a smoothed trace of it."""
    coords, kernel, image, want = _shift_case(dilation, width)
    size = 128
    mask = _frame_mask(image, size, THR, dilation)
    shifted = np.zeros_like(mask)
    shifted[size // 8:, size // 16:] = mask[:-(size // 8), :-(size // 16)]
    assert (shifted & ~mask).sum() > 1000, "the shift must carry filled values onto unmasked pixels"
    t = _transform(tuple(coords), size, None, (size // 8, size // 16))
    got = t.apply(image, dtype=dtype, **_sat(THR, dilation, width))
    _check(got, want, image, mask, dtype)


# ------------------------------------------------------------------ 3. settings at their edges
@pytest.mark.parametrize("dilation", [0, -1])
def test_dilation_until_stable_masks_everything_and_returns_the_input(dilation):
    """dilation < 1 is scipy's "until nothing changes": with one pixel above the threshold the whole padded frame is
    masked, every fill is NaN, and the output is the input bit for bit."""
    import torch
    side, size = 2048, 256
    coords = _covering((side, side), size)
    image = oracle.starfield((side, side), seed=3)
    image[1000, 1000] = 70000.0
    t = _transform(tuple(coords), size)
    for dtype in ("float32", "float64"):
        got = t.apply(image, dtype=dtype, **_sat(THR, dilation, 7))
        assert np.array_equal(got, image.astype(np.float64)), dtype
    dev = t.apply(torch.from_numpy(image).cuda(), **_sat(THR, dilation, 7))
    assert torch.equal(dev.cpu(), torch.from_numpy(image))


def test_threshold_below_every_pixel_returns_the_input():
    side, size = 512, 64
    coords = _covering((side, side), size)
    image = oracle.starfield((side, side), seed=4)
    t = _transform(tuple(coords), size)
    for dtype in ("float32", "float64"):
        got = t.apply(image, dtype=dtype, **_sat(float(image.min()) - 1.0, 1, 7))
        assert np.array_equal(got, image.astype(np.float64)), dtype


def test_nan_threshold_is_the_branch_switched_off():
    side, size = 512, 64
    coords = _covering((side, side), size)
    image = _full_scene((side, side), seed=5, n_stars=20, rect=False)
    t = _transform(tuple(coords), size)
    for dtype in ("float32", "float64"):
        assert np.array_equal(t.apply(image, dtype=dtype), t.apply(image, dtype=dtype, **_sat(math.nan, 2, 7)))


EDGE_SHAPE, EDGE_SIZE = (256, 192), 64


@functools.lru_cache(maxsize=None)
def _edge_scene():
    """Small scene with masked pixels whose padded position is within a window half-width of the padded frame's
    top/left (numpy's empty slice) and bottom/right (the clamped slice), a pixel exactly at the threshold, and NaN
    input pixels inside and right next to masked blobs."""
    h, w = EDGE_SHAPE
    p = EDGE_SIZE
    image = _full_scene(EDGE_SHAPE, seed=21, n_stars=10, rect=False)
    # symmetric pad: frame row 2P-1 lands on padded row 0, frame row H-2P on padded row Hp-1 (same for columns)
    for r, c in [(2 * p - 1, 2 * p - 1), (2 * p - 1, 40), (20, 2 * p - 1), (h - 2 * p, w - 2 * p), (h - 2 * p, 30),
                 (200, w - 2 * p)]:
        _blob(image, r, c, 120000.0)
    image[150, 100] = THR                          # exactly the threshold: stays unmasked
    _blob(image, 60, 150, 90000.0)
    image[60, 150] = np.nan                        # inside a masked blob
    image[60, 152] = np.nan                        # next to its core, inside the dilated mask
    image[60, 153] = np.nan                        # next to the dilated mask, in the fill window of its pixels
    return image


@pytest.mark.parametrize("width", [1, 0, 2, 8, 15, 7])
def test_edge_scene_neighbourhood_widths_against_oracle(width):
    image = _edge_scene()
    coords = _covering(EDGE_SHAPE, EDGE_SIZE)
    kernel = _kernel(EDGE_SIZE, len(coords), fwhm=2.0, shift=(7, 5))
    want = _oracle(image, coords, kernel, **_sat(THR, 1, width))
    mask = _frame_mask(image, EDGE_SIZE, THR, 1)
    padded = _padded_mask(image, EDGE_SIZE, THR, 1)
    half = max(width // 2, 1)
    assert padded[:half].any() and padded[:, :half].any() and padded[-half:].any() and padded[:, -half:].any()
    assert image[150, 100] == THR and not mask[150, 100]
    t = _transform(tuple(coords), EDGE_SIZE, 2.0, (7, 5))
    for dtype in ("float32", "float64"):
        got = t.apply(image, dtype=dtype, **_sat(THR, 1, width))
        _check(got, want, image, mask, dtype)


def test_nan_input_next_to_a_masked_region_poisons_the_same_footprint():
    """A NaN pixel just outside the dilated mask: the fill skips it (nanmean), the patches that read it are NaN."""
    image = _edge_scene().copy()
    image[60, 156] = np.nan
    coords = _covering(EDGE_SHAPE, EDGE_SIZE)
    kernel = _kernel(EDGE_SIZE, len(coords), fwhm=2.0, shift=(7, 5))
    mask = _frame_mask(image, EDGE_SIZE, THR, 1)
    assert mask[60, 152] and not mask[60, 153] and not mask[60, 156]
    want = _oracle(image, coords, kernel, **_sat(THR, 1, 7))
    assert np.isnan(want).any() and not np.isnan(want).all()
    t = _transform(tuple(coords), EDGE_SIZE, 2.0, (7, 5))
    for dtype in ("float32", "float64"):
        _check(t.apply(image, dtype=dtype, **_sat(THR, 1, 7)), want, image, mask, dtype)


def test_constant_pad_with_a_negative_threshold_masks_the_margin():
    image = _edge_scene() - 200.0
    threshold = -50.0
    coords = _covering(EDGE_SHAPE, EDGE_SIZE)
    kernel = _kernel(EDGE_SIZE, len(coords), fwhm=2.0, shift=(7, 5))
    padded = _padded_mask(image, EDGE_SIZE, threshold, 1, "constant")
    assert padded[0].all() and padded[:, 0].all() and not padded.all()
    want = _oracle(image, coords, kernel, pad_mode="constant", **_sat(threshold, 1, 7))
    t = _transform(tuple(coords), EDGE_SIZE, 2.0, (7, 5))
    mask = _frame_mask(image, EDGE_SIZE, threshold, 1, "constant")
    for dtype in ("float32", "float64"):
        _check(t.apply(image, pad_mode="constant", dtype=dtype, **_sat(threshold, 1, 7)), want, image, mask, dtype)


@pytest.mark.parametrize("pad_mode", ["reflect", "edge", "wrap", "constant"])
def test_index_map_pad_modes_at_full_size(pad_mode):
    """symmetric is test_full_size_scene_against_oracle; the other four modes mirror the blobs differently."""
    side, size = 2048, 256
    coords, kernel, image, _ = _full_case(side, size, 1, 7)
    want = _oracle(image, coords, kernel, pad_mode=pad_mode, **_sat(THR, 1, 7))
    got = _transform(tuple(coords), size).apply(image, pad_mode=pad_mode, **_sat(THR, 1, 7))
    _check(got, want, image, _frame_mask(image, size, THR, 1, pad_mode), "float32")


# ------------------------------------------------------------------ 4. both K1 kernels on the fill buffer
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("width_px", [192, 191])
def test_both_k1_kernels_read_the_fill_buffer(width_px, dtype):
    """K1 reads the materialised fill buffer, whose pitch is W + 4P: bulk row copies where (W + 4P) x sizeof(T) is a
    multiple of 16 (W = 192), the gather fallback where it is not (W = 191); and the older K1 (gather mode 1)."""
    import torch
    shape, size = (256, width_px), 64
    coords = _covering(shape, size)
    kernel = _kernel(size, len(coords), fwhm=2.0, shift=(7, 5))
    image = _full_scene(shape, seed=31, n_stars=15, rect=False)
    want = _oracle(image, coords, kernel, **_sat(THR, 2, 7))
    mask = _frame_mask(image, size, THR, 2)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    nt = t._native_transform(dtype)
    plan = nt.plan(shape[0], shape[1], 0, 0, shape[0], 1)
    tdtype = torch.float32 if dtype == "float32" else torch.float64
    frame = torch.from_numpy(image).to("cuda", tdtype)
    try:
        for mode in (0, 1):
            _native.check(nt.lib.rpsf_plan_set_gather_mode(plan, mode))
            got = t.apply(frame, dtype=dtype, **_sat(THR, 2, 7)).cpu().numpy()
            _check(got, want, image, mask, dtype)
    finally:
        nt.lib.rpsf_plan_set_gather_mode(plan, 0)


# ------------------------------------------------------------------ 5. combinations
def test_row_bands_stitch_into_the_whole_frame():
    import torch
    side, size = 2048, 256
    coords, _, image, _ = _full_case(side, size, 1, 7)
    t = _transform(tuple(coords), size)
    frame = torch.from_numpy(image).cuda()
    sat = (THR, 1, 7)
    whole = t._apply_device(frame, "float32", 0, sat=sat).cpu().numpy()
    for cuts in ([0, 384, 1024, 2048], [0, 1000, 1001, 1537, 2048]):      # on and off patch-row boundaries (P/2)
        bands = [t._apply_device(frame, "float32", 0, row_range=(lo, hi), sat=sat).cpu().numpy()
                 for lo, hi in zip(cuts[:-1], cuts[1:])]
        assert np.array_equal(np.concatenate(bands, axis=0), whole), cuts


@functools.lru_cache(maxsize=None)
def _batch_case():
    side, size = 2048, 256
    coords, kernel, busy, want_busy = _full_case(side, size, 1, 7)
    sparse = oracle.starfield((side, side), seed=9)
    for r, c in [(300, 1700), (1500, 200), (2000, 1000)]:
        _blob(sparse, r, c, 80000.0)
    clean = oracle.starfield((side, side), seed=10)
    assert not (clean > THR).any()
    frames = np.stack([busy, clean, sparse])
    want = np.stack([want_busy, _oracle(clean, coords, kernel, **_sat()), _oracle(sparse, coords, kernel, **_sat())])
    return coords, kernel, frames, want


def test_host_batch_of_frames_with_very_different_masked_counts():
    """Three 2048^2 frames run one per host chunk and reuse the plan's saturation buffers; one has no masked pixel."""
    coords, _, frames, want = _batch_case()
    size = 256
    t = _transform(tuple(coords), size)
    counts = [int(_frame_mask(f, size, THR, 1).sum()) for f in frames]
    assert counts[1] == 0 and counts[2] > 0 and counts[0] > 100 * counts[2]
    assert t.HOST_CHUNK_BYTES < frames[0].nbytes * 2
    got = t.apply(frames, **_sat())
    for k in range(3):
        _check(got[k], want[k], frames[k], _frame_mask(frames[k], size, THR, 1), "float32")
        assert np.array_equal(got[k], t.apply(frames[k], **_sat())), k


def test_device_batch_equals_host_path():
    import torch
    coords, _, frames, _ = _batch_case()
    t = _transform(tuple(coords), 256)
    host = t.apply(frames, **_sat())
    dev = t.apply(torch.from_numpy(frames).cuda(), **_sat()).cpu().numpy()
    assert np.array_equal(dev.astype(np.float64), host)


@pytest.mark.parametrize("size", [48, 100])
def test_embedded_patch_sizes(size):
    shape = (300, 260)
    coords = _covering(shape, size)
    kernel = _kernel(size, len(coords), fwhm=2.0, shift=(size // 8, size // 16))
    image = _full_scene(shape, seed=size, n_stars=20, rect=False)
    want = _oracle(image, coords, kernel, **_sat(THR, 2, 7))
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    mask = _frame_mask(image, size, THR, 2)
    for dtype in ("float32", "float64"):
        _check(t.apply(image, dtype=dtype, **_sat(THR, 2, 7)), want, image, mask, dtype)


def test_irregular_coordinates():
    """The golden p16_irregular_coords geometry scaled by 8: 512^2, 128-px patches at scattered corners (several
    colour phases of overlap-add)."""
    from tests.helpers import load_golden
    g = load_golden("p16_irregular_coords")
    scale, size = 8, 128
    coords = [(r * scale, c * scale) for r, c in g["coords"]]
    shape = (g["image"].shape[0] * scale, g["image"].shape[1] * scale)
    kernel = _kernel(size, len(coords), fwhm=2.0, shift=(size // 8, size // 16))
    image = _full_scene(shape, seed=41, n_stars=60, rect=False)
    want = _oracle(image, coords, kernel, **_sat(THR, 1, 7))
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    mask = _frame_mask(image, size, THR, 1)
    for dtype in ("float32", "float64"):
        _check(t.apply(image, dtype=dtype, **_sat(THR, 1, 7)), want, image, mask, dtype)


def test_materialised_pad_median():
    image = _edge_scene()
    coords = _covering(EDGE_SHAPE, EDGE_SIZE)
    kernel = _kernel(EDGE_SIZE, len(coords), fwhm=2.0, shift=(7, 5))
    image = np.where(np.isnan(image), 0.0, image).astype(np.float32)     # np.pad's median of a NaN row is NaN
    want = _oracle(image, coords, kernel, pad_mode="median", **_sat(THR, 2, 7))
    mask = _frame_mask(image, EDGE_SIZE, THR, 2, "median")
    t = _transform(tuple(coords), EDGE_SIZE, 2.0, (7, 5))
    for dtype in ("float32", "float64"):
        _check(t.apply(image, pad_mode="median", dtype=dtype, **_sat(THR, 2, 7)), want, image, mask, dtype)


def test_cached_plan_with_changing_settings_equals_fresh_transforms():
    side, size = 1024, 128
    coords, kernel, image, _ = _full_case(side, size, 2, 3)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    calls = [_sat(THR, 2, 3), {}, _sat(THR, 1, 8), _sat(60000.0, 3, 7), _sat(THR, 0, 7), _sat(THR, 2, 3)]
    for kwargs in calls:
        fresh = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel)).apply(image, **kwargs)
        assert np.array_equal(t.apply(image, **kwargs), fresh), kwargs


# ------------------------------------------------------------------ 6. input dtypes near the threshold
def _near_threshold_scene(dtype):
    """A frame with pixels at threshold + delta and threshold - delta, delta below half a float32 ulp there."""
    shape = (256, 192)
    base = _full_scene(shape, seed=61, n_stars=8, rect=False).astype(np.float64)
    if dtype == np.int32:
        threshold = 2.0 ** 24 + 0.5                  # 2^24 + 1 rounds to 2^24 in float32
        image = np.rint(base).astype(np.int32)
        image[image > 2 ** 24] = 2 ** 24
        image[40, 50] = 2 ** 24 + 1                  # above the threshold, equal to 2^24 in float32
        image[41, 52] = 2 ** 24 + 1
        image[90, 100] = 2 ** 24                     # below
        image[200, 20] = 2 ** 24 + 3                 # above; 2^24 + 4 in float32
        image[180, 150] = 2 ** 24 + 1
        return image, threshold
    threshold = THR
    image = base.copy()
    spacing = float(np.spacing(np.float32(THR)))
    assert 0.001 < spacing / 2
    image[image > THR] = THR - 1000.0
    image[40, 50] = THR + 0.001                      # above; THR in float32
    image[41, 52] = THR + 0.001
    image[90, 100] = THR - 0.001                     # below; THR in float32
    image[200, 20] = THR + 0.0015
    image[180, 150] = THR + 0.001
    return image, threshold


@pytest.mark.parametrize("kind", ["float64 array", "float64 tensor", "int32 array", "int32 tensor", "float64 median"])
def test_mask_is_decided_on_the_unconverted_input(kind):
    """In float32 mode a float64 or int32 pixel just above the threshold converts to the threshold or below it; the
    reference masks it (it compares the float64 value), so the device must decide the mask before the conversion."""
    import torch
    dtype = np.int32 if kind.startswith("int32") else np.float64
    image, threshold = _near_threshold_scene(dtype)
    shape, size = image.shape, 64
    coords = _covering(shape, size)
    kernel = _kernel(size, len(coords), fwhm=2.0, shift=(7, 5))
    pad_mode = "median" if kind.endswith("median") else "symmetric"
    kwargs = dict(pad_mode=pad_mode, **_sat(threshold, 1, 7))
    want = _oracle(image, coords, kernel, **kwargs)
    mask = _frame_mask(image, size, threshold, 1, pad_mode)
    assert mask[40, 50] and mask[200, 20] and not mask[90, 100]
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    if kind.endswith("tensor"):
        got = t.apply(torch.from_numpy(image).cuda(), **kwargs).cpu().numpy()
    else:
        got = t.apply(image, **kwargs)
    _check(got, want, image, mask, "float32", exact=False)
    got64 = t.apply(image, dtype="float64", **kwargs)
    _check(got64, want, image, mask, "float64")
