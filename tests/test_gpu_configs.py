"""BASELINE.json's named configurations at FULL size on the GPU, plus the edge cases round 1 left open.

* config 1 exactly as tests/test_oracle_vs_reference.py pins the oracle to the reference: 1024^2, 128-px patches,
  make_gaussian fwhm 4 -> 3, alpha 3, epsilon 0.1 (regularizepsf/transform.py:53-83,85-177);
* config 4 with a real (coma) kernel at P = 512 on the 8192^2 mosaic: the oracle is run on the patches that cover one
  band of output rows (exact for that band: a row only ever receives the two patch rows that contain it,
  transform.py:157-169), at the top edge, in the interior and at the bottom edge of the frame;
* empty row bands, misaligned partial rows, tensors on a device that is not the current one, a caller that varies
  its batch size.
"""
import os

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native
from tests.helpers import make_gaussian, rel_err

pytestmark = pytest.mark.gpu
TOL = {"float32": 1e-5, "float64": 1e-10}


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]


@pytest.fixture(scope="module")
def config1():
    shape, size = (1024, 1024), 128
    coords = _covering(shape, size)
    g4, g3 = make_gaussian(size, fwhm=4), make_gaussian(size, fwhm=3)
    src = np.stack([g4 / g4.sum()] * len(coords))
    tgt = np.stack([g3 / g3.sum()] * len(coords))
    kernel = oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 3.0, 0.1)
    image = oracle.starfield(shape, seed=1234)
    want = oracle.apply_transform(image, coords, kernel, workers=-1)
    return coords, src, tgt, kernel, image, want


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_config1_full_size_given_kernel(config1, dtype):
    coords, _, _, kernel, image, want = config1
    assert len(coords) == 289 and np.all(np.isfinite(kernel))
    got = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel)).apply(image, dtype=dtype)
    assert got.dtype == np.float64 and got.shape == image.shape
    assert rel_err(got, want, float(image.max())) <= TOL[dtype]


def test_config1_full_size_device_fft_and_construct(config1):
    """ArrayPSF (device fft2) -> construct (device) -> apply, float64 PSF samples as in the reference's tests."""
    coords, src, tgt, _, image, want = config1
    source, target = rp.ArrayPSF(rp.IndexedCube(coords, src)), rp.ArrayPSF(rp.IndexedCube(coords, tgt))
    t = rp.ArrayPSFTransform.construct(source, target, 3.0, 0.1)
    assert rel_err(t.apply(image), want, float(image.max())) <= TOL["float32"]
    assert rel_err(t.apply(image, dtype="float64"), want, float(image.max())) <= TOL["float64"]
    # a batch of the same frame through the device path gives the same bits as the single frame
    import torch
    frames = torch.from_numpy(np.stack([image] * 3)).cuda()
    out = t.apply(frames)
    assert torch.equal(out[0], out[2]) and torch.equal(out[0], t.apply(frames[0]))


def test_config4_real_coma_kernel_row_bands():
    """8192^2, 512-px patches, spatially varying coma source -> Gaussian target: three bands against the oracle."""
    import torch
    shape, size = (8192, 8192), 512
    coords = _covering(shape, size)
    assert len(coords) == 1089
    rows = sorted({c[0] for c in coords})
    image = np.tile(oracle.starfield((2048, 2048), seed=77), (4, 4))
    image *= np.linspace(0.5, 1.5, shape[0], dtype=image.dtype)[:, None]            # no two bands alike
    dev_image = torch.from_numpy(image).cuda()
    # kernel cube on the device for all 1089 patches, built per patch row to bound host memory
    kernel = torch.empty((len(coords), size, size), dtype=torch.complex64, device="cuda")
    index = {c: i for i, c in enumerate(coords)}
    host_kernels = {}
    for r in rows:
        sub = [c for c in coords if c[0] == r]
        src = oracle.coma_psf_cube(sub, size, shape)
        tgt = oracle.gaussian_psf_cube(len(sub), size, 3.0)
        k = oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 1.0, 0.1).astype(np.complex64)
        assert np.all(np.isfinite(k))
        host_kernels[r] = (sub, k)
        kernel[[index[c] for c in sub]] = torch.from_numpy(k).cuda()
    from regularizepsf_b200.device import DeviceCube
    t = rp.ArrayPSFTransform(DeviceCube(coords, kernel))
    got = t.apply(dev_image).cpu().numpy()
    half = size // 2
    for band0 in (0, 2048, shape[0] - half):
        upper, lower = band0 - half, band0                   # corner rows of the two patch rows covering the band
        assert upper in host_kernels and lower in host_kernels
        lo, hi = max(upper, 0), min(lower + size, shape[0])
        sub_image = image[lo:hi]
        sub_coords, sub_kernel = [], []
        for r in (upper, lower):
            cs, k = host_kernels[r]
            sub_coords += [(c[0] - lo, c[1]) for c in cs]
            sub_kernel.append(k)
        want = oracle.apply_transform(sub_image, sub_coords, np.concatenate(sub_kernel), workers=-1)
        a, b = band0 - lo, band0 - lo + half
        err = rel_err(got[band0:band0 + half], want[a:b], float(image.max()))
        print(f"config 4 band rows [{band0},{band0 + half}): max rel err {err:.3e}")
        assert err <= TOL["float32"]


# ------------------------------------------------------------------ edge cases (ADVICE.md round 1)
def _small(shape=(96, 80), size=32, seed=3):
    coords = _covering(shape, size)
    rng = np.random.default_rng(seed)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    return coords, kernel.astype(np.complex64), oracle.starfield(shape, seed=seed)


def test_empty_row_band_is_a_no_op_on_host_and_device():
    import torch
    from regularizepsf_b200.distributed import slab_bounds
    coords, kernel, image = _small()
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    bounds = slab_bounds(image.shape[0], 32, 8)                # 6 half-patch rows for 8 ranks: empty bands exist
    assert any(lo == hi for lo, hi in bounds)
    whole = t.apply(image)
    parts = [t._apply_host(image, "float32", 0, row_range=b) for b in bounds]
    assert [p.shape[0] for p in parts] == [hi - lo for lo, hi in bounds]
    assert np.array_equal(np.concatenate(parts, axis=0), whole)
    dev = torch.from_numpy(image).cuda()
    dparts = [t._apply_device(dev, "float32", 0, row_range=b) for b in bounds]
    assert np.array_equal(torch.cat(dparts, dim=0).cpu().numpy().astype(np.float64), whole)


@pytest.mark.parametrize("pad_mode", ["symmetric", "reflect", "wrap", "edge", "constant"])
def test_patch_overhanging_both_frame_edges_with_a_misaligned_offset(pad_mode):
    """corner column -6 on a 20-px-wide frame: both ends of the in-frame span are 16-byte aligned but the landing
    offset in the stage row is not, so the row must take the gathered path (ADVICE: rpsf_stream.cuh `aligned`)."""
    size, shape = 16, (40, 20)
    coords = [(-6, -6), (2, -6), (10, 2), (-8, 4), (18, -6), (26, 2)]
    rng = np.random.default_rng(8)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    image = oracle.starfield(shape, seed=4)
    want = oracle.apply_transform(image, coords, kernel, pad_mode=pad_mode)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel.astype(np.complex128)))
    for dtype in ("float32", "float64"):
        got = t.apply(image, pad_mode=pad_mode, dtype=dtype)
        assert rel_err(got, want, float(image.max())) <= TOL[dtype]


def test_varying_batch_sizes_do_not_grow_the_plan_cache():
    import torch
    coords, kernel, image = _small()
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    frames = torch.from_numpy(np.stack([image] * 12)).cuda()
    single = t.apply(frames[0])
    for b in (1, 2, 3, 5, 8, 12, 7, 4, 9, 11, 6, 10):
        out = t.apply(frames[:b])
        assert torch.equal(out[b - 1], single)
    nt = t._native_transform("float32")
    assert len(nt._plans) <= nt.MAX_PLANS


def test_tensor_on_a_device_that_is_not_current():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    coords, kernel, image = _small()
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    want = t.apply(torch.from_numpy(image).to("cuda:0"))
    assert torch.cuda.current_device() == 0
    got = t.apply(torch.from_numpy(image).to("cuda:1"))          # current device stays 0
    assert got.device.index == 1 and torch.equal(got.cpu(), want.cpu())
    assert torch.cuda.current_device() == 0


def test_psf_fft2_returns_without_synchronising_and_reuses_its_tables():
    import torch
    values = torch.rand((4, 64, 64), device="cuda", dtype=torch.float32)
    lib = _native.load()
    outs = []
    for _ in range(3):
        out = torch.empty((4, 64, 64), dtype=torch.complex64, device="cuda")
        _native.check(lib.rpsf_psf_fft2(values.data_ptr(), out.data_ptr(), 4, 64, _native.F32, 0,
                                        _native.current_stream_ptr(torch)))
        outs.append(out)
    torch.cuda.synchronize()
    want = torch.fft.fft2(values.double()).to(torch.complex64)
    for out in outs:
        assert float((out - want).abs().max() / want.abs().max()) <= 2e-6


# ------------------------------------------------------------------ real multi-GPU runs (skipped on a one-GPU box)
def test_frame_and_slab_sharding_across_real_gpus_is_bit_identical():
    """Two ranks over NCCL on two GPUs: config 3 (frames sharded, gathered over NCCL and by peer stores fused into the
    overlap-add kernel, whole block and chunked) and config 4 (patch-row slabs, all-gather / root / none, sharded
    kernel cube and partial frame residency) must equal the single-GPU result bit for bit."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(root, "scripts", "multi_gpu_check.py"), "--assert"]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    print(proc.stdout[-3000:])
    assert proc.returncode == 0, proc.stderr[-3000:]
    assert '"config": 3' in proc.stdout and '"config": 4' in proc.stdout


def test_sharded_transform_on_one_gpu_stitches_bit_identically():
    """shard_transform_rows + frame_rows on a single device: every rank's band from its shard of the kernel cube and
    its rows of the frame equals the band of the complete transform (same colours, same summation order)."""
    import torch
    from regularizepsf_b200 import distributed as rdist
    from regularizepsf_b200.device import DeviceCube
    shape, size, world = (1536, 640), 128, 4
    coords = _covering(shape, size)
    g = torch.Generator(device="cuda").manual_seed(5)
    kernel = torch.randn((len(coords), size, size), dtype=torch.complex64, device="cuda", generator=g)
    full = rp.ArrayPSFTransform(DeviceCube(coords, kernel))
    image = torch.rand(shape, device="cuda", generator=g) * 500
    whole = full.apply(image)
    host = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel.cpu().numpy()))       # a host-resident cube shards too
    for rank in range(world):
        lo, hi = rdist.slab_bounds(shape[0], size, world)[rank]
        for source in (full, host):
            shard = rdist.shard_transform_rows(source, shape[0], rank, world)
            assert 0 < len(shard) < len(full)
            first, last = rdist.rows_needed(coords, size, shape[0], (lo, hi))
            band = shard._apply_device(image[first:last].contiguous(), "float32", 0, row_range=(lo, hi),
                                       frame_rows=(first, shape[0]))
            assert torch.equal(band, whole[lo:hi]), (rank, type(source._transfer_kernel).__name__)
        nt = shard._native_transform("float32")
        assert nt.plan_info(nt.plan(shape[0], shape[1], 0, lo, hi, 1))["rows_read"] == (first, last)
        with pytest.raises(ValueError):                                  # a shard cannot serve rows it has no kernels for
            other = (rank + 2) % world
            shard._apply_device(image, "float32", 0, row_range=rdist.slab_bounds(shape[0], size, world)[other])


# ------------------------------------------------------------------ every np.pad mode the reference accepts
@pytest.mark.parametrize("pad_mode", ["mean", "median", "maximum", "minimum", "linear_ramp"])
def test_statistical_pad_modes_match_np_pad(pad_mode):
    """transform.py:119-123 hands `pad_mode` straight to np.pad; modes without an index map are padded by np.pad on the
    host and the kernels read the materialised margin."""
    import torch
    shape, size = (200, 144), 32
    coords = _covering(shape, size)
    rng = np.random.default_rng(12)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel.astype(np.complex128)))
    frames = np.stack([oracle.starfield(shape, seed=s) for s in (31, 32)])
    want = np.stack([oracle.apply_transform(f, coords, kernel, pad_mode=pad_mode) for f in frames])
    scale = float(frames.max())
    for dtype in ("float32", "float64"):
        got = t.apply(frames, pad_mode=pad_mode, dtype=dtype)
        assert got.dtype == np.float64 and got.shape == frames.shape
        assert rel_err(got, want, scale) <= TOL[dtype], (pad_mode, dtype)
    one = t.apply(frames[1].astype(np.uint16), pad_mode=pad_mode)                     # integer pixels, single frame
    assert rel_err(one, oracle.apply_transform(frames[1].astype(np.uint16), coords, kernel, pad_mode=pad_mode), scale) <= TOL["float32"]
    dev = t.apply(torch.from_numpy(frames).cuda(), pad_mode=pad_mode)                 # device tensors take the same route
    assert dev.is_cuda and rel_err(dev.cpu().numpy(), want, scale) <= TOL["float32"]
    sat = t.apply(frames[0], pad_mode=pad_mode, saturation_threshold=float(np.percentile(frames[0], 99.9)))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want_sat = oracle.apply_transform(frames[0], coords, kernel, pad_mode=pad_mode,
                                          saturation_threshold=float(np.percentile(frames[0], 99.9)))
    assert np.array_equal(np.isnan(sat), np.isnan(want_sat)) and rel_err(sat, want_sat, scale) <= TOL["float32"]


def test_pad_mode_np_pad_rejects_is_rejected():
    coords, kernel, image = _small()
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    with pytest.raises(ValueError):
        t.apply(image, pad_mode="no such mode")


# ------------------------------------------------------------------ patch sizes that are not powers of two
@pytest.mark.parametrize("size,shape", [(48, (150, 120)), (100, (260, 300)), (21, (90, 75)), (6, (40, 33)), (200, (512, 420))])
def test_patch_sizes_without_a_native_fft_length(size, shape):
    """The reference takes any square patch size (transform.py:151-165; tests/test_util.py covers odd sizes).  Sizes that
    are not a power of two in 16..512 run embedded in the next power of two >= 2 P - 1 with a re-sampled kernel."""
    coords = _covering(shape, size)
    src = oracle.coma_psf_cube(coords, size, shape, core_sigma=min(2.5, size / 8), tail_scale=min(6.0, size / 6))
    tgt = oracle.gaussian_psf_cube(len(coords), size, min(3.0, size / 6))
    with np.errstate(all="ignore"):
        kernel = oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 1.0, 0.1)
    assert np.all(np.isfinite(kernel))
    frames = np.stack([oracle.starfield(shape, seed=s) for s in (41, 42)])
    want = np.stack([oracle.apply_transform(f, coords, kernel) for f in frames])
    scale = float(frames.max())
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    for dtype in ("float32", "float64"):
        got = t.apply(frames, dtype=dtype)
        assert got.shape == frames.shape and got.dtype == np.float64
        assert rel_err(got, want, scale) <= TOL[dtype], (size, dtype)
    # ArrayPSF -> construct -> apply end to end (direct DFT of the PSF cubes on the device)
    source, target = rp.ArrayPSF(rp.IndexedCube(coords, src)), rp.ArrayPSF(rp.IndexedCube(coords, tgt))
    assert np.max(np.abs(source.fft_evaluations - oracle.psf_fft(src))) <= 1e-12
    full = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    assert rel_err(full.apply(frames[0], dtype="float64"), want[0], scale) <= 1e-9
    # pad modes, row slabs and a NaN pixel keep the reference's footprint (the window ends at P, not at the FFT length)
    assert rel_err(t.apply(frames[0], pad_mode="reflect"), oracle.apply_transform(frames[0], coords, kernel, pad_mode="reflect"), scale) <= TOL["float32"]
    from regularizepsf_b200.distributed import slab_bounds
    parts = [t._apply_host(frames[1], "float32", 0, row_range=b) for b in slab_bounds(shape[0], size, 3)]
    assert np.array_equal(np.concatenate(parts, axis=0), t.apply(frames[1]))
    poisoned = frames[0].copy()
    poisoned[shape[0] // 2, shape[1] // 3] = np.nan
    want_nan = oracle.apply_transform(poisoned, coords, kernel)
    got_nan = t.apply(poisoned)
    assert np.array_equal(np.isnan(got_nan), np.isnan(want_nan))
    ok = ~np.isnan(want_nan)
    assert np.max(np.abs(got_nan[ok] - want_nan[ok])) <= TOL["float32"] * scale


# ------------------------------------------------------------------ coverings, row bands and pad modes against the oracle
@pytest.mark.parametrize("shape,size,dtype,batch,rows", [((2048, 2048), 256, "float32", 1, None), ((2048, 2048), 256, "float32", 3, None),
                                                        ((1024, 768), 128, "float32", 2, None), ((1024, 768), 128, "float64", 1, (256, 640)),
                                                        ((640, 512), 64, "float32", 9, None), ((700, 333), 64, "float64", 2, None),
                                                        ((2048, 1024), 256, "float32", 2, (512, 1408))])
def test_three_kernels_on_coverings_and_row_bands(shape, size, dtype, batch, rows):
    """The three kernels on coverings, whole frames and row bands: within the oracle tolerance, and bit-identical across
    fresh plans for 1 to 128 frames per call.  The planner cuts the overlap-add chains into more chunks for small calls
    than for large ones (every case here walks whole chains at 128): chunks recompute their seams, so every cut
    reproduces whole chains bit for bit."""
    import torch
    coords = _covering(shape, size)
    rng = np.random.default_rng(17)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    kernel = kernel.astype(np.complex64 if dtype == "float32" else np.complex128)
    frames = np.stack([oracle.starfield(shape, seed=60 + i) for i in range(batch)])
    tdtype = torch.float32 if dtype == "float32" else torch.float64
    dev = torch.from_numpy(frames).to("cuda", tdtype)
    lo, hi = rows if rows else (0, shape[0])

    def run(max_batch):
        """The batch through a fresh plan for `max_batch` frames per call, `max_batch` frames at a time."""
        t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))              # a fresh transform: a fresh plan
        nt = t._native_transform(dtype)
        plan = nt.plan(shape[0], shape[1], 0, lo, hi, max_batch)
        out = torch.empty((batch, hi - lo, shape[1]), dtype=tdtype, device="cuda")
        for b0 in range(0, batch, max_batch):
            nb = min(max_batch, batch - b0)
            _native.check(nt.lib.rpsf_apply(plan, dev[b0].data_ptr(), shape[1], shape[0] * shape[1], 0, shape[0],
                                            out[b0].data_ptr(), shape[1], (hi - lo) * shape[1], lo, nb,
                                            _native.current_stream_ptr(torch)))
        return out.cpu().numpy(), nt.plan_info(plan)

    three, info = run(batch)
    assert info["overlap_add"] == "streaming chains"
    assert np.array_equal(run(batch)[0], three)                            # bit-stable across fresh plans
    chunks = {info["overlap_chunks"]}
    for max_batch in (1, 2, 4, 8, 16, 32, 64, 128):
        got, info = run(max_batch)
        assert np.array_equal(got, three), max_batch                       # seams recompute, they do not approximate
        chunks.add(info["overlap_chunks"])
    groups = len({c for _, c in coords if c < shape[1] and c + size > 0})  # patch columns: groups of a row pair's chain
    if groups >= 2:
        assert 1 in chunks and len(chunks) >= 2, chunks
    if shape[0] * shape[1] <= 1_000_000:
        want = np.stack([oracle.apply_transform(f, coords, kernel) for f in frames])[:, lo:hi]
        assert rel_err(three, want, float(frames.max())) <= TOL[dtype]


@pytest.mark.parametrize("shape,size,dtype,batch,pad_mode", [((1024, 1024), 128, "float32", 2, "symmetric"), ((300, 260), 64, "float32", 3, "reflect"),
                                                            ((192, 160), 32, "float64", 2, "wrap"), ((96, 80), 16, "float32", 1, "constant"),
                                                            ((512, 384), 64, "float64", 1, "edge"), ((640, 384), 128, "float32", 5, "symmetric")])
def test_three_kernels_in_every_pad_mode_and_slab_stitching(shape, size, dtype, batch, pad_mode):
    """P <= 128 in every pad mode: the three kernels against the oracle; row slabs stitch bit-identically; repeated calls
    are bit-stable."""
    import torch
    coords = _covering(shape, size)
    rng = np.random.default_rng(23)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    kernel = kernel.astype(np.complex64 if dtype == "float32" else np.complex128)
    frames = np.stack([oracle.starfield(shape, seed=70 + i) for i in range(batch)])
    tdtype = torch.float32 if dtype == "float32" else torch.float64
    dev = torch.from_numpy(frames).to("cuda", tdtype)
    code = _native.PAD_MODES[pad_mode]

    def run(rows=None):
        t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
        nt = t._native_transform(dtype)
        lo, hi = rows if rows else (0, shape[0])
        nt.plan(shape[0], shape[1], code, lo, hi, batch)
        return t._apply_device(dev, dtype, code, row_range=(lo, hi)).cpu().numpy()

    three = run()
    assert np.array_equal(three, run())                                    # bit-stable
    want = np.stack([oracle.apply_transform(f, coords, kernel, pad_mode=pad_mode) for f in frames])
    assert rel_err(three, want, float(frames.max())) <= TOL[dtype]
    from regularizepsf_b200.distributed import slab_bounds
    parts = [run(rows=b) for b in slab_bounds(shape[0], size, 3) if b[1] > b[0]]
    assert np.array_equal(np.concatenate(parts, axis=1), three)


def test_nan_footprint_saturation_and_host_calls_at_64_px():
    coords, kernel, image = _small(shape=(256, 192), size=64, seed=5)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    poisoned = image.copy()
    poisoned[100, 77] = np.nan
    want = oracle.apply_transform(poisoned, coords, kernel)
    got = t.apply(poisoned)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.max(np.abs(got[ok] - want[ok])) <= TOL["float32"] * float(image.max())
    thr = float(np.percentile(image, 99.5))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want_sat = oracle.apply_transform(image, coords, kernel, saturation_threshold=thr, saturation_dilation=2)
    got_sat = t.apply(image, saturation_threshold=thr, saturation_dilation=2)
    assert rel_err(got_sat, want_sat, float(image.max())) <= TOL["float32"]
    hot = image > thr
    assert np.array_equal(got_sat[hot], image[hot].astype(np.float64))


# ------------------------------------------------------------------ programmatic dependent launch (round 2)
@pytest.mark.gpu
@pytest.mark.parametrize("size,shape", [(32, (256, 192)), (256, (1024, 768))])
def test_chained_calls_without_synchronisation_see_the_previous_result(size, shape):
    """The three kernels are launched so that a kernel's CTAs may start while its predecessor drains
    (rpsf_inst.cu: launch_chain).  Feeding each call's output to the next call, with nothing but stream order
    between them, must equal the same chain with the device drained after every call."""
    import torch
    coords, kernel, image = _small(shape=shape, size=size, seed=9)
    kernel = (kernel / np.abs(kernel).max()).astype(np.complex64)            # keeps the iterates bounded
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    start = torch.from_numpy(image.astype(np.float32)).cuda()
    bufs = [torch.empty_like(start) for _ in range(2)]

    def chain(drain):
        x = start
        for i in range(6):
            x = t._apply_device(x, "float32", 0, out=bufs[i % 2])
            if drain:
                torch.cuda.synchronize()
        return x.clone()

    want = chain(True)
    for _ in range(3):
        assert torch.equal(chain(False), want)
    first = t._apply_device(start, "float32", 0).cpu().numpy().astype(np.float64)
    want1 = oracle.apply_transform(image.astype(np.float32), coords, kernel, workers=-1)
    assert rel_err(first, want1, float(image.max())) <= TOL["float32"]


# ------------------------------------------------------------------ pageable batches staged by host threads (round 2)
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float32, np.uint16, np.float64])
def test_pageable_batch_in_several_chunks_equals_frame_by_frame(monkeypatch, dtype):
    """A pageable numpy batch that needs several chunks is staged into pinned buffers by host threads with
    non-temporal stores (rpsf_apply_host: parallel_copy); odd frame sizes and a misaligned base address exercise the
    head / tail handling of the copy.  The result must equal the same frames applied one call at a time.  On a
    host with 8 or more cores (4 copy threads) a float32 frame (4,276,588 bytes) is staged whole as one chunk of the
    batch on 4 threads, and in a single-frame call as one 4 MiB piece on 4 threads, then an 82,284-byte tail on one."""
    shape = (1031, 1037)                                        # > 1 MiB per frame so that several threads split a chunk
    coords, kernel, _ = _small(shape=shape, size=64, seed=13)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    monkeypatch.setattr(t, "HOST_CHUNK_BYTES", 1, raising=False)   # one frame per chunk: 5 chunks through the 3-slot ring
    rng = np.random.default_rng(3)
    raw = np.empty(5 * shape[0] * shape[1] + 3, dtype=dtype)
    frames = raw[3:].reshape(5, *shape)                         # base address off by 3 elements
    frames[...] = (rng.random((5, *shape)) * 1000).astype(dtype)
    got = t.apply(frames)
    assert got.shape == frames.shape and got.dtype == np.float64
    import torch
    for i in range(5):
        # one frame per call: staged in 4 MB pieces when it is at least that large (float32 / float64 here), through
        # the driver's pageable path otherwise (uint16)
        assert np.array_equal(got[i], t.apply(np.ascontiguousarray(frames[i]))), i
    # and no host staging at all: the same frames from a device tensor
    dev = torch.from_numpy(frames.astype(np.float32)).cuda()
    assert np.array_equal(got, t.apply(dev).cpu().numpy().astype(np.float64))


@pytest.mark.gpu
def test_one_and_two_tiles_per_cta_give_the_same_bytes():
    """The column pass walks two adjacent tiles per CTA when a CTA would see a single frame (only P = 256 in float32
    has it).  2048^2 frames, 256 px patches: a batch of 3 gives 289 patches x 8 tiles = 2,312 CTAs of 3 frames each,
    one tile per CTA; a single frame runs two tiles per CTA.  Each frame of the batch equals the frame alone."""
    import torch
    shape, size = (2048, 2048), 256
    coords = _covering(shape, size)
    rng = np.random.default_rng(29)
    kernel = (rng.standard_normal((len(coords), size, size)) + 1j * rng.standard_normal((len(coords), size, size)))
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel.astype(np.complex64)))
    frames = torch.from_numpy(rng.random((3, *shape), dtype=np.float32)).cuda()
    batch = t.apply(frames)
    for i in range(3):
        assert torch.equal(batch[i], t.apply(frames[i])), i


def test_bench_dump_outputs_writes_the_last_step(tmp_path):
    """bench.py --dump-outputs: the device-resident (float32) and host-API (float64) results of the last timed step,
    at the same seeded pixels, within 64 MB, and the pixels bench.py names in its JSON line."""
    import json
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--frames", "1", "--cpu-frames",
                          "1", "--dump-outputs", str(tmp_path)], cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["dump_outputs"]["files"] == ["device_out.npy", "host_out.npy"]
    device, host = np.load(tmp_path / "device_out.npy"), np.load(tmp_path / "host_out.npy")
    idx = bench.dump_indices(bench.H * bench.W)
    assert device.dtype == np.float32 and host.dtype == np.float64
    assert device.shape == host.shape == idx.shape and line["dump_outputs"]["pixels"] == idx.size
    assert device.nbytes + host.nbytes <= 64 << 20
    assert np.all(np.isfinite(device)) and np.array_equal(device.astype(np.float64), host)
