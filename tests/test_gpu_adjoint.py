"""The device transpose of apply (ArrayPSFTransform.apply_adjoint, rpsf_plan_create_adjoint) and autograd of apply.

Tolerances: max |device - oracle| <= 1e-5 (float32) / 1e-10 (float64) x max |oracle|, the reference being
tests/adjoint_oracle.apply_transform_adjoint in float64.
"""
import ctypes

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from tests.adjoint_oracle import apply_transform_adjoint
from regularizepsf_b200 import _native
from tests.helpers import load_golden

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-10}
PAD_MODES = ["symmetric", "reflect", "edge", "wrap", "constant"]


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]


def _kernel(coords, size, shape):
    src = oracle.coma_psf_cube(coords, size, shape)
    tgt = oracle.gaussian_psf_cube(len(coords), size, 3.0)
    return oracle.transfer_kernel(oracle.psf_fft(src), oracle.psf_fft(tgt), 1.0, 0.1)


def _geometry(name):
    if name == "irregular_p16":
        g = load_golden("p16_irregular_coords")
        return g["image"].shape, g["size"], g["coords"]
    shape, size = {"p16": ((64, 48), 16), "p64": ((192, 160), 64), "p256": ((640, 512), 256),
                   "embedded_p21": ((80, 70), 21), "embedded_p48": ((150, 130), 48), "p16_tiny": ((12, 10), 16)}[name]
    return shape, size, _covering(shape, size)


_CACHE = {}


def _setup(name):
    if name not in _CACHE:
        shape, size, coords = _geometry(name)
        _CACHE[name] = (shape, coords, _kernel(coords, size, shape))
    return _CACHE[name]


def _frames(shape, batch, seed):
    return np.random.default_rng(seed).normal(size=(batch,) + tuple(shape))


def _check_against_oracle(t, frames, coords, kernel, pad_mode, dtype):
    import torch
    want = np.stack([apply_transform_adjoint(f, coords, kernel, pad_mode) for f in frames])
    dev = torch.from_numpy(frames).cuda().to(torch.float32 if dtype == "float32" else torch.float64)
    got = t.apply_adjoint(dev, pad_mode=pad_mode, dtype=dtype)
    assert got.dtype == dev.dtype and tuple(got.shape) == frames.shape
    err = float(np.max(np.abs(got.cpu().numpy().astype(np.float64) - want)))
    assert err <= TOL[dtype] * float(np.max(np.abs(want))), (err, float(np.max(np.abs(want))))
    return got


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("name", ["p16", "p64", "p256", "embedded_p21", "embedded_p48", "irregular_p16", "p16_tiny"])
def test_adjoint_matches_oracle(name, pad_mode, batch, dtype):
    shape, coords, kernel = _setup(name)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    _check_against_oracle(t, _frames(shape, batch, seed=batch), coords, kernel, pad_mode, dtype)


def test_adjoint_matches_oracle_2048_p256():
    shape, size = (2048, 2048), 256
    coords = _covering(shape, size)
    kernel = _kernel(coords, size, shape)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    _check_against_oracle(t, _frames(shape, 1, seed=5), coords, kernel, "symmetric", "float32")


def test_numpy_input_returns_float64():
    shape, coords, kernel = _setup("p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    y = _frames(shape, 1, seed=9)[0].astype(np.float32)
    got = t.apply_adjoint(y, pad_mode="reflect")
    assert isinstance(got, np.ndarray) and got.dtype == np.float64 and got.shape == shape
    want = apply_transform_adjoint(y.astype(np.float64), coords, kernel, "reflect")
    assert np.max(np.abs(got - want)) <= TOL["float32"] * np.max(np.abs(want))


@pytest.mark.parametrize("pad_mode", PAD_MODES)
def test_device_dot_product_identity_float64(pad_mode):
    import torch
    shape, coords, kernel = _setup("p64")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x, y = (torch.from_numpy(f).cuda() for f in _frames(shape, 2, seed=11))
    ax = t.apply(x, pad_mode=pad_mode, dtype="float64")
    aty = t.apply_adjoint(y, pad_mode=pad_mode, dtype="float64")
    lhs, rhs = float(torch.sum(ax * y)), float(torch.sum(x * aty))
    assert abs(lhs - rhs) <= 1e-12 * float(torch.linalg.norm(ax) * torch.linalg.norm(y))


@pytest.mark.parametrize("pad_mode", ["symmetric", "constant"])
def test_gradcheck_and_gradgradcheck(pad_mode):
    import torch
    shape, size = (48, 40), 16
    coords = _covering(shape, size)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, _kernel(coords, size, shape)))
    x = torch.from_numpy(_frames(shape, 1, seed=2)[0]).cuda().requires_grad_()
    fn = lambda v: t.apply(v, pad_mode=pad_mode, dtype="float64")      # noqa: E731
    assert torch.autograd.gradcheck(fn, (x,))
    assert torch.autograd.gradgradcheck(fn, (x,), fast_mode=True)
    adj = lambda v: t.apply_adjoint(v, pad_mode=pad_mode, dtype="float64")    # noqa: E731
    assert torch.autograd.gradcheck(adj, (x,), fast_mode=True)


def test_backward_of_sum_is_adjoint_of_ones_bit_for_bit():
    import torch
    shape, coords, kernel = _setup("p64")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x = torch.from_numpy(_frames(shape, 2, seed=4)).cuda().float().requires_grad_()
    out = t.apply(x)
    assert out.grad_fn is not None
    out.sum().backward()
    with torch.no_grad():
        want = t.apply_adjoint(torch.ones_like(x))
    assert x.grad.dtype == x.dtype and torch.equal(x.grad, want)
    # the gradient comes back in the input's dtype
    x16 = torch.from_numpy(_frames(shape, 1, seed=4)[0]).cuda().double().requires_grad_()
    t.apply(x16).sum().backward()
    assert x16.grad.dtype == torch.float64


def test_adjoint_is_run_to_run_bit_stable():
    import torch
    shape, coords, kernel = _setup("irregular_p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    y = torch.from_numpy(_frames(shape, 3, seed=6)).cuda().float()
    first = t.apply_adjoint(y, pad_mode="edge")
    for _ in range(3):
        assert torch.equal(t.apply_adjoint(y, pad_mode="edge"), first)


def test_forward_unchanged_by_an_adjoint_plan():
    import torch
    shape, coords, kernel = _setup("p64")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x = torch.from_numpy(_frames(shape, 2, seed=8)).cuda().float()
    before = t.apply(x)
    t.apply_adjoint(x)
    assert torch.equal(t.apply(x), before)


def test_adjoint_plan_rejects_saturation_mirrors_and_materialised_pad():
    import torch
    shape, coords, kernel = _setup("p256")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    nt = t._native_transform("float32")
    plan = nt.plan(shape[0], shape[1], 0, 0, shape[0], 2, adjoint=True)
    lib = nt.lib
    assert lib.rpsf_plan_set_saturation(plan, 10.0, 1, 7) == _native.E_UNSUPPORTED
    assert lib.rpsf_plan_set_saturation(plan, float("inf"), 1, 7) == 0
    mirror = torch.empty(1, device="cuda")
    arr = (ctypes.c_void_p * 1)(mirror.data_ptr())
    assert lib.rpsf_plan_set_output_mirrors(plan, 1, arr) == _native.E_UNSUPPORTED
    out = ctypes.c_void_p()
    assert lib.rpsf_plan_create_adjoint(ctypes.byref(out), nt.handle, shape[0], shape[1], 5, 1) == _native.E_UNSUPPORTED


def test_not_differentiable_cases_raise_only_when_a_gradient_is_required():
    import torch
    shape, coords, kernel = _setup("p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x = torch.from_numpy(_frames(shape, 1, seed=1)[0]).cuda().float()
    xg = x.clone().requires_grad_()
    with pytest.raises(NotImplementedError, match="saturation"):
        t.apply(xg, saturation_threshold=1.0)
    with pytest.raises(NotImplementedError, match="pad mode"):
        t.apply(xg, pad_mode="mean")
    t.apply(x, saturation_threshold=1.0)                              # no gradient needed: as before
    t.apply(x, pad_mode="mean")
    keep = np.zeros(len(coords), dtype=bool)
    keep[: len(coords) // 2] = True
    shard = rp.ArrayPSFTransform.sharded(rp.IndexedCube([c for c, k in zip(coords, keep) if k], kernel[keep]), coords, keep)
    with pytest.raises(NotImplementedError, match="sharded"):
        shard.apply(xg)


def test_no_graph_without_grad():
    import torch
    shape, coords, kernel = _setup("p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    xg = torch.from_numpy(_frames(shape, 1, seed=1)[0]).cuda().float().requires_grad_()
    with torch.no_grad():
        assert t.apply(xg).grad_fn is None
        assert t.apply_adjoint(xg).grad_fn is None
    assert t.apply(xg.detach()).grad_fn is None
    assert t.apply_adjoint(xg).grad_fn is not None
