"""The gradient of apply with respect to the transfer kernel (transfer_kernel_gradient, rpsf_kernel_gradient, autograd).

Tolerances: max |device - oracle| <= 1e-5 (float32) / 1e-10 (float64) x max |oracle|, the reference being
tests/kernel_gradient_oracle.transfer_kernel_gradient in float64.
"""
import ctypes

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native
from tests.helpers import load_golden
from tests.kernel_gradient_oracle import transfer_kernel_gradient

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
        return g["image"].shape, int(g["size"]), [tuple(int(v) for v in c) for c in g["coords"]]
    shape, size = {"p16": ((64, 48), 16), "p64": ((192, 160), 64), "p256": ((640, 512), 256),
                   "p512": ((1024, 1024), 512), "p16_tiny": ((12, 10), 16)}[name]
    return shape, size, _covering(shape, size)


_CACHE = {}


def _setup(name):
    if name not in _CACHE:
        shape, size, coords = _geometry(name)
        _CACHE[name] = (shape, size, coords, _kernel(coords, size, shape))
    return _CACHE[name]


def _frames(shape, batch, seed):
    return np.random.default_rng(seed).normal(size=(batch,) + tuple(shape))


def _check_against_oracle(t, x, g, coords, size, pad_mode, dtype):
    import torch
    want = transfer_kernel_gradient(x, g, coords, size, pad_mode)
    real = torch.float32 if dtype == "float32" else torch.float64
    got = t.transfer_kernel_gradient(torch.from_numpy(x).cuda().to(real), torch.from_numpy(g).cuda().to(real),
                                     pad_mode=pad_mode, dtype=dtype)
    assert got.dtype == (torch.complex64 if dtype == "float32" else torch.complex128)
    assert tuple(got.shape) == want.shape
    err = float(np.max(np.abs(got.cpu().numpy().astype(np.complex128) - want)))
    assert err <= TOL[dtype] * float(np.max(np.abs(want))), (err, float(np.max(np.abs(want))))
    return got


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("batch", [1, 3])
@pytest.mark.parametrize("pad_mode", PAD_MODES)
@pytest.mark.parametrize("name", ["p16", "p64", "p256", "p512", "irregular_p16", "p16_tiny"])
def test_kernel_gradient_matches_oracle(name, pad_mode, batch, dtype):
    shape, size, coords, kernel = _setup(name)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x, g = _frames(shape, batch, seed=batch), _frames(shape, batch, seed=batch + 10)
    _check_against_oracle(t, x, g, coords, size, pad_mode, dtype)


def test_kernel_gradient_matches_oracle_2048_p256():
    shape, size = (2048, 2048), 256
    coords = _covering(shape, size)
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, _kernel(coords, size, shape)))
    _check_against_oracle(t, _frames(shape, 1, seed=5), _frames(shape, 1, seed=6), coords, size, "symmetric", "float32")


def test_numpy_input_returns_complex128():
    shape, size, coords, kernel = _setup("p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    x, g = _frames(shape, 1, seed=9)[0].astype(np.float32), _frames(shape, 1, seed=19)[0]
    got = t.transfer_kernel_gradient(x, g, pad_mode="reflect")
    assert isinstance(got, np.ndarray) and got.dtype == np.complex128 and got.shape == kernel.shape
    want = transfer_kernel_gradient(x.astype(np.float64), g, coords, size, "reflect")
    assert np.max(np.abs(got - want)) <= TOL["float32"] * np.max(np.abs(want))


@pytest.mark.parametrize("pad_mode", PAD_MODES)
def test_device_linearity_identity_float64(pad_mode):
    # sum_b <apply_D(x_b), g_b> = Re sum conj(grad) D for any complex cube D: apply is linear in the kernel
    import torch
    shape, size, coords, _ = _setup("p64")
    rng = np.random.default_rng(11)
    d = rng.normal(size=(len(coords), size, size)) + 1j * rng.normal(size=(len(coords), size, size))
    x, g = (torch.from_numpy(f).cuda() for f in (_frames(shape, 2, seed=12), _frames(shape, 2, seed=13)))
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, d))
    ax = t.apply(x, pad_mode=pad_mode, dtype="float64")
    grad = t.transfer_kernel_gradient(x, g, pad_mode=pad_mode, dtype="float64")
    lhs = float(torch.sum(ax * g))
    rhs = float(torch.sum(torch.real(torch.conj(grad) * torch.from_numpy(d).cuda())))
    assert abs(lhs - rhs) <= 1e-12 * float(torch.linalg.norm(ax) * torch.linalg.norm(g))


@pytest.mark.parametrize("pad_mode", ["symmetric", "constant"])
def test_gradcheck_in_the_kernel(pad_mode):
    import torch
    shape, size = (48, 40), 16
    coords = _covering(shape, size)
    x = torch.from_numpy(_frames(shape, 1, seed=2)[0]).cuda()
    k = torch.from_numpy(_kernel(coords, size, shape)).cuda().requires_grad_()

    def fn(kernel):
        # a fresh transform per call: gradcheck's perturbations need not bump the tensor's version
        return rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel)).apply(x, pad_mode=pad_mode, dtype="float64")

    assert torch.autograd.gradcheck(fn, (k,), fast_mode=True)


def test_backward_is_adjoint_and_kernel_gradient_bit_for_bit():
    import torch
    shape, size, coords, kernel = _setup("p64")
    k = torch.from_numpy(kernel).cuda().requires_grad_()               # complex128 kernel, float32 compute
    t = rp.ArrayPSFTransform(rp.DeviceCube(coords, k))
    x = torch.from_numpy(_frames(shape, 2, seed=4)).cuda().float().requires_grad_()
    g = torch.from_numpy(_frames(shape, 2, seed=14)).cuda().float()
    out = t.apply(x)
    assert out.grad_fn is not None and out.dtype == torch.float32
    out.backward(g)
    with torch.no_grad():
        want_x = t.apply_adjoint(g)
        want_k = t.transfer_kernel_gradient(x.detach(), g)
    assert x.grad.dtype == x.dtype and torch.equal(x.grad, want_x)
    assert k.grad.dtype == torch.complex128 and torch.equal(k.grad, want_k.to(torch.complex128))
    # the transpose: its kernel gradient is transfer_kernel_gradient with the roles swapped
    k.grad = None
    y = torch.from_numpy(_frames(shape, 1, seed=24)[0]).cuda().float()
    v = torch.from_numpy(_frames(shape, 1, seed=25)[0]).cuda().float()
    t.apply_adjoint(y).backward(v)
    with torch.no_grad():
        want_k = t.transfer_kernel_gradient(v, y)
    assert torch.equal(k.grad, want_k.to(torch.complex128))


def test_kernel_gradient_and_forward_are_bit_stable():
    import torch
    shape, size, coords, kernel = _setup("irregular_p16")
    k = torch.from_numpy(kernel).cuda().requires_grad_()
    t = rp.ArrayPSFTransform(rp.DeviceCube(coords, k))
    x = torch.from_numpy(_frames(shape, 3, seed=6)).cuda().float()
    g = torch.from_numpy(_frames(shape, 3, seed=7)).cuda().float()
    first = t.transfer_kernel_gradient(x, g, pad_mode="edge")
    for _ in range(3):
        assert torch.equal(t.transfer_kernel_gradient(x, g, pad_mode="edge"), first)
    out = t.apply(x, pad_mode="edge")
    assert out.grad_fn is not None
    with torch.no_grad():
        assert torch.equal(out.detach(), t.apply(x, pad_mode="edge"))


def test_in_place_kernel_update_is_applied():
    import torch
    shape, size, coords, kernel = _setup("p64")
    k = torch.from_numpy(kernel).cuda().to(torch.complex64).requires_grad_()
    cube = rp.DeviceCube(coords, k)
    t = rp.ArrayPSFTransform(cube)
    x = torch.from_numpy(_frames(shape, 2, seed=3)).cuda().float()
    target = torch.from_numpy(_frames(shape, 2, seed=33)).cuda().float()
    before_values = cube.values.copy()
    with torch.no_grad():
        before = t.apply(x)
    opt = torch.optim.SGD([k], lr=1e-3)
    loss = (t.apply(x) - target).square().sum()
    loss.backward()
    opt.step()
    with torch.no_grad():
        after = t.apply(x)
        fresh = rp.ArrayPSFTransform(rp.DeviceCube(coords, k.detach().clone())).apply(x)
    assert not torch.equal(after, before)
    assert torch.equal(after, fresh)
    assert np.array_equal(cube.values, k.detach().cpu().numpy()) and not np.array_equal(cube.values, before_values)


def _reads(corner, size, shape, pad_mode, pixel):
    rows = [oracle_pad_index(corner[0] + i, shape[0], pad_mode) for i in range(size)]
    cols = [oracle_pad_index(corner[1] + i, shape[1], pad_mode) for i in range(size)]
    return pixel[0] in rows and pixel[1] in cols


def oracle_pad_index(i, n, pad_mode):
    extra = {"constant_values": -1} if pad_mode == "constant" else {}
    pad = 4 * n + abs(i)
    return int(np.pad(np.arange(n), (pad, pad), mode=pad_mode, **extra)[i + pad])


@pytest.mark.parametrize("pad_mode", ["reflect", "wrap"])
def test_nan_poisons_exactly_the_patches_that_read_it(pad_mode):
    import torch
    shape, size, coords, kernel = _setup("p16")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    frame = _frames(shape, 1, seed=8)[0]
    pixel = (1, 0)
    frame[pixel] = np.nan
    x = torch.from_numpy(frame).cuda().float()
    g = torch.from_numpy(_frames(shape, 1, seed=18)[0]).cuda().float()
    grad = t.transfer_kernel_gradient(x, g, pad_mode=pad_mode).cpu().numpy()
    reads = np.array([_reads(c, size, shape, pad_mode, pixel) for c in coords])
    assert reads.any() and not reads.all()
    for i in range(len(coords)):
        if reads[i]:
            assert np.isnan(grad[i]).any(), i
        else:
            assert np.isfinite(grad[i]).all(), i


def test_unsupported_cases_raise_only_when_a_kernel_gradient_is_required():
    import torch
    shape, size, coords, kernel = _setup("p16")
    k = torch.from_numpy(kernel).cuda().requires_grad_()
    t = rp.ArrayPSFTransform(rp.DeviceCube(coords, k))
    x = torch.from_numpy(_frames(shape, 1, seed=1)[0]).cuda().float()
    with pytest.raises(NotImplementedError, match="saturation"):
        t.apply(x, saturation_threshold=1.0)
    with pytest.raises(NotImplementedError, match="pad mode"):
        t.apply(x, pad_mode="mean")
    with torch.no_grad():                                               # no gradient needed: as before
        t.apply(x, saturation_threshold=1.0)
        t.apply(x, pad_mode="mean")
    esize = 21
    ecoords = _covering(shape, esize)
    ek = torch.from_numpy(_kernel(ecoords, esize, shape)).cuda()
    embedded = rp.ArrayPSFTransform(rp.DeviceCube(ecoords, ek.clone().requires_grad_()))
    with pytest.raises(NotImplementedError, match="embedded"):
        embedded.apply(x)
    with torch.no_grad():
        embedded.apply(x)
    # the image gradient of an embedded transform still works when the kernel is fixed
    xg = x.clone().requires_grad_()
    rp.ArrayPSFTransform(rp.DeviceCube(ecoords, ek)).apply(xg).sum().backward()
    assert xg.grad is not None
    keep = np.zeros(len(coords), dtype=bool)
    keep[: len(coords) // 2] = True
    shard = rp.ArrayPSFTransform.sharded(rp.DeviceCube([c for c, kk in zip(coords, keep) if kk],
                                                       k.detach()[torch.from_numpy(keep).cuda()].requires_grad_()),
                                         coords, keep)
    with pytest.raises(NotImplementedError, match="sharded"):
        shard.apply(x)


def _call(lib, adjoint, forward, x, g, batch, out):
    h = x.shape[-2]
    return lib.rpsf_kernel_gradient(adjoint, forward, x.data_ptr(), x.stride(-2), h * x.stride(-2), g.data_ptr(),
                                    g.stride(-2), h * g.stride(-2), batch, out.data_ptr(),
                                    _native.current_stream_ptr(__import__("torch")))


def test_c_entry_point_status_codes():
    import torch
    shape, size, coords, kernel = _setup("p16")
    h, w = shape
    x = torch.from_numpy(_frames(shape, 2, seed=1)).cuda().float()
    out = torch.empty((len(coords), size, size), dtype=torch.complex64, device="cuda")
    t = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))
    nt = t._native_transform("float32")
    lib = nt.lib
    fwd = nt.plan(h, w, 0, 0, h, 2)
    adj = nt.plan(h, w, 0, 0, h, 2, adjoint=True)
    nt.set_saturation(fwd, (float("inf"), 1, 7))
    assert _call(lib, adj, fwd, x, x, 2, out) == 0
    assert _call(lib, fwd, adj, x, x, 2, out) == _native.E_INVALID_ARGUMENT          # plans swapped
    assert _call(lib, adj, fwd, x, x, 3, out) == _native.E_INVALID_ARGUMENT          # batch above capacity
    assert _call(lib, adj, nt.plan(h, w, 1, 0, h, 2), x, x, 2, out) == _native.E_INVALID_ARGUMENT   # pad modes differ
    assert _call(lib, adj, nt.plan(h, w - 2, 0, 0, h, 2), x, x, 2, out) == _native.E_INVALID_ARGUMENT  # shapes differ
    other = rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel))._native_transform("float32")
    assert _call(lib, adj, other.plan(h, w, 0, 0, h, 2), x, x, 2, out) == _native.E_INVALID_ARGUMENT  # transforms differ
    assert _call(lib, adj, nt.plan(h, w, 0, 0, h // 2, 2), x, x, 2, out) == _native.E_UNSUPPORTED     # row band
    assert _call(lib, adj, nt.plan(h, w, 5, 0, h, 2), x, x, 2, out) == _native.E_UNSUPPORTED          # materialised pad
    sat = nt.plan(h, w, 0, 0, h, 1)
    nt.set_saturation(sat, (10.0, 1, 7))
    assert _call(lib, adj, sat, x, x, 1, out) == _native.E_UNSUPPORTED                               # saturation
    nt.set_saturation(sat, (float("inf"), 1, 7))
    # embedded patch size
    ecoords = _covering(shape, 21)
    et = rp.ArrayPSFTransform(rp.IndexedCube(ecoords, _kernel(ecoords, 21, shape)))._native_transform("float32")
    eout = torch.empty((len(ecoords), 21, 21), dtype=torch.complex64, device="cuda")
    assert _call(lib, et.plan(h, w, 0, 0, h, 1, adjoint=True), et.plan(h, w, 0, 0, h, 1), x, x, 1,
                 eout) == _native.E_UNSUPPORTED
    # a shard that holds every patch touching the frame, but not a patch outside it
    scoords = coords + [(-20, 0)]
    keep = np.ones(len(scoords), dtype=bool)
    keep[-1] = False
    shard = rp.ArrayPSFTransform.sharded(rp.IndexedCube(coords, kernel), scoords, keep)._native_transform("float32")
    sout = torch.empty((len(scoords), size, size), dtype=torch.complex64, device="cuda")
    assert _call(lib, shard.plan(h, w, 0, 0, h, 1, adjoint=True), shard.plan(h, w, 0, 0, h, 1), x, x, 1,
                 sout) == _native.E_UNSUPPORTED
    torch.cuda.synchronize()


def test_double_backward_raises_through_the_kernel_and_works_for_the_image_only():
    import torch
    shape, size = (48, 40), 16
    coords = _covering(shape, size)
    kernel = torch.from_numpy(_kernel(coords, size, shape)).cuda()
    x = torch.from_numpy(_frames(shape, 1, seed=2)[0]).cuda().requires_grad_()
    t = rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel.clone().requires_grad_()))
    (gx,) = torch.autograd.grad(t.apply(x, dtype="float64").square().sum(), x, create_graph=True)
    with pytest.raises(RuntimeError, match="differentiate twice"):
        gx.sum().backward()
    fixed = rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel))
    fn = lambda v: fixed.apply(v, dtype="float64")      # noqa: E731
    assert torch.autograd.gradgradcheck(fn, (x,), fast_mode=True)
