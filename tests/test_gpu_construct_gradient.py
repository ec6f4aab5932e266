"""The gradient of construct and of the PSF FFT cube (rpsf_construct_kernel_backward, rpsf_psf_fft2_adjoint, autograd
through ArrayPSFTransform.construct / reconstruct).

Reference: tests/construct_gradient_oracle.py in float64, given the same (rounded) inputs.  Bars: max |device - oracle|
<= 1e-10 x max |oracle| in float64; in float32 1e-5 x max |oracle| for the cubes and 1e-4 relative for grad_alpha and
grad_eps.  Each parity test prints the error it reached ("reached: ...", visible with pytest -s).
"""
import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native
from tests.construct_gradient_oracle import construct_vjp, psf_fft_vjp

pytestmark = pytest.mark.gpu

CUBE_TOL = {"float32": 1e-5, "float64": 1e-10}
SCALAR_TOL = {"float32": 1e-4, "float64": 1e-10}


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


def _torch():
    import torch
    return torch


def _geometry(size):
    shape = {16: (64, 48), 64: (192, 160), 256: (2048, 2048), 512: (1024, 1024)}[size]
    return shape, [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]


_PSFS = {}


def _psf_values(size):
    """coma source and Gaussian target value cubes (float64 numpy) on the covering of _geometry(size)."""
    if size not in _PSFS:
        shape, coords = _geometry(size)
        _PSFS[size] = (coords, oracle.coma_psf_cube(coords, size, shape), oracle.gaussian_psf_cube(len(coords), size, 3.0))
    return _PSFS[size]


def _codes(dtype):
    torch = _torch()
    return ((torch.float32, torch.complex64, _native.F32) if dtype == "float32"
            else (torch.float64, torch.complex128, _native.F64))


def _native_backward(s, t, g, alpha, epsilon, want_s=True, want_t=True, want_scalars=True):
    """rpsf_construct_kernel_backward on CUDA tensors: (grad_s, grad_t, (grad_alpha, grad_eps)), None where not asked."""
    torch = _torch()
    code = _native.F32 if s.dtype == torch.complex64 else _native.F64
    gs = torch.full_like(s, complex(7, 7)) if want_s else None
    gt = torch.full_like(t, complex(7, 7)) if want_t else None
    ae = torch.full((2,), 7.0, dtype=torch.float64, device=s.device) if want_scalars else None
    _native.check(_native.load().rpsf_construct_kernel_backward(
        s.data_ptr(), t.data_ptr(), g.data_ptr(), s.numel(), code, alpha, epsilon,
        gs.data_ptr() if want_s else None, gt.data_ptr() if want_t else None, ae.data_ptr() if want_scalars else None,
        s.device.index, _native.current_stream_ptr(torch)))
    return gs, gt, ae


def _native_fft_adjoint(g, real):
    torch = _torch()
    n, p, _ = g.shape
    out = torch.empty(g.shape, dtype=real, device=g.device)
    code = _native.F32 if real == torch.float32 else _native.F64
    _native.check(_native.load().rpsf_psf_fft2_adjoint(g.data_ptr(), out.data_ptr(), n, p, code, g.device.index,
                                                         _native.current_stream_ptr(torch)))
    return out


def _random_complex(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=shape) + 1j * rng.normal(size=shape)


def _err(got, want):
    return float(np.max(np.abs(got - want)))


# --------------------------------------------------------------------------------------------- oracle parity
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("size,alpha,epsilon", [(16, 0.5, 0.05), (64, 1.5, 1.0), (256, 1.0, 0.1), (512, 3.0, 0.2)])
def test_entry_points_match_the_oracle(size, alpha, epsilon, dtype):
    torch = _torch()
    real, cplx, _ = _codes(dtype)
    coords, sv, tv = _psf_values(size)
    sv_t, tv_t = torch.from_numpy(sv).cuda().to(real), torch.from_numpy(tv).cuda().to(real)
    s = rp.ArrayPSF(rp.DeviceCube(coords, sv_t)).fft_cube.tensor
    t = rp.ArrayPSF(rp.DeviceCube(coords, tv_t)).fft_cube.tensor
    g = torch.from_numpy(_random_complex(s.shape, size)).cuda().to(cplx)
    gs, gt, ae = _native_backward(s, t, g, alpha, epsilon)
    s_np, t_np, g_np = (x.cpu().numpy().astype(np.complex128) for x in (s, t, g))
    want_s, want_t, want_a, want_e = construct_vjp(s_np, t_np, g_np, alpha, epsilon)
    scale = max(np.abs(want_s).max(), np.abs(want_t).max())
    err_s = _err(gs.cpu().numpy().astype(np.complex128), want_s)
    err_t = _err(gt.cpu().numpy().astype(np.complex128), want_t)
    got_a, got_e = ae.cpu().tolist()
    rel_a, rel_e = abs(got_a - want_a) / abs(want_a), abs(got_e - want_e) / abs(want_e)
    # the FFT adjoint of the same incoming gradient
    want_x = psf_fft_vjp(g_np)
    err_x = _err(_native_fft_adjoint(g, real).cpu().numpy().astype(np.float64), want_x)
    print(f"\nreached: P={size} {dtype} alpha={alpha} eps={epsilon}: grad_S {err_s / scale:.2e}, grad_T "
          f"{err_t / scale:.2e} (x max|oracle|), grad_alpha {rel_a:.2e}, grad_eps {rel_e:.2e} (relative), FFT VJP "
          f"{err_x / np.abs(want_x).max():.2e} (x max|oracle|)")
    assert np.all(np.isfinite(want_s)) and np.all(np.isfinite(want_t))
    assert err_s <= CUBE_TOL[dtype] * scale and err_t <= CUBE_TOL[dtype] * scale, (err_s, err_t, scale)
    assert rel_a <= SCALAR_TOL[dtype] and rel_e <= SCALAR_TOL[dtype], (got_a, want_a, got_e, want_e)
    assert err_x <= CUBE_TOL[dtype] * np.abs(want_x).max()


def _special_cube(seed):
    """Random bins plus S = 0, T = 0, S = T = 0 (0/0 in K), NaN and inf inputs, each with G = 0 and with G != 0."""
    rng = np.random.default_rng(seed)
    n = 4096
    s, t, g = _random_complex(n, seed), _random_complex(n, seed + 1), _random_complex(n, seed + 2)
    cases = [("s0", 0, None), ("t0", None, 0), ("st0", 0, 0), ("snan", np.nan, None), ("tinf", None, np.inf)]
    pos = 0
    for _, sval, tval in cases:
        for g_zero in (True, False):
            for _ in range(8):
                if sval is not None:
                    s[pos] = sval
                if tval is not None:
                    t[pos] = tval
                if g_zero:
                    g[pos] = 0
                pos += 1
    g[pos:pos + 16] = 0                                         # ordinary bins with G = 0
    perm = rng.permutation(n)
    return s[perm], t[perm], g[perm]


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("alpha,epsilon", [(1.0, 0.2), (1.5, 0.2), (0.5, 0.2), (1.0, 0.0)])
def test_special_bins_match_the_oracle_pattern(alpha, epsilon, dtype):
    torch = _torch()
    _, cplx, _ = _codes(dtype)
    s_np, t_np, g_np = _special_cube(3)
    s, t, g = (torch.from_numpy(x).cuda().to(cplx) for x in (s_np, t_np, g_np))
    gs, gt, ae = _native_backward(s, t, g, alpha, epsilon)
    s_np, t_np, g_np = (x.cpu().numpy().astype(np.complex128) for x in (s, t, g))
    want_s, want_t, want_a, want_e = construct_vjp(s_np, t_np, g_np, alpha, epsilon)
    got_s, got_t = gs.cpu().numpy().astype(np.complex128), gt.cpu().numpy().astype(np.complex128)
    for got, want in ((got_s, want_s), (got_t, want_t)):
        for part in (np.real, np.imag):
            np.testing.assert_array_equal(np.isfinite(part(got)), np.isfinite(part(want)))
            np.testing.assert_array_equal(part(got) == 0, part(want) == 0)
        finite = np.isfinite(want)
        assert _err(got[finite], want[finite]) <= CUBE_TOL[dtype] * np.abs(want[finite]).max()
    zero = g_np == 0
    assert np.all(got_s[zero] == 0) and np.all(got_t[zero] == 0)
    got_a, got_e = ae.cpu().tolist()
    assert not np.isfinite(want_a) and not np.isfinite(got_a) and not np.isfinite(got_e)   # the G != 0 0/0 bins
    # without the bins where K is not finite under G != 0, the sums are finite and match
    keep = zero | np.isfinite(oracle.transfer_kernel(s_np, t_np, alpha, epsilon))
    s2, t2, g2 = (torch.from_numpy(np.ascontiguousarray(x[keep])).cuda().to(cplx) for x in (s_np, t_np, g_np))
    _, _, ae2 = _native_backward(s2, t2, g2, alpha, epsilon, want_s=False, want_t=False)
    _, _, want_a, want_e = construct_vjp(s_np[keep], t_np[keep], g_np[keep], alpha, epsilon)
    got_a, got_e = ae2.cpu().tolist()
    for got, want in ((got_a, want_a), (got_e, want_e)):
        assert np.isfinite(got) and abs(got - want) <= SCALAR_TOL[dtype] * max(abs(want), 1e-300)
    if epsilon == 0:
        assert got_a == 0 and got_e == 0


def test_nullable_outputs_and_status_codes():
    torch = _torch()
    s = torch.from_numpy(_random_complex(1000, 1)).cuda()
    t = torch.from_numpy(_random_complex(1000, 2)).cuda()
    g = torch.from_numpy(_random_complex(1000, 3)).cuda()
    full = _native_backward(s, t, g, 1.5, 0.2)
    only_s = _native_backward(s, t, g, 1.5, 0.2, want_t=False, want_scalars=False)
    only_scalars = _native_backward(s, t, g, 1.5, 0.2, want_s=False, want_t=False)
    assert torch.equal(full[0], only_s[0]) and torch.equal(full[2], only_scalars[2])
    lib = _native.load()
    stream = _native.current_stream_ptr(torch)
    ae = torch.full((2,), 7.0, dtype=torch.float64, device="cuda")
    assert lib.rpsf_construct_kernel_backward(None, None, None, 0, _native.F64, 1.0, 0.1, None, None, ae.data_ptr(), 0,
                                              stream) == 0
    assert ae.tolist() == [0.0, 0.0]                              # an empty cube has zero sums
    assert lib.rpsf_construct_kernel_backward(None, t.data_ptr(), g.data_ptr(), 10, _native.F64, 1.0, 0.1, None, None,
                                              None, 0, stream) == _native.E_INVALID_ARGUMENT
    assert lib.rpsf_construct_kernel_backward(s.data_ptr(), t.data_ptr(), g.data_ptr(), 10, 7, 1.0, 0.1, None, None,
                                              None, 0, stream) == _native.E_UNSUPPORTED
    x = torch.empty((2, 21, 21), dtype=torch.float64, device="cuda")
    gc = torch.zeros((2, 21, 21), dtype=torch.complex128, device="cuda")
    assert lib.rpsf_psf_fft2_adjoint(gc.data_ptr(), x.data_ptr(), 2, 21, _native.F64, 0, stream) == _native.E_UNSUPPORTED
    assert lib.rpsf_psf_fft2_adjoint(None, x.data_ptr(), 2, 16, _native.F64, 0, stream) == _native.E_INVALID_ARGUMENT
    assert lib.rpsf_psf_fft2_adjoint(gc.data_ptr(), x.data_ptr(), 2, 16, 3, 0, stream) == _native.E_UNSUPPORTED


# --------------------------------------------------------------------------------------------- autograd
def _fit_setup(size=16, dtype=None, seed=0, target_fwhm=None):
    """Source / target value tensors that require grad, alpha and epsilon as 0-d CUDA tensors, and a frame.

    ``target_fwhm`` replaces the target by a narrower Gaussian: with FWHM 3 px, |T| falls to 4e-7 in the corners of the
    spectrum and K varies on the scale of eps |T| there, too fine for finite differences."""
    torch = _torch()
    real = dtype or torch.float64
    coords, sv, tv = _psf_values(size)
    if target_fwhm is not None:
        tv = oracle.gaussian_psf_cube(len(coords), size, target_fwhm)
    shape, _ = _geometry(size)
    sv_t = torch.from_numpy(sv).cuda().to(real).requires_grad_()
    tv_t = torch.from_numpy(tv).cuda().to(real).requires_grad_()
    alpha = torch.tensor(1.3, dtype=torch.float64, device="cuda", requires_grad=True)
    epsilon = torch.tensor(0.1, dtype=torch.float64, device="cuda", requires_grad=True)
    x = torch.from_numpy(np.random.default_rng(seed).normal(size=shape)).cuda().to(real)
    return coords, sv_t, tv_t, alpha, epsilon, x


def test_gradcheck_through_construct_and_apply():
    torch = _torch()
    coords, sv, tv, alpha, epsilon, x = _fit_setup(16, target_fwhm=1.0)
    w = torch.from_numpy(np.random.default_rng(9).normal(size=tuple(x.shape))).cuda() / x.numel()

    def f(sv_, tv_, a_, e_):
        transform = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, sv_)),
                                                   rp.ArrayPSF(rp.DeviceCube(coords, tv_)), a_, e_)
        return (transform.apply(x, dtype="float64") * w).sum()

    assert torch.autograd.gradcheck(f, (sv, tv, alpha, epsilon), eps=1e-6, atol=1e-7, rtol=1e-4, fast_mode=True)


def test_directional_derivative_at_config2_in_float64():
    torch = _torch()
    coords, sv, tv, _, epsilon, x = _fit_setup(256)
    alpha = torch.tensor(1.0, dtype=torch.float64, device="cuda", requires_grad=True)
    target = rp.ArrayPSF(rp.DeviceCube(coords, tv.detach()))
    w = torch.from_numpy(np.random.default_rng(11).normal(size=tuple(x.shape))).cuda()
    # a change of each patch's flux and of the coma core: a random direction would move the bins where |S| is 1e-20 by
    # far more than eps |T| (4e-8), where K is not smooth on the scale of a difference step
    shape, _ = _geometry(256)
    values = sv.detach().cpu().numpy()
    flux = np.random.default_rng(12).normal(size=(len(coords), 1, 1))
    direction = torch.from_numpy(flux * values + oracle.coma_psf_cube(coords, 256, shape, core_sigma=2.7) - values).cuda()
    da, de = 0.3, 0.05

    def loss(values, a, e):
        t = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, values)), target, a, e)
        return (t.apply(x, dtype="float64") * w).sum()

    loss(sv, alpha, epsilon).backward()
    analytic = float((sv.grad * direction).sum() + alpha.grad * da + epsilon.grad * de)
    h = 1e-4
    with torch.no_grad():
        up = float(loss(sv + h * direction, 1.0 + h * da, 0.1 + h * de))
        down = float(loss(sv - h * direction, 1.0 - h * da, 0.1 - h * de))
    numeric = (up - down) / (2 * h)
    print(f"\nreached: config-2 float64 directional derivative {analytic:.12e} vs central difference {numeric:.12e}")
    assert abs(analytic - numeric) <= 1e-5 * abs(numeric)


def test_backward_is_bit_stable():
    torch = _torch()
    coords, sv, tv, alpha, epsilon, x = _fit_setup(64)

    def grads():
        for p in (sv, tv, alpha, epsilon):
            p.grad = None
        t = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, sv)), rp.ArrayPSF(rp.DeviceCube(coords, tv)),
                                           alpha, epsilon)
        (t.apply(x, dtype="float64") ** 2).sum().backward()
        return [p.grad.clone() for p in (sv, tv, alpha, epsilon)]

    first, second = grads(), grads()
    for a, b in zip(first, second):
        assert torch.equal(a, b)
    # and the entry point on a full config-2 cube, float32
    s = torch.from_numpy(_random_complex((289, 256, 256), 1)).cuda().to(torch.complex64)
    t = torch.from_numpy(_random_complex((289, 256, 256), 2)).cuda().to(torch.complex64)
    g = torch.from_numpy(_random_complex((289, 256, 256), 3)).cuda().to(torch.complex64)
    one, two = _native_backward(s, t, g, 1.5, 0.2), _native_backward(s, t, g, 1.5, 0.2)
    for a, b in zip(one, two):
        assert torch.equal(a, b)


def test_gradients_come_back_in_each_inputs_dtype():
    torch = _torch()
    coords, sv, tv, alpha, epsilon, x = _fit_setup(16, dtype=torch.float32)
    tv64 = tv.detach().double().requires_grad_()
    alpha32 = torch.tensor(1.3, dtype=torch.float32, requires_grad=True)          # a CPU scalar
    t = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, sv)), rp.ArrayPSF(rp.DeviceCube(coords, tv64)),
                                       alpha32, epsilon)
    assert t._kernel_tensor.dtype == torch.complex128 and t._kernel_tensor.requires_grad
    t.apply(x).sum().backward()
    assert sv.grad.dtype == torch.float32 and tv64.grad.dtype == torch.float64
    assert alpha32.grad.dtype == torch.float32 and alpha32.grad.device.type == "cpu"
    assert epsilon.grad.dtype == torch.float64 and epsilon.grad.is_cuda
    # a DeviceCube FFT cube that requires grad is differentiated directly
    spectrum = rp.ArrayPSF(rp.DeviceCube(coords, sv.detach())).fft_cube.tensor.clone().requires_grad_()
    given = rp.ArrayPSF(rp.IndexedCube(coords, sv.detach().cpu().numpy()), rp.DeviceCube(coords, spectrum))
    t = rp.ArrayPSFTransform.construct(given, rp.ArrayPSF(rp.DeviceCube(coords, tv.detach())), 1.3, 0.1)
    t.apply(x).sum().backward()
    assert spectrum.grad is not None and spectrum.grad.dtype == torch.complex64


# --------------------------------------------------------------------------------------------- unchanged paths
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_construct_without_grad_is_the_plain_kernel(dtype):
    torch = _torch()
    real, _, code = _codes(dtype)
    coords, sv, tv = _psf_values(64)
    sv_t = torch.from_numpy(sv).cuda().to(real)
    host = rp.ArrayPSF(rp.IndexedCube(coords, sv_t.cpu().numpy()))
    device = rp.ArrayPSF(rp.DeviceCube(coords, sv_t))
    assert torch.equal(host.fft_cube.tensor, device.fft_cube.tensor)                 # the same FFT either way
    target = rp.ArrayPSF(rp.IndexedCube(coords, tv.astype(sv_t.cpu().numpy().dtype)))
    s, t = device.fft_cube.tensor, target.fft_cube.tensor
    want = torch.empty_like(s)
    _native.check(_native.load().rpsf_construct_kernel(s.data_ptr(), t.data_ptr(), want.data_ptr(), s.numel(), code, 1.5,
                                                       0.2, 0, _native.current_stream_ptr(torch)))
    for a, e in ((1.5, 0.2), (torch.tensor(1.5, device="cuda"), torch.tensor(0.2, dtype=torch.float64))):
        got = rp.ArrayPSFTransform.construct(device, target, a, e)._kernel_tensor
        assert got.grad_fn is None and not got.requires_grad and torch.equal(got, want)
    trainable = rp.ArrayPSF(rp.DeviceCube(coords, sv_t.clone().requires_grad_()))
    with torch.no_grad():
        got = rp.ArrayPSFTransform.construct(trainable, target, 1.5, 0.2)._kernel_tensor
    assert got.grad_fn is None and torch.equal(got, want)


def test_host_accessors_follow_in_place_updates_of_values_that_require_grad():
    torch = _torch()
    coords, sv, _ = _psf_values(16)
    values = torch.from_numpy(sv).cuda().requires_grad_()
    psf = rp.ArrayPSF(rp.DeviceCube(coords, values))
    before = psf.fft_evaluations.copy()
    np.testing.assert_allclose(before, oracle.psf_fft(sv), rtol=0, atol=1e-12 * np.abs(before).max())
    assert psf.fft_cube.tensor.grad_fn is None
    with torch.no_grad():
        values.mul_(2)
    np.testing.assert_allclose(psf.fft_evaluations, 2 * before, rtol=0, atol=1e-12 * np.abs(before).max())


# --------------------------------------------------------------------------------------------- reconstruct
def _plan_handles(transform):
    return {key: (nt.handle, dict(nt._plans)) for key, nt in transform._native.items()}


def test_reconstruct_keeps_plans_and_matches_a_fresh_construct():
    torch = _torch()
    coords, sv, tv, alpha, epsilon, x = _fit_setup(64, target_fwhm=1.0)
    source, target = rp.ArrayPSF(rp.DeviceCube(coords, sv)), rp.ArrayPSF(rp.DeviceCube(coords, tv))
    y = x.flip(0)
    transform = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)
    params = [sv, alpha, epsilon]
    losses, handles = [], None
    for _ in range(3):
        for p in params:
            p.grad = None
        transform.reconstruct(source, target, alpha, epsilon)
        loss = torch.nn.functional.mse_loss(transform.apply(x, dtype="float64"), y)
        loss.backward()
        losses.append(float(loss.detach()))
        if handles is None:
            handles = _plan_handles(transform)
        assert _plan_handles(transform) == handles
        with torch.no_grad():                                         # a short step along the normalised gradient
            norm = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in params))
            for p in params:
                p -= 1e-4 * p.grad / norm
    assert losses[1] < losses[0] and losses[2] < losses[1], losses
    # after reconstruct, apply is bit-identical to a fresh construct's
    transform.reconstruct(source, target, alpha, epsilon)
    fresh = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)
    for dtype in ("float64", "float32"):
        assert torch.equal(transform.apply(x, dtype=dtype), fresh.apply(x, dtype=dtype))
    with torch.no_grad():
        assert torch.equal(transform.apply(x), fresh.apply(x))


def test_reconstruct_checks_coordinates_and_patch_size():
    coords, sv, tv = _psf_values(16)
    transform = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.IndexedCube(coords, sv)),
                                               rp.ArrayPSF(rp.IndexedCube(coords, tv)), 1.0, 0.1)
    moved = [(r + 1, c) for r, c in coords]
    with pytest.raises(rp.InvalidCoordinateError):
        transform.reconstruct(rp.ArrayPSF(rp.IndexedCube(moved, sv)), rp.ArrayPSF(rp.IndexedCube(moved, tv)), 1.0, 0.1)
    small = sv[:, :8, :8].copy()
    with pytest.raises(rp.IncorrectShapeError):
        transform.reconstruct(rp.ArrayPSF(rp.IndexedCube(coords, small)), rp.ArrayPSF(rp.IndexedCube(coords, small)),
                              1.0, 0.1)


# --------------------------------------------------------------------------------------------- refusals
def test_refusals():
    torch = _torch()
    coords, sv, tv, alpha, epsilon, x = _fit_setup(16)
    source, target = rp.ArrayPSF(rp.DeviceCube(coords, sv)), rp.ArrayPSF(rp.DeviceCube(coords, tv))
    # embedded patch size with values that require grad
    emb = torch.ones((len(coords), 21, 21), dtype=torch.float64, device="cuda", requires_grad=True)
    with pytest.raises(NotImplementedError):
        rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, emb)),
                                       rp.ArrayPSF(rp.DeviceCube(coords, emb.detach())), 1.0, 0.1)
    # ... but not without grad
    with torch.no_grad():
        rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, emb)),
                                       rp.ArrayPSF(rp.DeviceCube(coords, emb)), 1.0, 0.1)
    transform = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)
    with pytest.raises(NotImplementedError):
        transform.apply(x, saturation_threshold=1.0)
    with pytest.raises(NotImplementedError):
        transform.apply(x, pad_mode="mean")
    # a sharded transform
    keep = np.zeros(len(coords), dtype=bool)
    keep[: len(coords) // 2] = True
    kept = [c for c, k in zip(coords, keep) if k]
    mask = torch.from_numpy(keep).cuda()
    plain = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.IndexedCube(coords, sv.detach().cpu().numpy())),
                                           rp.ArrayPSF(rp.IndexedCube(coords, tv.detach().cpu().numpy())), 1.0, 0.1)
    shard = rp.ArrayPSFTransform.sharded(rp.DeviceCube(kept, plain._kernel_tensor[mask]), coords, keep)
    sub = [rp.ArrayPSF(rp.DeviceCube(kept, v[mask])) for v in (sv, tv)]
    with pytest.raises(NotImplementedError):
        shard.reconstruct(sub[0], sub[1], alpha, epsilon)
    with torch.no_grad():
        shard.reconstruct(sub[0], sub[1], alpha, epsilon)               # without a gradient it is allowed
    # alpha must be a scalar
    with pytest.raises(ValueError):
        rp.ArrayPSFTransform.construct(source, target, alpha.reshape(1), epsilon)
    # double backward through Construct
    kernel = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)._kernel_tensor
    (g_alpha,) = torch.autograd.grad((kernel.abs() ** 2).sum(), alpha, create_graph=True)
    with pytest.raises(RuntimeError):
        g_alpha.backward()
