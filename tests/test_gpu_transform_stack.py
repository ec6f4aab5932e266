"""TransformStack: every member applied in one call, bit for bit what the member computes alone.

``stack.apply(x)[m]`` must equal ``stack[m].apply(x)`` (np.array_equal) for every argument ``apply`` takes, and the
kernels of ``TransformStack.construct`` must equal ``ArrayPSFTransform.construct``'s pair by pair.
"""
import ctypes
import itertools
import math
import os

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "builder", "c5_builder_p32.npz")
ALPHAS = (0.5, 1.0, 2.0, 3.0)
EPSILONS = (0.3, 0.1, 0.05, 0.01)


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


def _psfs(coords, size):
    src = oracle.coma_psf_cube(coords, size, (4096, 4096), core_sigma=min(2.5, size / 8), tail_scale=min(6.0, size / 6))
    tgt = oracle.gaussian_psf_cube(len(coords), size, min(3.0, size / 6))
    return rp.ArrayPSF(rp.IndexedCube(coords, src)), rp.ArrayPSF(rp.IndexedCube(coords, tgt))


def _stack(coords, size, m):
    pairs = list(itertools.product(ALPHAS, EPSILONS))[:m]
    source, target = _psfs(coords, size)
    return rp.TransformStack.construct(source, target, [a for a, _ in pairs], [e for _, e in pairs])


def _frames(rng, b, h, w):
    img = rng.normal(100.0, 20.0, (b, h, w))
    img[:, h // 3, w // 4] = 5000.0            # bright pixels for the saturation cases
    img[:, h // 2:h // 2 + 2, w // 2] = 3000.0
    return img


def _fused(stack, dtype):
    """Whether the stack's plan for its last call ran k2_stack (rpsf_plan_stack_info)."""
    import torch
    ns = stack._native[(dtype, torch.cuda.current_device())]
    flag = ctypes.c_int()
    _native.check(ns.lib.rpsf_plan_stack_info(next(reversed(ns._plans.values())), ctypes.byref(flag)))
    return bool(flag.value)


def _check(stack, x, **kw):
    """stack.apply(x)[m] equals stack[m].apply(x) bit for bit, through k2_stack and through the per-kernel column
    pass (rpsf_plan_set_stack_mode)."""
    wants = []
    for m in range(len(stack)):
        want = stack[m].apply(x, **kw)
        wants.append(want.cpu().numpy() if hasattr(want, "cpu") else want)
    dtype = kw.get("dtype") or "float32"
    size = stack.psf_shape[0]
    native = size in (16, 32, 64, 128, 256, 512)
    for mode in (0, 1):
        stack._stack_mode = mode
        got = stack.apply(x, **kw)
        got = got.cpu().numpy() if hasattr(got, "cpu") else got
        assert got.shape == (len(stack),) + tuple(x.shape)
        # k2_stack runs for two kernels or more at the native sizes whose column-pass stage ring fits (float32 to 256 px,
        # float64 to 64 px)
        fits = native and len(stack) >= 2 and (size <= 256 if dtype == "float32" else size <= 64)
        assert _fused(stack, dtype) == (mode == 0 and fits)
        for m in range(len(stack)):
            assert got.dtype == wants[m].dtype
            assert np.array_equal(got[m], wants[m], equal_nan=True), (mode, m, kw)
    stack._stack_mode = 0


# (patch, frame shape, kernels, frames, dtype, pad mode)
CASES = [
    (16, (96, 128), 2, 3, "float32", "symmetric"),
    (16, (64, 80), 5, 1, "float64", "wrap"),
    (32, (256, 256), 5, 3, "float32", "reflect"),
    (32, (200, 160), 2, 1, "float64", "edge"),
    (64, (256, 320), 2, 3, "float32", "constant"),
    (64, (256, 256), 1, 8, "float64", "symmetric"),
    (128, (1024, 1024), 4, 1, "float32", "symmetric"),       # config 1
    (128, (1024, 1024), 2, 3, "float64", "reflect"),
    (256, (2048, 2048), 16, 8, "float32", "symmetric"),      # config 2
    (256, (2048, 2048), 2, 1, "float64", "symmetric"),
]


@pytest.mark.parametrize("size,shape,m,b,dtype,pad", CASES)
def test_apply_equals_members(size, shape, m, b, dtype, pad):
    import torch
    stack = _stack(rp.calculate_covering(shape, size), size, m)
    x = torch.from_numpy(_frames(np.random.default_rng(size + m + b), b, *shape)).cuda()
    if b == 1:
        x = x[0]
    _check(stack, x, dtype=dtype, pad_mode=pad)


@pytest.mark.parametrize("dilation", [0, 1, 2])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_saturation(dilation, dtype):
    import torch
    shape = (192, 160)
    stack = _stack(rp.calculate_covering(shape, 32), 32, 3)
    x = torch.from_numpy(_frames(np.random.default_rng(dilation), 2, *shape)).cuda()
    _check(stack, x, dtype=dtype, saturation_threshold=2000.0, saturation_dilation=dilation)


@pytest.mark.parametrize("per_frame", [False, True])
@pytest.mark.parametrize("threshold", [math.inf, 2000.0])
def test_mask(per_frame, threshold):
    import torch
    shape = (160, 192)
    rng = np.random.default_rng(7)
    stack = _stack(rp.calculate_covering(shape, 32), 32, 3)
    x = torch.from_numpy(_frames(rng, 3, *shape)).cuda()
    mask = rng.random((3,) + shape if per_frame else shape) < 0.002
    mask[..., 40, 60:64] = True
    _check(stack, x, saturation_threshold=threshold, mask=torch.from_numpy(mask).cuda())
    _check(stack, x.cpu().numpy(), saturation_threshold=threshold, mask=mask)


def test_irregular_coordinates():
    import torch
    rng = np.random.default_rng(3)
    coords = sorted({(int(r), int(c)) for r, c in rng.integers(-20, 180, (40, 2))})
    stack = _stack(coords, 32, 3)
    x = torch.from_numpy(_frames(rng, 2, 200, 190)).cuda()
    _check(stack, x)
    _check(stack, x, dtype="float64", pad_mode="reflect")
    # mixed corner-row parities: the colour-phase overlap-add
    odd = [(r + (i % 2), c) for i, (r, c) in enumerate(rp.calculate_covering((128, 128), 32))]
    _check(_stack(odd, 32, 2), x[:, :128, :128])


@pytest.mark.parametrize("out_dtype", [np.float32, np.float64, None])
@pytest.mark.parametrize("src", [np.uint16, np.float64])
def test_numpy_input(out_dtype, src):
    shape = (128, 128)
    stack = _stack(rp.calculate_covering(shape, 32), 32, 3)
    x = np.clip(_frames(np.random.default_rng(1), 2, *shape), 0, 60000).astype(src)
    _check(stack, x, out_dtype=out_dtype)
    _check(stack, x[0], out_dtype=out_dtype, saturation_threshold=2000.0)
    _check(stack, x, out_dtype=out_dtype, dtype="float64")


@pytest.mark.parametrize("size", [21, 100])
def test_embedded_sizes(size):
    import torch
    shape = (4 * size, 3 * size + 7)
    stack = _stack(rp.calculate_covering(shape, size), size, 3)
    x = torch.from_numpy(_frames(np.random.default_rng(size), 2, *shape)).cuda()
    _check(stack, x)
    _check(stack, x, dtype="float64", saturation_threshold=2000.0)


# ------------------------------------------------------------------ construct
@pytest.mark.parametrize("wide", [False, True])
def test_construct_equals_per_pair(wide):
    import torch
    coords = rp.calculate_covering((256, 256), 32)
    source, target = _psfs(coords, 32)
    if not wide:
        source = rp.ArrayPSF(rp.IndexedCube(coords, source.values.astype(np.float32)))
        target = rp.ArrayPSF(rp.IndexedCube(coords, target.values.astype(np.float32)))
    pairs = list(itertools.product(ALPHAS, EPSILONS)) + [(1.0, 0.0), (2.0, 0.0), (0.5, 0.0), (1.7, 0.2), (0.0, 0.1)]
    alphas, epsilons = [a for a, _ in pairs], [e for _, e in pairs]
    host = rp.TransformStack.construct(source, target, alphas, epsilons)
    f64 = lambda v: torch.tensor(v, dtype=torch.float64, device="cuda")          # noqa: E731
    dev = rp.TransformStack.construct(source, target, [f64(a) for a in alphas], [f64(e) for e in epsilons])
    assert len(host) == len(pairs)
    for m, (a, e) in enumerate(pairs):
        want = rp.ArrayPSFTransform.construct(source, target, a, e)._kernel_tensor.cpu().numpy()
        want_dev = rp.ArrayPSFTransform.construct(source, target, f64(a), f64(e))._kernel_tensor.cpu().numpy()
        assert np.array_equal(want, want_dev, equal_nan=True)
        got = host.kernels[m].cpu().numpy()
        assert got.dtype == want.dtype
        assert np.array_equal(got, want, equal_nan=True), (a, e)
        assert np.array_equal(dev.kernels[m].cpu().numpy(), want, equal_nan=True), (a, e)
        if e == 0.0:
            assert np.array_equal(np.isnan(got), np.isnan(want))


def test_config5_sweep_in_one_call():
    """The 16-pair alpha / epsilon sweep of BASELINE.json configs[4] as one float64 stack.apply."""
    golden = np.load(GOLDEN)
    frames, _ = oracle.builder_frames()
    size = int(golden["size"])
    coords = [tuple(int(v) for v in c) for c in golden["coords"]]
    src = golden["values_median"]
    tgt = oracle.gaussian_psf_cube(len(coords), size, 3.0)
    source = rp.ArrayPSF(rp.IndexedCube(coords, src))
    target = rp.ArrayPSF(rp.IndexedCube(coords, tgt))
    s_fft, t_fft = oracle.psf_fft(src), oracle.psf_fft(tgt)
    pairs = list(itertools.product(ALPHAS, EPSILONS))
    stack = rp.TransformStack.construct(source, target, [a for a, _ in pairs], [e for _, e in pairs])
    image = frames[0]
    got = stack.apply(image, dtype="float64")
    assert got.shape == (16,) + image.shape
    scale = float(np.max(np.abs(image)))
    r0, r1, c0, c1 = (int(v) for v in golden["crop"])
    pinned = {tuple(p): k for k, p in enumerate(golden["sweep"])}
    for m, (alpha, epsilon) in enumerate(pairs):
        want = oracle.apply_transform(image, coords, oracle.transfer_kernel(s_fft, t_fft, alpha, epsilon))
        assert np.max(np.abs(got[m] - want)) <= 1e-10 * scale, (alpha, epsilon)
        if (alpha, epsilon) in pinned:
            ref = golden[f"out_crop_{pinned[(alpha, epsilon)]}"]
            assert np.max(np.abs(got[m][r0:r1, c0:c1] - ref)) <= 1e-10 * scale
        assert np.array_equal(got[m], stack[m].apply(image, dtype="float64"))


# ------------------------------------------------------------------ stacking transforms, views
def test_stack_of_transforms_and_views():
    import torch
    coords = rp.calculate_covering((128, 128), 32)
    source, target = _psfs(coords, 32)
    members = [rp.ArrayPSFTransform.construct(source, target, a, 0.1) for a in (1.0, 2.0, 3.0)]
    host_member = rp.ArrayPSFTransform(rp.IndexedCube(coords, members[0]._kernel_tensor.cpu().numpy()))
    stack = rp.ArrayPSFTransform.stack(members + [host_member])
    assert len(stack) == 4
    x = torch.from_numpy(_frames(np.random.default_rng(0), 2, 128, 128)).cuda()
    got = stack.apply(x)
    for m, tr in enumerate(members + [host_member]):
        assert np.array_equal(got[m].cpu().numpy(), tr.apply(x).cpu().numpy())
    view = stack[1]._kernel_tensor
    assert view.data_ptr() == stack.kernels[1].data_ptr()          # a view, not a copy
    assert not stack[1]._native                                     # no native state until it is applied
    assert stack[1] is stack[1]                                     # members are kept: one native state each


# ------------------------------------------------------------------ streams and graphs
def test_side_stream_and_graph():
    import torch
    shape = (256, 256)
    stack = _stack(rp.calculate_covering(shape, 64), 64, 4)
    x = torch.from_numpy(_frames(np.random.default_rng(5), 2, *shape)).float().cuda()
    eager = stack.apply(x)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        on_side = stack.apply(x)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(eager, on_side)

    static_in = x.clone()
    stack.apply(static_in)                                          # warm up the plan
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = stack.apply(static_in)
    static_in.mul_(1.5).add_(3.0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, stack.apply(static_in))


def test_capture_refuses_a_cold_plan():
    import torch
    stack = _stack(rp.calculate_covering((128, 128), 32), 32, 2)
    x = torch.zeros((1, 128, 128), device="cuda")
    stack.apply(x)
    x3 = torch.zeros((3, 128, 128), device="cuda")
    graph = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError):
        with torch.cuda.graph(graph):
            stack.apply(x3)


# ------------------------------------------------------------------ errors
def test_errors():
    import torch
    coords = rp.calculate_covering((128, 128), 32)
    source, target = _psfs(coords, 32)
    a = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    shifted = rp.ArrayPSFTransform(rp.IndexedCube([(r + 2, c) for r, c in coords], a._kernel_tensor.cpu().numpy()))
    with pytest.raises(rp.InvalidCoordinateError):
        rp.ArrayPSFTransform.stack([a, shifted])
    s16, t16 = _psfs(coords, 16)
    with pytest.raises(rp.IncorrectShapeError):
        rp.ArrayPSFTransform.stack([a, rp.ArrayPSFTransform.construct(s16, t16, 1.0, 0.1)])
    sharded = rp.ArrayPSFTransform.sharded(rp.IndexedCube(coords[:2], a._kernel_tensor.cpu().numpy()[:2]), coords,
                                           [True, True] + [False] * (len(coords) - 2))
    with pytest.raises(NotImplementedError):
        rp.ArrayPSFTransform.stack([a, sharded])
    far = rp.ArrayPSF(rp.IndexedCube([(r + 4, c) for r, c in coords], source.values))
    with pytest.raises(rp.InvalidCoordinateError):
        rp.TransformStack.construct(far, target, [1.0], [0.1])
    with pytest.raises(rp.IncorrectShapeError):
        rp.TransformStack.construct(source, t16, [1.0], [0.1])
    with pytest.raises(ValueError):
        rp.TransformStack.construct(source, target, [1.0, 2.0], [0.1])

    stack = rp.ArrayPSFTransform.stack([a, a])
    x = torch.zeros((128, 128), device="cuda")
    with pytest.raises(NotImplementedError):
        stack.apply(x.clone().requires_grad_(True))
    trainable = rp.TransformStack(coords, stack.kernels.clone().requires_grad_(True))
    with pytest.raises(NotImplementedError):
        trainable.apply(x)
    with torch.no_grad():
        assert trainable.apply(x).shape == (2, 128, 128)
    with pytest.raises(NotImplementedError):
        stack.apply_adjoint(x)
    with pytest.raises(NotImplementedError):
        stack.apply(x, pad_mode="mean")
    with pytest.raises(NotImplementedError):
        stack.apply(x.cpu().numpy(), out_dtype=np.int32)


def test_c_status_codes():
    import torch
    lib = _native.load()
    coords = np.ascontiguousarray(rp.calculate_covering((128, 128), 32), dtype=np.int32)
    st, plan = ctypes.c_void_p(), ctypes.c_void_p()
    assert lib.rpsf_stack_create(None, coords.ctypes.data, len(coords), 32, _native.F32, 0, 2) == _native.E_INVALID_ARGUMENT
    assert lib.rpsf_stack_create(ctypes.byref(st), coords.ctypes.data, len(coords), 32, _native.F32, 0, 0) == \
        _native.E_INVALID_ARGUMENT
    _native.check(lib.rpsf_stack_create(ctypes.byref(st), coords.ctypes.data, len(coords), 32, _native.F32, 0, 2))
    try:
        assert lib.rpsf_plan_create_stack(None, st, 128, 128, 0, 2) == _native.E_INVALID_ARGUMENT
        assert lib.rpsf_plan_create_stack(ctypes.byref(plan), st, 128, 128, 5, 2) == _native.E_UNSUPPORTED
        assert lib.rpsf_plan_create_stack(ctypes.byref(plan), st, 128, 128, 0, 40000) == _native.E_INVALID_ARGUMENT
        _native.check(lib.rpsf_plan_create_stack(ctypes.byref(plan), st, 128, 128, 0, 2))
        assert lib.rpsf_plan_set_stack_mode(plan, 2) == _native.E_INVALID_ARGUMENT
        assert lib.rpsf_plan_set_stack_mode(None, 0) == _native.E_INVALID_ARGUMENT
        fused = ctypes.c_int()
        _native.check(lib.rpsf_plan_stack_info(plan, ctypes.byref(fused)))
        assert fused.value == 1
        x = torch.zeros((3, 128, 128), device="cuda")
        out = torch.zeros((2, 3, 128, 128), device="cuda")
        k = torch.zeros((len(coords), 32, 32), dtype=torch.complex64, device="cuda")
        args = lambda m, b, pitch=128: (plan, x.data_ptr(), pitch, 128 * 128, out.data_ptr(), 128, 128 * 128, m, b,
                                        None, 0, 0, 0, None, 0, 0, None)
        assert lib.rpsf_apply_stack(*args(2, 1)) == _native.E_NO_KERNEL
        assert lib.rpsf_stack_set_kernel(st, 2, k.data_ptr(), _native.F32, None) == _native.E_INVALID_ARGUMENT
        assert lib.rpsf_stack_set_kernel(st, 0, None, _native.F32, None) == _native.E_INVALID_ARGUMENT
        for m in range(2):
            _native.check(lib.rpsf_stack_set_kernel(st, m, k.data_ptr(), _native.F32, None))
        assert lib.rpsf_apply_stack(None, *args(2, 1)[1:]) == _native.E_INVALID_ARGUMENT
        assert lib.rpsf_apply_stack(plan, None, *args(2, 1)[2:]) == _native.E_INVALID_ARGUMENT
        assert lib.rpsf_apply_stack(*args(2, 3)) == _native.E_INVALID_ARGUMENT         # above max_batch = 2
        assert lib.rpsf_apply_stack(*args(3, 1)) == _native.E_INVALID_ARGUMENT         # M of another stack
        assert lib.rpsf_apply_stack(*args(2, 1, 100)) == _native.E_INCORRECT_SHAPE     # pitch of a narrower frame
        _native.check(lib.rpsf_apply_stack(*args(2, 2)))
        # the ordinary entry points refuse a stack plan
        assert lib.rpsf_apply(plan, x.data_ptr(), 128, 128 * 128, 0, 128, out.data_ptr(), 128, 128 * 128, 0, 1,
                              None) == _native.E_INVALID_ARGUMENT
        torch.cuda.synchronize()
    finally:
        lib.rpsf_plan_destroy(plan)
        lib.rpsf_stack_destroy(st)
    kk = torch.zeros((2, 4), dtype=torch.complex64, device="cuda")
    assert lib.rpsf_construct_kernels(kk.data_ptr(), kk.data_ptr(), kk.data_ptr(), 4, _native.F32, None, 2, 0, None) == \
        _native.E_INVALID_ARGUMENT
    assert lib.rpsf_construct_kernels_dev(kk.data_ptr(), kk.data_ptr(), kk.data_ptr(), 4, 7, kk.data_ptr(), 1, 0,
                                          None) == _native.E_UNSUPPORTED
