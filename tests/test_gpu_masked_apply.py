"""apply(mask=), its transpose and its gradients on the device, against tests/masked_apply_oracle.py.

Bars as for the saturation branch: identical NaN pattern, max |diff| <= 1e-5 x max|image| in float32 mode and <= 1e-10 in
float64 mode, masked output pixels equal to the raw input; the masked map's transpose satisfies the dot-product identity
to 1e-12 in float64; everything that should equal another path does so bit for bit.
"""
import math

import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native
from regularizepsf_b200.exceptions import IncorrectShapeError
from tests import masked_apply_oracle as mo

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


def _torch():
    import torch
    return torch


def _covering(shape, size):
    return [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]


def _kernel(size, n, fwhm=2.5, shift=(1, 2)):
    """A Gaussian blur followed by a small circular shift, one spectrum for every patch."""
    k = np.arange(size)
    spec = np.exp(-2j * np.pi * (k[:, None] * shift[0] + k[None, :] * shift[1]) / size)
    r = np.minimum(k, size - k).astype(np.float64)
    g = np.exp(-4 * np.log(2) * (r[:, None] ** 2 + r[None, :] ** 2) / fwhm ** 2)
    spec = spec * np.fft.fft2(g / g.sum())
    return np.repeat(spec[np.newaxis], n, axis=0)


def _transform(shape, size):
    coords = _covering(shape, size)
    kernel = _kernel(size, len(coords))
    return rp.ArrayPSFTransform(rp.IndexedCube(coords, kernel)), coords, kernel


def _mask(shape, kind, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "random":
        return rng.random(shape) < 1e-3
    m = np.zeros(shape, bool)
    if kind == "columns":
        m[:, [3, shape[1] // 3, shape[1] // 3 + 1, shape[1] - 1]] = True
    elif kind == "nan_block":
        m[shape[0] // 2:shape[0] // 2 + 64, shape[1] // 4:shape[1] // 4 + 64] = True
    return m


def _scene(shape, kind, seed=0):
    image = oracle.starfield(shape, seed=11 + seed).astype(np.float64)
    mask = _mask(shape, kind, seed)
    if kind == "nan_block":
        image[mask] = np.nan
    return image, mask


def _check(got, want, image, mask, dtype):
    got = np.asarray(got, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.all(np.isfinite(got[~mask]))
    assert np.array_equal(got[mask], image[mask].astype(np.float32 if dtype == "float32" else np.float64),
                          equal_nan=True)
    scale = np.nanmax(np.abs(image))
    assert np.nanmax(np.abs(got - want)) <= TOL[dtype] * scale


_ORACLE = {}


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("kind", ["random", "columns", "nan_block"])
@pytest.mark.parametrize("config", [(2048, 256), (1024, 128)])
def test_parity_with_the_oracle(config, kind, dtype):
    torch = _torch()
    n, size = config
    t, coords, kernel = _transform((n, n), size)
    image, mask = _scene((n, n), kind)
    if (config, kind) not in _ORACLE:
        _ORACLE[(config, kind)] = mo.apply_masked(image, coords, kernel, mask)
    want = _ORACLE[(config, kind)]
    got = t.apply(torch.from_numpy(image).cuda(), mask=torch.from_numpy(mask).cuda(), dtype=dtype)
    _check(got.cpu().numpy(), want, image, mask, dtype)
    host = t.apply(image, mask=mask, dtype=dtype)
    assert host.dtype == np.float64 and np.array_equal(host, got.cpu().numpy().astype(np.float64), equal_nan=True)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_an_all_false_mask_is_the_plain_apply(dtype):
    torch = _torch()
    t, _, _ = _transform((1024, 1024), 128)
    image = oracle.starfield((1024, 1024), seed=3)
    none = np.zeros(image.shape, bool)
    x = torch.from_numpy(image).cuda()
    assert torch.equal(t.apply(x, dtype=dtype, mask=torch.from_numpy(none).cuda()), t.apply(x, dtype=dtype))
    assert np.array_equal(t.apply(image, dtype=dtype, mask=none), t.apply(image, dtype=dtype))


def test_the_saturation_frame_mask_is_the_threshold_call_and_a_union_matches_the_oracle():
    torch = _torch()
    shape, size = (1024, 1024), 128
    t, coords, kernel = _transform(shape, size)
    image = np.random.default_rng(2).normal(100.0, 5.0, shape)
    image[[200, 201, 600, 700], [300, 300, 500, 90]] = 1e5             # >= 2 px from the border after dilation
    frame_mask = np.zeros(shape, bool)
    for r, c in [(200, 300), (201, 300), (600, 500), (700, 90)]:
        frame_mask[r - 1:r + 2, c] = frame_mask[r, c - 1:c + 2] = True
    x = torch.from_numpy(image).cuda()
    for dtype in ("float32", "float64"):
        a = t.apply(x, saturation_threshold=1e4, dtype=dtype)
        b = t.apply(x, mask=torch.from_numpy(frame_mask).cuda(), dtype=dtype)
        assert torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(), b.nan_to_num())
    extra = _mask(shape, "columns")
    want = mo.apply_masked(image, coords, kernel, extra, saturation_threshold=1e4)
    got = t.apply(x, mask=torch.from_numpy(extra).cuda(), saturation_threshold=1e4, dtype="float64")
    full = extra | frame_mask
    _check(got.cpu().numpy(), want, image, full, "float64")


def test_shared_and_per_frame_masks_batch_like_single_frames():
    torch = _torch()
    shape = (512, 512)
    t, _, _ = _transform(shape, 64)
    frames = np.stack([oracle.starfield(shape, seed=s) for s in range(3)])
    masks = np.stack([_mask(shape, "random", seed=s) | _mask(shape, "columns") for s in range(3)])
    x = torch.from_numpy(frames).cuda()
    per_frame = t.apply(x, mask=torch.from_numpy(masks).cuda())
    shared = t.apply(x, mask=torch.from_numpy(masks[0]).cuda())
    for b in range(3):
        assert torch.equal(per_frame[b], t.apply(x[b], mask=torch.from_numpy(masks[b]).cuda()))
        assert torch.equal(shared[b], t.apply(x[b], mask=torch.from_numpy(masks[0]).cuda()))
    u8 = torch.from_numpy(masks.astype(np.uint8)).cuda()
    assert torch.equal(per_frame, t.apply(x, mask=u8))
    assert torch.equal(per_frame, t.apply(x, mask=torch.from_numpy(masks).cuda()))       # repeated: bit-identical


@pytest.mark.parametrize("pad_mode", PAD_MODES)
def test_every_pad_mode_forward_and_transpose(pad_mode):
    torch = _torch()
    shape, size = (256, 256), 32
    t, coords, kernel = _transform(shape, size)
    image, mask = _scene(shape, "random", seed=4)
    mask |= _mask(shape, "columns")
    want = mo.apply_masked(image, coords, kernel, mask, pad_mode)
    m = torch.from_numpy(mask).cuda()
    got = t.apply(torch.from_numpy(image).cuda(), pad_mode=pad_mode, mask=m, dtype="float64")
    _check(got.cpu().numpy(), want, image, mask, "float64")
    y = np.random.default_rng(5).normal(size=shape)
    want_t = mo.apply_masked_adjoint(y, coords, kernel, mask, pad_mode)
    got_t = t.apply_adjoint(torch.from_numpy(y).cuda(), pad_mode=pad_mode, mask=m, dtype="float64").cpu().numpy()
    assert np.max(np.abs(got_t - want_t)) <= 1e-10 * np.max(np.abs(want_t))


@pytest.mark.parametrize("size", [48, 100])
def test_embedded_sizes_forward_and_transpose(size):
    torch = _torch()
    shape = (300, 260)
    t, coords, kernel = _transform(shape, size)
    image, mask = _scene(shape, "random", seed=6)
    mask[:, 17] = True
    m = torch.from_numpy(mask).cuda()
    want = mo.apply_masked(image, coords, kernel, mask)
    _check(t.apply(torch.from_numpy(image).cuda(), mask=m, dtype="float64").cpu().numpy(), want, image, mask, "float64")
    y = np.random.default_rng(7).normal(size=shape)
    want_t = mo.apply_masked_adjoint(y, coords, kernel, mask)
    got_t = t.apply_adjoint(y, mask=mask, dtype="float64")
    assert np.max(np.abs(got_t - want_t)) <= 1e-10 * np.max(np.abs(want_t))


def _random_kernel_transform(shape, size, requires_grad=False):
    torch = _torch()
    coords = _covering(shape, size)
    g = torch.Generator(device="cuda").manual_seed(3)
    kernel = torch.randn((len(coords), size, size), dtype=torch.complex128, device="cuda", generator=g)
    if requires_grad:
        kernel.requires_grad_()
    return rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel)), coords, kernel


@pytest.mark.parametrize("width", [2, 7, 8])
def test_dot_product_identity_on_the_device(width):
    torch = _torch()
    shape, size = (512, 384), 64
    t, coords, kernel = _random_kernel_transform(shape, size)
    mask = _mask(shape, "random", seed=8) | _mask(shape, "columns")
    mask[100:140, 200:260] = True                                      # a run wider than a fill chunk, full windows
    m = torch.from_numpy(mask).cuda()
    rng = np.random.default_rng(9)
    x = torch.from_numpy(rng.normal(size=shape)).cuda()
    y = torch.from_numpy(rng.normal(size=shape)).cuda()
    lx = t.apply(x, mask=m, neighborhood_width=width, dtype="float64")
    lty = t.apply_adjoint(y, mask=m, neighborhood_width=width, dtype="float64")
    err = abs(float((lx * y).sum() - (x * lty).sum())) / float(lx.norm() * y.norm())
    assert err <= 1e-12
    assert torch.equal(lty, t.apply_adjoint(y, mask=m, neighborhood_width=width, dtype="float64"))
    want_t = mo.apply_masked_adjoint(y.cpu().numpy(), coords, kernel.cpu().numpy(), mask, neighborhood_width=width)
    assert np.max(np.abs(lty.cpu().numpy() - want_t)) <= 1e-10 * np.max(np.abs(want_t))


def test_autograd_image_gradient_is_the_transpose_and_double_backward_works():
    torch = _torch()
    shape = (512, 512)
    t, _, _ = _transform(shape, 64)
    mask = torch.from_numpy(_mask(shape, "random") | _mask(shape, "columns")).cuda()
    x = torch.from_numpy(oracle.starfield(shape, seed=2).astype(np.float64)).cuda().requires_grad_()
    g = torch.randn(shape, dtype=torch.float64, device="cuda")
    out = t.apply(x, mask=mask, dtype="float64")
    (grad,) = torch.autograd.grad(out, x, g, create_graph=True)
    assert torch.equal(grad, t.apply_adjoint(g, mask=mask, dtype="float64"))
    v = torch.randn(shape, dtype=torch.float64, device="cuda")
    gv = g.clone().requires_grad_()
    (gx,) = torch.autograd.grad(t.apply(x, mask=mask, dtype="float64"), x, gv, create_graph=True)
    (ggv,) = torch.autograd.grad((gx * v).sum(), gv)
    assert torch.equal(ggv, t.apply(v, mask=mask, dtype="float64"))


def test_kernel_gradient_matches_the_oracle():
    torch = _torch()
    shape, size = (512, 384), 64
    t, coords, kernel = _random_kernel_transform(shape, size, requires_grad=True)
    rng = np.random.default_rng(10)
    x, g = rng.normal(size=(2,) + shape), rng.normal(size=(2,) + shape)
    masks = np.stack([_mask(shape, "random", seed=s) | _mask(shape, "columns") for s in range(2)])
    want = mo.masked_kernel_gradient(x, g, coords, size, masks)
    got = t.transfer_kernel_gradient(x, g, mask=masks, dtype="float64")
    assert np.max(np.abs(got - want)) <= 1e-10 * np.max(np.abs(want))
    xt = torch.from_numpy(x).cuda()
    out = t.apply(xt, mask=torch.from_numpy(masks).cuda(), dtype="float64")
    (gk,) = torch.autograd.grad(out, kernel, torch.from_numpy(g).cuda())
    assert np.max(np.abs(gk.cpu().numpy() - want)) <= 1e-10 * np.max(np.abs(want))


def test_a_masked_construct_apply_loss_reaches_psf_values_alpha_and_epsilon():
    torch = _torch()
    shape, size = (256, 256), 32
    coords = _covering(shape, size)
    src = torch.from_numpy(oracle.coma_psf_cube(coords, size, shape)).cuda().requires_grad_()
    tgt = rp.ArrayPSF(rp.DeviceCube(coords, torch.from_numpy(oracle.gaussian_psf_cube(len(coords), size, 3.0)).cuda()))
    alpha = torch.tensor(1.5, dtype=torch.float64, device="cuda", requires_grad=True)
    eps = torch.tensor(0.3, dtype=torch.float64, device="cuda", requires_grad=True)
    image = torch.from_numpy(oracle.starfield(shape, seed=7).astype(np.float64)).cuda()
    mask = torch.from_numpy(_mask(shape, "random", seed=1) | _mask(shape, "columns")).cuda()
    w = torch.randn(shape, dtype=torch.float64, device="cuda")

    def loss(values, a, e):
        t = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, values)), tgt, a, e)
        return (t.apply(image, mask=mask, dtype="float64") * w).sum()

    gs, ga, ge = torch.autograd.grad(loss(src, alpha, eps), (src, alpha, eps))
    h = 1e-6
    with torch.no_grad():
        for got, bump in ((ga, lambda d: (src, alpha + d, eps)), (ge, lambda d: (src, alpha, eps + d))):
            fd = (loss(*bump(h)) - loss(*bump(-h))) / (2 * h)
            assert abs(float(got) - float(fd)) <= 1e-5 * max(1.0, abs(float(fd)))
        # along the values themselves: a direction that moves every spectrum bin in proportion (a single value would
        # move the near-zero bins of the spectrum by more than their size, where the kernel is far from linear)
        d = src.detach()
        fd = (loss(src + h * d, alpha, eps) - loss(src - h * d, alpha, eps)) / (2 * h)
        assert abs(float((gs * d).sum()) - float(fd)) <= 1e-5 * max(1.0, abs(float(fd)))


def _capture(fn, warmup=2):
    torch = _torch()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


def test_cuda_graphs_replay_a_masked_apply_and_a_fitting_step():
    torch = _torch()
    shape, size = (512, 512), 64
    t, _, _ = _transform(shape, size)
    x = torch.from_numpy(oracle.starfield(shape, seed=3)).cuda()
    mask = torch.from_numpy(_mask(shape, "random")).cuda()
    graph, out = _capture(lambda: t.apply(x, mask=mask))
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, t.apply(x, mask=mask))
    mask.copy_(torch.from_numpy(_mask(shape, "columns")).cuda())          # read again at every replay
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, t.apply(x, mask=mask))

    coords = _covering(shape, size)
    values = torch.from_numpy(oracle.coma_psf_cube(coords, size, shape)).cuda().float().requires_grad_()
    tgt = rp.ArrayPSF(rp.DeviceCube(coords, torch.from_numpy(oracle.gaussian_psf_cube(len(coords), size, 3.0)).cuda()
                                    .float()))
    fit = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, values)), tgt, 1.5, 0.3)
    opt = torch.optim.SGD([values], lr=1e-3)
    want = torch.from_numpy(oracle.starfield(shape, seed=4)).cuda()

    def step():
        opt.zero_grad(set_to_none=False)
        fit.reconstruct(rp.ArrayPSF(rp.DeviceCube(coords, values)), tgt, 1.5, 0.3)
        loss = ((fit.apply(x, mask=mask) - want) ** 2).mean()
        loss.backward()
        opt.step()
        return loss.detach()

    start = values.detach().clone()
    eager = []
    for _ in range(3):
        eager.append(step())
    end_eager = values.detach().clone()
    with torch.no_grad():
        values.copy_(start)
    step()                                                              # warm-up outside the capture
    with torch.no_grad():
        values.copy_(start)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = step()
    with torch.no_grad():
        values.copy_(start)
    replayed = []
    for _ in range(3):
        graph.replay()
        replayed.append(loss.clone())
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(eager, replayed))
    assert torch.equal(values.detach(), end_eager)


def test_errors():
    torch = _torch()
    shape = (256, 256)
    t, _, _ = _transform(shape, 32)
    x = torch.zeros(shape, dtype=torch.float64, device="cuda")
    with pytest.raises(IncorrectShapeError):
        t.apply(x, mask=torch.zeros((255, 256), dtype=torch.bool, device="cuda"))
    with pytest.raises(IncorrectShapeError):
        t.apply(np.zeros(shape), mask=np.zeros((2, 256, 256), bool))
    with pytest.raises(ValueError):
        t.apply(x, mask=torch.zeros(shape, dtype=torch.bool))
    with pytest.raises(ValueError):
        t.apply(x, mask=np.zeros(shape, bool))
    with pytest.raises(TypeError):
        t.apply(x, mask=torch.zeros(shape, dtype=torch.float32, device="cuda"))
    with pytest.raises(TypeError):
        t.apply(np.zeros(shape), mask=np.zeros(shape, np.int32))
    m = torch.zeros(shape, dtype=torch.bool, device="cuda")
    with pytest.raises(NotImplementedError):
        t.apply(x, pad_mode="mean", mask=m)
    with pytest.raises(NotImplementedError):
        t.apply(x.clone().requires_grad_(), saturation_threshold=10.0, mask=m)
    coords = _covering(shape, 32)
    keep = np.zeros(len(coords), bool)
    keep[:4] = True
    sharded = rp.ArrayPSFTransform.sharded(rp.IndexedCube([coords[i] for i in range(4)],
                                                          _kernel(32, 4)), coords, keep)
    with pytest.raises(NotImplementedError):
        sharded.apply(x, mask=m)
    assert math.isfinite(float(t.apply(x, mask=m).abs().max()))
