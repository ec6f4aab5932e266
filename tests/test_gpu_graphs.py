"""CUDA graphs: device-resident apply, its gradients and a whole fitting step captured with ``torch.cuda.graph``.

Each test warms its calls up outside the capture (plans, workspaces and the first kernel layout exist then), captures,
copies fresh inputs into the static input tensors and replays several times.  Unless a test says otherwise a replay is
compared bit for bit with the same eager calls: the kernels are run-to-run bit-stable.  The ordering tests hold a stream
with a spinning kernel (``torch.cuda._sleep``) as tests/test_gpu_streams.py does, and first check that the hold is still
pending, so that a set-up that synchronised by accident fails instead of passing vacuously.
"""
import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native

pytestmark = pytest.mark.gpu

HOLD_SECONDS = 0.3
REPLAYS = 3
_HOLD = {}


def _torch():
    import torch
    return torch


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    torch = _torch()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    torch.cuda._sleep(1000)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    torch.cuda._sleep(50_000_000)
    end.record()
    end.synchronize()
    _HOLD["cycles"] = int(50_000_000 * HOLD_SECONDS * 1000.0 / start.elapsed_time(end))
    before = _native.launch_count()
    yield
    assert _native.launch_count() > before, "no kernel of librpsf_b200.so was launched"


def _hold(stream):
    torch = _torch()
    with torch.cuda.stream(stream):
        torch.cuda._sleep(_HOLD["cycles"])
        event = torch.cuda.Event()
        event.record()
    return event


def _assert_pending(event):
    assert not event.query(), "the held stream finished before the calls under test were issued: nothing was raced"


def _bits(t):
    """The tensor's bytes as integers, so that NaNs compare equal to themselves."""
    torch = _torch()
    real = torch.view_as_real(t) if t.is_complex() else t
    return real.contiguous().view(torch.int32 if real.element_size() == 4 else torch.int64)


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and _torch().equal(_bits(a), _bits(b))


def _capture(fn, warmup=2):
    """Warm ``fn`` up on a side stream, then capture it: (graph, its output)."""
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


def _random_transform(shape, size, seed=1, requires_grad=False, dtype=None):
    torch = _torch()
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]
    g = torch.Generator(device="cuda").manual_seed(seed)
    kernel = torch.randn((len(coords), size, size), dtype=dtype or torch.complex64, device="cuda", generator=g)
    if requires_grad:
        kernel.requires_grad_()
    return rp.ArrayPSFTransform(rp.DeviceCube(coords, kernel)), kernel


def _frames(shape, batch, seed, dtype=None):
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(seed)
    full = (batch,) + tuple(shape) if batch else tuple(shape)
    return torch.rand(full, device="cuda", generator=g, dtype=dtype or torch.float32) * 100.0


# --------------------------------------------------------------------------------------------- forward and gradients
FORWARD = {"p64": ((192, 160), 64, 0), "p128_1024": ((1024, 1024), 128, 0), "p256_2048_b8": ((2048, 2048), 256, 8),
           "embedded_p100": ((300, 280), 100, 0)}


@pytest.mark.parametrize("case", sorted(FORWARD))
def test_replayed_apply_matches_eager(case):
    shape, size, batch = FORWARD[case]
    t, _ = _random_transform(shape, size)
    static = _frames(shape, batch, 0)
    graph, out = _capture(lambda: t.apply(static))
    for seed in range(1, REPLAYS + 1):
        x = _frames(shape, batch, seed)
        static.copy_(x)
        graph.replay()
        assert _same(out, t.apply(x)), seed


def test_replayed_saturation_branch_matches_eager():
    shape, size = (2048, 2048), 256
    t, _ = _random_transform(shape, size)
    static = _frames(shape, 0, 0)
    threshold = 99.0

    def call():
        return t.apply(static, saturation_threshold=threshold, saturation_dilation=2)

    graph, out = _capture(call)
    for seed in range(1, REPLAYS + 1):
        x = _frames(shape, 0, seed)
        static.copy_(x)
        graph.replay()
        assert _same(out, t.apply(x, saturation_threshold=threshold, saturation_dilation=2)), seed


@pytest.mark.parametrize("pad_mode", ["symmetric", "wrap"])
def test_replayed_apply_adjoint_matches_eager(pad_mode):
    shape, size = (192, 160), 64
    t, _ = _random_transform(shape, size)
    static = _frames(shape, 2, 0)
    graph, out = _capture(lambda: t.apply_adjoint(static, pad_mode=pad_mode))
    for seed in range(1, REPLAYS + 1):
        y = _frames(shape, 2, seed)
        static.copy_(y)
        graph.replay()
        assert _same(out, t.apply_adjoint(y, pad_mode=pad_mode)), seed


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_replayed_transfer_kernel_gradient_matches_eager(dtype):
    torch = _torch()
    shape, size = (192, 160), 64
    real = torch.float32 if dtype == "float32" else torch.float64
    t, _ = _random_transform(shape, size, dtype=torch.complex64 if dtype == "float32" else torch.complex128)
    sx, sg = _frames(shape, 2, 0, real), _frames(shape, 2, 50, real)
    graph, out = _capture(lambda: t.transfer_kernel_gradient(sx, sg, dtype=dtype))
    for seed in range(1, REPLAYS + 1):
        x, g = _frames(shape, 2, seed, real), _frames(shape, 2, 50 + seed, real)
        sx.copy_(x)
        sg.copy_(g)
        graph.replay()
        assert _same(out, t.transfer_kernel_gradient(x, g, dtype=dtype)), seed


# --------------------------------------------------------------------------------------------- ordering
def _psf_setup(shape=(192, 160), size=64):
    torch = _torch()
    coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]
    src = torch.from_numpy(oracle.coma_psf_cube(coords, size, shape)).cuda()
    tgt = torch.from_numpy(oracle.gaussian_psf_cube(len(coords), size, 3.0)).cuda()
    source, target = rp.ArrayPSF(rp.DeviceCube(coords, src)), rp.ArrayPSF(rp.DeviceCube(coords, tgt))
    for psf in (source, target):
        psf.fft_cube
    return coords, source, target


def test_replay_behind_a_reconstruct_on_a_held_stream_uses_the_new_kernel():
    torch = _torch()
    shape = (192, 160)
    _, source, target = _psf_setup(shape)
    t = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    static = _frames(shape, 0, 0)
    graph, out = _capture(lambda: t.apply(static))
    fresh = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.3)
    torch.cuda.synchronize()
    want = fresh.apply(static)
    torch.cuda.synchronize()
    held = torch.cuda.Stream()
    event = _hold(held)
    with torch.cuda.stream(held):
        t.reconstruct(source, target, 1.0, 0.3)
    other = torch.cuda.Stream()
    with torch.cuda.stream(other):
        graph.replay()
    _assert_pending(event)
    torch.cuda.synchronize()
    assert _same(out, want)


def _reconstructing_graph(shape, size, static):
    """A transform and a graph that holds ``reconstruct`` (epsilon read from a static 0-d tensor) and ``apply(static)``:
    each replay builds and lays out the kernel of the epsilon it finds, so a call that reads the layout after the
    replay sees the new kernel only if it is ordered behind the replay."""
    torch = _torch()
    _, source, target = _psf_setup(shape, size)
    t = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    alpha, epsilon = (torch.tensor(v, dtype=torch.float64, device="cuda") for v in (1.0, 0.1))

    def call():
        with torch.no_grad():
            t.reconstruct(source, target, alpha, epsilon)
            return t.apply(static)

    graph, out = _capture(call)
    torch.cuda.synchronize()
    return t, source, target, epsilon, graph, out


def test_eager_and_numpy_calls_after_a_held_replay_run_in_order():
    torch = _torch()
    shape, size = (192, 160), 64
    static = _frames(shape, 0, 0)
    t, source, target, epsilon, graph, out = _reconstructing_graph(shape, size, static)
    x2, frame_np = _frames(shape, 0, 2), _frames(shape, 0, 3).cpu().numpy()
    graph.replay()
    t.apply(x2)                                    # lays the replay's kernel out once: later eager calls read the layout
    torch.cuda.synchronize()
    for eps, numpy_call in ((0.3, False), (0.5, True)):
        fresh = rp.ArrayPSFTransform.construct(source, target, 1.0, eps)
        want_replay = fresh.apply(static).clone()
        want = fresh.apply(frame_np) if numpy_call else fresh.apply(x2).clone()
        epsilon.fill_(eps)
        torch.cuda.synchronize()
        held = torch.cuda.Stream()
        event = _hold(held)
        with torch.cuda.stream(held):
            graph.replay()                         # lays out the kernel of `eps`
        _assert_pending(event)
        # the current stream is not held: without the order the call would read the previous layout
        got = t.apply(frame_np) if numpy_call else t.apply(x2)
        torch.cuda.synchronize()
        assert _same(out, want_replay), eps
        if numpy_call:
            assert np.array_equal(got, want), eps
        else:
            assert _same(got, want), eps


def test_two_replays_sharing_a_plan_on_two_streams_run_one_after_the_other():
    torch = _torch()
    shape, size = (1024, 1024), 128
    s1, s2 = _frames(shape, 0, 0), _frames(shape, 0, 1)
    t, source, target, epsilon, g1, out1 = _reconstructing_graph(shape, size, s1)
    g2, out2 = _capture(lambda: t.apply(s2))       # lays out, in the graph, the kernel g1 builds
    g1.replay()
    g2.replay()
    fresh = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.3)
    want1, want2 = fresh.apply(s1).clone(), fresh.apply(s2).clone()
    epsilon.fill_(0.3)
    torch.cuda.synchronize()
    held, other = torch.cuda.Stream(), torch.cuda.Stream()
    event = _hold(held)
    with torch.cuda.stream(held):
        g1.replay()
    with torch.cuda.stream(other):
        g2.replay()                                # without the order it would read g1's kernel before g1 builds it
    _assert_pending(event)
    torch.cuda.synchronize()
    assert _same(out1, want1) and _same(out2, want2)


def _churn(like, n=4):
    """Allocate and fill blocks like ``like``, so that a block a graph reads but nobody keeps would be overwritten."""
    torch = _torch()
    return [torch.full_like(like, complex(7.0, -7.0) if like.is_complex() else 7.0) for _ in range(n)]


def test_eager_reconstruct_reaches_a_graph_that_lays_out_an_earlier_kernel():
    torch = _torch()
    shape = (192, 160)
    coords, source, target = _psf_setup(shape)
    values = source._values_cube.tensor.clone().requires_grad_()
    trainable = rp.ArrayPSF(rp.DeviceCube(coords, values))
    t = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.1)
    t.reconstruct(trainable, target, 1.0, 0.2)     # a kernel that requires grad: captured calls lay it out
    static = _frames(shape, 0, 0)

    def call():
        with torch.no_grad():
            return t.apply(static)

    graph, out = _capture(call)
    t.reconstruct(trainable, target, 1.0, 0.3)     # eager, after the capture
    junk = _churn(t._kernel_tensor)
    graph.replay()
    want = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.3).apply(static)
    torch.cuda.synchronize()
    assert _same(out, want)
    del junk
    # a kernel tensor the caller gave is not overwritten: reconstruct refuses and leaves the transform as it was
    user, kernel = _random_transform(shape, 64, requires_grad=True)

    def call_user():
        with torch.no_grad():
            return user.apply(static)

    _capture(call_user)
    with pytest.raises(RuntimeError, match="kernel tensor it was given"):
        user.reconstruct(source, target, 1.0, 0.3)
    assert user._kernel_tensor is kernel


def test_replay_after_an_eager_upload_of_the_same_host_fft_cube():
    torch = _torch()
    shape = (192, 160)
    coords, source, target = _psf_setup(shape)
    host_target = rp.ArrayPSF(rp.IndexedCube(coords, target.values), rp.IndexedCube(coords, target.fft_evaluations))
    t = rp.ArrayPSFTransform.construct(source, host_target, 1.0, 0.1)
    alpha, epsilon = (torch.tensor(v, dtype=torch.float64, device="cuda") for v in (1.0, 0.2))
    static = _frames(shape, 0, 0)

    def call():
        with torch.no_grad():
            t.reconstruct(source, host_target, alpha, epsilon)
            return t.apply(static)

    graph, out = _capture(call)
    other = rp.ArrayPSFTransform.construct(source, host_target, 1.0, 0.1)   # an eager upload of the same host cube
    junk = _churn(other._kernel_tensor)
    graph.replay()
    want = rp.ArrayPSFTransform.construct(source, target, 1.0, 0.2).apply(static)
    torch.cuda.synchronize()
    assert _same(out, want)
    del junk


# --------------------------------------------------------------------------------------------- kernel updates, fitting
def test_optimizer_step_between_replays_reaches_the_next_replay():
    torch = _torch()
    shape, size = (192, 160), 64
    t, kernel = _random_transform(shape, size, requires_grad=True)
    static = _frames(shape, 0, 0)
    with torch.no_grad():
        t.apply(static)                             # the native transform and its first layout, outside the capture
    opt = torch.optim.SGD([kernel], lr=0.05)

    def call():
        with torch.no_grad():
            return t.apply(static)

    graph, out = _capture(call)
    for seed in range(1, REPLAYS + 1):
        kernel.grad = torch.randn(kernel.shape, dtype=kernel.dtype, device="cuda",
                                  generator=torch.Generator(device="cuda").manual_seed(seed))
        opt.step()
        graph.replay()
        with torch.no_grad():
            want = t.apply(static)
        assert _same(out, want), seed


FIT = {"config1_float32": ((1024, 1024), 128, 8, "float32"), "p64_float64": ((192, 160), 64, 2, "float64")}


class _Fit:
    """PSF values, alpha and epsilon that require grad, a target and frames; ``step`` is one fitting step."""

    def __init__(self, case):
        torch = _torch()
        shape, size, batch, dtype = FIT[case]
        self.dtype = dtype
        real = torch.float32 if dtype == "float32" else torch.float64
        coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(shape, size)]
        src = torch.from_numpy(oracle.coma_psf_cube(coords, size, shape)).cuda().to(real)
        tgt = torch.from_numpy(oracle.gaussian_psf_cube(len(coords), size, 3.0)).cuda().to(real)
        self.values = src.clone().requires_grad_()
        self.alpha = torch.tensor(1.2, dtype=torch.float64, device="cuda", requires_grad=True)
        self.epsilon = torch.tensor(0.15, dtype=torch.float64, device="cuda", requires_grad=True)
        self.source = rp.ArrayPSF(rp.DeviceCube(coords, self.values))
        self.target = rp.ArrayPSF(rp.DeviceCube(coords, tgt))
        self.target.fft_cube
        self.x = _frames(shape, batch, 7, real)
        ref = rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(coords, src)), self.target, 1.0, 0.1)
        self.y = ref.apply(self.x, dtype=dtype).detach()
        self.transform = rp.ArrayPSFTransform.construct(self.source, self.target, self.alpha.detach(),
                                                        self.epsilon.detach())
        self.params = [self.values, self.alpha, self.epsilon]
        self.initial = [p.detach().clone() for p in self.params]
        self.opt = torch.optim.Adam(self.params, lr=1e-3, capturable=True)

    def step(self):
        self.transform.reconstruct(self.source, self.target, self.alpha, self.epsilon)
        out = self.transform.apply(self.x, dtype=self.dtype)
        loss = ((out - self.y) ** 2).mean()
        loss.backward()
        self.opt.step()

    def reset(self):
        torch = _torch()
        with torch.no_grad():
            for p, p0 in zip(self.params, self.initial):
                p.copy_(p0)
            for state in self.opt.state.values():
                for value in state.values():
                    if torch.is_tensor(value):
                        value.zero_()


@pytest.mark.parametrize("case", sorted(FIT))
def test_captured_fitting_step_matches_eager_steps(case):
    torch = _torch()
    steps = 5
    eager = _Fit(case)
    for _ in range(steps):
        eager.opt.zero_grad(set_to_none=True)
        eager.step()
    torch.cuda.synchronize()
    fit = _Fit(case)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fit.opt.zero_grad(set_to_none=True)
            fit.step()
    torch.cuda.current_stream().wait_stream(side)
    fit.opt.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fit.step()
    fit.reset()
    for _ in range(steps):
        graph.replay()
    torch.cuda.synchronize()
    for got, want in zip(fit.params, eager.params):
        assert _same(got.detach(), want.detach())


# --------------------------------------------------------------------------------------------- device scalars
ALPHA_EPSILON = [(0.5, 0.05), (1.5, 1.0), (1.0, 0.1), (3.0, 0.2), (1.0, 0.2), (1.5, 0.2), (0.5, 0.2), (1.0, 0.0)]


def _special_cube(seed):
    """Random bins plus S = 0, T = 0, S = T = 0, NaN and inf inputs, each with G = 0 and with G != 0."""
    rng = np.random.default_rng(seed)
    n = 4096

    def rc():
        return rng.normal(size=n) + 1j * rng.normal(size=n)

    s, t, g = rc(), rc(), rc()
    pos = 0
    for sval, tval in ((0, None), (None, 0), (0, 0), (np.nan, None), (None, np.inf)):
        for g_zero in (True, False):
            for _ in range(8):
                if sval is not None:
                    s[pos] = sval
                if tval is not None:
                    t[pos] = tval
                if g_zero:
                    g[pos] = 0
                pos += 1
    return s, t, g


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("alpha,epsilon", ALPHA_EPSILON)
def test_device_scalar_entry_points_are_bit_identical(alpha, epsilon, dtype):
    torch = _torch()
    cplx = torch.complex64 if dtype == "float32" else torch.complex128
    code = _native.F32 if dtype == "float32" else _native.F64
    lib = _native.load()
    stream = _native.current_stream_ptr(torch)
    _, source, target = _psf_setup()
    cubes = [(source.fft_cube.tensor.to(cplx), target.fft_cube.tensor.to(cplx),
              torch.randn(source.fft_cube.tensor.shape, dtype=cplx, device="cuda"))]
    cubes.append(tuple(torch.from_numpy(c).cuda().to(cplx) for c in _special_cube(3)))
    ae = torch.tensor([alpha, epsilon], dtype=torch.float64, device="cuda")
    for s, t, g in cubes:
        n = s.numel()
        k_host, k_dev = torch.empty_like(s), torch.empty_like(s)
        _native.check(lib.rpsf_construct_kernel(s.data_ptr(), t.data_ptr(), k_host.data_ptr(), n, code, alpha, epsilon,
                                                0, stream))
        _native.check(lib.rpsf_construct_kernel_dev(s.data_ptr(), t.data_ptr(), k_dev.data_ptr(), n, code, ae.data_ptr(),
                                                    0, stream))
        assert _same(k_host, k_dev)
        outs = []
        for on_device in (False, True):
            gs, gt = torch.empty_like(s), torch.empty_like(s)
            sums = torch.empty(2, dtype=torch.float64, device="cuda")
            if on_device:
                rc = lib.rpsf_construct_kernel_backward_dev(s.data_ptr(), t.data_ptr(), g.data_ptr(), n, code,
                                                            ae.data_ptr(), gs.data_ptr(), gt.data_ptr(), sums.data_ptr(),
                                                            0, stream)
            else:
                rc = lib.rpsf_construct_kernel_backward(s.data_ptr(), t.data_ptr(), g.data_ptr(), n, code, alpha, epsilon,
                                                        gs.data_ptr(), gt.data_ptr(), sums.data_ptr(), 0, stream)
            _native.check(rc)
            outs.append((gs, gt, sums))
        for a, b in zip(*outs):
            assert _same(a, b)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_construct_with_tensor_scalars_is_bit_identical_and_does_not_synchronise(dtype):
    torch = _torch()
    real = torch.float32 if dtype == "float32" else torch.float64
    coords, source, target = _psf_setup()
    values = source._values_cube.tensor.to(real)
    results = {}
    for kind in ("float", "tensor"):
        v = values.clone().requires_grad_()
        psf = rp.ArrayPSF(rp.DeviceCube(coords, v))
        if kind == "float":
            alpha, epsilon = 1.25, 0.125                  # exact in float32, so both kinds hold the same values
        else:
            alpha = torch.tensor(1.25, dtype=real, device="cuda", requires_grad=True)
            epsilon = torch.tensor(0.125, dtype=torch.float64, device="cuda", requires_grad=True)
        torch.cuda.synchronize()
        if kind == "tensor":
            torch.cuda.set_sync_debug_mode("error")
        try:
            kernel = rp.ArrayPSFTransform.construct(psf, target, alpha, epsilon)._kernel_tensor
            (kernel.abs() ** 2).sum().backward()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        results[kind] = (kernel.detach(), v.grad)
        if kind == "tensor":
            assert alpha.grad is not None and epsilon.grad is not None and alpha.grad.dtype == real
    for a, b in zip(results["float"], results["tensor"]):
        assert _same(a, b)
    # without autograd too
    plain = rp.ArrayPSFTransform.construct(source, target, 1.3, 0.1)._kernel_tensor
    alpha, epsilon = (torch.tensor(v, dtype=torch.float64, device="cuda") for v in (1.3, 0.1))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        dev = rp.ArrayPSFTransform.construct(source, target, alpha, epsilon)._kernel_tensor
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert _same(plain, dev)


# --------------------------------------------------------------------------------------------- plans and refusals
def test_captured_plan_survives_the_cache_bound():
    torch = _torch()
    shape, size = (192, 160), 64
    t, _ = _random_transform(shape, size)
    static = _frames(shape, 0, 0)
    graph, out = _capture(lambda: t.apply(static))
    nt = t._native[("float32", torch.cuda.current_device())]
    captured = [k for k in nt._plans if k[:2] == shape]
    assert len(captured) == 1 and captured[0] in nt._pinned
    for i in range(nt.MAX_PLANS + 1):               # widths other than the captured one: every call makes a plan
        t.apply(_frames((192, 176 + 16 * i), 0, 100 + i))
    assert all(k[:2] != shape for k in list(nt._plans)[-nt.MAX_PLANS:])
    assert captured[0] in nt._plans
    x = _frames(shape, 0, 9)
    static.copy_(x)
    graph.replay()
    assert _same(out, t.apply(x))


def test_refusals_inside_a_capture_leave_the_device_usable():
    torch = _torch()
    shape, size = (192, 160), 64
    t, _ = _random_transform(shape, size)
    x = _frames(shape, 0, 0)
    want = t.apply(x).clone()
    other_shape = _frames((176, 160), 0, 1)
    untouched, _ = _random_transform(shape, size, seed=2)
    host_frame = x.cpu().numpy()
    torch.cuda.synchronize()
    cases = {
        "plan": (lambda: t.apply(other_shape), "no plan"),
        "layout": (lambda: untouched.apply(x), "no native state"),
        "numpy": (lambda: t.apply(host_frame), "numpy array"),
    }
    for name, (call, words) in cases.items():
        graph = torch.cuda.CUDAGraph()
        with pytest.raises(RuntimeError, match=words):
            with torch.cuda.graph(graph):
                call()
        assert _same(t.apply(x), want), name
        assert not torch.cuda.is_current_stream_capturing()
