"""Calls from several CUDA streams, and the default dtype on every path.

The library owns device state that outlives a call: the laid-out transfer kernel (and its conjugate), and each plan's
spectrum workspace, adjoint box and saturation scratch.  A call must see the kernel as of the moment it was issued and
must not share a plan's scratch with a call still queued on another stream, whatever streams the earlier calls or
kernel layouts used (INTEGRATION.md, "Streams").

The races are made deterministic by holding one stream with a spinning kernel (``torch.cuda._sleep``) and issuing the
calls under test behind it without synchronising; each test first checks that the hold is still pending, so a set-up
that synchronised by accident fails instead of passing vacuously.  Expected values are the same calls made with the
device drained before and after; the kernels are run-to-run bit-stable, so they compare with ``torch.equal`` /
``np.array_equal``.  Each hazard also compares its expected value with the float64 oracle (1e-5 x max in float32).
"""
import numpy as np
import pytest

import regularizepsf_b200 as rp
from oracle import cpu_oracle as oracle
from regularizepsf_b200 import _native
from tests.adjoint_oracle import apply_transform_adjoint
from tests.kernel_gradient_oracle import transfer_kernel_gradient

pytestmark = pytest.mark.gpu

TOL = {"float32": 1e-5, "float64": 1e-10}
HOLD_SECONDS = 0.3
ALPHA, EPSILONS = 1.0, (0.1, 0.3)                 # the kernels K0 and K1
GEOMETRIES = {"p64": ((192, 160), 64), "p256_2048": ((2048, 2048), 256), "embedded_p48": ((150, 130), 48)}
_HOLD = {}


def _torch():
    import torch
    return torch


@pytest.fixture(scope="module", autouse=True)
def _native_must_be_loaded():
    torch = _torch()
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    _native.load()
    # cycles of torch.cuda._sleep per second on this device
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


@pytest.fixture
def float64_default():
    rp.set_default_dtype("float64")
    try:
        yield
    finally:
        rp.set_default_dtype("float32")


def _hold(stream=None):
    """Keep ``stream`` (default: the current one) busy for about HOLD_SECONDS; the event recorded right behind it."""
    torch = _torch()
    with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
        torch.cuda._sleep(_HOLD["cycles"])
        event = torch.cuda.Event()
        event.record()
    return event


def _assert_pending(event):
    assert not event.query(), "the held stream finished before the calls under test were issued: nothing was raced"


def _drained(fn):
    torch = _torch()
    torch.cuda.synchronize()
    out = fn()
    torch.cuda.synchronize()
    return out


class _Setup:
    """One geometry: device PSF models, the kernels K0 and K1 they make, two frames (numpy float32 and on the device)."""

    def __init__(self, name):
        torch = _torch()
        self.shape, self.size = GEOMETRIES[name]
        self.coords = [tuple(int(v) for v in c) for c in rp.calculate_covering(self.shape, self.size)]
        n = len(self.coords)
        self.src = oracle.coma_psf_cube(self.coords, self.size, self.shape)
        self.tgt = oracle.gaussian_psf_cube(n, self.size, 3.0)
        self.values = torch.from_numpy(self.src).cuda()
        self.source = rp.ArrayPSF(rp.DeviceCube(self.coords, self.values))
        self.target = rp.ArrayPSF(rp.DeviceCube(self.coords, torch.from_numpy(self.tgt).cuda()))
        for psf in (self.source, self.target):
            psf.fft_cube                                  # the spectra exist before any stream is held
        self.k = [rp.ArrayPSFTransform.construct(self.source, self.target, ALPHA, e)._kernel_tensor for e in EPSILONS]
        self.frames = [oracle.starfield(self.shape, seed=s) for s in (11, 12)]
        self.x = [torch.from_numpy(f).cuda() for f in self.frames]
        self.grad = torch.from_numpy(np.random.default_rng(5).normal(size=self.shape).astype(np.float32)).cuda()
        self.sat_threshold = float(np.quantile(self.frames[0], 0.999))
        torch.cuda.synchronize()

    def oracle_kernel(self, which):
        return oracle.transfer_kernel(oracle.psf_fft(self.src), oracle.psf_fft(self.tgt), ALPHA, EPSILONS[which])

    def transform(self, kernel, trainable=False):
        k = kernel.clone().requires_grad_() if trainable else kernel
        return rp.ArrayPSFTransform(rp.DeviceCube(self.coords, k))


_SETUPS = {}


def _setup(name="p64"):
    if name not in _SETUPS:
        _SETUPS[name] = _Setup(name)
    return _SETUPS[name]


def _check_oracle(got, want):
    got = got.cpu().numpy() if hasattr(got, "cpu") else np.asarray(got)
    err = float(np.max(np.abs(got.astype(np.complex128 if np.iscomplexobj(got) else np.float64) - want)))
    assert err <= TOL["float32"] * float(np.max(np.abs(want))), err


# --------------------------------------------------------------------------------------------- default dtype
@pytest.mark.parametrize("input_dtype", ["float32", "float64"])
def test_device_apply_follows_the_default_dtype(float64_default, input_dtype):
    torch = _torch()
    s = _setup()
    t = rp.ArrayPSFTransform(rp.DeviceCube(s.coords, torch.from_numpy(s.oracle_kernel(0)).cuda()))
    x = s.x[0].to(getattr(torch, input_dtype))
    y = t.apply(x)
    assert y.dtype == torch.float64, f"{y.dtype} returned after set_default_dtype('float64')"
    assert torch.equal(y, t.apply(x, dtype="float64"))
    want = oracle.apply_transform(s.frames[0], s.coords, s.oracle_kernel(0))
    assert float(np.max(np.abs(y.cpu().numpy() - want))) <= TOL["float64"] * float(np.max(np.abs(want)))


def test_other_entry_points_follow_the_default_dtype(float64_default):
    torch = _torch()
    s = _setup()
    kernel = s.oracle_kernel(0)
    t = rp.ArrayPSFTransform(rp.DeviceCube(s.coords, torch.from_numpy(kernel).cuda()))
    x, g = s.x[0], s.grad

    def close(got, want):
        got = got.cpu().numpy() if hasattr(got, "cpu") else got
        assert float(np.max(np.abs(got - want))) <= TOL["float64"] * float(np.max(np.abs(want)))

    adj = t.apply_adjoint(g)
    assert adj.dtype == torch.float64 and torch.equal(adj, t.apply_adjoint(g, dtype="float64"))
    close(adj, apply_transform_adjoint(g.cpu().numpy().astype(np.float64), s.coords, kernel))
    kg = t.transfer_kernel_gradient(x, g)
    assert kg.dtype == torch.complex128 and torch.equal(kg, t.transfer_kernel_gradient(x, g, dtype="float64"))
    close(kg, transfer_kernel_gradient(s.frames[0], g.cpu().numpy(), s.coords, s.size))
    host = t.apply(s.frames[0])
    assert np.array_equal(host, t.apply(s.frames[0], dtype="float64"))
    close(host, oracle.apply_transform(s.frames[0], s.coords, kernel))
    assert np.array_equal(t.apply_adjoint(s.frames[0]), t.apply_adjoint(s.frames[0], dtype="float64"))
    assert np.array_equal(t.transfer_kernel_gradient(s.frames[0], g.cpu().numpy()),
                          t.transfer_kernel_gradient(s.frames[0], g.cpu().numpy(), dtype="float64"))
    with torch.no_grad():
        lifted = s.x[0].clone().requires_grad_()
    assert t.apply(lifted).dtype == torch.float64


# --------------------------------------------------------------------------------------------- host path after a re-layout
_HOST_CASES = [(v, g, False) for g in GEOMETRIES for v in ("reconstruct", "inplace", "side_first_layout")]
_HOST_CASES.append(("reconstruct", "p64", True))


@pytest.mark.parametrize("variant,geometry,saturation", _HOST_CASES)
def test_host_apply_sees_a_kernel_laid_out_on_a_held_stream(variant, geometry, saturation):
    """A numpy call runs its kernels on private streams; the kernel it must use is laid out on the caller's stream,
    which is still held when the call is issued."""
    torch = _torch()
    s = _setup(geometry)
    kw = {"saturation_threshold": s.sat_threshold} if saturation else {}
    frame = s.frames[0]
    # (the first-layout case gets a kernel of its own, so that a freshly allocated layout cannot hold it by chance)
    k1 = s.k[1] * 0.75 if variant == "side_first_layout" else s.k[1]
    expected = s.transform(k1)
    want = _drained(lambda: expected.apply(frame, **kw))
    if variant == "reconstruct":
        t = rp.ArrayPSFTransform.construct(s.source, s.target, ALPHA, EPSILONS[0])
        _drained(lambda: t.apply(frame, **kw))
        held = _hold()
        t.reconstruct(s.source, s.target, ALPHA, EPSILONS[1])
        _assert_pending(held)
        got = t.apply(frame, **kw)
    elif variant == "inplace":
        t = s.transform(s.k[0], trainable=True)
        _drained(lambda: t.apply(frame, **kw))
        held = _hold()
        with torch.no_grad():
            t._kernel_tensor.copy_(k1)
        _assert_pending(held)
        got = t.apply(frame, **kw)
    else:
        t = s.transform(s.k[0], trainable=True)
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            held = _hold(side)
            with torch.no_grad():
                t._kernel_tensor.copy_(k1)
            _assert_pending(held)
            # the first call: the layout is issued on `side`, behind the hold.  (At 2048^2 this call also allocates
            # the new plan's pinned staging buffers, and a page-locked allocation synchronises the device: there the
            # case guards the result rather than racing.)
            got = t.apply(frame, **kw)
    torch.cuda.synchronize()
    old = _drained(lambda: s.transform(s.k[0]).apply(frame, **kw))
    assert not np.array_equal(old, want)
    assert not np.array_equal(got, old), "the host call used the kernel from before the re-layout"
    assert np.array_equal(got, want)
    if geometry == "p64" and variant == "reconstruct" and not saturation:
        _check_oracle(want, oracle.apply_transform(frame, s.coords, s.oracle_kernel(1)))


# --------------------------------------------------------------------------------------------- first layout, another stream
def test_first_layout_on_a_held_stream_orders_a_call_on_another():
    torch = _torch()
    s = _setup()
    kernel = s.k[0] * 1.25                       # a kernel of its own (see above)
    expected = s.transform(kernel)
    want = _drained(lambda: expected.apply(s.x[0]))
    t = s.transform(kernel)
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    held = _hold(a)
    with torch.cuda.stream(a):
        ya = t.apply(s.x[0])                     # lays the kernel out on `a`, behind the hold
    with torch.cuda.stream(b):
        yb = t.apply(s.x[0])
    _assert_pending(held)
    torch.cuda.synchronize()
    assert torch.equal(yb, want), "the call on the second stream ran before the first layout"
    assert torch.equal(ya, want)
    _check_oracle(want, oracle.apply_transform(s.frames[0], s.coords, 1.25 * s.oracle_kernel(0)))


# --------------------------------------------------------------------------------------------- one plan, two streams
@pytest.mark.parametrize("kind", ["apply", "apply_adjoint", "kernel_gradient_then_apply", "device_then_host"])
def test_streams_sharing_a_plan_are_ordered(kind):
    """Two calls of one geometry share a plan (its workspace, box and scratch): the second, on another stream, must
    wait for the first, queued behind a hold."""
    torch = _torch()
    s = _setup()
    t = s.transform(s.k[0])
    x1, x2 = s.x
    first = {"apply": lambda: t.apply(x1), "apply_adjoint": lambda: t.apply_adjoint(x1),
             "kernel_gradient_then_apply": lambda: t.transfer_kernel_gradient(x1, s.grad),
             "device_then_host": lambda: t.apply(x1)}[kind]
    second = {"apply_adjoint": lambda: t.apply_adjoint(x2), "device_then_host": lambda: t.apply(s.frames[1])}.get(
        kind, lambda: t.apply(x2))
    want1, want2 = _drained(first), _drained(second)      # (this also makes the plans)
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    held = _hold(a)
    with torch.cuda.stream(a):
        r1 = first()
        done_a = torch.cuda.Event()
        done_a.record()
    if kind == "device_then_host":
        _assert_pending(held)
        r2 = second()                            # synchronous: returns when its own streams are done
    else:
        with torch.cuda.stream(b):
            r2 = second()
        _assert_pending(held)
        b.synchronize()
    assert done_a.query(), "the second call finished while the first, sharing its plan, was still queued"
    torch.cuda.synchronize()
    same = np.array_equal if kind == "device_then_host" else torch.equal
    assert torch.equal(r1, want1) and same(r2, want2)
    kernel = s.oracle_kernel(0)
    if kind == "apply":
        _check_oracle(want2, oracle.apply_transform(s.frames[1], s.coords, kernel))
    elif kind == "apply_adjoint":
        _check_oracle(want2, apply_transform_adjoint(s.frames[1].astype(np.float64), s.coords, kernel))
    elif kind == "kernel_gradient_then_apply":
        _check_oracle(want1, transfer_kernel_gradient(s.frames[0], s.grad.cpu().numpy(), s.coords, s.size))
    else:
        _check_oracle(want2, oracle.apply_transform(s.frames[1], s.coords, kernel))


# --------------------------------------------------------------------------------------------- write after read
@pytest.mark.parametrize("kind", ["reconstruct", "inplace", "adjoint_reconstruct"])
def test_a_call_sees_the_kernel_it_was_issued_with(kind):
    """y0 is queued on a held stream with K0; the kernel becomes K1 on another stream and y1 follows there."""
    torch = _torch()
    s = _setup()
    x = s.x[0]
    adjoint = kind == "adjoint_reconstruct"
    if kind == "inplace":
        t = s.transform(s.k[0], trainable=True)
    else:
        t = rp.ArrayPSFTransform.construct(s.source, s.target, ALPHA, EPSILONS[0])
    with torch.no_grad():
        call = (lambda tr: tr.apply_adjoint(x)) if adjoint else (lambda tr: tr.apply(x))
        _drained(lambda: call(t))                           # laid out, plans made
        want0 = _drained(lambda: call(s.transform(s.k[0])))
        want1 = _drained(lambda: call(s.transform(s.k[1])))
        a, b = torch.cuda.Stream(), torch.cuda.Stream()
        torch.cuda.synchronize()
        held = _hold(a)
        with torch.cuda.stream(a):
            y0 = call(t)
        with torch.cuda.stream(b):
            if kind == "inplace":
                t._kernel_tensor.copy_(s.k[1])
            else:
                t.reconstruct(s.source, s.target, ALPHA, EPSILONS[1])
            y1 = call(t)
        _assert_pending(held)
    torch.cuda.synchronize()
    assert not torch.equal(want0, want1)
    assert not torch.equal(y0, want1), "y0 was computed with the kernel laid out after it was issued"
    assert torch.equal(y0, want0) and torch.equal(y1, want1)
    for got, which in ((want0, 0), (want1, 1)):
        kernel = s.oracle_kernel(which)
        _check_oracle(got, apply_transform_adjoint(s.frames[0].astype(np.float64), s.coords, kernel) if adjoint
                      else oracle.apply_transform(s.frames[0], s.coords, kernel))


# --------------------------------------------------------------------------------------------- user tensors (guards)
@pytest.mark.parametrize("kind", ["apply", "apply_adjoint", "kernel_gradient", "construct", "psf_fft"])
def test_inputs_written_on_a_held_side_stream(kind):
    """Inputs written on a side stream behind a hold, then the call on that stream: PyTorch's stream order."""
    torch = _torch()
    s = _setup()
    t = s.transform(s.k[0])
    ops = {
        "apply": lambda x, v: t.apply(x),
        "apply_adjoint": lambda x, v: t.apply_adjoint(x),
        "kernel_gradient": lambda x, v: t.transfer_kernel_gradient(x, s.grad),
        "construct": lambda x, v: rp.ArrayPSFTransform.construct(rp.ArrayPSF(rp.DeviceCube(s.coords, v)),
                                                                 s.target, ALPHA, EPSILONS[0])._kernel_tensor,
        "psf_fft": lambda x, v: rp.ArrayPSF(rp.DeviceCube(s.coords, v)).fft_cube.tensor,
    }
    op = ops[kind]
    want = _drained(lambda: op(s.x[0], s.values))
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    held = _hold(side)
    with torch.cuda.stream(side):
        x = torch.empty_like(s.x[0])
        x.copy_(s.x[0])
        v = torch.empty_like(s.values)
        v.copy_(s.values)
        got = op(x, v)
    _assert_pending(held)
    torch.cuda.synchronize()
    assert torch.equal(got, want)


def test_backward_runs_on_the_forward_stream():
    torch = _torch()
    s = _setup()
    t = s.transform(s.k[0], trainable=True)
    kernel = t._kernel_tensor
    g = s.grad
    x = s.x[0].clone().requires_grad_()

    def forward_backward():
        x.grad = kernel.grad = None
        (t.apply(x) * g).sum().backward()

    _drained(forward_backward)                                  # plans of both directions
    with torch.no_grad():
        want_x = _drained(lambda: t.apply_adjoint(g))
        want_k = _drained(lambda: t.transfer_kernel_gradient(s.x[0], g).to(kernel.dtype))
    x.grad = kernel.grad = None
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    held = _hold(side)
    with torch.cuda.stream(side):
        loss = (t.apply(x) * g).sum()
    loss.backward()
    _assert_pending(held)
    torch.cuda.synchronize()
    assert torch.equal(x.grad, want_x)
    assert torch.equal(kernel.grad, want_k)


def test_chain_alternating_between_two_streams():
    torch = _torch()
    s = _setup()
    t = s.transform(s.k[0])

    def chain(streams):
        outs, prev = [s.x[0]], None
        for i in range(6):
            stream = streams[i % len(streams)]
            if prev is not None:
                stream.wait_stream(prev)
            with torch.cuda.stream(stream):
                outs.append(t.apply(outs[-1]) if i % 2 == 0 else t.apply_adjoint(outs[-1]))
            prev = stream
        return outs, prev

    want = _drained(lambda: chain([torch.cuda.current_stream()])[0])
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    held = _hold(a)
    outs, last = chain([a, b])
    _assert_pending(held)
    torch.cuda.current_stream().wait_stream(last)
    torch.cuda.synchronize()
    for got, expected in zip(outs[1:], want[1:], strict=True):
        assert torch.equal(got, expected)


def _device_count():
    torch = _torch()
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.skipif(_device_count() < 2, reason="needs two CUDA devices")
def test_second_device_orders_a_kernel_update():
    """The write-after-read case on a second device: its transform, plans and event live there."""
    torch = _torch()
    s = _setup()
    k0, k1 = (k.to("cuda:1") for k in s.k)
    x = s.x[0].to("cuda:1")
    t = rp.ArrayPSFTransform(rp.DeviceCube(s.coords, k0.clone().requires_grad_()))
    with torch.no_grad(), torch.cuda.device(1):
        _drained(lambda: t.apply(x))
        want0 = _drained(lambda: rp.ArrayPSFTransform(rp.DeviceCube(s.coords, k0)).apply(x))
        want1 = _drained(lambda: rp.ArrayPSFTransform(rp.DeviceCube(s.coords, k1)).apply(x))
        a, b = torch.cuda.Stream(1), torch.cuda.Stream(1)
        torch.cuda.synchronize(1)
        held = _hold(a)
        with torch.cuda.stream(a):
            y0 = t.apply(x)
        with torch.cuda.stream(b):
            t._kernel_tensor.copy_(k1)
            y1 = t.apply(x)
        _assert_pending(held)
        torch.cuda.synchronize(1)
    assert torch.equal(y0, want0) and torch.equal(y1, want1)
