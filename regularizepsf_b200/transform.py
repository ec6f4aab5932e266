"""``ArrayPSFTransform`` — the drop-in for the reference's correction path, running on a B200.

Mirrors regularizepsf/transform.py:25-177 (``__init__``, ``psf_shape``, ``coordinates``,
``__len__``, ``construct``, ``apply``, ``__eq__``) with the same names, argument order, defaults
and error types.  ``construct`` and ``apply`` are thin calls through the C ABI
(include/rpsf_b200.h) into hand-written sm_100a kernels; see DESIGN.md.  No CPU fallback.
"""
from __future__ import annotations

import ctypes
import math
import weakref

import numpy as np

from regularizepsf_b200 import _native
from regularizepsf_b200.device import DeviceCube, cube_tensor, pinned_empty
from regularizepsf_b200.exceptions import IncorrectShapeError, InvalidCoordinateError
from regularizepsf_b200.util import IndexedCube

_DTYPES = {"float32": _native.F32, "float64": _native.F64}
_NATIVE_SIZES = (16, 32, 64, 128, 256, 512)           # patch sizes with an FFT length of their own (no embedding)
_default_dtype = "float32"


def set_default_dtype(name: str) -> None:
    """Select the arithmetic precision of ``apply``: "float32" (default) or "float64" (validation mode)."""
    global _default_dtype
    if name not in _DTYPES:
        raise ValueError(f"dtype must be one of {sorted(_DTYPES)}, got {name!r}")
    _default_dtype = name


def _normalize_dtype(dtype) -> str:
    if dtype is None:
        return _default_dtype
    name = np.dtype(dtype).name if not isinstance(dtype, str) else dtype
    if name not in _DTYPES:
        raise ValueError(f"dtype must be one of {sorted(_DTYPES)}, got {dtype!r}")
    return name


def _destroy(lib, kind: str, handle: int) -> None:
    try:
        getattr(lib, f"rpsf_{kind}_destroy")(handle)
    except Exception:  # pragma: no cover - interpreter shutdown
        pass


class _NativeTransform:
    """Owns one ``rpsf_transform`` (per compute dtype) and its plans."""

    def __init__(self, coords: np.ndarray, patch: int, dtype_name: str, device: int, kernel_tensor, stream: int,
                 keep: np.ndarray | None = None):
        self.lib = _native.load()
        self.dtype_name = dtype_name
        self.device = device
        handle = ctypes.c_void_p()
        if keep is None:
            _native.check(self.lib.rpsf_transform_create(
                ctypes.byref(handle), coords.ctypes.data, coords.shape[0], patch, _DTYPES[dtype_name], device))
        else:       # a row-slab shard: the whole coordinate list, kernels of the kept patches only
            keep = np.ascontiguousarray(keep, dtype=np.uint8)
            _native.check(self.lib.rpsf_transform_create_subset(
                ctypes.byref(handle), coords.ctypes.data, coords.shape[0], patch, _DTYPES[dtype_name], device,
                keep.ctypes.data))
        self.handle = handle.value
        # geometry key -> plan handle, most recently used last (bounded: see plan())
        self._plans: dict[tuple, int] = {}
        self._saturation: dict[int, tuple] = {}          # plan handle -> the saturation settings it was last given
        self._finalizer = weakref.finalize(self, _NativeTransform._cleanup, self.lib, self.handle, self._plans)
        # a kernel tensor that requires grad may be updated in place (optimizer.step()): the tensor and the version it
        # had when it was laid out, so that the next call lays it out again (ArrayPSFTransform._native_transform)
        self.kernel_source = None
        self.kernel_version = None
        self.captured = False           # a CUDA graph holds calls of this transform (reconstruct lays out at once)
        # the kernel tensors captured layouts read, kept alive with the transform: [(tensor, made by construct)]
        self.graph_sources: list = []
        self.set_kernel(kernel_tensor, stream)

    def set_kernel(self, kernel_tensor, stream: int) -> None:
        """Lay out ``kernel_tensor`` (contiguous, on this device) for the kernels; stream-ordered on ``stream``."""
        kcode = _native.F32 if str(kernel_tensor.dtype) == "torch.complex64" else _native.F64
        _native.check(self.lib.rpsf_transform_set_kernel(self.handle, kernel_tensor.data_ptr(), kcode, stream))

    @staticmethod
    def _cleanup(lib, handle, plans):
        for plan in plans.values():
            _destroy(lib, "plan", plan)
        plans.clear()
        _destroy(lib, "transform", handle)

    #: keys of plans a CUDA graph has captured: never evicted, freed with the transform (a replay uses their workspaces)
    _pinned: frozenset = frozenset()

    #: at most this many plans stay alive per transform and compute dtype; each owns max_batch spectrum
    #: workspaces (75.8 MB per 2048^2 / 256-px frame), so an unbounded cache is an HBM leak
    MAX_PLANS = 6

    def plan(self, height: int, width: int, pad_mode: int, row_begin: int, row_end: int, max_batch: int,
             adjoint: bool = False, capturing: bool = False) -> int:
        """Plan for this geometry able to take ``max_batch`` frames per call (``adjoint``: the transpose of the
        whole-frame plan, ``rpsf_plan_create_adjoint``; it has workspaces of its own).

        A cached plan of the same geometry is reused when its capacity is in [max_batch, 2 * max_batch]
        (``rpsf_apply`` accepts any batch up to the plan's; the factor keeps a single-frame call off a plan
        whose work lists were cut for large batches).  Plans are evicted least-recently-used beyond
        ``MAX_PLANS``; eviction calls ``rpsf_plan_destroy`` (its ``cudaFree`` waits for work in flight).

        ``capturing``: the call is being captured in a CUDA graph.  The plan must exist (creating one allocates and
        synchronises: RuntimeError), and it is pinned: never evicted, freed with the transform, since every replay of
        the graph uses its workspaces.
        """
        geometry = (height, width, pad_mode, row_begin, row_end, adjoint)
        exact = geometry + (max_batch,)
        if exact in self._plans:
            if next(reversed(self._plans)) != exact:
                self._plans[exact] = self._plans.pop(exact)
            if capturing:
                self._pinned = self._pinned | {exact}
            return self._plans[exact]
        best = None
        for key in self._plans:
            if key[:-1] == geometry and max_batch <= key[-1] <= 2 * max_batch and (best is None or key[-1] < best[-1]):
                best = key
        if best is not None:
            plan = self._plans.pop(best)
            self._plans[best] = plan                      # most recently used last
            if capturing:
                self._pinned = self._pinned | {best}
            return plan
        if capturing:
            raise RuntimeError(f"no plan for {'adjoint ' if adjoint else ''}frames of {height} x {width} (pad mode "
                               f"{pad_mode}, rows [{row_begin}, {row_end}), {max_batch} frames) exists, and creating one "
                               "cannot be captured in a CUDA graph: run the same call once before capturing")
        out = ctypes.c_void_p()
        if adjoint:
            _native.check(self.lib.rpsf_plan_create_adjoint(ctypes.byref(out), self.handle, height, width, pad_mode,
                                                            max_batch))
        else:
            _native.check(self.lib.rpsf_plan_create(ctypes.byref(out), self.handle, height, width, pad_mode,
                                                    row_begin, row_end, max_batch))
        self._plans[geometry + (max_batch,)] = out.value
        while len(self._plans) - len(self._pinned) > self.MAX_PLANS:
            oldest = next(key for key in self._plans if key not in self._pinned)
            handle = self._plans.pop(oldest)
            self._saturation.pop(handle, None)
            _destroy(self.lib, "plan", handle)
        return out.value

    def set_saturation(self, plan: int, sat: tuple) -> None:
        """``rpsf_plan_set_saturation`` only when the settings of this plan change."""
        if self._saturation.get(plan) != sat:
            _native.check(self.lib.rpsf_plan_set_saturation(plan, *sat))
            self._saturation[plan] = sat

    def plan_info(self, plan: int) -> dict:
        info = (ctypes.c_int64 * 9)()
        _native.check(self.lib.rpsf_plan_info(plan, info))
        return {"active_patches": info[0], "colours": info[1], "workspace_bytes": info[2],
                "rows_read": (info[3], info[4]), "colour0_tiles_band": bool(info[5]),
                "overlap_add": {2: "streaming chains", 1: "row-pair gather", 0: "colour phases"}[int(info[6])],
                "gather_teams": info[7], "overlap_chunks": info[8]}


class ArrayPSFTransform:
    """A source→target PSF transform that can be applied to images (transform.py:25-51)."""

    #: host-buffer path: frames are streamed through the GPU in chunks of about this many input
    #: bytes (at least one frame), so upload, kernels and download of successive chunks overlap
    HOST_CHUNK_BYTES = 8 << 20

    def __init__(self, transfer_kernel: IndexedCube) -> None:
        self._transfer_kernel = transfer_kernel
        # the CUDA tensor of a device-resident kernel: the transform is differentiable in it when it requires grad
        self._kernel_tensor = transfer_kernel.tensor if isinstance(transfer_kernel, DeviceCube) else None
        self._native: dict[tuple[str, int], _NativeTransform] = {}
        self._coords_i32: np.ndarray | None = None
        # row-slab shard (distributed.shard_transform_rows): coordinates of the COMPLETE transform and which of them
        # this object holds kernels for; None for an ordinary transform
        self._shard_coordinates = None
        self._shard_keep: np.ndarray | None = None

    @classmethod
    def sharded(cls, transfer_kernel: IndexedCube, all_coordinates, keep) -> "ArrayPSFTransform":
        """A transform that holds the kernels of only some patches of a larger one (one rank of a patch-row slab
        split, SURVEY.md section 8e).  ``transfer_kernel`` carries the kept patches in the order they have in
        ``all_coordinates``; ``keep`` is the boolean mask over ``all_coordinates``.  Colour classes, and with them
        the summation order, are those of the complete transform, so slabs stitch bit-identically."""
        keep = np.asarray(keep, dtype=bool)
        full = np.asarray(all_coordinates)
        if full.ndim != 2 or full.shape[1] != 2 or keep.shape != (full.shape[0],):
            raise InvalidCoordinateError("all_coordinates must be (N, 2) and keep a mask of length N")
        kept = [tuple(c) for c in np.asarray(transfer_kernel.coordinates).reshape(-1, 2).tolist()]
        if kept != [tuple(c) for c in full[keep].tolist()]:
            raise InvalidCoordinateError("the shard's coordinates are not all_coordinates[keep], in order")
        obj = cls(transfer_kernel)
        obj._shard_coordinates, obj._shard_keep = full, keep
        return obj

    # ------------------------------------------------------------------ container plumbing
    @property
    def psf_shape(self) -> tuple[int, int]:
        return self._transfer_kernel.sample_shape

    @property
    def coordinates(self):
        return self._transfer_kernel.coordinates

    def __len__(self) -> int:
        return len(self._transfer_kernel)

    def __eq__(self, other) -> bool:
        if not isinstance(other, ArrayPSFTransform):
            raise TypeError("Can only compare ArrayPSFTransform to another ArrayPSFTransform.")
        return self._transfer_kernel == other._transfer_kernel

    __hash__ = None

    # ------------------------------------------------------------------ persistence (transform.py:220-282)
    def save(self, path, overwrite: bool = False) -> None:
        """Save the transfer kernel: ``.h5`` (coordinates, transfer_kernel) or ``.fits`` (transfer_real/_imag)."""
        from regularizepsf_b200 import persistence
        persistence.write_cubes(path, self.coordinates, {"transfer_kernel": self._transfer_kernel.values},
                                exclusive=True, overwrite=overwrite)

    @classmethod
    def load(cls, path) -> "ArrayPSFTransform":
        """Load a transform written by this class or by the reference package; the kernel is uploaded to
        HBM (and re-laid out for the column kernel) at the first ``apply``."""
        from regularizepsf_b200 import persistence
        coordinates, cubes = persistence.read_cubes(path, {"transfer_kernel": True})
        return cls(IndexedCube(coordinates, cubes["transfer_kernel"]))

    # ------------------------------------------------------------------ construct
    @classmethod
    def construct(cls, source, target, alpha, epsilon) -> "ArrayPSFTransform":
        """Build the regularised transfer kernel on the device (transform.py:53-83).

        ``K = conj(S) |S|^(alpha-1) / (|S|^(alpha+1) + (epsilon |T|)^(alpha+1)) * T`` elementwise over
        the two FFT cubes, in the cubes' precision, with no zero guard (0/0 bins are NaN, as in
        the reference).

        Differentiable on the device: when grad mode is on and the values of either PSF (an ``ArrayPSF`` built on a
        ``DeviceCube`` whose tensor requires grad), a given ``DeviceCube`` FFT cube, or ``alpha`` / ``epsilon`` require
        grad, the result's kernel tensor requires grad, so ``loss(apply(x)).backward()`` reaches them through
        ``rpsf_construct_kernel_backward`` and ``rpsf_psf_fft2_adjoint`` (DESIGN.md section 6).  ``alpha`` and ``epsilon``
        are numbers or 0-d real tensors.  A tensor is never read to the host: the kernels take both values from device
        memory (``rpsf_construct_kernel_dev``, bit-identical to passing them as numbers), so the call does not
        synchronise and can be captured in a CUDA graph.  PSF values that require grad need a native patch size (16, 32,
        ..., 512).  Otherwise the kernel is computed exactly as without autograd.
        """
        if np.any(np.array(source.coordinates) != np.array(target.coordinates)):
            raise InvalidCoordinateError("Source PSF coordinates do not match target PSF coordinates.")
        torch = _native.require_cuda()
        differentiable = torch.is_grad_enabled() and (
            any(_is_torch_tensor(x) and x.requires_grad for x in (alpha, epsilon))
            or any(_spectrum_source(psf) is not None for psf in (source, target)))
        if not differentiable:
            lib = _native.load()
            s_cube = source.fft_cube if hasattr(source, "fft_cube") else source._fft_cube
            t_cube = target.fft_cube if hasattr(target, "fft_cube") else target._fft_cube
            if s_cube.sample_shape != t_cube.sample_shape:
                raise IncorrectShapeError(f"source and target sample shapes differ: "
                                          f"{s_cube.sample_shape} != {t_cube.sample_shape}")
            s, t = _plain_spectrum(source, s_cube, torch), _plain_spectrum(target, t_cube, torch)
            if s.device != t.device:
                raise ValueError(f"source and target FFT cubes live on different devices: {s.device} and {t.device}")
            wide = torch.complex128 if torch.complex128 in (s.dtype, t.dtype) else torch.complex64
            with torch.cuda.device(s.device):                 # the launch stream must belong to the cubes' device
                s = s.to(wide) if s.dtype != wide else s
                t = t.to(wide) if t.dtype != wide else t
                kernel = torch.empty_like(s)
                code = _native.F32 if wide == torch.complex64 else _native.F64
                stream = _native.current_stream_ptr(torch)
                if _is_torch_tensor(alpha) or _is_torch_tensor(epsilon):
                    values = _device_scalars(torch, alpha, epsilon, s.device)
                    _native.check(lib.rpsf_construct_kernel_dev(s.data_ptr(), t.data_ptr(), kernel.data_ptr(), s.numel(),
                                                                code, values.data_ptr(), s.device.index, stream))
                else:
                    _native.check(lib.rpsf_construct_kernel(s.data_ptr(), t.data_ptr(), kernel.data_ptr(), s.numel(),
                                                            code, float(alpha), float(epsilon), s.device.index, stream))
            return cls._constructed(source.coordinates, kernel)
        from regularizepsf_b200._autograd import Construct
        for name, value in (("alpha", alpha), ("epsilon", epsilon)):
            if _is_torch_tensor(value) and (value.dim() != 0 or value.is_complex()):
                raise ValueError(f"{name} must be a number or a 0-d real tensor, got shape {tuple(value.shape)} "
                                 f"{value.dtype}")
        s, t = _spectrum(source, torch), _spectrum(target, torch)
        if tuple(s.shape[1:]) != tuple(t.shape[1:]):
            raise IncorrectShapeError(f"source and target sample shapes differ: {tuple(s.shape[1:])} != "
                                      f"{tuple(t.shape[1:])}")
        if s.device != t.device:
            raise ValueError(f"source and target FFT cubes live on different devices: {s.device} and {t.device}")
        wide = torch.complex128 if torch.complex128 in (s.dtype, t.dtype) else torch.complex64
        with torch.cuda.device(s.device):
            s = (s.to(wide) if s.dtype != wide else s).contiguous()
            t = (t.to(wide) if t.dtype != wide else t).contiguous()
            if _is_torch_tensor(alpha) or _is_torch_tensor(epsilon):
                kernel = Construct.apply(s, t, alpha, epsilon, None, None, _device_scalars(torch, alpha, epsilon, s.device))
            else:
                kernel = Construct.apply(s, t, alpha, epsilon, float(alpha), float(epsilon))
        return cls._constructed(source.coordinates, kernel)

    #: the kernel tensor was made by construct / reconstruct, not given by the caller (reconstruct may write into it)
    _kernel_owned = False

    @staticmethod
    def stack(transforms) -> "TransformStack":
        """A ``TransformStack`` of the kernels of ``transforms`` (copied into one (M, N, P, P) tensor), which must share
        their coordinates (InvalidCoordinateError) and patch size (IncorrectShapeError); a sharded transform raises
        NotImplementedError.  ``stack.apply(x)[m]`` is bit-identical to ``transforms[m].apply(x)``."""
        from regularizepsf_b200.stack import TransformStack
        return TransformStack.from_transforms(transforms)

    @classmethod
    def _constructed(cls, coordinates, kernel) -> "ArrayPSFTransform":
        obj = cls(DeviceCube(coordinates, kernel))
        obj._kernel_owned = True
        return obj

    def reconstruct(self, source, target, alpha, epsilon) -> None:
        """Replace the transfer kernel by ``construct(source, target, alpha, epsilon)``'s, in place.

        For a fitting loop that builds the kernel from its parameters at every step: the transform keeps its native
        transforms and plans (with their spectrum workspaces, 75.8 MB per 2048^2 frame at 256 px) and lays the new
        kernel out at its next call, where a fresh ``construct`` would create them again.  A transform whose calls a CUDA
        graph has captured lays it out in this call instead, so that replays launched after it read the new kernel; a
        graph that lays the kernel out itself reads the kernel tensor it was captured with, so the new kernel is copied
        into that tensor too (RuntimeError if that tensor is one the caller gave, not one ``construct`` made).  If the
        new kernel cannot be built, the transform is left as it was (inside a capture: with the previous kernel
        detached from its autograd graph, which a captured call lets go of before it builds the next).  The coordinates and the patch
        size must be the transform's (InvalidCoordinateError / IncorrectShapeError).  A kernel that requires grad on a
        sharded transform raises NotImplementedError.
        """
        if np.any(np.array(source.coordinates) != np.array(self.coordinates)):
            raise InvalidCoordinateError("the PSF coordinates do not match the transform's coordinates")
        torch = _native.require_cuda()
        capturing = _native.capturing(torch)
        if not capturing and any(not owned for nt in self._native.values() for _, owned in nt.graph_sources):
            raise RuntimeError("CUDA graphs of this transform lay out the kernel tensor it was given, and reconstruct "
                               "would leave them reading that tensor: update the tensor in place instead, or capture "
                               "the graphs again on a fresh transform")
        old = self._kernel_tensor
        if capturing and old is not None and old.grad_fn is not None:
            # let go of the previous kernel's autograd graph before building the next: otherwise the new graph reuses
            # the PSF values' gradient accumulators it holds, which belong to the stream of the eager call that made
            # them, and the captured backward would accumulate on a stream outside the capture
            old = old.detach()
            self._kernel_tensor, self._transfer_kernel = old, DeviceCube(self.coordinates, old)
            for nt in self._native.values():
                if nt.kernel_source is not None:
                    nt.kernel_source = old
        saved = (self._kernel_tensor, self._transfer_kernel, [(nt, nt.kernel_source) for nt in self._native.values()])
        try:
            new = type(self).construct(source, target, alpha, epsilon)
            if new.psf_shape != self.psf_shape:
                raise IncorrectShapeError(f"the PSFs' sample shape {new.psf_shape} is not the transform's "
                                          f"{self.psf_shape}")
            kernel = new._kernel_tensor
            if kernel.requires_grad and self._shard_keep is not None:
                raise NotImplementedError("the kernel gradient of a sharded transform is not implemented")
        except BaseException:
            self._kernel_tensor, self._transfer_kernel, sources = saved     # the transform is as it was
            for nt, source_tensor in sources:
                nt.kernel_source = source_tensor
            raise
        self._transfer_kernel = DeviceCube(self.coordinates, kernel)
        self._kernel_tensor = kernel
        self._kernel_owned = True
        for (_, device), nt in self._native.items():
            nt.kernel_source, nt.kernel_version = kernel, None     # laid out again at the next call
            if nt.captured and not capturing:
                # a replay runs no Python: lay the kernel out now, stream-ordered, so that replays launched after this
                # call read it (inside a capture, the next captured call lays it out).  Captured layouts read the
                # kernel tensors they were captured with: the new kernel is copied into them, after every call issued
                # so far (rpsf_transform_order) and before every call issued after this one (the layout records).
                with torch.cuda.device(device):
                    stream = _native.current_stream_ptr(torch)
                    if nt.graph_sources:
                        _native.check(nt.lib.rpsf_transform_order(nt.handle, stream))
                        for tensor, _ in nt.graph_sources:
                            tensor.copy_(kernel.detach())
                    nt.set_kernel(self._kernel_on(torch, device), stream)
                nt.kernel_version = kernel._version if kernel.requires_grad else None

    # ------------------------------------------------------------------ native state
    def _coords(self) -> np.ndarray:
        if self._coords_i32 is None:
            raw = np.asarray(self.coordinates if self._shard_coordinates is None else self._shard_coordinates)
            if raw.size == 0:
                raw = raw.reshape(0, 2)
            if raw.ndim != 2 or raw.shape[1] != 2:
                raise InvalidCoordinateError("coordinates must be (row, col) pairs")
            as_int = np.rint(raw).astype(np.int64)
            if not np.array_equal(as_int, raw):
                raise InvalidCoordinateError("patch corners must be integers to slice an image")
            if as_int.size and (as_int.min() < -2**30 or as_int.max() > 2**30):
                raise InvalidCoordinateError("patch corners out of range")
            self._coords_i32 = np.ascontiguousarray(as_int, dtype=np.int32)
        return self._coords_i32

    def _native_transform(self, dtype_name: str, device: int | None = None, capturing: bool = False,
                          reads_kernel: bool = True) -> _NativeTransform:
        """The native transform for (compute dtype, device); ``device`` defaults to the current CUDA device.
        Call with that device current (``_apply_device`` / ``_apply_host`` do).

        ``capturing``: the call is being captured in a CUDA graph.  The native transform must exist (RuntimeError
        otherwise: creating it and the first kernel layout allocate and synchronise).  A kernel tensor that requires
        grad, or one not laid out yet (``reconstruct``), is laid out again inside the graph at every captured call, so
        that each replay reads the tensor as it is then (``optimizer.step()`` between replays updates it in place, where
        no Python runs to see the new version); the transform keeps that tensor alive (``graph_sources``).
        ``reads_kernel=False`` (the kernel gradient, which reads no kernel) skips that layout."""
        torch = _native.require_cuda()
        if device is None:
            device = torch.cuda.current_device()
        key = (dtype_name, device)
        nt = self._native.get(key)
        if capturing:
            if nt is not None:
                nt.captured = True
            if nt is None:
                raise RuntimeError(f"this transform has no native state for {dtype_name} on cuda:{device} yet, and "
                                   "creating it (with the first kernel layout) cannot be captured in a CUDA graph: run "
                                   "the same call once before capturing")
            if (nt.kernel_source is not None and reads_kernel
                    and (nt.kernel_source.requires_grad or nt.kernel_version is None)):
                # the graph reads the kernel tensor by address at every replay: keep it alive with the transform
                source = self._transfer_kernel.tensor.detach()
                if not any(t.data_ptr() == source.data_ptr() for t, _ in nt.graph_sources):
                    nt.graph_sources.append((source, self._kernel_owned))
                with torch.cuda.device(device):
                    nt.set_kernel(self._kernel_on(torch, device), _native.current_stream_ptr(torch))
                nt.kernel_version = None       # the layout happens at replays: the next eager call lays it out again
            return nt
        if nt is None:
            p0, p1 = self.psf_shape
            if p0 != p1:
                # the reference's apodization window only broadcasts for square patches (transform.py:151-155)
                raise IncorrectShapeError(f"patches must be square, got {(p0, p1)}")
            with torch.cuda.device(device):
                # set_kernel is stream-ordered on this device's current stream, the stream `kt` was made on, so
                # the caching allocator cannot hand kt's block to anyone before the layout kernel has read it
                kt = self._kernel_on(torch, device)
                nt = _NativeTransform(self._coords(), p0, dtype_name, device, kt, _native.current_stream_ptr(torch),
                                      keep=self._shard_keep)
            source = self._kernel_tensor
            if source is not None and source.requires_grad:
                nt.kernel_source, nt.kernel_version = source, source._version
            self._native[key] = nt
        elif nt.kernel_source is not None and nt.kernel_source._version != nt.kernel_version:
            # the kernel tensor was updated in place since it was laid out (optimizer.step()): lay it out again
            version = nt.kernel_source._version
            with torch.cuda.device(device):
                nt.set_kernel(self._kernel_on(torch, device), _native.current_stream_ptr(torch))
            nt.kernel_version = version
        return nt

    def _kernel_on(self, torch, device: int):
        """The transfer kernel as a contiguous complex tensor on ``device`` (without autograd history)."""
        kernel = self._transfer_kernel
        if isinstance(kernel, DeviceCube):
            kt = kernel.tensor.detach()
            if kt.device.index != device:
                kt = kt.to(f"cuda:{device}")
        else:
            values = np.ascontiguousarray(kernel.values)
            if values.dtype not in (np.complex64, np.complex128):
                values = values.astype(np.complex128)
            kt = torch.from_numpy(values).to(f"cuda:{device}")
        return kt.contiguous()

    def _trainable_kernel(self):
        """The kernel tensor when the transform is differentiable in it (it requires grad), else None."""
        kt = self._kernel_tensor
        return kt if kt is not None and kt.requires_grad else None

    # ------------------------------------------------------------------ apply
    def apply(self, image, workers: int | None = None, pad_mode: str = "symmetric",
              saturation_threshold: float = math.inf, saturation_dilation: int = 1,
              neighborhood_width: int = 7, *, dtype=None, out_dtype=None, mask=None):
        """Apply the transform to an image (transform.py:85-177).

        ``image`` may be a numpy array (any real dtype; returns a fresh float64 numpy array exactly
        like the reference) or a CUDA ``torch.Tensor`` (stays on the device; returns a tensor in
        the compute dtype).  A leading batch axis ``(B, H, W)`` is accepted.  ``workers`` is
        accepted for signature parity and ignored.  ``dtype`` picks the arithmetic precision:
        "float32" or "float64" (validation mode); ``None`` means ``set_default_dtype``'s choice
        ("float32" unless changed), for every kind of input.  ``out_dtype`` (numpy input only) is the
        dtype of the returned array: float64 like the reference by default; ``np.float32`` halves the
        device-to-host copy, which is what bounds a host-to-host call (DESIGN.md section 5).

        Streams (INTEGRATION.md): a tensor is read and the result written in order on the current
        stream, and backward runs on the forward's stream.  The call sees the transfer kernel as it
        is when the call is issued (after ``reconstruct`` or an in-place update of the kernel tensor
        too), whatever streams earlier calls used: the library orders its own device state — the
        laid-out kernel, the plans' workspaces and scratch — across streams, the private streams of a
        numpy call included.  A tensor call does not synchronise with the host, and once warmed up it can be
        captured in a CUDA graph (INTEGRATION.md, "CUDA graphs"); a numpy call synchronises and cannot.

        ``mask``: a caller-given bad-pixel mask, boolean (or uint8 0/1) of shape (H, W), shared by every frame, or
        (B, H, W): a numpy array with numpy input, a CUDA tensor on the image's device with tensor input.  A pixel marked
        True is treated exactly like a saturated pixel after dilation: the image and the mask are padded alike (with
        "constant" the margin is unmasked), the padded mask is ORed into the dilated saturation mask (it alone with an
        infinite threshold), the masked pixels are filled in raster order with the nanmean of their neighbourhood, and
        they get their raw values back after the correction.  So a NaN or a defect under the mask stays at its own pixel
        instead of poisoning every patch that holds it.  With an infinite threshold the map is linear in the image and
        differentiable (``apply_adjoint(mask=)``, ``transfer_kernel_gradient(mask=)``).  A numpy image with a mask is
        uploaded and corrected on the device path and returned as float64 (or ``out_dtype``).  Pad modes without an
        index map and sharded transforms raise NotImplementedError (DESIGN.md section 6).
        """
        del workers
        if mask is not None:
            return self._apply_masked(image, pad_mode, saturation_threshold, saturation_dilation, neighborhood_width,
                                      mask, dtype, out_dtype)
        kt = self._kernel_tensor
        if (_is_torch_tensor(image) and (image.requires_grad or (kt is not None and kt.requires_grad))
                and _native.require_cuda().is_grad_enabled()):
            return self._apply_differentiable(image, pad_mode, saturation_threshold, dtype, adjoint=False)
        if (pad_mode == "symmetric" and saturation_threshold == math.inf and dtype is None and out_dtype is None
                and _is_torch_tensor(image)):
            # the common device-resident call: nothing to normalise (the host side of such a call costs as much as
            # the kernels of a 512^2 frame, scripts/host_cost.py)
            return self._apply_device(image, _default_dtype, 0)
        dtype_name = _normalize_dtype(dtype)
        # (threshold, dilation, neighbourhood width) of the saturation branch, transform.py:125-138;
        # +inf switches it off.  The mask, its dilation, the raster-ordered fill and the final
        # restore all run on the device, so no host pass over the frame decides anything.
        sat = (float(saturation_threshold), int(saturation_dilation), int(neighborhood_width))
        if math.isnan(sat[0]):
            sat = (math.inf,) + sat[1:]                    # `padded > nan` is all False in the reference
        out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
        if out_np not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise NotImplementedError(f"out_dtype must be float32 or float64, got {out_np}")
        if pad_mode not in _native.PAD_MODES:
            return self._apply_materialized_pad(image, dtype_name, pad_mode, out_np, sat)
        if _is_torch_tensor(image):
            return self._apply_device(image, dtype_name, _native.PAD_MODES[pad_mode], sat=sat)
        _native.refuse_in_capture(_native.require_cuda(), "apply() of a numpy array (a host-to-host call)")
        image = np.asarray(image)
        if image.ndim not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {image.shape}")
        return self._apply_host(image, dtype_name, _native.PAD_MODES[pad_mode], out_dtype=out_np.type, sat=sat)

    def apply_adjoint(self, image, pad_mode: str = "symmetric", *, dtype=None, mask=None, neighborhood_width: int = 7):
        """The transpose of ``apply`` without saturation, a linear map of the image: ``<apply(x), y> = <x,
        apply_adjoint(y)>``.  For forward modelling and iterative solvers (Landweber, CG on the normal equations), and
        the backward of ``apply`` under autograd.

        Takes what ``apply`` takes: a numpy array (any real dtype; returns float64) or a CUDA tensor (returns the
        compute dtype ``dtype``, "float32" by default), shaped (H, W) or (B, H, W).  ``pad_mode`` is one of the five
        modes with an index map ("symmetric", "reflect", "edge", "wrap", "constant").  A tensor that requires grad
        gives a differentiable result whose backward is ``apply``; so does a transform whose kernel tensor
        (``DeviceCube``) requires grad, whose kernel gradient is ``transfer_kernel_gradient`` with the roles swapped.

        ``mask`` (as in ``apply``) with ``neighborhood_width``: the transpose of ``apply(x, mask=mask,
        neighborhood_width=neighborhood_width)`` with an infinite threshold, in which the pixels that contribute to a
        fill are decided by the mask alone (as if the image were finite outside it).
        """
        if pad_mode not in _native.PAD_MODES:
            raise NotImplementedError(f"apply_adjoint supports the pad modes {sorted(_native.PAD_MODES)}, got {pad_mode!r}")
        if self._shard_keep is not None:
            raise NotImplementedError("apply_adjoint needs the kernels of every patch; a sharded transform holds a subset")
        sat = (math.inf, 1, int(neighborhood_width))
        if _is_torch_tensor(image):
            if ((image.requires_grad or self._trainable_kernel() is not None)
                    and _native.require_cuda().is_grad_enabled()):
                return self._apply_differentiable(image, pad_mode, math.inf, dtype, adjoint=True, mask=mask, width=sat[2])
            if mask is not None:
                return self._apply_device(image, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint=True,
                                          sat=sat, mask=mask)
            return self._apply_device(image, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint=True)
        torch = _native.require_cuda()
        _native.refuse_in_capture(torch, "apply_adjoint() of a numpy array (a host-to-host call)")
        host = np.asarray(image)
        if host.ndim not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {host.shape}")
        dev = torch.from_numpy(np.ascontiguousarray(host, dtype=np.float64)).to(f"cuda:{torch.cuda.current_device()}")
        if mask is not None:
            out = self._apply_device(dev, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint=True, sat=sat,
                                     mask=_upload_mask(torch, mask, host.shape, dev.device))
            return out.cpu().numpy().astype(np.float64, copy=False)
        out = self._apply_device(dev, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint=True)
        return out.cpu().numpy().astype(np.float64, copy=False)

    def _apply_masked(self, image, pad_mode: str, threshold, dilation, width, mask, dtype, out_dtype):
        """``apply(mask=...)``: the saturation branch with the caller's mask ORed into its own, on the device path."""
        if pad_mode not in _native.PAD_MODES:
            raise NotImplementedError(f"a mask needs one of the pad modes {sorted(_native.PAD_MODES)}; {pad_mode!r} is "
                                      "computed by np.pad on the host")
        if self._shard_keep is not None:
            raise NotImplementedError("a mask needs the whole frame: a sharded transform holds a subset of the patches")
        torch = _native.require_cuda()
        threshold = float(threshold)
        if math.isnan(threshold):
            threshold = math.inf                           # `padded > nan` is all False in the reference
        sat = (threshold, int(dilation), int(width))
        dtype_name = _normalize_dtype(dtype)
        pad_code = _native.PAD_MODES[pad_mode]
        if _is_torch_tensor(image):
            kt = self._kernel_tensor
            if (image.requires_grad or (kt is not None and kt.requires_grad)) and torch.is_grad_enabled():
                return self._apply_differentiable(image, pad_mode, threshold, dtype, adjoint=False, mask=mask, width=sat[2])
            return self._apply_device(image, dtype_name, pad_code, sat=sat, mask=mask)
        _native.refuse_in_capture(torch, "apply() of a numpy array (a host-to-host call)")
        out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
        if out_np not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise NotImplementedError(f"out_dtype must be float32 or float64, got {out_np}")
        host = np.asarray(image)
        if host.ndim not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {host.shape}")
        dev = torch.from_numpy(np.ascontiguousarray(host, dtype=np.float64)).to(f"cuda:{torch.cuda.current_device()}")
        out = self._apply_device(dev, dtype_name, pad_code, sat=sat, mask=_upload_mask(torch, mask, host.shape, dev.device))
        return out.cpu().numpy().astype(out_np.type, copy=False)

    def _apply_differentiable(self, image, pad_mode: str, saturation_threshold: float, dtype, adjoint: bool, mask=None,
                              width: int = 7):
        """``apply`` / ``apply_adjoint`` of a CUDA tensor that requires grad, or with a kernel tensor that does: a linear
        map whose backward is the other, and, for the kernel, ``transfer_kernel_gradient`` (``mask`` and the
        neighbourhood ``width`` carried along)."""
        if not (saturation_threshold == math.inf or math.isnan(saturation_threshold)):
            raise NotImplementedError("apply is not differentiable with a finite saturation_threshold: the mask and "
                                      "the restored pixels depend on the image")
        if pad_mode not in _native.PAD_MODES:
            raise NotImplementedError(f"apply is differentiable for the pad modes {sorted(_native.PAD_MODES)} only; "
                                      f"{pad_mode!r} is computed by np.pad on the host")
        if self._shard_keep is not None:
            raise NotImplementedError("a sharded transform is not differentiable: its transpose needs every patch's kernel")
        kernel = self._trainable_kernel()
        if kernel is None:
            from regularizepsf_b200._autograd import LinearMap
            return LinearMap.apply(image, self, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint, mask,
                                   width)
        self._check_kernel_gradient(pad_mode)
        for nt in self._native.values():
            if nt.kernel_source is None:       # requires_grad was switched on after the layout: track it from now on
                nt.kernel_source, nt.kernel_version = kernel, None
        from regularizepsf_b200._autograd import KernelMap
        return KernelMap.apply(image, kernel, self, _normalize_dtype(dtype), _native.PAD_MODES[pad_mode], adjoint, mask,
                               width)

    def _check_kernel_gradient(self, pad_mode: str) -> None:
        """NotImplementedError for what ``transfer_kernel_gradient`` has no device path for (DESIGN.md section 6)."""
        if pad_mode not in _native.PAD_MODES:
            raise NotImplementedError(f"the kernel gradient supports the pad modes {sorted(_native.PAD_MODES)}, got "
                                      f"{pad_mode!r}")
        if self._shard_keep is not None:
            raise NotImplementedError("the kernel gradient of a sharded transform is not implemented")
        if self.psf_shape[0] not in _NATIVE_SIZES:
            raise NotImplementedError(f"the kernel gradient is implemented for the patch sizes {_NATIVE_SIZES}; "
                                      f"{self.psf_shape[0]} runs embedded in a larger FFT")

    def transfer_kernel_gradient(self, image, grad_output, pad_mode: str = "symmetric", *, dtype=None, mask=None,
                                 neighborhood_width: int = 7):
        """The gradient of ``<apply(image), grad_output>`` with respect to the transfer kernel, without saturation: the
        vector-Jacobian product of ``apply`` in the kernel, for fitting a kernel to calibration pairs.  For patch p,
        ``conj(X_p) * G_p / P**2`` summed over the frames, with ``X_p`` and ``G_p`` the FFT2 of the apodized patch of
        the padded image and of the zero-extended ``grad_output``; patches that do not touch the frame get 0.  It uses
        PyTorch's convention for complex gradients (dL/dRe + i dL/dIm) and is Hermitian per patch.

        ``image`` and ``grad_output`` have the same shape, (H, W) or (B, H, W): numpy arrays (any real dtype; returns an
        (N, P, P) complex128 array, computed on the device) or CUDA tensors (returns complex64 for the compute dtype
        "float32", the default, complex128 for "float64").  ``pad_mode`` is one of the five modes with an index map.
        Embedded patch sizes (not a power of two) and sharded transforms raise NotImplementedError.

        ``mask`` (as in ``apply``) with ``neighborhood_width``: the gradient of ``<apply(image, mask=mask), grad_output>``
        with an infinite threshold; ``X_p`` is then taken from the padded image filled under the mask, and ``G_p`` from
        ``grad_output`` with the masked pixels set to 0.
        """
        self._check_kernel_gradient(pad_mode)
        dtype_name = _normalize_dtype(dtype)
        pad_code = _native.PAD_MODES[pad_mode]
        if _is_torch_tensor(image) or _is_torch_tensor(grad_output):
            if not (_is_torch_tensor(image) and _is_torch_tensor(grad_output)):
                raise TypeError("image and grad_output must both be numpy arrays or both CUDA tensors")
            return self._kernel_gradient_device(image.detach(), grad_output.detach(), dtype_name, pad_code, mask=mask,
                                                width=int(neighborhood_width))
        torch = _native.require_cuda()
        _native.refuse_in_capture(torch, "transfer_kernel_gradient() of numpy arrays (a host-to-host call)")
        x, g = np.asarray(image), np.asarray(grad_output)
        if x.shape != g.shape or x.ndim not in (2, 3):
            raise IncorrectShapeError(f"image and grad_output must share a shape (H, W) or (B, H, W), got {x.shape} "
                                      f"and {g.shape}")
        device = f"cuda:{torch.cuda.current_device()}"
        xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(device)
        gt = torch.from_numpy(np.ascontiguousarray(g, dtype=np.float64)).to(device)
        if mask is not None:
            mask = _upload_mask(torch, mask, x.shape, xt.device)
        out = self._kernel_gradient_device(xt, gt, dtype_name, pad_code, mask=mask, width=int(neighborhood_width))
        return out.cpu().numpy().astype(np.complex128, copy=False)

    def _kernel_gradient_device(self, image, grad, dtype_name: str, pad_code: int = 0, mask=None, width: int = 7):
        """``transfer_kernel_gradient`` of two CUDA tensors (no autograd history): the (N, P, P) complex tensor."""
        torch = _native.require_cuda()
        if not (image.is_cuda and grad.is_cuda) or image.device != grad.device:
            raise ValueError("image and grad_output must be CUDA tensors on one device")
        if tuple(image.shape) != tuple(grad.shape) or image.dim() not in (2, 3):
            raise IncorrectShapeError(f"image and grad_output must share a shape (H, W) or (B, H, W), got "
                                      f"{tuple(image.shape)} and {tuple(grad.shape)}")
        want = torch.float32 if dtype_name == "float32" else torch.float64
        if mask is not None:
            mask, mask_pitch, mask_stride = _mask_view(torch, mask, tuple(image.shape), image.device)
        with torch.cuda.device(image.device):
            capturing = _native.capturing(torch)
            nt = self._native_transform(dtype_name, image.device.index, capturing, reads_kernel=False)
            frames = [t.unsqueeze(0) if t.dim() == 2 else t for t in (image, grad)]
            frames = [t.to(want) if t.dtype != want else t for t in frames]
            x, g = [t.contiguous() if t.stride(-1) != 1 else t for t in frames]
            b, h, w = x.shape
            forward = nt.plan(h, w, pad_code, 0, h, b, capturing=capturing)
            adjoint = nt.plan(h, w, pad_code, 0, h, b, adjoint=True, capturing=capturing)
            nt.set_saturation(forward, self._NO_SAT if mask is None else (math.inf, 1, width))
            p = self.psf_shape[0]
            out = torch.empty((len(self), p, p), dtype=torch.complex64 if dtype_name == "float32" else torch.complex128,
                              device=x.device)
            if mask is not None:
                _native.check(nt.lib.rpsf_kernel_gradient_masked(
                    adjoint, forward, x.data_ptr(), x.stride(1), x.stride(0) if b > 1 else h * x.stride(1),
                    g.data_ptr(), g.stride(1), g.stride(0) if b > 1 else h * g.stride(1), b, out.data_ptr(),
                    mask.data_ptr(), mask_pitch, mask_stride, _native.current_stream_ptr(torch, x.device.index)))
                return out
            _native.check(nt.lib.rpsf_kernel_gradient(
                adjoint, forward, x.data_ptr(), x.stride(1), x.stride(0) if b > 1 else h * x.stride(1),
                g.data_ptr(), g.stride(1), g.stride(0) if b > 1 else h * g.stride(1), b, out.data_ptr(),
                _native.current_stream_ptr(torch, x.device.index)))
        return out

    _NO_SAT = (math.inf, 1, 7)
    _PAD_MATERIALIZED = 5                                  # RPSF_PAD_MATERIALIZED

    def _apply_materialized_pad(self, image, dtype_name: str, pad_mode, out_np, sat: tuple):
        """``pad_mode`` values without an on-device index map (np.pad's statistical modes, "linear_ramp", ...: the
        reference hands any mode string to np.pad, transform.py:119-123).  The margin is what np.pad makes of it, so it
        is computed by np.pad itself, on the host, in float64 like the reference (2P per side: "linear_ramp" depends on
        the width); the padded frames are uploaded and the kernels read the margin in place.  Slower than the five
        index-map modes (4.5 x the upload at 2048^2 / 256 px) — those stay the fast path."""
        torch = _native.require_cuda()
        _native.refuse_in_capture(torch, f"apply() with pad_mode={pad_mode!r} (np.pad on the host)")
        is_tensor = _is_torch_tensor(image)
        host = image.detach().cpu().numpy() if is_tensor else np.asarray(image)
        if host.ndim not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {host.shape}")
        squeeze = host.ndim == 2
        frames = host[np.newaxis] if squeeze else host
        pad = 2 * self.psf_shape[0]
        padded = np.stack([np.pad(f.astype(float), ((pad, pad), (pad, pad)), mode=pad_mode) for f in frames])
        want = torch.float32 if dtype_name == "float32" else torch.float64
        device = image.device if is_tensor else torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(device):
            dev64 = torch.from_numpy(padded).to(device)
            dev = dev64.to(want)
            b, h, w = frames.shape
            inner = dev[:, pad:pad + h, pad:pad + w]            # a view: the kernels address the margin through its pitch
            # the saturation mask is decided on the float64 padded frames, as the reference decides it
            out = self._apply_device(inner, dtype_name, self._PAD_MATERIALIZED, sat=sat,
                                     source=dev64[:, pad:pad + h, pad:pad + w])
        if is_tensor:
            return out[0] if squeeze else out
        result = out.cpu().numpy().astype(out_np.type, copy=False)
        return result[0] if squeeze else result

    def _apply_host(self, image: np.ndarray, dtype_name: str, pad_code: int, out_dtype=np.float64,
                    row_range: tuple[int, int] | None = None, sat: tuple = _NO_SAT) -> np.ndarray:
        nt = self._native_transform(dtype_name)
        squeeze = image.ndim == 2
        frames = image[np.newaxis] if squeeze else image
        code = _native.dtype_code(frames.dtype)
        if code is None:
            frames = frames.astype(np.float64)
            code = _native.F64
        frames = np.ascontiguousarray(frames)
        b, h, w = frames.shape
        r0, r1 = row_range if row_range is not None else (0, h)
        if r1 <= r0:                                       # an empty band (more ranks than half-patch rows)
            empty = np.empty((b, 0, w), out_dtype)
            return empty[0] if squeeze else empty
        chunk = max(1, min(b, self.HOST_CHUNK_BYTES // max(1, h * w * frames.dtype.itemsize)))
        plan = nt.plan(h, w, pad_code, r0, r1, chunk)
        nt.set_saturation(plan, sat)
        out = pinned_empty((b, r1 - r0, w), out_dtype)
        ocode = _native.dtype_code(out.dtype)
        _native.check(nt.lib.rpsf_apply_host(plan, frames.ctypes.data, code, out.ctypes.data, ocode, b))
        return out[0] if squeeze else out

    def _apply_device(self, image, dtype_name: str, pad_code: int, row_range: tuple[int, int] | None = None,
                      out=None, sat: tuple = _NO_SAT, mirrors: list[int] | None = None,
                      frame_rows: tuple[int, int] | None = None, adjoint: bool = False, source=None, mask=None):
        """``frame_rows = (first, height)``: ``image`` holds only rows [first, first + image.shape[-2]) of frames that
        are ``height`` rows tall (a row slab keeps just the rows its patches read: ``plan_info()["rows_read"]``).
        ``adjoint``: run the transpose (whole frames, no saturation).  ``source``: the frames of ``image`` before a
        conversion to the compute dtype, laid out alike, on which the saturation mask is decided (by default
        ``image`` itself, before this call converts it).  ``mask``: the caller's bad-pixel mask (``apply(mask=)``), a CUDA
        tensor; with ``adjoint`` the transpose of the masked map."""
        torch = _native.require_cuda()
        if not image.is_cuda:
            raise ValueError("apply() takes a numpy array or a CUDA tensor; move the tensor to the GPU first")
        if image.device.index == torch._C._cuda_getDevice():
            return self._apply_device_on(torch, image, dtype_name, pad_code, row_range, out, sat, mirrors, frame_rows,
                                         adjoint, source, mask)
        with torch.cuda.device(image.device):             # plans, streams and launches follow the image's device
            return self._apply_device_on(torch, image, dtype_name, pad_code, row_range, out, sat, mirrors, frame_rows,
                                         adjoint, source, mask)

    def _apply_device_on(self, torch, image, dtype_name, pad_code, row_range, out, sat, mirrors, frame_rows=None,
                         adjoint=False, source=None, mask=None):
        if mask is not None:
            if image.dim() not in (2, 3):
                raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {tuple(image.shape)}")
            mask, mask_pitch, mask_stride = _mask_view(torch, mask, tuple(image.shape), image.device)
        capturing = _native.capturing(torch)
        nt = self._native_transform(dtype_name, image.device.index, capturing)
        want = torch.float32 if dtype_name == "float32" else torch.float64
        squeeze = image.dim() == 2
        frames = image.unsqueeze(0) if squeeze else image
        if frames.dim() != 3:
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {tuple(image.shape)}")
        if source is None and frames.dtype != want and sat[0] != math.inf:
            source = frames                               # the saturation mask compares the unconverted pixels
        if frames.dtype != want:
            frames = frames.to(want)
        if frames.stride(-1) != 1:
            frames = frames.contiguous()
        b, held, w = frames.shape
        first, h = frame_rows if frame_rows is not None else (0, held)
        r0, r1 = row_range if row_range is not None else (0, h)
        if out is None:
            out = torch.empty((b, r1 - r0, w), dtype=want, device=frames.device)
        else:
            if out.device != frames.device:
                raise ValueError(f"`out` lives on {out.device}, the frames on {frames.device}")
            if squeeze and out.dim() == 2:
                out = out.unsqueeze(0)
            if tuple(out.shape) != (b, r1 - r0, w) or out.dtype != want or out.stride(-1) != 1:
                raise IncorrectShapeError(f"`out` must be a {want} tensor of shape {(b, r1 - r0, w)} with unit column "
                                          f"stride, got {out.dtype} {tuple(out.shape)}")
        if r1 <= r0:                                       # an empty band: nothing to compute, no native call
            return out[0] if squeeze else out
        plan = nt.plan(h, w, pad_code, r0, r1, b, adjoint=adjoint, capturing=capturing)
        nt.set_saturation(plan, sat)
        if mirrors:        # device pointers of peer buffers laid out like `out` (distributed.PeerFrames)
            import ctypes
            arr = (ctypes.c_void_p * len(mirrors))(*mirrors)
            _native.check(nt.lib.rpsf_plan_set_output_mirrors(plan, len(mirrors), arr))
        src_code = None
        if source is not None and sat[0] != math.inf:
            source = source.unsqueeze(0) if source.dim() == 2 else source
            if source.stride(-1) != 1:
                source = source.contiguous()
            src_code = _TORCH_CODES.get(str(source.dtype))
        try:
            args = (plan, frames.data_ptr(), frames.stride(1), frames.stride(0) if b > 1 else held * frames.stride(1),
                    first, held, out.data_ptr(), out.stride(1), out.stride(0) if b > 1 else (r1 - r0) * out.stride(1),
                    r0, b)
            stream = _native.current_stream_ptr(torch, frames.device.index)
            if mask is not None:
                src_args = (None, 0, 0, 0) if src_code is None else (
                    source.data_ptr(), src_code, source.stride(1), source.stride(0) if b > 1 else held * source.stride(1))
                rc = nt.lib.rpsf_apply_masked(*args, *src_args, mask.data_ptr(), mask_pitch, mask_stride, stream)
            elif src_code is None:
                rc = nt.lib.rpsf_apply(*args, stream)
            else:
                rc = nt.lib.rpsf_apply_source(*args, source.data_ptr(), src_code, source.stride(1),
                                              source.stride(0) if b > 1 else held * source.stride(1), stream)
            if rc:
                _native.check(rc)
        finally:
            if mirrors:
                _native.check(nt.lib.rpsf_plan_set_output_mirrors(plan, 0, None))
        return out[0] if squeeze else out


# element type codes of the torch dtypes the native code reads (str(dtype) -> code)
_TORCH_CODES = {"torch.float32": _native.F32, "torch.float64": _native.F64, "torch.uint8": _native.U8,
                "torch.int16": _native.I16, "torch.uint16": _native.U16, "torch.int32": _native.I32,
                "torch.int64": _native.I64, "torch.uint32": _native.U32}


def _mask_view(torch, mask, image_shape: tuple, device):
    """The caller's mask for an image of ``image_shape`` on CUDA ``device``: a uint8 tensor with unit column stride (a
    view of a bool or uint8 tensor when it has one), its row pitch, and its frame stride (0: one mask for every frame).
    IncorrectShapeError for a shape other than (H, W) or the image's (B, H, W), ValueError for a mask that is not a
    CUDA tensor on ``device``, TypeError for a dtype other than bool or uint8."""
    if not _is_torch_tensor(mask) or mask.device != device:
        where = mask.device if _is_torch_tensor(mask) else type(mask).__name__
        raise ValueError(f"with a CUDA tensor image, mask must be a CUDA tensor on {device}, got {where}")
    if mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError(f"mask must be bool or uint8, got {mask.dtype}")
    shape = tuple(mask.shape)
    if shape != tuple(image_shape[-2:]) and not (len(image_shape) == 3 and shape == tuple(image_shape)):
        raise IncorrectShapeError(f"mask must be (H, W) or the image's (B, H, W) for an image of shape "
                                  f"{tuple(image_shape)}, got {shape}")
    view = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
    if view.stride(-1) != 1:
        view = view.contiguous()
    return view, view.stride(-2), (view.stride(0) if view.dim() == 3 and view.shape[0] > 1 else 0)


def _upload_mask(torch, mask, image_shape: tuple, device):
    """A numpy mask for a numpy image of ``image_shape``, checked and copied to ``device`` (a tensor: ValueError)."""
    if _is_torch_tensor(mask):
        raise ValueError("with a numpy image, mask must be a numpy array, got a tensor")
    host = np.asarray(mask)
    if host.dtype not in (np.dtype(np.bool_), np.dtype(np.uint8)):
        raise TypeError(f"mask must be bool or uint8, got {host.dtype}")
    if host.shape != tuple(image_shape[-2:]) and not (len(image_shape) == 3 and host.shape == tuple(image_shape)):
        raise IncorrectShapeError(f"mask must be (H, W) or the image's (B, H, W) for an image of shape "
                                  f"{tuple(image_shape)}, got {host.shape}")
    return torch.from_numpy(np.ascontiguousarray(host).view(np.uint8)).to(device)


def _spectrum_source(psf):
    """The tensor through which ``psf``'s FFT cube depends on something that requires grad, or None: a given
    ``DeviceCube`` FFT cube that requires grad, else a ``DeviceCube`` of values that does."""
    given = getattr(psf, "_given_fft_cube", None)
    if given is not None:
        return given.tensor if isinstance(given, DeviceCube) and given.tensor.requires_grad else None
    values = getattr(psf, "_values_device_tensor", None)
    return values if values is not None and values.requires_grad else None


def _plain_spectrum(psf, cube, torch):
    """The FFT cube ``cube`` of ``psf`` as a CUDA tensor without autograd history (``ArrayPSF._device_spectrum`` for an
    ``ArrayPSF``, so that a host cube is not copied inside a CUDA graph capture)."""
    if hasattr(psf, "_device_spectrum"):
        return psf._device_spectrum(torch)
    return cube_tensor(cube, torch)


def _spectrum(psf, torch):
    """``psf``'s FFT cube as a CUDA tensor, differentiable in what ``_spectrum_source`` finds: a values tensor goes
    through ``_autograd.PsfFFT``, afresh at every call."""
    source = _spectrum_source(psf)
    if source is None:
        if hasattr(psf, "_device_spectrum"):
            return psf._device_spectrum(torch)
        return cube_tensor(psf.fft_cube if hasattr(psf, "fft_cube") else psf._fft_cube, torch)
    if psf._given_fft_cube is not None:
        return source
    if source.dim() != 3 or source.shape[1] not in _NATIVE_SIZES or source.shape[1] != source.shape[2]:
        raise NotImplementedError(f"PSF values that require grad need square patches of a native size {_NATIVE_SIZES}; "
                                  f"got {tuple(source.shape[1:])}, which runs embedded in a larger FFT")
    if source.is_complex() or not source.is_cuda:
        raise ValueError(f"PSF values that require grad must be a real CUDA tensor, got {source.dtype} on "
                         f"{source.device}")
    from regularizepsf_b200._autograd import PsfFFT
    return PsfFFT.apply(source if source.dtype in (torch.float32, torch.float64) else source.to(torch.float64))


def _device_scalars(torch, alpha, epsilon, device):
    """[alpha, epsilon] as a float64 tensor on ``device``, without a host synchronisation: a CUDA tensor is copied on the
    device, a number (or a CPU tensor, whose value the host has) is filled in."""
    values = torch.empty(2, dtype=torch.float64, device=device)
    for i, x in enumerate((alpha, epsilon)):
        if _is_torch_tensor(x) and x.is_cuda:
            values[i].copy_(x.detach().reshape(()))
        else:
            values[i].fill_(float(x.detach()) if _is_torch_tensor(x) else float(x))
    return values


def _is_torch_tensor(obj) -> bool:
    mod = type(obj).__module__
    return mod == "torch" or mod.startswith("torch.")
