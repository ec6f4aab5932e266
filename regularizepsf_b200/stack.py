"""``TransformStack`` — M transfer kernels on one set of patch corners, applied to the same frames in one call.

Picking ``alpha`` and ``epsilon`` means applying many kernels built from the same PSFs to the same frames.  A stack
does the work that does not depend on the kernel once per frame instead of once per kernel: the saturation / mask fill
and the row pass (gather, window, row FFT).  The column pass then runs once per kernel from the shared row spectra,
and one overlap-add writes every output (``rpsf_apply_stack``, DESIGN.md section 6, "Transform stacks").  ``construct`` builds all M
kernels in one pass over the two FFT cubes (``rpsf_construct_kernels``).

``stack.apply(x)[m]`` is bit-identical to ``stack[m].apply(x)`` with the same arguments.
"""
from __future__ import annotations

import ctypes
import math
import weakref

import numpy as np

from regularizepsf_b200 import _native
from regularizepsf_b200.device import DeviceCube
from regularizepsf_b200.exceptions import IncorrectShapeError, InvalidCoordinateError
from regularizepsf_b200.transform import (
    _DTYPES, ArrayPSFTransform, _device_scalars, _is_torch_tensor, _mask_view, _normalize_dtype, _plain_spectrum,
    _spectrum_source, _TORCH_CODES, _upload_mask)


class _NativeStack:
    """Owns one ``rpsf_stack`` (per compute dtype and device) and its plans."""

    #: plans kept per native stack; a plan holds the spectra of M x max_batch frames (75.8 MB each at 2048^2 / 256 px,
    #: float32), so few are kept
    MAX_PLANS = 2

    def __init__(self, coords: np.ndarray, patch: int, dtype_name: str, device: int, kernels, stream: int, version: int):
        self.lib = _native.load()
        self.m = int(kernels.shape[0])
        handle = ctypes.c_void_p()
        _native.check(self.lib.rpsf_stack_create(ctypes.byref(handle), coords.ctypes.data, coords.shape[0], patch,
                                                 _DTYPES[dtype_name], device, self.m))
        self.handle = handle.value
        self._plans: dict[tuple, int] = {}
        self._pinned: frozenset = frozenset()
        self._saturation: dict[int, tuple] = {}
        self._plans_batch: dict[int, int] = {}           # plan handle -> its max_batch
        self._finalizer = weakref.finalize(self, _NativeStack._cleanup, self.lib, self.handle, self._plans)
        self.kernel_version = None
        self.set_kernels(kernels, stream, version)

    def set_kernels(self, kernels, stream: int, version: int) -> None:
        """Lay out every kernel of the contiguous (M, N, P, P) tensor ``kernels``, stream-ordered on ``stream``;
        ``version``: that of the stack's kernel tensor it was taken from."""
        kcode = _native.F32 if str(kernels.dtype) == "torch.complex64" else _native.F64
        for m in range(self.m):
            _native.check(self.lib.rpsf_stack_set_kernel(self.handle, m, kernels[m].data_ptr(), kcode, stream))
        self.kernel_version = version

    @staticmethod
    def _cleanup(lib, handle, plans):
        for plan in plans.values():
            try:
                lib.rpsf_plan_destroy(plan)
            except Exception:  # pragma: no cover - interpreter shutdown
                pass
        plans.clear()
        try:
            lib.rpsf_stack_destroy(handle)
        except Exception:  # pragma: no cover - interpreter shutdown
            pass

    def plan(self, height: int, width: int, pad_mode: int, max_batch: int, capturing: bool = False) -> int:
        """A plan for this geometry taking ``max_batch`` frames per call: a cached one of capacity in [max_batch,
        2 * max_batch], else a new one (RuntimeError inside a CUDA graph capture).  Captured plans are never evicted."""
        geometry = (height, width, pad_mode)
        best = None
        for key in self._plans:
            if key[:-1] == geometry and max_batch <= key[-1] <= 2 * max_batch and (best is None or key[-1] < best[-1]):
                best = key
        if best is not None:
            self._plans[best] = self._plans.pop(best)          # most recently used last
            if capturing:
                self._pinned = self._pinned | {best}
            return self._plans[best]
        if capturing:
            raise RuntimeError(f"no stack plan for frames of {height} x {width} (pad mode {pad_mode}, {max_batch} frames) "
                               "exists, and creating one cannot be captured in a CUDA graph: run the same call once "
                               "before capturing")
        out = ctypes.c_void_p()
        _native.check(self.lib.rpsf_plan_create_stack(ctypes.byref(out), self.handle, height, width, pad_mode, max_batch))
        self._plans[geometry + (max_batch,)] = out.value
        self._plans_batch[out.value] = max_batch
        while len(self._plans) - len(self._pinned) > self.MAX_PLANS:
            oldest = next(key for key in self._plans if key not in self._pinned)
            handle = self._plans.pop(oldest)
            self._saturation.pop(handle, None)
            self._plans_batch.pop(handle, None)
            self.lib.rpsf_plan_destroy(handle)
        return out.value

    def set_saturation(self, plan: int, sat: tuple) -> None:
        if self._saturation.get(plan) != sat:
            _native.check(self.lib.rpsf_plan_set_saturation(plan, *sat))
            self._saturation[plan] = sat


class TransformStack:
    """M transfer kernels sharing one set of patch corners and one patch size, held as one (M, N, P, P) complex CUDA
    tensor.  ``len(stack)`` is M; ``stack[m]`` is an ``ArrayPSFTransform`` whose ``DeviceCube`` is a view of slice m
    (no copy), with native state of its own only once it is applied itself.

    Build one with ``TransformStack.construct(source, target, alphas, epsilons)`` or
    ``ArrayPSFTransform.stack(transforms)``.
    """

    def __init__(self, coordinates, kernels) -> None:
        if kernels.dim() != 4 or not kernels.is_complex():
            raise IncorrectShapeError(f"the kernels must be an (M, N, P, P) complex tensor, got {kernels.dtype} "
                                      f"{tuple(kernels.shape)}")
        if kernels.shape[0] < 1:
            raise ValueError("a transform stack needs at least one kernel")
        if len(coordinates) != kernels.shape[1]:
            raise IncorrectShapeError(f"{len(coordinates)} coordinates defined but {kernels.shape[1]} patches found.")
        self._coordinates = coordinates
        self._kernels = kernels.contiguous()
        self._template = ArrayPSFTransform(DeviceCube(coordinates, self._kernels[0]))
        self._native: dict[tuple[str, int], _NativeStack] = {}
        self._members: dict[int, ArrayPSFTransform] = {}
        #: column pass of the stack's plans (rpsf_plan_set_stack_mode): 0 = k2_stack where it exists, 1 = the per-kernel
        #: column pass.  Both give the same bits; a test and benchmark hook.
        self._stack_mode = 0

    # ------------------------------------------------------------------ container
    @property
    def kernels(self):
        """The (M, N, P, P) complex tensor of the transfer kernels."""
        return self._kernels

    @property
    def coordinates(self):
        return self._coordinates

    @property
    def psf_shape(self) -> tuple[int, int]:
        return int(self._kernels.shape[2]), int(self._kernels.shape[3])

    def __len__(self) -> int:
        return int(self._kernels.shape[0])

    def __getitem__(self, m: int) -> ArrayPSFTransform:
        """Member m, made at its first access and kept, so that its native state and plans (made at its first apply)
        serve every later ``stack[m]``."""
        m = range(len(self))[m]
        member = self._members.get(m)
        if member is None:
            member = self._members[m] = ArrayPSFTransform(DeviceCube(self._coordinates, self._kernels[m]))
        return member

    # ------------------------------------------------------------------ construction
    @classmethod
    def construct(cls, source, target, alphas, epsilons) -> "TransformStack":
        """Kernel m is ``ArrayPSFTransform.construct(source, target, alphas[m], epsilons[m])``'s, bit for bit (NaN
        bins included), built for all m in one pass over the two FFT cubes.  ``alphas`` and ``epsilons`` are
        equal-length sequences of numbers or 0-d real tensors (a grid: ``zip(*itertools.product(...))``); tensors are
        read on the device, so the call does not synchronise.  Not differentiable: PSF values or an ``alpha`` /
        ``epsilon`` that requires grad while grad mode is on raise NotImplementedError."""
        if np.any(np.array(source.coordinates) != np.array(target.coordinates)):
            raise InvalidCoordinateError("Source PSF coordinates do not match target PSF coordinates.")
        alphas, epsilons = list(alphas), list(epsilons)
        if len(alphas) != len(epsilons):
            raise ValueError(f"alphas and epsilons must have one length, got {len(alphas)} and {len(epsilons)}")
        if not alphas:
            raise ValueError("a transform stack needs at least one (alpha, epsilon) pair")
        torch = _native.require_cuda()
        for name, values in (("alpha", alphas), ("epsilon", epsilons)):
            for v in values:
                if _is_torch_tensor(v) and (v.dim() != 0 or v.is_complex()):
                    raise ValueError(f"{name} must be a number or a 0-d real tensor, got shape {tuple(v.shape)} {v.dtype}")
        if torch.is_grad_enabled() and (
                any(_is_torch_tensor(v) and v.requires_grad for v in alphas + epsilons)
                or any(_spectrum_source(psf) is not None for psf in (source, target))):
            raise NotImplementedError("TransformStack.construct is not differentiable; use ArrayPSFTransform.construct "
                                      "per pair, or build the stack under torch.no_grad()")
        lib = _native.load()
        s_cube = source.fft_cube if hasattr(source, "fft_cube") else source._fft_cube
        t_cube = target.fft_cube if hasattr(target, "fft_cube") else target._fft_cube
        if s_cube.sample_shape != t_cube.sample_shape:
            raise IncorrectShapeError(f"source and target sample shapes differ: {s_cube.sample_shape} != "
                                      f"{t_cube.sample_shape}")
        s, t = _plain_spectrum(source, s_cube, torch), _plain_spectrum(target, t_cube, torch)
        if s.device != t.device:
            raise ValueError(f"source and target FFT cubes live on different devices: {s.device} and {t.device}")
        wide = torch.complex128 if torch.complex128 in (s.dtype, t.dtype) else torch.complex64
        m = len(alphas)
        with torch.cuda.device(s.device):
            s = (s.to(wide) if s.dtype != wide else s).contiguous()
            t = (t.to(wide) if t.dtype != wide else t).contiguous()
            kernels = torch.empty((m,) + tuple(s.shape), dtype=wide, device=s.device)
            code = _native.F32 if wide == torch.complex64 else _native.F64
            stream = _native.current_stream_ptr(torch)
            if any(_is_torch_tensor(v) for v in alphas + epsilons):
                pairs = torch.stack([_device_scalars(torch, a, e, s.device) for a, e in zip(alphas, epsilons)])
                _native.check(lib.rpsf_construct_kernels_dev(s.data_ptr(), t.data_ptr(), kernels.data_ptr(), s.numel(),
                                                             code, pairs.data_ptr(), m, s.device.index, stream))
            else:
                pairs = np.ascontiguousarray([[float(a), float(e)] for a, e in zip(alphas, epsilons)], dtype=np.float64)
                _native.check(lib.rpsf_construct_kernels(s.data_ptr(), t.data_ptr(), kernels.data_ptr(), s.numel(),
                                                         code, pairs.ctypes.data, m, s.device.index, stream))
        return cls(source.coordinates, kernels)

    @classmethod
    def from_transforms(cls, transforms) -> "TransformStack":
        """``ArrayPSFTransform.stack``: the kernels of ``transforms`` copied into one (M, N, P, P) tensor (complex128
        if any of them is, else complex64) on the device of the first device-resident kernel, else the current one."""
        transforms = list(transforms)
        if not transforms:
            raise ValueError("a transform stack needs at least one transform")
        for tr in transforms:
            if not isinstance(tr, ArrayPSFTransform):
                raise TypeError(f"can only stack ArrayPSFTransform objects, got {type(tr).__name__}")
            if tr._shard_keep is not None:
                raise NotImplementedError("a sharded transform cannot be stacked: it holds a subset of the patches")
        first = transforms[0]
        coords = np.asarray(first.coordinates)
        for tr in transforms[1:]:
            other = np.asarray(tr.coordinates)
            if other.shape != coords.shape or np.any(other != coords):
                raise InvalidCoordinateError("the transforms of a stack must share their patch coordinates")
            if tr.psf_shape != first.psf_shape:
                raise IncorrectShapeError(f"the transforms of a stack must share a patch size, got {first.psf_shape} "
                                          f"and {tr.psf_shape}")
        torch = _native.require_cuda()
        device = next((tr._kernel_tensor.device.index for tr in transforms if tr._kernel_tensor is not None),
                      torch.cuda.current_device())
        with torch.cuda.device(device):
            parts = [tr._kernel_on(torch, device) for tr in transforms]
            wide = torch.complex128 if any(p.dtype == torch.complex128 for p in parts) else torch.complex64
            kernels = torch.stack([p.to(wide) for p in parts])
        return cls(first.coordinates, kernels)

    # ------------------------------------------------------------------ apply
    def _native_stack(self, torch, dtype_name: str, device: int, capturing: bool) -> _NativeStack:
        key = (dtype_name, device)
        ns = self._native.get(key)
        kernels = self._kernels
        if capturing:
            if ns is None:
                raise RuntimeError(f"this transform stack has no native state for {dtype_name} on cuda:{device} yet, "
                                   "and creating it cannot be captured in a CUDA graph: run the same call once before "
                                   "capturing")
            return ns
        if kernels.device.index != device:
            kernels = kernels.to(f"cuda:{device}")
        if ns is None:
            p0, p1 = self.psf_shape
            if p0 != p1:
                raise IncorrectShapeError(f"patches must be square, got {(p0, p1)}")
            ns = _NativeStack(self._template._coords(), p0, dtype_name, device, kernels.detach(),
                              _native.current_stream_ptr(torch), self._kernels._version)
            self._native[key] = ns
        elif self._kernels._version != ns.kernel_version:
            # the kernel tensor was written in place since its layout: lay it out again
            ns.set_kernels(kernels.detach(), _native.current_stream_ptr(torch), self._kernels._version)
        return ns

    def apply(self, image, workers: int | None = None, pad_mode: str = "symmetric",
              saturation_threshold: float = math.inf, saturation_dilation: int = 1, neighborhood_width: int = 7, *,
              dtype=None, out_dtype=None, mask=None):
        """Every kernel of the stack applied to ``image``: (M, H, W) for an (H, W) image, (M, B, H, W) for (B, H, W).
        Takes what ``ArrayPSFTransform.apply`` takes, and ``result[m]`` is bit-identical to ``self[m].apply`` with the
        same arguments.  A numpy image returns float64 numpy (or ``out_dtype``); a CUDA tensor returns a tensor of the
        compute dtype, with ``apply``'s stream rules, and once warmed up a tensor call allocates nothing in the library
        and can be captured in a CUDA graph.  The kernel tensor is read as it is at the last eager call.

        Not implemented (NotImplementedError): autograd (an image or kernel tensor that requires grad while grad mode is
        on), the pad modes without an index map (np.pad's statistical modes and the like)."""
        del workers
        torch = _native.require_cuda()
        if pad_mode not in _native.PAD_MODES:
            raise NotImplementedError(f"a transform stack supports the pad modes {sorted(_native.PAD_MODES)}; "
                                      f"{pad_mode!r} is computed by np.pad on the host")
        if torch.is_grad_enabled() and (self._kernels.requires_grad or (_is_torch_tensor(image) and image.requires_grad)):
            raise NotImplementedError("TransformStack.apply is not differentiable; apply the members one by one, or "
                                      "call it under torch.no_grad()")
        threshold = float(saturation_threshold)
        if math.isnan(threshold):
            threshold = math.inf                           # `padded > nan` is all False in the reference
        sat = (threshold, int(saturation_dilation), int(neighborhood_width))
        dtype_name = _normalize_dtype(dtype)
        pad_code = _native.PAD_MODES[pad_mode]
        if _is_torch_tensor(image):
            if not image.is_cuda:
                raise ValueError("apply() takes a numpy array or a CUDA tensor; move the tensor to the GPU first")
            with torch.cuda.device(image.device):
                return self._apply_device(torch, image, dtype_name, pad_code, sat, mask)
        _native.refuse_in_capture(torch, "TransformStack.apply() of a numpy array (a host-to-host call)")
        out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
        if out_np not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise NotImplementedError(f"out_dtype must be float32 or float64, got {out_np}")
        host = np.asarray(image)
        if host.ndim not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {host.shape}")
        device = torch.cuda.current_device()
        dev = torch.from_numpy(np.ascontiguousarray(host, dtype=np.float64)).to(f"cuda:{device}")
        if mask is not None:
            mask = _upload_mask(torch, mask, host.shape, dev.device)
        out = self._apply_device(torch, dev, dtype_name, pad_code, sat, mask)
        return out.cpu().numpy().astype(out_np.type, copy=False)

    def apply_adjoint(self, *args, **kwargs):
        """Not implemented for a stack: apply the members' ``apply_adjoint`` one by one."""
        raise NotImplementedError("apply_adjoint of a transform stack is not implemented; use stack[m].apply_adjoint")

    def _apply_device(self, torch, image, dtype_name: str, pad_code: int, sat: tuple, mask):
        if image.dim() not in (2, 3):
            raise IncorrectShapeError(f"image must be (H, W) or (B, H, W), got shape {tuple(image.shape)}")
        if mask is not None:
            mask, mask_pitch, mask_stride = _mask_view(torch, mask, tuple(image.shape), image.device)
        capturing = _native.capturing(torch)
        ns = self._native_stack(torch, dtype_name, image.device.index, capturing)
        want = torch.float32 if dtype_name == "float32" else torch.float64
        squeeze = image.dim() == 2
        frames = image.unsqueeze(0) if squeeze else image
        source = frames if frames.dtype != want and sat[0] != math.inf else None
        if frames.dtype != want:
            frames = frames.to(want)
        if frames.stride(-1) != 1:
            frames = frames.contiguous()
        b, h, w = frames.shape
        plan = ns.plan(h, w, pad_code, b, capturing=capturing)
        ns.set_saturation(plan, sat)
        _native.check(ns.lib.rpsf_plan_set_stack_mode(plan, self._stack_mode))
        out = torch.empty((ns.m, b, h, w), dtype=want, device=frames.device)
        src_args = (None, 0, 0, 0)
        if source is not None and _TORCH_CODES.get(str(source.dtype)) is not None:
            if source.stride(-1) != 1:
                source = source.contiguous()
            src_args = (source.data_ptr(), _TORCH_CODES.get(str(source.dtype)), source.stride(1),
                        source.stride(0) if b > 1 else h * source.stride(1))
        mask_args = (None, 0, 0) if mask is None else (mask.data_ptr(), mask_pitch, mask_stride)
        _native.check(ns.lib.rpsf_apply_stack(
            plan, frames.data_ptr(), frames.stride(1), frames.stride(0) if b > 1 else h * frames.stride(1),
            out.data_ptr(), w, h * w, ns.m, b, *src_args, *mask_args,
            _native.current_stream_ptr(torch, frames.device.index)))
        return out[:, 0] if squeeze else out
