"""Autograd of the device-resident ``apply`` / ``apply_adjoint`` (imported when a tensor that requires grad arrives).

Without saturation, ``apply`` is linear in the image, so the vector-Jacobian product of ``apply`` is ``apply_adjoint``
of the output gradient and that of ``apply_adjoint`` is ``apply``.  ``LinearMap`` saves nothing for backward, and the
backward goes through it again, so double backward works too.  ``KernelMap`` is used when the transfer kernel requires
grad: ``apply`` is linear in the kernel as well, and its kernel gradient is ``transfer_kernel_gradient``.  ``Construct``
and ``PsfFFT`` carry that gradient on from the kernel to the PSF values, alpha and epsilon
(``ArrayPSFTransform.construct``).
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable


def _run(transform, image, dtype_name: str, pad_code: int, adjoint: bool, mask, width: int):
    """The map itself: ``apply`` / ``apply_adjoint`` of a tensor without autograd history (with a caller's ``mask``: the
    masked map with an infinite threshold and neighbourhood ``width``)."""
    if mask is None:
        return transform._apply_device(image, dtype_name, pad_code, adjoint=adjoint)
    return transform._apply_device(image, dtype_name, pad_code, adjoint=adjoint, sat=(float("inf"), 1, width), mask=mask)


class LinearMap(torch.autograd.Function):
    """``forward(image, transform, dtype_name, pad_code, adjoint, mask=None, width=7)``: ``transform``'s map (its
    transpose when ``adjoint``) in the compute dtype ``dtype_name``, under the caller's bad-pixel ``mask`` with
    neighbourhood width ``width`` when one is given; the gradient comes back in ``image.dtype``."""

    @staticmethod
    def forward(ctx, image, transform, dtype_name: str, pad_code: int, adjoint: bool, mask=None, width: int = 7):
        ctx.transform, ctx.dtype_name, ctx.pad_code, ctx.adjoint = transform, dtype_name, pad_code, adjoint
        ctx.mask, ctx.width = mask, width
        ctx.image_dtype = image.dtype
        return _run(transform, image.detach(), dtype_name, pad_code, adjoint, mask, width)

    @staticmethod
    def backward(ctx, grad_output):
        # .sum().backward() hands over a stride-0 gradient: the kernels need real rows
        grad = LinearMap.apply(grad_output.contiguous(), ctx.transform, ctx.dtype_name, ctx.pad_code, not ctx.adjoint,
                               ctx.mask, ctx.width)
        return grad.to(ctx.image_dtype), None, None, None, None, None, None


class KernelMap(torch.autograd.Function):
    """``forward(image, kernel, transform, dtype_name, pad_code, adjoint, mask=None, width=7)``: ``LinearMap`` that is
    differentiable in the transfer kernel too (with the same ``mask`` and ``width``).  ``kernel`` is the tensor of the transform's ``DeviceCube``; ``transform`` lays it out again
    when it has been updated in place.  The image gradient is the same ``apply_adjoint`` / ``apply`` as ``LinearMap``'s;
    the kernel gradient is ``transfer_kernel_gradient(image, grad)`` (for the transpose: ``(grad, image)``) in the
    kernel's dtype and device.  The image is saved only when the kernel needs a gradient.  The kernel gradient has no
    derivative of its own on the device, so the backward is once-differentiable."""

    @staticmethod
    def forward(ctx, image, kernel, transform, dtype_name: str, pad_code: int, adjoint: bool, mask=None, width: int = 7):
        ctx.transform, ctx.dtype_name, ctx.pad_code, ctx.adjoint = transform, dtype_name, pad_code, adjoint
        ctx.mask, ctx.width = mask, width
        ctx.image_dtype = image.dtype
        ctx.kernel_dtype, ctx.kernel_device = kernel.dtype, kernel.device
        if ctx.needs_input_grad[1]:
            ctx.save_for_backward(image)
        return _run(transform, image.detach(), dtype_name, pad_code, adjoint, mask, width)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        grad = grad_output.contiguous()
        transform = ctx.transform
        grad_image = grad_kernel = None
        if ctx.needs_input_grad[0]:
            grad_image = _run(transform, grad, ctx.dtype_name, ctx.pad_code, not ctx.adjoint, ctx.mask,
                              ctx.width).to(ctx.image_dtype)
        if ctx.needs_input_grad[1]:
            (image,) = ctx.saved_tensors
            x, g = (grad, image) if ctx.adjoint else (image, grad)
            grad_kernel = transform._kernel_gradient_device(x.detach(), g.detach(), ctx.dtype_name, ctx.pad_code,
                                                            mask=ctx.mask, width=ctx.width)
            grad_kernel = grad_kernel.to(device=ctx.kernel_device, dtype=ctx.kernel_dtype)
        return grad_image, grad_kernel, None, None, None, None, None, None


class PsfFFT(torch.autograd.Function):
    """``forward(values)``: the FFT cube of a real (N, P, P) CUDA tensor (``rpsf_psf_fft2``, psf.py:216-219), complex64
    for float32 values and complex128 for float64.  The backward is ``rpsf_psf_fft2_adjoint``, Re(fft2(conj(G))), in the
    values' dtype; native patch sizes only.  Used by ``ArrayPSFTransform.construct`` for values that require grad, once
    per call: a graph kept across calls could not be backpropagated twice."""

    @staticmethod
    def forward(ctx, values):
        from regularizepsf_b200.psf import _psf_fft2
        ctx.values_dtype = values.dtype
        return _psf_fft2(values.detach().contiguous(), torch)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        from regularizepsf_b200 import _native
        wide = torch.complex64 if ctx.values_dtype == torch.float32 else torch.complex128
        grad = grad_output.to(wide).contiguous()
        n, p, _ = grad.shape
        out = torch.empty(grad.shape, dtype=ctx.values_dtype, device=grad.device)
        with torch.cuda.device(grad.device):
            _native.check(_native.load().rpsf_psf_fft2_adjoint(
                grad.data_ptr(), out.data_ptr(), n, p, _native.F32 if wide == torch.complex64 else _native.F64,
                grad.device.index, _native.current_stream_ptr(torch)))
        return out


class Construct(torch.autograd.Function):
    """``forward(source_fft, target_fft, alpha, epsilon, alpha_value, epsilon_value, values)``: the transfer kernel
    (``rpsf_construct_kernel``, transform.py:78-82) of two complex cubes of one dtype.  ``alpha`` / ``epsilon`` are the
    caller's objects (floats or 0-d tensors, which get gradients).  Their values are either ``alpha_value`` /
    ``epsilon_value`` as floats (``values`` None), or ``values``, a float64 CUDA tensor [alpha, epsilon] on the cubes'
    device, read there by ``rpsf_construct_kernel_dev`` (no host synchronisation; used whenever alpha or epsilon is a
    tensor).  The backward is ``rpsf_construct_kernel_backward`` (``_dev``): the cube gradients in the cubes' dtype,
    those of alpha and epsilon accumulated in double and returned in each tensor's dtype and device.
    Once-differentiable."""

    @staticmethod
    def forward(ctx, source_fft, target_fft, alpha, epsilon, alpha_value, epsilon_value, values=None):
        from regularizepsf_b200 import _native
        ctx.values = (alpha_value, epsilon_value)
        ctx.on_device = values is not None
        ctx.scalars = tuple((x.dtype, x.device) if torch.is_tensor(x) else None for x in (alpha, epsilon))
        ctx.save_for_backward(source_fft, target_fft, values)
        kernel = torch.empty_like(source_fft)
        code = _native.F32 if source_fft.dtype == torch.complex64 else _native.F64
        lib = _native.load()
        with torch.cuda.device(source_fft.device):
            stream = _native.current_stream_ptr(torch)
            if values is not None:
                _native.check(lib.rpsf_construct_kernel_dev(
                    source_fft.data_ptr(), target_fft.data_ptr(), kernel.data_ptr(), source_fft.numel(), code,
                    values.data_ptr(), source_fft.device.index, stream))
            else:
                _native.check(lib.rpsf_construct_kernel(
                    source_fft.data_ptr(), target_fft.data_ptr(), kernel.data_ptr(), source_fft.numel(), code,
                    alpha_value, epsilon_value, source_fft.device.index, stream))
        return kernel

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        from regularizepsf_b200 import _native
        s, t, values = ctx.saved_tensors
        grad = grad_output.to(s.dtype).contiguous()
        need_s, need_t, need_a, need_e = ctx.needs_input_grad[:4]
        grad_s = torch.empty_like(s) if need_s else None
        grad_t = torch.empty_like(t) if need_t else None
        scalars = torch.empty(2, dtype=torch.float64, device=s.device) if need_a or need_e else None
        code = _native.F32 if s.dtype == torch.complex64 else _native.F64
        outputs = (grad_s.data_ptr() if need_s else None, grad_t.data_ptr() if need_t else None,
                   scalars.data_ptr() if scalars is not None else None)
        lib = _native.load()
        with torch.cuda.device(s.device):
            stream = _native.current_stream_ptr(torch)
            if ctx.on_device:
                _native.check(lib.rpsf_construct_kernel_backward_dev(
                    s.data_ptr(), t.data_ptr(), grad.data_ptr(), s.numel(), code, values.data_ptr(), *outputs,
                    s.device.index, stream))
            else:
                _native.check(lib.rpsf_construct_kernel_backward(
                    s.data_ptr(), t.data_ptr(), grad.data_ptr(), s.numel(), code, ctx.values[0], ctx.values[1], *outputs,
                    s.device.index, stream))
        grad_a = grad_e = None
        if need_a:
            grad_a = scalars[0].to(dtype=ctx.scalars[0][0], device=ctx.scalars[0][1])
        if need_e:
            grad_e = scalars[1].to(dtype=ctx.scalars[1][0], device=ctx.scalars[1][1])
        return grad_s, grad_t, grad_a, grad_e, None, None, None
