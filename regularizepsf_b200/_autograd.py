"""Autograd of the device-resident ``apply`` / ``apply_adjoint`` (imported when a tensor that requires grad arrives).

Without saturation, ``apply`` is linear in the image, so the vector-Jacobian product of ``apply`` is ``apply_adjoint``
of the output gradient and that of ``apply_adjoint`` is ``apply``.  ``LinearMap`` saves nothing for backward, and the
backward goes through it again, so double backward works too.  ``KernelMap`` is used when the transfer kernel requires
grad: ``apply`` is linear in the kernel as well, and its kernel gradient is ``transfer_kernel_gradient``.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable


class LinearMap(torch.autograd.Function):
    """``forward(image, transform, dtype_name, pad_code, adjoint)``: ``transform``'s map (its transpose when
    ``adjoint``) in the compute dtype ``dtype_name``; the gradient comes back in ``image.dtype``."""

    @staticmethod
    def forward(ctx, image, transform, dtype_name: str, pad_code: int, adjoint: bool):
        ctx.transform, ctx.dtype_name, ctx.pad_code, ctx.adjoint = transform, dtype_name, pad_code, adjoint
        ctx.image_dtype = image.dtype
        return transform._apply_device(image.detach(), dtype_name, pad_code, adjoint=adjoint)

    @staticmethod
    def backward(ctx, grad_output):
        # .sum().backward() hands over a stride-0 gradient: the kernels need real rows
        grad = LinearMap.apply(grad_output.contiguous(), ctx.transform, ctx.dtype_name, ctx.pad_code, not ctx.adjoint)
        return grad.to(ctx.image_dtype), None, None, None, None


class KernelMap(torch.autograd.Function):
    """``forward(image, kernel, transform, dtype_name, pad_code, adjoint)``: ``LinearMap`` that is differentiable in the
    transfer kernel too.  ``kernel`` is the tensor of the transform's ``DeviceCube``; ``transform`` lays it out again
    when it has been updated in place.  The image gradient is the same ``apply_adjoint`` / ``apply`` as ``LinearMap``'s;
    the kernel gradient is ``transfer_kernel_gradient(image, grad)`` (for the transpose: ``(grad, image)``) in the
    kernel's dtype and device.  The image is saved only when the kernel needs a gradient.  The kernel gradient has no
    derivative of its own on the device, so the backward is once-differentiable."""

    @staticmethod
    def forward(ctx, image, kernel, transform, dtype_name: str, pad_code: int, adjoint: bool):
        ctx.transform, ctx.dtype_name, ctx.pad_code, ctx.adjoint = transform, dtype_name, pad_code, adjoint
        ctx.image_dtype = image.dtype
        ctx.kernel_dtype, ctx.kernel_device = kernel.dtype, kernel.device
        if ctx.needs_input_grad[1]:
            ctx.save_for_backward(image)
        return transform._apply_device(image.detach(), dtype_name, pad_code, adjoint=adjoint)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        grad = grad_output.contiguous()
        transform = ctx.transform
        grad_image = grad_kernel = None
        if ctx.needs_input_grad[0]:
            grad_image = transform._apply_device(grad, ctx.dtype_name, ctx.pad_code,
                                                 adjoint=not ctx.adjoint).to(ctx.image_dtype)
        if ctx.needs_input_grad[1]:
            (image,) = ctx.saved_tensors
            x, g = (grad, image) if ctx.adjoint else (image, grad)
            grad_kernel = transform._kernel_gradient_device(x.detach(), g.detach(), ctx.dtype_name, ctx.pad_code)
            grad_kernel = grad_kernel.to(device=ctx.kernel_device, dtype=ctx.kernel_dtype)
        return grad_image, grad_kernel, None, None, None, None
