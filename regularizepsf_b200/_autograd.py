"""Autograd of the device-resident ``apply`` / ``apply_adjoint`` (imported when a tensor that requires grad arrives).

Without saturation, ``apply`` is linear in the image, so the vector-Jacobian product of ``apply`` is ``apply_adjoint``
of the output gradient and that of ``apply_adjoint`` is ``apply``.  Nothing is saved for backward, and the backward
goes through this Function again, so double backward works too.
"""
from __future__ import annotations

import torch


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
