"""ctypes binding of librpsf_b200.so (C ABI declared in include/rpsf_b200.h).

The library is built in-tree by ``python -m regularizepsf_b200.csrc.build`` (or
``__graft_entry__.build()``).  There is no CPU fallback: if the library or a CUDA device is
missing every compute entry point raises ``NativeLibraryError``.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np

from regularizepsf_b200 import exceptions
from regularizepsf_b200.exceptions import NativeLibraryError

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "librpsf_b200.so")

# element type codes (include/rpsf_b200.h)
F32, F64, U8, I16, U16, I32, I64, U32 = range(8)
_NP_CODES = {
    np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.uint8): U8, np.dtype(np.int16): I16,
    np.dtype(np.uint16): U16, np.dtype(np.int32): I32, np.dtype(np.int64): I64, np.dtype(np.uint32): U32,
}
PAD_MODES = {"symmetric": 0, "reflect": 1, "edge": 2, "wrap": 3, "constant": 4}

E_INVALID_ARGUMENT, E_INVALID_COORDINATE, E_INCORRECT_SHAPE, E_UNSUPPORTED, E_CUDA, E_NO_KERNEL = -1, -2, -3, -4, -5, -6

# every symbol include/rpsf_b200.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
SIGNATURES = {
    "rpsf_abi_version": (_i, []),
    "rpsf_last_error": (ctypes.c_char_p, []),
    "rpsf_patch_size_supported": (_i, [_i]),
    "rpsf_transform_create": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i]),
    "rpsf_transform_create_subset": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _vp]),
    "rpsf_transform_destroy": (_i, [_vp]),
    "rpsf_transform_set_kernel": (_i, [_vp, _vp, _i, _vp]),
    "rpsf_transform_num_colours": (_i, [_vp]),
    "rpsf_transform_order": (_i, [_vp, _vp]),
    "rpsf_construct_kernel": (_i, [_vp, _vp, _vp, _i64, _i, _d, _d, _i, _vp]),
    "rpsf_construct_kernel_backward": (_i, [_vp, _vp, _vp, _i64, _i, _d, _d, _vp, _vp, _vp, _i, _vp]),
    "rpsf_construct_kernel_dev": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _i, _vp]),
    "rpsf_construct_kernel_backward_dev": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _vp, _vp, _vp, _i, _vp]),
    "rpsf_psf_fft2": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp]),
    "rpsf_psf_fft2_adjoint": (_i, [_vp, _vp, _i64, _i, _i, _i, _vp]),
    "rpsf_average_patches": (_i, [_vp, _i64, _i, _vp, _vp, _i64, _i, _d, _vp, _i, _vp]),
    "rpsf_plane_background": (_i, [_vp, _i64, _i, _vp, _i, _vp]),
    "rpsf_star_cutouts": (_i, [_vp, _i, _i, _i, _vp, _i64, _i, _d, _d, _d, _vp, _vp, _i, _vp]),
    "rpsf_isolate_cores": (_i, [_vp, _i64, _i, _i, _vp]),
    "rpsf_plan_create": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, _i]),
    "rpsf_plan_create_adjoint": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i]),
    "rpsf_kernel_gradient": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _i, _vp, _vp]),
    "rpsf_kernel_gradient_masked": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _i64, _i64, _i, _vp, _vp, _i64, _i64, _vp]),
    "rpsf_plan_destroy": (_i, [_vp]),
    "rpsf_plan_info": (_i, [_vp, ctypes.POINTER(_i64)]),
    "rpsf_plan_set_overlap_mode": (_i, [_vp, _i]),
    "rpsf_plan_set_gather_mode": (_i, [_vp, _i]),
    "rpsf_plan_column_info": (_i, [_vp, ctypes.POINTER(_i64)]),
    "rpsf_plan_set_saturation": (_i, [_vp, _d, _i, _i]),
    "rpsf_plan_set_output_mirrors": (_i, [_vp, _i, ctypes.POINTER(_vp)]),
    "rpsf_ipc_alloc": (_i, [ctypes.POINTER(_vp), _i64, _i, ctypes.c_char_p]),
    "rpsf_ipc_open": (_i, [ctypes.POINTER(_vp), ctypes.c_char_p, _i]),
    "rpsf_ipc_close": (_i, [_vp, _i]),
    "rpsf_upload": (_i, [ctypes.POINTER(_vp), _vp, _i64, _i]),
    "rpsf_device_free": (_i, [_vp, _i]),
    "rpsf_apply": (_i, [_vp, _vp, _i64, _i64, _i, _i, _vp, _i64, _i64, _i, _i, _vp]),
    "rpsf_apply_source": (_i, [_vp, _vp, _i64, _i64, _i, _i, _vp, _i64, _i64, _i, _i, _vp, _i, _i64, _i64, _vp]),
    "rpsf_apply_masked": (_i, [_vp, _vp, _i64, _i64, _i, _i, _vp, _i64, _i64, _i, _i, _vp, _i, _i64, _i64, _vp, _i64, _i64,
                               _vp]),
    "rpsf_apply_host": (_i, [_vp, _vp, _i, _vp, _i, _i]),
    "rpsf_construct_kernels": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _i, _i, _vp]),
    "rpsf_construct_kernels_dev": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _i, _i, _vp]),
    "rpsf_stack_create": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i]),
    "rpsf_stack_set_kernel": (_i, [_vp, _i, _vp, _i, _vp]),
    "rpsf_stack_destroy": (_i, [_vp]),
    "rpsf_plan_create_stack": (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i]),
    "rpsf_plan_set_stack_mode": (_i, [_vp, _i]),
    "rpsf_plan_stack_info": (_i, [_vp, ctypes.POINTER(_i)]),
    "rpsf_apply_stack": (_i, [_vp, _vp, _i64, _i64, _vp, _i64, _i64, _i, _i, _vp, _i, _i64, _i64, _vp, _i64, _i64, _vp]),
    "rpsf_convert": (_i, [_vp, _i, _i64, _vp, _i, _i64, _i, _i, _i, _vp]),
    "rpsf_plan_workspace": (_i, [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_i64)]),
    "rpsf_apply_stages": (_i, [_vp, _vp, _i64, _i64, _i, _i, _vp, _i64, _i64, _i, _i, _i, _vp]),
    "rpsf_plan_enable_timing": (_i, [_vp, _i]),
    "rpsf_plan_read_timing": (_i, [_vp, ctypes.POINTER(_d), ctypes.POINTER(_i)]),
    "rpsf_pad_index": (_i, [_i, _i, _i]),
    "rpsf_copy_to_host": (_i, [_vp, _vp, _i64, _i]),
    "rpsf_launch_count": (_i64, []),
}

_lib = None
_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """Load the shared library once; raise ``NativeLibraryError`` if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found. Build it with `python -m regularizepsf_b200.csrc.build` "
                "(needs nvcc); regularizepsf_b200 has no CPU fallback.")
        try:
            lib = ctypes.CDLL(LIB_PATH)
        except OSError as exc:  # pragma: no cover - depends on the box
            raise NativeLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def last_error() -> str:
    msg = load().rpsf_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


#: what the library's refusals on a capturing stream say (rpsf_api.cu, refuse_capture)
CAPTURE_REFUSAL = "while a CUDA graph is being captured"


def check(rc: int) -> None:
    """Translate a status code into the reference's exception types (a refusal during graph capture: RuntimeError)."""
    if rc == 0:
        return
    msg = last_error()
    if rc == E_UNSUPPORTED and CAPTURE_REFUSAL in msg:
        raise RuntimeError(msg)
    raise exceptions.for_status(rc)(msg)


def dtype_code(dtype) -> int | None:
    return _NP_CODES.get(np.dtype(dtype))


_torch = None


def require_cuda():
    """Return torch after checking that a CUDA device is visible (checked once: a visible device stays visible)."""
    global _torch
    if _torch is None:
        import torch

        if not torch.cuda.is_available():
            raise NativeLibraryError("no CUDA device is visible; regularizepsf_b200 has no CPU fallback")
        _torch = torch
    return _torch


def current_stream_ptr(torch, device: int | None = None) -> int:
    """cudaStream_t of torch's current stream on ``device`` (default: the current device).  The raw-stream getter is
    one C call; ``torch.cuda.current_stream()`` builds a Stream object through several Python layers (13 us of a
    30 us device-resident apply() call, scripts/host_cost_profile.py)."""
    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:
        return int(raw(torch._C._cuda_getDevice() if device is None else device))
    return int(torch.cuda.current_stream(device).cuda_stream)


def capturing(torch) -> bool:
    """Whether torch's current stream is capturing a CUDA graph (one C call)."""
    return torch.cuda.is_current_stream_capturing()


def refuse_in_capture(torch, what: str) -> None:
    """RuntimeError when the current stream is capturing: ``what`` allocates, synchronises or runs on the host."""
    if capturing(torch):
        raise RuntimeError(f"{what} cannot run while a CUDA graph is being captured; call it outside the capture "
                           "(INTEGRATION.md, \"CUDA graphs\")")


def launch_count() -> int:
    return int(load().rpsf_launch_count())
