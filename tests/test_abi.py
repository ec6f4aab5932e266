"""The C-ABI library loads and exports every symbol include/rpsf_b200.h declares (no GPU compute)."""
import ctypes
import os
import re

import numpy as np
import pytest

from regularizepsf_b200 import _native

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rpsf_b200.h")


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rpsf_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree(native_lib):
    names = declared_functions()
    assert len(names) >= 18
    assert sorted(_native.SIGNATURES) == names
    for name in names:
        assert hasattr(native_lib, name), name


def test_abi_version_3_and_supported_patch_sizes(native_lib):
    # static CUDA runtime: the only CUDA dependency is the driver, resolved lazily.  Version 3: rpsf_plan_info fills
    # nine entries (info[8] = overlap-add chunks per chain), so a caller built for version 2 must not pass its array.
    assert native_lib.rpsf_abi_version() == 3
    for p in (16, 32, 64, 128, 256, 512):
        assert native_lib.rpsf_patch_size_supported(p) == 1
    for p in (2, 8, 11, 100, 255, 256 - 1):            # embedded in the next power of two >= 2 P - 1
        assert native_lib.rpsf_patch_size_supported(p) == 2
    for p in (0, 1, 257, 300, 1024, -4):
        assert native_lib.rpsf_patch_size_supported(p) == 0


@pytest.mark.parametrize("mode", sorted(_native.PAD_MODES))
@pytest.mark.parametrize("n", [1, 2, 3, 7, 16])
def test_pad_index_matches_numpy_pad(native_lib, mode, n):
    if mode == "reflect" and n == 1:
        pytest.skip("np.pad special-cases length-1 reflect")
    code = _native.PAD_MODES[mode]
    pad = 3 * n + 2                      # several reflections deep
    axis = np.arange(n) + 1
    want = np.pad(axis, (pad, pad), mode=mode)
    got = []
    for i in range(-pad, n + pad):
        j = native_lib.rpsf_pad_index(i, n, code)
        got.append(axis[j] if j >= 0 else 0)
    assert np.array_equal(want, np.array(got))


def test_argument_errors_without_a_gpu(native_lib):
    out = ctypes.c_void_p()
    coords = np.zeros((1, 2), dtype=np.int32)
    rc = native_lib.rpsf_transform_create(ctypes.byref(out), coords.ctypes.data, 1, 300, _native.F32, 0)
    assert rc == _native.E_UNSUPPORTED and b"patch size 300" in native_lib.rpsf_last_error()
    with pytest.raises(NotImplementedError):
        _native.check(rc)
    rc = native_lib.rpsf_transform_create(ctypes.byref(out), coords.ctypes.data, 1, 32, 5, 0)
    assert rc == _native.E_UNSUPPORTED
    rc = native_lib.rpsf_plan_create(ctypes.byref(out), None, 10, 10, 0, 0, 10, 1)
    assert rc == _native.E_INVALID_ARGUMENT
