"""Device-resident cubes and small torch helpers (torch is plumbing: memory, streams, NCCL)."""
from __future__ import annotations

import numpy as np

from regularizepsf_b200 import _native
from regularizepsf_b200.util import IndexedCube


class DeviceCube(IndexedCube):
    """An ``IndexedCube`` whose values live in HBM as an (N, P, P) torch CUDA tensor.

    ``values`` downloads (once) to a numpy array in the reference layout, so host-side users —
    ``save()``, ``==``, ``cube[coord]`` — see exactly what the reference's cube would hold
    (regularizepsf/util.py:147-150).  A tensor that requires grad (a transfer kernel being fitted) is downloaded again
    after each in-place update (``optimizer.step()``), so ``save()`` and ``==`` see the fitted values; writes through
    ``tensor.data`` do not bump the tensor's version and are not seen.
    """

    def __init__(self, coordinates, tensor) -> None:
        if tensor.dim() != 3:
            from regularizepsf_b200.exceptions import IncorrectShapeError
            raise IncorrectShapeError("Values must be three dimensional")
        if len(coordinates) != tensor.shape[0]:
            from regularizepsf_b200.exceptions import IncorrectShapeError
            raise IncorrectShapeError(f"{len(coordinates)} coordinates defined but {tensor.shape[0]} values found.")
        self._coordinates = coordinates
        self._tensor = tensor
        self._host = None
        self._host_version = None
        self._index = {tuple(c): i for i, c in enumerate(coordinates)}

    @property
    def tensor(self):
        return self._tensor

    @property
    def sample_shape(self) -> tuple[int, int]:
        return int(self._tensor.shape[1]), int(self._tensor.shape[2])

    @property
    def values(self) -> np.ndarray:
        t = self._tensor
        if t.requires_grad:
            if self._host is None or self._host_version != t._version:
                self._host = t.detach().cpu().numpy()
                self._host_version = t._version
            return self._host
        if self._host is None:
            self._host = t.cpu().numpy()
        return self._host

    @property
    def _values(self):          # IndexedCube internals read this name
        return self.values

    def __setitem__(self, coordinate, value) -> None:
        raise TypeError("device-resident cubes are immutable; build a new IndexedCube from .values")


def cube_tensor(cube: IndexedCube, torch, dtype=None):
    """The cube's values as a contiguous CUDA tensor (upload if it lives on the host)."""
    if isinstance(cube, DeviceCube):
        t = cube.tensor
    else:
        t = torch.from_numpy(np.ascontiguousarray(cube.values)).cuda()
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """A numpy array backed by page-locked memory (torch's caching host allocator)."""
    torch = _native.require_cuda()
    tdtype = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64,
              np.dtype(np.uint16): torch.uint16, np.dtype(np.int16): torch.int16,
              np.dtype(np.uint8): torch.uint8, np.dtype(np.int32): torch.int32,
              np.dtype(np.int64): torch.int64}[np.dtype(dtype)]
    return torch.empty(tuple(shape), dtype=tdtype, pin_memory=True).numpy()
