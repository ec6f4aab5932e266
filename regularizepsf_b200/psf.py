"""``ArrayPSF`` with its FFT cube resident in HBM.

Mirrors regularizepsf/psf.py:192-416 for the part of the class the correction path uses
(construction, accessors, equality).  ``fft_evaluations`` keeps the reference layout —
(N, P, P) complex, full unshifted spectrum, complex64 for float32 values and complex128 for
float64 — but is computed by the library's own batched 2-D FFT (``rpsf_psf_fft2``) instead of
``scipy.fft.fft2`` (psf.py:216-219) and stays on the device until a host accessor asks for it.
The cube is computed the first time something needs it (``fft_evaluations``, ``fft_at``,
``ArrayPSFTransform.construct``, ``save``, ``==``), so building models on a host without a GPU works
and only the spectrum itself needs the device.  ``save`` / ``load`` keep the reference's h5 and FITS
layouts (psf.py:262-330).

The values may be a ``DeviceCube``: a real (N, P, P) CUDA tensor of float32 or float64, transformed where it lies.  When
that tensor requires grad, ``ArrayPSFTransform.construct`` differentiates through the FFT (``_autograd.PsfFFT``), and the
host accessors see a detached cube that is computed again after each in-place update of the tensor
(``optimizer.step()``).
"""
from __future__ import annotations

import numpy as np

from regularizepsf_b200 import _native
from regularizepsf_b200.device import DeviceCube
from regularizepsf_b200.exceptions import IncorrectShapeError, InvalidCoordinateError
from regularizepsf_b200.util import IndexedCube


def _values_tensor(values_cube: IndexedCube, torch):
    """The values as a contiguous real CUDA tensor of float32 or float64 (an upload unless they are a ``DeviceCube``),
    without autograd history."""
    if isinstance(values_cube, DeviceCube):
        values = values_cube.tensor.detach()
        if values.dtype not in (torch.float32, torch.float64):
            values = values.to(torch.float64)       # scipy.fft promotes the same way
        return (values if values.is_cuda else values.cuda()).contiguous()
    values = values_cube.values
    if values.dtype not in (np.float32, np.float64):
        values = values.astype(np.float64)          # scipy.fft promotes the same way
    return torch.from_numpy(np.ascontiguousarray(values)).cuda()


def _psf_fft2(values, torch):
    """``rpsf_psf_fft2`` of a contiguous real (N, P, P) CUDA tensor: the complex spectrum cube, on the same device."""
    lib = _native.load()
    n, p0, p1 = values.shape
    if p0 != p1:
        raise IncorrectShapeError(f"PSF samples must be square for the device FFT, got {(p0, p1)}")
    if n and not 1 <= p0 <= 512:
        raise NotImplementedError(f"patch size {p0} has no device path (1..512: radix-2 kernels for powers of two "
                                  "16..512, a direct DFT otherwise)")
    cdtype = torch.complex64 if values.dtype == torch.float32 else torch.complex128
    out = torch.empty((n, p0, p1), dtype=cdtype, device=values.device)
    if n:
        code = _native.F32 if values.dtype == torch.float32 else _native.F64
        with torch.cuda.device(values.device):
            _native.check(lib.rpsf_psf_fft2(values.data_ptr(), out.data_ptr(), n, p0, code, values.device.index,
                                            _native.current_stream_ptr(torch)))
    return out


def _device_fft_cube(values_cube: IndexedCube) -> DeviceCube:
    torch = _native.require_cuda()
    values = _values_tensor(values_cube, torch)
    if values.dim() != 3:
        raise IncorrectShapeError(f"PSF values must be (N, P, P), got shape {tuple(values.shape)}")
    return DeviceCube(values_cube.coordinates, _psf_fft2(values, torch))


class ArrayPSF:
    """A PSF model sampled on a grid of patches (regularizepsf/psf.py:192-237)."""

    def __init__(self, values_cube: IndexedCube, fft_cube: IndexedCube | None = None,
                 workers: int | None = None) -> None:
        self._values_cube = values_cube
        self._workers = workers                      # accepted for API parity; the GPU ignores it
        self._given_fft_cube = fft_cube              # None: computed on the device at first use
        self._computed_fft_cube = None
        self._computed_version = None                # values tensor version the computed cube was made from
        self._uploaded_fft = None                    # the last upload of a host FFT cube given here (_device_spectrum)
        self._captured_uploads = []                  # uploads CUDA graphs read: never freed before the PSF
        if fft_cube is None:
            return                                   # a computed cube matches the values cube by construction
        if fft_cube.sample_shape != self._values_cube.sample_shape:
            raise IncorrectShapeError(
                f"Values cube and FFT cube have different sample shapes: "
                f"{self._values_cube.sample_shape} != {fft_cube.sample_shape}.")
        if len(fft_cube) != len(self._values_cube):
            raise IncorrectShapeError(
                f"Values cube and FFT cube have different sample counts: "
                f"{len(self._values_cube)} != {len(fft_cube)}.")
        if np.any(np.array(self._values_cube.coordinates) != np.array(fft_cube.coordinates)):
            raise InvalidCoordinateError("Values cube and FFT cube have different coordinates")

    @property
    def _fft_cube(self) -> IndexedCube:
        if self._given_fft_cube is not None:
            return self._given_fft_cube
        tensor = self._values_device_tensor
        version = tensor._version if tensor is not None and tensor.requires_grad else None
        if self._computed_fft_cube is None or version != self._computed_version:
            self._computed_fft_cube = _device_fft_cube(self._values_cube)
            self._computed_version = version
        return self._computed_fft_cube

    def _device_spectrum(self, torch):
        """The FFT cube as a CUDA tensor.  A host cube given to the constructor is uploaded at every eager call; the last
        upload serves calls captured in a CUDA graph, which cannot copy from the host (RuntimeError when no eager call
        has made one), and an upload a capture has used is kept with the PSF, since its graphs read it at every
        replay."""
        cube = self._fft_cube
        if isinstance(cube, DeviceCube):
            return cube.tensor.contiguous()
        if _native.capturing(torch):
            if self._uploaded_fft is None:
                raise RuntimeError("this PSF's FFT cube is on the host, and uploading it cannot be captured in a CUDA "
                                   "graph: run the same call once before capturing")
            if not any(u is self._uploaded_fft for u in self._captured_uploads):
                self._captured_uploads.append(self._uploaded_fft)
            return self._uploaded_fft
        self._uploaded_fft = torch.from_numpy(np.ascontiguousarray(cube.values)).cuda()
        return self._uploaded_fft

    @property
    def _values_device_tensor(self):
        """The CUDA tensor of the values when they are a ``DeviceCube``, else None."""
        return self._values_cube.tensor if isinstance(self._values_cube, DeviceCube) else None

    @property
    def coordinates(self):
        return self._values_cube.coordinates

    @property
    def values(self) -> np.ndarray:
        return self._values_cube.values

    @property
    def fft_evaluations(self) -> np.ndarray:
        return self._fft_cube.values

    @property
    def fft_cube(self) -> IndexedCube:
        """The FFT cube object itself (a ``DeviceCube`` when it was computed on the GPU)."""
        return self._fft_cube

    def __getitem__(self, coord) -> np.ndarray:
        return self._values_cube[coord]

    def fft_at(self, coord) -> np.ndarray:
        return self._fft_cube[coord]

    @property
    def sample_shape(self) -> tuple[int, int]:
        return self._values_cube.sample_shape

    def __len__(self) -> int:
        return len(self._values_cube)

    def __eq__(self, other) -> bool:
        if not isinstance(other, ArrayPSF):
            raise TypeError("Can only compare ArrayPSF to other ArrayPSF.")
        return self._values_cube == other._values_cube and self._fft_cube == other._fft_cube

    __hash__ = None

    # ------------------------------------------------------------------ persistence (psf.py:262-330)
    def save(self, path) -> None:
        """Save the model: ``.h5`` (coordinates, values, fft_evaluations) or ``.fits``."""
        from regularizepsf_b200 import persistence
        persistence.write_cubes(path, self.coordinates, {"values": self.values, "fft_evaluations": self.fft_evaluations})

    @classmethod
    def load(cls, path) -> "ArrayPSF":
        """Load a model written by this class or by the reference package."""
        from regularizepsf_b200 import persistence
        coordinates, cubes = persistence.read_cubes(path, {"values": False, "fft_evaluations": True})
        return cls(IndexedCube(coordinates, cubes["values"]), IndexedCube(coordinates, cubes["fft_evaluations"]))
