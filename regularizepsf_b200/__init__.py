"""regularizepsf_b200 — B200-native drop-in for regularizepsf's correction hot path.

Same public names as the reference package (regularizepsf/__init__.py:5-16): ``ArrayPSF``,
``ArrayPSFTransform`` (``construct`` / ``apply`` / ``save`` / ``load``), ``IndexedCube``,
``calculate_covering``, the functional PSF decorators, ``ArrayPSFBuilder`` (stack averaging on the
GPU, star finding through the optional ``sep`` dependency as in the reference) and the exception
types.  ``DeviceCube`` holds a cube as a CUDA tensor: a transform built on one whose tensor requires grad is
trainable (``ArrayPSFTransform.apply`` differentiates with respect to the transfer kernel), and an ``ArrayPSF`` whose
values are a ``DeviceCube`` that requires grad makes ``ArrayPSFTransform.construct`` differentiable in the PSF values,
as 0-d tensors ``alpha`` and ``epsilon`` do.  ``TransformStack`` applies many transfer kernels (an alpha / epsilon
sweep) to the same frames in one call.  Plotting is out of scope (see DESIGN.md).
"""
from regularizepsf_b200.exceptions import (
    FunctionParameterMismatchError,
    IncorrectShapeError,
    InvalidCoordinateError,
    InvalidDataError,
    InvalidFunctionError,
    NativeLibraryError,
    PSFBuilderError,
    RegularizePSFError,
)
from regularizepsf_b200.builder import ArrayPSFBuilder
from regularizepsf_b200.device import DeviceCube
from regularizepsf_b200.psf import ArrayPSF
from regularizepsf_b200.functional import (
    SimpleFunctionalPSF,
    VariedFunctionalPSF,
    simple_functional_psf,
    varied_functional_psf,
)
from regularizepsf_b200.transform import ArrayPSFTransform, set_default_dtype
from regularizepsf_b200.stack import TransformStack
from regularizepsf_b200.util import IndexedCube, calculate_covering

__version__ = "0.1.0"

__all__ = [
    "ArrayPSF", "ArrayPSFBuilder", "ArrayPSFTransform", "TransformStack", "DeviceCube", "IndexedCube", "calculate_covering", "set_default_dtype",
    "SimpleFunctionalPSF", "VariedFunctionalPSF", "simple_functional_psf", "varied_functional_psf",
    "RegularizePSFError", "InvalidCoordinateError", "IncorrectShapeError", "InvalidFunctionError",
    "FunctionParameterMismatchError", "PSFBuilderError", "InvalidDataError", "NativeLibraryError",
    "__version__",
]
