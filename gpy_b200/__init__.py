"""gpy_b200 — B200-native exact-GP engine behind GPy's kernel / exact-inference plugin interface.

Host side (Python, mirrors the reference's operator interface for the hot path) over a ctypes C ABI
(include/gpx.h) into hand-written sm_100a CUDA (gpy_b200/csrc). No CPU fallback: importing works everywhere,
computing requires libgpx.so and a B200.
"""
from . import _ffi  # noqa: F401
from ._ffi import Engine, GpxError, kern_K, kern_Kdiag, kern_grad_full  # noqa: F401

from .kern import (RBF, Exponential, Matern32, Matern52, Stationary, DeviceGradient, Add, Prod, White, Bias,  # noqa: F401
                   Kern, CombinationKernel, Coregionalize)
from .inference import (ExactGaussianInference, Gaussian, HeteroscedasticGaussian, MixedNoise,  # noqa: F401
                        PosteriorExact)
from .model import GP, GPCoregionalizedRegression, GPHeteroscedasticRegression, GPRegression  # noqa: F401
from .multioutput import ICM, LCM, build_XY  # noqa: F401
from .sparse import SparseGPRegression, VarDTC  # noqa: F401

__version__ = "0.1.0"
