"""Multi-output helpers mirroring GPy.util.multioutput (multioutput.py:40-135): stack per-output data with an output-index
column and build intrinsic (ICM) / linear (LCM) coregionalization kernels from gpy_b200 kernels."""
import warnings

import numpy as np

from .inference import Gaussian, MixedNoise
from .kern import Coregionalize


def get_slices(input_list):
    """multioutput.py:40-45: the row slice of each output in the stacked data."""
    _s = np.cumsum([0] + [_x.shape[0] for _x in input_list])
    return [slice(a, b) for a, b in zip(_s[:-1], _s[1:])]


def build_XY(input_list, output_list=None, index=None):
    """multioutput.py:48-67 -> (X with the output index as its last column, stacked Y or None, index column)."""
    num_outputs = len(input_list)
    if output_list is not None:
        assert num_outputs == len(output_list)
        Y = np.vstack(output_list)
    else:
        Y = None
    if index is not None:
        assert len(index) == num_outputs
        I = np.hstack([np.repeat(j, _x.shape[0]) for _x, j in zip(input_list, index)])
    else:
        I = np.hstack([np.repeat(j, _x.shape[0]) for _x, j in zip(input_list, range(num_outputs))])
    X = np.vstack(input_list)
    X = np.hstack([X, I[:, None]])
    return X, Y, I[:, None]


def build_likelihood(Y_list, noise_index, likelihoods_list=None):
    """multioutput.py:70-84: a MixedNoise of one Gaussian per output."""
    Ny = len(Y_list)
    if likelihoods_list is None:
        likelihoods_list = [Gaussian(name="Gaussian_noise_%s" % j) for j in range(Ny)]
    else:
        assert len(likelihoods_list) == Ny
    return MixedNoise(likelihoods_list=likelihoods_list)


def ICM(input_dim, num_outputs, kernel, W_rank=1, W=None, kappa=None, name="ICM"):
    """multioutput.py:86-116: kernel * Coregionalize on the column after the inputs (the output index)."""
    if kernel.input_dim != input_dim:
        kernel.input_dim = input_dim
        warnings.warn("kernel's input dimension overwritten to fit input_dim parameter.")
    return kernel.prod(Coregionalize(1, num_outputs, active_dims=[input_dim], rank=W_rank, W=W, kappa=kappa, name="B"),
                       name=name)


def LCM(input_dim, num_outputs, kernels_list, W_rank=1, name="ICM"):
    """multioutput.py:118-135: the sum of one ICM per kernel."""
    K = ICM(input_dim, num_outputs, kernels_list[0], W_rank, name="%s%s" % (name, 0))
    for j, kernel in enumerate(kernels_list[1:], start=1):
        K += ICM(input_dim, num_outputs, kernel, W_rank, name="%s%s" % (name, j))
    return K
