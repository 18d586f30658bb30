"""Host-side mirror of GPy's stationary-kernel plugin interface, computing on the B200 through libgpx.

Same names, argument meaning and error behaviour as the reference classes:
    GPy.kern.RBF           GPy/kern/src/rbf.py:13-52,177-178
    GPy.kern.Exponential   GPy/kern/src/stationary.py:378-386
    GPy.kern.Matern32      GPy/kern/src/stationary.py:457-492
    GPy.kern.Matern52      GPy/kern/src/stationary.py:556-589
base: GPy.kern.src.stationary.Stationary (stationary.py:23-243) and GPy.kern.Kern (kern.py:12-145).
`K`, `Kdiag`, `update_gradients_full`, `update_gradients_diag` take/return NumPy arrays exactly like the reference;
there is no NumPy implementation behind them — every call goes through the C ABI (include/gpx.h).
"""
import numpy as np

from . import _ffi
from .param import Param, Parameterized


class DeviceGradient(object):
    """Lazy, device-backed stand-in for the N x N `dL_dK` that ExactGaussianInference hands to
    `kern.update_gradients_full` (GPy/core/gp.py:278-280). The fused device evaluation has already reduced it to
    the kernel's parameter gradients; this handle carries them (keyed by the kernel state they were computed for)
    and only materialises the matrix (2 GiB at N=16384) if somebody treats it as an ndarray."""

    def __init__(self, engine, key, dvariance, dlengthscale, N, part_grads=None):
        self._engine, self._key = engine, key
        self.dvariance, self.dlengthscale = dvariance, dlengthscale
        self.part_grads = part_grads          # composite kernels: one [variance, lengthscale..] array per flattened part
        self.shape = (N, N)
        self.ndim = 2
        self.dtype = np.dtype(np.float64)
        self._host = None

    def matches(self, key):
        return self._key == key

    def __array__(self, dtype=None, copy=None):
        if self._host is None:
            self._host = np.ascontiguousarray(self._engine.get("dL_dK"))  # symmetric: C == F order
        return self._host if dtype is None else self._host.astype(dtype)

    def __getitem__(self, idx):
        return self.__array__()[idx]


class Kern(Parameterized):
    """Subset of GPy.kern.Kern (kern.py:12-145) the exact-GP path uses: active_dims slicing + the abstract plugin
    methods."""

    def __init__(self, input_dim, active_dims, name):
        super(Kern, self).__init__(name)
        self.input_dim = int(input_dim)
        if active_dims is None:
            active_dims = np.arange(self.input_dim)
        self.active_dims = np.atleast_1d(np.asarray(active_dims, dtype=np.int64))
        assert self.active_dims.size == self.input_dim, "input_dim=%d does not match len(active_dim)=%d" % (
            self.input_dim, self.active_dims.size)

    def _slice_X(self, X):
        """kern.py:112-117: column-select the active dims and cast to float."""
        X = np.asarray(X)
        if X.shape[1] == self.input_dim and np.array_equal(self.active_dims, np.arange(self.input_dim)):
            return np.ascontiguousarray(X, dtype=np.float64)
        return np.ascontiguousarray(X[:, self.active_dims], dtype=np.float64)

    def K(self, X, X2=None):
        raise NotImplementedError

    def Kdiag(self, X):
        raise NotImplementedError

    def update_gradients_full(self, dL_dK, X, X2=None):
        raise NotImplementedError

    # kern.py:311-360: operator overloading builds combination kernels
    def __add__(self, other):
        return self.add(other)

    def add(self, other, name="sum"):
        assert isinstance(other, Kern), "only kernels can be added to kernels..."
        return Add([self, other], name=name)

    def __mul__(self, other):
        return self.prod(other)

    def prod(self, other, name="mul"):
        assert isinstance(other, Kern), "only kernels can be multiplied to kernels..."
        return Prod([self, other], name)

    @property
    def is_fixed(self):
        ps = self.flattened_parameters()
        return bool(ps) and all(p.is_fixed for p in ps)


class Stationary(Kern):
    """GPy.kern.src.stationary.Stationary (stationary.py:23-243): variance + (ARD) lengthscale, K = K_of_r(r)."""

    _kind = None

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name="stationary"):
        super(Stationary, self).__init__(input_dim, active_dims, name)
        self.ARD = bool(ARD)
        # stationary.py:61-77: default / shape checking of the lengthscale
        if not ARD:
            if lengthscale is None:
                lengthscale = np.ones(1)
            else:
                lengthscale = np.asarray(lengthscale, dtype=np.float64)
                assert lengthscale.size == 1, "Only 1 lengthscale needed for non-ARD kernel"
        else:
            if lengthscale is not None:
                lengthscale = np.asarray(lengthscale, dtype=np.float64)
                assert lengthscale.size in [1, input_dim], "Bad number of lengthscales"
                if lengthscale.size != input_dim:
                    lengthscale = np.ones(input_dim) * lengthscale
            else:
                lengthscale = np.ones(self.input_dim)
        self.lengthscale = Param("lengthscale", lengthscale)
        self.variance = Param("variance", variance)
        assert self.variance.size == 1
        self.link_parameters(self.variance, self.lengthscale)  # stationary.py:81

    # -- state key used to recognise gradients precomputed by the fused evaluation ------------------------------
    def _state_key(self):
        return (self._kind, self.ARD, float(self.variance[0]), tuple(self.lengthscale.values.tolist()),
                tuple(self.active_dims.tolist()))

    def _theta(self):
        ls = self.lengthscale.values if self.ARD else self.lengthscale.values[0]
        return self._kind, self.ARD, float(self.variance[0]), ls

    # -- plugin interface -------------------------------------------------------------------------------------
    def K(self, X, X2=None):
        """stationary.py:105-115 -> gpx_kern_K."""
        X = self._slice_X(X)
        X2 = None if X2 is None else self._slice_X(X2)
        kind, ard, var, ls = self._theta()
        return _ffi.kern_K(kind, ard, var, ls, X, X2)

    def Kdiag(self, X):
        """stationary.py:170-173 -> gpx_kern_Kdiag."""
        return _ffi.kern_Kdiag(self._kind, float(self.variance[0]), int(np.asarray(X).shape[0]))

    def update_gradients_full(self, dL_dK, X, X2=None, reset=True):
        """stationary.py:193-213. A DeviceGradient handle from our ExactGaussianInference short-circuits to the
        gradients the fused epilogue already reduced on the device; any other dL_dK goes through gpx_kern_grad_full."""
        if isinstance(dL_dK, DeviceGradient) and X2 is None and dL_dK.matches(self._state_key()):
            self.variance.gradient = np.atleast_1d(dL_dK.dvariance)
            self.lengthscale.gradient = np.atleast_1d(dL_dK.dlengthscale).copy()
            return
        Xs = self._slice_X(X)
        X2s = None if X2 is None else self._slice_X(X2)
        kind, ard, var, ls = self._theta()
        dv, dl = _ffi.kern_grad_full(kind, ard, var, ls, Xs, np.asarray(dL_dK, dtype=np.float64), X2s)
        self.variance.gradient = np.atleast_1d(dv)
        self.lengthscale.gradient = np.atleast_1d(dl)

    def gradients_X(self, dL_dK, X, X2=None):
        """stationary.py:245-252 -> gpx_kern_grad_X (needed by inducing-point / latent-variable models)."""
        Xs = self._slice_X(X)
        X2s = None if X2 is None else self._slice_X(X2)
        kind, ard, var, ls = self._theta()
        g = _ffi.kern_grad_X(kind, ard, var, ls, Xs, np.asarray(dL_dK, dtype=np.float64), X2s)
        if Xs.shape[1] == np.asarray(X).shape[1]:
            return g
        full = np.zeros(np.asarray(X).shape)       # kernel_slice_operations.py:138-150: scatter into the full X
        full[:, self.active_dims] = g
        return full

    def gradients_X_diag(self, dL_dKdiag, X):
        """stationary.py:368-369."""
        return np.zeros(np.asarray(X).shape)

    def update_gradients_diag(self, dL_dKdiag, X):
        """stationary.py:182-192."""
        self.variance.gradient = np.atleast_1d(np.sum(dL_dKdiag))
        self.lengthscale.gradient = np.zeros_like(self.lengthscale.values)

    def reset_gradients(self):
        """stationary.py:175-180."""
        self.variance.gradient = np.zeros(1)
        self.lengthscale.gradient = np.zeros_like(self.lengthscale.values)


class RBF(Stationary):
    """GPy.kern.RBF (rbf.py:13-52): k(r) = variance * exp(-0.5 r^2)."""
    _kind = "rbf"

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name="rbf"):
        super(RBF, self).__init__(input_dim, variance, lengthscale, ARD, active_dims, name)


class Exponential(Stationary):
    """GPy.kern.Exponential (stationary.py:378-386): k(r) = variance * exp(-r)."""
    _kind = "exponential"

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name="Exponential"):
        super(Exponential, self).__init__(input_dim, variance, lengthscale, ARD, active_dims, name)


class Matern32(Stationary):
    """GPy.kern.Matern32 (stationary.py:457-492)."""
    _kind = "matern32"

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name="Mat32"):
        super(Matern32, self).__init__(input_dim, variance, lengthscale, ARD, active_dims, name)


class Matern52(Stationary):
    """GPy.kern.Matern52 (stationary.py:556-589)."""
    _kind = "matern52"

    def __init__(self, input_dim, variance=1., lengthscale=None, ARD=False, active_dims=None, name="Mat52"):
        super(Matern52, self).__init__(input_dim, variance, lengthscale, ARD, active_dims, name)


# ----------------------------------------------------------------------------------------------------------------------
# combination / static kernels (SURVEY.md §8f item 4). Mirrors GPy/kern/src/add.py:60-99, prod.py:59-68,377-396,
# static.py:63-185. A GP whose kernel is a sum of products of stationary / White / Bias leaves is evaluated by ONE device
# call (gpx_exact_eval_multi: the K-build multiplies / adds the parts in registers, every part's gradient is reduced from
# the stored K^-1 with the other factors of its term recomputed on the fly); `flatten_parts` is the translation.
# The stand-alone K / update_gradients_full methods below (foreign dL_dK, nested structures the flattening does not cover)
# build the parts' matrices on the device and do the O(N^2) glue in NumPy on the host.
# ----------------------------------------------------------------------------------------------------------------------
def flatten_parts(kern):
    """-> list of (leaf kernel, term index) for a kernel that is a leaf, a product of leaves, or a sum of those; None for
    anything else (e.g. a product containing a sum), which then takes the generic inference path."""
    def leaf(k):
        return isinstance(k, (Stationary, White, Bias, Coregionalize))

    def product(k, term):
        if leaf(k):
            return [(k, term)]
        if isinstance(k, Prod) and all(leaf(q) for q in k.parts):
            return [(q, term) for q in k.parts]
        return None

    if isinstance(kern, Add):
        out = []
        for t, part in enumerate(kern.parts):
            fl = product(part, t)
            if fl is None:
                return None
            out.extend(fl)
        return out
    return product(kern, 0)


def part_descriptor(leaf, term):
    """(kind, ARD, term, dims, variance, lengthscale) of one leaf for Engine.exact_eval_multi"""
    if isinstance(leaf, White):
        return ("white", False, term, [], float(leaf.variance[0]), None)
    if isinstance(leaf, Bias):
        return ("bias", False, term, [], float(leaf.variance[0]), None)
    if isinstance(leaf, Coregionalize):
        return ("coregionalize", False, term, leaf.active_dims.tolist(), 1.0, leaf.B)
    kind, ard, var, ls = leaf._theta()
    return (kind, ard, term, leaf.active_dims.tolist(), var, ls)


def composite_state_key(kern):
    fl = flatten_parts(kern)
    if fl is None:
        return None
    return tuple((t, type(k).__name__) + (k._state_key() if isinstance(k, Coregionalize) else (
                  float(k.variance[0]), tuple(k.lengthscale.values.tolist()) if isinstance(k, Stationary) else (),
                  tuple(k.active_dims.tolist()))) for (k, t) in fl)


def scatter_part_gradients(kern, dL_dK):
    """hand the per-part gradients of a fused composite evaluation to the leaves (what Add / Prod.update_gradients_full do
    with a dense dL_dK); -> False if the handle does not belong to this kernel state"""
    if not (isinstance(dL_dK, DeviceGradient) and dL_dK.part_grads is not None and dL_dK.matches(composite_state_key(kern))):
        return False
    for (leaf, _), g in zip(flatten_parts(kern), dL_dK.part_grads):
        if isinstance(leaf, Coregionalize):
            leaf.set_gradients_from_S(np.asarray(g).reshape(leaf.output_dim, leaf.output_dim))
            continue
        leaf.variance.gradient = np.atleast_1d(g[0])
        if isinstance(leaf, Stationary):
            leaf.lengthscale.gradient = np.atleast_1d(g[1:]).copy()
    return True



class CombinationKernel(Kern):
    """GPy.kern.src.kern.CombinationKernel (kern.py:363-451): a kernel made of parts; active dims = union."""

    def __init__(self, kernels, name):
        assert all(isinstance(p, Kern) for p in kernels)
        input_dim = int(max(int(np.max(p.active_dims)) for p in kernels) + 1)
        super(CombinationKernel, self).__init__(input_dim, np.arange(input_dim), name)
        self.parts = list(kernels)
        for p in self.parts:
            self.link_parameter(p)

    def _slice_X(self, X):
        return np.ascontiguousarray(X, dtype=np.float64)


class Add(CombinationKernel):
    """GPy.kern.Add (add.py:11-86)."""

    def __init__(self, subkerns, name="sum"):
        flat = []
        for s in subkerns:                       # add.py:20-27: nested sums are flattened
            flat.extend(s.parts if isinstance(s, Add) else [s])
        super(Add, self).__init__(flat, name)

    def K(self, X, X2=None):
        out = None
        for p in self.parts:
            Kp = p.K(X, X2)
            out = Kp if out is None else out + Kp
        return out

    def Kdiag(self, X):
        return sum(p.Kdiag(X) for p in self.parts)

    def update_gradients_full(self, dL_dK, X, X2=None):
        if X2 is None and scatter_part_gradients(self, dL_dK):
            return
        dL_dK = np.asarray(dL_dK, dtype=np.float64)
        for p in self.parts:
            if not p.is_fixed:
                p.update_gradients_full(dL_dK, X, X2)

    def update_gradients_diag(self, dL_dKdiag, X):
        for p in self.parts:
            p.update_gradients_diag(dL_dKdiag, X)

    def gradients_X(self, dL_dK, X, X2=None):
        return sum(p.gradients_X(dL_dK, X, X2) for p in self.parts)


class Prod(CombinationKernel):
    """GPy.kern.Prod (prod.py:23-110)."""

    def __init__(self, kernels, name="mul"):
        flat = []
        for s in kernels:
            flat.extend(s.parts if isinstance(s, Prod) else [s])
        super(Prod, self).__init__(flat, name)

    def K(self, X, X2=None):
        out = None
        for p in self.parts:
            Kp = p.K(X, X2)
            out = Kp if out is None else out * Kp
        return out

    def Kdiag(self, X):
        out = None
        for p in self.parts:
            Kp = p.Kdiag(X)
            out = Kp if out is None else out * Kp
        return out

    def update_gradients_full(self, dL_dK, X, X2=None):
        """prod.py:377-385: each part sees dL_dK times the product of the other parts."""
        if X2 is None and scatter_part_gradients(self, dL_dK):
            return
        dL_dK = np.asarray(dL_dK, dtype=np.float64)
        Ks = [p.K(X, X2) for p in self.parts]
        for i, p in enumerate(self.parts):
            other = None
            for j, Kj in enumerate(Ks):
                if j != i:
                    other = Kj if other is None else other * Kj
            p.update_gradients_full(dL_dK * other if other is not None else dL_dK, X, X2)

    def gradients_X(self, dL_dK, X, X2=None):
        dL_dK = np.asarray(dL_dK, dtype=np.float64)
        Ks = [p.K(X, X2) for p in self.parts]
        out = 0.0
        for i, p in enumerate(self.parts):
            other = None
            for j, Kj in enumerate(Ks):
                if j != i:
                    other = Kj if other is None else other * Kj
            out = out + p.gradients_X(dL_dK * other if other is not None else dL_dK, X, X2)
        return out


class Static(Kern):
    """GPy.kern.src.static.Static (static.py:11-61): a variance parameter, no dependence on X."""

    def __init__(self, input_dim, variance, active_dims, name):
        super(Static, self).__init__(input_dim, active_dims, name)
        self.variance = Param("variance", variance)
        self.link_parameter(self.variance)

    def Kdiag(self, X):
        ret = np.empty((np.asarray(X).shape[0],), dtype=np.float64)
        ret[:] = self.variance[0]
        return ret

    def gradients_X(self, dL_dK, X, X2=None):
        return np.zeros(np.asarray(X).shape)

    def update_gradients_diag(self, dL_dKdiag, X):
        self.variance.gradient = np.atleast_1d(np.sum(dL_dKdiag))


class White(Static):
    """GPy.kern.White (static.py:63-99)."""

    def __init__(self, input_dim, variance=1., active_dims=None, name="white"):
        super(White, self).__init__(input_dim, variance, active_dims, name)

    def K(self, X, X2=None):
        n = np.asarray(X).shape[0]
        if X2 is None:
            return np.eye(n) * self.variance[0]
        return np.zeros((n, np.asarray(X2).shape[0]))

    def update_gradients_full(self, dL_dK, X, X2=None):
        self.variance.gradient = np.atleast_1d(np.trace(np.asarray(dL_dK)) if X2 is None else 0.)


class Bias(Static):
    """GPy.kern.Bias (static.py:142-185)."""

    def __init__(self, input_dim, variance=1., active_dims=None, name="bias"):
        super(Bias, self).__init__(input_dim, variance, active_dims, name)

    def K(self, X, X2=None):
        shape = (np.asarray(X).shape[0], np.asarray(X).shape[0] if X2 is None else np.asarray(X2).shape[0])
        return np.full(shape, self.variance[0], dtype=np.float64)

    def update_gradients_full(self, dL_dK, X, X2=None):
        self.variance.gradient = np.atleast_1d(np.asarray(dL_dK).sum())


class Coregionalize(Kern):
    """GPy.kern.Coregionalize (coregionalize.py:17-157): K(x, x') = B[int(x), int(x')] on one active dim holding the output
    index, B = W W^T + diag(kappa). W (output_dim x rank) is unconstrained, kappa (output_dim) positive (Logexp). Inside a
    model evaluated by ExactGaussianInference the part runs on the device (gpx_exact_eval_coreg), which hands back the
    O x O reduction S of dL_dK; K / Kdiag / update_gradients_full below are the host gathers and sums of the reference for
    any other caller."""

    def __init__(self, input_dim, output_dim, rank=1, W=None, kappa=None, active_dims=None, name="coregion"):
        super(Coregionalize, self).__init__(input_dim, active_dims, name)
        self.output_dim = int(output_dim)
        self.rank = int(rank)
        if W is None:                                                          # coregionalize.py:66-69
            W = 0.5 * np.random.randn(self.output_dim, self.rank) / np.sqrt(self.rank)
        else:
            W = np.asarray(W, dtype=np.float64)
            assert W.shape == (self.output_dim, self.rank)
        if kappa is None:                                                      # coregionalize.py:71-74
            kappa = 0.5 * np.ones(self.output_dim)
        else:
            kappa = np.asarray(kappa, dtype=np.float64)
            assert kappa.shape == (self.output_dim,)
        self.W = Param("W", W, transform=None)
        self.kappa = Param("kappa", kappa)
        self.link_parameters(self.W, self.kappa)

    @property
    def B(self):
        """coregionalize.py:80"""
        return np.dot(self.W.values, self.W.values.T) + np.diag(self.kappa.values)

    def _state_key(self):
        return (tuple(self.W.values.reshape(-1).tolist()), tuple(self.kappa.values.tolist()), tuple(self.active_dims.tolist()))

    def _index(self, X):
        return np.asarray(self._slice_X(X), dtype=int)[:, 0]

    def K(self, X, X2=None):
        """coregionalize.py:88-94 (a gather of B)"""
        i = self._index(X)
        j = i if X2 is None else self._index(X2)
        return self.B[i[:, None], j[None, :]]

    def Kdiag(self, X):
        """coregionalize.py:107-108"""
        return np.diag(self.B)[self._index(X)]

    def set_gradients_from_S(self, S):
        """coregionalize.py:123-128 from S[a, b] = sum of dL_dK over rows with index a and columns with index b"""
        S = np.array(S, dtype=np.float64)
        dkappa = np.diag(S).copy()
        S += S.T
        self.W.gradient = (self.W.values[:, None, :] * S[:, :, None]).sum(0)
        self.kappa.gradient = dkappa

    def update_gradients_full(self, dL_dK, X, X2=None):
        """coregionalize.py:110-137 with the NumPy reduction (:130-137)"""
        i = self._index(X)
        j = i if X2 is None else self._index(X2)
        dL_dK = np.asarray(dL_dK, dtype=np.float64)
        S = np.zeros((self.output_dim, self.output_dim))
        for a in range(self.output_dim):
            rows = dL_dK[i == a]
            for b in range(self.output_dim):
                S[a, b] = rows[:, j == b].sum()
        self.set_gradients_from_S(S)

    def update_gradients_diag(self, dL_dKdiag, X):
        """coregionalize.py:145-151"""
        i = self._index(X)
        dL_dKdiag_small = np.array([np.asarray(dL_dKdiag)[i == a].sum() for a in range(self.output_dim)])
        self.W.gradient = 2. * self.W.values * dL_dKdiag_small[:, None]
        self.kappa.gradient = dL_dKdiag_small

    def gradients_X(self, dL_dK, X, X2=None):
        """coregionalize.py:153-154"""
        return np.zeros(np.asarray(X).shape)

    def gradients_X_diag(self, dL_dKdiag, X):
        """coregionalize.py:156-157"""
        return np.zeros(np.asarray(X).shape)
