"""The reference-side binding: plugin classes that subclass GPy's OWN kernel / inference classes and route the hot
path through libgpx (see INTEGRATION.md). Use where GPy (+ paramz) is importable:

    import GPy
    from gpy_b200 import gpy_plugin
    B = gpy_plugin.load()                       # subclasses of GPy.kern.RBF/Matern32/Matern52/Exponential + inference
    m = GPy.models.GPRegression(X, Y, kernel=B.RBF(D, ARD=True))
    m.inference_method = B.ExactGaussianInference()      # same hook the reference's tests use (GPy/testing/fitc.py:31)
    m.optimize()                                # paramz loop unchanged; one gpx_exact_eval per iterate

`make(...)` takes the base classes explicitly so that the wiring can be exercised against the unmodified reference
modules in the build container (tests/test_gpy_plugin_cpu.py) where the full `import GPy` is impossible (no paramz).

The sparse model is a drop-in the same way — the reference's own `GPy.core.SparseGP` / `SparseGPRegression`, UNCHANGED:

    m = GPy.core.SparseGP(X, Y, Z, B.RBF(D, ARD=True), GPy.likelihoods.Gaussian(), inference_method=B.VarDTC())

`B.VarDTC.inference` makes ONE `gpx_sparse_eval` (or `gpx_sparse_eval_het`) and returns a grad_dict whose `dL_dKnm` /
`dL_dKmm` are handles carrying the gradients the device already reduced; `SparseGP._update_gradients`
(core/sparse_gp.py:108-119) then calls the plugin kernel's `update_gradients_diag / update_gradients_full / gradients_X`
exactly as written there and gets those numbers back (the N x M matrix dL_dKnm never exists).

The methods `K`, `Kdiag`, `update_gradients_full`, `update_gradients_diag`, `gradients_X` are defined in the class bodies on purpose:
`KernCallsViaSlicerMeta` only wraps names it finds in the class dict (GPy/kern/src/kernel_slice_operations.py:14-57), and
the wrapper hands them X already sliced to `active_dims` (GPy/kern/src/kern.py:112-117).
"""
import types

import numpy as np

from . import _ffi
from .inference import PosteriorExact, _DataKey, _LazyAlpha
from .kern import DeviceGradient

_KINDS = {"RBF": "rbf", "Exponential": "exponential", "Matern32": "matern32", "Matern52": "matern52"}


class SparseDeviceGradient(object):
    """Stand-in for `grad_dict['dL_dKnm']` (N x M) / `grad_dict['dL_dKmm']` (M x M) of VarDTC.inference
    (var_dtc.py:178-188). The device evaluation has already reduced both to d/d(variance, lengthscale) and dL/dZ
    (core/sparse_gp.py:110-118); the handle carries its share, keyed by the kernel state and the inducing inputs they were
    computed for. `.T` is the same handle (SparseGP passes `dL_dKnm.T` to `gradients_X`, :118). It cannot turn into an
    ndarray: the N x M matrix is never formed."""

    def __init__(self, key, role, shape, dvariance, dlengthscale, dZ):
        self._key, self.role, self.shape = key, role, shape
        self.dvariance, self.dlengthscale, self.dZ = dvariance, dlengthscale, dZ
        self.ndim, self.dtype = 2, np.dtype(np.float64)

    def matches(self, key):
        return self._key == key

    @property
    def T(self):
        h = SparseDeviceGradient(self._key, self.role, self.shape[::-1], self.dvariance, self.dlengthscale, self.dZ)
        return h

    def __array__(self, dtype=None, copy=None):
        raise TypeError("%s of the device VarDTC evaluation is a handle to already-reduced gradients; the matrix itself is "
                        "never materialised (use a gpy_plugin kernel, or the stock VarDTC)" % (
                            "dL_dKnm" if self.role == "knm" else "dL_dKmm"))


def _make_kernel(base, kind, ffi):
    class B200Kernel(base):
        _gpx_kind = kind

        def _gpx_theta(self):
            ls = np.asarray(self.lengthscale.values if hasattr(self.lengthscale, "values") else self.lengthscale,
                            dtype=np.float64).reshape(-1)
            return kind, bool(self.ARD), float(np.asarray(self.variance).reshape(-1)[0]), (ls if self.ARD else float(ls[0]))

        def _gpx_state_key(self):
            k, ard, var, ls = self._gpx_theta()
            return (k, ard, var, tuple(np.atleast_1d(ls).tolist()), tuple(np.atleast_1d(self.active_dims).tolist()))

        def K(self, X, X2=None):
            k, ard, var, ls = self._gpx_theta()
            return ffi.kern_K(k, ard, var, ls, np.asarray(X, dtype=np.float64),
                              None if X2 is None else np.asarray(X2, dtype=np.float64))

        def Kdiag(self, X):
            return ffi.kern_Kdiag(kind, float(np.asarray(self.variance).reshape(-1)[0]), int(np.asarray(X).shape[0]))

        def update_gradients_full(self, dL_dK, X, X2=None, reset=True):
            if isinstance(dL_dK, DeviceGradient) and X2 is None and dL_dK.matches(self._gpx_state_key()):
                self.variance.gradient = dL_dK.dvariance
                self.lengthscale.gradient = dL_dK.dlengthscale
                return
            if isinstance(dL_dK, SparseDeviceGradient):          # core/sparse_gp.py:112,114 on the device's reductions
                if not dL_dK.matches(self._gpx_state_key()):
                    raise ValueError("stale gradient handle: the kernel parameters changed since the sparse evaluation")
                self.variance.gradient = dL_dK.dvariance
                self.lengthscale.gradient = dL_dK.dlengthscale if self.ARD else np.sum(dL_dK.dlengthscale)
                return
            k, ard, var, ls = self._gpx_theta()
            dv, dl = ffi.kern_grad_full(k, ard, var, ls, np.asarray(X, dtype=np.float64),
                                        np.asarray(dL_dK, dtype=np.float64),
                                        None if X2 is None else np.asarray(X2, dtype=np.float64))
            self.variance.gradient = dv
            self.lengthscale.gradient = dl if self.ARD else dl[0]

        def update_gradients_diag(self, dL_dKdiag, X):
            self.variance.gradient = np.sum(dL_dKdiag)
            self.lengthscale.gradient = 0.

        def gradients_X(self, dL_dK, X, X2=None):
            """stationary.py:245-252,348-366 (gpx_kern_grad_X); with a handle of the device VarDTC evaluation: the dL/dZ
            it already holds (core/sparse_gp.py:117-118)."""
            if isinstance(dL_dK, SparseDeviceGradient):
                if not dL_dK.matches(self._gpx_state_key()):
                    raise ValueError("stale gradient handle: the kernel parameters changed since the sparse evaluation")
                return dL_dK.dZ
            k, ard, var, ls = self._gpx_theta()
            return ffi.kern_grad_X(k, ard, var, ls, np.asarray(X, dtype=np.float64), np.asarray(dL_dK, dtype=np.float64),
                                   None if X2 is None else np.asarray(X2, dtype=np.float64))

    B200Kernel.__name__ = B200Kernel.__qualname__ = base.__name__
    return B200Kernel


def _make_combination(base, is_prod):
    """Add / Prod over GPy's own class: K, Kdiag, gradients_X ... stay the reference's; update_gradients_full recognises the
    handle of a fused composite evaluation and hands every leaf the gradient the device already reduced for it (the stock
    methods would build every factor's N x N matrix on the host: add.py:76-77, prod.py:377-385)."""

    class B200Combination(base):
        def update_gradients_full(self, dL_dK, X, X2=None):
            if isinstance(dL_dK, DeviceGradient) and X2 is None and dL_dK.part_grads is not None \
                    and dL_dK.matches(_composite_key(self)):
                for (leaf, _), g in zip(_flatten(self), dL_dK.part_grads):
                    if getattr(leaf, "_gpx_coreg", False):
                        _set_coreg_gradients(leaf, g)
                        continue
                    leaf.variance.gradient = g[0]
                    if hasattr(leaf, "lengthscale"):
                        leaf.lengthscale.gradient = g[1:] if leaf.ARD else g[1]
                return
            return super(B200Combination, self).update_gradients_full(np.asarray(dL_dK, dtype=np.float64), X, X2)

    B200Combination.__name__ = B200Combination.__qualname__ = base.__name__
    B200Combination._gpx_is_prod = is_prod
    return B200Combination


def _set_coreg_gradients(leaf, S):
    """coregionalize.py:123-128 from the device's S[a, b] = sum of dL_dK over rows of output a and columns of output b"""
    S = np.array(S, dtype=np.float64).reshape(leaf.output_dim, leaf.output_dim)
    dkappa = np.diag(S).copy()
    S += S.T
    leaf.W.gradient = (np.asarray(leaf.W)[:, None, :] * S[:, :, None]).sum(0)
    leaf.kappa.gradient = dkappa


def _coreg_B(leaf):
    """coregionalize.py:80, from the current W and kappa"""
    W = np.asarray(leaf.W, dtype=np.float64)
    return np.dot(W, W.T) + np.diag(np.asarray(leaf.kappa, dtype=np.float64))


def _make_coregionalize(base):
    """GPy.kern.Coregionalize whose update_gradients_full takes the O x O reduction S a fused evaluation of this kernel
    alone already made on the device; any other dL_dK goes to the stock method (coregionalize.py:110-137). K, Kdiag and
    the rest are the reference's. Inside a sum / product, the plugin Add / Prod hand the leaf its S."""

    class B200Coregionalize(base):
        _gpx_coreg = True

        def update_gradients_full(self, dL_dK, X, X2=None):
            if isinstance(dL_dK, DeviceGradient) and X2 is None and dL_dK.part_grads is not None \
                    and len(dL_dK.part_grads) == 1 and dL_dK.matches(_composite_key(self)):
                _set_coreg_gradients(self, dL_dK.part_grads[0])
                return
            return super(B200Coregionalize, self).update_gradients_full(np.asarray(dL_dK, dtype=np.float64), X, X2)

    B200Coregionalize.__name__ = B200Coregionalize.__qualname__ = base.__name__
    return B200Coregionalize


def _is_leaf(k):
    return hasattr(k, "_gpx_kind") or getattr(k, "_gpx_coreg", False) or type(k).__name__ in ("White", "Bias")


def _flatten(kern):
    """GPy kernel object -> [(leaf, term)] when it is a leaf, a product of leaves or a sum of those; else None"""
    def product(k, term):
        if _is_leaf(k):
            return [(k, term)]
        if getattr(k, "_gpx_is_prod", None) is True and all(_is_leaf(q) for q in k.parts):
            return [(q, term) for q in k.parts]
        return None

    if getattr(kern, "_gpx_is_prod", None) is False:
        out = []
        for t, part in enumerate(kern.parts):
            fl = product(part, t)
            if fl is None:
                return None
            out.extend(fl)
        return out
    return product(kern, 0)


def _leaf_descriptor(leaf, term):
    if getattr(leaf, "_gpx_coreg", False):
        return ("coregionalize", False, term, np.atleast_1d(leaf.active_dims).astype(int).tolist(), 1.0, _coreg_B(leaf))
    var = float(np.asarray(leaf.variance).reshape(-1)[0])
    if not hasattr(leaf, "_gpx_kind"):
        return (type(leaf).__name__.lower(), False, term, [], var, None)
    kind, ard, var, ls = leaf._gpx_theta()
    return (kind, ard, term, np.atleast_1d(leaf.active_dims).astype(int).tolist(), var, ls)


def _composite_key(kern):
    fl = _flatten(kern)
    if fl is None:
        return None
    return tuple((t,) + tuple(repr(tuple(x.ravel().tolist()) if isinstance(x, np.ndarray) else x)
                              for x in _leaf_descriptor(leaf, t)) for (leaf, t) in fl)


def _make_vardtc(base, kernel_types, ffi):
    from .sparse import LazySparsePosterior

    class B200VarDTC(base):
        """GPy.inference.latent_function_inference.VarDTC with the whole evaluation on the device (gpx_sparse_eval /
        gpx_sparse_eval_het). Certain inputs, Gaussian / HeteroscedasticGaussian noise, a plugin stationary kernel, no mean
        function; anything else goes to the stock method (var_dtc.py:66-215)."""

        def __init__(self, limit=1, device=0, engine=None):
            super(B200VarDTC, self).__init__(limit)
            self.device, self._engine, self._data_key = device, engine, _DataKey()

        @property
        def engine(self):
            if self._engine is None:
                self._engine = ffi.Engine(self.device)
            return self._engine

        def invalidate_data(self):
            self._data_key.invalidate()

        def __getstate__(self):
            """the stock class pickles as its cache limit (var_dtc.py:39-41: Cacher objects cannot be pickled); the device
            handle is dropped the same way (precedent: GPy/kern/src/rbf.py:313-318)"""
            return {"limit": self.limit, "device": self.device}

        def __setstate__(self, state):
            super(B200VarDTC, self).__setstate__(state["limit"])   # var_dtc.py:43-48 rebuilds the caches
            self.device, self._engine, self._data_key = state.get("device", 0), None, _DataKey()

        def inference(self, kern, X, Z, likelihood, Y, Y_metadata=None, mean_function=None, precision=None, Lm=None,
                      dL_dKmm=None, psi0=None, psi1=None, psi2=None, Z_tilde=None):
            plain_X = isinstance(X, np.ndarray)                    # a VariationalPosterior is not an ndarray subclass
            if (not isinstance(kern, kernel_types) or not plain_X or mean_function is not None or Lm is not None
                    or dL_dKmm is not None or psi0 is not None or psi1 is not None or psi2 is not None):
                return super(B200VarDTC, self).inference(kern, X, Z, likelihood, Y, Y_metadata, mean_function, precision,
                                                         Lm, dL_dKmm, psi0, psi1, psi2, Z_tilde)
            if precision is None:                                  # var_dtc.py:78-80
                variance = np.asarray(likelihood.gaussian_variance(Y_metadata), dtype=np.float64).reshape(-1)
            else:
                variance = 1.0 / np.asarray(precision, dtype=np.float64).reshape(-1)
            Xs = np.ascontiguousarray(kern._slice_X(np.asarray(X)), dtype=np.float64)
            Zs = np.ascontiguousarray(kern._slice_X(np.asarray(Z)), dtype=np.float64)
            Yc = np.ascontiguousarray(Y, dtype=np.float64)
            N, P = Yc.shape
            M = Zs.shape[0]
            eng = self.engine
            if not self._data_key.matches(Xs, Yc):
                eng.sparse_set_data(Xs, Yc)
                self._data_key.remember(Xs, Yc)
            k, ard, var, ls = kern._gpx_theta()
            if variance.size > 1:                                  # het_noise (var_dtc.py:82-84)
                lml, grad, dZ, dR = eng.sparse_eval_het(k, ard, var, ls, Zs, variance)
                beta = 1.0 / np.fmax(variance, self.const_jitter)
                dL_dthetaL = likelihood.exact_inference_gradients(dR, Y_metadata)         # :176
                gk = grad
            else:
                lml, grad, dZ = eng.sparse_eval(k, ard, var, ls, Zs, float(variance[0]))
                beta = np.full(N, 1.0 / max(float(variance[0]), self.const_jitter))
                dL_dthetaL = likelihood.exact_inference_gradients(np.atleast_1d(grad[-1]), Y_metadata)
                gk = grad[:-1]
            if Z_tilde is not None:
                lml += Z_tilde                                     # var_dtc.py:166-170
            dL_dKdiag = -0.5 * P * beta                            # _compute_dL_dpsi: dL_dpsi0 (:218)
            key = kern._gpx_state_key()
            dlen = np.atleast_1d(gk[1:])
            knm = SparseDeviceGradient(key, "knm", (N, M), gk[0] - dL_dKdiag.sum(), dlen, dZ)
            kmm = SparseDeviceGradient(key, "kmm", (M, M), 0.0, np.zeros_like(dlen), np.zeros_like(dZ))
            post = LazySparsePosterior(eng)
            return post, lml, {"dL_dKmm": kmm, "dL_dKdiag": dL_dKdiag, "dL_dKnm": knm, "dL_dthetaL": dL_dthetaL,
                               "dL_dm": None}

    B200VarDTC.__name__ = B200VarDTC.__qualname__ = "VarDTC"
    return B200VarDTC


def make(RBF, Exponential, Matern32, Matern52, ExactGaussianInference, ffi=_ffi, Add=None, Prod=None, VarDTC=None,
         Coregionalize=None):
    """Build the plugin classes on top of the given GPy base classes (Add / Prod optional: composite kernels; VarDTC
    optional: the sparse model; Coregionalize optional: multi-output kernels, fused inside Add / Prod or alone)."""
    kernels = {n: _make_kernel(b, _KINDS[n], ffi) for n, b in
               (("RBF", RBF), ("Exponential", Exponential), ("Matern32", Matern32), ("Matern52", Matern52))}
    kernel_types = tuple(kernels.values())
    if Add is not None and Prod is not None:
        kernels["Add"], kernels["Prod"] = _make_combination(Add, False), _make_combination(Prod, True)
    if Coregionalize is not None:
        kernels["Coregionalize"] = _make_coregionalize(Coregionalize)

    class B200ExactGaussianInference(ExactGaussianInference):
        """GPy.inference.latent_function_inference.ExactGaussianInference with the fused device evaluation; anything the
        accelerated path does not cover (mean function, precomputed K, foreign kernels) goes to the stock method."""

        def __init__(self, device=0, engine=None):
            super(B200ExactGaussianInference, self).__init__()
            self.device, self._engine, self._data_key = device, engine, _DataKey()

        @property
        def engine(self):
            if self._engine is None:
                self._engine = ffi.Engine(self.device)
            return self._engine

        def invalidate_data(self):
            """force an upload at the next inference whatever the content"""
            self._data_key.invalidate()

        def __getstate__(self):
            """pickling goes back to a device-less object (precedent: GPy/kern/src/rbf.py:313-318 drops its GPU state);
            the engine is re-created lazily and the data re-uploaded at the next inference"""
            d = dict(self.__dict__)
            d["_engine"], d["_data_key"] = None, _DataKey()
            return d

        def inference(self, kern, X, likelihood, Y, mean_function=None, Y_metadata=None, K=None, variance=None,
                      Z_tilde=None):
            parts = None
            if mean_function is None and K is None and not isinstance(kern, kernel_types):
                parts = _flatten(kern) if (hasattr(kern, "_gpx_is_prod") or getattr(kern, "_gpx_coreg", False)) else None
            if parts is None and (mean_function is not None or K is not None or not isinstance(kern, kernel_types)):
                return super(B200ExactGaussianInference, self).inference(kern, X, likelihood, Y, mean_function,
                                                                         Y_metadata, K, variance, Z_tilde)
            if variance is None:
                variance = likelihood.gaussian_variance(Y_metadata)
            nvec = np.asarray(variance, dtype=np.float64).reshape(-1)
            het = nvec.size > 1                      # HeteroscedasticGaussian (likelihoods/gaussian.py:347-362)
            if parts is not None:
                # sum / product kernel (add.py, prod.py, static.py, coregionalize.py): ONE device call, data resident;
                # with coregionalization parts or one noise variance per data point (MixedNoise, HeteroscedasticGaussian)
                # gpx_exact_eval_coreg, else gpx_exact_eval_multi
                Xc = np.ascontiguousarray(X, dtype=np.float64)
                Yc = np.ascontiguousarray(Y, dtype=np.float64)
                if het and nvec.size != Yc.shape[0]:
                    raise ValueError("heteroscedastic noise needs one variance per data point")
                if not self._data_key.matches(Xc, Yc):
                    self.engine.set_data(Xc, Yc)
                    self._data_key.remember(Xc, Yc)
                desc = [_leaf_descriptor(l, t) for (l, t) in parts]
                coreg = het or any(getattr(l, "_gpx_coreg", False) for (l, _) in parts)
                if coreg:
                    lml, grad, dnoise, _ = self.engine.exact_eval_coreg(desc, nvec if het else float(nvec[0]), jitter=1e-8,
                                                                        max_tries=5)
                else:
                    lml, grad, _ = self.engine.exact_eval_multi(desc, float(nvec[0]), jitter=1e-8, max_tries=5)
                if Z_tilde is not None:
                    lml += Z_tilde
                pg, i = [], 0
                for (leaf, _) in parts:
                    if getattr(leaf, "_gpx_coreg", False):
                        n = int(leaf.output_dim) ** 2
                    else:
                        n = 1 + (np.asarray(leaf.lengthscale).size if hasattr(leaf, "lengthscale") else 0)
                    pg.append(grad[i:i + n])
                    i += n
                key = _composite_key(kern)
                post = PosteriorExact(self.engine, Yc.shape[0], Yc.shape[1], key)
                dL_dK = DeviceGradient(self.engine, key, None, None, Yc.shape[0], part_grads=pg)
                # exact_gaussian_inference.py:72 with mixed_noise.py:38-41 / gaussian.py:358-359
                dL_dthetaL = likelihood.exact_inference_gradients(dnoise, Y_metadata) if het else grad[-1]
                return post, lml, {"dL_dK": dL_dK, "dL_dthetaL": dL_dthetaL, "dL_dm": _LazyAlpha(post)}
            noise = None if het else float(nvec[0])
            Xs = np.ascontiguousarray(kern._slice_X(X)[0] if _returns_tuple(kern, X) else kern._slice_X(X),
                                      dtype=np.float64)
            Yc = np.ascontiguousarray(Y, dtype=np.float64)
            if not self._data_key.matches(Xs, Yc):   # exact content comparison (GP.set_XY has no hook into inference)
                self.engine.set_data(Xs, Yc)
                self._data_key.remember(Xs, Yc)
            k, ard, var, ls = kern._gpx_theta()
            if het:
                lml, grad, dnoise, _ = self.engine.exact_eval_het(k, ard, var, ls, nvec, jitter=1e-8, max_tries=5)
                dL_dthetaL = likelihood.exact_inference_gradients(dnoise, Y_metadata)   # gaussian.py:358-359
            else:
                lml, grad, _ = self.engine.exact_eval(k, ard, var, ls, noise, jitter=1e-8, max_tries=5)
                dL_dthetaL = grad[-1]
            if Z_tilde is not None:
                lml += Z_tilde
            post = PosteriorExact(self.engine, Yc.shape[0], Yc.shape[1], kern._gpx_state_key())
            dlen = grad[1:-1] if ard else grad[1]
            dL_dK = DeviceGradient(self.engine, kern._gpx_state_key(), grad[0], dlen, Yc.shape[0])
            return post, lml, {"dL_dK": dL_dK, "dL_dthetaL": dL_dthetaL, "dL_dm": _LazyAlpha(post)}

    B200ExactGaussianInference.__name__ = B200ExactGaussianInference.__qualname__ = "ExactGaussianInference"
    extra = {}
    if VarDTC is not None:
        extra["VarDTC"] = _make_vardtc(VarDTC, kernel_types, ffi)
    return types.SimpleNamespace(ExactGaussianInference=B200ExactGaussianInference, **kernels, **extra)


def _returns_tuple(kern, X):
    """Kern._slice_X returns the sliced array; some paramz versions wrap cached results — accept both."""
    r = kern._slice_X(X)
    return isinstance(r, tuple)


def load():
    """Plugin classes over an installed GPy."""
    import GPy
    from GPy.inference.latent_function_inference import ExactGaussianInference, VarDTC
    return make(GPy.kern.RBF, GPy.kern.Exponential, GPy.kern.Matern32, GPy.kern.Matern52, ExactGaussianInference,
                Add=GPy.kern.Add, Prod=GPy.kern.Prod, VarDTC=VarDTC, Coregionalize=GPy.kern.Coregionalize)
