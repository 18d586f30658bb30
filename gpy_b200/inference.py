"""Host-side mirror of GPy's exact Gaussian inference plugin, computing on the B200 through libgpx.

Mirrors (same names, argument meaning, return structure and error behaviour):
    GPy.inference.latent_function_inference.ExactGaussianInference.inference
        GPy/inference/latent_function_inference/exact_gaussian_inference.py:37-74
    GPy.inference.latent_function_inference.posterior.PosteriorExact
        GPy/inference/latent_function_inference/posterior.py:9-77,273-302
    GPy.likelihoods.Gaussian (the three one-liners on the path)  GPy/likelihoods/gaussian.py:69-79,102-110
    GPy.likelihoods.HeteroscedasticGaussian / MixedNoise (vector noise)  GPy/likelihoods/gaussian.py:347-377, mixed_noise.py:14-53
"""
import numpy as np

from . import _ffi
from .kern import (Coregionalize, DeviceGradient, Stationary, White, Bias, composite_state_key, flatten_parts,
                   part_descriptor)
from .param import Param, Parameterized


class Gaussian(Parameterized):
    """GPy.likelihoods.Gaussian restricted to what exact inference touches (gaussian.py:35-79,102-110)."""

    def __init__(self, variance=1., name="Gaussian_noise"):
        super(Gaussian, self).__init__(name)
        self.variance = Param("variance", variance)
        self.link_parameter(self.variance)

    def gaussian_variance(self, Y_metadata=None):
        return self.variance

    def update_gradients(self, grad):
        self.variance.gradient = np.atleast_1d(grad)

    def exact_inference_gradients(self, dL_dKdiag, Y_metadata=None):
        return np.asarray(dL_dKdiag).sum()

    def predictive_values(self, mu, var, full_cov=False, Y_metadata=None):
        if full_cov:
            var = var + np.eye(var.shape[0]) * float(self.variance[0])
        else:
            var = var + float(self.variance[0])
        return mu, var


class HeteroscedasticGaussian(Gaussian):
    """GPy.likelihoods.HeteroscedasticGaussian (gaussian.py:347-377): one noise variance per output index."""

    def __init__(self, Y_metadata, variance=1., name="het_Gauss"):
        idx = np.asarray(Y_metadata["output_index"])
        super(HeteroscedasticGaussian, self).__init__(np.ones(idx.shape[0]) * variance, name)   # gaussian.py:356

    def gaussian_variance(self, Y_metadata=None):
        return self.variance.values[np.asarray(Y_metadata["output_index"]).flatten()]            # gaussian.py:361-362

    def exact_inference_gradients(self, dL_dKdiag, Y_metadata=None):
        return np.asarray(dL_dKdiag)[np.asarray(Y_metadata["output_index"]).flatten()]            # gaussian.py:358-359

    def update_gradients(self, grad):
        g = np.asarray(grad, dtype=np.float64).reshape(-1)
        if g.size != self.variance.values.size:
            # the reference assigns the array to the parameter's gradient and fails on the shape the same way
            # (gaussian.py:73): with P > 1 outputs VarDTC's dL_dR is N x P (var_dtc.py:245-257), not one value per variance
            raise ValueError("noise gradient of %d entries for %d noise variances" % (g.size, self.variance.values.size))
        self.variance.gradient = g

    def predictive_values(self, mu, var, full_cov=False, Y_metadata=None):
        _s = self.gaussian_variance(Y_metadata)                                                  # gaussian.py:364-373
        if full_cov:
            return mu, var + np.eye(var.shape[0]) * _s
        return mu, var + _s.reshape(-1, 1)


class MixedNoise(Parameterized):
    """GPy.likelihoods.MixedNoise (mixed_noise.py:14-53): a list of Gaussian likelihoods, data point n uses the one selected
    by Y_metadata['output_index'][n]. For exact inference it is a heteroscedastic variance vector going in
    (exact_gaussian_inference.py:52-56 -> gpx_exact_eval_het) and per-likelihood sums of diag(dL_dK) coming back."""

    def __init__(self, likelihoods_list, name="mixed_noise"):
        super(MixedNoise, self).__init__(name)
        self.likelihoods_list = list(likelihoods_list)
        if not all(isinstance(l, Gaussian) and not isinstance(l, HeteroscedasticGaussian) for l in self.likelihoods_list):
            raise AssertionError("MixedNoise works with a list of Gaussian likelihoods")          # mixed_noise.py:24,39
        self.link_parameters(*self.likelihoods_list)

    def gaussian_variance(self, Y_metadata):
        ind = np.asarray(Y_metadata["output_index"]).flatten()                                    # mixed_noise.py:23-29
        variance = np.zeros(ind.size)
        for j, lik in enumerate(self.likelihoods_list):
            variance[ind == j] = float(lik.variance[0])
        return variance

    def betaY(self, Y, Y_metadata):
        return Y / self.gaussian_variance(Y_metadata=Y_metadata)[:, None]                         # mixed_noise.py:31-33

    def exact_inference_gradients(self, dL_dKdiag, Y_metadata):
        ind = np.asarray(Y_metadata["output_index"]).flatten()                                    # mixed_noise.py:38-41
        d = np.asarray(dL_dKdiag).reshape(-1)
        return np.array([d[ind == i].sum() for i in range(len(self.likelihoods_list))])

    def update_gradients(self, gradients):
        g = np.asarray(gradients, dtype=np.float64).reshape(-1)                                   # mixed_noise.py:35-36: the
        for lik, gi in zip(self.likelihoods_list, g):                                             # container gradient is the
            lik.update_gradients(gi)                                                              # leaves' gradients in order

    def predictive_values(self, mu, var, full_cov=False, Y_metadata=None):
        ind = np.asarray(Y_metadata["output_index"]).flatten()                                    # mixed_noise.py:43-50
        _variance = np.array([float(self.likelihoods_list[j].variance[0]) for j in ind])
        if full_cov:
            return mu, var + np.eye(var.shape[0]) * _variance
        return mu, var + _variance.reshape(-1, 1)

    def predictive_variance(self, mu, sigma, Y_metadata):
        return self.gaussian_variance(Y_metadata) + sigma ** 2                                    # mixed_noise.py:52-54


class PosteriorExact(object):
    """Posterior whose big members live in HBM and are fetched lazily (posterior.py:21-77 constructor contract:
    woodbury_chol = L, woodbury_vector = alpha, K = noise-free kernel matrix)."""

    def __init__(self, engine, N, P, kern_key=None):
        self._engine, self._N, self._P = engine, N, P
        self._cache = {}
        self._serial = getattr(engine, "eval_serial", None)   # the evaluation this posterior describes
        self._kern_key = kern_key

    def _check_fresh(self):
        """The big members stay in HBM and the engine keeps only its LAST evaluation: a posterior handle kept across a
        later evaluation must not silently describe the new theta (the reference's posterior owns its arrays)."""
        if self._serial is not None and getattr(self._engine, "eval_serial", None) != self._serial:
            raise RuntimeError("this posterior belongs to an earlier evaluation; the device now holds a newer one "
                               "(read m.posterior again, or fetch what you need before the next parameter change)")

    def _get(self, which):
        if which not in self._cache:
            self._check_fresh()
            self._cache[which] = self._engine.get(which)
        return self._cache[which]

    @property
    def woodbury_chol(self):
        return self._get("L")

    @property
    def woodbury_vector(self):
        return self._get("alpha")

    @property
    def woodbury_inv(self):
        """posterior.py:183-203: (K + noise)^-1."""
        return self._get("Kinv")

    @property
    def K(self):
        return self._get("K")

    @property
    def mean(self):
        """posterior.py:98-110: K alpha."""
        return np.dot(self.K, self.woodbury_vector)

    def _raw_predict(self, kern, Xnew, pred_var=None, full_cov=False):
        """posterior.py:273-302 on the device (gpx_predict). `pred_var` (the training inputs) is what the engine holds."""
        key = kern._state_key() if hasattr(kern, "_state_key") else (
            kern._gpx_state_key() if hasattr(kern, "_gpx_state_key") else composite_state_key(kern))
        if self._kern_key is not None and key != self._kern_key:
            # a different kernel than the one evaluated (GP.predict(Xnew, kern=sub_kernel)): the reference's formula with
            # the kernel it is given (posterior.py:276-295), on the factor fetched from the device
            return HostPosterior(self.woodbury_chol, self.woodbury_vector, None)._raw_predict(kern, Xnew, pred_var, full_cov)
        self._check_fresh()
        Xn = kern._slice_X(Xnew) if hasattr(kern, "_slice_X") else np.asarray(Xnew, dtype=np.float64)
        if isinstance(Xn, tuple):
            Xn = Xn[0]
        return self._engine.predict(np.ascontiguousarray(Xn, dtype=np.float64), full_cov=full_cov)


class _DataKey(object):
    """Decides whether (X, Y) must be uploaded again: an exact comparison with a private host copy of what the device
    holds. (paramz keys its caches on object identity; the sliced X is a fresh array on every call without paramz's cache
    and callers may permute rows in place, so neither identity nor a moment/sample fingerprint is safe — a row swap keeps
    every moment.) Cost: one memcmp-speed pass, ~0.1 ms per MB, and N (D + P) doubles of host memory. Deliberately not a
    BLAS call: a multi-threaded BLAS spins up its worker pool for such a tiny product and, under a CPU quota, the
    spinning workers get the process throttled right when the evaluation's kernels have to be enqueued."""

    def __init__(self):
        self._X = self._Y = None

    def invalidate(self):
        self._X = self._Y = None

    def matches(self, X, Y):
        return (self._X is not None and self._X.shape == X.shape and self._Y.shape == Y.shape
                and np.array_equal(self._X, X) and np.array_equal(self._Y, Y))

    def remember(self, X, Y):
        self._X, self._Y = np.array(X, dtype=np.float64, copy=True), np.array(Y, dtype=np.float64, copy=True)


class ExactGaussianInference(object):
    """Drop-in for GPy's ExactGaussianInference: `inference(kern, X, likelihood, Y, ...)` returns
    (posterior, log_marginal, {'dL_dK', 'dL_dthetaL', 'dL_dm'}). For the stationary kernels of gpy_b200.kern the whole
    evaluation (K build, factorisation, solves, K^-1, gradient reductions) is ONE C-ABI call; `dL_dK` comes back as a
    DeviceGradient handle that `kern.update_gradients_full` recognises."""

    def __init__(self, device=0, engine=None):
        self.device = device
        self._engine = engine
        self._data_key = _DataKey()

    def on_optimization_start(self):
        pass

    def on_optimization_end(self):
        pass

    def to_dict(self):
        return {"class": "gpy_b200.inference.ExactGaussianInference", "name": "ExactGaussianInference"}

    def __getstate__(self):
        """pickle without the device handle (precedent: GPy/kern/src/rbf.py:313-318); re-created lazily after loading"""
        d = dict(self.__dict__)
        d["_engine"], d["_data_key"] = None, _DataKey()
        return d

    @property
    def engine(self):
        if self._engine is None:
            self._engine = _ffi.Engine(self.device)
        return self._engine

    def invalidate_data(self):
        """the model was handed new data (GP.set_XY): upload again at the next inference whatever the content."""
        self._data_key.invalidate()

    def _bind(self, X, Y, force=False):
        if force or not self._data_key.matches(X, Y):
            self.engine.set_data(X, Y)
            self._data_key.remember(X, Y)

    def inference(self, kern, X, likelihood, Y, mean_function=None, Y_metadata=None, K=None, variance=None,
                  Z_tilde=None):
        if variance is None:
            variance = likelihood.gaussian_variance(Y_metadata)
        nvec = np.asarray(variance, dtype=np.float64).reshape(-1)
        het = nvec.size > 1                          # HeteroscedasticGaussian: a vector reaches diag.add (:55-56)
        noise = nvec if het else float(nvec[0])
        if mean_function is None and K is None and not isinstance(kern, Stationary):
            parts = flatten_parts(kern)
            if parts is not None and (het or any(isinstance(k, Coregionalize) for k, _ in parts)):
                return self._coreg_inference(kern, parts, X, Y, noise, Z_tilde, likelihood, Y_metadata)
            if parts is not None and not het:
                return self._composite_inference(kern, parts, X, Y, noise, Z_tilde)
        if mean_function is not None or K is not None or not isinstance(kern, Stationary):
            return self._generic_inference(kern, X, Y, noise, mean_function, K, Z_tilde, likelihood, Y_metadata)
        Xs = kern._slice_X(X)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        self._bind(Xs, Y)
        kind, ard, var, ls = kern._theta()
        if het:
            if nvec.size != Y.shape[0]:
                raise ValueError("heteroscedastic noise needs one variance per data point")
            lml, grad, dnoise, _ = self.engine.exact_eval_het(kind, ard, var, ls, nvec, jitter=1e-8, max_tries=5)
            if Z_tilde is not None:
                lml += Z_tilde
            N, P = Y.shape
            post = PosteriorExact(self.engine, N, P, kern._state_key())
            dL_dK = DeviceGradient(self.engine, kern._state_key(), grad[0], grad[1:-1], N)
            dL_dthetaL = likelihood.exact_inference_gradients(dnoise, Y_metadata)              # :72 with gaussian.py:358
            return post, lml, {"dL_dK": dL_dK, "dL_dthetaL": dL_dthetaL, "dL_dm": _LazyAlpha(post)}
        # exact_gaussian_inference.py:56: +1e-8 on the diagonal, always; jitchol ladder of 5 (util/linalg.py:56)
        lml, grad, _ = self.engine.exact_eval(kind, ard, var, ls, noise, jitter=1e-8, max_tries=5)
        if Z_tilde is not None:
            lml += Z_tilde
        N, P = Y.shape
        post = PosteriorExact(self.engine, N, P, kern._state_key())
        dL_dK = DeviceGradient(self.engine, kern._state_key(), grad[0], grad[1:-1], N)
        grad_dict = {"dL_dK": dL_dK, "dL_dthetaL": grad[-1], "dL_dm": _LazyAlpha(post)}
        return post, lml, grad_dict


    def _composite_inference(self, kern, parts, X, Y, noise, Z_tilde):
        """Sum / product kernels (add.py, prod.py, static.py) on the fused device path: ONE gpx_exact_eval_multi per
        evaluation; the data stay resident, nothing of size N^2 crosses PCIe."""
        Xc = np.ascontiguousarray(kern._slice_X(X), dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        self._bind(Xc, Y)
        desc = [part_descriptor(leaf, term) for (leaf, term) in parts]
        lml, grad, _ = self.engine.exact_eval_multi(desc, noise, jitter=1e-8, max_tries=5)
        if Z_tilde is not None:
            lml += Z_tilde
        part_grads, i = [], 0
        for (leaf, _) in parts:
            n = 1 + (leaf.lengthscale.size if isinstance(leaf, Stationary) else 0)
            part_grads.append(grad[i:i + n])
            i += n
        N, P = Y.shape
        key = composite_state_key(kern)
        post = PosteriorExact(self.engine, N, P, key)
        dL_dK = DeviceGradient(self.engine, key, None, None, N, part_grads=part_grads)
        return post, lml, {"dL_dK": dL_dK, "dL_dthetaL": grad[-1], "dL_dm": _LazyAlpha(post)}

    def _coreg_inference(self, kern, parts, X, Y, noise, Z_tilde, likelihood, Y_metadata):
        """Composite kernels with coregionalization parts (coregionalize.py, util/multioutput.py ICM / LCM) and / or one
        noise variance per data point (MixedNoise, HeteroscedasticGaussian) on the fused path: ONE gpx_exact_eval_coreg per
        evaluation. dL_dthetaL = likelihood.exact_inference_gradients(diag(dL_dK)) (exact_gaussian_inference.py:72)."""
        Xc = np.ascontiguousarray(kern._slice_X(X), dtype=np.float64)
        Y = np.ascontiguousarray(Y, dtype=np.float64)
        if np.ndim(noise) > 0 and np.size(noise) != Y.shape[0]:
            raise ValueError("heteroscedastic noise needs one variance per data point")
        self._bind(Xc, Y)
        desc = [part_descriptor(leaf, term) for (leaf, term) in parts]
        lml, grad, dnoise, _ = self.engine.exact_eval_coreg(desc, noise, jitter=1e-8, max_tries=5)
        if Z_tilde is not None:
            lml += Z_tilde
        part_grads, i = [], 0
        for (leaf, _) in parts:
            n = (leaf.output_dim ** 2 if isinstance(leaf, Coregionalize) else
                 1 + (leaf.lengthscale.size if isinstance(leaf, Stationary) else 0))
            part_grads.append(grad[i:i + n])
            i += n
        N, P = Y.shape
        key = composite_state_key(kern)
        post = PosteriorExact(self.engine, N, P, key)
        dL_dK = DeviceGradient(self.engine, key, None, None, N, part_grads=part_grads)
        dL_dthetaL = grad[-1] if dnoise is None else likelihood.exact_inference_gradients(dnoise, Y_metadata)
        return post, lml, {"dL_dK": dL_dK, "dL_dthetaL": dL_dthetaL, "dL_dm": _LazyAlpha(post)}

    def _generic_inference(self, kern, X, Y, noise, mean_function, K, Z_tilde, likelihood=None, Y_metadata=None):
        """exact_gaussian_inference.py:37-74 for the cases the fused call does not cover (mean function, precomputed K,
        foreign kernel): the N^3 part (jitchol + dpotri, util/linalg.py:193-214) still runs on the device through
        gpx_pdinv; the O(N^2 P) remainder is NumPy on the host because K arrives as / has to be returned as ndarrays."""
        m = 0 if mean_function is None else mean_function.f(X)
        YYT_factor = np.asarray(Y, dtype=np.float64) - m
        if K is None:
            K = kern.K(X)
        Ky = np.array(K, dtype=np.float64, copy=True)
        Ky[np.diag_indices_from(Ky)] += np.asarray(noise) + 1e-8
        Wi, LW, _, W_logdet, _ = _ffi.pdinv(Ky, maxtries=5, want=("Ai", "L"), engine=self.engine)
        alpha = np.dot(Wi, YYT_factor)
        log_marginal = 0.5 * (-YYT_factor.size * np.log(2 * np.pi) - YYT_factor.shape[1] * W_logdet
                              - np.sum(alpha * YYT_factor))
        if Z_tilde is not None:
            log_marginal += Z_tilde
        dL_dK = 0.5 * (np.dot(alpha, alpha.T) - YYT_factor.shape[1] * Wi)
        self._data_key.invalidate()   # the context workspace was re-used
        if np.ndim(noise) > 0 and likelihood is not None:
            dL_dthetaL = likelihood.exact_inference_gradients(np.diag(dL_dK), Y_metadata)
        else:
            dL_dthetaL = float(np.trace(dL_dK))
        return (HostPosterior(LW, alpha, K), float(log_marginal),
                {"dL_dK": dL_dK, "dL_dthetaL": dL_dthetaL, "dL_dm": alpha})


class HostPosterior(object):
    """posterior.py:21-77,273-302 with host arrays (generic inference path)."""

    def __init__(self, woodbury_chol, woodbury_vector, K):
        self.woodbury_chol, self.woodbury_vector, self.K = woodbury_chol, woodbury_vector, K

    def _raw_predict(self, kern, Xnew, pred_var, full_cov=False):
        from scipy.linalg import solve_triangular
        Kx = kern.K(pred_var, Xnew)
        mu = np.dot(Kx.T, self.woodbury_vector)
        tmp = solve_triangular(self.woodbury_chol, Kx, lower=True)
        if full_cov:
            return mu, kern.K(Xnew) - np.dot(tmp.T, tmp)
        return mu, (kern.Kdiag(Xnew) - np.square(tmp).sum(0))[:, None]


class _LazyAlpha(object):
    """grad_dict['dL_dm'] is alpha (exact_gaussian_inference.py:74); fetched only if used."""

    def __init__(self, post):
        self._post = post

    def __array__(self, dtype=None, copy=None):
        a = self._post.woodbury_vector
        return a if dtype is None else a.astype(dtype)
