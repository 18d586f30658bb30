"""Host model mirroring GPy's GPRegression / GP runtime for the exact-GP hot path.

Mirrors:
    GPy.models.GPRegression                GPy/models/gp_regression.py:9-36
    GPy.core.GP.__init__/parameters_changed/log_likelihood/predict/optimize
                                           GPy/core/gp.py:38-108,269-288,290-365,663-684
    GPy.core.Model.objective_function[_gradients]   GPy/core/model.py:97-128
GPy obtains its optimizer loop, parameter transforms and gradient checking from the third-party `paramz`; here the same
three things are provided stand-alone (Logexp transform on all three hyper-parameters, SciPy L-BFGS-B, central
finite-difference checkgrad) so that `m.optimize()` / `m.checkgrad()` read like the reference's own tests. When GPy and
paramz are importable, use the real GPy model with the plugin classes of gpy_b200.gpy_plugin instead.
"""
import numpy as np

from .inference import ExactGaussianInference, Gaussian, HeteroscedasticGaussian
from .kern import RBF
from .param import Parameterized


class Standardize(object):
    """GPy.util.normalizer.Standardize (normalizer.py:85-113): per-output mean / standard deviation of Y; O(N P) host work,
    the device sees the normalised targets."""

    def __init__(self):
        self.mean = None

    def scale_by(self, Y):
        Y = np.ma.masked_invalid(Y, copy=False)
        self.mean = Y.mean(0).view(np.ndarray)
        self.std = Y.std(0).view(np.ndarray)
        self.std[np.where(self.std == 0)] = 1.                      # normalizer.py:93-96

    def scaled(self):
        return self.mean is not None

    def normalize(self, Y):
        return (Y - self.mean) / self.std

    def inverse_mean(self, X):
        return (X * self.std) + self.mean

    def inverse_variance(self, var):
        return var * (self.std ** 2)

    def inverse_covariance(self, covariance):
        return covariance[..., np.newaxis] * (self.std ** 2)


class GP(Parameterized):
    def __init__(self, X, Y, kernel, likelihood, mean_function=None, inference_method=None, name="gp", device=0,
                 engine=None, Y_metadata=None, normalizer=False):
        super(GP, self).__init__(name)
        self._initialised = False   # parameter writes during construction do not evaluate (paramz: after __init__)
        self.mean_function = mean_function
        self.Y_metadata = Y_metadata
        X = np.asarray(X, dtype=np.float64)
        Y = np.asarray(Y, dtype=np.float64)
        assert X.ndim == 2
        assert Y.ndim == 2 and Y.shape[0] == X.shape[0]  # gp.py:42-66
        self.X, self.Y = X, Y
        # gp.py:49-66: normalizer True -> Standardize, False / None -> none, else a _Norm-like object
        self.normalizer = Standardize() if normalizer is True else (None if normalizer in (False, None) else normalizer)
        self._normalize_Y()
        self.num_data, self.input_dim = X.shape
        self.output_dim = Y.shape[1]
        self.kern, self.likelihood = kernel, likelihood
        assert self.input_dim >= self.kern.input_dim
        if inference_method is None:  # gp.py:97-99: Gaussian likelihood -> exact inference
            inference_method = ExactGaussianInference(device=device, engine=engine)
        self.inference_method = inference_method
        self.link_parameter(self.kern)        # gp.py:106
        self.link_parameter(self.likelihood)  # gp.py:107
        self.posterior = None
        self._log_marginal_likelihood = None
        self.grad_dict = None
        self.update_model_flag = True
        self._initialised = True
        self.parameters_changed()  # paramz's metaclass triggers this after __init__

    def _normalize_Y(self):
        if self.normalizer is not None:
            self.normalizer.scale_by(self.Y)
            self.Y_normalized = np.ascontiguousarray(self.normalizer.normalize(self.Y), dtype=np.float64)
        else:
            self.Y_normalized = self.Y

    def __getstate__(self):
        """pickling returns a device-less model (precedent: GPy/kern/src/rbf.py:313-318 drops its GPU state): the engine
        handle is dropped, the inference object re-creates it lazily and uploads the data at the next evaluation"""
        d = dict(self.__dict__)
        d["posterior"] = None
        return d

    # ---- one evaluation: gp.py:269-282 -------------------------------------------------------------------------
    def parameters_changed(self):
        self.posterior, self._log_marginal_likelihood, self.grad_dict = self.inference_method.inference(
            self.kern, self.X, self.likelihood, self.Y_normalized, self.mean_function, self.Y_metadata)
        self.likelihood.update_gradients(self.grad_dict["dL_dthetaL"])
        self.kern.update_gradients_full(self.grad_dict["dL_dK"], self.X)

    def log_likelihood(self):
        """gp.py:284-288."""
        return self._log_marginal_likelihood

    # ---- data / parameter setters -------------------------------------------------------------------------------
    def set_XY(self, X=None, Y=None):
        """gp.py:188-230 (set_XY): swap the data, re-evaluate."""
        if X is not None:
            self.X = np.asarray(X, dtype=np.float64)
        if Y is not None:
            self.Y = np.asarray(Y, dtype=np.float64)
            self._normalize_Y()                                     # gp.py:224-226
        self.num_data = self.X.shape[0]
        if hasattr(self.inference_method, "invalidate_data"):
            self.inference_method.invalidate_data()
        if self.update_model_flag:
            self.parameters_changed()

    def update_model(self, flag):
        """paramz Parameterizable.update_model: False defers re-evaluation while several things are written."""
        was = self.update_model_flag
        self.update_model_flag = bool(flag)
        if flag and not was:
            self.parameters_changed()

    def set_theta(self, variance, lengthscale, noise_variance):
        """convenience: write all three hyper-parameters, then ONE parameters_changed()."""
        self.kern.variance.values[...] = variance
        self.kern.lengthscale.values[...] = lengthscale
        self.likelihood.variance.values[...] = noise_variance
        self.parameters_changed()

    # ---- paramz.Model surface: transformed optimizer space ---------------------------------------------------------
    def _free(self):
        return [p for p in self.flattened_parameters() if not p.is_fixed]

    @property
    def optimizer_array(self):
        return np.concatenate([(p.values if p.transform is None else p.transform.finv(p.values)).reshape(-1)
                               for p in self._free()])

    @optimizer_array.setter
    def optimizer_array(self, x):
        i = 0
        for p in self._free():
            v = x[i:i + p.size]
            p.values[...] = (v if p.transform is None else p.transform.f(v)).reshape(p.values.shape)
            i += p.size
        self.parameters_changed()

    def objective_function(self):
        """model.py:97-109 (no priors on the hot path)."""
        return -float(self.log_likelihood())

    def objective_function_gradients(self):
        """model.py:111-128, in the untransformed theta space."""
        return -self.gradient

    def _grads_transformed(self):
        g = []
        for p in self._free():
            gf = 1.0 if p.transform is None else p.transform.gradfactor(p.values).reshape(-1)   # W of Coregionalize: none
            g.append(np.asarray(p.gradient, dtype=np.float64).reshape(-1) * gf)
        return -np.concatenate(g)

    def _objective_and_grad(self, x):
        try:
            self.optimizer_array = x
            f, g = self.objective_function(), self._grads_transformed()
            self._fail_count = 0
        except (np.linalg.LinAlgError, ZeroDivisionError, ValueError):   # _ffi.check maps argument-domain errors to ValueError
            # paramz tolerates a bounded number of failed evaluations during optimisation
            self._fail_count = getattr(self, "_fail_count", 0) + 1
            if self._fail_count > 10:
                raise
            # paramz Model._objective_grads: objective = inf, gradient = the last good one (clipped)
            g = getattr(self, "_last_good_grad", None)
            return np.inf, (np.zeros_like(x) if g is None or g.shape != x.shape else np.clip(g, -1e10, 1e10))
        self._last_good_grad = g
        return f, g

    def optimize(self, optimizer="lbfgsb", max_iters=1000, messages=False, gtol=1e-5, ftol=2.220446049250313e-09):
        """gp.py:663-684 -> paramz Model.optimize: default 'lbfgsb' = scipy.optimize.fmin_l_bfgs_b on the transformed
        parameters. Returns the scipy result dict (paramz returns an Optimizer object)."""
        from scipy.optimize import fmin_l_bfgs_b
        assert optimizer in ("lbfgsb", "lbfgs", "bfgs", None)
        self.inference_method.on_optimization_start()
        self.n_evals = 0

        def fg(x):
            self.n_evals += 1
            f, g = self._objective_and_grad(x)
            if messages:
                print("eval %4d  objective %.10f" % (self.n_evals, f))
            return f, g

        x0 = self.optimizer_array
        x, f, d = fmin_l_bfgs_b(fg, x0, maxfun=max_iters, maxiter=max_iters, pgtol=gtol, factr=ftol / np.finfo(float).eps)
        self.optimizer_array = x
        self.inference_method.on_optimization_end()
        d["x"], d["f"], d["n_evals"] = x, f, self.n_evals
        return d

    def checkgrad(self, step=1e-6, tolerance=1e-3, verbose=False):
        """paramz Model.checkgrad: central finite differences vs the analytic gradient in the transformed space."""
        x = self.optimizer_array.copy()
        self.optimizer_array = x
        g = self._grads_transformed()
        num = np.zeros_like(x)
        for i in range(x.size):
            xp, xm = x.copy(), x.copy()
            xp[i] += step
            xm[i] -= step
            self.optimizer_array = xp
            fp = self.objective_function()
            self.optimizer_array = xm
            fm = self.objective_function()
            num[i] = (fp - fm) / (2 * step)
        self.optimizer_array = x
        ratio = np.where(num != 0, g / np.where(num == 0, 1, num), 1.0)
        if verbose:
            print("analytic", g, "numeric", num)
        return bool(np.all(np.abs(1.0 - ratio) < tolerance) or np.allclose(g, num, atol=tolerance * 1e-2))

    # ---- prediction: gp.py:290-365 --------------------------------------------------------------------------------
    def _raw_predict(self, Xnew, full_cov=False, kern=None):
        mu, var = self.posterior._raw_predict(kern=self.kern if kern is None else kern, Xnew=Xnew, pred_var=self.X,
                                              full_cov=full_cov)
        if self.mean_function is not None:
            mu = mu + self.mean_function.f(Xnew)   # gp.py:304-305
        return mu, var

    def predict(self, Xnew, full_cov=False, Y_metadata=None, kern=None, likelihood=None, include_likelihood=True):
        mean, var = self._raw_predict(Xnew, full_cov=full_cov, kern=kern)
        if include_likelihood:
            if likelihood is None:
                likelihood = self.likelihood
            mean, var = likelihood.predictive_values(mean, var, full_cov, Y_metadata=Y_metadata)
        if self.normalizer is not None:                             # gp.py:355-363
            mean = self.normalizer.inverse_mean(mean)
            if full_cov and mean.shape[1] > 1:
                var = self.normalizer.inverse_covariance(var)
            else:
                var = self.normalizer.inverse_variance(var)
        return mean, var

    def predict_noiseless(self, Xnew, full_cov=False, Y_metadata=None, kern=None):
        return self.predict(Xnew, full_cov, Y_metadata, kern, None, False)


class GPHeteroscedasticRegression(GP):
    """GPy.models.GPHeteroscedasticRegression (gp_heteroscedastic_regression.py:10-37): one Gaussian noise variance per
    data point (HeteroscedasticGaussian), exact inference; "does not make inference on the noise outside the training
    set", so predict() needs Y_metadata for the new points (or include_likelihood=False)."""

    def __init__(self, X, Y, kernel=None, Y_metadata=None, device=0, engine=None):
        Ny = np.asarray(Y).shape[0]
        if Y_metadata is None:
            Y_metadata = {"output_index": np.arange(Ny)[:, None]}          # :26-27
        else:
            assert Y_metadata["output_index"].shape[0] == Ny
        if kernel is None:
            kernel = RBF(np.asarray(X).shape[1])                             # :31-32
        likelihood = HeteroscedasticGaussian(Y_metadata)                      # :35
        super(GPHeteroscedasticRegression, self).__init__(X, Y, kernel, likelihood, name="gp_het", device=device,
                                                          engine=engine, Y_metadata=Y_metadata)


class GPRegression(GP):
    """GPy.models.GPRegression (gp_regression.py:9-36): Gaussian likelihood, default RBF kernel, exact inference."""

    def __init__(self, X, Y, kernel=None, Y_metadata=None, normalizer=None, noise_var=1., mean_function=None,
                 device=0, engine=None):
        if kernel is None:
            kernel = RBF(np.asarray(X).shape[1])  # gp_regression.py:31-32
        likelihood = Gaussian(variance=noise_var)  # gp_regression.py:34
        super(GPRegression, self).__init__(X, Y, kernel, likelihood, mean_function=mean_function, name="GP regression",
                                           device=device, engine=engine, Y_metadata=Y_metadata,
                                           normalizer=False if normalizer is None else normalizer)


class GPCoregionalizedRegression(GP):
    """GPy.models.GPCoregionalizedRegression (gp_coregionalized_regression.py:31-46): multi-output regression. X_list /
    Y_list hold one input / output array per output; the data are stacked with an output-index column (build_XY), the
    kernel defaults to ICM(RBF) and the likelihood is a MixedNoise of one Gaussian per output. predict() takes the output
    index as the last column of Xnew and, with include_likelihood, Y_metadata={'output_index': ...} for the noise."""

    def __init__(self, X_list, Y_list, kernel=None, likelihoods_list=None, name="GPCR", W_rank=1, kernel_name="coreg",
                 device=0, engine=None):
        from . import multioutput
        X, Y, self.output_index = multioutput.build_XY(X_list, Y_list)             # :34
        Ny = len(Y_list)
        if kernel is None:                                                           # :38-41
            kernel = RBF(X.shape[1] - 1)
            kernel = multioutput.ICM(input_dim=X.shape[1] - 1, num_outputs=Ny, kernel=kernel, W_rank=W_rank,
                                     name=kernel_name)
        likelihood = multioutput.build_likelihood(Y_list, self.output_index, likelihoods_list)   # :43
        super(GPCoregionalizedRegression, self).__init__(X, Y, kernel, likelihood, name=name, device=device, engine=engine,
                                                         Y_metadata={"output_index": self.output_index})
