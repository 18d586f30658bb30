"""The plugin classes of gpy_b200/gpy_plugin.py for multi-output models, wired onto the UNMODIFIED reference classes
(GPCoregionalizedRegression, GP, Add, Prod, Coregionalize, MixedNoise, util.multioutput, loaded from the reference tree).
The C ABI is replaced by a test double answering from the NumPy restatement (tests/coreg_oracle.py): what is tested is
the wiring — the stock model with plugin kernels issues ONE gpx_exact_eval_coreg per evaluation, the plugin Add / Prod /
Coregionalize hand every leaf its device-reduced gradient, the likelihood gets diag(dL_dK) through its own
exact_inference_gradients, and LML and gradient equal the stock model's."""
import importlib.util
import os
import types

import numpy as np
import pytest

import coreg_oracle as co

pytestmark = pytest.mark.skipif(not os.path.isdir(os.environ.get("GPX_REFERENCE", "/root/reference") + "/GPy"),
                                reason="reference tree not present")


class FakeEngine(object):
    def __init__(self, device=0):
        self.calls, self.eval_serial = [], 0

    def set_data(self, X, Y):
        self.X, self.Y = np.array(X), np.array(Y)
        self.calls.append("set_data")

    def exact_eval_coreg(self, parts, noise, jitter=1e-8, max_tries=5):
        self.calls.append("exact_eval_coreg")
        self.eval_serial += 1
        self.parts = []
        for (k, a, t, d, v, l) in parts:
            if k == "coregionalize":
                self.parts.append(dict(kind=k, term=t, dims=d, B=np.asarray(l)))
            else:
                self.parts.append(dict(kind=k, ARD=a, term=t, dims=d, variance=v, lengthscale=l))
        lml, _, self.res = co.eval_lml_grad(self.X, self.Y, self.parts, noise)
        return lml, self.res["device_grad"], (self.res["dnoise"] if np.ndim(noise) else None), 0.0

    def get(self, which):
        return {"L": self.res["L"], "alpha": self.res["alpha"], "K": self.res["K"]}[which]


def _fake_ffi():
    from oracle import gpy_oracle as o

    def kern_K(kind, ARD, var, ls, X, X2=None):
        return o.StationaryOracle(kind, X.shape[1], var, ls, ARD).K(X, X2)

    def kern_Kdiag(kind, var, N):
        return np.full(N, var)

    def kern_grad_full(kind, ARD, var, ls, X, dL_dK, X2=None):
        dv, dl = o.StationaryOracle(kind, X.shape[1], var, ls, ARD).update_gradients_full(dL_dK, X, X2)
        return dv, np.atleast_1d(dl)

    # the model's construction evaluates once with GPy's stock inference (dense dL_dK) before the plugin inference is set
    return types.SimpleNamespace(kern_K=kern_K, kern_Kdiag=kern_Kdiag, kern_grad_full=kern_grad_full, Engine=FakeEngine)


def _reference():
    spec = importlib.util.spec_from_file_location(
        "make_coreg_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_coreg_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.load_reference()


def plugin_pair(ffi):
    """-> (stock model, plugin model, B): the reference's GPCoregionalizedRegression once with its own ICM kernel and
    once with the plugin kernel B.Prod([B.RBF, B.Coregionalize]) (GPy's multioutput.ICM builds GPy.kern.Coregionalize,
    so the plugin kernel is built explicitly) and the plugin inference"""
    import sys
    from gpy_b200 import gpy_plugin
    G, C, M, mo, GPCR, R = _reference()
    Cref = sys.modules["GPy.kern"].Coregionalize
    B = gpy_plugin.make(G.RBF, G.Exponential, G.Matern32, G.Matern52, G.ExactGaussianInference, ffi=ffi, Add=C.Add,
                        Prod=C.Prod, Coregionalize=Cref)
    rng = np.random.RandomState(5)
    D, O = 2, 3
    Xl = [rng.uniform(-2, 2, (14 + j, D)) for j in range(O)]
    Yl = [np.sin(x).sum(1, keepdims=True) * (1 + 0.3 * j) + 0.1 * rng.randn(x.shape[0], 1) for j, x in enumerate(Xl)]
    W, kappa, ls = 0.5 * rng.randn(O, 2), np.array([0.3, 0.5, 0.7]), np.array([0.9, 1.4])
    stock = GPCR(Xl, Yl, kernel=mo.ICM(D, O, G.RBF(D, variance=1.2, lengthscale=ls, ARD=True), W_rank=2, W=W.copy(),
                                       kappa=kappa.copy()))
    k = B.Prod([B.RBF(D, variance=1.2, lengthscale=ls, ARD=True),
                B.Coregionalize(1, O, rank=2, W=W.copy(), kappa=kappa.copy(), active_dims=[D], name="B")], name="ICM")
    plug = GPCR(Xl, Yl, kernel=k)
    for m in (stock, plug):
        for j, v in enumerate([0.05, 0.11, 0.08]):
            m.likelihood.likelihoods_list[j].variance[:] = v
    plug.inference_method = B.ExactGaussianInference()
    plug.parameters_changed()
    stock.parameters_changed()
    return stock, plug, B


def test_stock_coregionalized_model_with_plugin_kernels_runs_fused():
    stock, plug, B = plugin_pair(_fake_ffi())
    assert type(plug) is type(stock)
    eng = plug.inference_method.engine
    assert eng.calls == ["set_data", "exact_eval_coreg"]
    assert abs(plug.log_likelihood() - stock.log_likelihood()) <= 1e-10 * abs(stock.log_likelihood())
    assert np.asarray(plug.gradient).size == np.asarray(stock.gradient).size == 1 + 2 + 6 + 3 + 3
    np.testing.assert_allclose(np.asarray(plug.gradient), np.asarray(stock.gradient), rtol=1e-9, atol=1e-12)


def test_plugin_coregionalize_alone_and_foreign_dL_dK():
    """a plugin Coregionalize as the whole kernel takes S from the handle; a dense dL_dK goes to the stock reduction"""
    import sys
    from gpy_b200 import gpy_plugin
    from gpy_b200.kern import DeviceGradient
    G, C, M, mo, GPCR, R = _reference()
    Cref = sys.modules["GPy.kern"].Coregionalize
    B = gpy_plugin.make(G.RBF, G.Exponential, G.Matern32, G.Matern52, G.ExactGaussianInference, ffi=_fake_ffi(),
                        Coregionalize=Cref)
    rng = np.random.RandomState(2)
    W = rng.randn(3, 1)
    ours, ref = B.Coregionalize(1, 3, W=W.copy()), Cref(1, 3, W=W.copy())
    idx = rng.randint(0, 3, (20, 1)).astype(float)
    dL = rng.randn(20, 20)
    dL = dL + dL.T
    ours.update_gradients_full(dL, idx)
    ref.update_gradients_full(dL, idx)
    np.testing.assert_array_equal(np.asarray(ours.W.gradient), np.asarray(ref.W.gradient))
    S = co.CoregOracle(W, np.full(3, 0.5)).S(dL, idx)
    h = DeviceGradient(None, gpy_plugin._composite_key(ours), None, None, 20, part_grads=[S.reshape(-1)])
    ours.update_gradients_full(h, idx)
    np.testing.assert_allclose(np.asarray(ours.W.gradient), np.asarray(ref.W.gradient), rtol=1e-12)
    np.testing.assert_allclose(np.asarray(ours.kappa.gradient), np.asarray(ref.kappa.gradient), rtol=1e-12)
