"""Multi-output (coregionalized) regression on the device: gpx_exact_eval_coreg against the NumPy restatement in
tests/coreg_oracle.py (itself checked against the reference GPy in tests/test_coreg_cpu.py). N = 150 takes the DMMA sweep
with the plain K^-1 store, N = 700 / 1300 the tcgen05 sweep that stores K^-1 itself (ragged last tile)."""
import glob
import json
import os

import numpy as np
import pytest

import coreg_oracle as co
import gpy_b200
from gpy_b200 import _ffi
from oracle import gpy_oracle as o

pytestmark = pytest.mark.gpu

LML_ATOL = 1e-8
GRAD_RTOL = 1e-6
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "coreg")


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - b)) / max(np.max(np.abs(b)), 1e-300))


def _data(N, D, O, P, seed):
    """inputs with the output index as last column, rows shuffled across outputs"""
    rng = np.random.default_rng(seed)
    Xi = rng.uniform(-3, 3, (N, D))
    idx = rng.integers(0, O, N).astype(np.float64)
    Y = np.stack([np.sin(Xi).sum(1) / np.sqrt(D) * (1 + 0.3 * idx) + 0.1 * rng.standard_normal(N) for _ in range(P)], 1)
    return np.hstack([Xi, idx[:, None]]), Y, idx.astype(int)


def _parts(case, D, O, seed):
    rng = np.random.default_rng(seed + 100)
    if case == "icm":
        return [dict(kind="rbf", term=0, dims=list(range(D)), variance=1.3, lengthscale=list(rng.uniform(0.8, 2.0, D)),
                     ARD=True),
                dict(kind="coregionalize", term=0, dims=[D], W=(0.6 * rng.standard_normal((O, 2))).tolist(),
                     kappa=list(rng.uniform(0.2, 0.8, O)))]
    return [dict(kind="rbf", term=0, dims=list(range(D)), variance=0.9, lengthscale=[1.3], ARD=False),
            dict(kind="coregionalize", term=0, dims=[D], W=(0.7 * rng.standard_normal((O, 1))).tolist(),
                 kappa=list(rng.uniform(0.2, 0.8, O))),
            dict(kind="matern32", term=1, dims=list(range(D)), variance=0.6, lengthscale=list(rng.uniform(0.8, 2.0, D)),
                 ARD=True),
            dict(kind="coregionalize", term=1, dims=[D], W=(0.7 * rng.standard_normal((O, 1))).tolist(),
                 kappa=list(rng.uniform(0.2, 0.8, O))),
            dict(kind="bias", term=2, variance=0.35)]


def _engine(N):
    eng = _ffi.Engine(0)
    eng.set_option("ozaki", 1 if N >= 700 else 0)
    return eng


@pytest.mark.parametrize("case", ["icm", "lcm"])
@pytest.mark.parametrize("P", [1, 2])
@pytest.mark.parametrize("N", [150, 700, 1300])
def test_coreg_parity_mixed_noise(N, P, case):
    D, O = 4, 3
    X, Y, idx = _data(N, D, O, P, seed=N + P)
    parts = _parts(case, D, O, seed=N)
    noise_out = np.array([0.05, 0.09, 0.03])
    eng = _engine(N)
    eng.set_data(X, Y)
    lml, g, dnoise, _ = eng.exact_eval_coreg(co.device_parts(parts), noise_out[idx])
    lml0, g0, res = co.eval_lml_grad(X, Y, parts, noise_out[idx])
    assert abs(lml - lml0) <= LML_ATOL
    np.testing.assert_allclose(g, res["device_grad"], rtol=GRAD_RTOL, atol=1e-9)
    np.testing.assert_allclose(co.per_output(dnoise, idx, O), co.per_output(res["dnoise"], idx, O), rtol=GRAD_RTOL, atol=1e-9)
    np.testing.assert_allclose(dnoise, res["dnoise"], rtol=1e-6, atol=1e-9)
    assert rel(eng.get("alpha"), res["alpha"]) < 1e-9
    assert rel(eng.get("K"), res["K"]) < 1e-12
    assert rel(eng.get("L"), res["L"]) < 1e-10


@pytest.mark.parametrize("N", [150, 1300])
def test_coreg_homoscedastic(N):
    D, O = 4, 3
    X, Y, idx = _data(N, D, O, 1, seed=7 + N)
    parts = _parts("icm", D, O, seed=3)
    eng = _engine(N)
    eng.set_data(X, Y)
    lml, g, dnoise, _ = eng.exact_eval_coreg(co.device_parts(parts), 0.06)
    lml0, g0, res = co.eval_lml_grad(X, Y, parts, 0.06)
    assert dnoise is None
    assert abs(lml - lml0) <= LML_ATOL
    np.testing.assert_allclose(g, res["device_grad"], rtol=GRAD_RTOL, atol=1e-9)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "*.npz"))), ids=os.path.basename)
def test_coreg_golden_through_the_device(path):
    """the reference's own numbers (tests/golden/coreg) through the model class: LML, every gradient in paramz order,
    alpha, predictions with and without the likelihood"""
    f = np.load(path)
    parts = json.loads(str(f["parts"]))
    X, Y, idx = f["X"], f["Y"], f["output_index"]
    m = _model_from_parts(parts, X, Y, idx, f["noise"])
    assert abs(m.log_likelihood() - float(f["lml"])) <= LML_ATOL
    np.testing.assert_allclose(m.gradient, f["grad"], rtol=GRAD_RTOL, atol=1e-9)
    assert rel(m.posterior.woodbury_vector, f["alpha"]) < 1e-9
    mu, var = m.predict(f["Xnew"], Y_metadata={"output_index": f["output_index_new"]})
    np.testing.assert_allclose(mu, f["mu"], rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(var, f["var"], rtol=1e-7, atol=1e-9)
    mu0, var0 = m.predict(f["Xnew"], include_likelihood=False)
    np.testing.assert_allclose(var0, f["var_noiseless"], rtol=1e-7, atol=1e-9)
    _, cov0 = m.predict(f["Xnew"], full_cov=True, include_likelihood=False)
    np.testing.assert_allclose(cov0, f["cov_noiseless"], rtol=1e-7, atol=1e-9)


def _model_from_parts(parts, X, Y, idx, noise):
    """gpy_b200 model with the kernel of `parts` (terms of products), MixedNoise with the given per-output variances"""
    terms = {}
    for p in parts:
        if p["kind"] == "coregionalize":
            W, kappa = np.asarray(p["W"]), np.asarray(p["kappa"])
            k = gpy_b200.Coregionalize(1, W.shape[0], rank=W.shape[1], W=W, kappa=kappa, active_dims=p["dims"], name="B")
        elif p["kind"] == "bias":
            k = gpy_b200.Bias(X.shape[1], variance=p["variance"])
        else:
            cls = {"rbf": gpy_b200.RBF, "matern32": gpy_b200.Matern32}[p["kind"]]
            k = cls(len(p["dims"]), variance=p["variance"], lengthscale=np.asarray(p["lengthscale"]), ARD=p["ARD"],
                    active_dims=p["dims"])
        terms[p["term"]] = k if p["term"] not in terms else terms[p["term"]] * k
    kern = None
    for t in sorted(terms):
        kern = terms[t] if kern is None else kern + terms[t]
    liks = [gpy_b200.Gaussian(variance=float(v), name="Gaussian_noise_%d" % j) for j, v in enumerate(noise)]
    return gpy_b200.GP(X, Y, kern, gpy_b200.MixedNoise(liks), Y_metadata={"output_index": idx})


def test_coreg_model_predict_checkgrad_optimize():
    """GPCoregionalizedRegression at N = 150: predictions across outputs against the restatement, checkgrad, and 10
    optimizer iterations lower the objective"""
    rng = np.random.default_rng(5)
    Xl = [rng.uniform(-3, 3, (50, 2)) for _ in range(3)]
    Yl = [np.sin(x).sum(1, keepdims=True) * (1 + 0.4 * j) + 0.1 * rng.standard_normal((50, 1)) for j, x in enumerate(Xl)]
    m = gpy_b200.GPCoregionalizedRegression(Xl, Yl, kernel=gpy_b200.ICM(2, 3, gpy_b200.RBF(2, ARD=True), W_rank=2,
                                                                          W=0.5 * rng.standard_normal((3, 2))))
    assert m.gradient.size == 1 + 2 + 6 + 3 + 3
    B = m.kern.parts[1]
    parts = [dict(kind="rbf", term=0, dims=[0, 1], variance=1.0, lengthscale=[1.0, 1.0], ARD=True),
             dict(kind="coregionalize", term=0, dims=[2], W=B.W.values.tolist(), kappa=B.kappa.values.tolist())]
    idx = m.output_index.reshape(-1)
    lml0, g0, res = co.fixture_eval(dict(X=m.X, Y=m.Y, output_index=idx, noise=np.ones(3), parts=json.dumps(parts)))[:3]
    assert abs(m.log_likelihood() - lml0) <= LML_ATOL
    np.testing.assert_allclose(m.gradient, g0, rtol=GRAD_RTOL, atol=1e-9)
    Xnew = np.hstack([rng.uniform(-3, 3, (7, 2)), (np.arange(7) % 3)[:, None]])
    mu0, var0 = co.predict(parts, m.X, res["L"], res["alpha"], Xnew)
    mu, var = m.predict(Xnew, Y_metadata={"output_index": (np.arange(7) % 3)[:, None]})
    np.testing.assert_allclose(mu, mu0, rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(var, var0 + 1.0, rtol=1e-7, atol=1e-9)
    _, cov = m.predict(Xnew, full_cov=True, include_likelihood=False)
    np.testing.assert_allclose(cov, co.predict(parts, m.X, res["L"], res["alpha"], Xnew, full_cov=True)[1], rtol=1e-7,
                               atol=1e-9)
    assert m.checkgrad()
    f0 = m.objective_function()
    m.optimize(max_iters=10)
    assert m.objective_function() < f0


@pytest.mark.parametrize("N", [150, 1300])
def test_coreg_deterministic(N):
    D, O = 4, 3
    X, Y, idx = _data(N, D, O, 1, seed=9)
    parts = co.device_parts(_parts("lcm", D, O, seed=9))
    eng = _engine(N)
    eng.set_data(X, Y)
    nv = np.array([0.05, 0.09, 0.03])[idx]
    a = eng.exact_eval_coreg(parts, nv)
    b = eng.exact_eval_coreg(parts, nv)
    assert a[0] == b[0]
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


def test_coreg_bad_index_then_reuse():
    """an output index >= output_dim is an error with the library's message; the context then evaluates correctly, and a
    plain exact_eval / exact_eval_multi afterwards still match the oracle"""
    D, O, N = 3, 3, 300
    X, Y, idx = _data(N, D, O, 1, seed=13)
    parts = _parts("icm", D, O, seed=13)
    eng = _engine(N)
    bad = X.copy()
    bad[17, D] = O
    eng.set_data(bad, Y)
    with pytest.raises(_ffi.GpxError, match="output index"):
        eng.exact_eval_coreg(co.device_parts(parts), 0.05)
    eng.set_data(X, Y)
    lml, g, _, _ = eng.exact_eval_coreg(co.device_parts(parts), 0.05)
    lml0, _, res = co.eval_lml_grad(X, Y, parts, 0.05)
    assert abs(lml - lml0) <= LML_ATOL
    np.testing.assert_allclose(g, res["device_grad"], rtol=GRAD_RTOL, atol=1e-9)
    Xnew = X[:4].copy()
    Xnew[2, D] = -1.0
    with pytest.raises(_ffi.GpxError, match="output index"):
        eng.predict(Xnew)
    # a B that is not exactly symmetric is rejected, and a rejected call leaves no posterior to predict from
    desc = co.device_parts(parts)
    Bbad = np.array(desc[1][5], copy=True)
    Bbad[0, 1] += 1e-3
    with pytest.raises(_ffi.GpxError, match="symmetric"):
        eng.exact_eval_coreg(desc[:1] + [desc[1][:5] + (Bbad,)], 0.05)
    with pytest.raises(_ffi.GpxError, match="no successful"):
        eng.predict(X[:4])
    Xs = np.ascontiguousarray(X[:, :D])
    eng.set_data(Xs, Y)
    lml1, g1, _ = eng.exact_eval("rbf", True, 1.1, [1.2, 1.5, 0.9], 0.05)
    lml2, g2, _ = o.eval_lml_grad(Xs, Y, "rbf", True, 1.1, [1.2, 1.5, 0.9], 0.05)
    assert abs(lml1 - lml2) <= LML_ATOL
    np.testing.assert_allclose(g1, g2, rtol=GRAD_RTOL, atol=1e-9)
    mp = [dict(kind="rbf", term=0, dims=[0, 1], variance=1.2, lengthscale=[1.3, 0.8], ARD=True),
          dict(kind="matern32", term=0, dims=[2], variance=0.8, lengthscale=[1.1]), dict(kind="bias", term=1, variance=0.3)]
    desc = [(p["kind"], p.get("ARD", False), p["term"], p.get("dims", []), p["variance"], p.get("lengthscale"))
            for p in mp]
    lml3, g3, _ = eng.exact_eval_multi(desc, 0.05)
    lml4, g4, _ = o.composite_eval_lml_grad(Xs, Y, mp, 0.05)
    assert abs(lml3 - lml4) <= LML_ATOL
    np.testing.assert_allclose(g3, g4, rtol=GRAD_RTOL, atol=1e-9)



def test_composite_after_single_kernel_on_the_tcgen05_route():
    """a single-kernel evaluation on the chain schedule (tcgen05 route) followed by composite evaluations on the same
    context: the composite K-build must be complete before the sweep's first diagonal block starts"""
    D, O, N = 4, 3, 2100
    X, Y, idx = _data(N, D, O, 1, seed=31)
    parts = _parts("icm", D, O, seed=31)
    eng = _engine(N)
    Xs = np.ascontiguousarray(X[:, :D])
    eng.set_data(Xs, Y)
    eng.exact_eval("rbf", True, 1.1, [1.2, 1.5, 0.9, 1.3], 0.05)
    eng.set_data(X, Y)
    nv = np.array([0.05, 0.09, 0.03])[idx]
    lml, g, _, _ = eng.exact_eval_coreg(co.device_parts(parts), nv)
    lml0, _, res = co.eval_lml_grad(X, Y, parts, nv)
    assert abs(lml - lml0) <= LML_ATOL
    np.testing.assert_allclose(g, res["device_grad"], rtol=GRAD_RTOL, atol=1e-9)


@pytest.mark.parametrize("N", [150, 1300])
def test_composite_with_per_point_noise_without_coregionalization(N):
    """RBF + Bias with a HeteroscedasticGaussian likelihood: a composite kernel with a noise vector and no coregionalization
    part takes gpx_exact_eval_coreg too (K-build with the per-point diagonal, diag(dL_dK) per point)"""
    D = 3
    rng = np.random.default_rng(N + 1)
    X = rng.uniform(-3, 3, (N, D))
    Y = (np.sin(X).sum(1) / np.sqrt(D) + 0.1 * rng.standard_normal(N))[:, None]
    nv = rng.uniform(0.02, 0.2, N)
    meta = {"output_index": np.arange(N)[:, None]}
    eng = _engine(N)
    k = gpy_b200.RBF(D, variance=1.1, lengthscale=np.array([1.2, 0.8, 1.6]), ARD=True) + gpy_b200.Bias(D, variance=0.3)
    lik = gpy_b200.HeteroscedasticGaussian(meta)
    lik.variance.values[...] = nv
    m = gpy_b200.GP(X, Y, k, lik, Y_metadata=meta, engine=eng)
    parts = [dict(kind="rbf", term=0, dims=[0, 1, 2], variance=1.1, lengthscale=[1.2, 0.8, 1.6], ARD=True),
             dict(kind="bias", term=1, variance=0.3)]
    lml0, g0, res = co.eval_lml_grad(X, Y, parts, nv)
    assert abs(m.log_likelihood() - lml0) <= LML_ATOL
    np.testing.assert_allclose(m.gradient, np.concatenate([g0[:-1], res["dnoise"]]), rtol=GRAD_RTOL, atol=1e-9)
    assert rel(m.posterior.K, res["K"]) < 1e-12
    assert rel(m.posterior.woodbury_chol, res["L"]) < 1e-10
    assert rel(m.posterior.woodbury_vector, res["alpha"]) < 1e-9


@pytest.mark.skipif(not os.path.isdir(os.environ.get("GPX_REFERENCE", "/root/reference") + "/GPy"),
                    reason="reference tree not present")
def test_stock_gpy_coregionalized_model_runs_fused():
    """the reference's own GPCoregionalizedRegression with plugin kernels and the plugin inference, on the device"""
    from gpy_b200 import _ffi as ffi
    from test_gpy_plugin_coreg_cpu import plugin_pair
    stock, plug, B = plugin_pair(ffi)
    assert abs(plug.log_likelihood() - stock.log_likelihood()) <= LML_ATOL
    np.testing.assert_allclose(np.asarray(plug.gradient), np.asarray(stock.gradient), rtol=GRAD_RTOL, atol=1e-9)
