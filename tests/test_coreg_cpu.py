"""Multi-output (coregionalized) regression without a GPU: the NumPy restatement (tests/coreg_oracle.py) against the
reference's stored numbers (tests/golden/coreg) and, where a reference tree exists, against the live reference objects;
the host routing of gpy_b200.GPCoregionalizedRegression with a test double of the engine; the S -> (dW, dkappa) step."""
import glob
import json
import os

import numpy as np
import pytest

import coreg_oracle as co

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "coreg")
FIXTURES = sorted(glob.glob(os.path.join(GOLDEN, "*.npz")))


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - b)) / max(np.max(np.abs(b)), 1e-300))


def test_fixtures_present():
    assert len(FIXTURES) == 3
    for path in FIXTURES:
        assert "unmodified reference" in str(np.load(path)["source"])


@pytest.mark.parametrize("path", FIXTURES, ids=os.path.basename)
def test_restatement_matches_reference_fixtures(path):
    f = np.load(path)
    lml, grad, res, parts = co.fixture_eval(f)
    assert abs(lml - float(f["lml"])) <= 1e-12 * abs(float(f["lml"]))
    assert grad.shape == f["grad"].shape
    np.testing.assert_allclose(grad, f["grad"], rtol=1e-12, atol=0)
    assert rel(res["alpha"], f["alpha"]) <= 1e-12
    mu, var = co.predict(parts, f["X"], res["L"], res["alpha"], f["Xnew"])
    assert rel(mu, f["mu_noiseless"]) <= 1e-12 and rel(var, f["var_noiseless"]) <= 1e-12
    _, cov = co.predict(parts, f["X"], res["L"], res["alpha"], f["Xnew"], full_cov=True)
    assert rel(cov, f["cov_noiseless"]) <= 1e-12
    noise = np.asarray(f["noise"])[np.asarray(f["output_index_new"]).reshape(-1)]
    assert rel(var + noise[:, None], f["var"]) <= 1e-12


def test_rows_not_grouped_by_output():
    """the shuffled fixture is the grouped one with its rows permuted: same LML and gradient"""
    a = np.load(os.path.join(GOLDEN, "icm_o3_r2_rbf_ard_n75_d2.npz"))
    b = np.load(os.path.join(GOLDEN, "icm_o3_r2_rbf_ard_n75_d2_shuffled.npz"))
    assert not np.all(np.diff(b["output_index"].reshape(-1)) >= 0)
    assert abs(float(a["lml"]) - float(b["lml"])) <= 1e-10 * abs(float(a["lml"]))
    np.testing.assert_allclose(a["grad"], b["grad"], rtol=1e-8, atol=1e-12)


def _reference():
    try:
        import importlib.util
        spec = importlib.util.spec_from_file_location(
            "make_coreg_golden", os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_coreg_golden.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod.load_reference()
    except ImportError as e:
        pytest.skip("no reference tree: %s" % e)


def test_restatement_matches_live_reference():
    G, C, M, mo, GPCR, R = _reference()
    rng = np.random.RandomState(21)
    Xl = [rng.uniform(-2, 2, (12 + j, 2)) for j in range(3)]
    Yl = [np.cos(x).sum(1, keepdims=True) + 0.1 * rng.randn(x.shape[0], 1) for x in Xl]
    W, kappa = rng.randn(3, 2) * 0.5, np.array([0.3, 0.6, 0.9])
    m = GPCR(Xl, Yl, kernel=mo.ICM(2, 3, G.Matern32(2, variance=0.8, lengthscale=1.3), W_rank=2, W=W, kappa=kappa))
    parts = [dict(kind="matern32", term=0, dims=[0, 1], variance=0.8, lengthscale=[1.3], ARD=False),
             dict(kind="coregionalize", term=0, dims=[2], W=W.tolist(), kappa=kappa.tolist())]
    f = dict(X=np.asarray(m.X), Y=np.asarray(m.Y), output_index=np.asarray(m.output_index), noise=np.ones(3),
             parts=json.dumps(parts))
    lml, grad, _, _ = co.fixture_eval(f)
    assert abs(lml - float(m.log_likelihood())) <= 1e-12 * abs(lml)
    np.testing.assert_allclose(grad, np.asarray(m.gradient), rtol=1e-12, atol=1e-14)


def test_S_to_W_kappa_gradients():
    """Coregionalize.set_gradients_from_S is coregionalize.py:123-128; the dense host reduction agrees with it"""
    import gpy_b200
    rng = np.random.default_rng(4)
    O, R = 4, 2
    W = rng.standard_normal((O, R))
    k = gpy_b200.Coregionalize(1, O, rank=R, W=W, kappa=np.full(O, 0.5))
    S = rng.standard_normal((O, O))
    k.set_gradients_from_S(S)
    Ssym = S + S.T
    np.testing.assert_array_equal(k.kappa.gradient, np.diag(S))
    np.testing.assert_array_equal(k.W.gradient, (W[:, None, :] * Ssym[:, :, None]).sum(0))
    idx = rng.integers(0, O, 30)[:, None].astype(float)
    dL = rng.standard_normal((30, 30))
    dL = dL + dL.T
    k.update_gradients_full(dL, idx)
    gW, gk = co.CoregOracle(W, np.full(O, 0.5)).update_gradients_full(dL, idx)
    np.testing.assert_allclose(k.W.gradient, gW, rtol=1e-13)
    np.testing.assert_allclose(k.kappa.gradient, gk, rtol=1e-13)
    np.testing.assert_array_equal(k.K(idx), co.CoregOracle(W, np.full(O, 0.5)).K(idx))
    np.testing.assert_array_equal(k.Kdiag(idx), np.diag(k.B)[idx.astype(int).reshape(-1)])


def test_S_to_W_kappa_matches_reference_class():
    G, C, M, mo, GPCR, R = _reference()
    import gpy_b200
    Cref = __import__("sys").modules["GPy.kern"].Coregionalize
    rng = np.random.RandomState(8)
    W, kappa = rng.randn(3, 2), np.array([0.2, 0.4, 0.6])
    ref = Cref(1, 3, rank=2, W=W.copy(), kappa=kappa.copy())
    ours = gpy_b200.Coregionalize(1, 3, rank=2, W=W, kappa=kappa)
    idx = rng.randint(0, 3, (25, 1)).astype(float)
    dL = rng.randn(25, 25)
    dL = dL + dL.T
    ref.update_gradients_full(dL, idx)
    ours.update_gradients_full(dL, idx)
    np.testing.assert_allclose(ours.W.gradient, np.asarray(ref.W.gradient), rtol=1e-13)
    np.testing.assert_allclose(ours.kappa.gradient, np.asarray(ref.kappa.gradient), rtol=1e-13)
    np.testing.assert_array_equal(ours.B, np.asarray(ref.B))


class FakeEngine(object):
    """test double of gpy_b200._ffi.Engine answering gpx_exact_eval_coreg from the restatement"""

    def __init__(self):
        self.calls, self.eval_serial = [], 0

    def set_data(self, X, Y):
        self.X, self.Y = np.array(X), np.array(Y)
        self.eval_serial += 1
        self.calls.append("set_data")

    def exact_eval_coreg(self, parts, noise, jitter=1e-8, max_tries=5):
        self.calls.append("exact_eval_coreg")
        self.eval_serial += 1
        self.parts = []
        for (k, a, t, d, v, l) in parts:
            if k == "coregionalize":
                self.parts.append(dict(kind=k, term=t, dims=d, B=l))
            else:
                self.parts.append(dict(kind=k, ARD=a, term=t, dims=d, variance=v, lengthscale=l))
        lml, _, self.res = co.eval_lml_grad(self.X, self.Y, self.parts, noise)
        return lml, self.res["device_grad"], (self.res["dnoise"] if np.ndim(noise) else None), 0.0

    def get(self, which):
        return {"L": self.res["L"], "alpha": self.res["alpha"], "K": self.res["K"]}[which]

    def predict(self, Xnew, full_cov=False):
        return co.predict(self.parts, self.X, self.res["L"], self.res["alpha"], Xnew, full_cov)


def _cpu_model(eng, seed=3):
    import gpy_b200
    from gpy_b200.inference import ExactGaussianInference
    rng = np.random.default_rng(seed)
    Xl = [rng.uniform(-2, 2, (10 + j, 2)) for j in range(3)]
    Yl = [np.sin(x).sum(1, keepdims=True) + 0.1 * rng.standard_normal((x.shape[0], 1)) for x in Xl]
    W = 0.5 * rng.standard_normal((3, 2))
    k = gpy_b200.ICM(2, 3, gpy_b200.RBF(2, variance=1.2, lengthscale=np.array([0.8, 1.3]), ARD=True), W_rank=2, W=W,
                     kappa=np.array([0.3, 0.5, 0.7]))
    m = gpy_b200.GPCoregionalizedRegression.__new__(gpy_b200.GPCoregionalizedRegression)
    inf = ExactGaussianInference(engine=eng)
    from gpy_b200 import model as mdl
    orig = mdl.ExactGaussianInference
    mdl.ExactGaussianInference = lambda device=0, engine=None: inf
    try:
        m.__init__(Xl, Yl, kernel=k)
    finally:
        mdl.ExactGaussianInference = orig
    return m, Xl, Yl, W


def test_model_routes_to_one_fused_call():
    eng = FakeEngine()
    m, Xl, Yl, W = _cpu_model(eng)
    assert eng.calls == ["set_data", "exact_eval_coreg"]
    assert m.gradient.size == 1 + 2 + 6 + 3 + 3          # rbf variance, lengthscale(2), B.W (3x2), B.kappa (3), noise (3)
    parts = [dict(kind="rbf", term=0, dims=[0, 1], variance=1.2, lengthscale=[0.8, 1.3], ARD=True),
             dict(kind="coregionalize", term=0, dims=[2], W=W.tolist(), kappa=[0.3, 0.5, 0.7])]
    f = dict(X=m.X, Y=m.Y, output_index=m.output_index, noise=np.ones(3), parts=json.dumps(parts))
    lml, grad, _, _ = co.fixture_eval(f)
    assert abs(m.log_likelihood() - lml) <= 1e-12 * abs(lml)
    np.testing.assert_allclose(m.gradient, grad, rtol=1e-12, atol=1e-14)
    assert [p.name for p in m.flattened_parameters()] == ["variance", "lengthscale", "W", "kappa"] + ["variance"] * 3
    m.kern.parts[1].kappa[1] = 0.9                      # a parameter write re-evaluates through the same call
    assert eng.calls[-1] == "exact_eval_coreg" and len(eng.calls) == 3
    Xnew = np.hstack([np.zeros((3, 2)), np.arange(3)[:, None]])
    mu, var = m.predict(Xnew, Y_metadata={"output_index": np.arange(3)[:, None]})
    assert mu.shape == (3, 1) and var.shape == (3, 1)


def test_model_matches_reference_gradient_layout():
    G, C, M, mo, GPCR, R = _reference()
    eng = FakeEngine()
    m, Xl, Yl, W = _cpu_model(eng)
    ref = GPCR(Xl, Yl, kernel=mo.ICM(2, 3, G.RBF(2, variance=1.2, lengthscale=np.array([0.8, 1.3]), ARD=True), W_rank=2,
                                     W=W.copy(), kappa=np.array([0.3, 0.5, 0.7])))
    assert np.asarray(ref.gradient).size == m.gradient.size
    np.testing.assert_allclose(m.gradient, np.asarray(ref.gradient), rtol=1e-10, atol=1e-12)
    assert abs(m.log_likelihood() - float(ref.log_likelihood())) <= 1e-10 * abs(m.log_likelihood())
