"""The oracle restatement (and the host mirror classes) against the UNMODIFIED reference, GPy 1.14.2.

The reference's numbers for every case below are stored in tests/golden/reference/: tests/golden/make_golden.py runs the
reference itself (through oracle/ref_gpy.py and the test-only paramz stand-in) on the inputs these tests build, and
`record_reference` below is what it records. The inputs are rebuilt here from the same seeds. Every vector (gradients,
alpha, woodbury vectors, predictions) and every array of up to WHOLE entries is stored whole; a larger matrix is kept as a
fixed, seeded sample of SAMPLE entries (see _picked). The comparisons use the tolerances the live comparison used."""
import json
import os
import zlib

import numpy as np
import pytest

from oracle import gpy_oracle as o

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
WHOLE = 512
SAMPLE = 96


def _picked(key, shape):
    """flat indices of the stored entries of an array of `shape`: all of them for a vector (at most one dimension > 1) or
    an array of at most WHOLE entries; else SAMPLE entries picked by a seed taken from `key`. The large square matrices
    compared here (K, dL_dK, L) are symmetric or lower triangular, so theirs are picked from the lower triangle."""
    size = int(np.prod(shape))
    if size <= WHOLE or sum(n > 1 for n in shape) <= 1:
        return np.arange(size)
    pool = np.arange(size)
    if len(shape) == 2 and shape[0] == shape[1]:
        pool = np.ravel_multi_index(np.tril_indices(shape[0]), shape)
    return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(pool, SAMPLE, replace=False))


def _sample(key, a):
    """the stored part of array `a`"""
    return np.asarray(a, dtype=np.float64).reshape(-1)[_picked(key, np.shape(a))]


def put(store, key, a):
    """record the reference's array `a` under `key` (used by make_golden.py)"""
    store[key] = (_sample(key, a), np.shape(a))


def pack(store):
    """-> the two arrays of crosscheck.npz: every recorded entry end to end, and a JSON index key -> [offset, size, shape]"""
    index, offset = {}, 0
    for key, (v, shape) in store.items():
        index[key] = [offset, int(v.size), [int(n) for n in shape]]
        offset += v.size
    values = np.concatenate([v for v, _ in store.values()])
    return {"values": values, "index": np.array(json.dumps(index))}


@pytest.fixture(scope="module")
def R():
    """R(key, ours) -> (the same sample of ours, the reference's), after checking that the shapes agree; R.get(key) -> the
    reference's recorded entries"""
    z = np.load(os.path.join(GOLDEN, "crosscheck.npz"))
    values, index = z["values"], json.loads(str(z["index"]))

    def get(key):
        off, n, _ = index[key]
        return values[off:off + n]

    def ref(key, ours):
        assert tuple(index[key][2]) == np.shape(ours), (key, index[key][2], np.shape(ours))
        return _sample(key, ours), get(key)
    ref.get = get
    return ref


def _close(R, key, ours, **tol):
    a, b = R(key, ours)
    np.testing.assert_allclose(a, b, err_msg=key, **tol)


def _equal(R, key, ours):
    a, b = R(key, ours)
    np.testing.assert_array_equal(a, b, err_msg=key)


# ---- inputs (the same seeds for the recording and for the tests) ---------------------------------------------------
def _exact_inputs(kind, ARD):
    for (N, D, seed) in ((60, 1, 0), (150, 4, 1), (333, 8, 2)):
        X, Y = o.synthetic(N, D, seed)
        rng = np.random.default_rng(seed)
        ls = rng.uniform(0.8, 2.5, D) if ARD else float(rng.uniform(0.8, 2.5))
        var, noise = float(rng.uniform(0.5, 2)), float(rng.uniform(0.01, 0.2))
        Xn = rng.uniform(-3, 3, (6, D))
        yield "exact_%s_%d_n%d" % (kind, ARD, N), X, Y, var, ls, noise, Xn


def _linalg_inputs():
    from test_oracle import _corrupt
    B = np.random.default_rng(0).standard_normal((50, 7))
    return _corrupt(3), B, B.dot(B.T) + 50 * np.eye(50)


def _native_inputs():
    rng = np.random.default_rng(1)
    X, Z = rng.standard_normal((300, 10)), rng.standard_normal((20, 10))
    return [(rng.standard_normal((300, 300)), X, X), (rng.standard_normal((300, 20)), X, Z)]


def _gradients_X_inputs():
    rng = np.random.default_rng(2)
    X, Z = rng.standard_normal((60, 4)), rng.standard_normal((25, 4))
    for name, kind in (("RBF", "rbf"), ("Matern32", "matern32"), ("Matern52", "matern52"), ("Exponential", "exponential")):
        for ARD in (False, True):
            ls = np.array([1.0, 1.5, 2.0, 0.8]) if ARD else 1.3
            d1, d2 = rng.standard_normal((60, 60)), rng.standard_normal((60, 25))
            yield "gradX_%s_%d" % (kind, ARD), name, kind, ARD, ls, X, Z, d1, d2


VARDTC_CASES = [(k, a) for k in ("rbf", "matern32", "exponential") for a in (False, True)]


def _vardtc_inputs(kind, ARD):
    X, Y = o.synthetic(300, 3, 4)
    Z = X[np.random.default_rng(4).permutation(300)[:20]].copy()
    return "vardtc_%s_%d" % (kind, ARD), X, Y, Z, (np.array([1.2, 1.7, 2.1]) if ARD else 1.6)


VARDTC_HET_CASES = [("rbf", True, 1), ("matern52", False, 1), ("exponential", True, 2)]


def _vardtc_het_inputs(kind, ARD, P):
    rng = np.random.default_rng(14)
    N, M = 260, 24
    X = rng.uniform(-3, 3, (N, 3))
    Y = np.stack([np.sin(X).sum(1) + 0.2 * rng.standard_normal(N) for _ in range(P)], 1)
    Z = X[rng.permutation(N)[:M]].copy()
    ls = np.array([1.2, 1.7, 2.1]) if ARD else 1.6
    return "vardtc_het_%s_%d_p%d" % (kind, ARD, P), X, Y, Z, ls, rng.uniform(0.01, 0.4, N)


HET_CASES = [("rbf", True), ("matern32", False)]


def _het_inputs(kind, ARD):
    for (N, D, seed) in ((70, 2, 3), (211, 5, 4)):
        X, Y = o.synthetic(N, D, seed)
        rng = np.random.default_rng(seed)
        ls = rng.uniform(0.8, 2.5, D) if ARD else float(rng.uniform(0.8, 2.5))
        var = float(rng.uniform(0.5, 2))
        yield "het_%s_%d_n%d" % (kind, ARD, N), X, Y, var, ls, rng.uniform(0.01, 0.3, N)


def _mirror_het_inputs():
    rng = np.random.default_rng(0)
    N = 17
    md = {"output_index": np.arange(N)[:, None]}
    nv = rng.uniform(0.1, 1.0, N)
    sub = {"output_index": np.array([3, 0, 11])[:, None]}
    dd = rng.standard_normal(N)
    mu, var = rng.standard_normal((3, 1)), rng.uniform(0.1, 1, (3, 1))
    return md, nv, sub, dd, mu, var


MIXED_NOISE = [0.02, 0.3, 0.11]


def _mixed_inputs():
    rng = np.random.default_rng(7)
    N, D = 157, 3
    X, Y = o.synthetic(N, D, 5)
    idx = rng.integers(0, 3, N)
    ls = rng.uniform(0.8, 2.5, D)
    sub = {"output_index": np.array([2, 0, 1, 1])[:, None]}
    mu, var = rng.standard_normal((4, 1)), rng.uniform(0.1, 1, (4, 1))
    return X, Y, idx, ls, sub, mu, var


def _composite_inputs():
    rng = np.random.default_rng(5)
    N, D = 40, 5
    X = rng.uniform(-2, 2, (N, D))
    X2 = rng.uniform(-2, 2, (17, D))
    Y = np.sin(X).sum(1, keepdims=True) + 0.1 * rng.standard_normal((N, 1))
    return X, X2, Y


# ---- the tests ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", o.KINDS)
@pytest.mark.parametrize("ARD", [False, True])
def test_oracle_equals_reference(R, kind, ARD):
    for key, X, Y, var, ls, noise, Xn in _exact_inputs(kind, ARD):
        lml, g, res = o.eval_lml_grad(X, Y, kind, ARD, var, ls, noise)
        lml_r = float(R(key + "_lml", lml)[1][0])
        assert abs(lml_r - lml) <= 1e-10 * max(1.0, abs(lml))
        _close(R, key + "_grad", g, rtol=1e-10, atol=1e-12)
        _close(R, key + "_K", res["K"], rtol=0, atol=1e-14)
        _close(R, key + "_L", res["L"], rtol=1e-12, atol=1e-14)
        _close(R, key + "_alpha", res["alpha"], rtol=1e-10, atol=1e-12)
        _close(R, key + "_dL_dK", res["dL_dK"], rtol=1e-10, atol=1e-12)
        kern = o.StationaryOracle(kind, X.shape[1], var, ls, ARD)
        mu, pv = o.predict(kern, X, res["L"], res["alpha"], Xn, noise)
        _close(R, key + "_mu", mu, rtol=1e-10, atol=1e-12)
        _close(R, key + "_var", pv, rtol=1e-9, atol=1e-12)


def test_oracle_linalg_equals_reference_linalg(R):
    """jitchol ladder / pdinv / tdot / symmetrify of GPy/util/linalg.py, same inputs as GPy/testing/test_linalg.py:8-18."""
    A, B, S = _linalg_inputs()
    L, jit = o.jitchol(A, maxtries=5)
    _equal(R, "linalg_jitchol_L", L)
    assert R.get("linalg_jitchol_4_raises")[0] == 1     # the reference's ladder gives up after 4 tries on this matrix
    with pytest.raises(np.linalg.LinAlgError):
        o.jitchol(A, maxtries=4)
    _equal(R, "linalg_tdot", o.tdot(B))
    Ai2, L2, Li2, ld2 = o.pdinv(S)
    # dpotri's last bits depend on the BLAS thread count, which the stored numbers cannot share with every machine: a few
    # units of rounding of the sums that make each entry, i.e. relative to the largest entries for the smallest ones
    eps = np.finfo(float).eps
    _close(R, "linalg_pdinv_Ai", Ai2, rtol=4 * eps, atol=4 * eps * np.abs(Ai2).max())
    _equal(R, "linalg_pdinv_L", L2)
    _equal(R, "linalg_pdinv_logdet", ld2)


def test_reference_native_helper_matches(R):
    """The reference's NumPy reduction Stationary._lengthscale_grads_pure (stationary.py:234-235) against our C restatement
    of the serial Cython loop and, where oracle/Makefile compiled it into oracle/_ref, the reference's own
    stationary_utils.c: mirrors GPy/testing/test_cython.py:83-98."""
    which = ["port"] + (["ref"] if o._load_native()["ref"] is not None else [])
    for i, (tmp, A, B) in enumerate(_native_inputs()):
        for w in which:
            g_c = o.lengthscale_grads_native(tmp, A, B, np.ones(10), w)
            ours, ref = R("native_%d" % i, g_c)
            assert np.allclose(ref, ours), w


def test_oracle_gradients_X_equals_reference(R):
    for key, name, kind, ARD, ls, X, Z, d1, d2 in _gradients_X_inputs():
        ko = o.StationaryOracle(kind, 4, 0.9, ls, ARD)
        _close(R, key + "_XX", ko.gradients_X(d1, X), rtol=1e-12, atol=1e-14)
        _close(R, key + "_XZ", ko.gradients_X(d2, X, Z), rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("kind", ["rbf", "matern32", "exponential"])
@pytest.mark.parametrize("ARD", [False, True])
def test_oracle_vardtc_equals_reference(R, kind, ARD):
    """Sparse GP regression: oracle.vardtc_inference / sparse_eval against the unmodified
    GPy/inference/latent_function_inference/var_dtc.py (+ gradient wiring of core/sparse_gp.py:108-119)."""
    key, X, Y, Z, ls = _vardtc_inputs(kind, ARD)
    lml, g, Zg, res = o.sparse_eval(X, Y, Z, kind, ARD, 1.3, ls, 0.07)
    lml_r = float(R(key + "_lml", lml)[1][0])
    assert abs(lml - lml_r) <= 1e-9 * abs(lml_r)
    _close(R, key + "_grad", g, rtol=1e-8, atol=1e-10)
    _close(R, key + "_Zgrad", Zg, rtol=1e-8, atol=1e-10)
    _close(R, key + "_woodbury_vector", res["woodbury_vector"], rtol=1e-8, atol=1e-12)
    _close(R, key + "_woodbury_inv", res["woodbury_inv"], rtol=1e-7, atol=1e-10)
    _close(R, key + "_dL_dKnm", res["dL_dKnm"], rtol=1e-8, atol=1e-12)


@pytest.mark.parametrize("kind,ARD,P", VARDTC_HET_CASES)
def test_oracle_vardtc_heteroscedastic_equals_reference(R, kind, ARD, P):
    """Sparse GP regression with one noise variance per data point: the het_noise branches of the unmodified
    var_dtc.py (:127-128, :221-227, :241-257, :267-269) with the reference's HeteroscedasticGaussian, against
    oracle.vardtc_inference with a noise vector."""
    key, X, Y, Z, ls, nv = _vardtc_het_inputs(kind, ARD, P)
    lml, g, Zg, res = o.sparse_eval(X, Y, Z, kind, ARD, 1.3, ls, nv)
    lml_r = float(R(key + "_lml", lml)[1][0])
    assert abs(lml - lml_r) <= 1e-9 * abs(lml_r)
    _close(R, key + "_grad", g, rtol=1e-8, atol=1e-9)
    _close(R, key + "_Zgrad", Zg, rtol=1e-8, atol=1e-10)
    _close(R, key + "_woodbury_vector", res["woodbury_vector"], rtol=1e-8, atol=1e-12)
    _close(R, key + "_woodbury_inv", res["woodbury_inv"], rtol=1e-7, atol=1e-10)


@pytest.mark.parametrize("kind,ARD", HET_CASES)
def test_oracle_heteroscedastic_equals_reference(R, kind, ARD):
    """One noise variance per data point: oracle restatement against the reference's HeteroscedasticGaussian +
    ExactGaussianInference objects (likelihoods/gaussian.py:347-362, models/gp_heteroscedastic_regression.py:22-37)."""
    for key, X, Y, var, ls, nv in _het_inputs(kind, ARD):
        N, D = X.shape
        lml, g, res = o.eval_lml_grad(X, Y, kind, ARD, var, ls, nv)
        assert g.size == 1 + (D if ARD else 1) + N
        lml_r = float(R(key + "_lml", lml)[1][0])
        assert abs(lml_r - lml) <= 1e-10 * max(1.0, abs(lml))
        _close(R, key + "_grad", g, rtol=1e-10, atol=1e-12)
        _close(R, key + "_alpha", res["alpha"], rtol=1e-10, atol=1e-12)


def test_mirror_heteroscedastic_likelihood_matches_reference_class(R):
    """gpy_b200.inference.HeteroscedasticGaussian (host mirror) against the reference class: variance lookup, gradient
    routing and predictive values for the same Y_metadata (likelihoods/gaussian.py:347-373)."""
    from gpy_b200.inference import HeteroscedasticGaussian
    md, nv, sub, dd, mu, var = _mirror_het_inputs()
    mir = HeteroscedasticGaussian(md)
    mir.variance.values[...] = nv
    _equal(R, "mirror_het_gaussian_variance", mir.gaussian_variance(sub).reshape(-1))
    _equal(R, "mirror_het_gradients", np.asarray(mir.exact_inference_gradients(dd, md)).reshape(-1))
    m1, v1 = mir.predictive_values(mu.copy(), var.copy(), False, sub)
    _close(R, "mirror_het_pred_var", np.asarray(v1).reshape(-1), rtol=0, atol=0)
    _equal(R, "mirror_het_pred_mu", m1)


def test_mixed_noise_mirror_and_oracle_equal_reference(R):
    """MixedNoise (likelihoods/mixed_noise.py:14-53): the reference's own MixedNoise + ExactGaussianInference objects against
    (a) the oracle fed the per-point variance vector, with the noise gradients summed per output index, and (b) the host
    mirror class (variance lookup, gradient routing, predictive values)."""
    from gpy_b200.inference import Gaussian, MixedNoise
    X, Y, idx, ls, sub, mu, var = _mixed_inputs()
    D = X.shape[1]
    nv = np.asarray(MIXED_NOISE)[idx]
    _equal(R, "mixed_variance", nv)
    lml, g, res = o.eval_lml_grad(X, Y, "matern52", True, 1.3, ls, nv)
    gk, dn = g[:1 + D], g[1 + D:]
    gsum = np.array([dn[idx == j].sum() for j in range(3)])
    lml_r = float(R("mixed_lml", lml)[1][0])
    assert abs(lml_r - lml) <= 1e-10 * max(1.0, abs(lml))
    _close(R, "mixed_grad", np.concatenate([gk, gsum]), rtol=1e-10, atol=1e-12)
    _close(R, "mixed_alpha", res["alpha"], rtol=1e-10, atol=1e-12)
    mir = MixedNoise([Gaussian(v) for v in MIXED_NOISE])
    md = {"output_index": idx.reshape(-1, 1)}
    np.testing.assert_array_equal(mir.gaussian_variance(md), nv)
    dn_rec = R.get("mixed_dn")                      # the gradient vector the reference's routing was given
    _equal(R, "mixed_routed", np.asarray(mir.exact_inference_gradients(dn_rec, md)))
    m1, v1 = mir.predictive_values(mu.copy(), var.copy(), False, sub)
    _close(R, "mixed_pred_var", np.asarray(v1).reshape(-1), rtol=0, atol=0)
    _equal(R, "mixed_pred_mu", m1)
    mir.update_gradients(gsum)
    np.testing.assert_allclose([float(l.variance.gradient[0]) for l in mir.likelihoods_list], gsum)


def test_cited_reference_locations_exist():
    """Every `GPy/...:line` location cited in include/gpx.h, INTEGRATION.md and DESIGN.md §1 must exist in the reference tree
    (file present, at least that many lines) — the citations are how parity is audited. The line count of every source file
    of the reference is stored in tests/golden/reference/gpy_line_counts.json."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(GOLDEN, "gpy_line_counts.json")) as f:
        lines = json.load(f)
    texts = [open(os.path.join(root, "include", "gpx.h")).read(), open(os.path.join(root, "INTEGRATION.md")).read()]
    pat = re.compile(r"(GPy/[A-Za-z0-9_/]+\.(?:py|pyx|c)):(\d+)(?:-(\d+))?")
    seen = 0
    for t in texts:
        for m in pat.finditer(t):
            assert m.group(1) in lines, m.group(0)
            last = int(m.group(3) or m.group(2))
            assert last <= lines[m.group(1)], (m.group(0), lines[m.group(1)])
            seen += 1
    assert seen >= 20


COMPOSITE_PARTS = [dict(kind="rbf", term=0, dims=[0, 1], variance=1.2, lengthscale=np.array([1.0, 2.0]), ARD=True),
                   dict(kind="matern32", term=0, dims=[2, 3], variance=0.8, lengthscale=1.5, ARD=False),
                   dict(kind="matern52", term=1, dims=list(range(5)), variance=0.5, lengthscale=np.linspace(1.5, 2.5, 5),
                        ARD=True),
                   dict(kind="white", term=2, dims=None, variance=0.05), dict(kind="bias", term=3, dims=None, variance=0.3)]


def test_composite_oracle_equals_reference_add_prod_static(R):
    """oracle.composite_* (restating add.py:60-99, prod.py:59-68,377-396, static.py:63-185) against the reference's own
    Add / Prod / White / Bias objects: K, Kdiag and every parameter gradient for a foreign dL_dK."""
    X, X2, Y = _composite_inputs()
    kp = o.composite_parts(COMPOSITE_PARTS)
    _close(R, "composite_K", o.composite_K(kp, X), rtol=1e-14, atol=1e-15)
    _close(R, "composite_K2", o.composite_K(kp, X, X2), rtol=1e-14, atol=1e-15)
    _close(R, "composite_Kdiag", o.composite_Kdiag(kp, X), rtol=1e-14)
    lml0, g0, _ = o.composite_eval_lml_grad(X, Y, COMPOSITE_PARTS, 0.1)
    assert abs(lml0 - float(R("composite_lml", lml0)[1][0])) < 1e-10
    _close(R, "composite_grad", g0, rtol=1e-10, atol=1e-12)


# ---- what the reference computes for the inputs above (run by make_golden.py where the reference is importable) ------
def record_reference(store):
    from oracle import ref_gpy
    G = ref_gpy.load()
    for kind in o.KINDS:
        for ARD in (False, True):
            for key, X, Y, var, ls, noise, Xn in _exact_inputs(kind, ARD):
                r = ref_gpy.evaluate(G, X, Y, kind, ARD, var, ls, noise, Xn)
                for f in ("lml", "grad", "K", "L", "alpha", "dL_dK", "mu", "var"):
                    put(store, key + "_" + f, r[f])

    A, B, S = _linalg_inputs()
    put(store, "linalg_jitchol_L", G.linalg.jitchol(A, maxtries=5))
    try:
        G.linalg.jitchol(A, maxtries=4)
        put(store, "linalg_jitchol_4_raises", 0.0)
    except np.linalg.LinAlgError:
        put(store, "linalg_jitchol_4_raises", 1.0)
    put(store, "linalg_tdot", G.linalg.tdot(B))
    Ai, Lr, Li, ld = G.linalg.pdinv(S)
    put(store, "linalg_pdinv_Ai", Ai)
    put(store, "linalg_pdinv_L", Lr)
    put(store, "linalg_pdinv_logdet", ld)

    k = G.RBF(10)
    for i, (tmp, A_, B_) in enumerate(_native_inputs()):
        put(store, "native_%d" % i, k._lengthscale_grads_pure(tmp, A_, B_))

    for key, name, kind, ARD, ls, X, Z, d1, d2 in _gradients_X_inputs():
        kr = getattr(G, name)(4, variance=0.9, lengthscale=ls, ARD=ARD)
        put(store, key + "_XX", kr.gradients_X(d1, X))
        put(store, key + "_XZ", kr.gradients_X(d2, X, Z))

    for kind, ARD in VARDTC_CASES:
        key, X, Y, Z, ls = _vardtc_inputs(kind, ARD)
        r = ref_gpy.evaluate_sparse(G, X, Y, Z, kind, ARD, 1.3, ls, 0.07)
        for f in ("lml", "grad", "Zgrad", "woodbury_vector", "woodbury_inv", "dL_dKnm"):
            put(store, key + "_" + f, r[f])

    for kind, ARD, P in VARDTC_HET_CASES:
        key, X, Y, Z, ls, nv = _vardtc_het_inputs(kind, ARD, P)
        r = ref_gpy.evaluate_sparse_het(G, X, Y, Z, kind, ARD, 1.3, ls, nv)
        for f in ("lml", "grad", "Zgrad", "woodbury_vector", "woodbury_inv"):
            put(store, key + "_" + f, r[f])

    for kind, ARD in HET_CASES:
        for key, X, Y, var, ls, nv in _het_inputs(kind, ARD):
            r = ref_gpy.evaluate_het(G, X, Y, kind, ARD, var, ls, nv)
            for f in ("lml", "grad", "alpha"):
                put(store, key + "_" + f, r[f])

    md, nv, sub, dd, mu, var = _mirror_het_inputs()
    ref = G.HeteroscedasticGaussian(md)
    ref.variance[:] = nv.reshape(ref.variance.shape)
    put(store, "mirror_het_gaussian_variance", np.asarray(ref.gaussian_variance(sub)).reshape(-1))
    put(store, "mirror_het_gradients", np.asarray(ref.exact_inference_gradients(dd, md)).reshape(-1))
    m0, v0 = ref.predictive_values(mu.copy(), var.copy(), False, sub)
    put(store, "mirror_het_pred_var", np.asarray(v0).reshape(-1))
    put(store, "mirror_het_pred_mu", m0)

    X, Y, idx, ls, sub, mu, var = _mixed_inputs()
    D = X.shape[1]
    r = ref_gpy.evaluate_mixed(G, X, Y, "matern52", True, 1.3, ls, MIXED_NOISE, idx)
    for f in ("lml", "grad", "alpha", "variance"):
        put(store, "mixed_" + f, r[f])
    _, g, _ = o.eval_lml_grad(X, Y, "matern52", True, 1.3, ls, np.asarray(MIXED_NOISE)[idx])
    put(store, "mixed_dn", g[1 + D:])
    put(store, "mixed_routed", np.asarray(r["likelihood"].exact_inference_gradients(g[1 + D:], r["Y_metadata"])))
    m0, v0 = r["likelihood"].predictive_values(mu.copy(), var.copy(), False, sub)
    put(store, "mixed_pred_var", np.asarray(v0).reshape(-1))
    put(store, "mixed_pred_mu", m0)

    C = ref_gpy.load_combination()
    X, X2, Y = _composite_inputs()
    D = X.shape[1]
    k_rbf = G.RBF(2, variance=1.2, lengthscale=[1.0, 2.0], ARD=True, active_dims=[0, 1])
    k_m32 = G.Matern32(2, variance=0.8, lengthscale=1.5, active_dims=[2, 3])
    k_m52 = G.Matern52(D, variance=0.5, lengthscale=np.linspace(1.5, 2.5, D), ARD=True)
    kern = C.Add([C.Prod([k_rbf, k_m32]), k_m52, C.White(D, variance=0.05), C.Bias(D, variance=0.3)])
    put(store, "composite_K", kern.K(X))
    put(store, "composite_K2", kern.K(X, X2))
    put(store, "composite_Kdiag", kern.Kdiag(X))
    post, lml, gd = G.ExactGaussianInference().inference(kern, X, G.Gaussian(variance=0.1), Y)
    kern.update_gradients_full(gd["dL_dK"], X)
    k_rbf, k_m32 = kern.parts[0].parts            # Prod copies its factors (prod.py:36-41): read the linked copies
    k_m52, k_w, k_b = kern.parts[1:]
    put(store, "composite_lml", float(lml))
    put(store, "composite_grad", np.concatenate([
        np.atleast_1d(k_rbf.variance.gradient), np.atleast_1d(k_rbf.lengthscale.gradient).reshape(-1),
        np.atleast_1d(k_m32.variance.gradient), np.atleast_1d(k_m32.lengthscale.gradient).reshape(-1),
        np.atleast_1d(k_m52.variance.gradient), np.atleast_1d(k_m52.lengthscale.gradient).reshape(-1),
        np.atleast_1d(k_w.variance.gradient), np.atleast_1d(k_b.variance.gradient), np.atleast_1d(gd["dL_dthetaL"])]))
    return G


def record_line_counts():
    """-> {path under the reference tree: number of lines} for every .py / .pyx / .c file of GPy/"""
    from oracle import ref_gpy
    counts = {}
    for dp, _, fs in os.walk(os.path.join(ref_gpy.REF, "GPy")):
        for f in fs:
            if f.endswith((".py", ".pyx", ".c")):
                p = os.path.join(dp, f)
                with open(p, errors="replace") as fh:
                    counts[os.path.relpath(p, ref_gpy.REF)] = sum(1 for _ in fh)
    return dict(sorted(counts.items()))
