"""Generates tests/golden/*.npz. Run in the build container (has /root/reference):  python tests/golden/make_golden.py

Source of the numbers:
  * if the unmodified reference can be imported (GPy from /root/reference through the test-only paramz stand-in in
    oracle/paramz_shim), every fixture is produced by the REFERENCE ITSELF — GPy.models.GPRegression(...):
    m.log_likelihood(), m.gradient, posterior.woodbury_vector, m.predict — and the oracle is asserted against it here;
  * otherwise by the oracle restatement (fixtures then carry source='oracle').
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import gpy_oracle as o  # noqa: E402

CASES = [
    # name, kind, ARD, N, D, seed
    ("rbf_iso_n512_d2", "rbf", False, 512, 2, 0),          # BASELINE.json configs[0]
    ("rbf_ard_n300_d8", "rbf", True, 300, 8, 1),
    ("matern52_ard_n257_d5", "matern52", True, 257, 5, 2),
    ("matern32_iso_n128_d3", "matern32", False, 128, 3, 3),
    ("exponential_ard_n200_d4", "exponential", True, 200, 4, 4),
    ("rbf_ard_n1100_d8", "rbf", True, 1100, 8, 5),
    ("matern52_iso_n40_d1", "matern52", False, 40, 1, 6),
]


def try_reference():
    try:
        from oracle import ref_gpy
        return ref_gpy.load()
    except Exception as e:  # noqa: BLE001
        print("reference not importable (%r): fixtures come from the oracle" % (e,))
        return None


def main():
    GPy = try_reference()
    for name, kind, ARD, N, D, seed in CASES:
        X, Y = o.synthetic(N, D, seed)
        rng = np.random.default_rng(100 + seed)
        var = float(rng.uniform(0.5, 2.0))
        ls = np.sqrt(D) * rng.uniform(0.6, 1.5, D) if ARD else float(np.sqrt(D) * rng.uniform(0.6, 1.5))
        noise = float(rng.uniform(0.005, 0.1))
        Xn = rng.uniform(-3, 3, (7, D))
        lml, grad, res = o.eval_lml_grad(X, Y, kind, ARD, var, ls, noise)
        kern = o.StationaryOracle(kind, D, var, ls, ARD)
        mu, pv = o.predict(kern, X, res["L"], res["alpha"], Xn, noise)
        source = "oracle"
        if GPy is not None:
            from oracle import ref_gpy
            r = ref_gpy.evaluate(GPy, X, Y, kind, ARD, var, ls, noise, Xn)
            assert abs(r["lml"] - lml) <= 1e-9 * max(1, abs(lml)), (name, r["lml"], lml)
            np.testing.assert_allclose(r["grad"], grad, rtol=1e-8, atol=1e-10, err_msg=name)
            np.testing.assert_allclose(r["alpha"], res["alpha"], rtol=1e-7, atol=1e-10, err_msg=name)
            np.testing.assert_allclose(r["mu"], mu, rtol=1e-8, atol=1e-10, err_msg=name)
            np.testing.assert_allclose(r["var"], pv, rtol=1e-7, atol=1e-10, err_msg=name)
            lml, grad, alpha, mu, pv = r["lml"], r["grad"], r["alpha"], r["mu"], r["var"]
            source = "GPy %s (unmodified /root/reference via oracle/paramz_shim)" % GPy.__version__
        else:
            alpha = res["alpha"]
        np.savez_compressed(os.path.join(HERE, name + ".npz"), X=X, Y=Y, kind=kind, ARD=ARD, variance=var,
                            lengthscale=ls, noise=noise, lml=lml, grad=grad, alpha=alpha, Xnew=Xn, mu=mu, var=pv,
                            source=source)
        print("%-28s lml %.10f source %s" % (name, lml, source))


HET_CASES = [("het_matern32_ard_n150_d3", "matern32", True, 150, 3, 11), ("het_rbf_iso_n260_d2", "rbf", False, 260, 2, 12)]


def main_het():
    """tests/golden/het/*.npz: one noise variance per data point (GPHeteroscedasticRegression), produced by the
    reference's own HeteroscedasticGaussian + ExactGaussianInference objects when importable."""
    GPy = try_reference()
    os.makedirs(os.path.join(HERE, "het"), exist_ok=True)
    for name, kind, ARD, N, D, seed in HET_CASES:
        X, Y = o.synthetic(N, D, seed)
        rng = np.random.default_rng(100 + seed)
        var = float(rng.uniform(0.5, 2.0))
        ls = np.sqrt(D) * rng.uniform(0.6, 1.5, D) if ARD else float(np.sqrt(D) * rng.uniform(0.6, 1.5))
        nv = rng.uniform(0.005, 0.3, N)
        lml, grad, res = o.eval_lml_grad(X, Y, kind, ARD, var, ls, nv)
        alpha, source = res["alpha"], "oracle"
        if GPy is not None:
            from oracle import ref_gpy
            r = ref_gpy.evaluate_het(GPy, X, Y, kind, ARD, var, ls, nv)
            assert abs(r["lml"] - lml) <= 1e-9 * max(1, abs(lml)), (name, r["lml"], lml)
            np.testing.assert_allclose(r["grad"], grad, rtol=1e-8, atol=1e-10, err_msg=name)
            lml, grad, alpha = r["lml"], r["grad"], r["alpha"]
            source = "GPy %s (unmodified /root/reference via oracle/paramz_shim)" % GPy.__version__
        np.savez_compressed(os.path.join(HERE, "het", name + ".npz"), X=X, Y=Y, kind=kind, ARD=ARD, variance=var,
                            lengthscale=ls, noise_variances=nv, lml=lml, grad=grad, alpha=alpha, source=source)
        print("%-28s lml %.10f source %s" % (name, lml, source))


SPARSE_CASES = [("sparse_rbf_ard_n400_m50_d3", "rbf", True, 400, 50, 3, 21), ("sparse_matern52_iso_n333_m129_d2", "matern52", False, 333, 129, 2, 22)]


def main_sparse():
    """tests/golden/sparse/*.npz: SparseGPRegression (VarDTC) bound, gradients and inducing-input gradients produced by
    the reference's own VarDTC + kernel + Gaussian objects (gradient wiring of core/sparse_gp.py:108-119)."""
    GPy = try_reference()
    os.makedirs(os.path.join(HERE, "sparse"), exist_ok=True)
    for name, kind, ARD, N, M, D, seed in SPARSE_CASES:
        rng = np.random.default_rng(100 + seed)
        X = rng.uniform(-3, 3, (N, D))
        Y = np.sin(X).sum(1, keepdims=True) / np.sqrt(D) + 0.1 * rng.standard_normal((N, 1))
        Z = X[rng.permutation(N)[:M]].copy() + 0.01 * rng.standard_normal((M, D))
        var = float(rng.uniform(0.5, 2.0))
        ls = np.sqrt(D) * rng.uniform(0.6, 1.5, D) if ARD else float(np.sqrt(D) * rng.uniform(0.6, 1.5))
        noise = float(rng.uniform(0.01, 0.1))
        lml, grad, Zg, res = o.sparse_eval(X, Y, Z, kind, ARD, var, ls, noise)
        wv, source = res["woodbury_vector"], "oracle"
        if GPy is not None:
            from oracle import ref_gpy
            r = ref_gpy.evaluate_sparse(GPy, X, Y, Z, kind, ARD, var, ls, noise)
            assert abs(r["lml"] - lml) <= 1e-8 * max(1, abs(lml)), (name, r["lml"], lml)
            np.testing.assert_allclose(r["grad"], grad, rtol=1e-6, atol=1e-8, err_msg=name)
            np.testing.assert_allclose(r["Zgrad"], Zg, rtol=1e-6, atol=1e-8, err_msg=name)
            lml, grad, Zg, wv = r["lml"], r["grad"], r["Zgrad"], r["woodbury_vector"]
            source = "GPy %s (unmodified /root/reference via oracle/paramz_shim)" % GPy.__version__
        np.savez_compressed(os.path.join(HERE, "sparse", name + ".npz"), X=X, Y=Y, Z=Z, kind=kind, ARD=ARD, variance=var,
                            lengthscale=ls, noise=noise, lml=lml, grad=grad, Zgrad=Zg, woodbury_vector=wv, source=source)
        print("%-36s lml %.10f source %s" % (name, lml, source))


SPARSE_HET_CASES = [("sparse_het_rbf_ard_n300_m40_d3", "rbf", True, 300, 40, 3, 1, 31),
                    ("sparse_het_matern32_iso_n450_m130_d2", "matern32", False, 450, 130, 2, 1, 32)]


def main_sparse_het():
    """tests/golden/sparse_het/*.npz: VarDTC with one noise variance per data point (the het_noise branches
    var_dtc.py:127-128,221-227,241-257,267-269), produced by the reference's own VarDTC + HeteroscedasticGaussian."""
    GPy = try_reference()
    os.makedirs(os.path.join(HERE, "sparse_het"), exist_ok=True)
    for name, kind, ARD, N, M, D, P, seed in SPARSE_HET_CASES:
        rng = np.random.default_rng(100 + seed)
        X = rng.uniform(-3, 3, (N, D))
        Y = np.sin(X).sum(1, keepdims=True) / np.sqrt(D) + 0.1 * rng.standard_normal((N, P))
        Z = X[rng.permutation(N)[:M]].copy() + 0.01 * rng.standard_normal((M, D))
        var = float(rng.uniform(0.5, 2.0))
        ls = np.sqrt(D) * rng.uniform(0.6, 1.5, D) if ARD else float(np.sqrt(D) * rng.uniform(0.6, 1.5))
        nv = rng.uniform(0.01, 0.3, N)
        lml, grad, Zg, res = o.sparse_eval(X, Y, Z, kind, ARD, var, ls, nv)
        wv, wi, source = res["woodbury_vector"], res["woodbury_inv"], "oracle"
        if GPy is not None:
            from oracle import ref_gpy
            r = ref_gpy.evaluate_sparse_het(GPy, X, Y, Z, kind, ARD, var, ls, nv)
            assert abs(r["lml"] - lml) <= 1e-8 * max(1, abs(lml)), (name, r["lml"], lml)
            np.testing.assert_allclose(r["grad"], grad, rtol=1e-6, atol=1e-7, err_msg=name)
            np.testing.assert_allclose(r["Zgrad"], Zg, rtol=1e-6, atol=1e-7, err_msg=name)
            lml, grad, Zg, wv, wi = r["lml"], r["grad"], r["Zgrad"], r["woodbury_vector"], r["woodbury_inv"]
            source = "GPy %s (unmodified /root/reference via oracle/paramz_shim)" % GPy.__version__
        np.savez_compressed(os.path.join(HERE, "sparse_het", name + ".npz"), X=X, Y=Y, Z=Z, kind=kind, ARD=ARD, variance=var,
                            lengthscale=ls, noise_variances=nv, lml=lml, grad=grad, Zgrad=Zg, woodbury_vector=wv,
                            woodbury_inv=wi, source=source)
        print("%-40s lml %.10f source %s" % (name, lml, source))


def main_reference():
    """tests/golden/reference/: what the reference computes for the inputs of tests/test_reference_crosscheck.py, and the
    line count of each of its source files (the GPy/...:line citations of include/gpx.h and INTEGRATION.md are checked
    against it). Needs the reference (GPX_REFERENCE)."""
    import json
    sys.path.insert(0, os.path.dirname(HERE))
    import test_reference_crosscheck as t
    out = os.path.join(HERE, "reference")
    os.makedirs(out, exist_ok=True)
    store = {}
    G = t.record_reference(store)
    source = "GPy %s (unmodified, via oracle/paramz_shim)" % G.__version__
    np.savez_compressed(os.path.join(out, "crosscheck.npz"), source=source, **t.pack(store))
    with open(os.path.join(out, "gpy_line_counts.json"), "w") as f:
        json.dump(t.record_line_counts(), f, indent=0)
        f.write("\n")
    print("reference numbers of %d arrays, source %s" % (len(store), source))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "sparse_het":   # only the fixtures added last (the others stay byte-identical)
        main_sparse_het()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "reference":    # the crosscheck numbers only
        main_reference()
        sys.exit(0)
    main()
    main_het()
    main_sparse()
    main_sparse_het()
