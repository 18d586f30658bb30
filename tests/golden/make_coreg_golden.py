"""Writes tests/golden/coreg/*.npz: multi-output (coregionalized) regression evaluated by the UNMODIFIED reference GPy
objects (GPCoregionalizedRegression / GP, Prod, Add, Coregionalize, MixedNoise, util.multioutput ICM / LCM), loaded by
oracle/ref_gpy.py. Run from the repository root: python tests/golden/make_coreg_golden.py

Each file holds the inputs (X with the output index as last column, Y, output_index), the parameters, the kernel spec as
JSON (`parts`, the layout tests/coreg_oracle.py takes), the log marginal likelihood, the model gradient in paramz order,
alpha, and predictions at Xnew (noise-free mean / variance / full covariance and the variance with the likelihood)."""
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "coreg")


def load_reference():
    """oracle.ref_gpy's loaders plus the three names the multi-output modules take from their stub packages."""
    from oracle import ref_gpy as R
    G = R.load()
    C = R.load_combination()
    M = R.load_models()
    sys.modules["GPy.util"].multioutput = importlib.import_module("GPy.util.multioutput")
    sys.modules["GPy.kern"].Coregionalize = importlib.import_module("GPy.kern.src.coregionalize").Coregionalize
    sys.modules["GPy.likelihoods"].mixed_noise = importlib.import_module("GPy.likelihoods.mixed_noise")
    gcr = importlib.import_module("GPy.models.gp_coregionalized_regression")
    return G, C, M, sys.modules["GPy.util"].multioutput, gcr.GPCoregionalizedRegression, R


def data(O, D, n_per, seed):
    rng = np.random.RandomState(seed)
    Xl = [rng.uniform(-2, 2, (n_per + j, D)) for j in range(O)]
    Yl = [np.sin(x.sum(1, keepdims=True) * (1 + 0.3 * j)) + 0.2 * j + 0.1 * rng.randn(x.shape[0], 1)
          for j, x in enumerate(Xl)]
    return Xl, Yl, rng


def record(name, m, parts, X, Y, idx, Xnew, idx_new, mo_meta, source):
    mu, var = m.predict(Xnew, Y_metadata={"output_index": idx_new})
    mu0, var0 = m.predict(Xnew, include_likelihood=False)
    _, cov0 = m.predict(Xnew, full_cov=True, include_likelihood=False)
    os.makedirs(OUT, exist_ok=True)
    np.savez(os.path.join(OUT, name + ".npz"), X=X, Y=Y, output_index=idx, parts=json.dumps(parts),
             lml=float(m.log_likelihood()), grad=np.asarray(m.gradient, dtype=np.float64).copy(),
             alpha=np.asarray(m.posterior.woodbury_vector), Xnew=Xnew, output_index_new=idx_new, mu=np.asarray(mu),
             var=np.asarray(var), mu_noiseless=np.asarray(mu0), var_noiseless=np.asarray(var0), cov_noiseless=np.asarray(cov0),
             noise=np.asarray(mo_meta), source=source)
    print(name, "lml %.12f" % float(m.log_likelihood()), "ngrad", np.asarray(m.gradient).size)


def main():
    G, C, M, mo, GPCR, R = load_reference()
    src = "GPy %s (unmodified reference), make_coreg_golden.py" % G.__version__
    # ICM: O = 3 outputs, rank 2, RBF-ARD on D = 2; rows grouped by output as build_XY makes them
    O, D = 3, 2
    Xl, Yl, rng = data(O, D, 24, seed=11)
    W = 0.6 * rng.randn(O, 2)
    kappa = np.array([0.4, 0.7, 0.3])
    ls = np.array([0.9, 1.4])
    k = mo.ICM(input_dim=D, num_outputs=O, kernel=G.RBF(D, variance=1.3, lengthscale=ls, ARD=True), W_rank=2, W=W,
               kappa=kappa)
    m = GPCR(Xl, Yl, kernel=k)
    noise = [0.05, 0.11, 0.08]
    for j, v in enumerate(noise):
        m.likelihood.likelihoods_list[j].variance[:] = v
    X, Y, idx = np.asarray(m.X), np.asarray(m.Y), np.asarray(m.output_index)
    Xn = rng.uniform(-2, 2, (9, D))
    idx_new = (np.arange(9) % O)[:, None]
    Xnew = np.hstack([Xn, idx_new])
    parts = [dict(kind="rbf", term=0, dims=list(range(D)), variance=1.3, lengthscale=ls.tolist(), ARD=True),
             dict(kind="coregionalize", term=0, dims=[D], W=W.tolist(), kappa=kappa.tolist())]
    record("icm_o3_r2_rbf_ard_n75_d2", m, parts, X, Y, idx, Xnew, idx_new, noise, src + " GPCoregionalizedRegression")

    # the same ICM with the rows shuffled across outputs: GP + MixedNoise with Y_metadata (gp_coregionalized_regression.py:46)
    perm = np.random.RandomState(3).permutation(X.shape[0])
    k2 = mo.ICM(input_dim=D, num_outputs=O, kernel=G.RBF(D, variance=1.3, lengthscale=ls, ARD=True), W_rank=2, W=W,
                kappa=kappa)
    lik = mo.build_likelihood(Yl, idx[perm])
    for j, v in enumerate(noise):
        lik.likelihoods_list[j].variance[:] = v
    m2 = M.GP(X[perm], Y[perm], k2, lik, Y_metadata={"output_index": idx[perm]})
    record("icm_o3_r2_rbf_ard_n75_d2_shuffled", m2, parts, X[perm], Y[perm], idx[perm], Xnew, idx_new, noise,
           src + " GP + MixedNoise, shuffled rows")

    # LCM: RBF (iso) and Matern32 (ARD) each times its own Coregionalize (rank 1), plus a Bias term; O = 2, shuffled rows
    O, D = 2, 3
    Xl, Yl, rng = data(O, D, 40, seed=12)
    W0, W1 = np.array([[0.8], [-0.5]]), np.array([[0.3], [0.9]])
    k0, k1 = np.array([0.2, 0.5]), np.array([0.6, 0.1])
    ls1 = np.array([1.1, 0.7, 1.9])
    kern = (mo.ICM(D, O, G.RBF(D, variance=0.9, lengthscale=1.2), W_rank=1, W=W0, kappa=k0, name="ICM0")
            + mo.ICM(D, O, G.Matern32(D, variance=0.6, lengthscale=ls1, ARD=True), W_rank=1, W=W1, kappa=k1, name="ICM1")
            + C.Bias(D + 1, variance=0.35))
    X, Y, idx = mo.build_XY(Xl, Yl)
    perm = np.random.RandomState(4).permutation(X.shape[0])
    X, Y, idx = X[perm], Y[perm], idx[perm]
    lik = mo.build_likelihood(Yl, idx)
    noise = [0.07, 0.04]
    for j, v in enumerate(noise):
        lik.likelihoods_list[j].variance[:] = v
    m3 = M.GP(X, Y, kern, lik, Y_metadata={"output_index": idx})
    Xn = rng.uniform(-2, 2, (8, D))
    idx_new = (np.arange(8) % O)[:, None]
    Xnew = np.hstack([Xn, idx_new])
    parts = [dict(kind="rbf", term=0, dims=list(range(D)), variance=0.9, lengthscale=[1.2], ARD=False),
             dict(kind="coregionalize", term=0, dims=[D], W=W0.tolist(), kappa=k0.tolist()),
             dict(kind="matern32", term=1, dims=list(range(D)), variance=0.6, lengthscale=ls1.tolist(), ARD=True),
             dict(kind="coregionalize", term=1, dims=[D], W=W1.tolist(), kappa=k1.tolist()),
             dict(kind="bias", term=2, variance=0.35)]
    record("lcm_o2_rbf_matern32_bias_n81_d3_shuffled", m3, parts, X, Y, idx, Xnew, idx_new, noise,
           src + " GP + Add(ICM, ICM, Bias) + MixedNoise, shuffled rows")


if __name__ == "__main__":
    main()
