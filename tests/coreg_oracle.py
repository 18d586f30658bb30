"""NumPy restatement of GPy's coregionalized regression for the tests: Coregionalize (GPy/kern/src/coregionalize.py:80-137)
inside the composite kernel of oracle/gpy_oracle.py (add.py, prod.py, static.py, stationary kernels), with one noise
variance per data point (exact_gaussian_inference.py:52-74 with a vector variance, mixed_noise.py:23-41)."""
import numpy as np

from oracle import gpy_oracle as o


class CoregOracle(object):
    """coregionalize.py:80-137: K = B[idx, idx'], Kdiag = diag(B)[idx], dL_dK -> S -> (dW, dkappa)."""

    def __init__(self, W, kappa, B=None):
        self.W, self.kappa = np.asarray(W, dtype=np.float64), np.asarray(kappa, dtype=np.float64)
        self.B = np.dot(self.W, self.W.T) + np.diag(self.kappa) if B is None else np.asarray(B, dtype=np.float64)   # :80

    def K(self, X, X2=None):
        i = np.asarray(X, dtype=int)
        j = i if X2 is None else np.asarray(X2, dtype=int)
        return self.B[i, j.T]                                                    # :88-94

    def Kdiag(self, X):
        return np.diag(self.B)[np.asarray(X, dtype=int).flatten()]              # :107-108

    def S(self, dL_dK, X, X2=None):
        """dL_dK_small, with S[a, b] = sum over rows of index a and columns of index b (:130-137 stores its transpose,
        equal for a symmetric dL_dK)"""
        i = np.asarray(X, dtype=int)[:, 0]
        j = i if X2 is None else np.asarray(X2, dtype=int)[:, 0]
        O = self.B.shape[0]
        S = np.zeros((O, O))
        for a in range(O):
            rows = dL_dK[i == a]
            for b in range(O):
                S[a, b] = rows[:, j == b].sum()
        return S

    def grads_from_S(self, S):
        """:123-128 -> (dW, dkappa)"""
        dkappa = np.diag(S).copy()
        S = S + S.T
        return (self.W[:, None, :] * S[:, :, None]).sum(0), dkappa

    def update_gradients_full(self, dL_dK, X, X2=None):
        dW, dk = self.grads_from_S(self.S(dL_dK, X, X2))
        return dW, dk


def kparts(parts):
    """parts: dicts as oracle.gpy_oracle.composite_parts takes, plus {"kind": "coregionalize", "dims": [col], "W", "kappa"}"""
    out = []
    for p in parts:
        if p["kind"] == "coregionalize":
            out.append((CoregOracle(p.get("W", np.zeros((0, 0))), p.get("kappa", np.zeros(0)), p.get("B")),
                        np.asarray(p["dims"]), p["term"]))
        else:
            out.extend(o.composite_parts([p]))
    return out


def K(parts, X, X2=None):
    return o.composite_K(kparts(parts), X, X2)


def Kdiag(parts, X):
    return o.composite_Kdiag(kparts(parts), X)


def eval_lml_grad(X, Y, parts, noise):
    """One GP.parameters_changed(): noise is a float or N per-point variances; a coregionalization part is given by W and
    kappa, or by B alone (then only res["device_grad"] is meaningful for it).
    -> (lml, grad, res): grad = per part [variance, lengthscale..] or [W (row-major), kappa], then tr(dL_dK);
    res["device_grad"] = the same with S (row-major) for a coregionalization part (gpx_exact_eval_coreg's layout);
    res["dnoise"] = diag(dL_dK)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    Y = np.ascontiguousarray(Y, dtype=np.float64)
    kp = kparts(parts)
    Kx = o.composite_K(kp, X)
    Ky = Kx.copy()
    o.diag_add(Ky, np.asarray(noise, dtype=np.float64) + 1e-8)
    Wi, LW, LWi, W_logdet = o.pdinv(Ky)
    alpha, _ = o.dpotrs(LW, Y, lower=1)
    lml = 0.5 * (-Y.size * np.log(2 * np.pi) - Y.shape[1] * W_logdet - np.sum(alpha * Y))
    dL_dK = 0.5 * (o.tdot(alpha) - Y.shape[1] * Wi)
    grad, dev, S_list = [], [], []
    for i, (k, dims, t) in enumerate(kp):
        other = None
        for j, (k2, dims2, t2) in enumerate(kp):
            if j != i and t2 == t:
                Kj = k2.K(o._slice(X, dims2))
                other = Kj if other is None else other * Kj
        g = dL_dK if other is None else dL_dK * other
        if isinstance(k, CoregOracle):
            S = k.S(g, o._slice(X, dims))
            S_list.append(S)
            dev.append(S.reshape(-1))
            if k.W.size:
                dW, dk = k.grads_from_S(S)
                grad.append(np.concatenate([dW.reshape(-1), dk]))
        else:
            dv, dl = k.update_gradients_full(g, o._slice(X, dims), None)
            grad.append(np.concatenate([[dv], np.atleast_1d(dl).reshape(-1)]))
            dev.append(grad[-1])
    grad.append([np.trace(dL_dK)])
    dev.append([np.trace(dL_dK)])
    return float(lml), np.concatenate(grad), dict(L=LW, alpha=alpha, K=Kx, Wi=Wi, dL_dK=dL_dK, S=S_list,
                                                  dnoise=np.diag(dL_dK).copy(), device_grad=np.concatenate(dev))



def predict(parts, X, L, alpha, Xnew, full_cov=False):
    """posterior.py:273-302 with the composite kernel (noise-free)"""
    from scipy.linalg import solve_triangular
    kp = kparts(parts)
    Kx = o.composite_K(kp, X, Xnew)
    mu = Kx.T.dot(alpha)
    tmp = solve_triangular(L, Kx, lower=True)
    if full_cov:
        return mu, o.composite_K(kp, Xnew) - tmp.T.dot(tmp)
    return mu, (o.composite_Kdiag(kp, Xnew) - np.square(tmp).sum(0))[:, None]


def per_output(dnoise, index, O):
    """mixed_noise.py:38-41"""
    index = np.asarray(index).reshape(-1)
    return np.array([dnoise[index == j].sum() for j in range(O)])


def fixture_eval(f):
    """evaluate a tests/golden/coreg fixture with the restatement -> (lml, model gradient in paramz order, res)"""
    import json
    parts = json.loads(str(f["parts"]))
    idx = np.asarray(f["output_index"]).reshape(-1)
    noise = np.asarray(f["noise"])
    lml, g, res = eval_lml_grad(f["X"], f["Y"], parts, noise[idx])
    grad = np.concatenate([g[:-1], per_output(res["dnoise"], idx, noise.size)])
    return lml, grad, res, parts


def device_parts(parts):
    """parts dicts -> Engine.exact_eval_coreg descriptors"""
    out = []
    for p in parts:
        if p["kind"] == "coregionalize":
            W, kappa = np.asarray(p["W"]), np.asarray(p["kappa"])
            out.append(("coregionalize", False, p["term"], p["dims"], 1.0, np.dot(W, W.T) + np.diag(kappa)))
        elif p["kind"] in ("white", "bias"):
            out.append((p["kind"], False, p["term"], [], p["variance"], None))
        else:
            out.append((p["kind"], p.get("ARD", False), p["term"], p["dims"], p["variance"], p["lengthscale"]))
    return out
