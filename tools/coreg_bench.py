"""Times the fused multi-output (coregionalized) evaluation on one GPU against the single-kernel evaluation of the same run,
and the host route it replaces (_generic_inference: K as host arrays, gpx_pdinv, NumPy algebra) at N = 4096.

Workload (inputs from --seed): ICM with RBF-ARD on D = 8 inputs, O = 4 outputs, rank 2, MixedNoise (one variance per
output), rows in random output order. Single kernel: RBF-ARD on the same inputs, scalar noise. The fused outputs are checked
against the NumPy restatement (tests/coreg_oracle.py) at N = 4096 before any timing.
    python tools/coreg_bench.py [--sizes 4096 16384] [--reps 10] [--seed 0]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def workload(N, D, O, seed):
    rng = np.random.default_rng(seed + N)
    Xi = rng.uniform(-3, 3, (N, D))
    idx = rng.integers(0, O, N)
    Y = (np.sin(Xi).sum(1) / np.sqrt(D) * (1 + 0.3 * idx) + 0.1 * rng.standard_normal(N))[:, None]
    X = np.hstack([Xi, idx[:, None].astype(np.float64)])
    ls = rng.uniform(0.8, 2.0, D)
    W = 0.6 * rng.standard_normal((O, 2))
    kappa = rng.uniform(0.2, 0.8, O)
    noise = rng.uniform(0.02, 0.1, O)
    parts = [dict(kind="rbf", term=0, dims=list(range(D)), variance=1.3, lengthscale=ls.tolist(), ARD=True),
             dict(kind="coregionalize", term=0, dims=[D], W=W.tolist(), kappa=kappa.tolist())]
    return X, Y, idx, parts, noise, ls


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()                      # every engine call ends in a device synchronise before it returns
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, float(np.min(ts)) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import coreg_oracle as co
    import gpy_b200
    from gpy_b200 import _ffi
    from gpy_b200.inference import ExactGaussianInference
    D, O = 8, 4
    res = dict(card=card(), workload="ICM RBF-ARD D=8 O=4 rank 2 MixedNoise", reps=a.reps, seed=a.seed, rows=[])
    print("card, power limit:", res["card"])
    eng = _ffi.Engine(0)
    for N in a.sizes:
        X, Y, idx, parts, noise, ls = workload(N, D, O, a.seed)
        desc = co.device_parts(parts)
        nv = noise[idx]
        eng.set_data(X, Y)
        if N == 4096:
            lml, g, dn, _ = eng.exact_eval_coreg(desc, nv)
            lml0, _, r0 = co.eval_lml_grad(X, Y, parts, nv)
            err_l = abs(lml - lml0)
            err_g = float(np.max(np.abs(g - r0["device_grad"]) / np.maximum(np.abs(r0["device_grad"]), 1e-12)))
            err_n = float(np.max(np.abs(co.per_output(dn, idx, O) - co.per_output(r0["dnoise"], idx, O))
                                 / np.abs(co.per_output(r0["dnoise"], idx, O))))
            print("N=%d check vs restatement: |dLML| %.2e  grad max rel %.2e  noise grad max rel %.2e" % (N, err_l, err_g, err_n))
            res["check_n4096"] = dict(dlml=err_l, grad_rel=err_g, noise_rel=err_n)
            assert err_l <= 1e-8 and err_g <= 1e-6 and err_n <= 1e-6, "fused result differs from the restatement"
        t_co = timed(lambda: eng.exact_eval_coreg(desc, nv), a.reps)
        st = eng.stats()
        Xs = np.ascontiguousarray(X[:, :D])
        eng.set_data(Xs, Y)
        t_one = timed(lambda: eng.exact_eval("rbf", True, 1.3, ls, 0.05), a.reps)
        row = dict(N=N, coreg_ms_median=t_co[0], coreg_ms_min=t_co[1], single_ms_median=t_one[0], single_ms_min=t_one[1],
                   overhead_pct=100.0 * (t_co[0] / t_one[0] - 1.0), coreg_device_total_ms=st["total_ms"],
                   coreg_grad_ms=st["lauum_ms"])
        if N == 4096:
            m = gpy_b200.GPCoregionalizedRegression.__new__(gpy_b200.GPCoregionalizedRegression)
            inf = ExactGaussianInference(engine=eng)
            k = gpy_b200.ICM(D, O, gpy_b200.RBF(D, variance=1.3, lengthscale=ls, ARD=True), W_rank=2,
                             W=np.asarray(parts[1]["W"]), kappa=np.asarray(parts[1]["kappa"]))
            liks = [gpy_b200.Gaussian(variance=float(v)) for v in noise]
            lik = gpy_b200.MixedNoise(liks)
            meta = {"output_index": idx[:, None]}
            row["generic_ms_median"], row["generic_ms_min"] = timed(
                lambda: inf._generic_inference(k, X, Y, lik.gaussian_variance(meta), None, None, None, lik, meta), max(3, a.reps // 3))
        res["rows"].append(row)
        print(json.dumps(row))
        eng.set_data(X[:256], Y[:256])          # release nothing big between sizes; the next set_data resizes
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
