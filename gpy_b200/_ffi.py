"""ctypes binding of libgpx.so (C ABI: include/gpx.h). The CUDA library is the product: if it is missing or
cannot be loaded this module raises — there is NO CPU fallback anywhere in gpy_b200."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libgpx.so")

KIND = {"rbf": 0, "exponential": 1, "matern32": 2, "matern52": 3, "white": 4, "bias": 5, "coregionalize": 6}
GET = {"L": 0, "alpha": 1, "Kinv": 2, "dL_dK": 3, "K": 4, "Linv": 5}

_dp = ctypes.POINTER(ctypes.c_double)
_vp = ctypes.c_void_p


class GpxStats(ctypes.Structure):
    _fields_ = [("total_ms", ctypes.c_float), ("kbuild_ms", ctypes.c_float), ("sweep_ms", ctypes.c_float),
                ("update_ms", ctypes.c_float), ("lauum_ms", ctypes.c_float), ("solve_ms", ctypes.c_float),
                ("update_flops", ctypes.c_double), ("lauum_flops", ctypes.c_double), ("kbuild_bytes", ctypes.c_double),
                ("launches", ctypes.c_int64), ("update_launches", ctypes.c_int32), ("tries", ctypes.c_int32),
                ("update_int8_ops", ctypes.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class GpxKernPart(ctypes.Structure):
    """gpx_kern_part of include/gpx.h: one factor of a composite kernel."""
    _fields_ = [("kind", ctypes.c_int), ("ard", ctypes.c_int), ("term", ctypes.c_int), ("ndims", ctypes.c_int),
                ("dims", ctypes.POINTER(ctypes.c_int)), ("variance", ctypes.c_double), ("lengthscale", _dp)]


class GpxCoreg(ctypes.Structure):
    """gpx_coreg of include/gpx.h: output_dim and B of one coregionalization part."""
    _fields_ = [("output_dim", ctypes.c_int), ("B", _dp)]


EXPORTS = {
    # name: (restype, argtypes)
    "gpx_last_error": (ctypes.c_char_p, []),
    "gpx_version": (ctypes.c_char_p, []),
    "gpx_device_count": (ctypes.c_int, []),
    "gpx_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_vp)]),
    "gpx_destroy": (ctypes.c_int, [_vp]),
    "gpx_set_data": (ctypes.c_int, [_vp, _dp, ctypes.c_int64, ctypes.c_int, _dp, ctypes.c_int]),
    "gpx_exact_eval": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, ctypes.c_double,
                                      ctypes.c_double, ctypes.c_int, _dp, _dp, _dp]),
    "gpx_exact_eval_het": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_double,
                                          ctypes.c_int, _dp, _dp, _dp, _dp]),
    "gpx_exact_eval_multi": (ctypes.c_int, [_vp, ctypes.POINTER(GpxKernPart), ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                            ctypes.c_int, _dp, _dp, _dp]),
    "gpx_exact_eval_coreg": (ctypes.c_int, [_vp, ctypes.POINTER(GpxKernPart), ctypes.c_int, ctypes.POINTER(GpxCoreg),
                                            ctypes.c_double, _dp, ctypes.c_double, ctypes.c_int, _dp, _dp, _dp, _dp]),
    "gpx_get": (ctypes.c_int, [_vp, ctypes.c_int, _dp]),
    "gpx_predict": (ctypes.c_int, [_vp, _dp, ctypes.c_int64, ctypes.c_int, _dp, _dp]),
    "gpx_kern_K": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_int64, _dp,
                                  ctypes.c_int64, ctypes.c_int, _dp]),
    "gpx_kern_Kdiag": (ctypes.c_int, [ctypes.c_int, ctypes.c_double, ctypes.c_int64, _dp]),
    "gpx_kern_grad_full": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_int64,
                                          _dp, ctypes.c_int64, ctypes.c_int, _dp, _dp, _dp]),
    "gpx_kern_grad_X": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_int64, _dp,
                                       ctypes.c_int64, ctypes.c_int, _dp, _dp]),
    "gpx_sparse_set_data": (ctypes.c_int, [_vp, _dp, ctypes.c_int64, ctypes.c_int, _dp, ctypes.c_int]),
    "gpx_sparse_eval": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_int64,
                                       ctypes.c_double, _dp, _dp, _dp]),
    "gpx_sparse_get": (ctypes.c_int, [_vp, ctypes.c_int, _dp]),
    "gpx_sparse_eval_het": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_double, _dp, _dp, ctypes.c_int64,
                                           _dp, _dp, _dp, _dp, _dp]),
    "gpx_pdinv": (ctypes.c_int, [_vp, _dp, ctypes.c_int64, ctypes.c_int, _dp, _dp, _dp, _dp, _dp]),
    "gpx_get_stats": (ctypes.c_int, [_vp, ctypes.POINTER(GpxStats)]),
    "gpx_total_launches": (ctypes.c_int64, [_vp]),
    "gpx_measure_fp64_peak": (ctypes.c_int, [_vp, _dp]),
    "gpx_set_option": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_int64]),
    "gpx_comm_unique_id": (ctypes.c_int, [ctypes.c_char_p]),
    "gpx_comm_init": (ctypes.c_int, [_vp, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]),
}

_lib = None


def lib():
    """Load libgpx.so (once). Raises RuntimeError if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("gpy_b200: CUDA library %s not built (run `python -c 'import __graft_entry__ as g; "
                               "g.build()'` or `make -C gpy_b200/csrc`); there is no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


class GpxError(RuntimeError):
    pass


class GpxArgumentError(GpxError, ValueError):
    """rc == -2: an argument outside its domain (variance / lengthscale <= 0 or NaN, bad shapes). It is a ValueError so
    that an optimizer loop counts it as a failed evaluation the way paramz does (a Logexp underflow to exactly 0 or a
    NaN iterate must not abort `optimize()`), and still a GpxError for callers that catch the library's own class."""


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def check(rc, what):
    """rc < 0: CUDA/argument error -> GpxError; rc > 0: not positive definite -> numpy.linalg.LinAlgError, the class
    GPy raises from jitchol (GPy/util/linalg.py:64,75)."""
    if rc == 0:
        return
    msg = lib().gpx_last_error().decode()
    if rc > 0:
        raise np.linalg.LinAlgError("not positive definite, even with jitter. (leading minor %d)" % rc)
    if rc == -2:
        raise GpxArgumentError("%s: %s" % (what, msg))
    raise GpxError("%s failed (%d): %s" % (what, rc, msg))


def _theta(kind, ARD, lengthscale, D):
    ls = _f64(np.atleast_1d(lengthscale)).reshape(-1)
    if ARD:
        if ls.size != D:
            raise ValueError("ARD lengthscale must have %d entries" % D)
    elif ls.size != 1:
        raise ValueError("isotropic lengthscale must be a scalar")
    return KIND[kind], int(bool(ARD)), ls


class Engine(object):
    """One device context (gpx_ctx): owns the HBM-resident X, Y and the N x N factor workspace of one model."""

    def __init__(self, device=0):
        self._h = _vp()
        self._L = lib()
        check(self._L.gpx_create(int(device), ctypes.byref(self._h)), "gpx_create")
        self.N = self.D = self.P = 0
        self.device = device
        self.eval_serial = 0      # bumped by every evaluation: lazy posterior views check it before fetching

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.gpx_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name, value):
        check(self._L.gpx_set_option(self._h, name.encode(), int(value)), "gpx_set_option")

    def set_data(self, X, Y):
        X, Y = _f64(X), _f64(Y)
        if X.ndim != 2 or Y.ndim != 2 or X.shape[0] != Y.shape[0]:
            raise ValueError("X must be N x D and Y N x P")
        self.N, self.D = X.shape
        self.P = Y.shape[1]
        self.eval_serial += 1
        check(self._L.gpx_set_data(self._h, _ptr(X), self.N, self.D, _ptr(Y), self.P), "gpx_set_data")

    def exact_eval(self, kind, ARD, variance, lengthscale, noise, jitter=1e-8, max_tries=5):
        """-> (log_marginal, gradient[variance, lengthscale.., noise], extra_jitter_used)"""
        k, a, ls = _theta(kind, ARD, lengthscale, self.D)
        lml = ctypes.c_double()
        jit = ctypes.c_double()
        grad = np.zeros(ls.size + 2)
        rc = self._L.gpx_exact_eval(self._h, k, a, float(variance), _ptr(ls), float(noise), float(jitter), int(max_tries),
                                    ctypes.byref(lml), _ptr(grad), ctypes.byref(jit))
        self.eval_serial += 1
        check(rc, "gpx_exact_eval")
        return lml.value, grad, jit.value

    def exact_eval_het(self, kind, ARD, variance, lengthscale, noise_variances, jitter=1e-8, max_tries=5):
        """one noise variance per data point -> (log_marginal, gradient[variance, lengthscale.., sum], dnoise (N,), jitter)"""
        k, a, ls = _theta(kind, ARD, lengthscale, self.D)
        nv = _f64(np.asarray(noise_variances).reshape(-1))
        if nv.size != self.N:
            raise ValueError("need one noise variance per data point")
        lml = ctypes.c_double()
        jit = ctypes.c_double()
        grad = np.zeros(ls.size + 2)
        dnoise = np.zeros(self.N)
        rc = self._L.gpx_exact_eval_het(self._h, k, a, float(variance), _ptr(ls), _ptr(nv), float(jitter), int(max_tries),
                                        ctypes.byref(lml), _ptr(grad), _ptr(dnoise), ctypes.byref(jit))
        self.eval_serial += 1
        check(rc, "gpx_exact_eval_het")
        return lml.value, grad, dnoise, jit.value

    def exact_eval_multi(self, parts, noise, jitter=1e-8, max_tries=5):
        """composite kernel: parts = [(kind, ARD, term, dims, variance, lengthscale)], ordered by term ->
        (log_marginal, gradient [per part: variance, lengthscale.. (none for white / bias); then noise], extra_jitter)"""
        arr = (GpxKernPart * len(parts))()
        keep, ngrad = [], 1
        for i, (kind, ard, term, dims, variance, lengthscale) in enumerate(parts):
            static = kind in ("white", "bias")
            d = np.ascontiguousarray([] if static else dims, dtype=np.int32)
            ls = np.ascontiguousarray([1.0] if static else np.atleast_1d(lengthscale), dtype=np.float64).reshape(-1)
            if not static and ls.size != (d.size if ard else 1):
                raise ValueError("part %d: lengthscale does not match its active dims" % i)
            keep += [d, ls]
            arr[i].kind, arr[i].ard, arr[i].term, arr[i].ndims = KIND[kind], int(bool(ard)), int(term), int(d.size)
            arr[i].dims = d.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
            arr[i].variance, arr[i].lengthscale = float(variance), _ptr(ls)
            ngrad += 1 + (0 if static else ls.size)
        lml, jit = ctypes.c_double(), ctypes.c_double()
        grad = np.zeros(ngrad)
        rc = self._L.gpx_exact_eval_multi(self._h, arr, len(parts), float(noise), float(jitter), int(max_tries),
                                          ctypes.byref(lml), _ptr(grad), ctypes.byref(jit))
        self.eval_serial += 1
        check(rc, "gpx_exact_eval_multi")
        return lml.value, grad, jit.value

    def exact_eval_coreg(self, parts, noise, jitter=1e-8, max_tries=5):
        """composite kernel with coregionalization parts and scalar or per-point noise (gpx_exact_eval_coreg).
        parts = [(kind, ARD, term, dims, variance, lengthscale)], ordered by term; a "coregionalize" part carries its
        O x O matrix B in place of the lengthscale and one dim (the output-index column). noise: a float or N variances.
        -> (log_marginal, gradient [per part: variance, lengthscale.. (none for white / bias) or S (O*O, row-major);
        then noise], dnoise (N,) or None, extra_jitter)"""
        arr = (GpxKernPart * len(parts))()
        co = []
        keep, ngrad = [], 1
        for i, (kind, ard, term, dims, variance, lengthscale) in enumerate(parts):
            if kind == "coregionalize":
                B = np.ascontiguousarray(lengthscale, dtype=np.float64)
                d = np.ascontiguousarray(np.atleast_1d(dims), dtype=np.int32)
                if B.ndim != 2 or B.shape[0] != B.shape[1] or d.size != 1:
                    raise ValueError("part %d: a coregionalization part needs one dim and a square B" % i)
                keep += [d, B]
                arr[i].kind, arr[i].ard, arr[i].term, arr[i].ndims = KIND[kind], 0, int(term), 1
                arr[i].dims = d.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
                arr[i].variance, arr[i].lengthscale = 1.0, None
                co.append((B.shape[0], B))
                ngrad += B.size
                continue
            static = kind in ("white", "bias")
            d = np.ascontiguousarray([] if static else dims, dtype=np.int32)
            ls = np.ascontiguousarray([1.0] if static else np.atleast_1d(lengthscale), dtype=np.float64).reshape(-1)
            if not static and ls.size != (d.size if ard else 1):
                raise ValueError("part %d: lengthscale does not match its active dims" % i)
            keep += [d, ls]
            arr[i].kind, arr[i].ard, arr[i].term, arr[i].ndims = KIND[kind], int(bool(ard)), int(term), int(d.size)
            arr[i].dims = d.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
            arr[i].variance, arr[i].lengthscale = float(variance), _ptr(ls)
            ngrad += 1 + (0 if static else ls.size)
        carr = (GpxCoreg * max(1, len(co)))()
        for k, (O, B) in enumerate(co):
            carr[k].output_dim, carr[k].B = int(O), _ptr(B)
        nv = np.asarray(noise, dtype=np.float64).reshape(-1)
        vec = nv.size > 1 or np.ndim(noise) > 0
        if vec:
            nv = _f64(nv)
            if nv.size != self.N:
                raise ValueError("need one noise variance per data point")
        dnoise = np.zeros(self.N) if vec else None
        lml, jit = ctypes.c_double(), ctypes.c_double()
        grad = np.zeros(ngrad)
        rc = self._L.gpx_exact_eval_coreg(self._h, arr, len(parts), carr, float(nv.mean()) if vec else float(nv[0]),
                                          _ptr(nv) if vec else None, float(jitter), int(max_tries), ctypes.byref(lml),
                                          _ptr(grad), _ptr(dnoise), ctypes.byref(jit))
        self.eval_serial += 1
        check(rc, "gpx_exact_eval_coreg")
        return lml.value, grad, dnoise, jit.value

    def get(self, which):
        if which == "alpha":
            out = np.empty((self.N, self.P))
        else:
            out = np.empty((self.N, self.N), order="F")
        check(self._L.gpx_get(self._h, GET[which], _ptr(out)), "gpx_get")
        return out

    def predict(self, Xnew, full_cov=False):
        Xnew = _f64(Xnew)
        M = Xnew.shape[0]
        mu = np.empty((M, self.P))
        var = np.empty((M, M), order="F") if full_cov else np.empty(M)
        check(self._L.gpx_predict(self._h, _ptr(Xnew), M, int(full_cov), _ptr(mu), _ptr(var)), "gpx_predict")
        return mu, (var if full_cov else var[:, None])

    def kern_K_device_only(self, kind, ARD, variance, lengthscale, X, X2=None):
        """build K(X, X2) on the device without bringing it back; -> (kernel ms, algorithmic GB/s)."""
        X = _f64(X)
        N, D = X.shape
        k, a, ls = _theta(kind, ARD, lengthscale, D)
        X2c = None if X2 is None else _f64(X2)
        M = N if X2 is None else X2c.shape[0]
        check(self._L.gpx_kern_K(self._h, k, a, float(variance), _ptr(ls), _ptr(X), N, _ptr(X2c), M, D, None), "gpx_kern_K")
        st = self.stats()
        return st["kbuild_ms"], st["kbuild_bytes"] / st["kbuild_ms"] * 1e-6

    # ---- sparse GP regression (VarDTC) building blocks ---------------------------------------------------------
    def sparse_set_data(self, X, Y):
        X, Y = _f64(X), _f64(Y)
        self.sN, self.sD = X.shape
        self.sP = Y.shape[1]
        check(self._L.gpx_sparse_set_data(self._h, _ptr(X), self.sN, self.sD, _ptr(Y), self.sP), "gpx_sparse_set_data")

    def sparse_eval(self, kind, ARD, variance, lengthscale, Z, noise_variance):
        """one whole VarDTC evaluation on the device -> (lml, grad [variance, lengthscale.., noise], dZ (M x D))"""
        Z = _f64(Z)
        M = Z.shape[0]
        k, a, ls = _theta(kind, ARD, lengthscale, self.sD)
        lml = ctypes.c_double()
        grad = np.zeros(ls.size + 2)
        dZ = np.empty((M, self.sD))
        check(self._L.gpx_sparse_eval(self._h, k, a, float(variance), _ptr(ls), _ptr(Z), M, float(noise_variance),
                                      ctypes.byref(lml), _ptr(grad), _ptr(dZ)), "gpx_sparse_eval")
        self.sM, self._snl = M, ls.size
        self.sparse_serial = getattr(self, "sparse_serial", 0) + 1
        return lml.value, grad, dZ

    def sparse_eval_het(self, kind, ARD, variance, lengthscale, Z, noise_variances):
        """VarDTC with one noise variance per data point (var_dtc.py het_noise branches) ->
        (lml, grad [variance, lengthscale..], dZ (M x D), dL_dR (N x P))"""
        Z = _f64(Z)
        M = Z.shape[0]
        k, a, ls = _theta(kind, ARD, lengthscale, self.sD)
        nv = _f64(np.asarray(noise_variances, dtype=np.float64).reshape(-1))
        if nv.size != self.sN:
            raise ValueError("one noise variance per data point expected (%d given, N = %d)" % (nv.size, self.sN))
        lml = ctypes.c_double()
        grad = np.zeros(ls.size + 1)
        dZ = np.empty((M, self.sD))
        dR = np.empty((self.sN, self.sP))
        check(self._L.gpx_sparse_eval_het(self._h, k, a, float(variance), _ptr(ls), _ptr(Z), M, _ptr(nv),
                                          ctypes.byref(lml), _ptr(grad), _ptr(dZ), _ptr(dR)), "gpx_sparse_eval_het")
        self.sM, self._snl = M, ls.size
        self.sparse_serial = getattr(self, "sparse_serial", 0) + 1
        return lml.value, grad, dZ, dR

    SPARSE_GET = {"woodbury_vector": 0, "woodbury_inv": 1, "Kmm": 2, "Lm": 3}

    def sparse_get(self, what):
        which = self.SPARSE_GET[what]
        out = np.empty((self.sM, self.sP)) if which == 0 else np.empty((self.sM, self.sM), order="F")
        check(self._L.gpx_sparse_get(self._h, which, _ptr(out)), "gpx_sparse_get")
        return out

    def stats(self):
        s = GpxStats()
        check(self._L.gpx_get_stats(self._h, ctypes.byref(s)), "gpx_get_stats")
        return s.as_dict()

    def measure_fp64_peak(self):
        """fp64 DMMA issue peak of this device in TFLOP/s (roofline denominator, measured live)."""
        v = ctypes.c_double()
        check(self._L.gpx_measure_fp64_peak(self._h, ctypes.byref(v)), "gpx_measure_fp64_peak")
        return v.value

    def total_launches(self):
        return int(self._L.gpx_total_launches(self._h))


def kern_K(kind, ARD, variance, lengthscale, X, X2=None):
    X = _f64(X)
    N, D = X.shape
    k, a, ls = _theta(kind, ARD, lengthscale, D)
    if X2 is not None:
        X2 = _f64(X2)
        M = X2.shape[0]
    else:
        M = N
    out = np.empty((N, M))
    check(lib().gpx_kern_K(None, k, a, float(variance), _ptr(ls), _ptr(X), N, _ptr(X2), M, D, _ptr(out)), "gpx_kern_K")
    return out


def kern_Kdiag(kind, variance, N):
    out = np.empty(N)
    check(lib().gpx_kern_Kdiag(KIND[kind], float(variance), N, _ptr(out)), "gpx_kern_Kdiag")
    return out


def kern_grad_X(kind, ARD, variance, lengthscale, X, dL_dK, X2=None):
    """Stationary.gradients_X (stationary.py:245-252) on the device -> N x D."""
    X = _f64(X)
    N, D = X.shape
    k, a, ls = _theta(kind, ARD, lengthscale, D)
    X2c = None if X2 is None else _f64(X2)
    M = N if X2 is None else X2c.shape[0]
    dL_dK = _f64(dL_dK)
    if dL_dK.shape != (N, M):
        raise ValueError("dL_dK must be %d x %d" % (N, M))
    out = np.empty((N, D))
    check(lib().gpx_kern_grad_X(None, k, a, float(variance), _ptr(ls), _ptr(X), N, _ptr(X2c), M, D, _ptr(dL_dK), _ptr(out)),
          "gpx_kern_grad_X")
    return out


def pdinv(A, maxtries=5, want=("Ai", "L", "Li"), engine=None):
    """GPy.util.linalg.pdinv (linalg.py:193-214) on the device: -> (Ai, L, Li, logdet) (entries not in `want` are None)
    plus the jitter the jitchol ladder (linalg.py:56-75) had to add. Raises numpy.linalg.LinAlgError like the reference."""
    A = _f64(A)
    N = A.shape[0]
    if A.ndim != 2 or A.shape[1] != N:
        raise ValueError("A must be square")
    outs = {k: (np.empty((N, N), order="F") if k in want else None) for k in ("Ai", "L", "Li")}
    logdet, jit = ctypes.c_double(), ctypes.c_double()
    h = engine._h if engine is not None else None
    rc = lib().gpx_pdinv(h, _ptr(np.ascontiguousarray(A)), N, int(maxtries), _ptr(outs["Ai"]), _ptr(outs["L"]), _ptr(outs["Li"]),
                         ctypes.byref(logdet), ctypes.byref(jit))
    if rc > 0:
        raise np.linalg.LinAlgError(lib().gpx_last_error().decode())
    check(rc, "gpx_pdinv")
    return outs["Ai"], outs["L"], outs["Li"], logdet.value, jit.value


def jitchol(A, maxtries=5, engine=None):
    """GPy.util.linalg.jitchol (linalg.py:56-75) on the device: lower Cholesky factor, jitter ladder included."""
    return pdinv(A, maxtries, want=("L",), engine=engine)[1]


def kern_grad_full(kind, ARD, variance, lengthscale, X, dL_dK, X2=None):
    X = _f64(X)
    N, D = X.shape
    k, a, ls = _theta(kind, ARD, lengthscale, D)
    if X2 is not None:
        X2 = _f64(X2)
        M = X2.shape[0]
    else:
        M = N
    dL_dK = _f64(dL_dK)
    if dL_dK.shape != (N, M):
        raise ValueError("dL_dK must be %d x %d" % (N, M))
    dv = ctypes.c_double()
    dl = np.zeros(ls.size)
    check(lib().gpx_kern_grad_full(None, k, a, float(variance), _ptr(ls), _ptr(X), N, _ptr(X2), M, D, _ptr(dL_dK),
                                   ctypes.byref(dv), _ptr(dl)), "gpx_kern_grad_full")
    return dv.value, dl
