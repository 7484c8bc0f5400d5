"""
ctypes binding of libibo_b200.so (include/ibo_b200.h) -- the same mechanism the reference uses
for its optional libego (ego/acquisition/__init__.py:335-364), minus the find_library loop that
spins forever when the library is absent (:336-342): the library is looked up next to this
package and a missing or unbuildable library is a hard error.  There is no CPU fallback.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_long, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libibo_b200.so")

# every symbol include/ibo_b200.h declares (checked by tests/test_abi.py)
EXPORTED = [
    "ibo_last_error", "ibo_version", "ibo_device_count",
    "ibo_model_create", "ibo_model_create_pref", "ibo_model_create_laplace", "ibo_model_create_from_inverse", "ibo_model_append", "ibo_model_destroy", "ibo_model_n", "ibo_model_dim",
    "ibo_model_get_matrix", "ibo_model_set_variance_model", "ibo_pref_fit",
    "ibo_nlml", "ibo_kernel_matrix",
    "ibo_posterior_batch", "ibo_score_batch", "ibo_posterior_cov", "ibo_posterior_sample",
    "ibo_posterior_grad", "ibo_score_grad", "ibo_qei", "ibo_qnei", "ibo_max_value_gumbel", "ibo_mes",
    "ibo_paths_create", "ibo_paths_eval", "ibo_paths_grad", "ibo_paths_destroy",
    "ibo_cands_create", "ibo_cands_destroy", "ibo_score_resident", "ibo_get_profile", "ibo_launch_count",
    "ibo_fp64_peak", "ibo_i8_peak", "ibo_i8_peak2", "ibo_host_register", "ibo_host_unregister", "ibo_stream_mark", "ibo_stream_elapsed_ms",
    "ibo_device_synchronize", "ibo_debug_exp",
    "ibo_direct_batched", "ibo_acqmax", "ibo_acqmax_many", "direct", "acqmaxGP",
    "ibo_comm_unique_id", "ibo_comm_init", "ibo_comm_destroy", "ibo_comm_argmax", "ibo_comm_bcast", "ibo_comm_barrier",
    "ibo_comm_rank", "ibo_comm_size", "ibo_comm_allgather",
    "ibo_set_option", "ibo_get_option", "ibo_model_last_guarded",
]

KERNEL_SE_ARD, KERNEL_SE_ISO, KERNEL_MATERN3, KERNEL_MATERN5, KERNEL_MATERN5_ARD = 0, 1, 2, 3, 4
ACQ_EI, ACQ_PI, ACQ_UCB = 0, 1, 2
FLAG_MODE_CPP, FLAG_MODE_PY, FLAG_KSTAR_EXPAND, FLAG_DIRECT_SEQ, FLAG_PROFILE, FLAG_GRAD_EXACT, FLAG_SHARD = 0x0, 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
FLAG_DIRECT_SPECULATE = 0x40
FLAG_INT8 = 0x80      # take the INT8 tensor-core path of wide batches even when option "int8" is 0 (it is on by default)
FLAG_FP64 = 0x100     # FP64 DMMA kernels for every candidate
E_BADARG, E_CUDA, E_NOTSPD, E_NOMEM, E_COMM, E_OBJECTIVE = -1, -2, -3, -4, -5, -6

BATCH_OBJECTIVE = ctypes.CFUNCTYPE(None, c_void_p, c_long, c_int, POINTER(c_double), POINTER(c_double))
OBJECTIVE = ctypes.CFUNCTYPE(c_double, c_int, POINTER(c_double))

_lib = None


class IBOError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "libibo_b200 error %d: %s" % (code, msg))
        self.code = code


class NotPositiveDefinite(IBOError, np.linalg.LinAlgError):
    """Raised when the device Cholesky meets a non-positive pivot (numpy.linalg.LinAlgError-compatible so
    that the reference's `C += I` retry loop, ego/gaussianprocess/__init__.py:487-498, keeps working)."""

    def __init__(self, code, msg, pivot):
        IBOError.__init__(self, code, msg)
        self.pivot = pivot


def dptr(a):
    return a.ctypes.data_as(POINTER(c_double))


def as_f64(a, ndmin=1):
    return np.ascontiguousarray(np.array(a, dtype=np.float64, ndmin=ndmin))


def lib():
    """Load (once) and return the shared library with argtypes set."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s not found: build it with `make -C ibo_b200/csrc` (or __graft_entry__.build()); "
                          "ibo_b200 has no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    pd, pi, pl = POINTER(c_double), POINTER(c_int), POINTER(c_long)
    L.ibo_last_error.restype = c_char_p
    L.ibo_version.restype = c_char_p
    L.ibo_device_count.restype = c_int
    L.ibo_launch_count.restype = c_long
    L.ibo_model_create.restype = c_int
    L.ibo_model_create.argtypes = [c_int, c_int, pd, c_int, pd, pd, c_int, c_int, c_double, pd,
                                   c_int, pd, pd, c_double, pd, pd, POINTER(c_void_p), pi]
    L.ibo_model_create_pref.argtypes = [c_int, c_int, pd, c_int, pd, pd, c_int, c_int, c_double, c_int, pi, pi, pd, c_double,
                                        POINTER(c_void_p), pi]
    L.ibo_model_create_laplace.argtypes = [c_int, c_int, pd, c_int, pd, pd, c_int, c_int, c_double, pd, POINTER(c_void_p), pi]
    L.ibo_model_create_from_inverse.restype = c_int
    L.ibo_model_create_from_inverse.argtypes = [c_int, c_int, pd, c_int, pd, pd, c_int, c_int, c_double, pd, c_double,
                                                c_int, pd, pd, c_double, pd, pd, POINTER(c_void_p), pi]
    L.ibo_model_append.argtypes = [c_void_p, pd, pd, c_int, pi]
    L.ibo_model_destroy.argtypes = [c_void_p]
    L.ibo_model_n.argtypes = [c_void_p]
    L.ibo_model_dim.argtypes = [c_void_p]
    L.ibo_model_get_matrix.argtypes = [c_void_p, c_int, pd]
    L.ibo_model_set_variance_model.argtypes = [c_void_p, c_void_p]
    L.ibo_pref_fit.argtypes = [c_void_p, c_int, pi, pi, pd, pd, c_int, c_double, pd, pd, pi]
    L.ibo_nlml.argtypes = [c_int, c_int, pd, c_int, pd, pd, c_int, c_int, c_double, c_int, pd, pd, pi]
    L.ibo_kernel_matrix.argtypes = [c_int, c_int, pd, c_int, pd, c_int, c_int, c_int, c_int, pd]
    L.ibo_posterior_batch.argtypes = [c_void_p, pd, c_long, c_int, pd, pd]
    L.ibo_score_batch.argtypes = [c_void_p, pd, c_long, c_int, c_double, c_double, c_int, pd, pd, pd, pd, pl]
    L.ibo_posterior_cov.argtypes = [c_void_p, pd, c_long, pd, pd]
    L.ibo_posterior_sample.argtypes = [c_void_p, pd, c_long, pd, c_int, c_double, pd, pl, pi]
    L.ibo_posterior_grad.argtypes = [c_void_p, pd, c_long, c_int, pd, pd, pd, pd]
    L.ibo_score_grad.argtypes = [c_void_p, pd, c_long, c_int, c_double, c_double, c_int, pd, pd]
    L.ibo_qei.argtypes = [c_void_p, pd, c_long, c_int, pd, c_int, c_double, c_double, c_double, pd, pd, pi]
    L.ibo_qnei.argtypes = [c_void_p, pd, c_long, c_int, pd, c_long, pd, c_int, c_double, pd, pd, pd, pi, pi]
    L.ibo_max_value_gumbel.argtypes = [c_void_p, pd, c_long, c_int, pd, pd, pd]
    L.ibo_mes.argtypes = [c_void_p, pd, c_long, pd, c_int, c_int, pd, pd, pd, pl]
    L.ibo_paths_create.argtypes = [c_void_p, c_int, c_int, pd, pd, pd, pd, POINTER(c_void_p), pi]
    L.ibo_paths_eval.argtypes = [c_void_p, pd, c_long, pd, pd, pl]
    L.ibo_paths_grad.argtypes = [c_void_p, pd, c_long, pi, pd, pd]
    L.ibo_paths_destroy.argtypes = [c_void_p]
    L.ibo_cands_create.argtypes = [c_void_p, pd, c_long, POINTER(c_void_p)]
    L.ibo_cands_destroy.argtypes = [c_void_p]
    L.ibo_score_resident.argtypes = [c_void_p, c_void_p, c_int, c_double, c_double, c_int, pd, pd, pl, POINTER(c_float)]
    L.ibo_get_profile.argtypes = [c_void_p, pd]
    L.ibo_fp64_peak.argtypes = [c_int, pd]
    L.ibo_i8_peak.argtypes = [c_int, pd]
    L.ibo_i8_peak2.argtypes = [c_int, c_double, pd, pd]
    L.ibo_host_register.argtypes = [c_void_p, ctypes.c_ulong]
    L.ibo_host_unregister.argtypes = [c_void_p]
    L.ibo_stream_mark.argtypes = [c_void_p, c_int]
    L.ibo_stream_elapsed_ms.argtypes = [c_void_p, POINTER(c_float)]
    L.ibo_device_synchronize.argtypes = [c_int]
    L.ibo_debug_exp.argtypes = [c_int, pd, c_long, pd, pd]
    L.ibo_direct_batched.argtypes = [BATCH_OBJECTIVE, c_void_p, c_int, pd, pd, c_int, c_int, c_int, c_int, pd, pd, pl, pi]
    L.ibo_acqmax.argtypes = [c_void_p, pd, pd, c_int, c_double, c_double, c_int, c_int, c_int, c_int, pd, pd, pl, pi]
    L.ibo_acqmax_many.argtypes = [c_int, POINTER(c_void_p), pd, pd, c_int, pd, pd, c_int, c_int, c_int, c_int, pd, pd, pl, pi, pi]
    L.direct.restype = POINTER(c_double)
    L.direct.argtypes = [OBJECTIVE, c_int, pd, pd, c_int, c_int, c_int]
    L.acqmaxGP.restype = POINTER(c_double)
    L.acqmaxGP.argtypes = [c_int, pd, pd, pd, pd, pd, c_int, c_int, c_int, pd, c_int, pd, pd, c_double, pd, pd,
                           c_double, c_double, c_int, c_int, c_int]       # ego/acquisition/__init__.py:343-364
    L.ibo_comm_unique_id.argtypes = [ctypes.c_char_p]
    L.ibo_comm_init.argtypes = [c_int, c_int, c_int, ctypes.c_char_p]
    L.ibo_comm_argmax.argtypes = [pd, pl]
    L.ibo_comm_bcast.argtypes = [pd, c_long, c_int]
    L.ibo_comm_allgather.argtypes = [pd, c_long, pd]
    L.ibo_set_option.argtypes = [c_char_p, c_long]
    L.ibo_get_option.argtypes = [c_char_p, pl]
    L.ibo_model_last_guarded.argtypes = [c_void_p]
    _lib = L
    return L


def check(rc, info=None):
    if rc == 0:
        return
    msg = lib().ibo_last_error().decode("utf-8", "replace")
    if rc == E_NOTSPD:
        raise NotPositiveDefinite(rc, msg, info)
    raise IBOError(rc, msg)


def set_option(name, value):
    """Process-wide tuning switch of the library (include/ibo_b200.h, "options")."""
    check(lib().ibo_set_option(name.encode(), int(value)))


def get_option(name):
    v = c_long(0)
    check(lib().ibo_get_option(name.encode(), ctypes.byref(v)))
    return v.value


def require_gpu():
    """Fail loudly when no device is usable -- the product path never degrades to the CPU."""
    n = lib().ibo_device_count()
    if n <= 0:
        raise IBOError(E_CUDA, "no CUDA device visible; ibo_b200 has no CPU fallback (%s)"
                       % lib().ibo_last_error().decode("utf-8", "replace"))
    return n


def nlml(kind, hyper, X, Y, noise, want_grad=True, flags=0, device=0):
    """ibo_nlml: (nlml, dnlml or None) of trainhyper.marginalLikelihood on the device."""
    hyper = as_f64(hyper)
    X = as_f64(X, 2)
    Y = as_f64(Y)
    if X.shape[0] != Y.shape[0]:
        raise ValueError("X and Y differ in length")
    val = c_double(0.0)
    grad = np.zeros(len(hyper)) if want_grad else None
    info = c_int(0)
    rc = lib().ibo_nlml(device, kind, dptr(hyper), len(hyper), dptr(X), dptr(Y), X.shape[0], X.shape[1], float(noise), flags,
                        ctypes.byref(val), dptr(grad) if want_grad else None, ctypes.byref(info))
    check(rc, info.value)
    return val.value, grad


def kernel_matrix(kind, hyper, X, which=-1, flags=0, device=0):
    """ibo_kernel_matrix: covMatrix(X) (which < 0) or derivative(X, which) as an N x N array."""
    hyper = as_f64(hyper)
    X = as_f64(X, 2)
    out = np.empty((X.shape[0], X.shape[0]))
    check(lib().ibo_kernel_matrix(device, kind, dptr(hyper), len(hyper), dptr(X), X.shape[0], X.shape[1], int(which), flags, dptr(out)))
    return out


class Model(object):
    """Owner of an `ibo_model*` handle (device-resident L, W = inv(L), beta)."""

    def __init__(self, kind, hyper, X, Y, noise, Cinv=None, prior=None, device=0, invR=None, sf2=1.0, pref=None, C=None):
        """pref = (a, b, w, cdiag): Laplace term as preference pairs, C = dense Laplace matrix -- inv(C) is then formed on the
        device (ibo_model_create_pref / ibo_model_create_laplace); Cinv = explicit inverse (ibo_model_create)"""
        L = lib()
        self.X = as_f64(X, 2)
        self.Y = as_f64(Y, 1).reshape(-1)
        self.N, self.d = self.X.shape
        if self.Y.shape[0] != self.N:
            raise ValueError("X and Y disagree")
        hyper = as_f64(hyper, 1)
        self._h = c_void_p()
        info = c_int(0)
        if prior is None:
            npb, pm, pb, pt = 0, as_f64([0.0]), as_f64([0.0]), 0.0
            plb, pw = as_f64([0.0]), as_f64([1.0])
        else:
            pm = as_f64(prior.means, 2)
            npb = pm.shape[0]
            pb, pt = as_f64(prior.beta), float(prior.theta)
            plb, pw = as_f64(prior.lowerb), as_f64(prior.width)
        if pref is not None:
            a = np.ascontiguousarray(pref[0], dtype=np.int32); b = np.ascontiguousarray(pref[1], dtype=np.int32)
            w = as_f64(pref[2], 1)
            ip = lambda z: z.ctypes.data_as(POINTER(c_int))
            rc = L.ibo_model_create_pref(device, kind, dptr(hyper), len(hyper), dptr(self.X), dptr(self.Y), self.N, self.d, float(noise),
                                         len(a), ip(a), ip(b), dptr(w), float(pref[3]), ctypes.byref(self._h), ctypes.byref(info))
        elif C is not None:
            C = as_f64(C, 2)
            rc = L.ibo_model_create_laplace(device, kind, dptr(hyper), len(hyper), dptr(self.X), dptr(self.Y), self.N, self.d, float(noise),
                                            dptr(C), ctypes.byref(self._h), ctypes.byref(info))
        elif invR is not None:
            invR = as_f64(invR, 2)
            rc = L.ibo_model_create_from_inverse(device, kind, dptr(hyper), len(hyper), dptr(self.X), dptr(self.Y), self.N, self.d,
                                                 float(noise), dptr(invR), float(sf2), npb, dptr(pm), dptr(pb), pt, dptr(plb), dptr(pw),
                                                 ctypes.byref(self._h), ctypes.byref(info))
        else:
            ci = None
            if Cinv is not None:
                Cinv = as_f64(Cinv, 2)
                ci = dptr(Cinv)
            rc = L.ibo_model_create(device, kind, dptr(hyper), len(hyper), dptr(self.X), dptr(self.Y), self.N, self.d,
                                    float(noise), ci, npb, dptr(pm), dptr(pb), pt, dptr(plb), dptr(pw),
                                    ctypes.byref(self._h), ctypes.byref(info))
        check(rc, info.value)
        self._var = None

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().ibo_model_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def handle(self):
        return self._h

    def append(self, X, Y):
        """rank-1 device append of observations (ibo_model_append); raises NotPositiveDefinite like a rebuild would"""
        X = as_f64(X, 2)
        Y = as_f64(Y, 1).reshape(-1)
        if X.shape[1] != self.d or X.shape[0] != Y.shape[0]:
            raise ValueError("appended X / Y have the wrong shape")
        info = c_int(0)
        rc = lib().ibo_model_append(self._h, dptr(X), dptr(Y), X.shape[0], ctypes.byref(info))
        if rc == E_NOTSPD:       # the handle is unusable now
            self.close()
        check(rc, info.value)
        self.X = np.r_[self.X, X]
        self.Y = np.r_[self.Y, Y]
        self.N = self.X.shape[0]

    def pref_fit(self, v, u, deg, start, maxit=100, gtol=1e-9):
        """Laplace MAP latents of a preference model (ibo_pref_fit) -> (Y, S(Y), |grad|_inf, Newton iterations)"""
        v = np.ascontiguousarray(v, dtype=np.int32)
        u = np.ascontiguousarray(u, dtype=np.int32)
        deg = as_f64(deg, 1)
        y = as_f64(start, 1).copy()
        if y.shape[0] != self.N or len(v) != len(u) or len(v) != len(deg):
            raise ValueError("preference arrays have the wrong shape")
        S, g, it = c_double(0), c_double(0), c_int(0)
        ip = lambda a: a.ctypes.data_as(POINTER(c_int))
        check(lib().ibo_pref_fit(self._h, len(v), ip(v), ip(u), dptr(deg), dptr(y), int(maxit), float(gtol),
                                 ctypes.byref(S), ctypes.byref(g), ctypes.byref(it)))
        return y, S.value, g.value, it.value

    def matrix(self, which):
        out = np.empty((self.N, self.N))
        check(lib().ibo_model_get_matrix(self._h, which, dptr(out)))
        return out

    def set_variance_model(self, other):
        self._var = other
        check(lib().ibo_model_set_variance_model(self._h, other._h if other is not None else None))

    def posterior(self, Xs, flags=FLAG_MODE_PY):
        Xs = as_f64(Xs, 2)
        M = Xs.shape[0]
        mu, s2 = np.empty(M), np.empty(M)
        check(lib().ibo_posterior_batch(self._h, dptr(Xs), M, flags, dptr(mu), dptr(s2)))
        return mu, s2

    def _candidates(self, Xs):
        Xs = as_f64(Xs, 2)
        if Xs.shape[1] != self.d:
            raise ValueError("candidates have %d columns, the model %d" % (Xs.shape[1], self.d))
        return Xs

    def posterior_cov(self, Xs):
        """joint posterior over the candidates (ibo_posterior_cov) -> (mu[M], cov[M, M]); diag(cov) is the unclipped sigma^2"""
        Xs = self._candidates(Xs)
        M = Xs.shape[0]
        mu, cov = np.empty(M), np.empty((M, M))
        check(lib().ibo_posterior_cov(self._h, dptr(Xs), M, dptr(mu), dptr(cov)))
        return mu, cov

    def posterior_sample(self, Xs, Z, jitter=0.0, want_F=True):
        """joint posterior samples F = mu + chol(cov + jitter I) Z for standard normals Z[M, S] (ibo_posterior_sample)
        -> (F[M, S] or None, argmax[S]); raises NotPositiveDefinite (pivot = 1-based candidate) when cov + jitter I is not SPD"""
        Xs = self._candidates(Xs)
        Z = as_f64(Z, 2)
        M, S = Xs.shape[0], Z.shape[1]
        if Z.shape[0] != M:
            raise ValueError("Z has %d rows for %d candidates" % (Z.shape[0], M))
        F = np.empty((M, S)) if want_F else None
        am = np.empty(S, dtype=np.int64)
        info = c_int(0)
        rc = lib().ibo_posterior_sample(self._h, dptr(Xs), M, dptr(Z), S, float(jitter), dptr(F) if want_F else None,
                                        am.ctypes.data_as(POINTER(c_long)), ctypes.byref(info))
        check(rc, info.value)
        return F, am

    def posterior_grad(self, Xs, flags=FLAG_MODE_PY):
        """posterior and its gradient with respect to the candidate (ibo_posterior_grad) -> (mu[M], s2[M], dmu[M, d], ds2[M, d]);
        values are ibo_posterior_batch's with FLAG_FP64, ds2 = 0 where s2 is clipped"""
        Xs = self._candidates(Xs)
        M = Xs.shape[0]
        mu, s2, dmu, ds2 = np.empty(M), np.empty(M), np.empty((M, self.d)), np.empty((M, self.d))
        check(lib().ibo_posterior_grad(self._h, dptr(Xs), M, flags, dptr(mu), dptr(s2), dptr(dmu), dptr(ds2)))
        return mu, s2, dmu, ds2

    def score_grad(self, Xs, acq, ymax, parm, flags=FLAG_MODE_PY):
        """acquisition values and their gradient with respect to the candidate (ibo_score_grad) -> (scores[M], dscores[M, d]);
        scores are ibo_score_batch's with FLAG_FP64"""
        Xs = self._candidates(Xs)
        M = Xs.shape[0]
        sc, dsc = np.empty(M), np.empty((M, self.d))
        check(lib().ibo_score_grad(self._h, dptr(Xs), M, acq, float(ymax), float(parm), flags, dptr(sc), dptr(dsc)))
        return sc, dsc

    def qei(self, Xb, Z, ymax, xi, jitter=0.0, want_grad=True):
        """batch expected improvement of B batches of q points Xb[B, q, d] for standard normals Z[q, S] (ibo_qei) ->
        (values[B], dvalues[B, q, d] or None, number of batches whose covariance + jitter I is not positive definite: NaN rows)"""
        Xb = as_f64(Xb, 3)
        Z = as_f64(Z, 2)
        B, q, d = Xb.shape
        if d != self.d:
            raise ValueError("points have %d columns, the model %d" % (d, self.d))
        if Z.shape[0] != q:
            raise ValueError("Z has %d rows for batches of %d points" % (Z.shape[0], q))
        vals = np.empty(B)
        dv = np.empty((B, q, d)) if want_grad else None
        nbad = c_int(0)
        check(lib().ibo_qei(self._h, dptr(Xb), B, q, dptr(Z), Z.shape[1], float(ymax), float(xi), float(jitter), dptr(vals),
                            dptr(dv) if want_grad else None, ctypes.byref(nbad)))
        return vals, dv, nbad.value

    def qnei(self, Xb, Xbase, Z, jitter=0.0, want_grad=True):
        """noisy batch expected improvement of B batches of q points Xb[B, q, d] over the baseline Xbase[P, d] for standard normals
        Z[P + q, S], baseline rows first (ibo_qnei) -> (values[B], dvalues[B, q, d] or None, number of batches whose Schur
        complement + jitter I is not positive definite: NaN rows, incumbent draws m[S]).  Raises NotPositiveDefinite with the
        1-based pivot when the baseline's covariance + jitter I is not positive definite."""
        Xb = as_f64(Xb, 3)
        Xbase = as_f64(Xbase, 2)
        Z = as_f64(Z, 2)
        B, q, d = Xb.shape
        if d != self.d or Xbase.shape[1] != self.d:
            raise ValueError("points have %d and %d columns, the model %d" % (d, Xbase.shape[1], self.d))
        P = Xbase.shape[0]
        if Z.shape[0] != P + q:
            raise ValueError("Z has %d rows for %d baseline points and batches of %d" % (Z.shape[0], P, q))
        S = Z.shape[1]
        vals = np.empty(B)
        dv = np.empty((B, q, d)) if want_grad else None
        inc = np.empty(S)
        nbad, info = c_int(0), c_int(0)
        rc = lib().ibo_qnei(self._h, dptr(Xb), B, q, dptr(Xbase), P, dptr(Z), S, float(jitter), dptr(vals),
                            dptr(dv) if want_grad else None, dptr(inc), ctypes.byref(nbad), ctypes.byref(info))
        check(rc, info.value)
        return vals, dv, nbad.value, inc

    def max_value_gumbel(self, Xs, flags=FLAG_MODE_CPP):
        """Gumbel fit of the distribution of the maximum over the candidates (ibo_max_value_gumbel) -> (q[3], loc, scale): q solve
        F(q) = 0.25, 0.5, 0.75 for F(y) = prod_i Phi((y - mu_i) / s_i) with mu, s2 as `posterior` returns them with `flags`"""
        Xs = self._candidates(Xs)
        q, loc, scale = np.empty(3), c_double(0), c_double(0)
        check(lib().ibo_max_value_gumbel(self._h, dptr(Xs), Xs.shape[0], flags, dptr(q), ctypes.byref(loc), ctypes.byref(scale)))
        return q, loc.value, scale.value

    def mes(self, Xs, ystar, flags=FLAG_MODE_CPP, want_grad=False):
        """max-value entropy search at the candidates for samples ystar[K] of the maximum (ibo_mes) -> (values[M],
        dvalues[M, d] or None, best value, its index).  With want_grad, flags may carry FLAG_MODE_PY only and the values are
        those of the FP64 kernels."""
        Xs = self._candidates(Xs)
        ystar = as_f64(ystar)
        M = Xs.shape[0]
        vals = np.empty(M)
        dv = np.empty((M, self.d)) if want_grad else None
        best, bidx = c_double(0), c_long(-1)
        check(lib().ibo_mes(self._h, dptr(Xs), M, dptr(ystar), ystar.shape[0], flags, dptr(vals), dptr(dv) if want_grad else None,
                            ctypes.byref(best), ctypes.byref(bidx)))
        return vals, dv, best.value, bidx.value

    def sample_paths(self, omega, phase, w, e):
        """pathwise posterior samples for caller-supplied draws (ibo_paths_create): omega[F, d] spectral frequencies, phase[F],
        w[F, S] and e[Ng, S] standard normals (Ng: the training points of the variance model when one is attached) -> Paths;
        raises NotPositiveDefinite when inv(C) + (1 + noise - sf2) I of a Laplace model is not positive definite"""
        return Paths(self, omega, phase, w, e)

    def score(self, Xs, acq, ymax, parm, flags=FLAG_MODE_PY, want_scores=True, want_posterior=False, out=None):
        """`out` (optional, float64[M]) receives the scores in place (lets callers reuse a pinned buffer)."""
        if not (isinstance(Xs, np.ndarray) and Xs.dtype == np.float64 and Xs.ndim == 2 and Xs.flags.c_contiguous):
            Xs = as_f64(Xs, 2)
        M = Xs.shape[0]
        sc = (out if out is not None else np.empty(M)) if want_scores else None
        mu = np.empty(M) if want_posterior else None
        s2 = np.empty(M) if want_posterior else None
        best, bidx = c_double(0), c_long(-1)
        check(lib().ibo_score_batch(self._h, dptr(Xs), M, acq, float(ymax), float(parm), flags,
                                    dptr(sc) if want_scores else None, dptr(mu) if want_posterior else None,
                                    dptr(s2) if want_posterior else None, ctypes.byref(best), ctypes.byref(bidx)))
        return sc, mu, s2, best.value, bidx.value

    def acqmax(self, lb, ub, acq, ymax, parm, flags=FLAG_MODE_CPP, maxiter=50, maxtime=30, maxsample=10000):
        lb, ub = as_f64(lb), as_f64(ub)
        opt, optx = c_double(0), np.empty(self.d)
        ns, it = c_long(0), c_int(0)
        check(lib().ibo_acqmax(self._h, dptr(lb), dptr(ub), acq, float(ymax), float(parm), flags, int(maxiter), int(maxtime),
                               int(maxsample), ctypes.byref(opt), dptr(optx), ctypes.byref(ns), ctypes.byref(it)))
        return opt.value, optx, ns.value, it.value

    def last_guarded(self):
        """candidates the last scoring call re-scored on the DMMA path (guard of the INT8 path)"""
        return int(lib().ibo_model_last_guarded(self._h))

    def profile(self):
        out = np.zeros(6)
        check(lib().ibo_get_profile(self._h, dptr(out)))
        return dict(k1_ms=out[0], k2_ms=out[1], k3_ms=out[2], total_ms=out[3], launches=int(out[4]), k2_launches=int(out[5]))


class Paths(object):
    """Owner of an `ibo_paths*` handle: S posterior sample paths, a snapshot of the model they were drawn from"""

    def __init__(self, model, omega, phase, w, e):
        omega, phase, w, e = as_f64(omega, 2), as_f64(phase), as_f64(w, 2), as_f64(e, 2)
        F, S = w.shape
        ng = (model._var or model).N           # the training points Sigma comes from: the variance model's when one is attached
        if omega.shape != (F, model.d) or phase.shape != (F,) or e.shape != (ng, S):
            raise ValueError("draws have inconsistent shapes: omega %s, phase %s, w %s, e %s" % (omega.shape, phase.shape, w.shape, e.shape))
        self.d, self.S, self.F = model.d, S, F
        self._h = c_void_p()
        info = c_int(0)
        check(lib().ibo_paths_create(model.handle, F, S, dptr(omega), dptr(phase), dptr(w), dptr(e), ctypes.byref(self._h),
                                     ctypes.byref(info)), info.value)

    def _points(self, X):
        X = as_f64(X, 2)
        if X.shape[1] != self.d:
            raise ValueError("points have %d columns, the paths %d" % (X.shape[1], self.d))
        return X

    def eval(self, X, want_values=True):
        """(values[M, S] or None, best[S], argmax[S]) at the points X[M, d] (ibo_paths_eval)"""
        X = self._points(X)
        M = X.shape[0]
        vals = np.empty((M, self.S)) if want_values else None
        best, idx = np.empty(self.S), np.empty(self.S, dtype=np.int64)
        check(lib().ibo_paths_eval(self._h, dptr(X), M, dptr(vals) if want_values else None, dptr(best), idx.ctypes.data_as(POINTER(c_long))))
        return vals, best, idx

    def grad(self, X, which):
        """point j on path which[j] -> (values[M], gradients[M, d]) (ibo_paths_grad); values are eval's bits"""
        X = self._points(X)
        M = X.shape[0]
        wh = np.ascontiguousarray(np.broadcast_to(np.asarray(which), (M,)), dtype=np.int32)
        vals, g = np.empty(M), np.empty((M, self.d))
        check(lib().ibo_paths_grad(self._h, dptr(X), M, wh.ctypes.data_as(POINTER(c_int)), dptr(vals), dptr(g)))
        return vals, g

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().ibo_paths_destroy(self._h)
            self._h = None

    __del__ = close


def acqmax_many(models, lb, ub, acq, ymax, parm, flags=FLAG_MODE_CPP, maxiter=50, maxtime=30, maxsample=10000):
    """independent queries side by side (ibo_acqmax_many): models[q] with incumbent ymax[q] and parameter parm[q];
    returns (opt[nq], optx[nq, d], nsamples[nq], iterations[nq])"""
    nq = len(models)
    lb, ub = as_f64(lb), as_f64(ub)
    ymax = as_f64(np.broadcast_to(np.asarray(ymax, dtype=float), (nq,)))
    parm = as_f64(np.broadcast_to(np.asarray(parm, dtype=float), (nq,)))
    handles = (c_void_p * nq)(*[m.handle for m in models])
    d = models[0].d
    opt, optx = np.empty(nq), np.empty((nq, d))
    ns, it, st = (c_long * nq)(), (c_int * nq)(), (c_int * nq)()
    check(lib().ibo_acqmax_many(nq, handles, dptr(lb), dptr(ub), acq, dptr(ymax), dptr(parm), flags, int(maxiter), int(maxtime),
                                int(maxsample), dptr(opt), dptr(optx), ns, it, st))
    return opt, optx, np.array(ns[:]), np.array(it[:])


class ResidentCandidates(object):
    def __init__(self, model, Xs):
        Xs = as_f64(Xs, 2)
        self.model, self.M = model, Xs.shape[0]
        self._h = c_void_p()
        check(lib().ibo_cands_create(model.handle, dptr(Xs), self.M, ctypes.byref(self._h)))

    def score(self, acq, ymax, parm, flags=FLAG_MODE_CPP, scores_out=None):
        best, bidx, ms = c_double(0), c_long(-1), c_float(0)
        check(lib().ibo_score_resident(self.model.handle, self._h, acq, float(ymax), float(parm), flags,
                                       dptr(scores_out) if scores_out is not None else None,
                                       ctypes.byref(best), ctypes.byref(bidx), ctypes.byref(ms)))
        return best.value, bidx.value, ms.value

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib().ibo_cands_destroy(self._h)
            self._h = None

    __del__ = close
