"""
GaussianProcess / PrefGaussianProcess with the reference's public surface
(ego/gaussianprocess/__init__.py:81-527) on top of the CUDA library.

Host code here only owns NumPy buffers and marshals them through ctypes; the correlation matrix,
its Cholesky factor, and every posterior / acquisition evaluation are computed on the GPU
(ibo_b200/csrc/model.cu, score.cu).  There is no CPU fallback: without the library or a device
every numeric method raises.

Differences from the reference that a user can observe (all opt-in or bug fixes, SURVEY.md App. A):
  * `posteriors` and the new `score_batch` evaluate whole candidate arrays in one launch sequence;
    `posterior` keeps the reference's "first point only" contract (:183-184,226).
  * gradient observations (`G`) are rejected: the reference's gradient branches call functions that
    do not exist (:199-206,292).
  * no `pdb.set_trace()` (:382-384) and no library-search spin loop.
"""
from time import time

import numpy as np

from .. import _lib
from .kernel import (GaussianKernel_ard, GaussianKernel_iso, Kernel, MaternKernel3, MaternKernel5,  # noqa: F401
                     MaternKernel5_ard, SVGaussianKernel_ard, SVGaussianKernel_iso, SVKernel)
from .prior import GPMeanPrior, RBFNMeanPrior  # noqa: F401

# -----------------------------------------------------------------------------------------------
# scalar erf / CDF / PDF with the reference's constants (ego/gaussianprocess/__init__.py:55-77).
# Host-side helpers for scalar callers (PrefGP's Laplace terms); the batched versions live in K3.
# -----------------------------------------------------------------------------------------------
_NR = (1.00002368, 0.37409196, 0.09678418, -0.18628806, 0.27886807, -1.13520398, 1.48851587, -0.82215223, 0.17087277)


def erf(z):
    t = 1.0 / (1.0 + 0.5 * abs(z))
    p = 0.0
    for c in reversed(_NR):
        p = c + t * p
    ans = 1 - t * np.exp(-z * z - 1.26551223 + t * p)
    return ans if z >= 0.0 else -ans


def CDF(x):
    return 0.5 * (1 + erf(x * 0.707106))


def PDF(x):
    return np.exp(-(x ** 2 / 2)) * 0.398942


def gumbel_draws(loc, scale, n, seed=None):
    """n draws loc - scale log(-log u) of a Gumbel distribution, u = k / 2^53 for k uniform in 1 .. 2^53 - 1 from
    numpy.random.default_rng(seed): strictly inside (0, 1), so every draw is finite"""
    u = np.random.default_rng(seed).integers(1, 2 ** 53, size=n) / 2.0 ** 53
    return loc - scale * np.log(-np.log(u))


def spectral_draws(kind, rng, F, d):
    """F frequencies [F, d] from the spectral density of kernel `kind` (_lib.KERNEL_*) in unit-length-scale coordinates: N(0, I)
    for the squared exponential; for Matern-nu (nu = 3/2, 5/2) the multivariate Student-t with 2 nu degrees of freedom,
    z sqrt(2 nu / u) with z ~ N(0, I) and one u ~ chi^2(2 nu) per frequency (z first, then u)"""
    if kind in (_lib.KERNEL_SE_ARD, _lib.KERNEL_SE_ISO):
        return rng.standard_normal((F, d))
    if kind == _lib.KERNEL_MATERN3:
        nu = 1.5
    elif kind in (_lib.KERNEL_MATERN5, _lib.KERNEL_MATERN5_ARD):
        nu = 2.5
    else:
        raise ValueError("unknown kernel kind %r" % (kind,))
    z = rng.standard_normal((F, d))
    u = rng.chisquare(2 * nu, size=F)
    return z * np.sqrt(2 * nu / u)[:, None]


def path_draws(kind, d, n_features, n_paths, n_train, seed=None):
    """the draws of GaussianProcess.sample_paths, from numpy.random.default_rng(seed) in this order: omega = spectral_draws(kind,
    rng, F, d), phase ~ U(0, 2 pi) [F], w ~ N(0, 1) [F, S], e ~ N(0, 1) [n_train, S]"""
    if n_features < 1 or n_paths < 1:
        raise ValueError("n_features and n_paths must be at least 1")
    rng = np.random.default_rng(seed)
    omega = spectral_draws(kind, rng, n_features, d)
    phase = rng.uniform(0.0, 2 * np.pi, n_features)
    w = rng.standard_normal((n_features, n_paths))
    e = rng.standard_normal((n_train, n_paths))
    return omega, phase, w, e


class PosteriorPaths(object):
    """S posterior sample paths f_s(x) = mu(x) + phi(x)^T w_s - k(x)^T c_s (GaussianProcess.sample_paths): deterministic functions,
    evaluated on the device at any number of points.  They sample the latent function (no observation noise).  A snapshot: later
    changes to the GP do not change them."""

    def __init__(self, paths):
        self._paths = paths
        self.n_paths = paths.S

    def __call__(self, X):
        """values F[M, S] of every path at the points X"""
        return self._paths.eval(_as_points(X), want_values=True)[0]

    def argmax(self, X):
        """per path the maximum over the points X and its index -> (best[S], idx[S]); lowest index wins ties"""
        _, best, idx = self._paths.eval(_as_points(X), want_values=False)
        return best, idx

    def grad(self, X, which):
        """point j on path which[j] -> (values[M], gradients[M, d])"""
        return self._paths.grad(_as_points(X), which)

    def close(self):
        self._paths.close()


def _as_points(X):
    X = np.asarray(X, dtype=float)
    return X.reshape(-1, 1) if X.ndim == 1 else X


class GaussianProcess(object):

    append_above = 256       # addData appends on the device when the resident model has at least this many points ...
    append_max_rows = 64     # ... and at most this many rows arrive at once (beyond that a rebuild is cheaper)

    def __init__(self, kernel, X=None, Y=None, prior=None, noise=.1, gnoise=1e-4, G=None, device=0):
        """
        @param kernel:  kernel object (ibo_b200.gaussianprocess.kernel)
        @param prior:   GP mean prior (RBFNMeanPrior) or None
        @param noise:   noise hyperparameter sigma^2_n
        @param X, Y:    initial training data / observations
        @param device:  CUDA device ordinal holding the model
        """
        self.kernel = kernel
        self.prior = prior
        self.noise = noise
        self.gnoise = np.array(gnoise, ndmin=1)
        self.device = device
        if (X is None) != (Y is None):
            raise ValueError
        if G is not None:
            raise NotImplementedError("gradient observations are not supported (dead code in the reference)")
        self.X = np.zeros((0, 0))
        self.Y = np.zeros((0))
        self.G = None
        self.name = 'GP'
        self.starttime = time()
        self._model = None          # _lib.Model for (X, Y [, Laplace term])
        self._laplace = None        # PrefGaussianProcess: ("pairs", a, b, w, cdiag) or ("dense", C); inv(C) is formed on the device
        self._Cinv_host = None
        self._augmodel = None
        self.augX = None
        self.selected = None
        self.endtime = None
        if X is not None:
            self.addData(X, Y)

    # ---- device model -------------------------------------------------------------------------
    def _invalidate(self):
        for attr in ("_model", "_augmodel"):
            m = getattr(self, attr, None)
            if m is not None:
                m.close()
            setattr(self, attr, None)

    def _build(self, X, Y, Cinv=None, laplace=None):
        kind, hyper = self.kernel.spec(X.shape[1])
        if laplace is not None:
            if self.prior is not None:
                raise NotImplementedError("a preference GP has no mean prior")
            if laplace[0] == "pairs":
                return _lib.Model(kind, hyper, X, Y, self.noise, pref=laplace[1:], device=self.device)
            return _lib.Model(kind, hyper, X, Y, self.noise, C=laplace[1], device=self.device)
        return _lib.Model(kind, hyper, X, Y, self.noise, Cinv=Cinv, prior=self.prior, device=self.device)

    @property
    def _Cinv(self):
        """inv(C) of a fitted preference model, read back from the device on demand (None for a plain GP)"""
        if self._laplace is None:
            return None
        if self._Cinv_host is None:
            self._Cinv_host = self.model.matrix(3)
        return self._Cinv_host

    @property
    def model(self):
        """the device-resident model (L, W = inv(L), beta), built on first use after a data change"""
        if self._model is None:
            if len(self.X) == 0:
                raise ValueError("GP has no data")
            self._model = self._build(self.X, self.Y, laplace=self._laplace)
            if self.augX is not None:
                self._attach_aug()
        return self._model

    @property
    def R(self):
        """correlation matrix K_offdiag + (1+noise) I (:134-143), computed on the device"""
        if len(self.X) == 0:
            return None
        A = self.model.matrix(0)
        return A if self._Cinv is None else A - self._Cinv

    @property
    def L(self):
        """lower Cholesky factor of R (or of R + inv(C) for a fitted PrefGaussianProcess)"""
        return None if len(self.X) == 0 else self.model.matrix(1)

    # ---- posterior ----------------------------------------------------------------------------
    def posterior(self, X, getvar=True):
        """Posterior mean and variance at a point X (first row if several are given, as the reference)."""
        if len(self.X) == 0:
            m = 0.0 if self.prior is None else self.prior.mu(np.array(X, dtype=float, ndmin=2)[0])
            return (m, 1.0) if getvar else m
        X = np.array(X, dtype=float, ndmin=2)
        mu, s2 = self.model.posterior(X[:1], _lib.FLAG_MODE_PY)
        if getvar:
            return float(mu[0]), float(s2[0])
        return float(mu[0])

    def posteriors(self, X):
        """arrays of posterior means and variances for the points in X, one batched launch (:231-244)"""
        X = np.asarray(X, dtype=float)
        if X.ndim == 1:
            X = X.reshape(-1, 1)
        if len(self.X) == 0:
            m = np.array([0.0 if self.prior is None else self.prior.mu(x) for x in X])
            return m, np.ones(len(X))
        return self.model.posterior(X, _lib.FLAG_MODE_PY)

    def _candidates(self, X):
        if len(self.X) == 0:
            raise ValueError("joint posterior of a GP without data")
        X = np.asarray(X, dtype=float)
        return X.reshape(-1, 1) if X.ndim == 1 else X

    def posterior_cov(self, X):
        """joint posterior over the points in X -> (mu[M], cov[M, M]).  mu is what `posteriors` returns; diag(cov) is its
        sigma^2 before clipping (the variance of an observation: 1 + noise - v.v)."""
        return self.model.posterior_cov(self._candidates(X))

    def sample_posterior(self, X, n_samples=1, seed=None, jitter=0.0):
        """joint draws of the posterior at the points in X -> F[M, n_samples] = mu + chol(cov + jitter I) Z, with
        Z = numpy.random.default_rng(seed).standard_normal((M, n_samples)): a seed reproduces the draws exactly.
        Raises NotPositiveDefinite when cov + jitter I is not positive definite (near-duplicate points); a small jitter helps."""
        X = self._candidates(X)
        Z = np.random.default_rng(seed).standard_normal((X.shape[0], n_samples))
        return self.model.posterior_sample(X, Z, jitter)[0]

    def score_batch(self, Xs, acq='ei', xi=0.01, parm=None, mode='py', want_posterior=False, out=None, int8=None):
        """Acquisition values for a candidate array (batched EI.negf / PI.negf / UCB.negf, negated).

        Returns (scores, best_score, best_index[, mu, sigma2]).  `parm` overrides xi (UCB multiplier).
        Batches of more than 2048 candidates take the INT8 tensor-core path by default (sigma^2 through an exact-integer
        emulation of the FP64 triangular GEMM, about 4x the DMMA rate at the accuracy of the FP64 GEMM; library option "int8");
        `int8=False` forces the FP64 DMMA kernels for this call (IBO_FLAG_FP64), `int8=True` the INT8 path (IBO_FLAG_INT8)."""
        acq_id = {'ei': _lib.ACQ_EI, 'pi': _lib.ACQ_PI, 'ucb': _lib.ACQ_UCB}[acq]
        flags = (_lib.FLAG_MODE_PY if mode == 'py' else _lib.FLAG_MODE_CPP) | (0 if int8 is None else (_lib.FLAG_INT8 if int8 else _lib.FLAG_FP64))
        sc, mu, s2, best, bidx = self.model.score(Xs, acq_id, np.max(self.Y), xi if parm is None else parm, flags,
                                                  want_posterior=want_posterior, out=out)
        if want_posterior:
            return sc, best, bidx, mu, s2
        return sc, best, bidx

    def posterior_grad(self, X, mode='py'):
        """posterior at the points in X and its gradient with respect to the point -> (mu[M], s2[M], dmu[M, d], ds2[M, d]).
        Values are those of the FP64 kernels; ds2 = 0 where s2 is clipped (floor by mode, ceiling 10)."""
        flags = _lib.FLAG_MODE_PY if mode == 'py' else _lib.FLAG_MODE_CPP
        return self.model.posterior_grad(self._candidates(X), flags)

    def score_grad(self, Xs, acq='ei', xi=0.01, parm=None, mode='py'):
        """acquisition values at the points in Xs and their gradient with respect to the point -> (scores[M], dscores[M, d]),
        with score_batch's incumbent and defaults; the values are score_batch's with int8=False."""
        acq_id = {'ei': _lib.ACQ_EI, 'pi': _lib.ACQ_PI, 'ucb': _lib.ACQ_UCB}[acq]
        flags = _lib.FLAG_MODE_PY if mode == 'py' else _lib.FLAG_MODE_CPP
        return self.model.score_grad(self._candidates(Xs), acq_id, np.max(self.Y), xi if parm is None else parm, flags)

    def qEI(self, batches, samples=512, seed=None, xi=0.01, jitter=0.0, Z=None, grad=False):
        """Monte-Carlo expected improvement of batches of points evaluated together (q-EI) over the incumbent max(Y):
        batches[B, q, d] (or one batch [q, d]) -> values[B] (a float for one batch), and with grad=True also the gradient with
        respect to the points [B, q, d] (or [q, d]).  The draws are mu + chol(cov + jitter I) Z with
        Z = numpy.random.default_rng(seed).standard_normal((q, samples)) unless Z[q, S] is given: the same Z makes every call
        score with the same common random numbers.  A batch whose cov + jitter I is not positive definite (e.g. a repeated point
        without noise) gets NaN."""
        if len(self.X) == 0:
            raise ValueError("q-EI of a GP without data")
        Xb = np.asarray(batches, dtype=float)
        one = Xb.ndim == 2
        Xb = Xb[None] if one else Xb
        if Z is None:
            Z = np.random.default_rng(seed).standard_normal((Xb.shape[1], samples))
        vals, dv, _ = self.model.qei(Xb, Z, np.max(self.Y), xi, jitter, want_grad=grad)
        if one:
            vals, dv = float(vals[0]), (dv[0] if grad else None)
        return (vals, dv) if grad else vals

    def qNEI(self, batches, baseline=None, samples=512, seed=None, jitter=1e-8, Z=None, grad=False):
        """Monte-Carlo noisy expected improvement of batches of points evaluated together (q-NEI, Letham et al. 2019): the
        incumbent is max_i f(x_i) over the `baseline` points (default: the distinct rows of X, in order of first appearance),
        drawn jointly with the batch from the latent posterior, instead of the fixed number max(Y).  batches[B, q, d] (or one
        batch [q, d]) -> values[B] (a float for one batch), and with grad=True also the gradient with respect to the points
        [B, q, d] (or [q, d]).  Z = numpy.random.default_rng(seed).standard_normal((P + q, samples)) unless Z[P + q, S] is given
        (baseline rows first).  Raises NotPositiveDefinite when the baseline's covariance + jitter I is not positive definite
        (a repeated baseline point with jitter 0); a batch whose own factorisation fails gets NaN."""
        if len(self.X) == 0:
            raise ValueError("q-NEI of a GP without data")
        Xb = np.asarray(batches, dtype=float)
        one = Xb.ndim == 2
        Xb = Xb[None] if one else Xb
        base = self.qnei_baseline() if baseline is None else np.array(baseline, dtype=float, ndmin=2)
        if Z is None:
            Z = np.random.default_rng(seed).standard_normal((base.shape[0] + Xb.shape[1], samples))
        vals, dv, _, _ = self.model.qnei(Xb, base, Z, jitter, want_grad=grad)
        if one:
            vals, dv = float(vals[0]), (dv[0] if grad else None)
        return (vals, dv) if grad else vals

    def qnei_baseline(self):
        """the distinct rows of X in order of first appearance: q-NEI's default baseline"""
        X = np.asarray(self.X, dtype=float)
        _, idx = np.unique(X, axis=0, return_index=True)
        return X[np.sort(idx)]

    def sample_paths(self, n_paths, n_features=2048, seed=None):
        """n_paths posterior sample paths by pathwise conditioning (Matheron's rule) with n_features random Fourier features of the
        prior -> PosteriorPaths.  The draws come from numpy.random.default_rng(seed) in the order of `path_draws` (frequencies,
        phases, w, e): a seed reproduces the paths exactly.  Unlike sample_posterior there is no limit on the number of points."""
        if len(self.X) == 0:
            raise ValueError("sample paths of a GP without data")
        kind, _ = self.kernel.spec(self.X.shape[1])
        ng = len(self.augX) if self.augX is not None else len(self.X)
        omega, phase, w, e = path_draws(kind, self.X.shape[1], n_features, n_paths, ng, seed)
        return PosteriorPaths(self.model.sample_paths(omega, phase, w, e))

    def sample_max_values(self, X, n_samples=10, seed=None, floor=None, method='gumbel', jitter=0.0, n_features=2048):
        """samples y*[n_samples] of the maximum of f over the points in X, for max-value entropy search (`mes`).
        method='gumbel' (Wang & Jegelka 2017): the Gumbel fit of F(y) = prod_i Phi((y - mu_i) / s_i) over X
        (ibo_max_value_gumbel), y* = loc - scale log(-log u) for u from numpy.random.default_rng(seed), strictly inside (0, 1).
        method='joint': the maxima over X of joint posterior draws (sample_posterior with seed and jitter; at most 16384
        points), which ignore no correlation.  method='paths': the maxima over X of sample_paths(n_samples, n_features, seed), with
        no limit on the number of points.  Samples below `floor` (default max(Y)) are raised to it."""
        X = self._candidates(X)
        if method == 'gumbel':
            _, loc, scale = self.model.max_value_gumbel(X, _lib.FLAG_MODE_PY)
            ys = gumbel_draws(loc, scale, n_samples, seed)
        elif method == 'joint':
            ys = np.max(self.sample_posterior(X, n_samples, seed, jitter), axis=0)
        elif method == 'paths':
            paths = self.sample_paths(n_samples, n_features, seed)
            ys = paths.argmax(X)[0]
            paths.close()
        else:
            raise ValueError("unknown method %r" % (method,))
        return np.maximum(ys, np.max(self.Y) if floor is None else floor)

    def mes(self, Xs, ystar, grad=False, int8=None, mode='py'):
        """max-value entropy search at the points in Xs for samples ystar of the maximum (sample_max_values): the mean over
        the samples of h(g) = g psi(g) / 2 - log Phi(g), g = (y* - mu) / sigma, psi = phi / Phi -> values[M], and with grad=True
        also their gradient with respect to the point [M, d] (values then those of the FP64 kernels).  `int8` and `mode` as in
        score_batch; sigma^2 is the same clipped variance of a noisy observation."""
        flags = (_lib.FLAG_MODE_PY if mode == 'py' else _lib.FLAG_MODE_CPP) | (0 if int8 is None else (_lib.FLAG_INT8 if int8 else _lib.FLAG_FP64))
        vals, dv, _, _ = self.model.mes(self._candidates(Xs), ystar, flags, want_grad=grad)
        return (vals, dv) if grad else vals

    def mu(self, x):
        return self.posterior(x, getvar=False)

    def negmu(self, x):
        return -self.mu(x)

    # ---- data ---------------------------------------------------------------------------------
    def addData(self, X, Y, G=None):
        """Add observations and update (:267-308).  X is (N,D) (or one D-vector), Y an N-vector."""
        if G is not None:
            raise NotImplementedError("gradient observations are not supported (dead code in the reference)")
        X = np.array(X, dtype=float, ndmin=2)
        Y = np.array(Y, dtype=float, ndmin=1).flatten()
        assert len(Y) == len(X), 'wrong number of Y-observations given'
        if len(self.X) == 0 and len(self.gnoise) == 1:
            self.gnoise = np.tile(self.gnoise, X.shape[1])
        if len(self.X) == 0:
            self.X, self.Y = X.copy(), Y.copy()
            self._invalidate()
            return
        nold = len(self.X)
        self.X = np.r_[self.X, X]
        self.Y = np.r_[self.Y, Y]
        # The factor of the enlarged matrix has the old factor as its leading block (:300-308).  Large resident
        # models get the new rows appended on the device (O(N^2) per point, ibo_model_append); small ones are simply
        # rebuilt (sub-millisecond, and a rebuilt model is a pure function of (X, Y), which keeps the reference's
        # sequential == batch training property, ego/unittest_GP.py:109-156, exact).
        if (self._model is not None and self._laplace is None and self._augmodel is None and self.augX is None
                and nold >= self.append_above and len(X) <= self.append_max_rows):
            try:
                self._model.append(X, Y)
                return
            except np.linalg.LinAlgError:
                self._invalidate()
                raise
        self._invalidate()

    def getYfromX(self, qx):
        for x, y in zip(self.X, self.Y):
            if np.all(qx == x):
                return y
        return None

    def done(self, x):
        self.selected = x
        self.endtime = time()

    # aug* attributes exist on every GP in the reference (:118-120)
    @property
    def augR(self):
        return None if self._augmodel is None else self._augmodel.matrix(0) - self._augCinv

    @property
    def augL(self):
        return None if self._augmodel is None else self._augmodel.matrix(1)

    def _attach_aug(self):
        n, na = len(self.X), len(self.augX)
        Cinv = np.zeros((na, na))
        if self._Cinv is not None:
            Cinv[:n, :n] = self._Cinv
        self._augCinv = Cinv
        # build the new factor first and swap it in before the old one goes away: if the build fails (not positive definite,
        # out of memory) the main model must not keep pointing at a destroyed variance model
        old = self._augmodel
        try:
            new = self._build(self.augX, np.zeros(na), Cinv)
        except Exception:
            self._model.set_variance_model(None)
            self._augmodel = None
            if old is not None:
                old.close()
            raise
        self._model.set_variance_model(new)
        self._augmodel = new
        if old is not None:
            old.close()

    def __del__(self):
        try:
            self._invalidate()
        except Exception:
            pass


class PrefGaussianProcess(GaussianProcess):
    """
    GP trained on pairwise preferences with a Laplace approximation (:331-527).  Triples are
    (xv, xu, d): xv preferred to xu, d = degree (0 standard, 1 greatly preferred).

    Everything numerical runs on the device: the MAP fit of the latents (ibo_pref_fit, Newton in whitened coordinates), the
    assembly of the Laplace matrix C from the preference pairs, inv(C) (Cholesky + triangular inverse + Gram product -- no
    explicit inverse on the host), L = chol(R + inv(C)), posteriors and acquisition.  The host indexes the distinct points and
    evaluates the P pair weights.  `reference_exact = True` restores the reference's optimiser for the latents (SciPy BFGS on
    numerical gradients, :441-442; ibo_b200/gaussianprocess/reference_fit.py) for problems small enough to afford it.
    `fromLaplace` builds the process directly from a fitted (X, Y, C).
    """

    reference_exact = False

    def __init__(self, kernel, prefs=None, **kwargs):
        super(PrefGaussianProcess, self).__init__(kernel, **kwargs)
        self.preferences = []
        self._pairs = None          # (a, b, w): C = cdiag I + sum w (e_a - e_b)(e_a - e_b)^T
        self._denseC = None
        self._cdiag = 5.0
        if prefs is not None:
            self.addPreferences(prefs)

    @classmethod
    def fromLaplace(cls, kernel, X, Y, C, **kwargs):
        gp = cls(kernel, **kwargs)
        gp.X = np.array(X, dtype=float, ndmin=2)
        gp.Y = np.array(Y, dtype=float).reshape(-1)
        gp._denseC = np.array(C, dtype=float)
        gp._factor_with_C()
        return gp

    @property
    def C(self):
        """the Laplace matrix (:461-486), assembled on the host only when somebody asks for it"""
        if self._denseC is not None:
            return self._denseC
        if self._pairs is None:
            return None
        a, b, w = self._pairs
        n = len(self.X)
        C = np.eye(n) * self._cdiag
        keep = a != b
        np.add.at(C, (a[keep], a[keep]), w[keep]); np.add.at(C, (b[keep], b[keep]), w[keep])
        np.subtract.at(C, (a[keep], b[keep]), w[keep]); np.subtract.at(C, (b[keep], a[keep]), w[keep])
        return C

    def _factor_with_C(self):
        """L = chol(R + inv(C)) on the device, retrying with C += I up to 10 times when not SPD (:487-498)."""
        for attempt in range(11):
            self._invalidate()
            self._Cinv_host = None
            if self._denseC is not None:
                self._laplace = ("dense", self._denseC)
            else:
                self._laplace = ("pairs",) + tuple(self._pairs) + (self._cdiag,)
            try:
                self.model   # builds and factorises on the device; raises NotPositiveDefinite
                return
            except np.linalg.LinAlgError:
                print('[addPreferences] GP.C matrix is ill-conditioned, adding regularizer delta = %d' % (attempt + 1))
                if self._denseC is not None:
                    self._denseC = self._denseC + np.eye(len(self.X))
                else:
                    self._cdiag += 1.0
        raise np.linalg.LinAlgError("R + inv(C) is not positive definite after 10 regularisation steps")

    def addPreferences(self, prefs, useC=True, showPrefLikelihood=False):
        self.preferences.extend(prefs)
        # index the distinct points in order of first appearance (:391-408)
        x2ind, prefinds, winners = {}, [], set()
        for v, u, d in self.preferences:
            v, u = tuple(v), tuple(u)
            winners.add(v)
            for p in (v, u):
                if p not in x2ind:
                    x2ind[p] = len(x2ind)
            prefinds.append((x2ind[v], x2ind[u], d))
        newX = np.array([x for x, _ in sorted(x2ind.items(), key=lambda kv: kv[1])], dtype=float)
        # warm start from the previous latent values (:410-430)
        lastY = dict((tuple(x), y) for x, y in zip(self.X, self.Y))
        ymax, ymin = (max(self.Y), min(self.Y)) if len(self.Y) > 0 else (.5, -.5)
        start = np.array([lastY.get(tuple(x), ymax if tuple(x) in winners else ymin) for x in newX], dtype=float)
        # R and its factor come from the device (:433-438)
        self._invalidate()
        self._laplace, self._pairs, self._denseC, self._Cinv_host, self.augX = None, None, None, None, None
        self._cdiag = 5.0
        self.X, self.Y = newX, start.copy()
        vi = np.array([p[0] for p in prefinds]); ui = np.array([p[1] for p in prefinds])
        dg = np.array([p[2] for p in prefinds], dtype=float)
        # The reference minimises S (:373-386) with BFGS on *numerical* gradients (:442), i.e. N+1 evaluations of an O(N^2)
        # functional per step -- hopeless at BASELINE config #3's ~1000 points.  Here S is minimised on the device by Newton's
        # method (ibo_pref_fit: same functional, same minimiser, reached to 1e-9 instead of BFGS's 1e-5 tolerance).
        self.fit_info = None
        if self.reference_exact:
            from .reference_fit import bfgs_latents
            self.Y = bfgs_latents(self.L, vi, ui, dg, start)
        else:
            self.Y, Sval, gnorm, iters = self.model.pref_fit(vi, ui, dg, start)
            self.fit_info = dict(S=Sval, gnorm=gnorm, newton_iterations=iters)
        # ordering fix-up (:445-458)
        losers = set(tuple(c1) for _, c1, _ in self.preferences)
        for r, c, _ in self.preferences:
            r, c = tuple(r), tuple(c)
            if self.Y[x2ind[r]] <= self.Y[x2ind[c]]:
                if r not in losers:          # nothing is preferred to r: bump it above c
                    self.Y[x2ind[r]] = self.Y[x2ind[c]] + .1
        # Laplace C matrix (:461-486): each preference (a,b) adds w to C[a,a], C[b,b] and -w to C[a,b], C[b,a]
        self._invalidate()
        mu_all = self.posteriors(self.X)[0]
        dd = (mu_all[vi] - mu_all[ui]) / (np.sqrt(2) * np.sqrt(self.noise))
        cdf = np.maximum(np.array([CDF(z) for z in dd]), 1e-10)
        pdf = np.maximum(np.array([PDF(z) for z in dd]), 1e-10)
        w = 1.0 / (2 * self.noise) * (pdf ** 2 / cdf ** 2 + dd * pdf / cdf)
        self._pairs = (vi.astype(np.int32), ui.astype(np.int32), w)
        self._factor_with_C()

    def addObservationPoint(self, X):
        """Add a point at which we will observe but have no observation yet (:502-519): the variance is
        then taken from the augmented factor chol(augR + pad(inv(C))) while the mean keeps (X, L)."""
        X = np.array(X, dtype=float, ndmin=2)
        self.augX = self.X.copy() if self.augX is None else self.augX
        self.augX = np.r_[self.augX, X]
        self.model
        self._attach_aug()

    def addData(self, X, Y, G=None):
        raise NotImplementedError("can't (yet) add explicit ratings to preference GP")
