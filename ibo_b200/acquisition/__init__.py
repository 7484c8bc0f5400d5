"""
Acquisition functions and their maximisers with the reference's public surface
(ego/acquisition/__init__.py:60-197,307-468): EI / PI / UCB objects with scalar `.negf/.f`
(Python-path arithmetic, evaluated on the GPU), and maximizeEI / maximizePI / maximizeUCB /
cdirectGP which run the batched DIRECT driver against the GPU objective.

Not carried over: the RandomForest surrogate branch (cdirectRF / maxRF, out of scope), the
library search loop that spins forever (:336-342) and the broken bare-except fallback (:449-457).
"""
import ctypes

import numpy as np

from .. import _lib
from ..gaussianprocess import GaussianProcess, PrefGaussianProcess, gumbel_draws
from ..utils.optimize import direct, cdirect  # noqa: F401
from ..utils.latinhypercube import lhcSample  # noqa: F401


def _ucb_sbeta(nY, NA, delta):
    """sqrt(2 log(t^(NA/2+2) pi^2 / (3 delta))), t = len(Y)+1; NA/2 is Python-2 integer division (:66)."""
    t = nY + 1
    return np.sqrt(2.0 * np.log(t ** (NA // 2 + 2) * np.pi ** 2 / (3.0 * delta)))


class _Acquisition(object):
    acq = None

    def __init__(self, GP):
        self.GP = GP

    def _parm(self):
        raise NotImplementedError

    def _ymax(self):
        return 0.0

    def negf(self, x):
        """scalar objective at one point (the reference's call shape); prefer f_batch for arrays"""
        x = np.array(x, dtype=float, ndmin=1).reshape(1, -1)
        return -float(self.f_batch(x)[0])

    def f(self, x):
        return -self.negf(x)

    def f_batch(self, Xs):
        """acquisition values for an array of points in one GPU batch (Python-path arithmetic)"""
        if len(self.GP.X) == 0:
            raise ValueError("acquisition over a GP without data")
        sc, _, _, _, _ = self.GP.model.score(Xs, self.acq, self._ymax(), self._parm(), _lib.FLAG_MODE_PY)
        return sc


class UCB(_Acquisition):
    """mu + sqrt(scale * sBeta) * sigma  (:60-75)"""
    acq = _lib.ACQ_UCB

    def __init__(self, GP, NA, delta=0.1, scale=0.2, **kwargs):
        super(UCB, self).__init__(GP)
        self.scale = scale
        self.sBeta = _ucb_sbeta(len(GP.Y), NA, delta)

    def _parm(self):
        return np.sqrt(self.scale * self.sBeta)


class PI(_Acquisition):
    """CDF((mu - (max(Y) + xi)) / sigma)  (:100-114)"""
    acq = _lib.ACQ_PI

    def __init__(self, GP, xi=.01, **kwargs):
        super(PI, self).__init__(GP)
        self.ymax = max(GP.Y)
        self.xi = xi
        self.Z = self.ymax + xi

    def _parm(self):
        return self.xi

    def _ymax(self):
        return self.ymax


class EI(_Acquisition):
    """(mu - max(Y) - xi) CDF(Z) + sigma PDF(Z)  (:138-169)"""
    acq = _lib.ACQ_EI

    def __init__(self, GP, xi=.01, **kwargs):
        super(EI, self).__init__(GP)
        self.ymax = max(GP.Y)
        self.xi = xi

    def _parm(self):
        return self.xi

    def _ymax(self):
        return self.ymax


class MES(_Acquisition):
    """max-value entropy search (Wang & Jegelka 2017) for samples ystar of the maximum: the mean over the samples of
    h(g) = g psi(g) / 2 - log Phi(g), g = (y* - mu) / sigma, psi = phi / Phi (ibo_mes, Python-path arithmetic)"""

    def __init__(self, GP, ystar, **kwargs):
        super(MES, self).__init__(GP)
        self.ystar = np.array(ystar, dtype=float, ndmin=1)
        self.evaluations = 0

    def f_batch(self, Xs):
        if len(self.GP.X) == 0:
            raise ValueError("acquisition over a GP without data")
        self.evaluations += len(Xs)
        return self.GP.model.mes(Xs, self.ystar, _lib.FLAG_MODE_PY)[0]


def cdirectGP(model, bounds, maxiter, maxtime, maxsample, acqfunc=None, xi=-1, beta=-1, scale=-1, delta=-1, polish=0, **kwargs):
    """DIRECT over the GPU acquisition (replaces the ctypes marshalling into libego.acqmaxGP, :307-447).

    Same arguments and return value (opt, optx).  The arithmetic is libego's: libm erf, sigma^2 floor
    1e-8, and the UCB multiplier of :317-319.  No explicit inverse of R is formed (the reference does
    linalg.inv(R) / inv(R + inv(C)) per call, :385-388): the model's device-resident factor is reused.

    polish = k > 0 refines DIRECT's answer by gradient ascent (polishAcquisition) from k starts: DIRECT's optx and the best
    k - 1 of 1024 seeded Latin-hypercube points.  The best polished point is returned, with its FP64 value, only when that
    value beats DIRECT's optx re-scored in the same call; otherwise DIRECT's (opt, optx) come back unchanged.
    cdirectGP.last['polish'] gives the objective evaluations and whether the point moved.
    """
    if polish and kwargs.get('shard'):
        raise ValueError("polish is not supported with shard")
    if acqfunc == 'ei':
        acquisition, parm = _lib.ACQ_EI, xi
    elif acqfunc == 'pi':
        acquisition, parm = _lib.ACQ_PI, xi
    elif acqfunc == 'ucb':
        acquisition = _lib.ACQ_UCB
        t = len(model.Y) + 1
        NA = len(bounds)
        parm = np.sqrt(scale * 2.0 * np.log(t ** (NA // 2 + 2) * np.pi ** 2 / (3.0 * delta)))
    else:
        raise NotImplementedError('unknown acquisition function %s' % acqfunc)
    lower = np.array([b[0] for b in bounds], dtype=float)
    upper = np.array([b[1] for b in bounds], dtype=float)
    flags = _lib.FLAG_MODE_CPP | (_lib.FLAG_DIRECT_SEQ if kwargs.get('sequential') else 0)
    if kwargs.get('shard'):
        # one process per GPU, communicator set up with ibo_comm_init: every DIRECT batch is cut into one slice per rank
        # and the values are all-gathered over NVLink; all ranks must call with the same arguments (SURVEY 8e, config #5)
        flags |= _lib.FLAG_SHARD
    opt, optx, nsamples, iters = model.model.acqmax(lower, upper, acquisition, np.max(model.Y), parm, flags,
                                                   maxiter=maxiter, maxtime=maxtime, maxsample=maxsample)
    cdirectGP.last = dict(nsamples=nsamples, iterations=iters)
    if polish > 0:
        fp64 = _lib.FLAG_MODE_CPP | _lib.FLAG_FP64
        P = np.array(lhcSample(bounds, 1024, seed=_POLISH_SEED), dtype=float)
        sc = model.model.score(P, acquisition, np.max(model.Y), parm, fp64)[0]
        starts = np.r_[np.asarray(optx, dtype=float)[None, :], P[np.argsort(-sc, kind='stable')[:polish - 1]]]
        acq = {_lib.ACQ_EI: 'ei', _lib.ACQ_PI: 'pi', _lib.ACQ_UCB: 'ucb'}[acquisition]
        vals, X, v0, nfev = _polish_model(model, bounds, starts, acq, parm, 'cpp', 100)
        b = int(np.argmax(vals))
        moved = bool(vals[b] > v0[0])
        cdirectGP.last['polish'] = dict(evaluations=nfev, moved=moved)
        if moved:
            return float(vals[b]), X[b]
    return opt, optx


_POLISH_SEED = 0


def _polish(fg, bounds, X0, maxiter=100):
    """Maximise a separable sum of S acquisitions from the starts X0[S, d] with L-BFGS-B.  fg(X[S, d]) -> (values[S],
    gradients[S, d]) is called once per objective evaluation for all starts.  Dimensions with equal bounds stay at that
    bound; the others are clipped into the box.  One final call scores the starts and the results together, and each row keeps
    whichever is better.  Returns (values[S], X[S, d], values of the starts[S], evaluations)."""
    from scipy.optimize import minimize
    b = np.array(bounds, dtype=float).reshape(-1, 2)
    lo, hi = b[:, 0], b[:, 1]
    X0 = np.clip(np.array(X0, dtype=float, ndmin=2), lo, hi)
    S = X0.shape[0]
    free = lo < hi
    nf = int(free.sum())
    state = dict(n=0, scale=None)

    def X_of(z):
        X = X0.copy()
        X[:, free] = np.clip(z.reshape(S, nf), lo[free], hi[free])
        return X

    def obj(z):
        v, g = fg(X_of(z))
        state['n'] += 1
        if state['scale'] is None:       # the first evaluation is at the starts: a fixed scale keeps EI of any size well conditioned
            m = np.max(np.abs(v[np.isfinite(v)])) if np.any(np.isfinite(v)) else 0.0
            state['scale'] = 1.0 / m if m > 0 else 1.0
        f = -state['scale'] * np.sum(v)
        gr = -state['scale'] * g[:, free].ravel()
        if not np.isfinite(f) or not np.all(np.isfinite(gr)):
            return np.inf, np.zeros_like(gr)
        return f, gr

    X = X0
    if nf > 0:
        res = minimize(obj, X0[:, free].ravel(), jac=True, method='L-BFGS-B', bounds=list(zip(np.tile(lo[free], S), np.tile(hi[free], S))),
                       options=dict(maxiter=maxiter, ftol=1e-15, gtol=1e-12))
        X = X_of(res.x)
    v, _ = fg(np.r_[X0, X])
    state['n'] += 1
    v0, v1 = v[:S], v[S:]
    better = v1 > v0
    return np.where(better, v1, v0), np.where(better[:, None], X, X0), v0, state['n']


def _polish_model(GP, bounds, X0, acq, parm, mode, maxiter):
    flags = _lib.FLAG_MODE_PY if mode == 'py' else _lib.FLAG_MODE_CPP
    acq_id = {'ei': _lib.ACQ_EI, 'pi': _lib.ACQ_PI, 'ucb': _lib.ACQ_UCB}[acq]
    ymax = np.max(GP.Y)
    return _polish(lambda X: GP.model.score_grad(X, acq_id, ymax, parm, flags), bounds, X0, maxiter)


def polishAcquisition(GP, bounds, X0, acq='ei', xi=0.01, parm=None, mode='cpp', maxiter=100):
    """Gradient refinement of acquisition maximisers: L-BFGS-B from each start in X0[S, d] within `bounds`, all starts in one
    batched value-and-gradient call (GaussianProcess.score_grad) per evaluation.  Dimensions with equal bounds stay fixed.  Each
    returned row is at least as good as its start (FP64 values).  Returns (values[S], X[S, d])."""
    if len(GP.X) == 0:
        raise ValueError("acquisition over a GP without data")
    vals, X, _, _ = _polish_model(GP, bounds, X0, acq, xi if parm is None else parm, mode, maxiter)
    return vals, X


def thompsonBatch(GP, bounds, q, samples=2048, candidates=None, seed=None, jitter=0.0, method='joint', n_features=2048, polish=False):
    """Thompson sampling of a batch of q points to evaluate in parallel: q posterior draws over a candidate set, each draw's
    maximiser is one point of the batch.

    Candidates are `samples` Latin-hypercube points within `bounds` (lhcSample with `seed`) unless given as an array.
    method='joint': the draws are mu + chol(cov + jitter I) Z with Z = numpy.random.default_rng(seed).standard_normal((M, q))
    (at most 16384 candidates).  method='paths': q sample paths (GaussianProcess.sample_paths with n_features and seed), with no
    limit on the candidates; with polish=True each path's maximiser is then refined by L-BFGS-B on that path's gradient within
    `bounds`, every path in one call per evaluation, and a point is kept only where its path value beats the start's.  Only the
    q argmax indices leave the device.  Two draws can pick the same candidate, so a point may appear more than once in the
    batch.  Returns (points[q, d], indices[q]); the indices name the starting candidates."""
    if len(GP.X) == 0:
        raise ValueError("Thompson sampling over a GP without data")
    if method not in ('joint', 'paths'):
        raise ValueError("unknown method %r" % (method,))
    if polish and method != 'paths':
        raise ValueError("polish=True needs method='paths'")
    if candidates is None:
        candidates = lhcSample(bounds, samples, seed=seed)
    C = np.array(candidates, dtype=float, ndmin=2)
    if method == 'joint':
        Z = np.random.default_rng(seed).standard_normal((C.shape[0], q))
        _, idx = GP.model.posterior_sample(C, Z, jitter, want_F=False)
        return C[idx], idx
    paths = GP.sample_paths(q, n_features, seed)
    try:
        _, idx = paths.argmax(C)
        if np.any(idx < 0):
            raise ValueError("a sample path is NaN at every candidate (NaN in the candidates?)")
        X = C[idx]
        if polish:
            _, X, _, _ = _polish(lambda P: paths.grad(P, np.arange(len(P)) % q), bounds, X)
    finally:
        paths.close()
    return X, idx


def _polish_batches(fg, bounds, starts, pending=None, maxiter=100):
    """L-BFGS-B over whole batches: fg(X[S, n, d]) -> (values[S], gradients[S, n, d]) for S batches of n = q + p points, starts[S, q, d],
    pending[p, d] appended to every batch and held fixed (lo = hi bounds).  Returns (best value, its q free points[q, d], the values
    of the starts[S], evaluations)."""
    b = np.array(bounds, dtype=float).reshape(-1, 2)
    starts = np.array(starts, dtype=float, ndmin=3)
    S, q, d = starts.shape
    P = np.zeros((0, d)) if pending is None else np.array(pending, dtype=float, ndmin=2).reshape(-1, d)
    n = q + P.shape[0]
    X0 = np.concatenate([starts, np.broadcast_to(P, (S,) + P.shape)], axis=1).reshape(S, n * d)
    tb = np.r_[np.tile(b, (q, 1)), np.repeat(P.reshape(-1, 1), 2, axis=1)]

    def flat(X):
        v, g = fg(X.reshape(-1, n, d))
        return v, g.reshape(-1, n * d)
    vals, X, v0, nfev = _polish(flat, tb, X0, maxiter)
    vs = np.where(np.isnan(vals), -np.inf, vals)
    k = int(np.argmax(vs))
    return float(vals[k]), X[k].reshape(n, d)[:q], v0, nfev


def maximizeQEI(GP, bounds, q, samples=512, seed=0, xi=0.01, starts=8, pending=None, jitter=0.0, maxiter=100):
    """Choose q points to evaluate in parallel by maximising their Monte-Carlo batch expected improvement (GaussianProcess.qEI) with
    L-BFGS-B on its exact gradient.  Z is drawn once (numpy.random.default_rng(seed), q + p rows, `samples` columns), so every
    evaluation uses the same common random numbers and the objective is deterministic.  The starts are
    thompsonBatch(GP, bounds, q, seed=seed + k) for k < starts; all of them are polished together, one ibo_qei call per evaluation.
    pending[p, d] are points already under evaluation: they join every batch, held fixed, so the q new points improve on them too.
    Returns (value, batch[q, d]); the value is at least the best start's.  maximizeQEI.last records the evaluations and the values
    of the starts."""
    if len(GP.X) == 0:
        raise ValueError("q-EI over a GP without data")
    p = 0 if pending is None else np.array(pending, dtype=float, ndmin=2).shape[0]
    Z = np.random.default_rng(seed).standard_normal((q + p, samples))
    ymax = np.max(GP.Y)
    X0 = np.array([thompsonBatch(GP, bounds, q, seed=seed + k, jitter=jitter)[0] for k in range(starts)])

    def fg(X):
        v, g, _ = GP.model.qei(X, Z, ymax, xi, jitter)
        return v, g
    val, batch, v0, nfev = _polish_batches(fg, bounds, X0, pending, maxiter)
    maximizeQEI.last = dict(evaluations=nfev, start_values=v0)
    return val, batch


def maximizeQNEI(GP, bounds, q, baseline=None, samples=512, seed=0, starts=8, pending=None, jitter=1e-8, maxiter=100):
    """Choose q points to evaluate in parallel by maximising their Monte-Carlo noisy batch expected improvement
    (GaussianProcess.qNEI): the incumbent is drawn jointly over the `baseline` points (default: the distinct rows of GP.X) instead
    of the fixed max(Y).  maximizeQEI's driver: Z is drawn once (numpy.random.default_rng(seed), P + q + p rows, `samples`
    columns, baseline rows first); the starts are thompsonBatch(GP, bounds, q, seed=seed + k) for k < starts, polished together
    by L-BFGS-B, one ibo_qnei call per evaluation; pending[p, d] join every batch, held fixed.  Returns (value, batch[q, d]); the
    value is at least the best start's.  maximizeQNEI.last records the evaluations, the values of the starts and the baseline."""
    if len(GP.X) == 0:
        raise ValueError("q-NEI over a GP without data")
    base = GP.qnei_baseline() if baseline is None else np.array(baseline, dtype=float, ndmin=2)
    p = 0 if pending is None else np.array(pending, dtype=float, ndmin=2).shape[0]
    Z = np.random.default_rng(seed).standard_normal((base.shape[0] + q + p, samples))
    X0 = np.array([thompsonBatch(GP, bounds, q, seed=seed + k, jitter=jitter)[0] for k in range(starts)])

    def fg(X):
        v, g, _, _ = GP.model.qnei(X, base, Z, jitter)
        return v, g
    val, batch, v0, nfev = _polish_batches(fg, bounds, X0, pending, maxiter)
    maximizeQNEI.last = dict(evaluations=nfev, start_values=v0, baseline=base)
    return val, batch


def _polish_from(fg, bounds, opt, optx, C, cvals, k, maxiter=100):
    """Gradient polish of a DIRECT answer: L-BFGS-B (_polish, fg(X) -> (values, gradients)) from DIRECT's optx and the k - 1
    candidates C with the largest values cvals.  The best polished point replaces (opt, optx) only when its value beats optx
    re-scored in the same call.  Returns (opt, optx, dict(evaluations, moved, starts))."""
    starts = np.r_[np.asarray(optx, dtype=float)[None, :], np.asarray(C, dtype=float)[np.argsort(-np.asarray(cvals), kind='stable')[:k - 1]]]
    vals, X, v0, nfev = _polish(fg, bounds, starts, maxiter)
    b = int(np.argmax(vals))
    moved = bool(vals[b] > v0[0])
    rec = dict(evaluations=nfev, moved=moved, starts=starts)
    return (float(vals[b]), X[b], rec) if moved else (opt, optx, rec)


def maximizeMES(GP, bounds, n_samples=10, seed=0, candidates=None, samples=16384, floor=None, maxiter=50, maxtime=30,
                maxsample=10000, polish=0):
    """Maximise max-value entropy search (MES) with DIRECT.  The samples y* of the maximum come from the Gumbel fit over the
    `candidates` or, by default, over `samples` Latin-hypercube points (lhcSample with `seed`), drawn with `seed` and raised to
    `floor` (GaussianProcess.sample_max_values).  polish = k > 0 refines DIRECT's answer by L-BFGS-B on the gradient of MES from
    DIRECT's optx and the k - 1 candidates of largest MES; the polished point (with its FP64 value) is returned only when it beats
    DIRECT's optx re-scored in the same call.  Returns (opt, optx); maximizeMES.last records ystar, loc, scale, DIRECT's samples
    and the polish evaluations."""
    if len(GP.X) == 0:
        raise ValueError("MES over a GP without data")
    C = np.array(lhcSample(bounds, samples, seed=seed) if candidates is None else candidates, dtype=float, ndmin=2)
    _, loc, scale = GP.model.max_value_gumbel(C, _lib.FLAG_MODE_PY)
    ystar = np.maximum(gumbel_draws(loc, scale, n_samples, seed), np.max(GP.Y) if floor is None else floor)
    obj = MES(GP, ystar)
    opt, optx = _python_direct(obj, bounds, maxiter=maxiter, maxtime=maxtime, maxsample=maxsample)
    maximizeMES.last = dict(ystar=ystar, loc=loc, scale=scale, samples=obj.evaluations, polish=None)
    if polish > 0:
        cvals = GP.model.mes(C, ystar, _lib.FLAG_MODE_PY)[0]
        fg = lambda X: GP.model.mes(X, ystar, _lib.FLAG_MODE_PY, want_grad=True)[:2]        # noqa: E731
        opt, optx, rec = _polish_from(fg, bounds, opt, optx, C, cvals, polish)
        maximizeMES.last['polish'] = dict(evaluations=rec['evaluations'], moved=rec['moved'])
    return opt, optx


def _python_direct(obj, bounds, **kw):
    """useCDIRECT=False route: the same DIRECT driver over the Python-path objective (batched)."""
    opt, optx = direct(obj.negf, bounds, batch_objective=lambda P: -obj.f_batch(P), pure=True, **kw)
    return -opt, optx


def maximizeUCB(model, bounds, delta=0.1, scale=0.2, useCDIRECT=True, maxiter=50, maxtime=30, maxsample=10000, **kwargs):
    """Maximize the upper confidence bound [Srinivas 2009a]  (:78-96)."""
    if not useCDIRECT:
        return _python_direct(UCB(model, len(bounds), delta=delta, scale=scale), bounds,
                              maxiter=maxiter, maxtime=maxtime, maxsample=maxsample)
    if isinstance(model, GaussianProcess):
        return cdirectGP(model, bounds, maxiter, maxtime, maxsample, acqfunc='ucb', delta=delta, scale=scale, **kwargs)
    raise ValueError


def maximizePI(model, bounds, xi=0.01, maxiter=50, maxtime=30, maxsample=10000, useCDIRECT=True, **kwargs):
    """Maximize the probability of improvement [Lizotte 2008]  (:117-134)."""
    if not useCDIRECT:
        return _python_direct(PI(model, xi), bounds, maxiter=maxiter, maxtime=maxtime, maxsample=maxsample)
    if isinstance(model, GaussianProcess):
        return cdirectGP(model, bounds, maxiter, maxtime, maxsample, acqfunc='pi', xi=xi, **kwargs)
    raise ValueError


def maximizeEI(model, bounds, useCDIRECT=True, xi=0.01, maxiter=50, maxtime=30, maxsample=10000, **kwargs):
    """Maximize expected improvement with DIRECT  (:174-197).  Returns (opt, optx)."""
    if not useCDIRECT:
        return _python_direct(EI(model, xi), bounds, maxiter=maxiter, maxtime=maxtime, maxsample=maxsample)
    if isinstance(model, GaussianProcess):
        return cdirectGP(model, bounds, maxiter, maxtime, maxsample, acqfunc='ei', xi=xi, **kwargs)
    raise ValueError


from .gallery import fastUCBGallery  # noqa: E402,F401
