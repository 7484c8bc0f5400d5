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
from ..gaussianprocess import GaussianProcess, PrefGaussianProcess
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


def cdirectGP(model, bounds, maxiter, maxtime, maxsample, acqfunc=None, xi=-1, beta=-1, scale=-1, delta=-1, **kwargs):
    """DIRECT over the GPU acquisition (replaces the ctypes marshalling into libego.acqmaxGP, :307-447).

    Same arguments and return value (opt, optx).  The arithmetic is libego's: libm erf, sigma^2 floor
    1e-8, and the UCB multiplier of :317-319.  No explicit inverse of R is formed (the reference does
    linalg.inv(R) / inv(R + inv(C)) per call, :385-388): the model's device-resident factor is reused.
    """
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
    return opt, optx


def thompsonBatch(GP, bounds, q, samples=2048, candidates=None, seed=None, jitter=0.0):
    """Thompson sampling of a batch of q points to evaluate in parallel: q joint posterior draws over a candidate set, each
    draw's maximiser is one point of the batch.

    Candidates are `samples` Latin-hypercube points within `bounds` (lhcSample with `seed`) unless given as an array.  The
    draws are mu + chol(cov + jitter I) Z with Z = numpy.random.default_rng(seed).standard_normal((M, q)); only the q
    argmax indices leave the device.  Two draws can pick the same candidate, so a point may appear more than once in the
    batch.  Returns (points[q, d], indices[q])."""
    if len(GP.X) == 0:
        raise ValueError("Thompson sampling over a GP without data")
    if candidates is None:
        candidates = lhcSample(bounds, samples, seed=seed)
    C = np.array(candidates, dtype=float, ndmin=2)
    Z = np.random.default_rng(seed).standard_normal((C.shape[0], q))
    _, idx = GP.model.posterior_sample(C, Z, jitter, want_F=False)
    return C[idx], idx


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
