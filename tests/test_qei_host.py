"""CPU tests of the batch expected improvement: the oracle's gradient against central finite differences of its own values (fixed
Z, points away from argmax ties and from zero improvement), its reverse Cholesky, its value at q = 1, the batch polish driver run on
the oracle, and the argument checks of ibo_qei (no device touched)."""
import ctypes

import numpy as np
import pytest

from ibo_b200 import _lib
from ibo_b200.acquisition import _polish_batches
from oracle import ibo_oracle as orc
import joint_oracle as jo
import qei_oracle as qo

KINDS = [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_SE_ISO, [.3]), (orc.K_MATERN3, [.5, .9]), (orc.K_MATERN5, [.4, .8]),
         (orc.K_MATERN5_ARD, [.3, .4, .5, .95])]


def _oracle(kind, hyper, N, d, seed, noise=0.1, prior=None):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    return orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior), rs


def _margin(o, Xb, Z, ymax, xi):
    """smallest distance of any sample to a kink of the integrand: the gap between its two largest draws, and |improvement|"""
    mu, Sig = jo.posterior_joint(o, Xb)
    F = mu[:, None] + np.linalg.cholesky(Sig).dot(Z)
    Fs = np.sort(F, axis=0)
    gap = Fs[-1] - Fs[-2] if F.shape[0] > 1 else np.full(F.shape[1], np.inf)
    return min(np.min(gap), np.min(np.abs(Fs[-1] - ymax - xi)))


def _check_fd(o, Xb, Z, ymax, xi, h=1e-6, tol=1e-6):
    assert _margin(o, Xb, Z, ymax, xi) > 1e-4
    v, G = qo.qei_batch(o, Xb, Z, ymax, xi)
    assert v > 0 and np.any(G != 0)
    fd = np.zeros_like(Xb)
    for j in range(Xb.shape[0]):
        for t in range(Xb.shape[1]):
            E = np.zeros_like(Xb)
            E[j, t] = h
            fd[j, t] = (qo.qei_batch(o, Xb + E, Z, ymax, xi, grad=False) - qo.qei_batch(o, Xb - E, Z, ymax, xi, grad=False)) / (2 * h)
    assert np.max(np.abs(G - fd)) <= tol * np.max(np.abs(fd)), np.max(np.abs(G - fd)) / np.max(np.abs(fd))


@pytest.mark.parametrize("kind,hyper", KINDS)
def test_gradient_matches_finite_differences(kind, hyper):
    o, rs = _oracle(kind, hyper, 40, 3, 1)
    Xb = rs.rand(3, 3)
    Z = np.random.default_rng(2).standard_normal((3, 24))
    _check_fd(o, Xb, Z, o.Y.max() - 0.3, 0.01)


@pytest.mark.parametrize("q,S", [(1, 32), (3, 32), (32, 8)])
def test_gradient_matches_finite_differences_over_q(q, S):
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 3)
    Xb = rs.rand(q, 3)
    Z = np.random.default_rng(q).standard_normal((q, S))
    _check_fd(o, Xb, Z, o.Y.max() - 0.5, 0.01)


def test_gradient_with_prior_and_variance_model():
    d = 2
    prior = orc.PriorSpec(np.random.RandomState(5).rand(3, d), [0.5, -0.2, 0.3], 3.0, np.zeros(d), np.ones(d))
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, d, 3, prior=prior)
    Xb = rs.rand(4, d)
    Z = np.random.default_rng(7).standard_normal((4, 24))
    _check_fd(o, Xb, Z, o.Y.max() - 0.3, 0.01)
    o.augX = np.r_[o.X, rs.rand(4, d)]
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, o.augX, o.noise))
    _check_fd(o, Xb, Z, o.Y.max() - 0.3, 0.01)


def test_reverse_cholesky_matches_finite_differences():
    rs = np.random.RandomState(11)
    for q in (1, 2, 5, 12):
        A = rs.randn(q, q)
        Sig = A.dot(A.T) + q * np.eye(q)
        C = np.tril(rs.randn(q, q))                                   # f(Sigma) = sum C o chol(Sigma): Lbar = C
        Gbar = qo.chol_rev(np.linalg.cholesky(Sig), C)
        assert np.allclose(Gbar, Gbar.T, rtol=0, atol=1e-14)
        E = rs.randn(q, q)
        E = E + E.T
        h = 1e-6
        fd = (np.sum(C * np.linalg.cholesky(Sig + h * E)) - np.sum(C * np.linalg.cholesky(Sig - h * E))) / (2 * h)
        assert abs(np.sum(Gbar * E) - fd) <= 1e-7 * max(1.0, abs(fd))


def test_q1_value_is_the_mean_improvement_of_one_point():
    o, rs = _oracle(orc.K_MATERN5_ARD, [.3, .4, .5, .95], 40, 3, 4)
    x = rs.rand(1, 3)
    Z = np.random.default_rng(0).standard_normal((1, 1000))
    ymax, xi, jitter = o.Y.max(), 0.01, 1e-3
    mu, s2 = o.posterior_batch(x, floor=-np.inf)
    ref = np.mean(np.maximum(0.0, mu[0] + np.sqrt(s2[0] + jitter) * Z[0] - ymax - xi))
    assert abs(qo.qei_batch(o, x, Z, ymax, xi, jitter, grad=False) - ref) <= 1e-12 * max(ref, 1e-5)


def test_batch_polish_never_loses_keeps_pending_and_bounds():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 6)
    bounds = [[0., 1.], [0.1, 0.9], [0.2, 0.9]]
    q, S = 3, 64
    pending = rs.rand(2, 3) * 0.5
    Z = np.random.default_rng(1).standard_normal((q + 2, S))
    ymax = o.Y.max()
    fg = lambda X: qo.qei(o, X, Z, ymax, 0.01)                         # noqa: E731
    b = np.array(bounds)
    starts = b[:, 0] + (b[:, 1] - b[:, 0]) * rs.rand(4, q, 3)
    val, batch, v0, nfev = _polish_batches(fg, bounds, starts, pending, maxiter=30)
    assert batch.shape == (q, 3) and nfev >= 2
    assert np.array_equal(v0, fg(np.concatenate([starts, np.broadcast_to(pending, (4, 2, 3))], axis=1))[0])
    assert val >= np.max(v0)
    assert np.all(batch >= b[:, 0]) and np.all(batch <= b[:, 1])
    full = np.r_[batch, pending][None]
    assert abs(fg(full)[0][0] - val) <= 1e-12 * val
    assert val > np.max(v0)                                           # the gradient steps moved the best start


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    fake = ctypes.create_string_buffer(1 << 16)                       # never dereferenced: every scalar check comes first
    h = ctypes.cast(fake, ctypes.c_void_p)
    x = np.zeros((4, 2)); z = np.zeros(64); o = np.zeros(64)
    p = _lib.dptr
    nbad = ctypes.c_int(5)
    good = dict(m=h, X=p(x), B=2, q=2, Z=p(z), S=4, jitter=0.0, v=p(o))
    bad = [dict(m=None), dict(X=None), dict(Z=None), dict(v=None), dict(B=0), dict(B=-3), dict(q=0), dict(q=33), dict(S=0),
           dict(S=65537), dict(jitter=-1e-9), dict(jitter=float("nan"))]
    for change in bad:
        a = dict(good, **change)
        rc = L.ibo_qei(a["m"], a["X"], a["B"], a["q"], a["Z"], a["S"], 0.0, 0.01, a["jitter"], a["v"], p(o), ctypes.byref(nbad))
        assert rc == _lib.E_BADARG, change
        assert nbad.value == 0
