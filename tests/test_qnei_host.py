"""CPU tests of the noisy batch expected improvement (q-NEI): the oracle's gradient against central finite differences of its own
values (fixed Z, away from argmax ties and from zero improvement), its Monte-Carlo value against the closed form at q = P = 1, its
identity with q-EI for a baseline point no kernel reaches, the batch polish driver run on it, and the argument checks of ibo_qnei
(no device touched)."""
import ctypes
import math

import numpy as np
import pytest

from ibo_b200 import _lib
from ibo_b200.acquisition import _polish_batches
from oracle import ibo_oracle as orc
import qei_oracle as qo
import qnei_oracle as no

KINDS = [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_SE_ISO, [.3]), (orc.K_MATERN3, [.5, .9]), (orc.K_MATERN5, [.4, .8]),
         (orc.K_MATERN5_ARD, [.3, .4, .5, .95])]


def _oracle(kind, hyper, N, d, seed, noise=0.1, prior=None, Cinv=None):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    return orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior, Cinv=Cinv), rs


def _low(o, P):
    """the P training points of lowest Y: a baseline the batch can improve on"""
    return o.X[np.argsort(o.Y, kind='stable')[:P]]


def _margin(o, Xb, Xbase, Z):
    """smallest distance of any sample to a kink of the integrand: the gaps between the two largest draws of the batch and of the
    baseline, and |improvement|"""
    P = len(Xbase)
    mu, Sig = no.latent_joint(o, np.r_[Xbase, Xb])
    F = mu[:, None] + np.linalg.cholesky(Sig).dot(Z)
    gaps = []
    for part in (F[:P], F[P:]):
        Fs = np.sort(part, axis=0)
        gaps.append(np.min(Fs[-1] - Fs[-2]) if part.shape[0] > 1 else np.inf)
    imp = np.max(F[P:], axis=0) - np.max(F[:P], axis=0)
    return min(gaps + [np.min(np.abs(imp))])


def _check_fd(o, Xb, Xbase, Z, h=1e-6, tol=1e-6):
    assert _margin(o, Xb, Xbase, Z) > 1e-4
    v, G = no.qnei_batch(o, Xb, Xbase, Z)
    assert v > 0 and np.any(G != 0)
    fd = np.zeros_like(Xb)
    for j in range(Xb.shape[0]):
        for t in range(Xb.shape[1]):
            E = np.zeros_like(Xb)
            E[j, t] = h
            fd[j, t] = (no.qnei_batch(o, Xb + E, Xbase, Z, grad=False) - no.qnei_batch(o, Xb - E, Xbase, Z, grad=False)) / (2 * h)
    assert np.max(np.abs(G - fd)) <= tol * np.max(np.abs(fd)), np.max(np.abs(G - fd)) / np.max(np.abs(fd))


@pytest.mark.parametrize("kind,hyper", KINDS)
def test_gradient_matches_finite_differences(kind, hyper):
    o, rs = _oracle(kind, hyper, 40, 3, 1)
    Xb = rs.rand(3, 3)
    Xbase = _low(o, 6)
    Z = np.random.default_rng(3).standard_normal((9, 24))
    _check_fd(o, Xb, Xbase, Z)


@pytest.mark.parametrize("q,S", [(1, 32), (3, 32), (32, 8)])
def test_gradient_matches_finite_differences_over_q(q, S):
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 3)
    Xb = rs.rand(q, 3)
    Xbase = _low(o, 5)
    Z = np.random.default_rng(q).standard_normal((5 + q, S))
    _check_fd(o, Xb, Xbase, Z)


def test_gradient_with_prior_and_variance_model():
    d = 2
    prior = orc.PriorSpec(np.random.RandomState(5).rand(3, d), [0.5, -0.2, 0.3], 3.0, np.zeros(d), np.ones(d))
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, d, 3, prior=prior)
    Xb = rs.rand(4, d)
    Z = np.random.default_rng(7).standard_normal((10, 24))
    _check_fd(o, Xb, _low(o, 6), Z)
    o.augX = np.r_[o.X, rs.rand(4, d)]
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, o.augX, o.noise))
    _check_fd(o, Xb, _low(o, 6), Z)


def test_gradient_of_a_laplace_model():
    B = np.random.RandomState(9).randn(30, 30) * 0.3
    o, rs = _oracle(orc.K_MATERN5_ARD, [.3, .4, .5, .95], 30, 3, 8, Cinv=np.linalg.inv(5 * np.eye(30) + B.dot(B.T)))
    Xb = rs.rand(3, 3)
    Z = np.random.default_rng(8).standard_normal((7, 24))
    _check_fd(o, Xb, _low(o, 4), Z)


def test_q1_p1_monte_carlo_matches_the_closed_form():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 40, 3, 4)
    x, xb = rs.rand(1, 3), o.X[:1]
    S = 200000
    Z = np.random.default_rng(0).standard_normal((2, S))
    mu, Sig = no.latent_joint(o, np.r_[xb, x])
    md = mu[1] - mu[0]
    sd = math.sqrt(Sig[0, 0] + Sig[1, 1] - 2 * Sig[0, 1])
    u = md / sd
    ref = sd * math.exp(-0.5 * u * u) / math.sqrt(2 * math.pi) + md * 0.5 * math.erfc(-u / math.sqrt(2))
    v = no.qnei_batch(o, x, xb, Z, grad=False)
    L = np.linalg.cholesky(Sig)
    F = mu[:, None] + L.dot(Z)
    se = np.std(np.maximum(0.0, F[1] - F[0])) / math.sqrt(S)
    assert ref > 1e-3 and abs(v - ref) <= 5 * se, (v, ref, se)


@pytest.mark.parametrize("kind,hyper", [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_MATERN3, [.5]), (orc.K_MATERN5_ARD, [.3, .4, .5])])
def test_identity_with_qei_for_an_unreachable_baseline_point(kind, hyper):
    noise = 0.1
    hyper = hyper + [math.sqrt(1 + noise)]                              # sf2 = 1 + noise: the latent and the observed Sigma agree
    o, rs = _oracle(kind, hyper, 40, 3, 5, noise=noise)
    assert o.kernel.sf2 == pytest.approx(1 + noise, rel=1e-15)
    far = np.full((1, 3), 1e4)                                          # thousands of length scales: every k to it is exactly 0
    assert np.all(o.kernel.cross(np.r_[o.X, rs.rand(3, 3)], far) == 0)
    Xb = rs.rand(3, 3)
    Zq = np.random.default_rng(3).standard_normal((3, 64))
    Z = np.r_[np.zeros((1, 64)), Zq]
    v, G = no.qnei_batch(o, Xb, far, Z)
    ve, Ge = qo.qei_batch(o, Xb, Zq, 0.0, 0.0)
    assert v > 0 and abs(v - ve) <= 1e-13 * abs(ve)
    assert np.all(np.abs(G - Ge) <= 1e-12 * np.max(np.abs(Ge)))


def test_baseline_that_is_not_positive_definite_raises():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 20, 3, 2)
    far = np.full((2, 3), 1e4)                                          # a repeated point: Sigma_bb = sf2 [[1, 1], [1, 1]]
    with pytest.raises(no.BaselineNotPD):
        no.qnei_batch(o, rs.rand(2, 3), far, np.zeros((4, 8)))


def test_batch_polish_never_loses_keeps_pending_and_bounds():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 6)
    bounds = [[0., 1.], [0.1, 0.9], [0.2, 0.9]]
    q, S, P = 3, 64, 8
    pending = rs.rand(2, 3) * 0.5
    Xbase = _low(o, P)
    Z = np.random.default_rng(1).standard_normal((P + q + 2, S))
    fg = lambda X: no.qnei(o, X, Xbase, Z, 1e-8)                      # noqa: E731
    b = np.array(bounds)
    starts = b[:, 0] + (b[:, 1] - b[:, 0]) * rs.rand(4, q, 3)
    val, batch, v0, nfev = _polish_batches(fg, bounds, starts, pending, maxiter=30)
    assert batch.shape == (q, 3) and nfev >= 2
    assert val >= np.max(v0)
    assert np.all(batch >= b[:, 0]) and np.all(batch <= b[:, 1])
    full = np.r_[batch, pending][None]
    assert abs(fg(full)[0][0] - val) <= 1e-12 * val
    assert val > np.max(v0)


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    fake = ctypes.create_string_buffer(1 << 16)                       # never dereferenced: every scalar check comes first
    h = ctypes.cast(fake, ctypes.c_void_p)
    x = np.zeros((4, 2)); xb = np.zeros((4, 2)); z = np.zeros(64); o = np.zeros(64)
    p = _lib.dptr
    nbad, info = ctypes.c_int(5), ctypes.c_int(7)
    good = dict(m=h, X=p(x), B=2, q=2, Xb=p(xb), P=2, Z=p(z), S=4, jitter=0.0, v=p(o))
    bad = [dict(m=None), dict(X=None), dict(Xb=None), dict(Z=None), dict(v=None), dict(B=0), dict(B=-3), dict(q=0), dict(q=33),
           dict(P=0), dict(P=8193), dict(S=0), dict(S=8193), dict(jitter=-1e-9), dict(jitter=float("nan"))]
    for change in bad:
        a = dict(good, **change)
        rc = L.ibo_qnei(a["m"], a["X"], a["B"], a["q"], a["Xb"], a["P"], a["Z"], a["S"], a["jitter"], a["v"], p(o), p(o),
                        ctypes.byref(nbad), ctypes.byref(info))
        assert rc == _lib.E_BADARG, change
        assert nbad.value == 0 and info.value == 0
