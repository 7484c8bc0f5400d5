"""CPU tests of max-value entropy search: the float64 restatement of h and h' against 50-digit mpmath, the oracle's gradient against
central differences of its own values, the Gumbel fit's closed forms, the polish step of maximizeMES on an oracle objective, and the
argument checks of ibo_mes and ibo_max_value_gumbel (no device touched)."""
import ctypes
import math

import numpy as np
import pytest
from scipy.stats import norm

from ibo_b200 import _lib
from ibo_b200.acquisition import _polish_from
from ibo_b200.gaussianprocess import gumbel_draws
from oracle import ibo_oracle as orc
import mes_oracle as mo

KINDS = [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_SE_ISO, [.3]), (orc.K_MATERN3, [.5, .9]), (orc.K_MATERN5, [.4, .8]),
         (orc.K_MATERN5_ARD, [.3, .4, .5, .95])]


def _oracle(kind, hyper, N, d, seed, noise=0.1, prior=None):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    return orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior), rs


def test_float64_h_matches_mpmath():
    G = np.r_[-np.logspace(4, -3, 200), 0.0, np.logspace(-3, math.log10(37), 200)]
    h, dh = mo.h_np(G)
    for g, a, b in zip(G, h, dh):
        hr, dr = mo.h_mp(g)
        bound = 1e-13 if g <= 8 else 16 * (1 + g * g) * 2.0 ** -53
        assert abs(a - float(hr)) <= bound * abs(float(hr)), g
        assert abs(b - float(dr)) <= bound * abs(float(dr)), g
    assert np.all(h >= 0) and np.all(dh < 0)


def _check_fd(o, Xs, ystar, mode="py", h=1e-6, tol=1e-6):
    v, G = mo.mes(o, Xs, ystar, mode)
    fd = np.zeros_like(Xs)
    for t in range(Xs.shape[1]):
        E = np.zeros_like(Xs)
        E[:, t] = h
        fd[:, t] = (mo.mes(o, Xs + E, ystar, mode, grad=False) - mo.mes(o, Xs - E, ystar, mode, grad=False)) / (2 * h)
    scale = np.max(np.abs(fd), axis=1, keepdims=True) + 1e-12
    assert np.all(np.abs(G - fd) <= tol * scale), np.max(np.abs(G - fd) / scale)
    return v, G


@pytest.mark.parametrize("kind,hyper", KINDS)
def test_gradient_matches_finite_differences(kind, hyper):
    o, rs = _oracle(kind, hyper, 40, 3, 1)
    ystar = o.Y.max() + np.array([0.05, 0.3, 1.0])
    _check_fd(o, rs.rand(6, 3), ystar)


def test_gradient_with_prior_and_variance_model():
    d = 2
    prior = orc.PriorSpec(np.random.RandomState(5).rand(3, d), [0.5, -0.2, 0.3], 3.0, np.zeros(d), np.ones(d))
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, d, 3, prior=prior)
    Xs = rs.rand(5, d)
    ystar = o.Y.max() + np.array([0.1, 0.4])
    _check_fd(o, Xs, ystar, mode="cpp")
    o.augX = np.r_[o.X, rs.rand(4, d)]
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, o.augX, o.noise))
    _check_fd(o, Xs, ystar)


def test_clipped_variance_contributes_no_gradient():
    """at a training point of a model with noise 1e-9 s2 is clipped to the floor: only d mu carries the gradient"""
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 4, noise=1e-9)
    Xs = np.r_[o.X[:2], rs.rand(2, 3)]
    mu, s2, dmu, ds2 = mo.grad_oracle.posterior_grad(o, Xs, "py")
    assert s2[0] == 10e-8 and s2[1] == 10e-8 and np.all(ds2[:2] == 0)
    ystar = np.array([o.Y.max() + 0.2])
    v, G = mo.mes(o, Xs, ystar)
    _, a, _ = mo.mes_partials(mu, s2, ystar)
    assert np.array_equal(G[:2], a[:2, None] * dmu[:2])


def test_gumbel_closed_forms():
    mu, s2 = np.array([0.3]), np.array([0.49])
    q, (loc, scale) = mo.gumbel_quantiles(mu, s2)
    for qq, p in zip(q, (0.25, 0.5, 0.75)):
        assert abs(qq - (0.3 + 0.7 * norm.ppf(p))) <= 1e-14
    rs = np.random.RandomState(0)
    mu, s2 = rs.randn(7), 0.1 + rs.rand(7)
    n = 5
    q1, _ = mo.gumbel_quantiles(np.tile(mu, n), np.tile(s2, n))
    for qq, p in zip(q1, (0.25, 0.5, 0.75)):                          # the set duplicated n times solves F = p^(1/n)
        assert abs(mo.log_F(qq, mu, np.sqrt(s2)) - math.log(p) / n) <= 1e-14
    assert loc == q[1] + scale * math.log(-math.log(.5))


def test_gumbel_draws_are_finite_and_seeded():
    u = gumbel_draws(1.0, 0.5, 100000, seed=3)
    assert np.all(np.isfinite(u)) and np.array_equal(u, gumbel_draws(1.0, 0.5, 100000, seed=3))
    assert abs(np.median(u) - (1.0 - 0.5 * math.log(-math.log(0.5)))) < 0.01


def test_polish_starts_and_keeps_only_a_better_point():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, 2, 6)
    bounds = [[0., 1.], [0.1, 0.9]]
    ystar = o.Y.max() + np.array([0.05, 0.2, 0.6])
    fg = lambda X: mo.mes(o, X, ystar)                                 # noqa: E731
    C = rs.rand(50, 2) * [1.0, 0.8] + [0.0, 0.1]
    cv = mo.mes(o, C, ystar, grad=False)
    optx = np.array([0.5, 0.5])
    opt = float(fg(optx[None])[0][0])
    val, x, rec = _polish_from(fg, bounds, opt, optx, C, cv, 4, maxiter=30)
    assert np.array_equal(rec["starts"][0], optx)
    assert np.array_equal(rec["starts"][1:], C[np.argsort(-cv)[:3]])
    assert rec["moved"] and val > max(opt, np.max(cv)) and abs(fg(x[None])[0][0] - val) <= 1e-15 * val
    assert np.all(x >= [0.0, 0.1]) and np.all(x <= [1.0, 0.9])
    # DIRECT's point is the maximum, which no polished start can beat: (opt, optx) come back unchanged
    quad = lambda X: (-np.sum((X - optx) ** 2, axis=1), -2.0 * (X - optx))      # noqa: E731
    v2, x2, rec2 = _polish_from(quad, bounds, 123.0, optx, C, -np.sum((C - optx) ** 2, axis=1), 3, maxiter=30)
    assert not rec2["moved"] and v2 == 123.0 and x2 is optx and rec2["evaluations"] >= 2


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    fake = ctypes.create_string_buffer(1 << 16)                       # never dereferenced: every scalar check comes first
    h = ctypes.cast(fake, ctypes.c_void_p)
    p = _lib.dptr
    x = np.zeros((4, 2)); ys = np.zeros(2048); v = np.zeros(64); g = np.zeros(128)
    best, idx = ctypes.c_double(0), ctypes.c_long(0)
    good = dict(m=h, X=p(x), M=4, y=p(ys), K=2, fl=0, v=p(v), dv=None)
    bad = [dict(m=None), dict(X=None), dict(M=0), dict(M=-1), dict(y=None), dict(v=None), dict(K=0), dict(K=1025), dict(K=-1),
           dict(fl=0x2), dict(fl=0x8), dict(fl=0x200), dict(dv=p(g), fl=_lib.FLAG_INT8), dict(dv=p(g), fl=_lib.FLAG_FP64),
           dict(dv=p(g), fl=_lib.FLAG_MODE_PY | _lib.FLAG_INT8)]
    for nonfinite in (float("nan"), float("inf"), -float("inf")):
        y2 = np.zeros(3); y2[2] = nonfinite
        bad.append(dict(y=p(y2), K=3, _keep=y2))
    for change in bad:
        a = dict(good, **change)
        rc = L.ibo_mes(a["m"], a["X"], a["M"], a["y"], a["K"], a["fl"], a["v"], a["dv"], ctypes.byref(best), ctypes.byref(idx))
        assert rc == _lib.E_BADARG, change
    q = np.zeros(3)
    for change in [dict(m=None), dict(X=None), dict(M=0), dict(fl=0x2), dict(fl=0x8), dict(fl=0x40)]:
        a = dict(good, **change)
        rc = L.ibo_max_value_gumbel(a["m"], a["X"], a["M"], a["fl"], p(q), None, None)
        assert rc == _lib.E_BADARG, change
