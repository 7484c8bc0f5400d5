"""CPU tests of the candidate gradients: the oracle's gradients against central finite differences of its own values, the
polish driver run on the oracle, and the argument checks of the two C entry points (no device touched)."""
import ctypes

import numpy as np
import pytest

from ibo_b200 import _lib
from ibo_b200.acquisition import _polish
from oracle import ibo_oracle as orc
import grad_oracle as go

KINDS = [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_SE_ISO, [.3]), (orc.K_MATERN3, [.5, .9]), (orc.K_MATERN5, [.4, .8]),
         (orc.K_MATERN5_ARD, [.3, .4, .5, .95])]


def _oracle(kind, hyper, N, d, seed, noise=0.1, prior=None):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    return orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior), rs


def _fd(f, Xs, h=1e-6):
    """central differences of f(Xs[M, d]) -> [M] per coordinate"""
    G = np.zeros(Xs.shape)
    for t in range(Xs.shape[1]):
        E = np.zeros(Xs.shape)
        E[:, t] = h
        G[:, t] = (f(Xs + E) - f(Xs - E)) / (2 * h)
    return G


def _close(G, G_fd, tol=1e-6):
    scale = np.maximum(np.max(np.abs(G_fd), axis=1, keepdims=True), 1e-3)
    assert np.max(np.abs(G - G_fd) / scale) <= tol, np.max(np.abs(G - G_fd) / scale)


@pytest.mark.parametrize("mode", ["py", "cpp"])
@pytest.mark.parametrize("kind,hyper", KINDS)
def test_posterior_gradient_matches_finite_differences(kind, hyper, mode):
    o, rs = _oracle(kind, hyper, 40, 3, 1)
    Xs = rs.rand(30, 3)
    Xs[:2] = o.X[:2]                         # candidates on training points: every h(r) is finite at r = 0
    floor = 10e-8 if mode == "py" else 1e-8
    mu, s2, dmu, ds2 = go.posterior_grad(o, Xs, mode)
    mu_b, s2_b = o.posterior_batch(Xs, floor=floor)
    assert np.allclose(mu, mu_b, rtol=1e-12, atol=1e-13) and np.allclose(s2, s2_b, rtol=1e-12, atol=1e-15)
    _close(dmu, _fd(lambda P: o.posterior_batch(P, floor=floor)[0], Xs))
    _close(ds2, _fd(lambda P: o.posterior_batch(P, floor=floor)[1], Xs))


@pytest.mark.parametrize("mode", ["py", "cpp"])
@pytest.mark.parametrize("acq", [orc.ACQ_EI, orc.ACQ_PI, orc.ACQ_UCB])
def test_acquisition_gradient_matches_finite_differences(acq, mode):
    o, rs = _oracle(orc.K_MATERN5_ARD, [.3, .4, .5, .95], 40, 3, 2)
    Xs = rs.rand(40, 3)
    ymax, parm = o.Y.max() - 0.3, (0.01 if acq != orc.ACQ_UCB else 1.7)
    floor = 10e-8 if mode == "py" else 1e-8
    sc, dsc = go.score_grad(o, Xs, acq, ymax, parm, mode)

    def val(P):
        mu, s2 = o.posterior_batch(P, floor=floor)
        return orc.score(acq, mode, mu, s2, ymax, parm)
    assert np.allclose(sc, val(Xs), rtol=1e-11, atol=1e-14)
    mu, s2 = o.posterior_batch(Xs, floor=floor)
    keep = np.abs((mu - ymax - parm) / np.sqrt(s2)) > 1e-3       # the Chebyshev erf steps by ~1e-9 at 0
    _close(dsc[keep], _fd(val, Xs)[keep])


def test_erf_derivative_is_that_of_the_chebyshev_formula():
    z = np.r_[-np.linspace(0.01, 6, 50), np.linspace(0.01, 6, 50)]
    h = 1e-6
    fd = (orc.erf_py(z + h) - orc.erf_py(z - h)) / (2 * h)
    assert np.max(np.abs(go.erf_py_deriv(z) - fd)) < 1e-8
    exact = 2 / np.sqrt(np.pi) * np.exp(-z * z)
    assert np.max(np.abs(go.erf_py_deriv(z) - exact)) > 1e-9          # not the derivative of the exact erf


@pytest.mark.parametrize("mode", ["py", "cpp"])
def test_prior_and_variance_factor(mode):
    d = 2
    prior = orc.PriorSpec(np.random.RandomState(5).rand(3, d), [0.5, -0.2, 0.3], 3.0, np.zeros(d), np.ones(d))
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, d, 3, prior=prior)
    o.augX = np.r_[o.X, rs.rand(4, d)]
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, o.augX, o.noise))
    Xs = rs.rand(25, d)
    floor = 10e-8 if mode == "py" else 1e-8
    _, _, dmu, ds2 = go.posterior_grad(o, Xs, mode)
    _close(dmu, _fd(lambda P: o.posterior_batch(P, floor=floor)[0], Xs))
    _close(ds2, _fd(lambda P: o.posterior_batch(P, floor=floor)[1], Xs))
    sc, dsc = go.score_grad(o, Xs, orc.ACQ_EI, o.Y.max(), 0.01, mode)
    _close(dsc, _fd(lambda P: orc.score(orc.ACQ_EI, mode, *o.posterior_batch(P, floor=floor), o.Y.max(), 0.01), Xs))


def test_clipped_variance_has_zero_gradient():
    """noise 0: sigma^2 at a training point cancels to (about) 0 and is clipped to the floor"""
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 20, 3, 4, noise=0.0)
    Xs = np.r_[o.X[:5], rs.rand(5, 3)]
    mu, s2, dmu, ds2 = go.posterior_grad(o, Xs, "py")
    assert np.all(s2[:5] == 10e-8) and np.all(ds2[:5] == 0.0)
    assert np.all(s2[5:] > 10e-8) and np.all(np.any(ds2[5:] != 0, axis=1))
    assert np.all(np.isfinite(dmu))


def _oracle_fg(o, acq, parm, mode):
    ymax = o.Y.max()
    return lambda X: go.score_grad(o, X, acq, ymax, parm, mode)


def _projected_gradient(X, G, lo, hi):
    P = G.copy()
    P[(X <= lo) & (G < 0)] = 0
    P[(X >= hi) & (G > 0)] = 0
    P[:, lo == hi] = 0
    return P


def test_polish_never_loses_respects_bounds_and_reaches_a_stationary_point():
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4, .5], 30, 3, 6)
    bounds = [[0., 1.], [0.25, 0.25], [0.2, 0.9]]          # the middle dimension is fixed
    X0 = np.c_[rs.rand(6), np.full(6, 0.25), 0.2 + 0.7 * rs.rand(6)]
    fg = _oracle_fg(o, orc.ACQ_EI, 0.01, "cpp")
    v0 = fg(X0)[0]
    vals, X, v0b, nfev = _polish(fg, bounds, X0)
    assert np.array_equal(v0, v0b) and nfev >= 2
    assert np.all(vals >= v0)
    assert np.all(X[:, 1] == 0.25)
    b = np.array(bounds)
    assert np.all(X >= b[:, 0]) and np.all(X <= b[:, 1])
    assert np.allclose(vals, fg(X)[0], rtol=1e-12, atol=0)
    G = _projected_gradient(X, fg(X)[1], b[:, 0], b[:, 1])
    assert np.max(np.abs(G) / np.maximum(np.abs(vals), 1e-12)[:, None]) < 1e-3


@pytest.mark.parametrize("name", ["branin", "shekel"])
def test_polish_from_direct_ends_at_or_above_direct(name):
    if name == "branin":
        bounds = [[-5., 10.], [0., 15.]]
        X = np.array(orc.lhc_sample(bounds, 10, seed=0))
        o = orc.GPOracle(orc.KernelSpec(orc.K_MATERN3, [1.0, 1.0], 2), X, -orc.branin(X) / 100.0, 0.01)
    else:
        bounds = [[0., 10.]] * 4
        X = np.array(orc.lhc_sample(bounds, 10, seed=0))
        o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ISO, [2.0], 4), X, np.array([-orc.shekel5(x) for x in X]), 0.1)
    opt, optx = orc.acqmax_cpp(o, bounds, orc.ACQ_EI, 0.01, maxiter=20, maxsample=2000)
    fg = _oracle_fg(o, orc.ACQ_EI, 0.01, "cpp")
    vals, Xp, v0, _ = _polish(fg, bounds, optx[None, :])
    assert abs(v0[0] - opt) <= 1e-9 * max(1.0, abs(opt))
    assert vals[0] >= opt - 1e-12
    b = np.array(bounds)
    assert np.all(Xp >= b[:, 0]) and np.all(Xp <= b[:, 1])


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    fake = ctypes.create_string_buffer(1 << 16)          # never dereferenced: every scalar check comes first
    h = ctypes.cast(fake, ctypes.c_void_p)
    x = np.zeros((3, 2)); o = np.zeros(6)
    p = _lib.dptr
    for args in [(None, p(x), 3, 0), (h, None, 3, 0), (h, p(x), 0, 0), (h, p(x), -1, 0), (h, p(x), 3, _lib.FLAG_FP64),
                 (h, p(x), 3, 0x2)]:
        assert L.ibo_posterior_grad(*args, p(o), p(o), p(o), p(o)) == _lib.E_BADARG
    for args in [(None, p(x), 3, 0, 0), (h, None, 3, 0, 0), (h, p(x), 0, 0, 0), (h, p(x), 3, -1, 0), (h, p(x), 3, 3, 0),
                 (h, p(x), 3, 0, _lib.FLAG_MODE_PY | _lib.FLAG_INT8)]:
        M, acq, flags = args[2], args[3], args[4]
        assert L.ibo_score_grad(args[0], args[1], M, acq, 0.0, 0.01, flags, p(o), p(o)) == _lib.E_BADARG


def test_polish_with_shard_is_refused():
    from ibo_b200.acquisition import cdirectGP
    with pytest.raises(ValueError):
        cdirectGP(object(), [[0., 1.]], 10, 10, 100, acqfunc='ei', xi=0.01, polish=2, shard=True)
