"""GPU tests of the candidate gradients (ibo_posterior_grad / ibo_score_grad and their Python surface) against the oracle's
grad_oracle, against finite differences of the device's own values, and of gradient polishing in maximizeEI."""
import ctypes

import numpy as np
import pytest

from oracle import ibo_oracle as orc
import grad_oracle as go

pytestmark = pytest.mark.gpu

# magnitudes below 1: R's diagonal is 1 + noise whatever sf2 is, so sf2 > 1 + noise can make R itself indefinite
KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}
# (kind, N, M): every kind, N = 1 and 50 (one row-block), 129 (two row-blocks with padding) and 1000; M from 1 to 2500 (across the
# 128-candidate tile and the 2048 boundary between the latency and throughput shapes of the scoring path)
CASES = [
    (orc.K_SE_ARD, 1, 7), (orc.K_SE_ISO, 50, 129), (orc.K_MATERN3, 129, 129), (orc.K_MATERN5, 1000, 7),
    (orc.K_MATERN5_ARD, 129, 1), (orc.K_SE_ARD, 1000, 2500), (orc.K_MATERN3, 50, 2500), (orc.K_SE_ISO, 1, 129),
    (orc.K_MATERN5_ARD, 1000, 129), (orc.K_MATERN5, 50, 1),
]


def _lib():
    from ibo_b200 import _lib as L
    return L


def _data(N, M, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    Xs = rs.rand(M, d)
    Xs[: min(2, M, N)] = X[: min(2, M, N)]        # candidates on training points
    return X, Y, Xs


def _check(G, G_o):
    """<= 1e-9 of the row's largest component + 1e-12"""
    bound = 1e-9 * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12
    assert np.all(np.abs(G - G_o) <= bound), np.max(np.abs(G - G_o) - bound)


def _flags(mode):
    L = _lib()
    return L.FLAG_MODE_PY if mode == "py" else L.FLAG_MODE_CPP


@pytest.mark.parametrize("mode", ["py", "cpp"])
@pytest.mark.parametrize("kind,N,M", CASES)
def test_gradients_match_oracle(kind, N, M, mode):
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs = _data(N, M, d, 10 * N + M + kind)
    hyper = KINDS[kind]
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise)
    m = L.Model(kind, hyper, X, Y, noise)
    fl = _flags(mode)
    mu, s2, dmu, ds2 = m.posterior_grad(Xs, fl)
    mu_b, s2_b = m.posterior(Xs, fl | L.FLAG_FP64)
    assert np.array_equal(mu, mu_b) and np.array_equal(s2, s2_b)
    _, _, dmu_o, ds2_o = go.posterior_grad(o, Xs, mode)
    _check(dmu, dmu_o)
    _check(ds2, ds2_o)
    ymax = Y.max()
    for acq, parm in ((L.ACQ_EI, 0.01), (L.ACQ_PI, 0.01), (L.ACQ_UCB, 1.3)):
        sc, dsc = m.score_grad(Xs, acq, ymax, parm, fl)
        sc_b = m.score(Xs, acq, ymax, parm, fl | L.FLAG_FP64)[0]
        assert np.array_equal(sc, sc_b)
        _check(dsc, go.score_grad(o, Xs, acq, ymax, parm, mode)[1])
    m.close()


@pytest.mark.parametrize("mode", ["py", "cpp"])
def test_gradients_match_finite_differences_of_device_values(mode):
    """the chain rule checked without the oracle: central differences of the device's own FP64 values"""
    L = _lib()
    d = 4
    X, Y, Xs = _data(300, 60, d, 21)
    Xs = Xs[5:]                                   # away from the training points
    m = L.Model(orc.K_MATERN5_ARD, [.3, .4, .5, .6, .95], X, Y, 0.1)
    fl = _flags(mode)
    ymax, h = Y.max() - 0.2, 1e-5
    mu, s2, dmu, ds2 = m.posterior_grad(Xs, fl)
    free = (s2 > 10e-8) & (s2 < 10)
    for acq, parm in ((L.ACQ_EI, 0.01), (L.ACQ_PI, 0.01), (L.ACQ_UCB, 1.3)):
        _, dsc = m.score_grad(Xs, acq, ymax, parm, fl)
        Z = (mu - ymax - parm) / np.sqrt(s2)
        keep = free & (np.abs(Z) > 1e-3)
        for t in range(d):
            E = np.zeros_like(Xs); E[:, t] = h
            fd = (m.score_grad(Xs + E, acq, ymax, parm, fl)[0] - m.score_grad(Xs - E, acq, ymax, parm, fl)[0]) / (2 * h)
            scale = np.maximum(np.max(np.abs(dsc), axis=1), 1e-6)
            assert np.max((np.abs(dsc[:, t] - fd) / scale)[keep]) < 1e-6
    for t in range(d):
        E = np.zeros_like(Xs); E[:, t] = h
        p, q = m.posterior_grad(Xs + E, fl), m.posterior_grad(Xs - E, fl)
        assert np.max(np.abs(dmu[:, t] - (p[0] - q[0]) / (2 * h)) / np.max(np.abs(dmu), axis=1)) < 1e-6
        assert np.max((np.abs(ds2[:, t] - (p[1] - q[1]) / (2 * h)) / np.max(np.abs(ds2), axis=1))[free]) < 1e-6


def test_rbf_prior():
    L = _lib()
    d = 2
    X, Y, Xs = _data(200, 300, d, 4)
    rs = np.random.RandomState(9)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1, prior=prior)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, prior=prior)
    for mode in ("py", "cpp"):
        _, _, dmu, ds2 = m.posterior_grad(Xs, _flags(mode))
        _, _, dmu_o, ds2_o = go.posterior_grad(o, Xs, mode)
        _check(dmu, dmu_o)
        _check(ds2, ds2_o)
        _check(m.score_grad(Xs, L.ACQ_EI, Y.max(), 0.01, _flags(mode))[1], go.score_grad(o, Xs, orc.ACQ_EI, Y.max(), 0.01, mode)[1])


def test_pref_gp_with_variance_model():
    """ds2 from the variance factor (augX, augL), dmu from the main model"""
    from ibo_b200.gaussianprocess import PrefGaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    rs = np.random.RandomState(8)
    N, d = 60, 4
    X = rs.rand(N, d) * 10
    Y = rs.randn(N)
    A = rs.randn(N, N) * 0.05
    C = np.eye(N) * 5 + A.dot(A.T)
    theta = [5.146, 4.189, 4.622, 5.843]
    gp = PrefGaussianProcess.fromLaplace(GaussianKernel_ard(theta), X, Y, C, noise=0.1)
    Cinv = np.linalg.inv(C)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, theta, d), X, Y, 0.1, Cinv=Cinv)
    q = rs.rand(150, d) * 10
    P = rs.rand(3, d) * 10
    gp.addObservationPoint(P)
    augX = np.r_[X, P]
    pad = np.zeros((N + 3, N + 3)); pad[:N, :N] = Cinv
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad); o.augX = augX
    mu, s2, dmu, ds2 = gp.posterior_grad(q)
    _, _, dmu_o, ds2_o = go.posterior_grad(o, q, "py")
    _check(dmu, dmu_o)
    _check(ds2, ds2_o)
    sc, dsc = gp.score_grad(q, 'ei')
    assert np.array_equal(sc, gp.score_batch(q, 'ei', int8=False)[0])
    _check(dsc, go.score_grad(o, q, orc.ACQ_EI, Y.max(), 0.01, "py")[1])


def test_model_from_inverse():
    L = _lib()
    d = 3
    X, Y, Xs = _data(150, 200, d, 6)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4, .5], d), X, Y, 0.1)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1, invR=o.invR(), sf2=1.0)
    _, _, dmu, ds2 = m.posterior_grad(Xs, L.FLAG_MODE_CPP)
    _, _, dmu_o, ds2_o = go.posterior_grad(o, Xs, "cpp")
    _check(dmu, dmu_o)
    _check(ds2, ds2_o)


def test_appended_model_equals_rebuilt_model():
    L = _lib()
    d = 3
    X, Y, Xs = _data(300, 400, d, 7)
    m = L.Model(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], X[:250], Y[:250], 0.1)
    m.posterior_grad(Xs)                          # a gradient call before the append: nothing cached may survive it
    m.append(X[250:], Y[250:])
    r = L.Model(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], X, Y, 0.1)
    a, b = m.posterior_grad(Xs), r.posterior_grad(Xs)
    for u, v in zip(a[2:], b[2:]):
        assert np.max(np.abs(u - v)) <= 1e-10 * max(1.0, np.max(np.abs(v)))


def test_chunks_are_batch_invariant_and_reproducible():
    """N = 1000: chunks of 32768 candidates, so 70000 candidates take three; a sub-range across a chunk boundary called alone gives
    the same rows bit for bit, and so does a second identical call"""
    L = _lib()
    d = 3
    X, Y, _ = _data(1000, 1, d, 30)
    Xs = np.random.RandomState(31).rand(70000, d)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1)
    mu, s2, dmu, ds2 = m.posterior_grad(Xs)
    mu2, s22, dmu2, ds22 = m.posterior_grad(Xs)
    assert np.array_equal(dmu, dmu2) and np.array_equal(ds2, ds22) and np.array_equal(mu, mu2) and np.array_equal(s2, s22)
    for lo, hi in ((32700, 32900), (65500, 65600), (0, 1), (69990, 70000)):
        _, _, a, b = m.posterior_grad(Xs[lo:hi])
        assert np.array_equal(a, dmu[lo:hi]) and np.array_equal(b, ds2[lo:hi])
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4, .5], d), X, Y, 0.1)
    rows = np.r_[0:50, 32740:32800, 65510:65560, 69950:70000]
    _, _, dmu_o, ds2_o = go.posterior_grad(o, Xs[rows])
    _check(dmu[rows], dmu_o)
    _check(ds2[rows], ds2_o)


def test_clipped_variance_has_zero_gradient():
    L = _lib()
    d = 3
    X, Y, _ = _data(40, 1, d, 32)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.0)
    Xs = np.r_[X[:6], np.random.RandomState(33).rand(4, d)]
    for mode, floor in (("py", 10e-8), ("cpp", 1e-8)):
        mu, s2, dmu, ds2 = m.posterior_grad(Xs, _flags(mode))
        assert np.all(s2[:6] == floor) and np.all(ds2[:6] == 0.0)
        assert np.all(np.any(ds2[6:] != 0, axis=1)) and np.all(np.isfinite(dmu))


def test_bad_arguments():
    L = _lib()
    lib = L.lib()
    X, Y, Xs = _data(20, 4, 2, 34)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1)
    p = L.dptr
    x = np.ascontiguousarray(Xs); o = np.zeros(64)
    h = m.handle
    assert lib.ibo_posterior_grad(None, p(x), 4, 0, p(o), p(o), p(o), p(o)) == L.E_BADARG
    assert lib.ibo_posterior_grad(h, None, 4, 0, p(o), p(o), p(o), p(o)) == L.E_BADARG
    assert lib.ibo_posterior_grad(h, p(x), 0, 0, p(o), p(o), p(o), p(o)) == L.E_BADARG
    assert lib.ibo_posterior_grad(h, p(x), 4, L.FLAG_FP64, p(o), p(o), p(o), p(o)) == L.E_BADARG
    for acq in (-1, 3):
        assert lib.ibo_score_grad(h, p(x), 4, acq, 0.0, 0.01, 0, p(o), p(o)) == L.E_BADARG
    assert lib.ibo_score_grad(h, p(x), 4, 0, 0.0, 0.01, L.FLAG_INT8, p(o), p(o)) == L.E_BADARG
    assert lib.ibo_score_grad(h, p(x), 4, 0, 0.0, 0.01, 0, None, None) == 0       # every output may be NULL
    d = 65
    Xw = np.random.RandomState(35).rand(8, d)
    try:
        wide = L.Model(orc.K_SE_ISO, [3.0], Xw, np.zeros(8), 0.1)
    except L.IBOError:
        return                                    # a model of more than 64 dimensions cannot be built at all
    xw = np.ascontiguousarray(Xw[:2])
    assert lib.ibo_posterior_grad(wide.handle, p(xw), 2, 0, None, None, None, None) == L.E_BADARG
    assert lib.ibo_score_grad(wide.handle, p(xw), 2, 0, 0.0, 0.01, 0, None, None) == L.E_BADARG


def _gp(name):
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, GaussianKernel_iso, MaternKernel3
    if name == "branin":
        bounds = [[-5., 10.], [0., 15.]]
        X = np.array(orc.lhc_sample(bounds, 10, seed=0))
        return GaussianProcess(MaternKernel3([1.0, 1.0]), X, -orc.branin(X) / 100.0, noise=0.01), bounds
    if name == "shekel":
        bounds = [[0., 10.]] * 4
        X = np.array(orc.lhc_sample(bounds, 10, seed=0))
        return GaussianProcess(GaussianKernel_iso([2.0]), X, np.array([-orc.shekel5(x) for x in X]), noise=0.1), bounds
    if name == "hartman6":
        X = np.random.RandomState(0).rand(200, 6)
        return GaussianProcess(GaussianKernel_ard([.53, .57, 2.5, .34, .27, .35]), X, orc.hartman6_neg(X), noise=0.1), [[0., 1.]] * 6
    rs = np.random.RandomState(5)                 # config #5's shape: d = 20, N = 4096
    X = rs.rand(4096, 20)
    return GaussianProcess(GaussianKernel_ard([1.0] * 20), X, np.sin(2 * X).sum(axis=1), noise=0.1), [[0., 1.]] * 20


@pytest.mark.parametrize("name", ["branin", "shekel", "hartman6", "d20"])
def test_maximize_ei_with_polish(name):
    from ibo_b200.acquisition import cdirectGP, maximizeEI
    L = _lib()
    gp, bounds = _gp(name)
    iters = 30 if name == "d20" else 50
    opt, optx = maximizeEI(gp, bounds, xi=0.01, maxiter=iters)
    last = dict(cdirectGP.last)
    opt_p, optx_p = maximizeEI(gp, bounds, xi=0.01, maxiter=iters, polish=8)
    assert cdirectGP.last["nsamples"] == last["nsamples"] and cdirectGP.last["polish"]["evaluations"] >= 2
    flags = L.FLAG_MODE_CPP | L.FLAG_FP64
    ref = gp.model.score(optx[None, :], L.ACQ_EI, gp.Y.max(), 0.01, flags)[0][0]
    got = gp.model.score(optx_p[None, :], L.ACQ_EI, gp.Y.max(), 0.01, flags)[0][0]
    assert got >= ref - 1e-15 * abs(ref)
    b = np.array(bounds)
    assert np.all(optx_p >= b[:, 0]) and np.all(optx_p <= b[:, 1])
    if cdirectGP.last["polish"]["moved"]:
        assert abs(opt_p - got) <= 1e-12 * max(1.0, abs(got))
    else:
        assert opt_p == opt and np.array_equal(optx_p, optx)
    # a fixed dimension stays at its bound
    fb = [list(v) for v in bounds]
    fb[0] = [bounds[0][0] + 0.3 * (bounds[0][1] - bounds[0][0])] * 2
    _, optx_f = maximizeEI(gp, fb, xi=0.01, maxiter=10, polish=4)
    assert optx_f[0] == fb[0][0]
