"""GPU tests of the batch expected improvement (ibo_qei and its Python surface) against the oracle's restatement (qei_oracle), against
ibo_posterior_sample, against finite differences of the device's own values, its exact identities, and maximizeQEI."""
import ctypes

import numpy as np
import pytest

from oracle import ibo_oracle as orc
import joint_oracle as jo
import qei_oracle as qo

pytestmark = pytest.mark.gpu

KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}
# (kind, N, q, S): every kind; N = 1, 50 (one row-block), 129 (two, with padding) and 1000; q = 1, 4 and 32; S = 1 and 1024
CASES = [
    (orc.K_SE_ARD, 1, 4, 1024), (orc.K_SE_ISO, 50, 32, 1024), (orc.K_MATERN3, 129, 1, 1024), (orc.K_MATERN5, 1000, 4, 1),
    (orc.K_MATERN5_ARD, 129, 32, 1), (orc.K_SE_ARD, 1000, 32, 1024), (orc.K_MATERN3, 50, 4, 1024), (orc.K_SE_ISO, 1, 1, 1),
    (orc.K_MATERN5_ARD, 1000, 4, 1024), (orc.K_MATERN5, 50, 1, 1024),
]


def _lib():
    from ibo_b200 import _lib as L
    return L


def _data(N, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    return X, np.sin(3 * X).sum(axis=1), rs


def _check_values(v, v_o):
    assert np.all(np.abs(v - v_o) <= 1e-10 * np.maximum(np.abs(v_o), 1e-5)), np.max(np.abs(v - v_o))


def _check_grad(G, G_o):
    """<= 1e-9 of the row's largest component + 1e-12"""
    G, G_o = G.reshape(-1, G.shape[-1]), G_o.reshape(-1, G_o.shape[-1])
    bound = 1e-9 * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12
    assert np.all(np.abs(G - G_o) <= bound), np.max(np.abs(G - G_o) - bound)


@pytest.mark.parametrize("kind,N,q,S", CASES)
def test_matches_oracle(kind, N, q, S):
    L = _lib()
    d = 3
    X, Y, rs = _data(N, d, 100 * N + 10 * q + kind)
    hyper = KINDS[kind]
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, 0.1)
    m = L.Model(kind, hyper, X, Y, 0.1)
    B = 6
    Xb = rs.rand(B, q, d)
    Xb[0, 0] = X[0]                                   # a point on a training point
    Z = np.random.default_rng(q + S).standard_normal((q, S))
    ymax = Y.max() - 0.3
    v, G, nbad = m.qei(Xb, Z, ymax, 0.01)
    assert nbad == 0
    v_o, G_o = qo.qei(o, Xb, Z, ymax, 0.01)
    assert np.any(v_o > 0)
    _check_values(v, v_o)
    _check_grad(G, G_o)
    m.close()


def test_prior_from_inverse_and_appended_models():
    L = _lib()
    d = 2
    X, Y, rs = _data(300, d, 4)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    Xb = rs.rand(20, 4, d)
    Z = np.random.default_rng(1).standard_normal((4, 256))
    ymax = Y.max() - 0.2
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1, prior=prior)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, prior=prior)
    v, G, _ = m.qei(Xb, Z, ymax, 0.01, jitter=1e-6)
    v_o, G_o = qo.qei(o, Xb, Z, ymax, 0.01, jitter=1e-6)
    _check_values(v, v_o)
    _check_grad(G, G_o)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, invR=o.invR(), sf2=1.0)
    v, G, _ = m.qei(Xb, Z, ymax, 0.01)
    v_o, G_o = qo.qei(o, Xb, Z, ymax, 0.01)
    _check_values(v, v_o)
    _check_grad(G, G_o)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X[:250], Y[:250], 0.1)
    m.qei(Xb, Z, ymax, 0.01)                          # a call before the append: nothing cached may survive it
    m.append(X[250:], Y[250:])
    v, G, _ = m.qei(Xb, Z, ymax, 0.01)
    _check_values(v, v_o)
    _check_grad(G, G_o)


def test_pref_gp_with_variance_model():
    """Sigma and its gradient from the variance factor (augX, augL), mu from the main model"""
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
    P = rs.rand(3, d) * 10
    gp.addObservationPoint(P)
    augX = np.r_[X, P]
    pad = np.zeros((N + 3, N + 3)); pad[:N, :N] = Cinv
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad); o.augX = augX
    Xb = rs.rand(30, 4, d) * 10
    Z = np.random.default_rng(3).standard_normal((4, 512))
    v, G = gp.qEI(Xb, Z=Z, grad=True)
    v_o, G_o = qo.qei(o, Xb, Z, Y.max(), 0.01)
    _check_values(v, v_o)
    _check_grad(G, G_o)
    assert np.array_equal(gp.qEI(Xb, Z=Z), v)


def test_equals_mean_improvement_of_posterior_samples():
    L = _lib()
    d = 3
    X, Y, rs = _data(500, d, 12)
    m = L.Model(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], X, Y, 0.1)
    Z = np.random.default_rng(4).standard_normal((8, 2048))
    ymax, xi, jitter = Y.max() - 0.2, 0.01, 1e-4
    Xb = rs.rand(5, 8, d)
    v, _, _ = m.qei(Xb, Z, ymax, xi, jitter, want_grad=False)
    for b in range(5):
        F, _ = m.posterior_sample(Xb[b], Z, jitter)
        ref = np.mean(np.maximum(0.0, F.max(axis=0) - ymax - xi))
        assert abs(v[b] - ref) <= 1e-10 * ref


def test_exact_identities():
    """a batch is worth at least its first point alone with Z's first row ((L z)_0 = L_00 z_0); values are the same bits with and
    without the gradient"""
    L = _lib()
    d = 3
    X, Y, rs = _data(400, d, 13)
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.1)
    Xb = rs.rand(200, 4, d)
    Z = np.random.default_rng(5).standard_normal((4, 1000))
    for ymax in (Y.max() - 0.3, Y.max() + 0.2):
        v, G, _ = m.qei(Xb, Z, ymax, 0.01, 1e-6)
        v1, _, _ = m.qei(Xb[:, :1], Z[:1], ymax, 0.01, 1e-6)
        assert np.all(v >= v1) and np.any(v > v1)
        vn, Gn, _ = m.qei(Xb, Z, ymax, 0.01, 1e-6, want_grad=False)
        assert Gn is None and np.array_equal(v, vn)


def test_chunks_are_batch_invariant_and_reproducible():
    """N = 1000: chunks of 32768 points, so q = 3 takes 10922 batches per chunk and 24000 batches take three; a sub-range across a
    chunk boundary called alone gives the same rows bit for bit, and so does a second identical call"""
    L = _lib()
    d = 3
    X, Y, _ = _data(1000, d, 30)
    Xb = np.random.RandomState(31).rand(24000, 3, d)
    Z = np.random.default_rng(6).standard_normal((3, 64))
    ymax = Y.max() - 0.3
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.1)
    v, G, _ = m.qei(Xb, Z, ymax, 0.01)
    v2, G2, _ = m.qei(Xb, Z, ymax, 0.01)
    assert np.array_equal(v, v2) and np.array_equal(G, G2)
    for lo, hi in ((10900, 10950), (21830, 21860), (0, 1), (23990, 24000)):
        a, b, _ = m.qei(Xb[lo:hi], Z, ymax, 0.01)
        assert np.array_equal(a, v[lo:hi]) and np.array_equal(b, G[lo:hi])
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], d), X, Y, 0.1)
    rows = np.r_[0:10, 10915:10930, 23990:24000]
    v_o, G_o = qo.qei(o, Xb[rows], Z, ymax, 0.01)
    _check_values(v[rows], v_o)
    _check_grad(G[rows], G_o)


def test_gradient_matches_finite_differences_of_device_values():
    L = _lib()
    d = 4
    X, Y, rs = _data(300, d, 21)
    hyper = [.3, .4, .5, .6, .95]
    m = L.Model(orc.K_MATERN5_ARD, hyper, X, Y, 0.1)
    o = orc.GPOracle(orc.KernelSpec(orc.K_MATERN5_ARD, hyper, d), X, Y, 0.1)
    Z = np.random.default_rng(7).standard_normal((3, 32))
    ymax, xi, h = Y.max() - 0.3, 0.01, 1e-6

    def margin(Xq):                                   # distance of the samples to a kink of the integrand (oracle draws)
        mu, Sig = jo.posterior_joint(o, Xq)
        F = np.sort(mu[:, None] + np.linalg.cholesky(Sig).dot(Z), axis=0)
        return min(np.min(F[-1] - F[-2]), np.min(np.abs(F[-1] - ymax - xi)))
    Xb = rs.rand(40, 3, d)
    Xb = Xb[[b for b in range(40) if margin(Xb[b]) > 1e-4]][:10]
    assert len(Xb) >= 5
    v, G, _ = m.qei(Xb, Z, ymax, xi)
    fd = np.zeros_like(Xb)
    for j in range(3):
        for t in range(d):
            E = np.zeros_like(Xb); E[:, j, t] = h
            fd[:, j, t] = (m.qei(Xb + E, Z, ymax, xi, want_grad=False)[0] - m.qei(Xb - E, Z, ymax, xi, want_grad=False)[0]) / (2 * h)
    live = v > 0
    assert np.sum(live) >= 3
    scale = np.max(np.abs(fd[live]).reshape(np.sum(live), -1), axis=1)
    assert np.max(np.abs(G[live] - fd[live]).reshape(np.sum(live), -1).max(axis=1) / scale) < 1e-6


def test_q1_agrees_with_analytic_ei():
    L = _lib()
    d = 3
    X, Y, rs = _data(200, d, 14)
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.1)
    x = rs.rand(1, d)
    ymax, xi = Y.max() - 0.1, 0.01
    mu, s2 = m.posterior(x, L.FLAG_MODE_CPP | L.FLAG_FP64)
    assert 1e-8 < s2[0] < 10
    ei = m.score_grad(x, L.ACQ_EI, ymax, xi, L.FLAG_MODE_CPP)[0][0]
    Z = np.random.default_rng(8).standard_normal((1, 1 << 16))
    v, _, _ = m.qei(x[None], Z, ymax, xi, want_grad=False)
    se = np.std(np.maximum(0.0, mu[0] + np.sqrt(s2[0]) * Z[0] - ymax - xi)) / np.sqrt(Z.shape[1])
    assert ei > 0 and abs(v[0] - ei) <= 5 * se


def test_batch_that_is_not_positive_definite_gets_nan():
    """noise 0 and one point twice, far from the data (V = 0): Sigma = [[1, 1], [1, 1]] exactly"""
    L = _lib()
    d = 3
    X, Y, rs = _data(40, d, 15)
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.0)
    Xb = rs.rand(5, 2, d)
    Xb[2] = 100.0
    Z = np.random.default_rng(9).standard_normal((2, 128))
    v, G, nbad = m.qei(Xb, Z, Y.max(), 0.01)
    assert nbad == 1 and np.isnan(v[2]) and np.all(np.isnan(G[2]))
    keep = [0, 1, 3, 4]
    v2, G2, nbad2 = m.qei(Xb[keep], Z, Y.max(), 0.01)
    assert nbad2 == 0 and np.array_equal(v2, v[keep]) and np.array_equal(G2, G[keep])
    assert np.all(np.isfinite(v2)) and np.all(np.isfinite(G2))


def test_bad_arguments():
    L = _lib()
    lib = L.lib()
    X, Y, rs = _data(20, 2, 34)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1)
    p = L.dptr
    x = rs.rand(4, 2); z = np.zeros(8); o = np.zeros(64)
    for args in [(None, p(x), 2, 2, p(z), 4, 0.0), (m.handle, p(x), 0, 2, p(z), 4, 0.0), (m.handle, p(x), 2, 33, p(z), 4, 0.0),
                 (m.handle, p(x), 2, 2, p(z), 0, 0.0), (m.handle, p(x), 2, 2, None, 4, 0.0), (m.handle, p(x), 2, 2, p(z), 4, -1.0)]:
        assert lib.ibo_qei(*args[:6], 0.0, 0.01, args[6], p(o), None, None) == L.E_BADARG
    assert lib.ibo_qei(m.handle, p(x), 2, 2, p(z), 4, 0.0, 0.01, 0.0, p(o), None, None) == 0
    Xw = rs.rand(8, 65)
    try:
        wide = L.Model(orc.K_SE_ISO, [3.0], Xw, np.zeros(8), 0.1)
    except L.IBOError:
        return                                        # a model of more than 64 dimensions cannot be built at all
    assert lib.ibo_qei(wide.handle, p(np.ascontiguousarray(Xw[:2])), 1, 2, p(z), 4, 0.0, 0.01, 0.0, p(o), None, None) == L.E_BADARG


def _gp(name):
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, MaternKernel3
    if name == "branin":
        bounds = [[-5., 10.], [0., 15.]]
        X = np.array(orc.lhc_sample(bounds, 10, seed=0))
        return GaussianProcess(MaternKernel3([1.0, 1.0]), X, -orc.branin(X) / 100.0, noise=0.01), bounds
    X = np.random.RandomState(0).rand(200, 6)
    return GaussianProcess(GaussianKernel_ard([.53, .57, 2.5, .34, .27, .35]), X, orc.hartman6_neg(X), noise=0.1), [[0., 1.]] * 6


@pytest.mark.parametrize("name", ["branin", "hartman6"])
def test_maximize_qei(name):
    from ibo_b200.acquisition import maximizeQEI, thompsonBatch
    gp, bounds = _gp(name)
    b = np.array(bounds)
    val, batch = maximizeQEI(gp, bounds, 4, samples=256, seed=3, starts=4, maxiter=50)
    last = maximizeQEI.last
    assert batch.shape == (4, len(bounds)) and last["evaluations"] >= 2
    assert val >= np.max(last["start_values"])
    assert np.all(batch >= b[:, 0]) and np.all(batch <= b[:, 1]) and not np.all(batch == batch[0])
    Z = np.random.default_rng(3).standard_normal((4, 256))
    assert abs(gp.qEI(batch, Z=Z) - val) <= 1e-12 * val
    starts = [thompsonBatch(gp, bounds, 4, seed=3 + k)[0] for k in range(4)]
    assert np.array_equal(last["start_values"], gp.qEI(np.array(starts), Z=Z))
    pending = b[:, 0] + (b[:, 1] - b[:, 0]) * np.random.RandomState(1).rand(2, len(bounds))
    val_p, batch_p = maximizeQEI(gp, bounds, 4, samples=256, seed=3, starts=4, pending=pending, maxiter=50)
    Zp = np.random.default_rng(3).standard_normal((6, 256))
    assert abs(gp.qEI(np.r_[batch_p, pending], Z=Zp) - val_p) <= 1e-12 * val_p
    assert val_p >= np.max(maximizeQEI.last["start_values"])
    assert np.all(batch_p >= b[:, 0]) and np.all(batch_p <= b[:, 1])
