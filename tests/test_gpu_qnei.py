"""GPU tests of the noisy batch expected improvement (ibo_qnei and its Python surface) against the oracle's full-form restatement
(qnei_oracle), its identity with ibo_qei, finite differences of the device's own values, its bit invariants, its errors, the shared
workspace, and maximizeQNEI."""
import ctypes

import numpy as np
import pytest

from oracle import ibo_oracle as orc
import qei_oracle as qo
import qnei_oracle as no

pytestmark = pytest.mark.gpu

KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}
# (kind, N, P, q, S, noise): every kind; N = 1, 50, 129, 1000; P = 1, 7, 129 and N; q = 1, 4, 32; S = 1, 1024; noise 0.1 and 1e-3
CASES = [
    (orc.K_SE_ARD, 1, 1, 4, 1024, 0.1), (orc.K_SE_ISO, 50, 7, 32, 1024, 0.1), (orc.K_MATERN3, 129, 129, 1, 1024, 1e-3),
    (orc.K_MATERN5, 1000, 7, 4, 1, 0.1), (orc.K_MATERN5_ARD, 129, 1, 32, 1, 1e-3), (orc.K_SE_ARD, 1000, 7, 32, 1024, 0.1),
    (orc.K_MATERN3, 50, 50, 4, 1024, 0.1), (orc.K_SE_ISO, 1, 1, 1, 1, 1e-3), (orc.K_MATERN5_ARD, 1000, 1000, 4, 1024, 1e-3),
    (orc.K_MATERN5, 50, 129, 1, 1024, 1e-3), (orc.K_SE_ARD, 129, 7, 4, 1024, 1e-3),
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


def _check_grad(G, G_o, rel=1e-9):
    """<= 1e-9 (rel) of the row's largest component + 1e-12"""
    G, G_o = G.reshape(-1, G.shape[-1]), G_o.reshape(-1, G_o.shape[-1])
    bound = rel * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12
    assert np.all(np.abs(G - G_o) <= bound), np.max(np.abs(G - G_o) - bound)


def _margin(o, Xq, Xbase, Z, jitter):
    """distance of the oracle's draws to a kink of the integrand: the two largest draws of the batch, of the baseline, and
    improvement 0"""
    P = len(Xbase)
    mu, Sig = no.latent_joint(o, np.r_[Xbase, Xq])
    F = mu[:, None] + np.linalg.cholesky(Sig + jitter * np.eye(len(Sig))).dot(Z)
    out = [np.min(np.abs(np.max(F[P:], axis=0) - np.max(F[:P], axis=0)))]
    for part in (F[:P], F[P:]):
        if part.shape[0] > 1:
            Fs = np.sort(part, axis=0)
            out.append(np.min(Fs[-1] - Fs[-2]))
    return min(out)


def _compare(o, Xb, Xbase, Z, jitter, v, G, inc=None, tie=1e-8, vfloor=1e-5, grel=1e-9):
    """values and incumbent everywhere; gradients of the batches whose draws are farther than `tie` from an argmax tie"""
    v_o, G_o = no.qnei(o, Xb, Xbase, Z, jitter)
    assert np.all(np.abs(v - v_o) <= 1e-10 * np.maximum(np.abs(v_o), vfloor)), np.max(np.abs(v - v_o))
    keep = [b for b in range(len(Xb)) if _margin(o, Xb[b], Xbase, Z, jitter) > tie]
    assert len(keep) >= max(1, len(Xb) // 2)
    _check_grad(G[keep], G_o[keep], grel)
    if inc is not None:
        inc_o = no.incumbent(o, Xbase, Z, jitter)
        assert np.all(np.abs(inc - inc_o) <= 1e-10 * np.maximum(np.abs(inc_o), 1e-5))
    return v_o


@pytest.mark.parametrize("kind,N,P,q,S,noise", CASES)
def test_matches_oracle(kind, N, P, q, S, noise):
    L = _lib()
    d = 3
    X, Y, rs = _data(N, d, 100 * N + 10 * q + kind)
    hyper = KINDS[kind]
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise)
    m = L.Model(kind, hyper, X, Y, noise)
    Xbase = np.r_[X[np.argsort(Y, kind='stable')], rs.rand(max(0, P - N), d)][:P]     # the lowest Y first: a baseline to improve on
    B = 6
    Xb = rs.rand(B, q, d)
    Z = np.random.default_rng(q + S + P).standard_normal((P + q, S))
    jitter = 1e-8
    v, G, nbad, inc = m.qnei(Xb, Xbase, Z, jitter)
    assert nbad == 0
    v_o = _compare(o, Xb, Xbase, Z, jitter, v, G, inc)
    assert S == 1 or np.any(v_o > 0)
    m.close()


def test_prior_from_inverse_and_appended_models():
    L = _lib()
    d = 2
    X, Y, rs = _data(300, d, 4)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    Xb = rs.rand(20, 4, d)
    Xbase = X[::10]
    Z = np.random.default_rng(1).standard_normal((len(Xbase) + 4, 256))
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1, prior=prior)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, prior=prior)
    v, G, _, inc = m.qnei(Xb, Xbase, Z, 1e-6)
    _compare(o, Xb, Xbase, Z, 1e-6, v, G, inc)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, invR=o.invR(), sf2=1.0)
    # a model built from the caller's inverse carries W only to cond(R) eps, and at training points the latent variance is a
    # difference of nearly equal terms: its baseline is taken off them, and values are compared with a floor of 1e-2 and gradients
    # to 1e-8 of the row's largest component
    Xoff = rs.rand(30, d)
    v, G, _, inc = m.qnei(Xb, Xoff, Z, 1e-8)
    _compare(o, Xb, Xoff, Z, 1e-8, v, G, inc, vfloor=1e-2, grel=1e-8)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X[:250], Y[:250], 0.1)
    m.qnei(Xb, Xoff, Z, 1e-8)                         # a call before the append: nothing cached may survive it
    m.append(X[250:], Y[250:])
    v, G, _, inc = m.qnei(Xb, Xoff, Z, 1e-8)         # the rank-1 appends' W, like the inverse's, off the training points
    _compare(o, Xb, Xoff, Z, 1e-8, v, G, inc, vfloor=1e-2, grel=1e-8)


def test_pref_gp_before_and_after_an_observation_point():
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
    base = gp.qnei_baseline()
    assert np.array_equal(base, X)
    Xb = rs.rand(30, 4, d) * 10
    Z = np.random.default_rng(3).standard_normal((N + 4, 512))
    v, G = gp.qNEI(Xb, Z=Z, grad=True)
    _compare(o, Xb, base, Z, 1e-8, v, G)
    assert np.array_equal(gp.qNEI(Xb, Z=Z), v)
    P = rs.rand(3, d) * 10
    gp.addObservationPoint(P)
    augX = np.r_[X, P]
    pad = np.zeros((N + 3, N + 3)); pad[:N, :N] = Cinv
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad); o.augX = augX
    v, G = gp.qNEI(Xb, Z=Z, grad=True)
    _compare(o, Xb, gp.qnei_baseline(), Z, 1e-8, v, G)


@pytest.mark.parametrize("kind,hyper", [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_MATERN3, [.5]), (orc.K_MATERN5_ARD, [.3, .4, .5])])
def test_identity_with_qei(kind, hyper):
    """sf2 = 1 + noise and one baseline point no kernel reaches, with a zero row of Z: q-NEI = q-EI with ymax = 0, xi = 0"""
    L = _lib()
    d, noise = 3, 0.1
    hyper = hyper + [np.sqrt(1 + noise)]
    X, Y, rs = _data(300, d, 40 + kind)
    m = L.Model(kind, hyper, X, Y, noise)
    far = np.full((1, d), 1e4)
    Xb = rs.rand(50, 4, d)
    Zq = np.random.default_rng(11).standard_normal((4, 512))
    v, G, _, inc = m.qnei(Xb, far, np.r_[np.zeros((1, 512)), Zq], 0.0)
    ve, Ge, _ = m.qei(Xb, Zq, 0.0, 0.0)
    assert np.all(inc == 0) and np.any(ve > 0)
    assert np.all(np.abs(v - ve) <= 1e-13 * np.abs(ve))
    assert np.all(np.abs(G - Ge) <= 1e-13 * np.max(np.abs(Ge), axis=(1, 2), keepdims=True))


def test_chunks_are_batch_invariant_and_reproducible():
    """N = 4000, P = 129, S = 1024: chunks of floor(2^26 / (2 4096 + 2 256 + 1024) / 128) 128 = 6784 points, 1696 batches of 4, so
    4000 batches take three; a sub-range across a chunk boundary called alone gives the same rows bit for bit, and so do a second
    identical call and the values without the gradient"""
    L = _lib()
    d = 3
    X, Y, _ = _data(4000, d, 30)
    Xbase = X[:129]
    Xb = np.random.RandomState(31).rand(4000, 4, d)
    Z = np.random.default_rng(6).standard_normal((133, 1024))
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.1)
    v, G, _, inc = m.qnei(Xb, Xbase, Z, 1e-8)
    v2, G2, _, inc2 = m.qnei(Xb, Xbase, Z, 1e-8)
    assert np.array_equal(v, v2) and np.array_equal(G, G2) and np.array_equal(inc, inc2)
    vn, Gn, _, _ = m.qnei(Xb, Xbase, Z, 1e-8, want_grad=False)
    assert Gn is None and np.array_equal(v, vn)
    for lo, hi in ((1690, 1700), (3390, 3395), (0, 1), (3999, 4000)):
        a, b, _, _ = m.qnei(Xb[lo:hi], Xbase, Z, 1e-8)
        assert np.array_equal(a, v[lo:hi]) and np.array_equal(b, G[lo:hi])
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], d), X, Y, 0.1)
    rows = np.r_[1694:1698, 3390:3394]
    _compare(o, Xb[rows], Xbase, Z, 1e-8, v[rows], G[rows], inc)


def test_gradient_matches_finite_differences_of_device_values():
    L = _lib()
    d = 4
    X, Y, rs = _data(300, d, 21)
    hyper = [.3, .4, .5, .6, .95]
    m = L.Model(orc.K_MATERN5_ARD, hyper, X, Y, 0.1)
    o = orc.GPOracle(orc.KernelSpec(orc.K_MATERN5_ARD, hyper, d), X, Y, 0.1)
    Xbase = X[np.argsort(Y)[:20]]
    Z = np.random.default_rng(7).standard_normal((23, 32))
    jitter, h = 1e-8, 1e-6
    Xb = rs.rand(40, 3, d)
    Xb = Xb[[b for b in range(40) if _margin(o, Xb[b], Xbase, Z, jitter) > 1e-4]][:10]
    assert len(Xb) >= 5
    v, G, _, _ = m.qnei(Xb, Xbase, Z, jitter)
    fd = np.zeros_like(Xb)
    for j in range(3):
        for t in range(d):
            E = np.zeros_like(Xb); E[:, j, t] = h
            fd[:, j, t] = (m.qnei(Xb + E, Xbase, Z, jitter, want_grad=False)[0] - m.qnei(Xb - E, Xbase, Z, jitter, want_grad=False)[0]) / (2 * h)
    live = v > 0
    assert np.sum(live) >= 3
    scale = np.max(np.abs(fd[live]).reshape(np.sum(live), -1), axis=1)
    assert np.max(np.abs(G[live] - fd[live]).reshape(np.sum(live), -1).max(axis=1) / scale) < 1e-6


def test_errors():
    """a repeated baseline point far from the data (Sigma_bb = [[1, 1], [1, 1]] exactly) with jitter 0: NotPositiveDefinite at
    pivot 2; a batch with a NaN coordinate: NaN and nbad, the other batches unchanged"""
    L = _lib()
    d = 3
    X, Y, rs = _data(40, d, 15)
    m = L.Model(orc.K_SE_ARD, KINDS[orc.K_SE_ARD], X, Y, 0.1)
    Xb = rs.rand(5, 2, d)
    Z = np.random.default_rng(9).standard_normal((5, 128))
    base = np.r_[X[:1], np.full((2, d), 100.0)]
    with pytest.raises(L.NotPositiveDefinite) as e:
        m.qnei(Xb, base, Z, 0.0)
    assert e.value.pivot == 3
    Xbase = X[:3]
    v0, G0, nbad0, _ = m.qnei(Xb, Xbase, Z, 1e-8)           # the handle works after the failure
    Xn = Xb.copy()
    Xn[2, 1, 0] = np.nan
    v, G, nbad, _ = m.qnei(Xn, Xbase, Z, 1e-8)
    assert nbad0 == 0 and nbad == 1 and np.isnan(v[2]) and np.all(np.isnan(G[2]))
    keep = [0, 1, 3, 4]
    assert np.array_equal(v[keep], v0[keep]) and np.array_equal(G[keep], G0[keep])


def test_bad_arguments():
    L = _lib()
    lib = L.lib()
    X, Y, rs = _data(20, 2, 34)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1)
    p = L.dptr
    x = rs.rand(4, 2); xb = rs.rand(3, 2); z = np.zeros(8 * 8); o = np.zeros(64)
    good = (m.handle, p(x), 2, 2, p(xb), 3, p(z), 4, 0.0)
    changes = [(0, None), (1, None), (2, 0), (3, 0), (3, 33), (4, None), (5, 0), (5, 8193), (6, None), (7, 0), (7, 8193), (8, -1.0),
               (8, float("nan"))]
    for i, val in changes:
        a = list(good); a[i] = val
        assert lib.ibo_qnei(*a, p(o), None, None, None, None) == L.E_BADARG, (i, val)
    assert lib.ibo_qnei(*good, p(o), None, None, None, None) == 0
    hot = L.Model(orc.K_SE_ARD, [.3, .4, 2.0], X * 100, Y, 0.1)           # sf2 = 4 > 1 + noise: the latent Sigma is not PSD
                                                                          # (points far apart, so that R itself is)
    assert lib.ibo_qnei(hot.handle, *good[1:], p(o), None, None, None, None) == L.E_BADARG
    Xw = rs.rand(8, 65)
    try:
        wide = L.Model(orc.K_SE_ISO, [3.0], Xw, np.zeros(8), 0.1)
    except L.IBOError:
        return                                        # a model of more than 64 dimensions cannot be built at all
    xw = np.ascontiguousarray(Xw[:2])
    assert lib.ibo_qnei(wide.handle, p(xw), 1, 2, p(xw), 1, p(z), 4, 0.0, p(o), None, None, None, None) == L.E_BADARG


def test_shared_workspace_gives_fresh_handle_bytes():
    """ibo_qnei interleaved with ibo_qei, ibo_posterior_sample, ibo_score_grad and ibo_mes on one handle: every call returns the
    bytes a fresh handle returns"""
    L = _lib()
    d = 3
    X, Y, rs = _data(700, d, 50)
    kind, hyper = orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD]
    Xb = rs.rand(300, 4, d)
    Xbase = X[:200]
    Z = np.random.default_rng(12).standard_normal((204, 512))
    Zq = Z[200:]
    C = rs.rand(500, d)
    Zs = np.random.default_rng(13).standard_normal((500, 8))
    ystar = Y.max() + np.linspace(0.1, 1.0, 5)
    calls = [
        lambda m: m.qnei(Xb, Xbase, Z, 1e-8),
        lambda m: m.qei(Xb, Zq, Y.max(), 0.01),
        lambda m: m.posterior_sample(C, Zs, 1e-8),
        lambda m: m.score_grad(C, L.ACQ_EI, Y.max(), 0.01),
        lambda m: m.mes(C, ystar, want_grad=True),
        lambda m: m.qnei(Xb[:50], Xbase[:30], np.r_[Z[:30], Zq], 0.0, want_grad=False),
    ]
    shared = L.Model(kind, hyper, X, Y, 0.1)
    for f in calls + calls[::-1]:
        fresh = L.Model(kind, hyper, X, Y, 0.1)
        a, b = f(shared), f(fresh)
        fresh.close()
        for x, y in zip(a, b):
            if isinstance(x, np.ndarray):
                assert x.tobytes() == y.tobytes()
            else:
                assert x == y


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
def test_maximize_qnei(name):
    from ibo_b200.acquisition import maximizeQNEI, thompsonBatch
    gp, bounds = _gp(name)
    b = np.array(bounds)
    base = gp.qnei_baseline()
    P = len(base)
    val, batch = maximizeQNEI(gp, bounds, 4, samples=256, seed=3, starts=4, maxiter=50)
    last = maximizeQNEI.last
    assert batch.shape == (4, len(bounds)) and last["evaluations"] >= 2 and np.array_equal(last["baseline"], base)
    assert val >= np.max(last["start_values"])
    assert np.all(batch >= b[:, 0]) and np.all(batch <= b[:, 1])
    Z = np.random.default_rng(3).standard_normal((P + 4, 256))
    assert abs(gp.qNEI(batch, Z=Z) - val) <= 1e-12 * val
    starts = [thompsonBatch(gp, bounds, 4, seed=3 + k, jitter=1e-8)[0] for k in range(4)]
    assert np.array_equal(last["start_values"], gp.qNEI(np.array(starts), Z=Z))
    pending = b[:, 0] + (b[:, 1] - b[:, 0]) * np.random.RandomState(1).rand(2, len(bounds))
    val_p, batch_p = maximizeQNEI(gp, bounds, 4, samples=256, seed=3, starts=4, pending=pending, maxiter=50)
    Zp = np.random.default_rng(3).standard_normal((P + 6, 256))
    vp, Gp = gp.qNEI(np.r_[batch_p, pending], Z=Zp, grad=True)
    assert abs(vp - val_p) <= 1e-12 * val_p
    assert val_p >= np.max(maximizeQNEI.last["start_values"])
    assert np.all(batch_p >= b[:, 0]) and np.all(batch_p <= b[:, 1])
