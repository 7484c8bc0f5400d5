"""GPU tests of the pathwise posterior samples (ibo_paths_*, GaussianProcess.sample_paths, thompsonBatch(method='paths')): parity with
the CPU restatement (tests/paths_oracle.py) on the same draws over every kernel and the model variants, exact identities, the paths'
covariance against its analytic form, argmax over 2^20 candidates, the snapshot rule, gradients, independence from the model's
workspace, argument checks, and Thompson batches end to end."""
import ctypes

import numpy as np
import pytest

from oracle import ibo_oracle as orc
import joint_oracle
import paths_oracle as po

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52
# values: |dev - oracle| <= C_VAL eps (sum of the magnitudes of the terms + the rounding of the cosines' arguments).  Both sides solve
# with R (condition numbers up to ~1e4 here at noise 0.1), so the coefficients a and c themselves differ by ~kappa eps.
C_VAL = 2.0 ** 18


def _lib():
    from ibo_b200 import _lib as L
    return L


def _hyper(kind, d):
    th = list(0.3 * np.sqrt(max(d, 3) / 3.0) * (1.0 + 0.5 * np.arange(d) / max(d, 1)))
    return {orc.K_SE_ARD: th, orc.K_SE_ISO: [th[0]], orc.K_MATERN3: [th[0], 0.9], orc.K_MATERN5: [th[0], 0.8],
            orc.K_MATERN5_ARD: th + [0.95]}[kind]


def _data(N, M, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    Xs = rs.rand(M, d)
    Xs[: min(2, M, N)] = X[: min(2, M, N)]
    return X, Y, Xs


def _draws(kind, d, F, S, Ng, seed=0):
    from ibo_b200.gaussianprocess import path_draws
    return path_draws(kind, d, F, S, Ng, seed)


def _check(dev, o, dr, Xs):
    v_o, mag = po.paths(o, *dr, Xs)
    omega, phase = dr[0], dr[1]
    th = o.kernel.theta
    amp = np.sqrt(2.0 * o.kernel.sf2 / omega.shape[0])
    argmag = np.abs(Xs / th[None, :]).dot(np.abs(omega).T) + np.abs(phase)[None, :] + np.abs(omega).dot(np.abs(o.X / th).max(axis=0))[None, :]
    bound = C_VAL * EPS * (mag + amp * argmag.dot(np.abs(dr[2])))
    err = np.abs(dev - v_o)
    assert np.all(err <= bound), float(np.max(err / bound))


# (kind, N, M, S, F, d): every kind, N 1 .. 1000, M 1 .. 2500, S in {1, 7, 128, 1024}, F in {1, 300, 4096}, d in {1, 6, 20, 40}
CASES = [
    (orc.K_SE_ARD, 1, 7, 1, 1, 1), (orc.K_SE_ISO, 50, 129, 7, 300, 6), (orc.K_MATERN3, 129, 129, 128, 4096, 6),
    (orc.K_MATERN5, 1000, 7, 1024, 300, 20), (orc.K_MATERN5_ARD, 129, 1, 7, 1, 40), (orc.K_SE_ARD, 1000, 2500, 128, 4096, 6),
    (orc.K_MATERN3, 50, 2500, 7, 300, 20), (orc.K_SE_ISO, 1, 129, 1024, 4096, 40), (orc.K_MATERN5_ARD, 300, 600, 128, 300, 1),
]


@pytest.mark.parametrize("kind,N,M,S,F,d", CASES)
def test_values_match_the_oracle(kind, N, M, S, F, d):
    L = _lib()
    X, Y, Xs = _data(N, M, d, N + M + S)
    hy = _hyper(kind, d)
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, 0.1)
    m = L.Model(kind, hy, X, Y, 0.1)
    dr = _draws(kind, d, F, S, N)
    p = m.sample_paths(*dr)
    vals, best, idx = p.eval(Xs)
    _check(vals, o, dr, Xs)
    assert np.array_equal(idx, np.argmax(vals, axis=0)) and np.array_equal(best, vals[idx, np.arange(S)])


def test_prior_legacy_appended_and_variance_models():
    L = _lib()
    d, kind, hy = 2, orc.K_SE_ARD, [.3, .4]
    X, Y, Xs = _data(300, 200, d, 4)
    rs = np.random.RandomState(4)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    dr = _draws(kind, d, 500, 9, 300)
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, 0.1, prior=prior)
    _check(L.Model(kind, hy, X, Y, 0.1, prior=prior).sample_paths(*dr).eval(Xs)[0], o, dr, Xs)
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, 0.1)
    _check(L.Model(kind, hy, X, Y, 0.1, invR=o.invR(), sf2=1.0).sample_paths(*dr).eval(Xs)[0], o, dr, Xs)
    m = L.Model(kind, hy, X[:250], Y[:250], 0.1)
    m.append(X[250:], Y[250:])
    _check(m.sample_paths(*dr).eval(Xs)[0], o, dr, Xs)
    # variance model: c over g's 320 points, the mean from the model's 300
    augX = np.r_[X, rs.rand(20, d)]
    aug = L.Model(kind, hy, augX, np.zeros(320), 0.1)
    m = L.Model(kind, hy, X, Y, 0.1)
    m.set_variance_model(aug)
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1)); o.augX = augX
    drg = _draws(kind, d, 500, 9, 320)
    _check(m.sample_paths(*drg).eval(Xs)[0], o, drg, Xs)


def test_identities():
    """argmax = numpy's argmax of the values (ties to the lowest index, NaN never wins); sub-ranges, repeated calls and a second
    object from the same draws give the same bits; the mean over 1024 paths is the posterior mean within 5 standard errors"""
    L = _lib()
    kind, d = orc.K_MATERN5_ARD, 3
    hy = _hyper(kind, d)
    X, Y, Xs = _data(200, 1000, d, 11)
    Xs[500] = Xs[100]; Xs[700] = Xs[100]; Xs[3, 1] = np.nan
    m = L.Model(kind, hy, X, Y, 0.1)
    dr = _draws(kind, d, 2048, 1024, 200, seed=3)
    p = m.sample_paths(*dr)
    vals, best, idx = p.eval(Xs)
    assert np.all(np.isnan(vals[3])) and np.array_equal(vals[500], vals[100]) and np.array_equal(vals[700], vals[100])
    v = np.where(np.isnan(vals), -np.inf, vals)
    assert np.array_equal(idx, np.argmax(v, axis=0)) and not np.any(idx == 500) and not np.any(idx == 3)
    assert np.array_equal(p.eval(Xs[37:901])[0], vals[37:901]) and np.array_equal(p.eval(Xs[999:])[0], vals[999:])
    assert np.array_equal(p.eval(Xs)[0], vals, equal_nan=True)
    assert np.array_equal(m.sample_paths(*dr).eval(Xs)[0], vals, equal_nan=True)
    mu = m.posterior(np.delete(Xs, 3, axis=0), L.FLAG_FP64)[0]
    vv = np.delete(vals, 3, axis=0)
    se = vv.std(axis=1) / np.sqrt(vv.shape[1])
    assert np.all(np.abs(vv.mean(axis=1) - mu) <= 5 * se)


def test_covariance_matches_the_analytic_form():
    """4096 paths (four objects of 1024 with the same F = 8192 features) on 64 points: the empirical covariance against the analytic
    covariance for these features (entrywise within 6 Monte-Carlo standard errors), which with exact kernels is
    Sigma - (1 + noise - sf2) I"""
    L = _lib()
    kind, d, noise = orc.K_MATERN3, 2, 0.1
    hy = _hyper(kind, d)
    X, Y, Xs = _data(40, 64, d, 21)
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, noise)
    m = L.Model(kind, hy, X, Y, noise)
    om, ph, _, _ = _draws(kind, d, 8192, 1, 40, seed=5)
    rng = np.random.default_rng(6)
    vals = np.concatenate([m.sample_paths(om, ph, rng.standard_normal((8192, 1024)), rng.standard_normal((40, 1024))).eval(Xs)[0]
                           for _ in range(4)], axis=1)
    P = lambda A: po.features(o.kernel, om, ph, A)                                        # noqa: E731
    Ps, Px = P(Xs), P(X)
    C = po.analytic_cov(Ps.dot(Ps.T), Ps.dot(Px.T), Px.dot(Px.T), o.kernel.cross(X, Xs), o.R,
                        (1 + noise - o.kernel.sf2) * np.eye(40))
    Ce = np.cov(vals)
    se = np.sqrt((np.outer(np.diag(C), np.diag(C)) + C * C) / vals.shape[1])
    assert np.all(np.abs(Ce - C) <= 6 * se), float(np.max(np.abs(Ce - C) / se))
    _, Sig = joint_oracle.posterior_joint(o, Xs)
    assert np.max(np.abs(C - (Sig - (1 + noise - o.kernel.sf2) * np.eye(64)))) < 0.05


def test_argmax_over_a_million_candidates():
    L = _lib()
    kind, d = orc.K_SE_ARD, 6
    hy = _hyper(kind, d)
    X, Y, _ = _data(256, 1, d, 3)
    Xs = np.random.RandomState(9).rand(1 << 20, d)
    p = L.Model(kind, hy, X, Y, 0.1).sample_paths(*_draws(kind, d, 1024, 16, 256))
    vals, best, idx = p.eval(Xs)
    assert np.array_equal(idx, np.argmax(vals, axis=0)) and np.array_equal(best, vals.max(axis=0))
    _, best2, idx2 = p.eval(Xs, want_values=False)
    assert np.array_equal(idx2, idx) and np.array_equal(best2, best)


def test_snapshot_survives_append_and_destroy():
    L = _lib()
    kind, d = orc.K_MATERN5, 3
    hy = _hyper(kind, d)
    X, Y, Xs = _data(300, 500, d, 5)
    m = L.Model(kind, hy, X[:280], Y[:280], 0.1)
    p = m.sample_paths(*_draws(kind, d, 300, 7, 280))
    v0 = p.eval(Xs)[0]
    g0 = p.grad(Xs[:20], np.arange(20) % 7)
    m.append(X[280:], Y[280:])
    assert np.array_equal(p.eval(Xs)[0], v0)
    m.close()
    assert np.array_equal(p.eval(Xs)[0], v0)
    g1 = p.grad(Xs[:20], np.arange(20) % 7)
    assert np.array_equal(g0[0], g1[0]) and np.array_equal(g0[1], g1[1])


@pytest.mark.parametrize("variant", ["plain", "prior", "variance"])
@pytest.mark.parametrize("kind", [orc.K_SE_ARD, orc.K_SE_ISO, orc.K_MATERN3, orc.K_MATERN5, orc.K_MATERN5_ARD])
def test_gradient(kind, variant):
    """values bit-equal to ibo_paths_eval's, the gradient against the oracle and against central differences of the device values"""
    L = _lib()
    d = 3
    hy = _hyper(kind, d)
    X, Y, Xs = _data(150, 40, d, 13)
    rs = np.random.RandomState(1)
    prior = orc.PriorSpec(rs.rand(3, d), 0.3 * rs.randn(3), 3.0, np.zeros(d), np.ones(d)) if variant == "prior" else None
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, 0.1, prior=prior)
    m = L.Model(kind, hy, X, Y, 0.1, prior=prior)
    ng = 150
    if variant == "variance":
        augX = np.r_[X, rs.rand(10, d)]
        aug = L.Model(kind, hy, augX, np.zeros(160), 0.1)
        m.set_variance_model(aug)
        o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1)); o.augX = augX
        ng = 160
    dr = _draws(kind, d, 600, 5, ng, seed=2)
    p = m.sample_paths(*dr)
    which = rs.randint(0, 5, len(Xs))
    v, G = p.grad(Xs, which)
    assert np.array_equal(v, p.eval(Xs)[0][np.arange(len(Xs)), which])
    v_o, G_o = po.paths_grad(o, *dr, Xs, which)
    assert np.all(np.abs(G - G_o) <= 1e-9 * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12)
    h = 1e-6
    for t in range(d):
        E = np.zeros(d); E[t] = h
        fd = (p.grad(Xs + E, which)[0] - p.grad(Xs - E, which)[0]) / (2 * h)
        assert np.all(np.abs(fd - G[:, t]) <= 1e-5 * (1 + np.abs(G).max()))


def test_paths_leave_the_model_workspace_alone():
    """joint samples, gradients, q-EI and MES interleaved with paths calls on one model: byte-identical to a fresh model's"""
    L = _lib()
    kind, d = orc.K_SE_ARD, 3
    hy = _hyper(kind, d)
    X, Y, Xs = _data(200, 300, d, 17)
    Z = np.random.default_rng(0).standard_normal((300, 8))
    Zq = np.random.default_rng(1).standard_normal((4, 64))
    ys = Y.max() + 0.1 + np.arange(5) * 0.05

    def calls(m, between):
        out = []
        for f in (lambda: m.posterior_sample(Xs, Z, 1e-10), lambda: m.posterior_grad(Xs),
                  lambda: m.qei(Xs[:256].reshape(64, 4, d), Zq, Y.max(), 0.01), lambda: m.mes(Xs, ys, want_grad=True)):
            between()
            out.append(f())
        return out

    fresh = calls(L.Model(kind, hy, X, Y, 0.1), lambda: None)
    m = L.Model(kind, hy, X, Y, 0.1)
    dr = _draws(kind, d, 400, 9, 200)
    ps = []

    def between():
        ps.append(m.sample_paths(*dr))
        ps[-1].eval(Xs)
        ps[-1].grad(Xs[:9], np.arange(9))

    got = calls(m, between)
    for a, b in zip(fresh, got):
        for x, y in zip(a, b):
            if isinstance(x, np.ndarray):
                assert x.tobytes() == y.tobytes()
            else:
                assert x == y
    assert all(np.array_equal(q.eval(Xs)[0], ps[0].eval(Xs)[0]) for q in ps)


def test_bad_arguments():
    L = _lib()
    lib = L.lib()
    kind, d = orc.K_SE_ARD, 2
    X, Y, Xs = _data(20, 5, d, 1)
    m = L.Model(kind, [.3, .4], X, Y, 0.1)
    om, ph, w, e = _draws(kind, d, 8, 3, 20)
    dp = L.dptr
    h = ctypes.c_void_p()
    info = ctypes.c_int(0)
    for F, S in ((0, 3), (65537, 3), (8, 0), (8, 1025)):
        assert lib.ibo_paths_create(m.handle, F, S, dp(om), dp(ph), dp(w), dp(e), ctypes.byref(h), ctypes.byref(info)) == L.E_BADARG
    assert lib.ibo_paths_create(m.handle, 8, 3, None, dp(ph), dp(w), dp(e), ctypes.byref(h), ctypes.byref(info)) == L.E_BADARG
    assert lib.ibo_paths_create(None, 8, 3, dp(om), dp(ph), dp(w), dp(e), ctypes.byref(h), ctypes.byref(info)) == L.E_BADARG
    big = L.Model(orc.K_MATERN3, [.4, 1.2], 100 * X, Y, 0.1)                   # sf2 = 1.44 > 1 + noise; far-apart points keep R SPD
    with pytest.raises(L.IBOError) as ei:
        big.sample_paths(om, ph, w, e)
    assert ei.value.code == L.E_BADARG
    p = m.sample_paths(om, ph, w, e)
    for which in ([0, 1, 2, 3, 0], [0, -1, 0, 0, 0]):
        with pytest.raises(L.IBOError) as ei:
            p.grad(Xs, which)
        assert ei.value.code == L.E_BADARG
    assert lib.ibo_paths_eval(p._h, None, 5, None, None, None) == L.E_BADARG
    assert lib.ibo_paths_eval(p._h, dp(Xs), 0, None, None, None) == L.E_BADARG
    assert lib.ibo_paths_destroy(None) == L.E_BADARG


def _branin_gp():
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    bb = [[-5., 10.], [0., 15.]]
    Xb = np.array(orc.lhc_sample(bb, 50, seed=0))
    return GaussianProcess(GaussianKernel_ard([3.4, 10.0]), Xb, np.array([-orc.branin(x) for x in Xb]) / 100.0, noise=0.1), bb


def _hartman_gp():
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    X = np.random.RandomState(2).rand(200, 6)
    return GaussianProcess(GaussianKernel_ard([0.3] * 6), X, -orc.hartman6_neg(X), noise=0.1), [[0., 1.]] * 6


@pytest.mark.parametrize("make", [_branin_gp, _hartman_gp])
def test_thompson_batch_with_paths_end_to_end(make):
    from ibo_b200.acquisition import thompsonBatch
    from ibo_b200.utils.latinhypercube import lhcSample
    gp, bounds = make()
    q = 4
    Xp, idx = thompsonBatch(gp, bounds, q, samples=4096, seed=0, method='paths', polish=True)
    b = np.array(bounds)
    assert Xp.shape == (q, len(bounds)) and np.all(Xp >= b[:, 0]) and np.all(Xp <= b[:, 1])
    C = np.array(lhcSample(bounds, 4096, seed=0), dtype=float)
    paths = gp.sample_paths(q, 2048, seed=0)
    v1 = paths.grad(Xp, np.arange(q))[0]
    v0 = paths.grad(C[idx], np.arange(q))[0]
    assert np.all(v1 >= v0)
    X0, i0 = thompsonBatch(gp, bounds, q, samples=4096, seed=0, method='paths')
    assert np.array_equal(i0, idx) and np.array_equal(X0, C[idx])
    # method='joint' (the default) is what it was: the argmax of mu + chol(cov) Z over the same candidates
    Xj, ij = thompsonBatch(gp, bounds, q, samples=512, seed=1)
    Cj = np.array(lhcSample(bounds, 512, seed=1), dtype=float)
    _, ref = gp.model.posterior_sample(Cj, np.random.default_rng(1).standard_normal((512, q)), 0.0, want_F=False)
    assert np.array_equal(ij, ref) and np.array_equal(Xj, Cj[ref])


def test_laplace_models():
    """the noise factor chol(inv(C) + (1 + noise - sf2) I) on the device: a preference model (ibo_model_create_pref, inv(C) formed on the
    device) with its gradient, and a PrefGaussianProcess after addObservationPoint, whose variance model carries a host inv(C) padded
    with zeros, through GaussianProcess.sample_paths"""
    from ibo_b200.gaussianprocess import PrefGaussianProcess, path_draws
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    L = _lib()
    kind, d, hy = orc.K_SE_ARD, 3, [.3, .4, .5]
    rs = np.random.RandomState(12)
    N, P, cdiag = 80, 60, 5.0
    X, Y = rs.rand(N, d), rs.randn(N)
    a = rs.randint(0, N, P)
    b = (a + 1 + rs.randint(0, N - 1, P)) % N
    wts = 0.5 + rs.rand(P)
    C = cdiag * np.eye(N)
    np.add.at(C, (a, a), wts); np.add.at(C, (b, b), wts); np.subtract.at(C, (a, b), wts); np.subtract.at(C, (b, a), wts)
    Cinv = np.linalg.inv(C)
    o = orc.GPOracle(orc.KernelSpec(kind, hy, d), X, Y, 0.1, Cinv=Cinv)
    m = L.Model(kind, hy, X, Y, 0.1, pref=(a, b, wts, cdiag))
    dr = _draws(kind, d, 500, 9, N)
    p = m.sample_paths(*dr)
    Xs = rs.rand(200, d)
    _check(p.eval(Xs)[0], o, dr, Xs)
    which = np.arange(40) % 9
    v, G = p.grad(Xs[:40], which)
    _, G_o = po.paths_grad(o, *dr, Xs[:40], which)
    assert np.all(np.abs(G - G_o) <= 1e-9 * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12)
    gp = PrefGaussianProcess.fromLaplace(GaussianKernel_ard(hy), X, Y, C, noise=0.1)
    Pts = rs.rand(5, d)
    gp.addObservationPoint(Pts)
    augX = np.r_[X, Pts]
    pad = np.zeros((N + 5, N + 5)); pad[:N, :N] = Cinv
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad); o.augX = augX; o.augCinv = pad
    paths = gp.sample_paths(7, 400, seed=3)
    _check(paths(Xs), o, path_draws(kind, d, 400, 7, N + 5, seed=3), Xs)
    best, idx = paths.argmax(Xs)
    assert np.array_equal(idx, np.argmax(paths(Xs), axis=0))


@pytest.mark.parametrize("variance", [False, True])
@pytest.mark.parametrize("noise", [1e-4, 1e-6])
def test_small_noise_against_longdouble(noise, variance):
    """at noise 1e-4 and 1e-6, where R is ill-conditioned, the device's values against the longdouble reference (tests/build_oracle.py):
    the device error stays within 4 x the larger error of two FP64 yardsticks (the oracle's triangular solves, and the same formulas
    through the device's own W = inv(L)) plus eps times the largest term.  SE-ARD without a magnitude has sf2 = 1, so
    R = K + noise I: condition numbers ~1e6 and ~1e8 here, and the noise draw is sqrt(noise) e"""
    import build_oracle as bo
    LD = np.longdouble
    L = _lib()
    kind, d, hy = orc.K_SE_ARD, 3, [.5, .6, .7]
    N, M, S, F = 200, 100, 8, 256
    X, Y, Xs = _data(N, M, d, 31)
    k = orc.KernelSpec(kind, hy, d)
    o = orc.GPOracle(k, X, Y, noise)
    m = L.Model(kind, hy, X, Y, noise)
    g, Xg, aug = m, X, None
    if variance:
        Xg = np.r_[X, np.random.RandomState(32).rand(16, d)]
        g = L.Model(kind, hy, Xg, np.zeros(len(Xg)), noise)
        m.set_variance_model(g)
        o.augL = np.linalg.cholesky(orc.build_R(k, Xg, noise)); o.augX = Xg
        aug = (Xg, bo.build_R(k, Xg, noise))
    om, ph, w, e = dr = _draws(kind, d, F, S, len(Xg), seed=4)
    dev = m.sample_paths(*dr).eval(Xs)[0]
    lo = bo._Model(k, X, Y, noise, None, aug)
    feat = lambda A: np.sqrt(LD(2 * k.sf2) / F) * np.cos((np.asarray(A, LD) / np.asarray(k.theta, LD)) @ np.asarray(om, LD).T  # noqa: E731
                                                           + np.asarray(ph, LD))
    c = bo.back_solve(lo.Lg, bo.forward_solve(lo.Lg, feat(Xg) @ np.asarray(w, LD) + np.sqrt(LD(1 + noise - k.sf2)) * np.asarray(e, LD)))
    ref = lo.mean(Xs)[0][:, None] + feat(Xs) @ np.asarray(w, LD) - bo.cross(k, Xg, Xs).T @ c
    y1, mag = po.paths(o, *dr, Xs)
    W, Wg = m.matrix(2), g.matrix(2)
    cw = Wg.T.dot(Wg.dot(po.features(k, om, ph, Xg).dot(w) + po.noise(o, e)))
    y2 = k.cross(X, Xs).T.dot(W.T.dot(W.dot(Y)))[:, None] + po.features(k, om, ph, Xs).dot(w) - k.cross(Xg, Xs).T.dot(cw)
    err = lambda v: float(np.max(np.abs(np.asarray(v, LD) - ref)))                                              # noqa: E731
    floor = EPS * float(np.max(mag))
    assert err(dev) <= 4 * max(err(y1), err(y2)) + floor, (err(dev), err(y1), err(y2), floor)
