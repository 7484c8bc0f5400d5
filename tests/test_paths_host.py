"""CPU tests of the pathwise posterior samples' host side: the spectral draws of every kernel against its covariance, the analytic
covariance of the paths against the joint posterior, the oracle's gradient against finite differences, and the argument checks and
draw order behind GaussianProcess.sample_paths."""
import numpy as np
import pytest

from oracle import ibo_oracle as orc
import joint_oracle
import paths_oracle as po

from ibo_b200.gaussianprocess import path_draws, spectral_draws

KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}


def _gp(kind, N=30, d=3, noise=0.1, seed=0, prior=False):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    pr = orc.PriorSpec(rs.rand(3, d), 0.3 * rs.randn(3), 3.0, np.zeros(d), np.ones(d)) if prior else None
    return orc.GPOracle(orc.KernelSpec(kind, KINDS[kind], d), X, Y, noise, prior=pr), rs


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_spectral_draws_reproduce_the_kernel(kind):
    """2^16 fixed-seed frequencies: the feature Gram matrix Phi Phi^T matches the kernel within 6 standard deviations of the Monte-Carlo
    estimate (each of the F terms lies in [-2 sf2, 2 sf2] with variance <= sf2^2, so the standard deviation is <= sf2 / sqrt(F)); the
    wrong Matern order misses that bound, so a wrong degree of freedom or scale is caught"""
    o, rs = _gp(kind)
    F = 1 << 16
    Xs = rs.rand(40, 3) * 0.8
    om = spectral_draws(kind, np.random.default_rng(7), F, 3)
    ph = np.random.default_rng(8).uniform(0, 2 * np.pi, F)
    P = po.features(o.kernel, om, ph, Xs)
    bound = 6 * o.kernel.sf2 / np.sqrt(F)
    assert np.max(np.abs(P.dot(P.T) - o.kernel.cross(Xs, Xs))) <= bound
    if kind in (orc.K_MATERN3, orc.K_MATERN5):
        wrong = orc.K_MATERN5 if kind == orc.K_MATERN3 else orc.K_MATERN3
        Pw = po.features(o.kernel, spectral_draws(wrong, np.random.default_rng(7), F, 3), ph, Xs)
        assert np.max(np.abs(Pw.dot(Pw.T) - o.kernel.cross(Xs, Xs))) > bound


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_analytic_covariance_with_exact_kernels_is_sigma_minus_the_noise(kind):
    o, rs = _gp(kind)
    Xs = rs.rand(9, 3)
    _, Sig = joint_oracle.posterior_joint(o, Xs)
    k = o.kernel
    Ks = k.cross(o.X, Xs)
    EEt = (1 + o.noise - k.sf2) * np.eye(len(o.X))
    C = po.analytic_cov(k.cross(Xs, Xs), Ks.T, k.cross(o.X, o.X), Ks, o.R, EEt)
    assert np.max(np.abs(C - (Sig - (1 + o.noise - k.sf2) * np.eye(9)))) < 1e-12


def test_analytic_covariance_with_features_converges():
    """with random Fourier features the covariance approaches Sigma - (1 + noise - sf2) I as F grows; at F = 2^14 within 0.02"""
    o, rs = _gp(orc.K_MATERN3)
    Xs = rs.rand(7, 3)
    _, Sig = joint_oracle.posterior_joint(o, Xs)
    target = Sig - (1 + o.noise - o.kernel.sf2) * np.eye(7)
    errs = []
    for F in (256, 1 << 14):
        om, ph, _, _ = path_draws(orc.K_MATERN3, 3, F, 1, 30, seed=1)
        Ps, Px = po.features(o.kernel, om, ph, Xs), po.features(o.kernel, om, ph, o.X)
        C = po.analytic_cov(Ps.dot(Ps.T), Ps.dot(Px.T), Px.dot(Px.T), o.kernel.cross(o.X, Xs), o.R,
                            (1 + o.noise - o.kernel.sf2) * np.eye(30))
        errs.append(np.max(np.abs(C - target)))
    assert errs[1] < 0.02 and errs[1] < errs[0]


@pytest.mark.parametrize("variant", ["plain", "prior", "variance", "laplace"])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_oracle_gradient_matches_finite_differences(kind, variant):
    o, rs = _gp(kind, prior=(variant == "prior"))
    ng = 30
    if variant == "laplace":
        B = rs.randn(30, 30) * 0.1
        o = orc.GPOracle(o.kernel, o.X, o.Y, o.noise, Cinv=np.linalg.inv(5 * np.eye(30) + B.dot(B.T)))
    if variant == "variance":
        augX = np.r_[o.X, rs.rand(5, 3)]
        o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, o.noise)); o.augX = augX
        ng = 35
    dr = path_draws(kind, 3, 200, 4, ng, seed=3)
    Xs = rs.rand(6, 3)
    which = np.arange(6) % 4
    v, G = po.paths_grad(o, *dr, Xs, which)
    h = 1e-6
    for t in range(3):
        E = np.zeros(3); E[t] = h
        fd = (po.paths(o, *dr, Xs + E)[0] - po.paths(o, *dr, Xs - E)[0])[np.arange(6), which] / (2 * h)
        assert np.all(np.abs(fd - G[:, t]) <= 1e-6 * (1 + np.abs(G).max()))
    assert np.array_equal(v, po.paths(o, *dr, Xs)[0][np.arange(6), which])


def test_laplace_noise_factor():
    """with inv(C) the noise draw is chol(inv(C) + (1 + noise - sf2) I) e: its covariance plus K is R + inv(C), and a zero inv(C)
    gives the plain sqrt(1 + noise - sf2) e"""
    o, rs = _gp(orc.K_MATERN5)
    B = rs.randn(30, 30) * 0.1
    Cinv = np.linalg.inv(5 * np.eye(30) + B.dot(B.T))
    ol = orc.GPOracle(o.kernel, o.X, o.Y, o.noise, Cinv=Cinv)
    E = po.noise(ol, np.eye(30))
    K = o.kernel.cross(o.X, o.X)
    assert np.max(np.abs(E.dot(E.T) + K - ol.A)) < 1e-12
    o.augL, o.augX, o.augCinv = o.L, o.X, np.zeros((30, 30))
    assert np.array_equal(po.noise(o, np.eye(30)), np.sqrt(1 + o.noise - o.kernel.sf2) * np.eye(30))


def test_draw_order_and_arguments():
    """sample_paths draws omega, then the phases, then w, then e from one default_rng(seed)"""
    rng = np.random.default_rng(42)
    z = rng.standard_normal((16, 3))
    u = rng.chisquare(3.0, size=16)
    ph = rng.uniform(0.0, 2 * np.pi, 16)
    w = rng.standard_normal((16, 5))
    e = rng.standard_normal((11, 5))
    got = path_draws(orc.K_MATERN3, 3, 16, 5, 11, seed=42)
    for a, b in zip(got, (z * np.sqrt(3.0 / u)[:, None], ph, w, e)):
        assert np.array_equal(a, b)
    assert all(np.array_equal(a, b) for a, b in zip(got, path_draws(orc.K_MATERN3, 3, 16, 5, 11, seed=42)))
    assert np.array_equal(path_draws(orc.K_SE_ISO, 2, 4, 1, 1, seed=0)[0], np.random.default_rng(0).standard_normal((4, 2)))
    for F, S in ((0, 1), (1, 0)):
        with pytest.raises(ValueError):
            path_draws(orc.K_SE_ARD, 2, F, S, 3)
    with pytest.raises(ValueError):
        spectral_draws(7, np.random.default_rng(0), 4, 2)


def test_paths_binding_checks_shapes_before_the_library():
    from ibo_b200 import _lib

    class Stub(object):
        d, N, _var = 3, 5, None
        handle = None

    om, ph, w, e = path_draws(orc.K_SE_ARD, 3, 8, 2, 5, seed=0)
    for bad in ((om[:, :2], ph, w, e), (om, ph[:7], w, e), (om, ph, w[:7], e), (om, ph, w, e[:, :1]), (om, ph, w, e[:4])):
        with pytest.raises(ValueError):
            _lib.Paths(Stub(), *bad)
