"""CPU tests of the extended-precision build reference (tests/build_oracle.py) that tests/test_gpu_build.py measures the device
against: it must itself be accurate far beyond FP64, agree with LAPACK to what LAPACK's conditioning allows, and be right on a
case worked by hand."""
import math

import numpy as np
import pytest
from scipy.linalg import lapack

import build_oracle as bo
from oracle import ibo_oracle as orc

LD = np.longdouble
EPS = np.finfo(float).eps


def _spd(n, cond, seed):
    """symmetric positive definite FP64 matrix with eigenvalues log-spaced over [1 / cond, 1]"""
    rs = np.random.RandomState(seed)
    Q, _ = np.linalg.qr(rs.randn(n, n))
    A = (Q * np.logspace(0, -np.log10(cond), n)).dot(Q.T)
    return 0.5 * (A + A.T)


def test_longdouble_is_extended_precision():
    assert np.finfo(LD).eps <= 1.1e-19


@pytest.mark.parametrize("n,cond", [(50, 1e2), (200, 1e6), (200, 1e10), (130, 1e10)])
def test_factor_and_inverse_are_accurate_at_the_longdouble_level(n, cond):
    A = _spd(n, cond, n)
    L = bo.cholesky(A)
    assert np.array_equal(np.triu(L, 1), np.zeros((n, n), dtype=LD))
    assert bo.rel(L @ L.T, A) <= 1e-17                                  # backward error: longdouble, not FP64
    W = bo.tri_inv(L)
    assert bo.rel(W @ L, np.eye(n)) <= 1e-17 * math.sqrt(cond)        # ||W L - I|| ~ cond(L) eps_ld
    # against LAPACK: each FP64 result is within cond * eps_64 of it
    Lp = np.tril(lapack.dpotrf(A, lower=1)[0])
    Wp = lapack.dtrtri(Lp, lower=1)[0]
    eL, eW = bo.rel(Lp, L), bo.rel(Wp, W)
    assert eL <= cond * EPS and eW <= cond * EPS
    # and LAPACK is not more accurate than FP64 allows: the reference is no mere copy of it
    assert eL >= EPS / 64


def test_three_by_three_by_hand():
    L0 = np.array([[2., 0, 0], [1, 3, 0], [-1, 1, 2]])
    A = L0.dot(L0.T)                                                    # [[4, 2, -2], [2, 10, 2], [-2, 2, 6]]
    assert np.array_equal(A, [[4, 2, -2], [2, 10, 2], [-2, 2, 6]])
    L = bo.cholesky(A)
    assert np.array_equal(L, L0.astype(LD))
    W = bo.tri_inv(L)
    want = np.array([[LD(1) / 2, 0, 0], [LD(-1) / 6, LD(1) / 3, 0], [LD(1) / 3, LD(-1) / 6, LD(1) / 2]], dtype=LD)
    assert np.max(np.abs(W - want)) <= 2 * np.finfo(LD).eps
    assert np.array_equal(bo.forward_solve(L, [2., 1, 0]), np.array([1, 0, LD(1) / 2], dtype=LD))


def test_blocking_does_not_change_the_factor_beyond_rounding():
    A = _spd(150, 1e4, 3)
    a, b = bo.cholesky(A, nb=64), bo.cholesky(A, nb=150)
    assert bo.rel(a, b) <= 1e-17 * 1e2


@pytest.mark.parametrize("p", [1, 64, 65, 97])
def test_first_failing_pivot_is_reported(p):
    """a near-duplicate pair (p - 2, p - 1) of a kernel whose variance exceeds the diagonal: the 2 x 2 minor is indefinite"""
    rs = np.random.RandomState(p)
    X = np.array([[a, b] for a in range(10) for b in range(10)], dtype=float)[:100]
    kern = orc.KernelSpec(orc.K_MATERN3, [0.01, 2.0], 2)
    if p > 1:
        X[p - 1] = X[p - 2] + 1e-9
        A = bo.build_R(kern, X, 0.1)
    else:
        A = bo.build_R(kern, X, 0.1)
        A[0, 0] = -rs.rand()
    with pytest.raises(np.linalg.LinAlgError) as ei:
        bo.cholesky(A)
    assert ei.value.pivot == p


def test_posterior_by_hand_and_against_the_fp64_oracle():
    kern = orc.KernelSpec(orc.K_SE_ISO, [0.5], 1)
    # one observation: mu = k y / (1 + nu), sigma^2 = 1 + nu - k^2 / (1 + nu)
    mu, s2 = bo.posterior(kern, [[0.0]], [3.0], 0.1, [[0.5]])
    k = np.exp(LD(-0.5) * (LD(0.5) / LD(0.5)) ** 2)
    assert abs(mu[0] - 3 * k / LD(1.1)) <= 4 * np.finfo(LD).eps and abs(s2[0] - (LD(1.1) - k * k / LD(1.1))) <= 4 * np.finfo(LD).eps
    # a well-conditioned model, with and without the prior: the FP64 oracle agrees to 1e-12
    rs = np.random.RandomState(8)
    for kind, hyper in ((orc.K_SE_ARD, [0.3, 0.4, 0.5]), (orc.K_MATERN3, [0.4, 0.9]), (orc.K_MATERN5, [0.5, 0.9])):
        kern = orc.KernelSpec(kind, hyper, 3)
        X, Xs = rs.rand(150, 3), rs.rand(40, 3)
        Y = np.sin(3 * X).sum(axis=1)
        pr = orc.PriorSpec(rs.rand(4, 3), rs.randn(4), 2.0, np.zeros(3), np.ones(3))
        for prior in (None, pr):
            o = orc.GPOracle(kern, X, Y, 0.1, prior=prior)
            mu_o, s2_o = o.posterior_batch(Xs, floor=-np.inf)
            mu, s2 = bo.posterior(kern, X, Y, 0.1, Xs, prior=prior)
            assert mu.dtype == LD and s2.dtype == LD
            assert np.max(np.abs(mu - mu_o)) <= 1e-12 and np.max(np.abs(s2 - s2_o)) <= 1e-12
        assert bo.rel(bo.build_R(kern, X, 0.1), o.R) <= 1e-15


# -- the candidate-side reference: joint posterior, gradients with respect to the candidate, reverse Cholesky, q-EI -----------------

CAND_KINDS = [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_MATERN3, [.5, .9]), (orc.K_MATERN5_ARD, [.3, .4, .5, .95])]


def _cand_problem(kind, hyper, seed, N=40, d=3, with_prior=False, with_aug=False, noise=0.1):
    """(spec, X, Y, prior, aug, FP64 GPOracle with the same prior / variance factor) on [0, 1]^d"""
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    spec = orc.KernelSpec(kind, hyper, d)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d)) if with_prior else None
    o = orc.GPOracle(spec, X, Y, noise, prior=prior)
    aug = None
    if with_aug:
        augX = np.r_[X, rs.rand(3, d)]
        A = rs.randn(N, N) * 0.05
        pad = np.zeros((N + 3, N + 3))
        pad[:N, :N] = np.linalg.inv(np.eye(N) * 5 + A.dot(A.T))
        aug = (augX, bo.build_R(spec, augX, noise) + pad)
        o.augX, o.augL = augX, np.linalg.cholesky(orc.build_R(spec, augX, noise) + pad)
    return spec, X, Y, prior, aug, o, rs


def _fd(f, x, h):
    """central differences of the longdouble function f at the longdouble point x, one coordinate at a time -> [..., x.size]"""
    x = np.asarray(x, dtype=LD)
    out = []
    for t in range(x.size):
        e = np.zeros(x.size, dtype=LD)
        e[t] = h
        e = e.reshape(x.shape)
        out.append((f(x + e) - f(x - e)) / (2 * h))
    return np.stack(out, axis=-1)


def _rel_max(a, b):
    a, b = np.asarray(a, dtype=LD), np.asarray(b, dtype=LD)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize("kind,hyper", CAND_KINDS)
@pytest.mark.parametrize("extra", ["", "prior", "aug"])
def test_posterior_gradient_agrees_with_longdouble_differences(kind, hyper, extra):
    spec, X, Y, prior, aug, _, rs = _cand_problem(kind, hyper, 20 + kind, with_prior=extra == "prior", with_aug=extra == "aug")
    Xs = rs.rand(4, 3).astype(LD)
    model = bo._Model(spec, X, Y, 0.1, prior, aug)
    mu, s2, dmu, ds2 = bo.posterior_grad(spec, X, Y, 0.1, Xs, model=model)
    h = LD(1e-7)
    for j in range(len(Xs)):
        f = lambda x: np.array(bo.posterior_grad(spec, X, Y, 0.1, x[None], model=model)[:2])[:, 0]
        g = _fd(f, Xs[j], h)
        assert _rel_max(dmu[j], g[0]) <= 1e-10 and _rel_max(ds2[j], g[1]) <= 1e-10, (j, dmu[j], g[0], ds2[j], g[1])


def test_chol_rev_agrees_with_longdouble_differences():
    """f(Sigma) = <Lbar, chol(Sigma)>: df / dSigma_kl over the symmetric perturbation of (k, l) and (l, k) is 2 Gbar_kl off the
    diagonal and Gbar_kk on it"""
    A = _spd(6, 10.0, 4)
    Lbar = np.tril(np.random.RandomState(5).randn(6, 6)).astype(LD)
    G = bo.chol_rev(bo.cholesky(A), Lbar)
    assert np.array_equal(G, G.T)
    h = LD(1e-7)
    for k in range(6):
        for l in range(k + 1):
            E = np.zeros((6, 6), dtype=LD)
            E[k, l] = E[l, k] = h
            fd = (np.sum(Lbar * bo.cholesky(A + E)) - np.sum(Lbar * bo.cholesky(A - E))) / (2 * h)
            want = G[k, l] * (1 if k == l else 2)
            assert abs(fd - want) <= 1e-10 * np.max(np.abs(G)), (k, l, fd, want)


@pytest.mark.parametrize("extra", ["", "prior", "aug"])
def test_qei_gradient_agrees_with_longdouble_differences(extra):
    spec, X, Y, prior, aug, _, rs = _cand_problem(orc.K_MATERN5_ARD, [.3, .4, .5, .95], 31, with_prior=extra == "prior",
                                                  with_aug=extra == "aug")
    model = bo._Model(spec, X, Y, 0.1, prior, aug)
    Z = np.random.default_rng(2).standard_normal((3, 64))
    ymax, xi = Y.max() - 0.3, 0.01
    Xb = rs.rand(12, 3, 3).astype(LD)
    v, G, gap, imp = bo.qei(spec, X, Y, 0.1, Xb, Z, ymax, xi, 1e-8, model=model)
    keep = [b for b in range(len(Xb)) if min(gap[b], imp[b]) > 1e-4 and v[b] > 0]
    assert len(keep) >= 3
    for b in keep[:3]:
        f = lambda x: bo.qei(spec, X, Y, 0.1, x[None], Z, ymax, xi, 1e-8, model=model)[0][0]
        g = _fd(f, Xb[b], LD(1e-7))
        assert _rel_max(G[b].reshape(-1), g) <= 1e-9, (b, G[b], g)


@pytest.mark.parametrize("kind,hyper", CAND_KINDS)
@pytest.mark.parametrize("extra", ["", "prior", "aug"])
def test_candidate_paths_agree_with_the_fp64_oracles(kind, hyper, extra):
    """noise 0.1, d = 3: the longdouble joint posterior, gradients, scores' gradients and q-EI agree with joint_oracle, grad_oracle
    and qei_oracle to about 1e-12"""
    import grad_oracle as go
    import joint_oracle as jo
    import qei_oracle as qo
    spec, X, Y, prior, aug, o, rs = _cand_problem(kind, hyper, 40 + kind, N=150, with_prior=extra == "prior", with_aug=extra == "aug")
    Xs = rs.rand(30, 3)
    Xs[:2] = X[:2]
    model = bo._Model(spec, X, Y, 0.1, prior, aug)
    close = lambda a, b: np.max(np.abs(np.asarray(a, dtype=float) - b)) <= 1e-12 * max(1.0, np.max(np.abs(b)))
    mu, Sig = bo.posterior_joint(spec, X, Y, 0.1, Xs, model=model)
    mu_o, Sig_o = jo.posterior_joint(o, Xs)
    assert close(mu, mu_o) and close(Sig, Sig_o)
    mu, s2, dmu, ds2 = bo.posterior_grad(spec, X, Y, 0.1, Xs, model=model)
    _, _, dmu_o, ds2_o = go.posterior_grad(o, Xs, "cpp")
    assert close(dmu, dmu_o) and close(ds2, ds2_o) and close(s2, np.diag(Sig_o))
    Z = np.random.default_rng(3).standard_normal((4, 128))
    Xb = rs.rand(5, 4, 3)
    v, G, _, _ = bo.qei(spec, X, Y, 0.1, Xb, Z, Y.max() - 0.3, 0.01, 0.0, model=model)
    v_o, G_o = qo.qei(o, Xb, Z, Y.max() - 0.3, 0.01)
    assert np.any(v_o > 0) and close(v, v_o) and close(G, G_o)


def test_joint_covariance_is_symmetric_and_bounded_below_by_the_noise():
    """Sigma = K** + noise I - k*^T inv(R) k*, and the posterior covariance of f is positive semi-definite; near-duplicate and
    on-data candidates make it singular up to the noise"""
    for noise in (0.1, 1e-4):
        spec, X, Y, _, _, _, rs = _cand_problem(orc.K_SE_ARD, [.6, .8, 1.0], 50, N=120, noise=noise)
        Xs = rs.rand(40, 3)
        Xs[:5] = X[:5]
        Xs[5:10] = Xs[10:15] + 1e-5
        _, Sig = bo.posterior_joint(spec, X, Y, noise, Xs)
        assert np.array_equal(Sig, Sig.T)
        ev = np.linalg.eigvalsh(np.asarray(Sig, dtype=float))
        assert np.min(ev) >= noise - 100 * EPS and np.min(ev) <= noise * 1.01
