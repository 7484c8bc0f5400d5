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
