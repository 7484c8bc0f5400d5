"""CPU tests of the joint posterior: the oracle's joint form against its marginal form, the argument checks of the two
C entry points (no device touched) and the Python surface on a GP without data."""
import ctypes

import numpy as np
import pytest

from ibo_b200 import _lib
from oracle import ibo_oracle as orc
from joint_oracle import posterior_joint


def _oracle(kind, hyper, N, d, seed, noise=0.1, prior=None):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    return orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior), rs


@pytest.mark.parametrize("kind,hyper", [(orc.K_SE_ARD, [.3, .4, .5]), (orc.K_SE_ISO, [.3]), (orc.K_MATERN3, [.5, 1.]),
                                        (orc.K_MATERN5, [.5, 1.]), (orc.K_MATERN5_ARD, [.3, .4, .5, 1.])])
def test_oracle_joint_agrees_with_marginals(kind, hyper):
    o, rs = _oracle(kind, hyper, 40, 3, 1)
    Xs = rs.rand(25, 3)
    Xs[:3] = o.X[:3]
    mu, S = posterior_joint(o, Xs)
    mu_b, s2_b = o.posterior_batch(Xs, floor=-np.inf)
    assert np.array_equal(mu, mu_b)
    assert np.array_equal(np.diag(S), s2_b)
    assert np.array_equal(S, S.T)


def test_oracle_joint_prior_mean_and_variance_factor():
    d = 2
    prior = orc.PriorSpec(np.random.RandomState(5).rand(3, d), [0.5, -0.2, 0.3], 3.0, np.zeros(d), np.ones(d))
    o, rs = _oracle(orc.K_SE_ARD, [.3, .4], 30, d, 2, prior=prior)
    P = rs.rand(4, d)
    o.augX = np.r_[o.X, P]
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, o.augX, o.noise))
    Xs = rs.rand(20, d)
    mu, S = posterior_joint(o, Xs)
    mu_b, s2_b = o.posterior_batch(Xs, floor=-np.inf)
    assert np.array_equal(mu, mu_b) and np.array_equal(np.diag(S), s2_b)


@pytest.mark.parametrize("noise", [0.1, 1e-3])
def test_oracle_joint_is_symmetric_with_eigenvalues_above_noise(noise):
    """R = K + noise I for a unit-magnitude kernel, so Sigma = (K** - K*^T inv(R) K*) + noise I >= noise I"""
    o, rs = _oracle(orc.K_SE_ARD, [.2, .3, .4], 60, 3, 3, noise=noise)
    Xs = rs.rand(80, 3)
    _, S = posterior_joint(o, Xs)
    assert np.array_equal(S, S.T)
    assert np.linalg.eigvalsh(S).min() >= noise - 1e-12


def test_bad_arguments_are_rejected_without_touching_a_gpu():
    L = _lib.lib()
    fake = ctypes.create_string_buffer(1 << 16)          # never dereferenced: every scalar check comes first
    h = ctypes.cast(fake, ctypes.c_void_p)
    x = np.zeros((3, 2)); z = np.zeros((3, 4)); mu = np.zeros(3); cov = np.zeros((3, 3)); F = np.zeros((3, 4))
    am = np.zeros(4, dtype=np.int64)
    pl = am.ctypes.data_as(ctypes.POINTER(ctypes.c_long))
    info = ctypes.c_int(7)
    d = _lib.dptr
    assert L.ibo_posterior_cov(None, d(x), 3, d(mu), d(cov)) == _lib.E_BADARG
    assert L.ibo_posterior_cov(h, None, 3, d(mu), d(cov)) == _lib.E_BADARG
    assert L.ibo_posterior_cov(h, d(x), 3, d(mu), None) == _lib.E_BADARG
    for M in (0, -1, 16385):
        assert L.ibo_posterior_cov(h, d(x), M, d(mu), d(cov)) == _lib.E_BADARG
        assert L.ibo_posterior_sample(h, d(x), M, d(z), 4, 0.0, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG
    assert L.ibo_posterior_sample(None, d(x), 3, d(z), 4, 0.0, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG
    assert info.value == 0
    assert L.ibo_posterior_sample(h, None, 3, d(z), 4, 0.0, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG
    assert L.ibo_posterior_sample(h, d(x), 3, None, 4, 0.0, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG
    for S in (0, -3):
        assert L.ibo_posterior_sample(h, d(x), 3, d(z), S, 0.0, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG
    for jitter in (-1e-12, float("nan"), -np.inf):
        assert L.ibo_posterior_sample(h, d(x), 3, d(z), 4, jitter, d(F), pl, ctypes.byref(info)) == _lib.E_BADARG


def test_gp_without_data_raises_value_error():
    from ibo_b200.acquisition import thompsonBatch
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    gp = GaussianProcess(GaussianKernel_ard([.3, .4]))
    X = np.random.RandomState(0).rand(5, 2)
    with pytest.raises(ValueError):
        gp.posterior_cov(X)
    with pytest.raises(ValueError):
        gp.sample_posterior(X, n_samples=3, seed=1)
    with pytest.raises(ValueError):
        thompsonBatch(gp, [[0., 1.]] * 2, 4, candidates=X, seed=1)
