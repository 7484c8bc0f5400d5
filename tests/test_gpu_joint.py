"""GPU tests of the joint posterior (ibo_posterior_cov / ibo_posterior_sample and their Python surface) against the oracle's
posterior_joint and against the library's own marginal posterior."""
import numpy as np
import pytest

from oracle import ibo_oracle as orc
from joint_oracle import posterior_joint

pytestmark = pytest.mark.gpu

# magnitudes below 1: R's diagonal is 1 + noise whatever sf2 is, so sf2 > 1 + noise can make R itself indefinite
KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}
# (kind, N, M): every kind, N = 1 and 50 (one row-block: mu from the fused small-model kernel), 129 (two row-blocks with
# padding) and 1000; M from 1 to 2500 (across the 2048 boundary between the latency and throughput shapes of the scoring path)
CASES = [
    (orc.K_SE_ARD, 1, 7), (orc.K_SE_ISO, 50, 128), (orc.K_MATERN3, 129, 129), (orc.K_MATERN5, 1000, 300),
    (orc.K_MATERN5_ARD, 129, 1), (orc.K_SE_ARD, 1000, 2500), (orc.K_MATERN3, 50, 2500), (orc.K_SE_ISO, 1, 300),
    (orc.K_MATERN5_ARD, 1000, 129), (orc.K_MATERN5, 50, 7),
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


def _check_consistency(m, Xs, mu, cov, noise):
    """exactly symmetric; mu = ibo_posterior_batch(FP64) bit for bit; diag(cov) = sigma^2 where sigma^2 is not clipped"""
    L = _lib()
    assert np.array_equal(cov, cov.T)
    mu_b, s2_b = m.posterior(Xs, L.FLAG_FP64)
    assert np.array_equal(mu, mu_b)
    free = (s2_b > 10e-8) & (s2_b < 10)
    assert np.all(np.abs(np.diag(cov)[free] - s2_b[free]) <= 1e-12)


def _check_cov(cov, S_o, noise):
    err = np.max(np.abs(cov - S_o))
    assert err <= 1e-10 * (1 + noise), "max |dSigma| = %.3e" % err


@pytest.mark.parametrize("kind,N,M", CASES)
def test_covariance_matches_oracle(kind, N, M):
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs = _data(N, M, d, 10 * N + M + kind)
    hyper = KINDS[kind]
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise)
    m = L.Model(kind, hyper, X, Y, noise)
    mu, cov = m.posterior_cov(Xs)
    mu_o, S_o = posterior_joint(o, Xs)
    _check_cov(cov, S_o, noise)
    assert np.max(np.abs(mu - mu_o) / np.maximum(np.abs(mu_o), 1e-3)) <= 1e-10
    _check_consistency(m, Xs, mu, cov, noise)
    m.close()


def test_rbf_prior_mean():
    L = _lib()
    d, noise = 2, 0.1
    X, Y, Xs = _data(200, 300, d, 4)
    rs = np.random.RandomState(9)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, noise, prior=prior)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, noise, prior=prior)
    mu, cov = m.posterior_cov(Xs)
    mu_o, S_o = posterior_joint(o, Xs)
    _check_cov(cov, S_o, noise)
    assert np.max(np.abs(mu - mu_o) / np.maximum(np.abs(mu_o), 1e-3)) <= 1e-10
    _check_consistency(m, Xs, mu, cov, noise)


def test_pref_gp_with_variance_model():
    """Sigma from the variance factor (augX, augL) as sigma^2 is, mu from the main model"""
    from ibo_b200.gaussianprocess import PrefGaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    L = _lib()
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
    mu0, cov0 = gp.posterior_cov(q)
    P = rs.rand(3, d) * 10
    gp.addObservationPoint(P)
    augX = np.r_[X, P]
    pad = np.zeros((N + 3, N + 3)); pad[:N, :N] = Cinv
    o.augL = np.linalg.cholesky(orc.build_R(o.kernel, augX, 0.1) + pad); o.augX = augX
    mu, cov = gp.posterior_cov(q)
    mu_o, S_o = posterior_joint(o, q)
    _check_cov(cov, S_o, 0.1)
    assert np.array_equal(mu, mu0)
    assert np.max(np.abs(mu - mu_o) / np.maximum(np.abs(mu_o), 1e-3)) <= 1e-10
    _check_consistency(gp.model, q, mu, cov, 0.1)
    assert not np.array_equal(cov, cov0)


def test_model_from_inverse():
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs = _data(150, 200, d, 6)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4, .5], d), X, Y, noise)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, noise, invR=o.invR(), sf2=1.0)
    mu, cov = m.posterior_cov(Xs)
    mu_o, S_o = posterior_joint(o, Xs)
    _check_cov(cov, S_o, noise)
    _check_consistency(m, Xs, mu, cov, noise)


def test_appended_model_equals_rebuilt_model():
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs = _data(300, 400, d, 7)
    m = L.Model(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], X[:250], Y[:250], noise)
    m.append(X[250:], Y[250:])
    r = L.Model(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], X, Y, noise)
    mu_a, cov_a = m.posterior_cov(Xs)
    mu_r, cov_r = r.posterior_cov(Xs)
    _check_cov(cov_a, cov_r, noise)
    assert np.max(np.abs(mu_a - mu_r) / np.maximum(np.abs(mu_r), 1e-3)) <= 1e-10
    o = orc.GPOracle(orc.KernelSpec(orc.K_MATERN5_ARD, KINDS[orc.K_MATERN5_ARD], d), X, Y, noise)
    _check_cov(cov_a, posterior_joint(o, Xs)[1], noise)
    _check_consistency(m, Xs, mu_a, cov_a, noise)


@pytest.mark.parametrize("N,M,S,jitter", [(50, 300, 5, 0.0), (1000, 700, 130, 1e-6), (129, 1, 3, 0.0)])
def test_samples_match_oracle_factor(N, M, S, jitter):
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs = _data(N, M, d, 11 + N)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4, .5], d), X, Y, noise)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, noise)
    Z = np.random.default_rng(N).standard_normal((M, S))
    F, am = m.posterior_sample(Xs, Z, jitter)
    mu, _ = m.posterior_cov(Xs)
    _, S_o = posterior_joint(o, Xs)
    F_o = mu[:, None] + np.linalg.cholesky(S_o + jitter * np.eye(M)).dot(Z)
    assert np.max(np.abs(F - F_o)) <= 1e-9
    assert np.array_equal(am, np.argmax(F, axis=0))
    F2, am2 = m.posterior_sample(Xs, Z, jitter, want_F=False)
    assert F2 is None and np.array_equal(am2, am)


def test_argmax_ties_go_to_the_lowest_index():
    """candidates far from the data and from each other: mu = 0 and Sigma = (1 + noise) I exactly, so equal rows of Z give
    equal rows of F; rows 3 and 7 hold every column's maximum and row 3 must win"""
    L = _lib()
    X, Y, _ = _data(40, 1, 2, 12)
    Xs = np.array([[100.0 * (i + 1), -50.0] for i in range(10)])
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1)
    Z = np.random.default_rng(3).standard_normal((10, 16))
    Z[3] = Z[7] = Z.max(axis=0) + 1.0
    F, am = m.posterior_sample(Xs, Z)
    assert np.array_equal(F[3], F[7])
    assert np.array_equal(am, np.argmax(F, axis=0)) and np.all(am == 3)


def test_sample_posterior_is_reproducible_and_uses_the_seeded_generator():
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    X, Y, Xs = _data(80, 200, 3, 13)
    gp = GaussianProcess(GaussianKernel_ard([.3, .4, .5]), X, Y, noise=0.1)
    F1 = gp.sample_posterior(Xs, n_samples=7, seed=42)
    F2 = gp.sample_posterior(Xs, n_samples=7, seed=42)
    assert F1.shape == (200, 7) and np.array_equal(F1, F2)
    Z = np.random.default_rng(42).standard_normal((200, 7))
    assert np.array_equal(F1, gp.model.posterior_sample(Xs, Z)[0])
    assert not np.array_equal(F1, gp.sample_posterior(Xs, n_samples=7, seed=43))


def test_empirical_covariance_of_many_draws():
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    X, Y, _ = _data(30, 1, 2, 14)
    Xs = np.random.RandomState(15).rand(6, 2)
    gp = GaussianProcess(GaussianKernel_ard([.3, .4]), X, Y, noise=0.1)
    mu, cov = gp.posterior_cov(Xs)
    n = 20000
    F = gp.sample_posterior(Xs, n_samples=n, seed=7)
    D = F - mu[:, None]
    C = D.dot(D.T) / n
    se = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / n)
    assert np.all(np.abs(C - cov) <= 6 * se)
    assert np.all(np.abs(F.mean(axis=1) - mu) <= 6 * np.sqrt(np.diag(cov) / n))


def test_indefinite_covariance_reports_the_pivot():
    """Matern-3/2 with sf2 = 4: two nearly coincident candidates far from the data have the Sigma block [[1.1, 4], [4, 1.1]]"""
    L = _lib()
    d = 2
    X = np.array([[3.0 * i, 0.0] for i in range(6)])
    Y = np.arange(6.0)
    hyper = [0.3, 2.0]
    m = L.Model(orc.K_MATERN3, hyper, X, Y, 0.1)
    Xs = np.array([[100., 100.], [100., 100. + 1e-9], [50., 50.], [70., 20.]])
    _, cov = m.posterior_cov(Xs)
    assert abs(cov[0, 1] - 4.0) < 1e-6 and abs(cov[0, 0] - 1.1) < 1e-12
    Z = np.random.default_rng(0).standard_normal((4, 3))
    with pytest.raises(L.NotPositiveDefinite) as ei:
        m.posterior_sample(Xs, Z)
    assert ei.value.pivot == 2
    F, am = m.posterior_sample(Xs, Z, jitter=10.0)
    o = orc.GPOracle(orc.KernelSpec(orc.K_MATERN3, hyper, d), X, Y, 0.1)
    mu, S_o = posterior_joint(o, Xs)
    assert np.max(np.abs(F - (mu[:, None] + np.linalg.cholesky(S_o + 10 * np.eye(4)).dot(Z)))) <= 1e-9


def test_thompson_batch():
    from ibo_b200.acquisition import thompsonBatch
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard
    X, Y, _ = _data(100, 1, 3, 16)
    gp = GaussianProcess(GaussianKernel_ard([.3, .4, .5]), X, Y, noise=0.1)
    C = np.random.RandomState(17).rand(500, 3)
    pts, idx = thompsonBatch(gp, [[0., 1.]] * 3, 8, candidates=C, seed=11)
    _, am = gp.model.posterior_sample(C, np.random.default_rng(11).standard_normal((500, 8)), want_F=False)
    assert np.array_equal(idx, am) and np.array_equal(pts, C[am])
    bounds = [[0., 1.], [-2., 2.], [5., 6.]]
    pts, idx = thompsonBatch(gp, bounds, 4, samples=300, seed=3)
    assert pts.shape == (4, 3) and idx.shape == (4,)
    assert np.all(pts >= np.array(bounds)[:, 0]) and np.all(pts <= np.array(bounds)[:, 1])
    from ibo_b200.utils.latinhypercube import lhcSample
    assert np.array_equal(pts, np.array(lhcSample(bounds, 300, seed=3))[idx])


def test_thompson_batch_picks_a_dominant_candidate():
    from ibo_b200.acquisition import thompsonBatch
    from ibo_b200.gaussianprocess import GaussianProcess
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_iso
    rs = np.random.RandomState(18)
    X = rs.rand(40, 2) * 10
    Y = np.zeros(40)
    Y[17] = 100.0
    gp = GaussianProcess(GaussianKernel_iso([0.2]), X, Y, noise=0.1)
    R = rs.rand(600, 2) * 10
    R = R[np.linalg.norm(R - X[17], axis=1) > 1.5]          # nothing near the dominant point but the point itself
    C = np.r_[R[:300], X[17:18], R[300:400]]
    mu, s2 = gp.posteriors(C)
    others = np.delete(np.arange(len(C)), 300)
    assert mu[300] - np.max(mu[others] + 10 * np.sqrt(s2[others])) > 10 * np.sqrt(s2[300])
    pts, idx = thompsonBatch(gp, [[0., 10.]] * 2, 16, candidates=C, seed=5, jitter=1e-9)
    assert np.all(idx == 300) and np.array_equal(pts, np.repeat(X[17:18], 16, axis=0))
