"""CPU checks of the longdouble reference of the hyperparameter and preference paths (tests/hyper_oracle.py): it agrees with the
FP64 oracle where FP64 is accurate, reproduces the reference's known answers, its gradient is the derivative of its value, and
its preference fixed point is a root of the gradient to longdouble rounding."""
import numpy as np
import pytest

import hyper_oracle as ho
from oracle import ibo_oracle as orc

HX = np.array([[.5, .1, .3], [.9, 1.2, .1], [.55, .234, .1], [.234, .547, .675]])
HY = np.array([.5, 1., .5, 2.])

KINDS = [
    (orc.K_SE_ARD, [.4, .6, .9, 1.3], False),          # with magnitude
    (orc.K_SE_ARD, [1e-5, 1e5, .7], False),            # clipped to [1e-4, 1e4]
    (orc.K_SE_ISO, [.7], False),
    (orc.K_MATERN3, [.8, 1.2], False),
    (orc.K_MATERN3, [.8, 1.2], True),
    (orc.K_MATERN5, [.8, 1.2], False),
    (orc.K_MATERN5_ARD, [.5, .6, .7, 1.1], False),
]


def _data(N, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    return X, np.sin(2 * X).sum(axis=1) + 0.1 * rs.randn(N)


@pytest.mark.parametrize("kind,hyper,exact", KINDS)
def test_matrices_and_likelihood_agree_with_the_fp64_oracle(kind, hyper, exact):
    X, Y = _data(40, 3, kind)
    spec = orc.KernelSpec(kind, hyper, 3)
    assert ho.rel(ho.cov_matrix(spec, X), orc.cov_matrix(spec, X)) <= 1e-14
    nh = ho.n_hyper(spec)
    for h in range(nh):
        assert ho.rel(ho.kernel_derivative(spec, X, h, exact), orc.kernel_derivative(spec, X, h, exact)) <= 1e-13
    nl, g, sc, _ = ho.marginal_likelihood(spec, X, Y, 0.1, exact)
    nl_o, g_o = orc.marginal_likelihood(spec, X, Y, nh, noise=0.1, exact_matern3=exact)
    assert abs(float(nl) - nl_o) <= 1e-12 * abs(nl_o)
    assert np.all(np.abs(g.astype(float) - g_o) <= 1e-12 * np.maximum(sc.astype(float), 1e-300))
    assert ho.marginal_likelihood(spec, X, Y, 0.1, exact, gradient=False) == nl


def test_reference_known_answers():
    """ego/unittest_GP.py:204-272, as tests/test_gpu_hyper.py checks them on the device"""
    cases = [(orc.K_SE_ARD, [2., 2., .1], 5.8404, [0.0039, 0.0302, -0.1733], 5e-5),
             (orc.K_SE_ARD, [1.5, 1.5, 1.5, 1.1], 7.514, [11.4659, -10.0714], 5e-4),    # SV-iso: ARD with equal length scales
             (orc.K_MATERN3, [1.5, 1.1], 5.1827, [1.6947897766, -2.9350], 5e-5),
             (orc.K_MATERN5, [1.5, 1.1], 5.6652, [4.4782, -4.8737], 5e-5)]
    for kind, hyper, nl_ref, g_ref, tol in cases:
        spec = orc.KernelSpec(kind, hyper, 3)
        nl, g, _, _ = ho.marginal_likelihood(spec, HX, HY, 0.0)
        if len(hyper) == 4:                     # d / d log theta of SV-iso: the sum of the per-dimension derivatives
            g = np.r_[np.sum(g[:3]), g[3]]
        assert abs(float(nl) - nl_ref) < tol
        assert np.max(np.abs(g.astype(float) - g_ref)) < 5e-5
    spec = orc.KernelSpec(orc.K_MATERN3, [1.5, 1.1], 3)
    assert abs(float(ho.marginal_likelihood(spec, HX, HY, 0.0)[1][0]) - 1.6947897766) < 1e-9


@pytest.mark.parametrize("kind,hyper,exact", [k for k in KINDS if k[0] != orc.K_MATERN3 or k[2]])
def test_gradient_is_the_derivative_of_the_value(kind, hyper, exact):
    """central differences in log hyperparameters (kinds whose derivative is exact; Matern-3/2 with exact_matern3 only); the
    clipped SE-ARD length scales have no effect, so their derivative is the formula's, not the value's, and is skipped"""
    X, Y = _data(30, 3, 7)
    spec = orc.KernelSpec(kind, hyper, 3)
    _, g, sc, _ = ho.marginal_likelihood(spec, X, Y, 1e-2, exact)
    clipped = [h for h in range(3) if kind == orc.K_SE_ARD and not 1e-4 <= hyper[h] <= 1e4]
    for h in range(ho.n_hyper(spec)):
        if h in clipped:
            continue
        e = np.zeros(len(hyper))
        e[h] = 1e-4
        fp = ho.marginal_likelihood(orc.KernelSpec(kind, np.exp(np.log(hyper) + e), 3), X, Y, 1e-2, gradient=False)
        fm = ho.marginal_likelihood(orc.KernelSpec(kind, np.exp(np.log(hyper) - e), 3), X, Y, 1e-2, gradient=False)
        assert abs(float((fp - fm) / 2e-4 - g[h])) <= 1e-7 * max(1.0, float(sc[h])), (h, g[h])


def _pref_problem(npts, nprefs, d, seed, theta):
    """the small problem of tests/test_gpu_laplace.py"""
    rs = np.random.RandomState(seed)
    X = rs.rand(npts, d)
    f = np.sin(3 * X).sum(axis=1)
    prefinds = []
    for _ in range(nprefs):
        a, b = rs.choice(npts, 2, replace=False)
        v, u = (a, b) if f[a] > f[b] else (b, a)
        prefinds.append((int(v), int(u), int(rs.rand() < 0.2)))
    spec = orc.KernelSpec(orc.K_SE_ARD, theta, d)
    winners = set(v for v, _, _ in prefinds)
    return spec, X, prefinds, np.array([.5 if i in winners else -.5 for i in range(npts)])


def test_preference_functional_and_fixed_point():
    spec, X, prefinds, start = _pref_problem(14, 12, 2, 3, [0.4, 0.5])
    R = orc.build_R(spec, X, 0.1)
    L64 = np.linalg.cholesky(R)
    Lld = ho.cholesky(ho.bo.build_R(spec, X, 0.1))
    rs = np.random.RandomState(0)
    for y in (start, rs.randn(14)):
        assert abs(float(ho.pref_S(y, prefinds, Lld)) - orc.pref_S(y, prefinds, L64)) <= 1e-12 * abs(orc.pref_S(y, prefinds, L64))
        assert np.max(np.abs(ho.pref_grad(y, prefinds, Lld).astype(float) - orc.pref_S_grad(y, prefinds, L64))) <= 1e-12
    y64 = ho.pref_fit_f64(start, prefinds, L64)
    ys, res = ho.pref_fixed_point(y64, prefinds, Lld)
    assert res <= 1e-15
    assert np.max(np.abs(ys.astype(float) - y64)) <= 1e-12
    assert np.max(np.abs(ys.astype(float) - orc.pref_fit_bfgs(start, prefinds, L64))) <= 2e-4     # BFGS's gtol 1e-5
    # the far start (every loser 10 above its winner) reaches the same point
    far = np.zeros(14)
    for v, u, _ in prefinds:
        far[u] = far[v] + 10.0 if far[u] == 0 else far[u]
    assert np.max(np.abs(ho.pref_fit_f64(far, prefinds, L64) - y64)) <= 1e-10
