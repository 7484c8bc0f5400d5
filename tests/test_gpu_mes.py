"""GPU tests of max-value entropy search (ibo_mes, ibo_max_value_gumbel and their Python surface): the device's h and h' against
50-digit mpmath over g in [-1e4, 37], MES values and gradients against the oracle (tests/mes_oracle.py), the INT8 path of wide
sets, exact identities, the Gumbel fit's quantiles, the shared candidate workspace, and maximizeMES."""
import ctypes
import math

import numpy as np
import pytest
from scipy.stats import norm

from oracle import ibo_oracle as orc
import mes_oracle as mo

pytestmark = pytest.mark.gpu

KINDS = {
    orc.K_SE_ARD: [.3, .4, .5],
    orc.K_SE_ISO: [.3],
    orc.K_MATERN3: [.5, .9],
    orc.K_MATERN5: [.4, .8],
    orc.K_MATERN5_ARD: [.3, .4, .5, .95],
}
# (kind, N, M, K): every kind, N from 1 to 1000, M from 1 to 2500, K in {1, 7, 100, 1024}
CASES = [
    (orc.K_SE_ARD, 1, 7, 1), (orc.K_SE_ISO, 50, 129, 7), (orc.K_MATERN3, 129, 129, 100), (orc.K_MATERN5, 1000, 7, 1024),
    (orc.K_MATERN5_ARD, 129, 1, 7), (orc.K_SE_ARD, 1000, 2500, 100), (orc.K_MATERN3, 50, 2500, 1024), (orc.K_SE_ISO, 1, 129, 1),
    (orc.K_MATERN5_ARD, 1000, 129, 100), (orc.K_MATERN5, 50, 1, 7),
]


def _lib():
    from ibo_b200 import _lib as L
    return L


def _data(N, M, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    Xs = rs.rand(M, d)
    Xs[: min(2, M, N)] = X[: min(2, M, N)]
    return X, Y, Xs, rs


def _ystar(Y, K, rs):
    return Y.max() + 0.05 + 0.5 * np.abs(rs.randn(K))


def _flags(mode):
    L = _lib()
    return L.FLAG_MODE_PY if mode == "py" else L.FLAG_MODE_CPP


def _check_values(v, v_o):
    """the repository's EI rule: 1e-10 relative, floor 1e-5"""
    assert np.all(np.abs(v - v_o) <= 1e-10 * np.maximum(np.abs(v_o), 1e-5)), np.max(np.abs(v - v_o) / np.maximum(np.abs(v_o), 1e-5))


def _check_grad(G, G_o):
    bound = 1e-9 * np.max(np.abs(G_o), axis=1, keepdims=True) + 1e-12
    assert np.all(np.abs(G - G_o) <= bound), np.max(np.abs(G - G_o) - bound)


def _h_at(y, mu, s2):
    """(h, h', g) at g = (y - mu) / sqrt(s2) computed at 50 digits from the doubles y, mu, s2"""
    with mo.mp.workdps(50):
        g = (mo.mp.mpf(float(y)) - mo.mp.mpf(float(mu))) / mo.mp.sqrt(mo.mp.mpf(float(s2)))
        Phi = mo.mp.ncdf(g)
        psi = mo.mp.npdf(g) / Phi
        h = g * psi / 2 - (mo.mp.log1p(-mo.mp.ncdf(-g)) if g > 0 else mo.mp.log(Phi))
        return h, -(psi / 2) * (1 + g * (g + psi)), float(g)


def _bound(g):
    return 1e-13 if g <= 8 else 16 * (1 + g * g) * 2.0 ** -53


@pytest.mark.parametrize("mode", ["py", "cpp"])
def test_h_and_its_derivatives_match_mpmath(mode):
    """K = 1, y* = mu_0 + s_0 g over g in [-1e4, 37]: values, d MES / d mu and d MES / d s against mpmath at the device's own
    doubles"""
    L = _lib()
    X, Y, Xs, _ = _data(50, 6, 3, 1)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1)
    fl = _flags(mode)
    mu, s2 = m.posterior(Xs, fl)
    mu_g, s2_g, dmu, ds2 = m.posterior_grad(Xs, fl)
    grid = np.r_[-np.logspace(4, -3, 40), 0.0, np.logspace(-3, math.log10(37), 40)]
    for g0 in grid:
        ys = np.array([mu[0] + math.sqrt(s2[0]) * g0])
        v = m.mes(Xs, ys, fl)[0]
        vg, dv, _, _ = m.mes(Xs, ys, fl, want_grad=True)
        for j in range(Xs.shape[0]):
            h, _, gf = _h_at(ys[0], mu[j], s2[j])
            assert abs(v[j] - float(h)) <= _bound(gf) * abs(float(h)), (gf, v[j], float(h))
            # the gradient path: mu and s of the FP64 kernels (ibo_posterior_grad's)
            _, dh, gg = _h_at(ys[0], mu_g[j], s2_g[j])
            with mo.mp.workdps(50):
                sg = mo.mp.sqrt(mo.mp.mpf(float(s2_g[j])))
                a = float(-dh / sg)
                b = float(-gg * dh / sg / (2 * sg))
            ref = a * dmu[j] + b * ds2[j]
            tol = _bound(gg) * (abs(a) * np.abs(dmu[j]) + abs(b) * np.abs(ds2[j]))
            assert np.all(np.abs(dv[j] - ref) <= 2 * tol + 1e-300), (gg, dv[j], ref)
    m.close()


@pytest.mark.parametrize("mode", ["py", "cpp"])
@pytest.mark.parametrize("kind,N,M,K", CASES)
def test_matches_oracle(kind, N, M, K, mode):
    L = _lib()
    d, noise = 3, 0.1
    X, Y, Xs, rs = _data(N, M, d, 10 * N + M + kind + K)
    hyper = KINDS[kind]
    o = orc.GPOracle(orc.KernelSpec(kind, hyper, d), X, Y, noise)
    m = L.Model(kind, hyper, X, Y, noise)
    fl = _flags(mode)
    ys = _ystar(Y, K, rs)
    v, _, best, bidx = m.mes(Xs, ys, fl)
    v_o, G_o = mo.mes(o, Xs, ys, mode)
    _check_values(v, v_o)
    assert bidx == int(np.argmax(v_o)) and best == v[bidx]
    vg, G, best_g, bidx_g = m.mes(Xs, ys, fl, want_grad=True)
    _check_values(vg, v_o)
    _check_grad(G, G_o)
    assert bidx_g == bidx and best_g == vg[bidx_g]
    m.close()


def test_prior_from_inverse_and_appended_models():
    L = _lib()
    d = 2
    X, Y, Xs, rs = _data(300, 200, d, 4)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d))
    ys = _ystar(Y, 9, rs)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1, prior=prior)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, prior=prior)
    v_o, G_o = mo.mes(o, Xs, ys)
    _check_values(m.mes(Xs, ys, L.FLAG_MODE_PY)[0], v_o)
    _check_grad(m.mes(Xs, ys, L.FLAG_MODE_PY, want_grad=True)[1], G_o)
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, [.3, .4], d), X, Y, 0.1)
    v_o, G_o = mo.mes(o, Xs, ys)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1, invR=o.invR(), sf2=1.0)
    _check_values(m.mes(Xs, ys, L.FLAG_MODE_PY)[0], v_o)
    _check_grad(m.mes(Xs, ys, L.FLAG_MODE_PY, want_grad=True)[1], G_o)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X[:250], Y[:250], 0.1)
    m.mes(Xs, ys, L.FLAG_MODE_PY, want_grad=True)           # a call before the append: nothing cached may survive it
    m.append(X[250:], Y[250:])
    _check_values(m.mes(Xs, ys, L.FLAG_MODE_PY)[0], v_o)
    _check_grad(m.mes(Xs, ys, L.FLAG_MODE_PY, want_grad=True)[1], G_o)


def test_pref_gp_with_variance_model():
    """sigma^2 and its gradient from the variance factor (augX, augL), mu from the main model"""
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
    Xs = rs.rand(300, d) * 10
    ys = _ystar(Y, 20, rs)
    v, G = gp.mes(Xs, ys, grad=True)
    v_o, G_o = mo.mes(o, Xs, ys)
    _check_values(v, v_o)
    _check_grad(G, G_o)
    assert np.array_equal(gp.mes(Xs, ys, int8=False), v)


def test_wide_sets_int8_path_and_guard():
    L = _lib()
    d = 3
    X, Y, _, rs = _data(1000, 1, d, 20)
    Xs = rs.rand(6000, d)
    ys = _ystar(Y, 50, rs)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1)
    v8, _, b8, i8 = m.mes(Xs, ys)
    v64, _, b64, i64 = m.mes(Xs, ys, L.FLAG_FP64)
    assert np.all(np.abs(v8 - v64) <= 1e-9 * np.maximum(np.abs(v64), 1e-5)) and i8 == i64
    # noise < 2^-10: candidates next to training points have sigma^2 under the guard and get the FP64 path's bits
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 1e-4)
    Xs[:300] = X[:300] + 1e-6
    v8, _, b8, i8 = m.mes(Xs, ys)
    assert m.last_guarded() > 0
    v64, _, b64, i64 = m.mes(Xs, ys, L.FLAG_FP64)
    guarded = m.posterior(Xs, L.FLAG_FP64)[1] < 2.0 ** -10
    assert guarded.sum() >= 300
    assert np.array_equal(v8[guarded], v64[guarded])
    assert np.all(np.abs(v8 - v64) <= 1e-9 * np.maximum(np.abs(v64), 1e-5)) and i8 == i64


def test_identities():
    L = _lib()
    d = 3
    X, Y, _, rs = _data(1000, 1, d, 30)
    Xs = rs.rand(70000, d)
    ys = _ystar(Y, 10, rs)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1)
    for fl in (L.FLAG_MODE_CPP, L.FLAG_MODE_PY):
        v, _, _, _ = m.mes(Xs, ys, fl)
        assert np.all(np.isfinite(v)) and np.all(v >= 0)
        v2 = m.mes(Xs, ys + 0.1, fl)[0]
        pos = v > 0
        assert np.all(v2[pos] < v[pos]) and np.all(v2[~pos] == 0)
        vf, _, bf, jf = m.mes(Xs, ys, fl | L.FLAG_FP64)
        vg, G, bg, jg = m.mes(Xs, ys, fl, want_grad=True)          # chunks of 32768 candidates on the gradient path
        assert np.array_equal(vf, vg) and bf == bg and jf == jg
        # sub-ranges across chunk boundaries: d mu and d s2 are the same bits (test_gpu_grad), but mu, and so MES and its chain
        # rule, come from the scoring path, whose FP64 sums are grouped by the size of the call: they agree to rounding
        for lo, hi in ((32700, 32900), (65500, 65600), (0, 1), (69990, 70000)):
            a, Ga, _, _ = m.mes(Xs[lo:hi], ys, fl, want_grad=True)
            assert np.all(np.abs(a - vg[lo:hi]) <= 1e-12 * np.abs(vg[lo:hi]))
            assert np.all(np.abs(Ga - G[lo:hi]) <= 1e-12 * np.max(np.abs(G[lo:hi]), axis=1, keepdims=True))
        assert np.array_equal(m.mes(Xs, ys, fl, want_grad=True)[1], G)
    # device central differences of the FP64 values
    P = Xs[:40]
    _, G, _, _ = m.mes(P, ys, L.FLAG_MODE_PY, want_grad=True)
    fd = np.zeros_like(P)
    h = 1e-6
    for t in range(d):
        E = np.zeros_like(P)
        E[:, t] = h
        fd[:, t] = (m.mes(P + E, ys, L.FLAG_MODE_PY | L.FLAG_FP64)[0] - m.mes(P - E, ys, L.FLAG_MODE_PY | L.FLAG_FP64)[0]) / (2 * h)
    assert np.all(np.abs(G - fd) <= 1e-6 * np.max(np.abs(fd), axis=1, keepdims=True) + 1e-12)


def test_clipped_variance_takes_no_share():
    L = _lib()
    d = 3
    X, Y, _, rs = _data(40, 1, d, 32)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.0)
    Xs = np.r_[X[:6], rs.rand(4, d)]
    ys = np.array([Y.max() + 0.3, Y.max() + 1.0])
    for mode, floor in (("py", 10e-8), ("cpp", 1e-8)):
        fl = _flags(mode)
        mu, s2, dmu, ds2 = m.posterior_grad(Xs, fl)
        assert np.all(s2[:6] == floor) and np.all(ds2[:6] == 0.0)
        _, G, _, _ = m.mes(Xs, ys, fl, want_grad=True)
        # G = (d MES / d mu) dmu on the clipped rows: parallel to dmu
        a = G[:6] / dmu[:6]
        assert np.all(np.abs(a - a[:, :1]) <= 1e-14 * np.abs(a[:, :1]))


@pytest.mark.parametrize("M", [1, 17, 4096, 1 << 20])
@pytest.mark.parametrize("flag", ["default", "fp64", "py"])
def test_gumbel_fit_solves_the_quantile_equations(M, flag):
    L = _lib()
    d = 3
    X, Y, _, rs = _data(1000, 1, d, 40 + M)
    Xs = rs.rand(M, d)
    m = L.Model(orc.K_SE_ARD, [.3, .4, .5], X, Y, 0.1)
    fl = {"default": 0, "fp64": L.FLAG_FP64, "py": L.FLAG_MODE_PY}[flag]
    q, loc, scale = m.max_value_gumbel(Xs, fl)
    mu, s2 = m.posterior(Xs, fl)
    s = np.sqrt(s2)
    for qq, p in zip(q, (0.25, 0.5, 0.75)):
        terms = mo.log_F_terms(qq, mu, s)
        err = abs(math.fsum(terms) - math.log(p))
        assert err <= (M + 8) * 2.0 ** -53 * math.fsum(np.abs(terms)) + 1e-15, (p, err)
    if M == 1:
        for qq, p in zip(q, (0.25, 0.5, 0.75)):
            assert abs(qq - (mu[0] + s[0] * norm.ppf(p))) <= 1e-13 * (abs(mu[0]) + s[0])
    loc_o, scale_o = mo.gumbel_loc_scale(q)
    assert loc == loc_o and scale == scale_o and q[0] < q[1] < q[2]
    q2, loc2, scale2 = m.max_value_gumbel(Xs, fl)
    assert np.array_equal(q, q2) and loc == loc2 and scale == scale2
    m.close()


def test_workspace_interleaved_with_joint_gradient_and_qei_calls():
    """MES and the Gumbel fit between joint, gradient and q-EI calls on one handle give a fresh handle's bytes"""
    L = _lib()
    d = 3
    X, Y, _, rs = _data(700, 1, d, 50)
    hyper = [.3, .4, .5]
    ys = _ystar(Y, 12, rs)
    Z = np.random.default_rng(0).standard_normal((3, 64))
    calls = [
        lambda m, P: m.mes(P[:3000], ys)[0],
        lambda m, P: m.posterior_cov(P[:200])[1],
        lambda m, P: m.mes(P[:500], ys, L.FLAG_MODE_PY, want_grad=True)[1],
        lambda m, P: m.max_value_gumbel(P[:5000])[0],
        lambda m, P: m.posterior_grad(P[:900])[2],
        lambda m, P: m.qei(P[:300].reshape(100, 3, d), Z, Y.max(), 0.01)[1],
        lambda m, P: m.mes(P[:40], ys, L.FLAG_MODE_CPP, want_grad=True)[1],
        lambda m, P: m.max_value_gumbel(P[:17], L.FLAG_MODE_PY)[0],
        lambda m, P: m.mes(P[:4000], ys, L.FLAG_FP64)[0],
        lambda m, P: m.posterior_sample(P[:100], Z[:, :8].repeat(34, axis=0)[:100], 1e-6)[0],
    ]
    P = rs.rand(6000, d)
    shared = L.Model(orc.K_SE_ARD, hyper, X, Y, 0.1)
    for c in calls:
        got = c(shared, P)
        fresh = L.Model(orc.K_SE_ARD, hyper, X, Y, 0.1)
        want = c(fresh, P)
        fresh.close()
        assert got.tobytes() == want.tobytes()
    shared.close()


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
def test_maximize_mes(name):
    from ibo_b200 import _lib as L
    from ibo_b200.acquisition import maximizeMES, MES
    from ibo_b200.utils.latinhypercube import lhcSample
    gp, bounds = _gp(name)
    b = np.array(bounds)
    opt, optx = maximizeMES(gp, bounds, n_samples=10, seed=2, maxiter=30, polish=8)
    last = maximizeMES.last
    assert np.all(optx >= b[:, 0]) and np.all(optx <= b[:, 1])
    assert last["samples"] > 0 and last["polish"]["evaluations"] >= 2 and np.all(last["ystar"] >= np.max(gp.Y))
    C = np.array(lhcSample(bounds, 16384, seed=2))
    q, loc, scale = gp.model.max_value_gumbel(C, L.FLAG_MODE_PY)
    assert loc == last["loc"] and scale == last["scale"]
    cv = gp.model.mes(C, last["ystar"], L.FLAG_MODE_PY | L.FLAG_FP64)[0]
    assert opt >= np.max(cv) * (1 - 1e-9)
    assert abs(MES(gp, last["ystar"]).f(optx) - opt) <= 1e-9 * abs(opt)
    opt2, optx2 = maximizeMES(gp, bounds, n_samples=10, seed=2, maxiter=30, polish=8)
    assert opt2 == opt and np.array_equal(optx2, optx) and np.array_equal(maximizeMES.last["ystar"], last["ystar"])


def test_sample_max_values():
    gp, bounds = _gp("hartman6")
    C = np.random.RandomState(3).rand(500, 6)
    F = gp.sample_posterior(C, 10, seed=4)
    assert np.array_equal(gp.sample_max_values(C, 10, seed=4, method="joint", floor=-np.inf), np.max(F, axis=0))
    assert np.array_equal(gp.sample_max_values(C, 10, seed=4, method="joint"), np.maximum(np.max(F, axis=0), np.max(gp.Y)))
    g1 = gp.sample_max_values(C, 7, seed=5, floor=-np.inf)
    assert np.array_equal(g1, gp.sample_max_values(C, 7, seed=5, floor=-np.inf)) and np.all(np.isfinite(g1))
    q, loc, scale = gp.model.max_value_gumbel(C, _lib().FLAG_MODE_PY)
    assert scale > 0 and np.median(gp.sample_max_values(C, 20001, seed=6, floor=-np.inf)) == pytest.approx(
        loc - scale * math.log(-math.log(0.5)), abs=0.05 * scale)


def test_bad_arguments():
    L = _lib()
    lib = L.lib()
    X, Y, Xs, rs = _data(20, 4, 2, 34)
    m = L.Model(orc.K_SE_ARD, [.3, .4], X, Y, 0.1)
    p = L.dptr
    v = np.zeros(4); g = np.zeros(8); ys = np.zeros(1025); best, idx = ctypes.c_double(0), ctypes.c_long(0)
    nan = np.array([0.0, float("nan")])
    for y, K, fl, dv in [(p(ys), 0, 0, None), (p(ys), 1025, 0, None), (p(nan), 2, 0, None), (p(ys), 2, L.FLAG_INT8, p(g))]:
        assert lib.ibo_mes(m.handle, p(Xs), 4, y, K, fl, p(v), dv, ctypes.byref(best), ctypes.byref(idx)) == L.E_BADARG
    assert lib.ibo_mes(m.handle, p(Xs), 4, p(ys), 1024, 0, p(v), p(g), ctypes.byref(best), ctypes.byref(idx)) == 0
    assert lib.ibo_max_value_gumbel(m.handle, p(Xs), 4, L.FLAG_INT8, None, None, None) == 0
