"""GPU tests of the workspace that the candidate-side entry points share on a model handle: the joint posterior, the candidate
gradients and q-EI, and the entry points that factorise in the workspace's scratch factor (samples, q-NEI, the Laplace fit, sample
paths of a Laplace model), interleaved on one handle with sizes that grow and shrink so that buffers grown by one are reused smaller
by another, give byte for byte what the same call gives on a freshly built handle (empty workspace; model builds are
bit-reproducible)."""
import ctypes

import numpy as np
import pytest

from oracle import ibo_oracle as orc

pytestmark = pytest.mark.gpu

D = 3
THETA = [.3, .4, .5]


def _lib():
    from ibo_b200 import _lib as L
    return L


def _chunk(N):
    """candidates per chunk of the gradient and q-EI paths (K* and V of 2 Np doubles per candidate in 512 MiB)"""
    Np = (N + 127) // 128 * 128
    return max(128, (512 << 20) // (2 * 8 * Np) // 128 * 128)


def _plain(N, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, D)
    Y = np.sin(3 * X).sum(axis=1)

    def make():
        L = _lib()
        return L.Model(orc.K_SE_ARD, THETA, X, Y, 0.1), []
    return make, Y.max()


def _prior(N, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, D)
    Y = np.sin(3 * X).sum(axis=1)
    prior = orc.PriorSpec(rs.rand(4, D), 0.3 * rs.randn(4), 3.0, np.zeros(D), np.ones(D))

    def make():
        L = _lib()
        return L.Model(orc.K_SE_ARD, THETA, X, Y, 0.1, prior=prior), []
    return make, Y.max()


def _pref(N, seed):
    """a preference model (A = R + inv(C), C inverted on the device) with a variance model over its points and three more"""
    rs = np.random.RandomState(seed)
    X = rs.rand(N, D)
    Y = 0.5 * rs.randn(N)
    A = rs.randn(N, N) * 0.05
    C = np.eye(N) * 5 + A.dot(A.T)
    augX = np.r_[X, rs.rand(3, D)]
    pad = np.zeros((N + 3, N + 3))
    pad[:N, :N] = np.linalg.inv(C)

    def make():
        L = _lib()
        m = L.Model(orc.K_SE_ARD, THETA, X, Y, 0.1, C=C)
        v = L.Model(orc.K_SE_ARD, THETA, augX, np.zeros(N + 3), 0.1, Cinv=pad)
        m.set_variance_model(v)
        return m, [v]
    return make, Y.max()


def _laplace(N, seed):
    """a Laplace model with a host-supplied inv(C): N <= 4096 keeps A = R + inv(C), from which sample paths form their noise factor"""
    rs = np.random.RandomState(seed)
    X = rs.rand(N, D)
    Y = 0.5 * rs.randn(N)
    A = rs.randn(N, N) * 0.05
    Cinv = np.linalg.inv(np.eye(N) * 5 + A.dot(A.T))

    def make():
        L = _lib()
        return L.Model(orc.K_SE_ARD, THETA, X, Y, 0.1, Cinv=Cinv), []
    return make, Y.max()


def _steps(N, ymax, seed):
    """(name, call) in order: sizes grow and shrink across the three entry points, with rejected calls in between"""
    L = _lib()
    rs = np.random.RandomState(seed)
    gen = np.random.default_rng(seed)
    chunk = _chunk(N)
    Xs1 = rs.rand(2500, D)
    Z1 = gen.standard_normal((2500, 16))
    Xs2 = rs.rand(2 * chunk + 800, D)                  # three chunks
    Xb3 = rs.rand(chunk // 4 + 50, 4, D)               # two chunks of whole batches of 4
    Z3 = gen.standard_normal((4, 64))
    Xs4 = rs.rand(300, D)
    Xs5 = rs.rand(64, D)
    Xb6 = rs.rand(3, 4, D)
    Z6 = gen.standard_normal((4, 33))
    Xs7 = rs.rand(100, D)
    Z7 = gen.standard_normal((100, 200))

    def rejected(m):
        lib, p = L.lib(), L.dptr
        x = np.ascontiguousarray(Xs5)
        o = np.zeros(64 * 64)
        rcs = (lib.ibo_posterior_cov(m.handle, p(x), 16385, p(o), p(o)),
               lib.ibo_score_grad(m.handle, p(x), 4, 3, 0.0, 0.01, 0, p(o), p(o)),
               lib.ibo_qei(m.handle, p(x), 1, 33, p(o), 4, 0.0, 0.01, 0.0, p(o), None, None))
        assert rcs == (L.E_BADARG,) * 3
        return ()

    return [
        ("sample M=2500", lambda m: m.posterior_sample(Xs1, Z1, jitter=1e-9)),
        ("score_grad three chunks", lambda m: m.score_grad(Xs2, L.ACQ_EI, ymax, 0.01)),
        ("qei two chunks", lambda m: m.qei(Xb3, Z3, ymax - 0.2, 0.01)),
        ("rejected", rejected),
        ("cov M=300", lambda m: m.posterior_cov(Xs4)),
        ("score_grad M=64", lambda m: m.score_grad(Xs5, L.ACQ_UCB, ymax, 1.3, L.FLAG_MODE_CPP)),
        ("posterior_grad M=64", lambda m: m.posterior_grad(Xs5)),
        ("qei B=3 q=4", lambda m: m.qei(Xb6, Z6, ymax - 0.2, 0.01, jitter=1e-8)),
        ("rejected", rejected),
        ("sample M=100", lambda m: m.posterior_sample(Xs7, Z7)),
        ("qei values only", lambda m: m.qei(Xb6, Z6, ymax - 0.2, 0.0, want_grad=False)),
    ]


def _factor_steps(N, ymax, seed, pref):
    """(name, call) in order over the entry points that factorise in the scratch factor: the factor grows and shrinks from one to
    the next (M = 2500, N, P = 300, N, M = 100, P = 50), and sample paths resize V, K*, the normals and a | b; the Laplace fit only
    on a plain model (pref)"""
    from ibo_b200.gaussianprocess import path_draws
    rs = np.random.RandomState(seed)
    gen = np.random.default_rng(seed)
    Xs1 = rs.rand(2500, D)
    Z1 = gen.standard_normal((2500, 16))
    Xb2, Xbase2 = rs.rand(20, 3, D), rs.rand(300, D)
    Z2 = gen.standard_normal((303, 64))
    dr3, Xs3 = path_draws(orc.K_SE_ARD, D, 1024, 80, N, seed), rs.rand(700, D)
    Xs4 = rs.rand(100, D)
    Z4 = gen.standard_normal((100, 40))
    Xb5, Xbase5 = rs.rand(5, 2, D), rs.rand(50, D)
    Z5 = gen.standard_normal((52, 33))
    dr6, Xs6 = path_draws(orc.K_SE_ARD, D, 300, 7, N, seed + 1), rs.rand(64, D)
    v, u = rs.randint(0, N, 400), rs.randint(0, N - 1, 400)
    u += u >= v                                        # distinct pairs
    deg = (rs.rand(400) < 0.2).astype(float)
    start = np.where(np.isin(np.arange(N), v), 0.5, -0.5)

    def paths(dr, Xs):
        def call(m):
            p = m.sample_paths(*dr)
            out = p.eval(Xs)
            p.close()
            return out
        return call

    fit = [("pref_fit", lambda m: m.pref_fit(v, u, deg, start))] if pref else []
    return [("sample M=2500", lambda m: m.posterior_sample(Xs1, Z1, jitter=1e-9))] + fit + [
        ("qnei P=300", lambda m: m.qnei(Xb2, Xbase2, Z2, jitter=1e-6)),
        ("paths S=80", paths(dr3, Xs3)),
        ("sample M=100", lambda m: m.posterior_sample(Xs4, Z4)),
    ] + fit + [
        ("qnei P=50", lambda m: m.qnei(Xb5, Xbase5, Z5, jitter=1e-6, want_grad=False)),
        ("paths S=7", paths(dr6, Xs6)),
    ] + fit


def _bytes(out):
    if not isinstance(out, tuple):
        out = (out,)
    return [None if a is None else np.asarray(a).tobytes() for a in out]


@pytest.mark.parametrize("case,N", [("plain", 8192), ("prior", 2048), ("pref", 300), ("plain_factor", 600), ("laplace_factor", 700)])
def test_interleaved_calls_on_one_handle_equal_fresh_handles(case, N):
    build = {"plain": _plain, "prior": _prior, "pref": _pref, "plain_factor": _plain, "laplace_factor": _laplace}[case]
    make, ymax = build(N, 40)
    steps = _factor_steps(N, ymax, 41, case == "plain_factor") if case.endswith("_factor") else _steps(N, ymax, 41)
    shared, keep = make()
    for name, call in steps:
        got = _bytes(call(shared))
        fresh, keep_f = make()
        want = _bytes(call(fresh))
        for h in [fresh] + keep_f:
            h.close()
        assert got == want, name
    for h in [shared] + keep:
        h.close()


def test_pref_fit_after_a_failed_sample_on_the_same_handle():
    """a failed ibo_posterior_sample leaves its pivot in the scratch factor's status word; a Laplace fit on the same handle from a
    start that already meets gtol (no Newton step, so no factorisation clears it) still succeeds, with a fresh handle's bytes"""
    L = _lib()
    X = np.array([[3.0 * i, 0.0] for i in range(6)])
    hyper = [0.3, 2.0]                                 # Matern-3/2, sf2 = 4 > 1 + noise: a repeated candidate is indefinite

    def make():
        return L.Model(orc.K_MATERN3, hyper, X, np.zeros(6), 0.1)
    Xs = np.array([[100., 100.], [100., 100.], [50., 50.]])
    Z = np.random.default_rng(0).standard_normal((3, 4))
    v, u, deg, start = [0, 2, 4], [1, 3, 5], [0.0, 1.0, 0.0], np.array([.5, -.5, .5, -.5, .5, -.5])
    m = make()
    with pytest.raises(L.NotPositiveDefinite) as ei:
        m.posterior_sample(Xs, Z)
    assert ei.value.pivot == 2
    got = m.pref_fit(v, u, deg, start, gtol=1e6)
    assert got[3] == 0
    fresh = make()
    assert _bytes(got) == _bytes(fresh.pref_fit(v, u, deg, start, gtol=1e6))
    for h in (m, fresh):
        h.close()
