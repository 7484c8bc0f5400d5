"""GPU tests of the workspace that the joint posterior, the candidate gradients and q-EI share on a model handle: the three entry
points interleaved on one handle, with sizes that grow and shrink so that buffers grown by one are reused smaller by another, give
byte for byte what the same call gives on a freshly built handle (empty workspace; model builds are bit-reproducible)."""
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


def _bytes(out):
    if not isinstance(out, tuple):
        out = (out,)
    return [None if a is None else np.asarray(a).tobytes() for a in out]


@pytest.mark.parametrize("case,N", [("plain", 8192), ("prior", 2048), ("pref", 300)])
def test_interleaved_calls_on_one_handle_equal_fresh_handles(case, N):
    make, ymax = {"plain": _plain, "prior": _prior, "pref": _pref}[case](N, 40)
    shared, keep = make()
    for name, call in _steps(N, ymax, 41):
        got = _bytes(call(shared))
        fresh, keep_f = make()
        want = _bytes(call(fresh))
        for h in [fresh] + keep_f:
            h.close()
        assert got == want, name
    for h in [shared] + keep:
        h.close()
