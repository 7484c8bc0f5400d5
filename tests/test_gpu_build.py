"""GPU tests of the model build (model.cu: R, the look-ahead blocked Cholesky in both schedules, W = inv(L), the packed blobs,
beta_Y = W Y, beta_1 = W 1, the rank-1 append, and the other entry points that end in the same factorisation) against an
extended-precision reference (tests/build_oracle.py) and against LAPACK.

An FP64 factorisation of an ill-conditioned matrix cannot be exact; what it can be is as accurate as FP64 allows.  So the device's
error is measured against the longdouble result and bounded by C times the error of LAPACK (dpotrf, dtrtri) on the same input,
or of the FP64 oracle for the posterior, plus a floor of N eps.  The input to both sides is the device's own A (matrix(0)),
which separates the factorisation from the build of R.  Small noise (down to 1e-6, cond(R) up to ~1e9) is where an explicit
inverse of the diagonal blocks could lose digits that a substitution keeps."""
import numpy as np
import pytest
from scipy.linalg import blas, cho_factor, cho_solve, lapack

import build_oracle as bo
from oracle import ibo_oracle as orc

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
C = 4.0
KINDS = {
    "se_ard_long": (orc.K_SE_ARD, [1.0, 1.5, 2.0]),       # long length scales: the ill-conditioned case
    "matern3": (orc.K_MATERN3, [0.5, 1.0]),
    "matern5_prior": (orc.K_MATERN5, [0.5, 1.0]),          # with the RBF prior mean: beta_1 enters mu
}
NOISES = [0.1, 1e-3, 1e-4, 1e-6]
GRID = [(N, k, nz) for N in (1, 127, 128, 129, 300, 640) for k in KINDS for nz in NOISES]
GRID += [(1100, "se_ard_long", nz) for nz in NOISES]       # 9 row-blocks; the host reference takes ~6 s per case here


@pytest.fixture
def options():
    """set_option for the test; every option it changed gets its old value back afterwards"""
    from ibo_b200 import _lib
    old = {}

    def set_(name, value):
        old.setdefault(name, _lib.get_option(name))
        _lib.set_option(name, value)
    try:
        yield set_
    finally:
        for name, value in old.items():
            _lib.set_option(name, value)


def _lapack(A):
    L, info = lapack.dpotrf(A, lower=1, clean=1)
    assert info == 0
    W, info = lapack.dtrtri(L, lower=1)
    assert info == 0
    return L, W


def _ld_mv(M, v):
    return np.asarray(M, dtype=bo.LD) @ np.asarray(v, dtype=bo.LD)


def _problem(N, name, seed):
    kind, hyper = KINDS[name]
    rs = np.random.RandomState(seed)
    X = rs.rand(N, 3)
    Y = np.sin(3 * X).sum(axis=1) + 0.1 * rs.randn(N)
    prior = orc.PriorSpec(rs.rand(4, 3), 0.3 * rs.randn(4), 3.0, np.zeros(3), np.ones(3)) if name == "matern5_prior" else None
    Xs = rs.rand(256, 3)
    k = min(N, 64)
    Xs[:k] = X[:k]                                                     # on training points
    Xs[64:64 + k] = X[N - k:] + 1e-5 * (2 * rs.rand(k, 3) - 1)         # within 1e-5 of them
    return orc.KernelSpec(kind, hyper, 3), X, Y, prior, Xs


def _check_posterior(tag, spec, X, Y, noise, prior, Xs, results, L_true=None):
    """results: [(label, (scores, mu, s2, best, bidx))] of the device; each within C x the FP64 oracle's error of the longdouble
    posterior (sigma^2: the larger of the substitution's and the explicit inverse's error), and its argmax as good as the
    oracle's accuracy can tell apart.  Returns (failures, measured ratios)."""
    N = len(Y)
    mu_s, s2_s = bo.posterior(spec, X, Y, noise, Xs, prior=prior, L=L_true)
    mu_s, s2_s = mu_s.astype(float), np.clip(s2_s, 1e-8, 10.0).astype(float)      # FLAG_MODE_CPP clips sigma^2 at 1e-8
    o = orc.GPOracle(spec, X, Y, noise, prior=prior)
    mu_o, s2_o = o.posterior_batch(Xs, floor=1e-8)
    # sigma^2 = (1 + noise) - |W k*|^2 through an explicit inverse loses more than the oracle's substitution (up to ~20x at noise
    # 1e-6, N = 1100): the same form with LAPACK's W (dtrtri) is what FP64 can deliver for it
    V = lapack.dtrtri(o.L, lower=1)[0].dot(spec.cross(X, Xs))
    s2_w = np.clip((1 + noise) - np.sum(V * V, axis=0), 1e-8, 10.0)
    ymax = Y.max()
    ei_s = orc.score(orc.ACQ_EI, "cpp", mu_s, s2_s, ymax, 0.01)
    ei_o = orc.score(orc.ACQ_EI, "cpp", mu_o, s2_o, ymax, 0.01)
    e_mu_o, e_s2_o = np.max(np.abs(mu_o - mu_s)), max(np.max(np.abs(s2_o - s2_s)), np.max(np.abs(s2_w - s2_s)))
    f_mu, f_s2 = N * EPS * max(1.0, np.max(np.abs(mu_s))), N * EPS
    tol_ei = C * np.max(np.abs(ei_o - ei_s)) + N * EPS * np.max(np.abs(ei_s))
    bad, ratios = [], {}
    for label, (sc, mu, s2, best, bidx) in results:
        e_mu, e_s2 = np.max(np.abs(mu - mu_s)), np.max(np.abs(s2 - s2_s))
        ratios["mu_" + label] = e_mu / max(e_mu_o, 1e-300)
        ratios["s2_" + label] = e_s2 / max(e_s2_o, 1e-300)
        if e_mu > C * e_mu_o + f_mu:
            bad.append("%s %s: mu error %.3e, oracle %.3e" % (tag, label, e_mu, e_mu_o))
        if e_s2 > C * e_s2_o + f_s2:
            bad.append("%s %s: sigma^2 error %.3e, oracle %.3e" % (tag, label, e_s2, e_s2_o))
        if ei_s[bidx] < ei_s.max() - tol_ei:
            bad.append("%s %s: argmax %d has EI %.17g, the best %.17g (tolerance %.3e)" % (tag, label, bidx, ei_s[bidx], ei_s.max(), tol_ei))
        if not (best == sc[bidx] and bidx == int(np.argmax(sc))):
            bad.append("%s %s: best / argmax are not the scores' own" % (tag, label))
    return bad, ratios


def _check_factor(tag, A, L, W, Ls, Ws, Lp, Wp):
    """L and W of the device against the longdouble factor of the same A, bounded by C x LAPACK's error + N eps"""
    N = A.shape[0]
    floor = N * EPS
    bad, ratios = [], {}
    for name, got, want, lap in (("L", L, Ls, Lp), ("W", W, Ws, Wp)):
        e, ep = bo.rel(got, want), bo.rel(lap, want)
        ratios[name] = e / max(ep, 1e-300)
        if e > C * ep + floor:
            bad.append("%s: e(%s) = %.3e, LAPACK %.3e" % (tag, name, e, ep))
        if not np.array_equal(np.triu(got, 1), np.zeros_like(got)):
            bad.append("%s: %s has non-zeros above the diagonal" % (tag, name))
    return bad, ratios


@pytest.mark.parametrize("N,name,noise", GRID)
def test_build_and_posterior_against_longdouble(N, name, noise, options):
    from ibo_b200 import _lib
    spec, X, Y, prior, Xs = _problem(N, name, 1000 + N)
    options("i8_min_batch", 192)               # a 256-point batch takes the INT8 kernels and gets the bits of a wide batch
    dev = {}
    for pair in (0, 1):
        options("chol_pair", pair)
        m = _lib.Model(spec.kind, spec.hyper, X, Y, noise, prior=prior)
        try:
            f64 = m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01, _lib.FLAG_MODE_CPP | _lib.FLAG_FP64, want_posterior=True)
            i8 = m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01, _lib.FLAG_MODE_CPP | _lib.FLAG_INT8, want_posterior=True)
            dev[pair] = (m.matrix(0), m.matrix(1), m.matrix(2), f64, i8)
        finally:
            m.close()
    A = dev[0][0]
    assert np.array_equal(A, dev[1][0])
    Ls = bo.cholesky(A)
    Ws = bo.tri_inv(Ls)
    Lp, Wp = _lapack(A)
    # beta_Y = W Y and beta_1 = W 1 through the device's W; the posterior below reaches the device's own beta vectors
    bY, b1 = _ld_mv(Ws, Y), Ws.sum(axis=1)
    eYp, e1p = bo.rel(_ld_mv(Wp, Y), bY), bo.rel(Wp.sum(axis=1), b1)
    L_true = Ls if N == 1 else bo.cholesky(bo.build_R(spec, X, noise))
    tag = "N=%d %s noise=%g" % (N, name, noise)
    bad, ratios = _check_posterior(tag, spec, X, Y, noise, prior, Xs,
                                   [("%s_pair%d" % (p, pair), dev[pair][k]) for pair in (0, 1) for k, p in ((3, "fp64"), (4, "int8"))], L_true)
    for pair in (0, 1):
        _, L, W, _, _ = dev[pair]
        b, r = _check_factor("%s chol_pair=%d" % (tag, pair), A, L, W, Ls, Ws, Lp, Wp)
        bad += b
        eY, e1 = bo.rel(_ld_mv(W, Y), bY), bo.rel(np.asarray(W, dtype=bo.LD).sum(axis=1), b1)
        if eY > C * eYp + N * EPS or e1 > C * e1p + N * EPS:
            bad.append("%s chol_pair=%d: e(W Y) = %.3e (LAPACK %.3e), e(W 1) = %.3e (LAPACK %.3e)" % (tag, pair, eY, eYp, e1, e1p))
        ratios.update(("%s_pair%d" % kv[0], kv[1]) for kv in [((k, pair), v) for k, v in r.items()])
    print("RATIO %s %s" % (tag, " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
    assert not bad, "\n".join(bad)


def _ld_free_backward(R, L, W):
    """||R - L L^T||_F / ||R||_F and ||W L - I||_F, in FP64 with triangular products"""
    LLt = blas.dtrmm(1.0, L, np.ascontiguousarray(L.T), lower=1)
    WL = blas.dtrmm(1.0, W, L, lower=1)
    WL[np.diag_indices_from(WL)] -= 1.0
    return np.linalg.norm(R - LLt) / np.linalg.norm(R), np.linalg.norm(WL)


@pytest.mark.parametrize("N", [2049, 6016, 6017, 6272])
def test_large_builds_schedule_bits_and_backward_error(N, options):
    """17, 47, 48 and 49 block columns: the default schedule is read from the bits (paired block columns from 48 on), two builds
    of one model give the same bits, and the factor is as good as LAPACK's on the same R"""
    from ibo_b200 import _lib
    rs = np.random.RandomState(N)
    d, noise = 4, 0.1
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    hyper = [0.3, 1.0]
    Xs = rs.rand(3000, d)
    nb = (N + 127) // 128
    got = {}
    for pair in (-1, 0, 1):
        options("chol_pair", pair)
        m = _lib.Model(orc.K_MATERN5, hyper, X, Y, noise)
        try:
            sc = m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01, _lib.FLAG_MODE_CPP)[0]
            got[pair] = (m.matrix(1), m.matrix(2), sc)
            if pair == -1:
                R = m.matrix(0) if N <= 4096 else orc.build_R(orc.KernelSpec(orc.K_MATERN5, hyper, d), X, noise)
                idx = np.unique(np.r_[np.arange(0, N, 97), np.arange(127, N, 128), N - 1])
                mu, s2 = m.posterior(X[idx], _lib.FLAG_MODE_CPP)
        finally:
            m.close()
    same = 1 if nb >= 48 else 0
    for k in range(3):
        assert np.array_equal(got[-1][k], got[same][k]), "default build at %d blocks is not chol_pair=%d bit for bit" % (nb, same)
    assert not np.array_equal(got[-1][0], got[1 - same][0])
    L, W = got[-1][0], got[-1][1]
    assert np.array_equal(np.triu(L, 1), np.zeros_like(L)) and np.array_equal(np.triu(W, 1), np.zeros_like(W))
    Lp, Wp = _lapack(R)
    bd, wd = _ld_free_backward(R, L, W)
    bp, wp = _ld_free_backward(R, Lp, Wp)
    print("RATIO N=%d backward=%.2f (%.2e / %.2e) WL-I=%.2f (%.2e / %.2e)" % (N, bd / bp, bd, bp, wd / wp, wd, wp))
    assert bd <= C * bp + EPS and wd <= C * wp + EPS
    # training-point identities (tests/test_gpu_fullsize.py) at every block's last row
    cf = cho_factor(R, lower=True)
    E = np.zeros((N, len(idx)))
    E[idx, np.arange(len(idx))] = 1.0
    mu_id = Y[idx] - noise * cho_solve(cf, Y)[idx]
    s2_id = 2 * noise - noise * noise * cho_solve(cf, E)[idx, np.arange(len(idx))]
    assert np.max(np.abs(mu - mu_id) / np.maximum(np.abs(mu_id), 1e-3)) <= 1e-10
    assert np.max(np.abs(s2 - s2_id) / s2_id) <= 1e-10


def test_two_builds_of_one_model_are_bit_identical():
    from ibo_b200 import _lib
    rs = np.random.RandomState(11)
    X = rs.rand(1100, 3)
    Y = np.sin(3 * X).sum(axis=1)
    Xs = rs.rand(3000, 3)
    out = []
    for _ in range(2):
        m = _lib.Model(orc.K_SE_ARD, [0.3, 0.4, 0.5], X, Y, 1e-4)
        out.append((m.matrix(1), m.matrix(2), m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01)[0]))
        m.close()
    for a, b in zip(*out):
        assert np.array_equal(a, b)


def _grid(N):
    g = np.arange(11) / 10.0
    return np.array([[a, b, c] for a in g for b in g for c in g])[:N]


@pytest.mark.parametrize("pivots", [(128,), (700,), (1099,), (700, 1099)])
@pytest.mark.parametrize("pair", [0, 1])
def test_first_failing_pivot_is_reported(pivots, pair, options):
    """Matern-3/2 with sf2 = 4 over a diagonal of 1 + noise on a grid 0.1 apart (length scale 0.01: off-diagonals ~ 1e-6, SPD); a
    near-duplicate pair at rows (p - 1, p) makes the 2 x 2 minor indefinite, so pivot p + 1 (1-based) is the first to fail"""
    from ibo_b200 import _lib
    X = _grid(1100)
    for p in pivots:
        X[p] = X[p - 1] + 1e-9
    Y = np.sin(3 * X).sum(axis=1)
    options("chol_pair", pair)
    with pytest.raises(np.linalg.LinAlgError) as ei:
        _lib.Model(_lib.KERNEL_MATERN3, [0.01, 2.0], X, Y, 0.1)
    assert ei.value.pivot == pivots[0] + 1


def test_indefinite_preference_matrix_reports_its_pivot():
    from ibo_b200 import _lib
    rs = np.random.RandomState(5)
    N, P = 1100, 900
    X = rs.rand(N, 4) * 10
    a = rs.randint(0, N, P).astype(np.int32)
    b = rs.randint(0, N, P).astype(np.int32)
    keep = (a != 600) & (b != 600)
    a, b = np.r_[a[keep], 600].astype(np.int32), np.r_[b[keep], 900].astype(np.int32)
    w = np.r_[rs.rand(keep.sum()) * 3, -5.0]          # C_600,600 = 0.5 - 5: rows before it form an SPD Laplacian + 0.5 I
    Cm = np.eye(N) * 0.5
    for i, j, v in zip(a, b, w):
        if i != j:
            Cm[i, i] += v; Cm[j, j] += v; Cm[i, j] -= v; Cm[j, i] -= v
    assert lapack.dpotrf(Cm, lower=1)[1] == 601
    for kw in (dict(pref=(a, b, w, 0.5)), dict(C=Cm)):
        with pytest.raises(np.linalg.LinAlgError) as ei:
            _lib.Model(_lib.KERNEL_SE_ARD, [5.1, 4.2, 4.6, 5.8], X, rs.randn(N), 0.1, **kw)
        assert ei.value.pivot == 601


@pytest.mark.parametrize("N", [1100, 2049])
def test_build_from_inverse_at_multi_block_sizes(N):
    """ibo_model_create_from_inverse: chol(J invR J) reversed and transposed; W^T W = invR as closely as the same procedure in
    LAPACK gets, W exactly lower triangular, and the legacy posterior of the oracle"""
    from ibo_b200 import _lib
    rs = np.random.RandomState(N)
    X = rs.rand(N, 3)
    Y = np.sin(3 * X).sum(axis=1)
    hyper = [0.3, 0.4, 0.5]
    o = orc.GPOracle(orc.KernelSpec(orc.K_SE_ARD, hyper, 3), X, Y, 0.1)
    invR = o.invR()
    invR = 0.5 * (invR + invR.T)
    m = _lib.Model(orc.K_SE_ARD, hyper, X, Y, 0.1, invR=invR, sf2=1.0)
    W = m.matrix(2)
    assert np.array_equal(np.triu(W, 1), np.zeros_like(W))
    G, info = lapack.dpotrf(np.ascontiguousarray(invR[::-1, ::-1]), lower=1, clean=1)
    assert info == 0
    Wp = np.ascontiguousarray(G.T[::-1, ::-1])
    e, ep = bo.rel(W.T.dot(W), invR), bo.rel(Wp.T.dot(Wp), invR)
    print("RATIO from_inverse N=%d %.2f (%.2e / %.2e)" % (N, e / ep, e, ep))
    assert e <= C * ep + N * EPS
    Xs = rs.rand(500, 3)
    Xs[:50] = X[:50]
    mu_o, sig_o = o.posterior_cpp(Xs, invR=invR)
    _, mu, s2, _, _ = m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01, _lib.FLAG_MODE_CPP, want_posterior=True)
    assert np.max(np.abs(mu - mu_o) / np.maximum(np.abs(mu_o), 1e-3)) <= 1e-10
    assert np.max(np.abs(np.sqrt(s2) - sig_o) / sig_o) <= 1e-10
    m.close()


def test_preference_build_at_multi_block_size():
    """ibo_model_create_pref at 9 row-blocks: inv(C) = Wc^T Wc against the longdouble inverse, and the factor of R + inv(C)"""
    from ibo_b200 import _lib
    rs = np.random.RandomState(12)
    N, d, P = 1100, 4, 2500
    X = rs.rand(N, d) * 10
    a = rs.randint(0, N, P).astype(np.int32)
    b = rs.randint(0, N, P).astype(np.int32)
    w = rs.rand(P) * 3
    Cm = np.eye(N) * 5.0
    for i, j, v in zip(a, b, w):
        if i != j:
            Cm[i, i] += v; Cm[j, j] += v; Cm[i, j] -= v; Cm[j, i] -= v
    m = _lib.Model(_lib.KERNEL_SE_ARD, [5.146, 4.189, 4.622, 5.843], X, rs.randn(N), 0.1, pref=(a, b, w, 5.0))
    Ci, A, L = m.matrix(3), m.matrix(0), m.matrix(1)
    m.close()
    Wc = bo.tri_inv(bo.cholesky(Cm))
    Cs = Wc.T @ Wc
    Cp = lapack.dpotri(lapack.dpotrf(Cm, lower=1, clean=1)[0], lower=1)[0]
    Cp = np.tril(Cp) + np.tril(Cp, -1).T
    e, ep = bo.rel(Ci, Cs), bo.rel(Cp, Cs)
    assert np.array_equal(Ci, Ci.T) and e <= C * ep + N * EPS, (e, ep)
    Ls = bo.cholesky(A)
    e, ep = bo.rel(L, Ls), bo.rel(_lapack(A)[0], Ls)
    print("RATIO pref N=%d L=%.2f (%.2e / %.2e)" % (N, e / max(ep, 1e-300), e, ep))
    assert e <= C * ep + N * EPS, (e, ep)


@pytest.mark.parametrize("N", [1100, 2049])
def test_nlml_at_multi_block_sizes(N):
    """ibo_nlml (create_model_with_diag and the Gram product) with the tolerances of tests/test_gpu_hyper.py"""
    from ibo_b200 import _lib
    rs = np.random.RandomState(N)
    X = rs.rand(N, 3)
    Y = np.sin(2 * X).sum(axis=1) + 0.1 * rs.randn(N)
    hyper, noise = [.4, .6, .9], 1e-3
    spec = orc.KernelSpec(orc.K_SE_ARD, hyper, 3)
    nl_o, g_o = orc.marginal_likelihood(spec, X, Y, len(hyper), noise=noise)
    nl, g = _lib.nlml(orc.K_SE_ARD, hyper, X, Y, noise)
    assert abs(nl - nl_o) <= 1e-10 * abs(nl_o)
    Ki = np.linalg.inv(orc.cov_matrix(spec, X) + noise * np.eye(N))
    al = Ki.dot(Y)
    G = Ki - np.outer(al, al)
    for h in range(len(hyper)):
        scale = 0.5 * np.sum(np.abs(G * orc.kernel_derivative(spec, X, h)))
        assert abs(g[h] - g_o[h]) <= 1e-8 * scale, (h, g[h], g_o[h], scale)


@pytest.mark.parametrize("N0,adds", [(100, [200]), (250, [1] * 8)])
def test_append_at_small_noise_against_longdouble(N0, adds, options):
    """100 + 200 in one call grows the buffers by two row-blocks at once; 250 + 1 x 8 crosses 255 -> 257 a point at a time.  The
    final L and W against the longdouble factor of the final R, then a batch on the INT8 kernels (slices rebuilt after growth)"""
    from ibo_b200 import _lib
    noise = 1e-4
    spec = orc.KernelSpec(orc.K_SE_ARD, [0.4, 0.5, 0.6], 3)
    rs = np.random.RandomState(N0)
    N = N0 + sum(adds)
    X = rs.rand(N, 3)
    Y = np.sin(3 * X).sum(axis=1)
    Xs = rs.rand(256, 3)
    Xs[:64] = X[N - 64:]
    Xs[64:128] = X[:64] + 1e-5 * (2 * rs.rand(64, 3) - 1)
    m = _lib.Model(spec.kind, spec.hyper, X[:N0], Y[:N0], noise)
    n = N0
    for k in adds:
        m.append(X[n:n + k], Y[n:n + k])
        n += k
    options("i8_min_batch", 192)
    i8 = m.score(Xs, _lib.ACQ_EI, Y.max(), 0.01, _lib.FLAG_MODE_CPP | _lib.FLAG_INT8, want_posterior=True)
    A, L, W = m.matrix(0), m.matrix(1), m.matrix(2)
    m.close()
    assert np.max(np.abs(A - orc.build_R(spec, X, noise))) <= 1e-14
    Ls = bo.cholesky(A)
    Ws = bo.tri_inv(Ls)
    Lp, Wp = _lapack(A)
    tag = "append N0=%d adds=%d" % (N0, len(adds))
    bad, r = _check_factor(tag, A, L, W, Ls, Ws, Lp, Wp)
    b, r2 = _check_posterior(tag, spec, X, Y, noise, None, Xs, [("int8", i8)], bo.cholesky(bo.build_R(spec, X, noise)))
    r.update(r2)
    print("RATIO %s %s" % (tag, " ".join("%s=%.2f" % kv for kv in sorted(r.items()))))
    assert not bad + b, "\n".join(bad + b)
