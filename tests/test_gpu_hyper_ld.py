"""GPU tests of the paths that produce a model's inputs -- the marginal likelihood and its gradient (ibo_nlml), the kernel and
derivative matrices (ibo_kernel_matrix) and the Laplace MAP fit of the preference latents (ibo_pref_fit) -- against the
longdouble reference of tests/hyper_oracle.py.

As in tests/test_gpu_build.py, an FP64 result of an ill-conditioned problem cannot be exact; what it can be is as accurate as FP64
allows.  So the device's error against longdouble is bounded by C times the error of FP64 on the same problem, plus a floor of
N eps times the magnitude of the terms.  The FP64 yardstick of the likelihood is the larger error of two forms: the oracle's
substitution (orc.marginal_likelihood) and the device's own explicit inverse with LAPACK (dpotrf, dtrtri, inv(K) = W^T W,
alpha = W^T (W Y)), applied to K as the library builds it: from coordinates scaled by 1 / theta and centred on their mean
before they are differenced (model.cu).  That rounding is relative to the coordinates, not to their difference, so for close
points at small noise it costs the device's nlml up to ~50x the error of the oracle's K (differences first); with it in the
yardstick the comparison measures the factorisation, the Gram product and the reductions."""
import math

import numpy as np
import pytest
from scipy.linalg import lapack

import hyper_oracle as ho
from oracle import ibo_oracle as orc

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
TINY = np.finfo(float).tiny
C = 4.0


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


# ---------------------------------------------------------------------------------------------
# a. kernel and derivative matrices, entry by entry
# ---------------------------------------------------------------------------------------------
# length scales that take the entries from 1 (duplicates) down to ~1e-300 over the unit cube in d = 3
KMAT = {
    "se_ard_mag": (orc.K_SE_ARD, [0.034, 0.042, 0.05, 1.3]),
    "se_ard_clip": (orc.K_SE_ARD, [1e-5, 1e5, 0.05]),          # clipped to 1e-4 and 1e4 (x_0 scaled by 1e-3 to stay in range)
    "se_iso": (orc.K_SE_ISO, [0.041]),
    "matern3": (orc.K_MATERN3, [0.0038, 1.2]),
    "matern5": (orc.K_MATERN5, [0.0048, 1.2]),
    "matern5_ard_mag": (orc.K_MATERN5_ARD, [0.0043, 0.005, 0.006, 1.1]),
}


def _kmat_bound(spec, X, which, exact):
    """per-entry bound on |device - exact| / |exact| from a first-order error analysis of kernel_matrix_kernel (u = eps / 2):
      - scaled coordinates a = x * fl(1 / theta) carry 2u, their difference u more; so the error of r^2 summed over d terms in
        a fixed order is rho <= u (4.02 sum_t |df_t| (|a_t| + |b_t|) + (d + 4) r^2)  (the last term: d - 1 additions, the squares,
        the common 1 / theta);
      - log k has slope at most 3/2 in r^2 for every kind (SE 1/2, Matern-3/2 3/(2(1 + z)), Matern-5/2 below 5/6), and the
        rounding of z = c r, exp and the products adds u (8 + 3 sqrt5 r);
      - a derivative multiplies by powers of s = c r (relative error rho / (2 r^2) + 3u, times the power, plus the extra z of
        exp(-z)) or by dh^2 (relative error 4.02 u (|a_h| + |b_h|) / |df_h| + 3u).
    The bound is twice that sum (c0 = 2 (8u + ...), c1 = 2 (d + 4) u, ...), so it is set by the formula, not by a measurement."""
    u = EPS / 2
    X = np.asarray(X, dtype=float)
    th = np.asarray(spec.theta, dtype=float)
    A = X * (1.0 / th)
    Ab = np.abs(A)
    df = np.abs(A[:, None, :] - A[None, :, :])
    sa = Ab[:, None, :] + Ab[None, :, :]
    r2 = np.sum(df * df, axis=2)
    d = X.shape[1]
    r = np.sqrt(r2)
    rho = u * (4.02 * np.sum(df * sa, axis=2) + (d + 4) * r2)
    with np.errstate(divide="ignore", invalid="ignore"):
        rel_s = np.where(r2 > 0, rho / (2 * r2), 0.0) + 3 * u
        rel_k = 1.5 * rho + u * (8 + 3 * math.sqrt(5) * r)
        nl = ho.nlen(spec)
        if which < 0 or (which == nl and spec.kind != orc.K_SE_ISO):
            b = rel_k + u
        elif spec.kind == orc.K_SE_ISO:
            b = rel_k + 2 * rel_s + u
        elif spec.kind in (orc.K_SE_ARD, orc.K_MATERN5_ARD):
            rel_h = np.where(df[:, :, which] > 0, 4.02 * u * sa[:, :, which] / df[:, :, which], 0.0) + 3 * u
            if spec.kind == orc.K_SE_ARD:
                b = rel_k + rel_h
            else:
                s = math.sqrt(5) * r
                b = (1 + s) * rel_s + rel_h + 3 * u
        elif spec.kind == orc.K_MATERN3:
            z = spec.hyper[0] * r if not exact else math.sqrt(3) * r
            b = (2 + z) * (rel_s + u) + 2 * u
        else:
            s = math.sqrt(5) * r
            b = (3 + s) * rel_s + 3 * u
    return 2 * b


def _kmat_points(name, N):
    rs = np.random.RandomState(N)
    X = rs.rand(N, 3)
    if name == "se_ard_clip":
        X[:, 0] *= 1e-3
    if N > 8:
        X[3] = X[2]                                      # a duplicate: r = 0 off the diagonal
        X[7] = X[6] + 1e-9                               # and a near-duplicate
    return X


@pytest.mark.parametrize("N", [1, 255, 256, 257])
@pytest.mark.parametrize("name", sorted(KMAT))
def test_kernel_and_derivative_matrices_entry_by_entry(name, N):
    """every kind, every hyperparameter index and FLAG_GRAD_EXACT, N across the 256-thread launch grid: each entry within the
    first-order bound of _kmat_bound relative to its own magnitude, plus the smallest normal (an absolute 1e-14 cannot see
    an error in the entries below 1e-14, most of the matrix at these length scales)"""
    from ibo_b200 import _lib
    kind, hyper = KMAT[name]
    X = _kmat_points(name, N)
    spec = orc.KernelSpec(kind, hyper, 3)
    p = ho._Pieces(spec, X)
    jobs = [(-1, False, p.K)] + [(h, False, ho.kernel_derivative(spec, X, h, pieces=p)) for h in range(ho.n_hyper(spec))]
    if kind == orc.K_MATERN3:
        jobs.append((0, True, ho.kernel_derivative(spec, X, 0, True, pieces=p)))
    bad, worst = [], 0.0
    for which, exact, ref in jobs:
        got = _lib.kernel_matrix(kind, hyper, X, which, flags=_lib.FLAG_GRAD_EXACT if exact else 0)
        err = np.abs(got.astype(ho.LD) - ref).astype(float)
        tol = _kmat_bound(spec, X, which, exact) * np.abs(ref).astype(float) + TINY
        worst = max(worst, float(np.max(err / tol)))
        if not np.all(err <= tol):
            i, j = np.unravel_index(np.argmax(err / tol), err.shape)
            bad.append("which=%d exact=%d: (%d, %d) got %.17g want %.17g (tolerance %.3e)" % (which, exact, i, j, got[i, j], ref[i, j], tol[i, j]))
        if N > 1 and which < 0:
            assert np.min(np.abs(ref[np.abs(ref) > 0])) < 1e-250 or kind == orc.K_SE_ARD and name == "se_ard_clip"
    print("RATIO kmat %s N=%d err/bound=%.3f" % (name, N, worst))
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------
# b. nlml and gradient
# ---------------------------------------------------------------------------------------------
def _kind_case(name):
    """(kind, hyper, d, exact): nh = 1, 2, 2, 2, 4, 8, 9, 16, 17"""
    if name == "se_iso":
        return orc.K_SE_ISO, [0.7], 4, False
    if name == "matern3":
        return orc.K_MATERN3, [0.8, 1.2], 3, False
    if name == "matern3_exact":
        return orc.K_MATERN3, [0.8, 1.2], 3, True
    if name == "matern5":
        return orc.K_MATERN5, [0.8, 1.2], 3, False
    d = int(name.split("_d")[1])
    base = orc.K_SE_ARD if name.startswith("se_ard") else orc.K_MATERN5_ARD
    return base, [0.4 * math.sqrt(d) * (1 + 0.5 * t / d) for t in range(d)] + [1.1], d, False


NLML_KINDS = ["se_iso", "matern3", "matern3_exact", "matern5", "se_ard_d3", "se_ard_d7", "se_ard_d8", "m52ard_d15", "m52ard_d16"]
NOISES = [0.1, 1e-3, 1e-4, 1e-6]
NLML_GRID = [(N, k, nz) for N in (1, 2) for k, nz in zip(NLML_KINDS, NOISES * 3)]
NLML_GRID += [(N, k, nz) for N in (63, 64, 65, 127, 128, 129, 300) for k in NLML_KINDS for nz in NOISES
              if N in (128, 300) or (NLML_KINDS.index(k) + NOISES.index(nz) + N) % 3 == 0]
NLML_GRID += [(1100, "se_ard_d3", 1e-6), (1100, "m52ard_d16", 1e-4), (1100, "matern3_exact", 1e-3), (1100, "se_iso", 0.1),
              (2049, "se_ard_d3", 1e-4)]


def _dK64(spec, X, h, exact):
    """orc.kernel_derivative without its N x N x d difference array for the ARD length scales"""
    if spec.kind in (orc.K_SE_ARD, orc.K_MATERN5_ARD) and h < spec.ndim:
        sc = (X[:, h][:, None] - X[:, h][None, :]) / spec.theta[h]
        if spec.kind == orc.K_SE_ARD:
            return orc.cov_matrix(spec, X) * sc ** 2
        D = (X[:, None, :] - X[None, :, :]) / spec.theta[None, None, :]
        s = math.sqrt(5.0) * np.sqrt(np.sum(D ** 2, axis=2))
        return spec.sf2 * (5.0 / 3.0) * (1.0 + s) * np.exp(-s) * sc ** 2
    return orc.kernel_derivative(spec, X, h, exact)


def _device_K(spec, X, noise):
    """covMatrix(X) + noise I in FP64 as model.cu builds it: x / theta minus the mean of those, differenced in dimension order"""
    it = 1.0 / np.asarray(spec.theta, dtype=float)
    ctr = np.zeros(X.shape[1])
    for x in X:
        ctr += x * it
    xt = X * it - ctr / len(X)
    r2 = np.zeros((len(X), len(X)))
    for t in range(X.shape[1]):
        df = xt[None, :, t] - xt[:, None, t]
        r2 += df * df
    if spec.kind in (orc.K_SE_ARD, orc.K_SE_ISO):
        K = spec.sf2 * np.exp(-0.5 * r2)
    elif spec.kind == orc.K_MATERN3:
        z = 1.7320508075688772 * np.sqrt(r2)
        K = spec.sf2 * (1.0 + z) * np.exp(-z)
    else:
        z = 2.23606797749979 * np.sqrt(r2)
        K = spec.sf2 * (1.0 + z + 5.0 * r2 / 3.0) * np.exp(-z)
    K = np.tril(K, -1) + np.tril(K, -1).T
    np.fill_diagonal(K, spec.sf2 + noise)
    return K


def _fp64_forms(spec, X, Y, noise, exact):
    """[(nlml, grad)] of (a) the oracle's substitution (orc.marginal_likelihood) and (b) the device's form with LAPACK, on K as
    the device builds it"""
    N = len(Y)
    K = orc.cov_matrix(spec, X) + noise * np.eye(N)
    nh = ho.n_hyper(spec)
    dKs = [_dK64(spec, X, h, exact) for h in range(nh)]
    L = np.linalg.cholesky(K)
    al = np.linalg.solve(L.T, np.linalg.solve(L, Y))
    nl_a = 0.5 * Y.dot(al) + np.sum(np.log(np.diag(L))) + 0.5 * N * math.log(2 * math.pi)
    Ga = np.linalg.solve(L.T, np.linalg.solve(L, np.eye(N))) - np.outer(al, al)
    Lp, info = lapack.dpotrf(_device_K(spec, X, noise), lower=1, clean=1)
    assert info == 0
    W = lapack.dtrtri(Lp, lower=1)[0]
    beta = W.dot(Y)
    alb = W.T.dot(beta)
    nl_b = 0.5 * beta.dot(beta) + np.sum(np.log(np.diag(Lp))) + 0.5 * N * math.log(2 * math.pi)
    Gb = W.T.dot(W) - np.outer(alb, alb)
    return [(nl_a, np.array([np.sum(Ga * dK) / 2 for dK in dKs])), (nl_b, np.array([np.sum(Gb * dK) / 2 for dK in dKs]))]


def _nlml_problem(N, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.rand(N, d)
    return X, np.sin(2 * X).sum(axis=1) + 0.1 * rs.randn(N)


def _check_nlml(tag, spec, X, Y, noise, exact, results):
    """results: [(label, nlml, grad)] of the device against the longdouble values: within C x the larger error of the two FP64
    forms plus (N + 10) eps x the magnitude of the terms (N for the sums; 10 for the roundings every term takes on its own: the K
    entry, the pivot's square root and reciprocal, the products and the log).  Returns (failures, ratios)."""
    N = len(Y)
    nf = N + 10
    nl_s, g_s, sc, mag_nl = ho.marginal_likelihood(spec, X, Y, noise, exact)
    mag_nl = float(mag_nl)
    forms = _fp64_forms(spec, X, Y, noise, exact)
    e64 = max(abs(float(nl - nl_s)) for nl, _ in forms)
    eg64 = np.max([np.abs((g - g_s).astype(float)) for _, g in forms], axis=0)
    sc = sc.astype(float)
    bad, ratios = [], {}
    for label, nl, g in results:
        e = abs(float(nl - nl_s))
        ratios["nlml_" + label] = e / max(e64, 1e-300)
        if e > C * e64 + nf * EPS * mag_nl:
            bad.append("%s %s: nlml error %.3e, FP64 %.3e (floor %.3e)" % (tag, label, e, e64, nf * EPS * mag_nl))
        eg = np.abs((np.asarray(g, dtype=ho.LD) - g_s).astype(float))
        ratios["grad_" + label] = float(np.max(eg / np.maximum(eg64, 1e-300)))
        for h in np.nonzero(eg > C * eg64 + nf * EPS * sc)[0]:
            bad.append("%s %s: dnlml[%d] error %.3e, FP64 %.3e, scale %.3e" % (tag, label, h, eg[h], eg64[h], sc[h]))
    return bad, ratios


@pytest.mark.parametrize("N,name,noise", NLML_GRID)
def test_nlml_and_gradient_against_longdouble(N, name, noise, options):
    """both Cholesky schedules; the value-only call gives the bits of the value of the full call, and a second call the same bits
    (the fixed summation order of hyper.cu)"""
    from ibo_b200 import _lib
    kind, hyper, d, exact = _kind_case(name)
    X, Y = _nlml_problem(N, d, 100 * N + d)
    spec = orc.KernelSpec(kind, hyper, d)
    flags = _lib.FLAG_GRAD_EXACT if exact else 0
    res = []
    for pair in (0, 1):
        options("chol_pair", pair)
        nl, g = _lib.nlml(kind, hyper, X, Y, noise, flags=flags)
        nl2, g2 = _lib.nlml(kind, hyper, X, Y, noise, flags=flags)
        assert nl2 == nl and np.array_equal(g2, g), "two calls differ"
        assert _lib.nlml(kind, hyper, X, Y, noise, want_grad=False, flags=flags)[0] == nl
        res.append(("pair%d" % pair, nl, g))
    tag = "N=%d %s noise=%g" % (N, name, noise)
    bad, ratios = _check_nlml(tag, spec, X, Y, noise, exact, res)
    print("RATIO %s %s" % (tag, " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------
# c. the dimension sweep of the gradient kernel's shared memory (1024 d + 512 bytes: opt-in above 48 KiB, refused above 200 KiB)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [47, 48, 120, 199])
def test_gradient_kernel_across_dimensions(d):
    from ibo_b200 import _lib
    kind, hyper = orc.K_SE_ARD, [0.5 * math.sqrt(d) * (1 + 0.5 * t / d) for t in range(d)]
    X, Y = _nlml_problem(300, d, d)
    spec = orc.KernelSpec(kind, hyper, d)
    nl, g = _lib.nlml(kind, hyper, X, Y, 1e-3)
    bad, ratios = _check_nlml("d=%d" % d, spec, X, Y, 1e-3, False, [("dev", nl, g)])
    print("RATIO d=%d %s" % (d, " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
    assert not bad, "\n".join(bad)


def test_dimension_above_the_gradient_kernel_limit_is_refused():
    """d = 200 needs 205312 bytes of shared memory: refused with IBO_E_BADARG (the value alone has no such limit), and the library
    serves the next call normally"""
    from ibo_b200 import _lib
    X, Y = _nlml_problem(100, 200, 200)
    hyper = [8.0] * 200
    with pytest.raises(_lib.IBOError) as ei:
        _lib.nlml(_lib.KERNEL_SE_ARD, hyper, X, Y, 1e-3)
    assert ei.value.code == _lib.E_BADARG and "dimension too large" in str(ei.value)
    nl = _lib.nlml(_lib.KERNEL_SE_ARD, hyper, X, Y, 1e-3, want_grad=False)[0]
    assert abs(nl - orc.marginal_likelihood(orc.KernelSpec(orc.K_SE_ARD, hyper, 200), X, Y, 200, 1e-3, compute_gradient=False)) <= 1e-10 * abs(nl)
    X, Y = _nlml_problem(65, 3, 3)
    spec = orc.KernelSpec(orc.K_SE_ARD, [.4, .5, .6], 3)
    nl, g = _lib.nlml(orc.K_SE_ARD, spec.hyper, X, Y, 1e-3)
    bad, _ = _check_nlml("after refusal", spec, X, Y, 1e-3, False, [("dev", nl, g)])
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------
# d. the Python surface
# ---------------------------------------------------------------------------------------------
def test_python_surface_against_longdouble():
    from ibo_b200.gaussianprocess.kernel import GaussianKernel_ard, MaternKernel5
    from ibo_b200.gaussianprocess.trainhyper import dnlml, marginalLikelihood
    X, Y = _nlml_problem(300, 3, 77)
    hyper = [.5, .6, .7]
    spec = orc.KernelSpec(orc.K_SE_ARD, hyper, 3)
    for noise, (nl, g) in ((1e-6, marginalLikelihood(GaussianKernel_ard(hyper), X, Y, 3, noise=1e-6)),
                           (1e-3, (None, dnlml(np.log(hyper), GaussianKernel_ard, X, Y)))):      # dnlml: the default noise 1e-3
        res = [("py", nl if nl is not None else float(ho.marginal_likelihood(spec, X, Y, noise, gradient=False)), g)]
        bad, ratios = _check_nlml("python noise=%g" % noise, spec, X, Y, noise, False, res)
        print("RATIO python noise=%g %s" % (noise, " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
        assert not bad, "\n".join(bad)
    hk = KMAT["matern5"][1]
    k = MaternKernel5(hk)
    Xk = _kmat_points("matern5", 257)
    spec = orc.KernelSpec(orc.K_MATERN5, hk, 3)
    for which, got in ((-1, k.covMatrix(Xk)), (0, k.derivative(Xk, 0)), (1, k.derivative(Xk, 1))):
        ref = ho.cov_matrix(spec, Xk) if which < 0 else ho.kernel_derivative(spec, Xk, which)
        tol = _kmat_bound(spec, Xk, which, False) * np.abs(ref).astype(float) + TINY
        assert np.all(np.abs(got.astype(ho.LD) - ref).astype(float) <= tol), which


# ---------------------------------------------------------------------------------------------
# e. the Laplace fit
# ---------------------------------------------------------------------------------------------
PREF_THETA = [0.3, 0.35, 0.4]
# (N, P, noise, appended rows): P = 1, P < N, P > N; 37 and 200 are not multiples of BK = 16
PREF_GRID = [(14, 1, 0.1, 0), (14, 37, 1e-4, 0), (127, 37, 0.1, 0), (127, 300, 1e-4, 0), (128, 200, 1e-4, 0), (128, 1, 0.1, 0),
             (129, 100, 0.1, 29), (129, 250, 1e-4, 0), (600, 450, 1e-4, 0), (600, 900, 0.1, 100), (1100, 700, 1e-4, 0),
             (1100, 1300, 0.1, 0)]


def _pref_problem(N, P, seed):
    """winners from one half of the points, losers from the other (so a start can put every loser 10 above its winner), five
    points in no preference, degree weights 0 and 1, a repeated pair and a self-pair"""
    rs = np.random.RandomState(seed)
    X = rs.rand(N, 3)
    perm = rs.permutation(N - 5 if N > 10 else N)
    A, B = perm[:len(perm) // 2], perm[len(perm) // 2:]
    pr = [(int(rs.choice(A)), int(rs.choice(B)), int(rs.rand() < 0.3)) for _ in range(P)]
    if P >= 3:
        pr[1] = pr[0]
        pr[2] = (pr[2][0], pr[2][0], 1)
    v = np.array([p[0] for p in pr]); u = np.array([p[1] for p in pr])
    default = np.where(np.isin(np.arange(N), v), 0.5, -0.5)
    far = np.zeros(N)
    far[u] = 10.0
    far[v] = 0.0
    return X, pr, default, far


def _check_S(tag, S, y, pr, Lld, L64):
    """the returned S against the longdouble S at the returned y: within C x the error of FP64's evaluation there (orc.pref_S)
    plus N eps x the sum of the magnitudes of its terms"""
    N = len(y)
    Ss, mag = ho.pref_S_terms(y, pr, Lld)
    e, e64 = abs(float(S - Ss)), abs(float(orc.pref_S(y, pr, L64) - Ss))
    return ([] if e <= C * e64 + N * EPS * float(mag) else ["%s: S error %.3e, FP64 %.3e, terms %.3e" % (tag, e, e64, float(mag))]), \
        e / max(e64, 1e-300)


def _pref_model(X, noise, nappend):
    from ibo_b200 import _lib
    N = len(X)
    m = _lib.Model(_lib.KERNEL_SE_ARD, PREF_THETA, X[:N - nappend], np.zeros(N - nappend), noise)
    if nappend:
        m.append(X[N - nappend:], np.zeros(nappend))
    return m


@pytest.mark.parametrize("N,P,noise,nappend", PREF_GRID)
def test_laplace_fit_against_longdouble_fixed_point(N, P, noise, nappend, options):
    """both Cholesky schedules, the default start and a far start (every loser 10 above its winner: the 1e-10 guard, Hessian weights
    clipped to 0).  With the default gtol the fit ends with gnorm <= gtol, and maxit = the iterations it took gives the same bits.
    Run to rounding (gtol below reach, 100 steps), y is within ||y - y*|| <= C ||y64 - y*|| + N eps ||y*|| of the longdouble root
    y* of the gradient the device solves for, y64 the FP64 Newton on the same equations with LAPACK, also run to rounding (at
    gtol = 1e-9 the distance to y* is the stopping rule's, up to ~1e-10, not the arithmetic's); and S is checked at that y"""
    from ibo_b200 import _lib
    X, pr, default, far = _pref_problem(N, P, N + P)
    spec = orc.KernelSpec(orc.K_SE_ARD, PREF_THETA, 3)
    L64 = np.linalg.cholesky(orc.build_R(spec, X, noise))
    Lld = ho.cholesky(ho.bo.build_R(spec, X, noise))
    y64 = ho.pref_fit_f64(default, pr, L64, gtol=0.0, maxit=40)
    ys, res = ho.pref_fixed_point(y64, pr, Lld)
    ysf = ys.astype(float)
    e64 = float(np.max(np.abs(y64 - ys)))
    floor = N * EPS * float(np.max(np.abs(ys)))
    v, u, dg = [p[0] for p in pr], [p[1] for p in pr], [float(p[2]) for p in pr]
    bad, ratios = [], {}
    for pair in (0, 1):
        options("chol_pair", pair)
        m = _pref_model(X, noise, nappend)
        try:
            for sname, start in (("default", default), ("far", far)):
                tag = "N=%d P=%d noise=%g append=%d pair=%d start=%s" % (N, P, noise, nappend, pair, sname)
                y, S, gn, it = m.pref_fit(v, u, dg, start)
                if not gn <= 1e-9:
                    bad.append("%s: gnorm %.3e after %d iterations" % (tag, gn, it))
                y2, S2, gn2, it2 = m.pref_fit(v, u, dg, start, maxit=it)
                if not (np.array_equal(y2, y) and S2 == S and it2 == it):
                    bad.append("%s: maxit = %d (the iterations taken) does not give the same fit" % (tag, it))
                y, S, _, _ = m.pref_fit(v, u, dg, start, maxit=100, gtol=1e-300)
                e = float(np.max(np.abs(y - ysf)))
                ratios["y_%s_pair%d" % (sname, pair)] = e / max(e64, 1e-300)
                if e > C * e64 + floor:
                    bad.append("%s: |y - y*| = %.3e, FP64 %.3e, floor %.3e" % (tag, e, e64, floor))
                b, r = _check_S(tag, S, y, pr, Lld, L64)
                bad += b
                ratios["S_%s_pair%d" % (sname, pair)] = r
        finally:
            m.close()
    print("RATIO pref N=%d P=%d noise=%g res=%.1e %s" % (N, P, noise, float(res), " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
    assert not bad, "\n".join(bad)


# ---------------------------------------------------------------------------------------------
# f. a fit that takes no step
# ---------------------------------------------------------------------------------------------
def test_zero_step_fit_after_a_failed_build():
    """a fit whose start already meets gtol runs no factorisation, so the pivot it reports must come from a cleared flag, not
    from whatever a recycled allocation held -- such as the pivot of a model whose build failed just before"""
    from ibo_b200 import _lib
    N, P, noise = 128, 200, 0.1
    X, pr, default, _ = _pref_problem(N, P, 5)
    v, u, dg = [p[0] for p in pr], [p[1] for p in pr], [float(p[2]) for p in pr]
    m = _pref_model(X, noise, 0)
    try:
        assert m.pref_fit(v, u, dg, default)[2] <= 1e-9
        Xd = np.array([[0.1, 0.2], [0.1, 0.2], [0.5, 0.5]])          # duplicate point, no noise: K is singular
        with pytest.raises(np.linalg.LinAlgError) as ei:
            _lib.nlml(_lib.KERNEL_SE_ARD, [1., 1.], Xd, [1., 2., 3.], 0.0)
        assert ei.value.pivot > 0
        y, S, gn, it = m.pref_fit(v, u, dg, default, gtol=1e30)
        assert it == 0
        Ld, Wd = m.matrix(1).astype(ho.LD), m.matrix(2).astype(ho.LD)
        want = Ld @ (Wd @ default.astype(ho.LD))
        tol = 2 * N * EPS * (np.abs(Ld) @ (np.abs(Wd) @ np.abs(default))).astype(float)
        assert np.all(np.abs((y - want).astype(float)) <= tol)
        spec = orc.KernelSpec(orc.K_SE_ARD, PREF_THETA, 3)
        bad, _ = _check_S("zero step", S, y, pr, ho.cholesky(ho.bo.build_R(spec, X, noise)),
                          np.linalg.cholesky(orc.build_R(spec, X, noise)))
        assert not bad, "\n".join(bad)
    finally:
        m.close()
