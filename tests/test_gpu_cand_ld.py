"""GPU tests of the candidate-side paths (joint.cu: ibo_posterior_cov / ibo_posterior_sample; grad.cu: ibo_posterior_grad /
ibo_score_grad; qei.cu: ibo_qei) against the extended-precision reference (tests/build_oracle.py), across dimensions on both
sides of the 16-dimension slabs of the gradient reduction, noise down to 1e-6, q-EI batch shapes and sample counts, and the
Cholesky of the joint covariance at 47 to 49 block columns and at the 16384-candidate cap.

The tolerance model is the build test's: the device's error against the longdouble result must stay within C = 4 times the error
of an FP64 yardstick on the same problem, plus a floor of a few eps scaled to the quantity.  The yardstick is the FP64 oracle
(joint_oracle, grad_oracle, qei_oracle).  The device forms an explicit W = inv(L), which at small noise loses more than a
substitution does, so the yardstick is the larger of two errors: the oracle's, and that of the same formulas with every solve
against L replaced by a product with LAPACK's W (dtrtri).  Each case prints one RATIO line: device error over yardstick error."""
import contextlib

import numpy as np
import pytest
from scipy.linalg import blas, lapack

import build_oracle as bo
import grad_oracle as go
import joint_oracle as jo
import qei_oracle as qo
from oracle import ibo_oracle as orc

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps
C = 4.0
FLOORS = {"py": 10e-8, "cpp": 1e-8}               # sigma^2 clipping floors of the two modes; both clip at 10 from above


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


def _lib():
    from ibo_b200 import _lib as L
    return L


@contextlib.contextmanager
def _explicit_inverse(o, W):
    """the FP64 oracles' formulas with every triangular solve against o.L or o.augL replaced by a product with the inverse W[k] of
    that factor (k = 0: o.L, 1: o.augL), as the device computes them: inv(L) B -> W B, inv(L)^T B -> W^T B (the oracles import
    solve_triangular when called)"""
    import scipy.linalg
    inv = {id(F): Wk for F, Wk in zip((o.L, o.augL), W) if F is not None}
    real = scipy.linalg.solve_triangular

    def solve(F, B, lower=False, trans=0, **kw):
        Wk = inv.get(id(F))
        if Wk is None:
            return real(F, B, lower=lower, trans=trans, **kw)
        return (Wk.T if trans in ("T", 1) else Wk).dot(B)
    scipy.linalg.solve_triangular = solve
    try:
        yield
    finally:
        scipy.linalg.solve_triangular = real


def _yardsticks(c, f):
    """f(o) evaluated by the FP64 oracle as written, with LAPACK's W (dtrtri) and with the W the device's build produced (tested
    against LAPACK's by tests/test_gpu_build.py): the last keeps the build's own error, within its test's bound, out of what is
    measured here"""
    out = [f(c.o)]
    for W in (c.W_lapack, c.W_dev):
        with _explicit_inverse(c.o, W):
            out.append(f(c.o))
    return out


class Case(object):
    """one problem on the device and in both references: spec, X, Y, noise, prior, variance model (aug); .m the device model, .o the
    FP64 oracle, .ld the longdouble factors"""

    def __init__(self, spec, X, Y, noise, prior=None, aug_pts=None, seed=0):
        L = _lib()
        self.spec, self.X, self.Y, self.noise, self.prior = spec, X, Y, noise, prior
        N, d = X.shape
        self.m = L.Model(spec.kind, spec.hyper, X, Y, noise, prior=prior)
        self.o = orc.GPOracle(spec, X, Y, noise, prior=prior)
        self.aug = None
        self.vm = None
        if aug_pts is not None:
            augX = np.r_[X, aug_pts]
            na = len(augX)
            A = np.random.RandomState(seed).randn(N, N) * 0.05
            pad = np.zeros((na, na))
            pad[:N, :N] = np.linalg.inv(np.eye(N) * 5 + A.dot(A.T))
            self.vm = L.Model(spec.kind, spec.hyper, augX, np.zeros(na), noise, Cinv=pad)
            self.m.set_variance_model(self.vm)
            self.aug = (augX, bo.build_R(spec, augX, noise) + pad)
            self.o.augX, self.o.augL = augX, np.linalg.cholesky(orc.build_R(spec, augX, noise) + pad)
        self.ld = bo._Model(spec, X, Y, noise, prior, self.aug)
        facs = [self.o.L] + ([self.o.augL] if self.vm is not None else [])
        self.W_lapack = [lapack.dtrtri(F, lower=1)[0] for F in facs]
        self.W_dev = [self.m.matrix(2)] + ([self.vm.matrix(2)] if self.vm is not None else [])

    def close(self):
        self.m.close()
        if self.vm is not None:
            self.vm.close()


def _err(a, ref):
    return float(np.max(np.abs(np.asarray(a, dtype=bo.LD) - ref))) if np.size(a) else 0.0


def _compare(bad, ratios, tag, name, dev, ref, yard, floor):
    """device error <= C x the largest yardstick error + floor (all against the longdouble ref); the ratio is recorded against all
    three yardsticks (name) and against the substitution and LAPACK's W alone (name/lp)"""
    errs = [_err(y, ref) for y in yard]
    e, ey = _err(dev, ref), max(errs)
    ratios[name] = e / max(ey, 1e-300)
    ratios[name + "/lp"] = e / max(max(errs[:2]), 1e-300)
    if not e <= C * ey + floor:
        bad.append("%s %s: device error %.3e, FP64 yardstick %.3e, floor %.3e" % (tag, name, e, ey, floor))


def _scale(x):
    return float(np.max(np.abs(np.asarray(x, dtype=float)))) if np.size(x) else 0.0


def _report(tag, ratios, bad):
    print("RATIO %s %s" % (tag, " ".join("%s=%.2f" % kv for kv in sorted(ratios.items()))))
    assert not bad, "\n".join(bad)


def _candidates(X, M, rs):
    """M random points, 8 of them on training points and 8 within 1e-5 of one"""
    N, d = X.shape
    Xs = rs.rand(M, d)
    k = min(8, N)
    Xs[:k] = X[:k]
    Xs[8:8 + k] = X[N - k:] + 1e-5 * (2 * rs.rand(k, d) - 1)
    return Xs


# -- gradients ---------------------------------------------------------------------------------------------------------------------

def _check_grad(c, Xs, tag, bad, ratios, acqs=((orc.ACQ_EI, 0.01), (orc.ACQ_PI, 0.01), (orc.ACQ_UCB, 1.3))):
    """posterior_grad and score_grad in both modes against the longdouble gradient; candidates whose longdouble sigma^2 lies in
    the error band of a clipping floor are left out (on either side of it the device rightly returns 0 or a nonzero ds2)"""
    L = _lib()
    N = len(c.Y)
    mu_l, s2_l, dmu_l, ds2_l = bo.posterior_grad(c.spec, c.X, c.Y, c.noise, Xs, model=c.ld)
    ymax = float(np.max(c.Y))
    for mode in ("py", "cpp"):
        fl = L.FLAG_MODE_PY if mode == "py" else L.FLAG_MODE_CPP
        floor = FLOORS[mode]
        mu, s2, dmu, ds2 = c.m.posterior_grad(Xs, fl)
        ys = _yardsticks(c, lambda o: go.posterior_grad(o, Xs, mode))
        e_s2 = max(_err(np.clip(y[1], floor, 10), np.clip(s2_l, floor, 10)) for y in ys)
        band = C * e_s2 + N * EPS
        keep = (np.abs(s2_l - floor) > band) & (np.abs(s2_l - 10) > band)
        clipped = (s2_l <= floor) | (s2_l >= 10)
        ds2_lc = np.where(clipped[:, None], 0, ds2_l)
        t = "%s %s" % (tag, mode)
        _compare(bad, ratios, t, "dmu_" + mode, dmu[keep], dmu_l[keep], [y[2][keep] for y in ys], N * EPS * _scale(dmu_l))
        _compare(bad, ratios, t, "ds2_" + mode, ds2[keep], ds2_lc[keep], [y[3][keep] for y in ys], N * EPS * _scale(ds2_l))
        mu_f, s2_f = mu_l.astype(float), np.clip(s2_l, floor, 10).astype(float)
        for acq, parm in acqs:
            sc, dsc = c.m.score_grad(Xs, acq, ymax, parm, fl)
            a_mu, a_s = go.acq_partials(acq, mode, mu_f, s2_f, ymax, parm)
            dsc_l = np.asarray(a_mu, dtype=bo.LD)[:, None] * dmu_l + np.asarray(a_s / (2 * np.sqrt(s2_f)), dtype=bo.LD)[:, None] * ds2_lc
            ysc = _yardsticks(c, lambda o: go.score_grad(o, Xs, acq, ymax, parm, mode)[1])
            # the acquisitions' CDFs have only absolute accuracy (DESIGN.md section 5 compares EI with a floor of 1e-5): far in the
            # tail the score's gradient is that small a fraction of the posterior's
            _compare(bad, ratios, t, "dsc%d_%s" % (acq, mode), dsc[keep], dsc_l[keep], [y[keep] for y in ysc],
                     N * EPS * max(_scale(dsc_l), 1e-5 * (_scale(dmu_l) + _scale(ds2_l))))
        assert np.sum(keep) >= len(Xs) // 2


# -- joint posterior ---------------------------------------------------------------------------------------------------------------

def _check_cov(c, Xs, tag, bad, ratios):
    N = len(c.Y)
    mu, Sig = c.m.posterior_cov(Xs)
    mu_l, Sig_l = bo.posterior_joint(c.spec, c.X, c.Y, c.noise, Xs, model=c.ld)
    ys = _yardsticks(c, lambda o: jo.posterior_joint(o, Xs))
    _compare(bad, ratios, tag, "mu_cov", mu, mu_l, [y[0] for y in ys], N * EPS * max(1.0, _scale(mu_l)))
    _compare(bad, ratios, tag, "Sigma", Sig, Sig_l, [y[1] for y in ys], N * EPS * (1 + c.noise))
    if not np.array_equal(Sig, Sig.T):
        bad.append("%s: Sigma is not exactly symmetric" % tag)
    return Sig_l, ys


def _check_sample(c, Xs, jitter, Sig_l, ys, tag, bad, ratios):
    """F = mu + chol(Sigma + jitter I) Z against the longdouble factor; where FP64 cannot factor the device's own Sigma + jitter I
    either, the device must report it rather than return samples"""
    L = _lib()
    M = len(Xs)
    Z = np.random.default_rng(M).standard_normal((M, 9))
    try:
        F, am = c.m.posterior_sample(Xs, Z, jitter)
    except L.NotPositiveDefinite:
        _, Sig = c.m.posterior_cov(Xs)
        if lapack.dpotrf(Sig + jitter * np.eye(M), lower=1)[1] == 0:
            bad.append("%s jitter=%g: the device reports an indefinite Sigma that LAPACK factorises" % (tag, jitter))
        ratios["F_j%g" % jitter] = float("nan")
        return
    mu_l = c.ld.mean(Xs)[0]
    F_l = mu_l[:, None] + bo.cholesky(Sig_l + bo.LD(jitter) * np.eye(M, dtype=bo.LD)) @ np.asarray(Z, dtype=bo.LD)
    Fy = []
    for mu_y, Sig_y in ys:
        Lf, info = lapack.dpotrf(Sig_y + jitter * np.eye(M), lower=1, clean=1)
        Fy.append(mu_y[:, None] + Lf.dot(Z) if info == 0 else np.full_like(Z, np.inf))
    _compare(bad, ratios, tag, "F_j%g" % jitter, F, F_l, Fy, M * EPS * _scale(F_l))
    if not np.array_equal(am, np.argmax(F, axis=0)):
        bad.append("%s jitter=%g: argmax is not the samples' own" % (tag, jitter))


# -- q-EI --------------------------------------------------------------------------------------------------------------------------

def _check_qei(c, Xb, Z, ymax, xi, jitter, tag, bad, ratios, min_keep):
    """values always; gradients on the batches whose longdouble margins (gap between the two largest draws, |improvement|) exceed
    C x the FP64 error of the draws, where the argmax and the sign of the improvement are the same for every FP64 evaluation"""
    N = len(c.Y)
    B, q, d = Xb.shape
    v, G, nbad = c.m.qei(Xb, Z, ymax, xi, jitter)
    if nbad:
        bad.append("%s: %d batches reported not positive definite" % (tag, nbad))
        return
    v_l, G_l, gap, imp = bo.qei(c.spec, c.X, c.Y, c.noise, Xb, Z, ymax, xi, jitter, model=c.ld)
    ys = _yardsticks(c, lambda o: qo.qei(o, Xb, Z, ymax, xi, jitter))
    _compare(bad, ratios, tag, "qei", v, v_l, [y[0] for y in ys], (N + Z.shape[1]) * EPS * max(_scale(v_l), EPS))
    # the FP64 error of the draws F = mu + L Z of each batch, from both yardsticks' mu and Sigma
    P = Xb.reshape(-1, d)
    mu_l, Sig_l = bo.posterior_joint(c.spec, c.X, c.Y, c.noise, P, model=c.ld)
    Zl = np.asarray(Z, dtype=bo.LD)
    fy = _yardsticks(c, lambda o: jo.posterior_joint(o, P))
    eF = np.zeros(B)
    for b in range(B):
        s = slice(b * q, (b + 1) * q)
        F_l = mu_l[s, None] + bo.cholesky(Sig_l[s, s] + bo.LD(jitter) * np.eye(q, dtype=bo.LD)) @ Zl
        for mu_y, Sig_y in fy:
            F_y = mu_y[s, None] + np.linalg.cholesky(Sig_y[s, s] + jitter * np.eye(q)).dot(Z)
            eF[b] = max(eF[b], _err(F_y, F_l))
    keep = (np.minimum(gap, imp) > C * eF + 1e-12) & (np.asarray(v_l, dtype=float) > 0)
    ratios["kept"] = float(np.sum(keep))
    if np.sum(keep) < min_keep:
        bad.append("%s: %d batches away from the kinks, %d wanted" % (tag, np.sum(keep), min_keep))
        return
    _compare(bad, ratios, tag, "dqei", G[keep], G_l[keep], [y[1][keep] for y in ys], N * EPS * _scale(G_l[keep]))


# -- a. dimensions -----------------------------------------------------------------------------------------------------------------

def _ard_theta(d):
    """length scales that differ per dimension and grow like sqrt(d): scaled distances between random points stay O(1)"""
    return 0.4 * np.sqrt(d) * (0.6 + 0.8 * np.arange(d) / max(d - 1, 1))


def _dim_spec(kind, d):
    th = _ard_theta(d)
    if kind == orc.K_SE_ARD:
        return orc.KernelSpec(kind, th, d)
    if kind == orc.K_MATERN5_ARD:
        return orc.KernelSpec(kind, np.r_[th, 0.95], d)
    return orc.KernelSpec(kind, [0.4 * np.sqrt(d), 0.9], d)        # isotropic Matern-3/2


DIMS = [1, 15, 16, 17, 31, 32, 33, 63, 64]


@pytest.mark.parametrize("N", [129, 300])
@pytest.mark.parametrize("kind", [orc.K_SE_ARD, orc.K_MATERN5_ARD, orc.K_MATERN3])
@pytest.mark.parametrize("d", DIMS)
def test_gradients_across_dimensions(d, kind, N):
    rs = np.random.RandomState(100 * d + 10 * kind + N)
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1) / np.sqrt(d)
    c = Case(_dim_spec(kind, d), X, Y, 0.1)
    tag = "dims d=%d kind=%d N=%d" % (d, kind, N)
    bad, ratios = [], {}
    try:
        _check_grad(c, _candidates(X, 97, rs), tag, bad, ratios)
        if d in (17, 64):
            _check_cov(c, _candidates(X, 161, rs), tag, bad, ratios)
            Xb = rs.rand(6, 4, d)
            Xb[0, 1] = X[3]
            _check_qei(c, Xb, np.random.default_rng(d).standard_normal((4, 64)), float(np.percentile(Y, 60)), 0.01, 0.0, tag,
                       bad, ratios, 3)
    finally:
        c.close()
    _report(tag, ratios, bad)


@pytest.mark.parametrize("extra", ["prior", "variance_model"])
@pytest.mark.parametrize("d", [17, 33, 64])
def test_gradient_launches_with_prior_and_variance_model_above_16_dims(d, extra):
    """the reductions <true,true,true> (prior) and <true,false,false> over the variance model then <false,true,*> over the model"""
    rs = np.random.RandomState(7 * d + len(extra))
    N = 129
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1) / np.sqrt(d)
    spec = _dim_spec(orc.K_MATERN5_ARD, d)
    if extra == "prior":
        c = Case(spec, X, Y, 0.1, prior=orc.PriorSpec(rs.rand(4, d), 0.5 * rs.randn(4), 3.0 / d, np.zeros(d), np.ones(d)))
    else:
        c = Case(spec, X, Y, 0.1, aug_pts=rs.rand(3, d), seed=d)
    tag = "launch d=%d %s" % (d, extra)
    bad, ratios = [], {}
    try:
        _check_grad(c, _candidates(X, 97, rs), tag, bad, ratios)
        Xb = rs.rand(6, 3, d)
        _check_qei(c, Xb, np.random.default_rng(d).standard_normal((3, 64)), float(np.percentile(Y, 60)), 0.01, 0.0, tag,
                   bad, ratios, 3)
    finally:
        c.close()
    _report(tag, ratios, bad)


# -- b. small noise ----------------------------------------------------------------------------------------------------------------

SMALL_KINDS = {
    "se_ard_long": (orc.K_SE_ARD, [1.0, 1.5, 2.0]),       # long length scales: the ill-conditioned case of the build test
    "matern5_prior": (orc.K_MATERN5, [0.5, 1.0]),          # with the RBF prior mean
}
SMALL = [(300, name, nz) for name in SMALL_KINDS for nz in (0.1, 1e-3, 1e-4, 1e-6)] + [(1100, "se_ard_long", 1e-6)]


@pytest.mark.parametrize("N,name,noise", SMALL)
def test_candidate_paths_at_small_noise(N, name, noise):
    kind, hyper = SMALL_KINDS[name]
    rs = np.random.RandomState(N + int(-np.log10(noise)))
    d = 3
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1) + 0.1 * rs.randn(N)
    prior = orc.PriorSpec(rs.rand(4, d), 0.3 * rs.randn(4), 3.0, np.zeros(d), np.ones(d)) if name == "matern5_prior" else None
    c = Case(orc.KernelSpec(kind, hyper, d), X, Y, noise, prior=prior)
    tag = "small N=%d %s noise=%g" % (N, name, noise)
    bad, ratios = [], {}
    try:
        Xs = _candidates(X, 333, rs)
        Sig_l, ys = _check_cov(c, Xs, tag, bad, ratios)
        for jitter in (0.0, 1e-8):
            _check_sample(c, Xs, jitter, Sig_l, ys, tag, bad, ratios)
        _check_grad(c, Xs[:161], tag, bad, ratios, acqs=((orc.ACQ_EI, 0.01),))
        # q-EI batches with near-duplicate points (1e-5 apart): Sigma_b is conditioned at the noise level
        Xb = rs.rand(8, 4, d)
        Xb[:4, 1] = Xb[:4, 0] + 1e-5 * (2 * rs.rand(4, d) - 1)
        Xb[4, 2] = X[5]
        _check_qei(c, Xb, np.random.default_rng(N).standard_normal((4, 256)), float(np.percentile(Y, 60)), 0.01, 1e-8, tag,
                   bad, ratios, 3)
    finally:
        c.close()
    _report(tag, ratios, bad)


# -- c. q-EI shapes ----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("S", [1, 3, 5, 1023])
@pytest.mark.parametrize("q", [1, 2, 3, 8, 17, 31, 32])
def test_qei_batch_shapes(q, S):
    """lane masking (lane < q), the pair -> (j, l) unpacking of the Sigma kernel (up to 17 items a thread) and the sample loop's
    stride of four warps (S not a multiple of 4: some warps take one sample fewer)"""
    rs = np.random.RandomState(10 * q + S)
    N, d = 129, 3
    X = rs.rand(N, d)
    Y = np.sin(3 * X).sum(axis=1)
    c = Case(orc.KernelSpec(orc.K_MATERN5_ARD, [.3, .4, .5, .95], d), X, Y, 0.1)
    tag = "qei q=%d S=%d" % (q, S)
    bad, ratios = [], {}
    try:
        B = 12
        Xb = rs.rand(B, q, d)
        Xb[0, 0] = X[0]
        ymax = float(np.percentile(Y, 30 if S < 5 else 60))
        _check_qei(c, Xb, np.random.default_rng(q * S).standard_normal((q, S)), ymax, 0.01, 0.0, tag, bad, ratios, 4)
    finally:
        c.close()
    _report(tag, ratios, bad)


# -- d. the joint factor at large M ------------------------------------------------------------------------------------------------

def _zero_mean_model(M, seed):
    """Y = 0 and no prior: mu = 0 exactly, so posterior_sample with Z = D = diag(+-1) returns F = chol(Sigma) D exactly (each entry
    is one product by +-1 plus exact zeros, and the bias added is 0)"""
    L = _lib()
    rs = np.random.RandomState(seed)
    N, d = 200, 3
    X = rs.rand(N, d)
    m = L.Model(orc.K_MATERN5, [0.3, 1.0], X, np.zeros(N), 0.1)
    return m, rs.rand(M, d)


def _signs(M):
    D = np.ones(M)
    D[1::2] = -1.0                                   # negated columns: zeros above the diagonal, -L_ss < 0 on it
    D[-1] = -1.0                                     # the last column is all zeros but its negative diagonal: a tie at row 0
    return D


@pytest.mark.parametrize("M", [6016, 6017, 6272])
def test_joint_factor_schedules_at_47_to_49_block_columns(M, options):
    """the invert-free Cholesky of ibo_posterior_sample at 47, 48 and 49 block columns under each schedule: F exactly triangular
    with the right signs on the diagonal, the default schedule bit for bit the paired one from 48 block columns on, the backward
    error as small as LAPACK's on the device's own Sigma, and argmax NumPy's first argmax (a negated column whose entries below the
    diagonal are all negative ties at its exact zeros above it)"""
    m, Xs = _zero_mean_model(M, M)
    D = _signs(M)
    F = {}
    try:
        _, Sig = m.posterior_cov(Xs)
        for pair in (-1, 0, 1):
            options("chol_pair", pair)
            f, am = m.posterior_sample(Xs, np.diag(D))
            F[pair] = f
            assert np.array_equal(am, np.argmax(f, axis=0)), "chol_pair=%d: argmax" % pair
    finally:
        m.close()
    nb = (M + 127) // 128
    same = 1 if nb >= 48 else 0
    assert np.array_equal(F[-1], F[same]), "default factor at %d block columns is not chol_pair=%d bit for bit" % (nb, same)
    assert not np.array_equal(F[-1], F[1 - same])
    ties = int(np.sum(np.max(F[-1], axis=0) == 0.0))
    assert ties >= 1                                  # the tie-break ran
    Lp, info = lapack.dpotrf(Sig, lower=1, clean=1)
    assert info == 0
    bp = np.linalg.norm(Sig - blas.dtrmm(1.0, Lp, np.ascontiguousarray(Lp.T), lower=1)) / np.linalg.norm(Sig)
    for pair in (0, 1):
        Lf = F[pair] * D[None, :]
        assert np.array_equal(np.triu(Lf, 1), np.zeros_like(Lf)) and np.all(np.diag(Lf) > 0)
        bd = np.linalg.norm(Sig - blas.dtrmm(1.0, Lf, np.ascontiguousarray(Lf.T), lower=1)) / np.linalg.norm(Sig)
        print("RATIO joint M=%d chol_pair=%d backward=%.2f (%.2e / %.2e) ties=%d" % (M, pair, bd / bp, bd, bp, ties))
        assert bd <= C * bp + EPS


def test_joint_factor_at_the_candidate_cap():
    """M = 16384: the backward error through random probes, |Sigma x - F (F^T x)| / (|Sigma|_F |x|) <= M eps"""
    M = 16384
    m, Xs = _zero_mean_model(M, 5)
    D = _signs(M)
    try:
        _, Sig = m.posterior_cov(Xs)
        F, am = m.posterior_sample(Xs, np.diag(D))
    finally:
        m.close()
    assert np.array_equal(am, np.argmax(F, axis=0))
    Lf = F * D[None, :]
    del F
    assert np.all(np.diag(Lf) > 0) and not np.any(np.triu(Lf[:512], 1)) and not np.any(np.triu(Lf[-512:], M - 512 + 1))
    x = np.random.RandomState(6).randn(M, 4)
    r = np.linalg.norm(Sig.dot(x) - Lf.dot(Lf.T.dot(x)), axis=0) / (np.linalg.norm(Sig) * np.linalg.norm(x, axis=0))
    print("RATIO joint M=%d probe backward %s (bound %.2e)" % (M, " ".join("%.2e" % v for v in r), M * EPS))
    assert np.all(r <= M * EPS)
