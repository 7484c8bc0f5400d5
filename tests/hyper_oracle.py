"""Extended-precision reference of the hyperparameter and preference paths (test infrastructure only): a plain NumPy restatement
in np.longdouble of Kernel.covMatrix / Kernel.derivative, of the marginal likelihood and its gradient, and of the Laplace MAP fit
of PrefGaussianProcess.  The formulas are those of oracle/ibo_oracle.py (cov_matrix, kernel_derivative, marginal_likelihood,
pref_S); the FP64 hyperparameters, noise and constants are part of the problem, as in tests/build_oracle.py, whose Cholesky,
triangular inverse and substitution this reuses."""
import math

import numpy as np

import build_oracle as bo
from oracle import ibo_oracle as orc

LD = bo.LD
cholesky, tri_inv, forward_solve, back_solve, rel = bo.cholesky, bo.tri_inv, bo.forward_solve, bo.back_solve, bo.rel


def nlen(kernel):
    """number of length-scale hyperparameters (d for the ARD kinds, else 1)"""
    return kernel.ndim if kernel.kind in (orc.K_SE_ARD, orc.K_MATERN5_ARD) else 1


def n_hyper(kernel):
    """hyperparameters with a derivative: the length scales, then the magnitude where the kind has one"""
    return nlen(kernel) + (1 if kernel.kind != orc.K_SE_ISO and len(kernel.hyper) > nlen(kernel) else 0)


def cov_matrix(kernel, X):
    """covMatrix(X): k(X_i, X_j) with the FP64 sf2 on the diagonal (the SE-ARD length scales are the clipped kernel.theta)"""
    K = bo.cross(kernel, X, X)
    np.fill_diagonal(K, LD(kernel.sf2))
    return K


class _Pieces(object):
    """what every derivative of one (kernel, X) reads: K, the scaled differences D[i, j, t] = (x_it - x_jt) / theta_t and r^2"""

    def __init__(self, kernel, X):
        self.K = cov_matrix(kernel, X)
        X = np.asarray(X, dtype=LD)
        self.U = X[:, None, :] - X[None, :, :]          # unscaled differences (the Matern-3/2 reference expression)
        self.D = self.U / np.asarray(kernel.theta, dtype=LD)
        self.r2 = np.sum(self.D * self.D, axis=2)


def kernel_derivative(kernel, X, hp, exact_matern3=False, pieces=None):
    """dK / d log(hyper[hp]) in longdouble: the expressions of orc.kernel_derivative"""
    p = pieces if pieces is not None else _Pieces(kernel, X)
    kind, nl, sf2 = kernel.kind, nlen(kernel), LD(kernel.sf2)
    if hp == nl and kind != orc.K_SE_ISO and len(kernel.hyper) > nl:
        return 2 * p.K
    if hp < 0 or hp >= nl:
        raise ValueError("kernel has no hyperparameter %d" % hp)
    if kind == orc.K_SE_ISO:
        return p.K * p.r2
    if kind == orc.K_SE_ARD:
        return p.K * p.D[:, :, hp] ** 2
    if kind == orc.K_MATERN3:
        if exact_matern3:
            z = np.sqrt(LD(3)) * np.sqrt(p.r2)
            return sf2 * z * z * np.exp(-z)
        r = np.sqrt(np.sum(p.U * p.U, axis=2))                     # kernel.py:217-222: not divided by theta
        return sf2 * r * r * np.exp(-r)
    s = np.sqrt(LD(5)) * np.sqrt(p.r2)
    if kind == orc.K_MATERN5:
        return sf2 * (s * s + s * s * s) * np.exp(-s) / 3
    return sf2 * LD(5) / 3 * (1 + s) * np.exp(-s) * p.D[:, :, hp] ** 2


def gram(W, nb=128):
    """W^T W of a lower triangular W, block row by block row over the columns it reaches (a third of the full product)"""
    n = W.shape[0]
    G = np.zeros((n, n), dtype=LD)
    for k0 in range(0, n, nb):
        k1 = min(k0 + nb, n)
        B = np.ascontiguousarray(W[k0:k1, :k1], dtype=LD)
        G[:k1, :k1] += np.ascontiguousarray(B.T) @ B
    return G


def marginal_likelihood(kernel, X, Y, noise, exact_matern3=False, gradient=True):
    """(nlml, dnlml[nh], scale[nh], magnitude of nlml's terms) of K = covMatrix(X) + noise I, all in longdouble; the diagonal is the FP64 sf2 + noise the
    library puts there.  nlml = Y.alpha / 2 + sum log L_ii + N log(2 pi) / 2; dnlml_h = sum (inv(K) - alpha alpha^T) o dK_h / 2 with
    inv(K) = W^T W, W = inv(L); scale_h = sum |(inv(K) - alpha alpha^T) o dK_h| / 2 (the magnitude of the terms); the
    magnitude of nlml's terms is Y.alpha / 2 + sum |log L_ii| + N log(2 pi) / 2."""
    Y = np.asarray(Y, dtype=LD)
    N = len(Y)
    K = cov_matrix(kernel, X)
    np.fill_diagonal(K, LD(kernel.sf2 + noise))
    L = cholesky(K)
    beta = forward_solve(L, Y)
    logd, log2pi = np.log(np.diag(L)), np.log(8 * np.arctan(LD(1)))
    nl = beta @ beta / 2 + np.sum(logd) + N * log2pi / 2
    if not gradient:
        return nl
    W = tri_inv(L)
    alpha = W.T @ beta
    G = gram(W) - np.outer(alpha, alpha)
    p = _Pieces(kernel, X)
    nh = n_hyper(kernel)
    g, sc = np.zeros(nh, dtype=LD), np.zeros(nh, dtype=LD)
    for h in range(nh):
        T = G * kernel_derivative(kernel, X, h, exact_matern3, pieces=p)
        g[h], sc[h] = np.sum(T) / 2, np.sum(np.abs(T)) / 2
    return nl, g, sc, beta @ beta / 2 + np.sum(np.abs(logd)) + N * log2pi / 2


# ---------------------------------------------------------------------------------------------
# Laplace fit of PrefGaussianProcess: the functional of orc.pref_S and the equations ibo_pref_fit solves (laplace.cu:19-50)
# ---------------------------------------------------------------------------------------------
_NR = [LD(c) for c in orc._NR]
SQRT2 = LD(1.4142135623730951)           # the FP64 constants of the device are part of the problem
INV_SQRT2 = LD(0.7071067811865476)
INV_SQRT2PI = LD(0.3989422804014327)
GUARD = LD(1e-10)


def erf_nr(z):
    """the Numerical-Recipes Chebyshev erf of the reference (orc.erf_py) in longdouble"""
    z = np.asarray(z, dtype=LD)
    t = 1 / (1 + np.abs(z) / 2)
    p = _NR[9]
    for c in _NR[8:0:-1]:
        p = c + t * p
    ans = 1 - t * np.exp(-z * z + _NR[0] + t * p)
    return np.where(z >= 0, ans, -ans)


def cdf(z):
    """the reference's CDF with its truncated constant 0.707106"""
    return (1 + erf_nr(np.asarray(z, dtype=LD) * LD(0.707106))) / 2


def _prefs(prefinds):
    v = np.array([p[0] for p in prefinds], dtype=int)
    u = np.array([p[1] for p in prefinds], dtype=int)
    dp1 = np.array([p[2] for p in prefinds], dtype=LD) + 1
    return v, u, dp1


def _terms(y, prefinds):
    """per preference: z, the log term (d + 1) log(cdf + 1e-10), dS/d(y_v - y_u) and the clipped curvature weight"""
    v, u, dp1 = _prefs(prefinds)
    z = (y[v] - y[u]) / SQRT2
    c = cdf(z) + GUARD
    q = np.exp(-z * z / 2) * INV_SQRT2PI / c
    w = dp1 * (z * q + q * q) / 2
    return v, u, dp1 * np.log(c), -dp1 * q * INV_SQRT2, np.where(w > 0, w, 0)


def pref_S_terms(y, prefinds, L):
    """(S, sum of the magnitudes of its terms) at y in longdouble; L: the lower factor of R (any precision)"""
    y = np.asarray(y, dtype=LD)
    _, _, lt, _, _ = _terms(y, prefinds)
    a = forward_solve(L, y)
    q = a @ a / 2
    return -np.sum(lt) + q, np.sum(np.abs(lt)) + q


def pref_S(y, prefinds, L):
    return pref_S_terms(y, prefinds, L)[0]


def pref_grad(y, prefinds, L):
    """g(y) = sum_p dS/d(delta_p) (e_v - e_u) + inv(R) y in longdouble"""
    y = np.asarray(y, dtype=LD)
    v, u, _, gd, _ = _terms(y, prefinds)
    g = np.zeros(len(y), dtype=LD)
    np.add.at(g, v, gd)
    np.add.at(g, u, -gd)
    return g + back_solve(L, forward_solve(L, y))


def pref_fit_f64(start, prefinds, L, gtol=1e-13, maxit=200):
    """the FP64 yardstick: damped Newton in whitened coordinates with LAPACK (the device's algorithm), from `start`; L: the FP64
    factor of R.  Returns y."""
    from scipy.linalg import cho_factor, cho_solve, solve_triangular
    L = np.asarray(L, dtype=float)
    a = solve_triangular(L, np.asarray(start, dtype=float), lower=True)

    def ev(a):
        y = L @ a
        v, u, dp1 = _prefs(prefinds)
        z = (y[v] - y[u]) / math.sqrt(2)
        c = orc.cdf_py(z) + 1e-10
        q = np.exp(-z * z / 2) * 0.3989422804014327 / c
        gl = np.zeros(len(y))
        gd = -dp1.astype(float) * q * 0.7071067811865476
        np.add.at(gl, v, gd)
        np.add.at(gl, u, -gd)
        w = np.maximum(dp1.astype(float) * (z * q + q * q) / 2, 0)
        return -np.sum(dp1.astype(float) * np.log(c)) + a @ a / 2, L.T @ gl + a, w
    S, g, w = ev(a)
    v, u, _ = _prefs(prefinds)
    for _ in range(maxit):
        if np.max(np.abs(g)) <= gtol:
            break
        G = (L[v] - L[u]).T * np.sqrt(w)
        da = -cho_solve(cho_factor(np.eye(len(a)) + G @ G.T, lower=True), g)
        t, ok = 1.0, False
        for _ in range(60):
            St, gt, wt = ev(a + t * da)
            if np.isfinite(St) and St <= S + 1e-12 * abs(S):
                ok = True
                break
            t /= 2
        if not ok:
            break
        a, S, g, w = a + t * da, St, gt, wt
    return L @ a


def pref_fixed_point(y0, prefinds, L, iters=8):
    """y* with g(y*) = 0 to longdouble rounding, from an FP64 solution y0; L: the longdouble factor of R.  Newton steps in
    whitened coordinates a = inv(L) y whose residual L^T g(y) and update are longdouble; the Hessian I + L^T Lambda L is formed
    once, at y0, in FP64 (a fixed-Jacobian Newton iteration: the residual decides the fixed point, the Jacobian only the rate,
    here ~1e-7 per step from the pdf standing in for the Chebyshev CDF's derivative).  Returns (y*, |L^T g(y*)|_inf)."""
    from scipy.linalg import cho_factor, cho_solve
    L = np.asarray(L, dtype=LD)
    y = np.asarray(y0, dtype=LD)
    v, u, _, _, w = _terms(y, prefinds)
    G = (L[v] - L[u]).astype(float).T * np.sqrt(w.astype(float))
    H = cho_factor(np.eye(len(y)) + G @ G.T, lower=True)
    best = None
    for _ in range(iters):
        r = L.T @ pref_grad(y, prefinds, L)                         # the gradient in whitened coordinates
        res = np.max(np.abs(r))
        if best is not None and res >= best[1]:
            break
        best = (y, res)
        y = y - L @ cho_solve(H, r.astype(float)).astype(LD)
    return best
