"""CPU restatement of the pathwise posterior samples (ibo_paths_*) for the tests (and smoke()), written on top of the GPOracle the way
joint_oracle.py restates the joint posterior: the same caller-supplied draws, triangular solves against the oracle's L (augL for a
variance factor), and the analytic covariance of the paths for given features."""
import numpy as np

from oracle import ibo_oracle as orc

import grad_oracle


def features(kernel, omega, phase, X):
    """phi[M, F] = sqrt(2 sf2 / F) cos(omega . (x / theta) + b)"""
    X = np.asarray(X, dtype=float)
    F = omega.shape[0]
    return np.sqrt(2.0 * kernel.sf2 / F) * np.cos((X / kernel.theta[None, :]).dot(omega.T) + phase[None, :])


def _g(o):
    """(L, X) of the model Sigma comes from: the variance factor when one is set"""
    return (o.augL, o.augX) if o.augL is not None else (o.L, o.X)


def noise(o, e):
    """E e: sqrt(1 + noise - sf2) e, or chol(inv(C) + (1 + noise - sf2) I) e for a g with a Laplace term (inv(C) = A - R of the oracle,
    or o.augCinv for a variance factor)"""
    c = 1.0 + o.noise - o.kernel.sf2
    Cinv = getattr(o, 'augCinv', None) if o.augL is not None else o.A - o.R
    if Cinv is None or not np.any(Cinv):
        return np.sqrt(c) * e
    return np.linalg.cholesky(Cinv + c * np.eye(len(Cinv))).dot(e)


def _solve(L, B):
    from scipy.linalg import solve_triangular
    return solve_triangular(L, solve_triangular(L, B, lower=True), lower=True, trans='T')


def coefficients(o, omega, phase, w, e):
    """c[Ng, S] = R_g^-1 (Phi_g w + E e)"""
    Lg, Xg = _g(o)
    return _solve(Lg, features(o.kernel, omega, phase, Xg).dot(w) + noise(o, e))


def mean(o, Xs):
    """mu = m0 + k^T a - m0 k^T b (a = R^-1 Y, b = R^-1 1; the prior terms with a prior only)"""
    Ks = o.kernel.cross(o.X, Xs)
    mu = Ks.T.dot(_solve(o.L, o.Y))
    if o.prior is not None:
        m = o.prior.mu_batch(Xs)
        mu = m + mu - m * Ks.T.dot(_solve(o.L, np.ones_like(o.Y)))
    return mu


def paths(o, omega, phase, w, e, Xs):
    """values[M, S] of the paths f_s = mu + phi^T w_s - k_g^T c_s, and the per-value sum of the magnitudes of its terms
    (|k a| + |phi w| + |k c| over the rows, and |m0| |k b| with a prior) that bounds its rounding error"""
    Xs = np.array(Xs, dtype=float, ndmin=2)
    _, Xg = _g(o)
    c = coefficients(o, omega, phase, w, e)
    Phi = features(o.kernel, omega, phase, Xs)
    Kg = o.kernel.cross(Xg, Xs)
    Ks = o.kernel.cross(o.X, Xs)
    a = _solve(o.L, o.Y)
    vals = mean(o, Xs)[:, None] + Phi.dot(w) - Kg.T.dot(c)
    mag = np.abs(Ks.T).dot(np.abs(a))[:, None] + np.abs(Phi).dot(np.abs(w)) + np.abs(Kg.T).dot(np.abs(c))
    if o.prior is not None:
        m = o.prior.mu_batch(Xs)
        mag = mag + (np.abs(m) * (1.0 + np.abs(Ks.T).dot(np.abs(_solve(o.L, np.ones_like(o.Y))))))[:, None]
    return vals, mag


def paths_grad(o, omega, phase, w, e, Xs, which):
    """(values[M], grad[M, d]) of point j on path which[j]"""
    Xs = np.array(Xs, dtype=float, ndmin=2)
    which = np.asarray(which)
    _, Xg = _g(o)
    th = o.kernel.theta
    c = coefficients(o, omega, phase, w, e)
    vals = paths(o, omega, phase, w, e, Xs)[0][np.arange(len(Xs)), which]
    o_mean = orc.GPOracle.__new__(orc.GPOracle)       # dmu of the mean model alone (grad_oracle reads augL for ds2 only)
    o_mean.__dict__.update(o.__dict__)
    o_mean.augL, o_mean.augX = None, None
    dmu = grad_oracle.posterior_grad(o_mean, Xs)[2]
    F = omega.shape[0]
    arg = (Xs / th[None, :]).dot(omega.T) + phase[None, :]
    W = w[:, which].T                                                              # [M, F]
    dfeat = -np.sqrt(2.0 * o.kernel.sf2 / F) * (W * np.sin(arg)).dot(omega) / th[None, :]
    dK = grad_oracle.kernel_grad(o.kernel, Xg, Xs)                                 # [Ng, M, d]
    dker = np.einsum('im,imt->mt', c[:, which], dK)
    return vals, dmu + dfeat - dker


def analytic_cov(Pss, Psx, Pxx, Ks, R, EEt):
    """covariance of the paths at the points X* for given features:
        Phi* Phi*^T - Phi* Phi_X^T R^-1 K* - K*^T R^-1 Phi_X Phi*^T + K*^T R^-1 (Phi_X Phi_X^T + E E^T) R^-1 K*
    with Pss = Phi* Phi*^T [M, M], Psx = Phi* Phi_X^T [M, N], Pxx = Phi_X Phi_X^T [N, N], Ks = K(X, X*) [N, M], EEt = E E^T.
    With the exact kernel in place of every feature Gram block this is Sigma - (1 + noise - sf2) I."""
    RiK = np.linalg.solve(R, Ks)
    C = Pss - Psx.dot(RiK) - RiK.T.dot(Psx.T) + RiK.T.dot(Pxx + EEt).dot(RiK)
    return 0.5 * (C + C.T)
