"""CPU restatement of the noisy batch expected improvement (q-NEI) and of its gradient for the tests, in the full form: one
Cholesky of the latent joint posterior of the P + q points [baseline; batch] (joint_oracle.posterior_joint minus (1 + noise - sf2) I on
the diagonal), and the gradient through qei_oracle.chol_rev over the whole joint, taking the rows of the batch points only (the
baseline does not move).  The device factors the same matrix blockwise with the baseline first; the two agree to rounding."""
import numpy as np

import grad_oracle as go
import joint_oracle as jo
from qei_oracle import chol_rev


class BaselineNotPD(np.linalg.LinAlgError):
    pass


def latent_joint(o, A):
    """mu[n], Sigma[n, n] of the latent function at the points A[n, d]: sf2 instead of 1 + noise on the diagonal"""
    mu, Sig = jo.posterior_joint(o, A)
    return mu, Sig - (1.0 + o.noise - o.kernel.sf2) * np.eye(len(A))


def qnei_batch(o, Xb, Xbase, Z, jitter=0.0, grad=True, incumbent=False):
    """value (and gradient [q, d]) of one batch Xb[q, d] over the baseline Xbase[P, d] for standard normals Z[P + q, S] (baseline
    rows first).  Raises BaselineNotPD when the baseline block + jitter I is not positive definite; NaN when only the batch's part
    fails.  incumbent=True also returns m[S]."""
    from scipy.linalg import solve_triangular
    Xb = np.array(Xb, dtype=float, ndmin=2)
    Xbase = np.array(Xbase, dtype=float, ndmin=2)
    q, d = Xb.shape
    P, S = Xbase.shape[0], Z.shape[1]
    A = np.r_[Xbase, Xb]
    mu, Sig = latent_joint(o, A)
    Sj = Sig + jitter * np.eye(P + q)
    try:
        Lb = np.linalg.cholesky(Sj[:P, :P])
    except np.linalg.LinAlgError:
        raise BaselineNotPD("baseline covariance + jitter I is not positive definite")
    m = np.max(mu[:P, None] + Lb.dot(Z[:P]), axis=0)
    out = []
    try:
        L = np.linalg.cholesky(Sj)
    except np.linalg.LinAlgError:
        out = [np.nan] + ([np.full((q, d), np.nan)] if grad else [])
        return tuple(out + [m]) if incumbent else (tuple(out) if grad else out[0])
    F = mu[:, None] + L.dot(Z)
    Fq = F[P:]
    jstar = np.argmax(Fq, axis=0)                                     # lowest index wins ties
    imp = Fq[jstar, np.arange(S)] - m
    val = np.sum(np.maximum(0.0, imp)) / S
    out = [val]
    if grad:
        pos = imp > 0
        mubar = np.bincount(jstar[pos], minlength=q) / S
        Lbar = np.zeros((P + q, P + q))
        for s in np.nonzero(pos)[0]:
            r = P + jstar[s]
            Lbar[r, :r + 1] += Z[:r + 1, s] / S
        Gbar = chol_rev(L, Lbar)
        _, _, dmu, _ = go.posterior_grad(o, Xb)
        if o.augL is not None:
            Xg, Lg = o.augX, o.augL
        else:
            Xg, Lg = o.X, o.L
        Kg = o.kernel.cross(Xg, A)
        Zm = solve_triangular(Lg, solve_triangular(Lg, Kg, lower=True), lower=True, trans='T')    # R_g^-1 k(X_g, a_l), [N, P + q]
        Y = Zm.dot(Gbar)
        dK = go.kernel_grad(o.kernel, Xg, A)                              # [N, P + q, d]
        dC = go.kernel_grad(o.kernel, A, A)                               # dC[l, j, t] = d k(a_l, a_j) / d a_j,t
        G = 2.0 * np.einsum('jl,ljt->jt', Gbar, dC) - 2.0 * np.einsum('ij,ijt->jt', Y, dK)
        out.append(mubar[:, None] * dmu + G[P:])
    if incumbent:
        return tuple(out + [m])
    return tuple(out) if grad else val


def qnei(o, Xb, Xbase, Z, jitter=0.0, grad=True):
    """values[B] (and gradients[B, q, d]) of the batches Xb[B, q, d]"""
    Xb = np.array(Xb, dtype=float, ndmin=3)
    res = [qnei_batch(o, X, Xbase, Z, jitter, grad) for X in Xb]
    if not grad:
        return np.array(res)
    return np.array([r[0] for r in res]), np.array([r[1] for r in res])


def incumbent(o, Xbase, Z, jitter=0.0):
    """m[S] = max over the baseline of mu_b + chol(Sigma_bb + jitter I) Z_b"""
    Xbase = np.array(Xbase, dtype=float, ndmin=2)
    P = Xbase.shape[0]
    mu, Sig = latent_joint(o, Xbase)
    return np.max(mu[:, None] + np.linalg.cholesky(Sig + jitter * np.eye(P)).dot(Z[:P]), axis=0)
