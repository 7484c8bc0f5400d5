"""CPU restatement of the batch expected improvement (q-EI) and of its gradient for the tests (and smoke()), on top of
joint_oracle.posterior_joint (mu, Sigma of a batch) and grad_oracle (kernel and prior gradients, dmu)."""
import numpy as np

import grad_oracle as go
import joint_oracle as jo


def chol_rev(L, Lbar):
    """reverse-mode Cholesky (Murray 2016): Sigma = L L^T, Lbar = df / dL (lower) -> the symmetric Gbar with
    df = sum_{k,l} Gbar_kl dSigma_kl over all ordered pairs: Gbar = sym(L^-T Phi(L^T Lbar) L^-1), Phi = lower triangle with the
    diagonal halved"""
    from scipy.linalg import solve_triangular
    P = np.tril(L.T.dot(np.tril(Lbar)))
    P[np.diag_indices_from(P)] *= 0.5
    X = solve_triangular(L, P, lower=True, trans='T')               # L^-T P
    S = solve_triangular(L, X.T, lower=True, trans='T').T           # X L^-1
    return 0.5 * (S + S.T)


def qei_batch(o, Xb, Z, ymax, xi, jitter=0.0, grad=True):
    """value (and gradient [q, d]) of one batch Xb[q, d] for the GPOracle o and standard normals Z[q, S]"""
    from scipy.linalg import solve_triangular
    Xb = np.array(Xb, dtype=float, ndmin=2)
    q, d = Xb.shape
    S = Z.shape[1]
    mu, Sigma = jo.posterior_joint(o, Xb)
    try:
        L = np.linalg.cholesky(Sigma + jitter * np.eye(q))
    except np.linalg.LinAlgError:
        return (np.nan, np.full((q, d), np.nan)) if grad else np.nan
    F = mu[:, None] + L.dot(Z)
    jstar = np.argmax(F, axis=0)                                      # lowest index wins ties
    imp = F[jstar, np.arange(S)] - ymax - xi
    val = np.sum(np.maximum(0.0, imp)) / S
    if not grad:
        return val
    pos = imp > 0
    mubar = np.bincount(jstar[pos], minlength=q) / S
    Lbar = np.zeros((q, q))
    for s in np.nonzero(pos)[0]:
        j = jstar[s]
        Lbar[j, :j + 1] += Z[:j + 1, s] / S
    Gbar = chol_rev(L, Lbar)
    _, _, dmu, _ = go.posterior_grad(o, Xb)
    if o.augL is not None:
        Xg, Lg = o.augX, o.augL
    else:
        Xg, Lg = o.X, o.L
    Kg = o.kernel.cross(Xg, Xb)
    Zm = solve_triangular(Lg, solve_triangular(Lg, Kg, lower=True), lower=True, trans='T')    # R_g^-1 k(X_g, x_l), [N, q]
    Y = Zm.dot(Gbar)                                                  # y_j = sum_l Gbar_jl z_l (Gbar symmetric)
    dK = go.kernel_grad(o.kernel, Xg, Xb)                             # [N, q, d]
    dC = go.kernel_grad(o.kernel, Xb, Xb)                             # dC[l, j, t] = d k(x_l, x_j) / d x_j,t
    G = mubar[:, None] * dmu + 2.0 * np.einsum('jl,ljt->jt', Gbar, dC) - 2.0 * np.einsum('ij,ijt->jt', Y, dK)
    return val, G


def qei(o, Xb, Z, ymax, xi, jitter=0.0, grad=True):
    """values[B] (and gradients[B, q, d]) of the batches Xb[B, q, d]"""
    Xb = np.array(Xb, dtype=float, ndmin=3)
    res = [qei_batch(o, X, Z, ymax, xi, jitter, grad) for X in Xb]
    if not grad:
        return np.array(res)
    return np.array([r[0] for r in res]), np.array([r[1] for r in res])
