"""Extended-precision reference of the model build (test infrastructure only): a plain NumPy restatement in np.longdouble of
the blocked Cholesky, the triangular inverse W = inv(L) and the posterior the model serves.

On x86-64 np.longdouble is the 80-bit format, eps ~ 1.1e-19, about 2000 times finer than FP64: where an FP64 result (the
device's or LAPACK's) disagrees with these values, the FP64 result is the one in error.  Inputs are FP64 arrays (they define
the problem exactly); outputs are longdouble.  A 512^3 longdouble product takes about a second, which makes this practical up
to N ~ 1100 and a few hundred candidates."""
import numpy as np

from oracle import ibo_oracle as orc

LD = np.longdouble


def cholesky(A, nb=64):
    """Lower L with L L^T = A: right-looking, nb columns at a time.  A non-positive pivot raises numpy.linalg.LinAlgError with
    `pivot` = its 1-based row, as the library reports it."""
    A = np.array(A, dtype=LD)
    n = A.shape[0]
    for k in range(0, n, nb):
        e = min(k + nb, n)
        for j in range(k, e):                    # diagonal block, one column at a time
            if not A[j, j] > 0:
                err = np.linalg.LinAlgError("not positive definite (pivot %d)" % (j + 1))
                err.pivot = j + 1
                raise err
            A[j, j] = np.sqrt(A[j, j])
            A[j + 1:e, j] /= A[j, j]
            A[j + 1:e, j + 1:e] -= np.outer(A[j + 1:e, j], A[j + 1:e, j])
        if e == n:
            break
        for j in range(k, e):                    # panel: A_ik <- A_ik inv(L_kk)^T, by substitution
            A[e:, j] = (A[e:, j] - A[e:, k:j] @ A[j, k:j]) / A[j, j]
        P = A[e:, k:e]
        for i in range(e, n, nb):                # trailing update, lower block rows only
            r = min(i + nb, n)
            A[i:r, e:r] -= P[i - e:r - e] @ P[:r - e].T
    return np.tril(A)


def tri_inv(L):
    """inv(L) of a lower triangular L, row by row: X_i = (e_i - L_i,<i X_<i) / L_ii."""
    L = np.asarray(L, dtype=LD)
    n = L.shape[0]
    X = np.zeros((n, n), dtype=LD)
    for i in range(n):
        X[i, :i] = -(L[i, :i] @ X[:i, :i]) / L[i, i]
        X[i, i] = 1 / L[i, i]
    return X


def forward_solve(L, B):
    """inv(L) B for a lower triangular L and B of shape (n,) or (n, m)."""
    L = np.asarray(L, dtype=LD)
    B = np.array(B, dtype=LD)
    for i in range(L.shape[0]):
        B[i] = (B[i] - L[i, :i] @ B[:i]) / L[i, i]
    return B


def cross(kernel, X, Xs):
    """k(X_i, Xs_j) in longdouble: the formulas of oracle.KernelSpec.cross (its FP64 theta and sf2 are part of the problem)."""
    X = np.asarray(X, dtype=LD)
    Xs = np.asarray(Xs, dtype=LD)
    th = np.asarray(kernel.theta, dtype=LD)
    D = (X[:, None, :] - Xs[None, :, :]) / th
    r2 = np.sum(D * D, axis=2)
    sf2 = LD(kernel.sf2)
    if kernel.kind in (orc.K_SE_ARD, orc.K_SE_ISO):
        return sf2 * np.exp(-r2 / 2)
    r = np.sqrt(r2)
    if kernel.kind == orc.K_MATERN3:
        z = np.sqrt(LD(3)) * r
        return sf2 * (1 + z) * np.exp(-z)
    s5r = np.sqrt(LD(5)) * r
    return sf2 * (1 + s5r + 5 * r2 / 3) * np.exp(-s5r)


def build_R(kernel, X, noise):
    """R = K_offdiag + (1 + noise) I; the diagonal is the FP64 number 1 + noise that the library (and the reference) puts there."""
    R = cross(kernel, X, X)
    np.fill_diagonal(R, LD(1.0 + noise))
    return R


def prior_mean(prior, Xs):
    """RBF-network prior mean (oracle.PriorSpec.mu_batch) in longdouble."""
    xs = (np.asarray(Xs, dtype=LD) - np.asarray(prior.lowerb, dtype=LD)) / np.asarray(prior.width, dtype=LD)
    d2 = np.sum((xs[:, None, :] - np.asarray(prior.means, dtype=LD)[None]) ** 2, axis=2)
    return np.sum(np.asarray(prior.beta, dtype=LD) * np.exp(-LD(prior.theta) * d2), axis=1)


def posterior(kernel, X, Y, noise, Xs, prior=None, L=None):
    """mu = m + k*^T inv(R) (Y - m 1) and sigma^2 = (1 + noise) - k*^T inv(R) k* (unclipped), with m the prior mean at the
    candidate (0 without a prior).  L: the longdouble factor of R when the caller has it."""
    if L is None:
        L = cholesky(build_R(kernel, X, noise))
    V = forward_solve(L, cross(kernel, X, Xs))
    mu = V.T @ forward_solve(L, Y)
    if prior is not None:
        m = prior_mean(prior, Xs)
        mu = m + mu - m * (V.T @ forward_solve(L, np.ones(len(Y))))
    return mu, LD(1.0 + noise) - np.sum(V * V, axis=0)


def rel(X, Xref):
    """||X - Xref||_F / ||Xref||_F, evaluated in longdouble, as a float."""
    Xref = np.asarray(Xref, dtype=LD)
    D = np.asarray(X, dtype=LD) - Xref
    return float(np.sqrt(np.sum(D * D)) / np.sqrt(np.sum(Xref * Xref)))
