"""Extended-precision reference of the model build (test infrastructure only): a plain NumPy restatement in np.longdouble of
the blocked Cholesky, the triangular inverse W = inv(L) and the posterior the model serves; and of the candidate-side paths on
top of it: the joint posterior, the gradients with respect to the candidate, the reverse Cholesky and the Monte-Carlo q-EI with its
gradient.

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


def back_solve(L, B):
    """inv(L)^T B for a lower triangular L and B of shape (n,) or (n, m)."""
    L = np.asarray(L, dtype=LD)
    B = np.array(B, dtype=LD)
    for i in range(L.shape[0] - 1, -1, -1):
        B[i] = (B[i] - L[i + 1:, i] @ B[i + 1:]) / L[i, i]
    return B


def kernel_grad(kernel, X, Xs):
    """dK[i, j, t] = d k(X_i, Xs_j) / d Xs_j,t = -(1 / theta_t) h(r) (Xs_j,t - X_i,t) / theta_t in longdouble, with h = k (SE),
    3 sf2 e^(-sqrt3 r) (Matern-3/2), (5/3) sf2 (1 + sqrt5 r) e^(-sqrt5 r) (Matern-5/2): the formulas of grad_oracle.kernel_grad"""
    X = np.asarray(X, dtype=LD)
    Xs = np.asarray(Xs, dtype=LD)
    th = np.asarray(kernel.theta, dtype=LD)
    D = (Xs[None, :, :] - X[:, None, :]) / th
    r2 = np.sum(D * D, axis=2)
    sf2 = LD(kernel.sf2)
    if kernel.kind in (orc.K_SE_ARD, orc.K_SE_ISO):
        h = sf2 * np.exp(-r2 / 2)
    elif kernel.kind == orc.K_MATERN3:
        h = 3 * sf2 * np.exp(-np.sqrt(LD(3)) * np.sqrt(r2))
    else:
        s5r = np.sqrt(LD(5)) * np.sqrt(r2)
        h = sf2 * (1 + s5r) * np.exp(-s5r) * 5 / 3
    return -h[:, :, None] * D / th


def prior_grad(prior, Xs):
    """d m0 / dx of the RBF-network prior mean in longdouble -> [M, d]"""
    w = np.asarray(prior.width, dtype=LD)
    xs = (np.asarray(Xs, dtype=LD) - np.asarray(prior.lowerb, dtype=LD)) / w
    Q = xs[:, None, :] - np.asarray(prior.means, dtype=LD)[None]
    e = np.asarray(prior.beta, dtype=LD) * np.exp(-LD(prior.theta) * np.sum(Q * Q, axis=2))
    return np.sum(e[:, :, None] * Q, axis=1) * (-2 * LD(prior.theta)) / w


class _Model(object):
    """the longdouble factors of one problem: L of R (the mean) and Lg of the matrix sigma^2 comes from (R, or the variance
    model's A = R(augX) + pad(inv(C)) when aug = (augX, augA) is given)"""

    def __init__(self, kernel, X, Y, noise, prior, aug):
        self.kernel, self.noise, self.prior = kernel, noise, prior
        self.X, self.Y = np.asarray(X, dtype=float), np.asarray(Y, dtype=float)
        self.L = cholesky(build_R(kernel, X, noise))
        self.Xg, self.Lg = (self.X, self.L) if aug is None else (np.asarray(aug[0], dtype=float), cholesky(aug[1]))
        self.a = back_solve(self.L, forward_solve(self.L, self.Y))                          # R^-1 Y
        self.b = None if prior is None else back_solve(self.L, forward_solve(self.L, np.ones(len(self.Y))))

    def mean(self, Xs, grad=False):
        """mu (and dmu) at the candidates"""
        Ks = cross(self.kernel, self.X, Xs)
        mu = Ks.T @ self.a
        dK = kernel_grad(self.kernel, self.X, Xs) if grad else None
        dmu = np.einsum('i,imt->mt', self.a, dK) if grad else None
        if self.prior is not None:
            m, kb = prior_mean(self.prior, Xs), Ks.T @ self.b
            mu = m + mu - m * kb
            if grad:
                dmu += prior_grad(self.prior, Xs) * (1 - kb)[:, None] - m[:, None] * np.einsum('i,imt->mt', self.b, dK)
        return mu, dmu

    def V(self, Xs):
        return forward_solve(self.Lg, cross(self.kernel, self.Xg, Xs))


def _model(kernel, X, Y, noise, prior, aug, model):
    return model if model is not None else _Model(kernel, X, Y, noise, prior, aug)


def posterior_joint(kernel, X, Y, noise, Xs, prior=None, aug=None, model=None):
    """(mu[M], Sigma[M, M]): Sigma = R(Xs, Xs) - V^T V with V = inv(L_g) k(X_g, Xs), so diag(Sigma) is sigma^2 before clipping.
    aug = (augX, augA): a variance model, A = R(augX) + inv(C) padded.  model: the factors of an earlier call on the problem."""
    o = _model(kernel, X, Y, noise, prior, aug, model)
    V = o.V(Xs)
    return o.mean(Xs)[0], build_R(kernel, Xs, noise) - V.T @ V


def posterior_grad(kernel, X, Y, noise, Xs, prior=None, aug=None, model=None):
    """(mu[M], s2[M] unclipped, dmu[M, d], ds2[M, d]) with ds2 = -2 sum_i z_i dk(X_g,i, x) / dx, z = inv(A_g) k(X_g, x)"""
    o = _model(kernel, X, Y, noise, prior, aug, model)
    mu, dmu = o.mean(Xs, grad=True)
    V = o.V(Xs)
    z = back_solve(o.Lg, V)
    ds2 = -2 * np.einsum('im,imt->mt', z, kernel_grad(kernel, o.Xg, Xs))
    return mu, LD(1.0 + noise) - np.sum(V * V, axis=0), dmu, ds2


def chol_rev(L, Lbar):
    """reverse-mode Cholesky (Murray 2016) in longdouble: Sigma = L L^T, Lbar = df / dL (lower) -> the symmetric
    Gbar = sym(L^-T Phi(L^T Lbar) L^-1) with df = sum_{k,l} Gbar_kl dSigma_kl (Phi: lower triangle, halved diagonal)"""
    L = np.asarray(L, dtype=LD)
    P = np.tril(L.T @ np.tril(np.asarray(Lbar, dtype=LD)))
    P[np.diag_indices_from(P)] /= 2
    S = back_solve(L, back_solve(L, P).T).T                       # (L^-T P) L^-1
    return (S + S.T) / 2


def qei(kernel, X, Y, noise, Xb, Z, ymax, xi, jitter, prior=None, aug=None, model=None):
    """values[B], gradients[B, q, d] of the Monte-Carlo q-EI of the batches Xb[B, q, d] for the standard normals Z[q, S] (FP64,
    part of the problem), and per batch two margins: the smallest gap between the two largest entries of F = mu + L Z over the
    samples with positive improvement (inf for q = 1 or no such sample), and the smallest |improvement| over all samples.  The
    gradient is discontinuous where either margin is 0.  A batch whose Sigma + jitter I is not positive definite raises."""
    o = _model(kernel, X, Y, noise, prior, aug, model)
    Xb = np.asarray(Xb, dtype=LD)
    B, q, d = Xb.shape
    Zl = np.asarray(Z, dtype=LD)
    S = Zl.shape[1]
    vals, grads, gaps, imps = np.zeros(B, dtype=LD), np.zeros((B, q, d), dtype=LD), np.zeros(B), np.zeros(B)
    mu_all, dmu_all = o.mean(Xb.reshape(-1, d), grad=True)
    V_all = o.V(Xb.reshape(-1, d))
    z_all = back_solve(o.Lg, V_all)                                # inv(A_g) k(X_g, x)
    for b in range(B):
        x, c = Xb[b], slice(b * q, (b + 1) * q)
        mu, dmu, V = mu_all[c], dmu_all[c], V_all[:, c]
        Sig = build_R(kernel, x, noise) - V.T @ V + LD(jitter) * np.eye(q, dtype=LD)
        Lb = cholesky(Sig)
        F = mu[:, None] + Lb @ Zl
        js = np.argmax(F, axis=0)                                  # lowest index wins ties
        imp = F[js, np.arange(S)] - LD(ymax) - LD(xi)
        pos = imp > 0
        vals[b] = np.sum(np.where(pos, imp, 0)) / S
        Fs = np.sort(F[:, pos], axis=0)
        gaps[b] = float(np.min(Fs[-1] - Fs[-2])) if q > 1 and pos.any() else np.inf
        imps[b] = float(np.min(np.abs(imp)))
        onehot = (js[pos][:, None] == np.arange(q)[None]).astype(LD)
        mubar = onehot.sum(axis=0) / S
        Gbar = chol_rev(Lb, np.tril(onehot.T @ Zl[:, pos].T) / S)
        y = z_all[:, c] @ Gbar                                     # y_j = sum_l Gbar_jl inv(A_g) k(X_g, x_l)
        dC = kernel_grad(kernel, x, x)                             # dC[l, j, t] = d k(x_l, x_j) / d x_j,t
        grads[b] = mubar[:, None] * dmu + 2 * np.einsum('jl,ljt->jt', Gbar, dC) - 2 * np.einsum('ij,ijt->jt', y, kernel_grad(kernel, o.Xg, x))
    return vals, grads, gaps, imps


def rel(X, Xref):
    """||X - Xref||_F / ||Xref||_F, evaluated in longdouble, as a float."""
    Xref = np.asarray(Xref, dtype=LD)
    D = np.asarray(X, dtype=LD) - Xref
    return float(np.sqrt(np.sum(D * D)) / np.sqrt(np.sum(Xref * Xref)))
