"""CPU restatement of the joint posterior for the tests (and smoke()), written the way oracle.GPOracle.posterior_batch is:
triangular solves against the oracle's L (augL for a variance factor) and build_R on the candidates."""
import numpy as np

from oracle import ibo_oracle as orc


def posterior_joint(o, Xs):
    """Joint posterior of the GPOracle `o` over the candidates -> mu[M], Sigma[M, M] = build_R(Xs) - V^T V with
    V = inv(L) k(X, Xs) (inv(augL) k(augX, Xs) when a variance factor is set): diag(Sigma) is o.posterior_batch's sigma^2
    before clipping, mu is its mu."""
    from scipy.linalg import solve_triangular
    Xs = np.array(Xs, dtype=float, ndmin=2)
    Ks = o.kernel.cross(o.X, Xs)
    V = solve_triangular(o.L, Ks, lower=True)
    bY = solve_triangular(o.L, o.Y, lower=True)
    if o.prior is None:
        mu = V.T.dot(bY)
    else:
        m = o.prior.mu_batch(Xs)
        b1 = solve_triangular(o.L, np.ones_like(o.Y), lower=True)
        mu = m + V.T.dot(bY) - m * V.T.dot(b1)
    if o.augL is not None:
        V = solve_triangular(o.augL, o.kernel.cross(o.augX, Xs), lower=True)
    G = V.T.dot(V)
    Sigma = orc.build_R(o.kernel, Xs, o.noise) - 0.5 * (G + G.T)
    np.fill_diagonal(Sigma, (1 + o.noise) - np.sum(V * V, axis=0))
    return mu, Sigma
