"""CPU restatement of the gradients with respect to the candidate for the tests (and smoke()), written on top of the GPOracle the
way joint_oracle.py restates the joint posterior: triangular solves against the oracle's L (augL for a variance factor),
kernel.cross, PriorSpec, the clipping floors, and the acquisition's chain rule in each mode's own arithmetic."""
import math

import numpy as np

from oracle import ibo_oracle as orc


def kernel_grad(kernel, X, Xs):
    """dK[i, j, t] = d k(X_i, Xs_j) / d Xs_j,t = -(1 / theta_t) h(r) (Xs_j,t - X_i,t) / theta_t with h = k (SE),
    3 sf2 e^(-sqrt3 r) (Matern-3/2), (5/3) sf2 (1 + sqrt5 r) e^(-sqrt5 r) (Matern-5/2)"""
    X = np.asarray(X, dtype=float)
    Xs = np.asarray(Xs, dtype=float)
    th = kernel.theta
    D = (Xs[None, :, :] - X[:, None, :]) / th[None, None, :]          # s_t - s_i,t
    r2 = np.sum(D * D, axis=2)
    if kernel.kind in (orc.K_SE_ARD, orc.K_SE_ISO):
        h = kernel.sf2 * np.exp(-.5 * r2)
    elif kernel.kind == orc.K_MATERN3:
        h = 3.0 * kernel.sf2 * np.exp(-math.sqrt(3) * np.sqrt(r2))
    else:
        r = np.sqrt(r2)
        h = (5.0 / 3.0) * kernel.sf2 * (1.0 + math.sqrt(5.0) * r) * np.exp(-math.sqrt(5.0) * r)
    return -h[:, :, None] * D / th[None, None, :]


def prior_grad(prior, Xs):
    """d m0 / dx for the RBF-network prior -> [M, d]"""
    xs = (np.asarray(Xs, dtype=float) - prior.lowerb[None, :]) / prior.width[None, :]
    Q = xs[:, None, :] - prior.means[None, :, :]                        # [M, B, d]
    e = prior.beta[None, :] * np.exp(-prior.theta * np.sum(Q * Q, axis=2))
    return np.sum(e[:, :, None] * (-2.0 * prior.theta) * Q, axis=1) / prior.width[None, :]


def posterior_grad(o, Xs, mode="py"):
    """(mu[M], s2[M] clipped as the mode clips it, dmu[M, d], ds2[M, d]); ds2 = 0 where s2 is clipped"""
    from scipy.linalg import solve_triangular
    Xs = np.array(Xs, dtype=float, ndmin=2)
    Ks = o.kernel.cross(o.X, Xs)
    V = solve_triangular(o.L, Ks, lower=True)
    a = solve_triangular(o.L, solve_triangular(o.L, o.Y, lower=True), lower=True, trans='T')
    dK = kernel_grad(o.kernel, o.X, Xs)
    dmu = np.einsum('i,imt->mt', a, dK)
    if o.prior is None:
        mu = Ks.T.dot(a)
    else:
        b = solve_triangular(o.L, solve_triangular(o.L, np.ones_like(o.Y), lower=True), lower=True, trans='T')
        m = o.prior.mu_batch(Xs)
        kb = Ks.T.dot(b)
        mu = m + Ks.T.dot(a) - m * kb
        dmu += prior_grad(o.prior, Xs) * (1.0 - kb)[:, None] - m[:, None] * np.einsum('i,imt->mt', b, dK)
    if o.augL is not None:
        Ka = o.kernel.cross(o.augX, Xs)
        V = solve_triangular(o.augL, Ka, lower=True)
        z = solve_triangular(o.augL, V, lower=True, trans='T')
        dK = kernel_grad(o.kernel, o.augX, Xs)
    else:
        z = solve_triangular(o.L, V, lower=True, trans='T')
    floor = 10e-8 if mode == "py" else 1e-8
    s2 = np.clip((1 + o.noise) - np.sum(V * V, axis=0), floor, 10)
    ds2 = -2.0 * np.einsum('im,imt->mt', z, dK)
    ds2[(s2 <= floor) | (s2 >= 10)] = 0.0
    return mu, s2, dmu, ds2


def erf_py_deriv(z):
    """derivative of orc.erf_py: erf_py(z) = sign(z) g(|z|), g(u) = 1 - t e^E, t = 1 / (1 + u / 2), E = -u^2 + c0 + t p(t)"""
    u = np.abs(np.asarray(z, dtype=float))
    t = 1.0 / (1.0 + 0.5 * u)
    p, dp = orc._NR[9], 0.0
    for c in orc._NR[8:0:-1]:
        dp = p + t * dp
        p = c + t * p
    e = np.exp(-u * u + orc._NR[0] + t * p)
    dt = -0.5 * t * t
    return -e * (dt + t * (-2.0 * u + dt * (p + t * dp)))


def acq_partials(acq, mode, mu, s2, ymax, parm):
    """(d acq / d mu, d acq / d s) in the mode's own arithmetic"""
    s = np.sqrt(s2)
    if acq == orc.ACQ_UCB:
        return np.ones_like(mu), np.full_like(mu, parm)
    Z = (mu - ymax - parm) / s
    if mode == "py":
        cdf, dcdf = orc.cdf_py(Z), 0.5 * 0.707106 * erf_py_deriv(Z * 0.707106)
        if acq == orc.ACQ_PI:
            return dcdf / s, -Z * dcdf / s
        pdf = orc.pdf_py(Z)
        return cdf + Z * dcdf - Z * pdf, pdf - Z * Z * dcdf + Z * Z * pdf
    pdf = orc.pdf_cpp(Z)
    if acq == orc.ACQ_PI:
        return pdf / s, -Z * pdf / s
    return orc.cdf_cpp(Z), pdf


def score_grad(o, Xs, acq, ymax, parm, mode="py"):
    """(scores[M], dscores[M, d]) through (mu, s = sqrt(s2))"""
    mu, s2, dmu, ds2 = posterior_grad(o, Xs, mode)
    a_mu, a_s = acq_partials(acq, mode, mu, s2, ymax, parm)
    sc = orc.score(acq, mode, mu, s2, ymax, parm)
    return sc, a_mu[:, None] * dmu + (a_s / (2 * np.sqrt(s2)))[:, None] * ds2
