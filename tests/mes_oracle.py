"""CPU restatement of max-value entropy search for the tests (and smoke()), on top of the GPOracle and grad_oracle: h and h' in
mpmath at 50 digits, MES and its gradient in float64 over the FP64 posterior oracle, and the Gumbel fit's quantiles by brentq over a
math.fsum of scipy's log_ndtr terms."""
import math

import mpmath as mp
import numpy as np
from scipy.optimize import brentq
from scipy.special import erfc, erfcx, log_ndtr

import grad_oracle

SQRT2 = math.sqrt(2.0)


def h_mp(g, dps=50):
    """(h, h') at the double g as mpmath numbers: h = g psi / 2 - log Phi, h' = -(psi / 2)(1 + g (g + psi)), psi = phi / Phi.
    log Phi(g) for g > 0 is log1p(-Phi(-g)): log(Phi(g)) loses the digits of Phi(g) ~ 1 at 50 digits for g >~ 15."""
    with mp.workdps(dps):
        g = mp.mpf(float(g))
        Phi = mp.ncdf(g)
        psi = mp.npdf(g) / Phi
        lphi = mp.log1p(-mp.ncdf(-g)) if g > 0 else mp.log(Phi)
        return g * psi / 2 - lphi, -(psi / 2) * (1 + g * (g + psi))


def h_np(G):
    """(h, h') in float64, elementwise: the textbook form for t = -g / sqrt2 < 1.5, the continued fraction of erfc above"""
    G = np.asarray(G, dtype=float)
    t = -G / SQRT2
    cf = t >= 1.5
    tt = np.where(cf, t, 1.5)
    r = np.zeros_like(tt)
    for k in range(120, 1, -1):
        r = (0.5 * k) / (tt + r)
    r1 = 0.5 / (tt + r)
    h_cf = (0.5 * G) * (SQRT2 * r1) + np.log(2.0 * math.sqrt(math.pi) * (tt + r1))
    dh_cf = -(SQRT2 * (tt + r1) / 2.0) * (r / (tt + r))
    tb = np.where(cf, 0.0, t)
    gb = np.where(cf, 0.0, G)
    with np.errstate(over='ignore', divide='ignore', invalid='ignore'):
        e = erfcx(tb)
        psi = math.sqrt(2.0 / math.pi) / e
        lphi = np.where(gb < 0, np.log(0.5 * e) - 0.5 * gb * gb, np.log1p(-0.5 * erfc(gb / SQRT2)))
        h_tb = 0.5 * gb * psi - lphi
        dh_tb = -0.5 * psi * (1.0 + gb * (gb + psi))
    return np.where(cf, h_cf, h_tb), np.where(cf, dh_cf, dh_tb)


def mes_partials(mu, s2, ystar):
    """(values[M], d MES / d mu [M], d MES / d s [M]) at the posterior (mu, s2) for samples ystar[K]"""
    mu, s = np.asarray(mu, dtype=float), np.sqrt(np.asarray(s2, dtype=float))
    ystar = np.asarray(ystar, dtype=float)
    K = ystar.shape[0]
    G = (ystar[None, :] - mu[:, None]) / s[:, None]
    h, dh = h_np(G)
    return np.sum(h, axis=1) / K, -np.sum(dh, axis=1) / (K * s), -np.sum(G * dh, axis=1) / (K * s)


def mes(o, Xs, ystar, mode="py", grad=True):
    """(values[M], gradient[M, d]) over the FP64 posterior oracle: d MES = d MES / d mu  d mu + d MES / d s  d s2 / (2 s), with
    d s2 = 0 where s2 is clipped"""
    mu, s2, dmu, ds2 = grad_oracle.posterior_grad(o, Xs, mode)
    v, a, b = mes_partials(mu, s2, ystar)
    if not grad:
        return v
    return v, a[:, None] * dmu + (b / (2.0 * np.sqrt(s2)))[:, None] * ds2


def log_F(y, mu, s):
    """log F(y) = sum_i log Phi((y - mu_i) / s_i), summed exactly rounded (math.fsum)"""
    return math.fsum(log_ndtr((y - np.asarray(mu)) / np.asarray(s)))


def log_F_terms(y, mu, s):
    return log_ndtr((y - np.asarray(mu)) / np.asarray(s))


def gumbel_quantiles(mu, s2):
    """q[3] with log F(q) = log 0.25, log 0.5, log 0.75 (brentq to a few ulp), and (loc, scale) of the header's formula"""
    mu, s = np.asarray(mu, dtype=float), np.sqrt(np.asarray(s2, dtype=float))
    lo = np.max(mu - s)
    hi = np.max(mu + math.sqrt(2.0 * math.log(5.0 * mu.shape[0])) * s)
    q = np.array([brentq(lambda y: log_F(y, mu, s) - math.log(p), lo, hi, xtol=1e-300, rtol=4 * np.finfo(float).eps, maxiter=500)
                  for p in (0.25, 0.5, 0.75)])
    return q, gumbel_loc_scale(q)


def gumbel_loc_scale(q):
    """(loc, scale) from q exactly as the header computes them (libm log)"""
    scale = (q[2] - q[0]) / (math.log(-math.log(.25)) - math.log(-math.log(.75)))
    return q[1] + scale * math.log(-math.log(.5)), scale
