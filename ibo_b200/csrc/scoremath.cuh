// Device math shared by the scoring kernels (score.cu: K1-K3, tiny.cu: the fused small-model kernel) and the other kernels that
// need the same arithmetic: covariance from the scaled squared distance, the kernels' own exp, the reference's two erf / EI / PI /
// UCB arithmetics, the RBF prior mean.
#pragma once
#include "common.cuh"
#include "../../include/ibo_b200.h"

namespace ibo {

// covariance from the scaled squared distance r2 = sum_j ((x_j - y_j) / theta_j)^2: the model build, the scoring path and the
// marginal likelihood all evaluate it here (ego/gaussianprocess/kernel.py:87-89,147-149,207-210,246-248; cpp/optimizeGP.cpp:70-112)
__device__ __forceinline__ double cov_r2(int kind, double sf2, double r2) {
    if (kind <= IBO_KERNEL_SE_ISO) return sf2 * exp(-0.5 * r2);
    double r = sqrt(r2);
    if (kind == IBO_KERNEL_MATERN3) {
        double z = 1.7320508075688772 * r;
        return sf2 * (1.0 + z) * exp(-z);
    }
    double z = 2.23606797749979 * r;
    return sf2 * (1.0 + z + 5.0 * r2 / 3.0) * exp(-z);
}

// dk/dx_t = -(1 / theta_t) h(r) (s_t - s_i,t) in the scaled coordinates s = x / theta - centre: h = k for SE,
// 3 sf2 e^(-sqrt3 r) for Matern-3/2, (5/3) sf2 (1 + sqrt5 r) e^(-sqrt5 r) for Matern-5/2 -- finite at r = 0 for all of them.
// *k receives k(r) (cov_r2's formulas).
__device__ __forceinline__ double cov_grad_h(int kind, double sf2, double r2, double* k) {
    if (kind <= IBO_KERNEL_SE_ISO) { *k = sf2 * exp(-0.5 * r2); return *k; }
    const double r = sqrt(r2);
    if (kind == IBO_KERNEL_MATERN3) {
        const double z = 1.7320508075688772 * r, e = sf2 * exp(-z);
        *k = (1.0 + z) * e;
        return 3.0 * e;
    }
    const double z = 2.23606797749979 * r, e = sf2 * exp(-z);
    *k = (1.0 + z + 5.0 * r2 / 3.0) * e;
    return (5.0 / 3.0) * (1.0 + z) * e;
}

// exp(x) for x <= 0 with the coefficients in the constant bank.  K1 is issue bound (ncu: 78 % of the issue slots, FP64 pipe
// 39 %), and libdevice's exp materialises its eleven 64-bit polynomial constants with two uniform moves each per call
// (UMOV = 26 % of all executed instructions of K1): here every coefficient is a constant-bank operand of its DFMA.
// exp(x) = 2^k exp(r), k = rint(x log2 e), r = x - k ln2 (two-term Cody-Waite with FMA), Taylor to degree 13 on
// |r| <= ln2 / 2 (truncation 4e-18), scaling through the exponent field; results below 2^-1021 flush to zero.
// Measured against libdevice exp on 10^7 arguments in [-745, 0]: <= 1 ulp (tests/test_gpu_api.py).
static __constant__ double EXPC[16] = {
    1.0 / 6227020800.0, 1.0 / 479001600.0, 1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 5040.0,
    1.0 / 720.0, 1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5,
    1.4426950408889634,            // [12] log2(e)
    6755399441055744.0,            // [13] 1.5 * 2^52: adding it rounds to the nearest integer
    -6.93147180369123816490e-01,   // [14] -ln2 (high part)
    -1.90821492927058770002e-10};  // [15] -ln2 (low part)

__device__ __forceinline__ double exp_nonpos(double x) {
    const double t = fma(x, EXPC[12], EXPC[13]);
    const int k = __double2loint(t);
    const double kf = t - EXPC[13];
    double r = fma(kf, EXPC[14], x);
    r = fma(kf, EXPC[15], r);
    double p = EXPC[0];
#pragma unroll
    for (int c = 1; c < 12; c++) p = fma(p, r, EXPC[c]);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const double res = __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
    return x < -707.0 ? 0.0 : res;
}

// covariance from the scaled squared distance with the kernel class fixed at compile time (0: SE, 1: Matern-3/2,
// 2: Matern-5/2) -- same formulas as cov_r2
template <int KC>
__device__ __forceinline__ double cov_r2_t(double sf2, double r2) {
    if (KC == 0) return sf2 * exp_nonpos(-0.5 * r2);
    const double r = sqrt(r2);
    if (KC == 1) {
        const double z = 1.7320508075688772 * r;
        return sf2 * (1.0 + z) * exp_nonpos(-z);
    }
    const double z = 2.23606797749979 * r;
    return sf2 * (1.0 + z + 5.0 * r2 / 3.0) * exp_nonpos(-z);
}

__device__ __forceinline__ double erf_nr(double z) {
    // Numerical-Recipes Chebyshev erf, ego/gaussianprocess/__init__.py:55-71 (same constants, Horner order)
    double t = 1.0 / (1.0 + 0.5 * fabs(z));
    double p = 0.17087277;
    p = -0.82215223 + t * p;
    p = 1.48851587 + t * p;
    p = -1.13520398 + t * p;
    p = 0.27886807 + t * p;
    p = -0.18628806 + t * p;
    p = 0.09678418 + t * p;
    p = 0.37409196 + t * p;
    p = 1.00002368 + t * p;
    double ans = 1 - t * exp(-z * z - 1.26551223 + t * p);
    return z >= 0.0 ? ans : -ans;
}

// d erf_nr / dz: erf_nr(z) = sign(z) g(|z|), g(u) = 1 - t e^E, t = 1 / (1 + u / 2), E = -u^2 - 1.26551223 + t p(t), so the
// derivative is g'(|z|) = -e^E (t' + t E') with t' = -t^2 / 2 and E' = -2 u + t' (p + t p').  The derivative of the formula
// erf_nr evaluates (same constants, Horner order), not of the exact erf.
__device__ __forceinline__ double erf_nr_deriv(double z) {
    const double u = fabs(z);
    const double t = 1.0 / (1.0 + 0.5 * u);
    double p = 0.17087277, dp = 0.0;
    dp = p + t * dp; p = -0.82215223 + t * p;
    dp = p + t * dp; p = 1.48851587 + t * p;
    dp = p + t * dp; p = -1.13520398 + t * p;
    dp = p + t * dp; p = 0.27886807 + t * p;
    dp = p + t * dp; p = -0.18628806 + t * p;
    dp = p + t * dp; p = 0.09678418 + t * p;
    dp = p + t * dp; p = 0.37409196 + t * p;
    dp = p + t * dp; p = 1.00002368 + t * p;
    const double e = exp(-u * u - 1.26551223 + t * p);
    const double dt = -0.5 * t * t;
    const double dE = -2.0 * u + dt * (p + t * dp);
    return -e * (dt + t * dE);
}

// partial derivatives of acq_value with respect to mu and s = sqrt(s2), in the same arithmetic: libm mode through the exact
// pair (Phi, phi); Python mode through the derivative of its own formula (erf_nr, 0.707106, 0.398942)
__device__ __forceinline__ void acq_partials(int acq, int mode_py, double mu, double s2, double ymax, double parm, double* dmu,
                                             double* ds) {
    const double s = sqrt(s2);
    if (acq == IBO_ACQ_UCB) { *dmu = 1.0; *ds = parm; return; }
    const double Z = (acq == IBO_ACQ_EI ? mu - ymax - parm : mu - (ymax + parm)) / s;
    if (mode_py) {
        const double cdf = 0.5 * (1 + erf_nr(Z * 0.707106));
        const double dcdf = 0.5 * 0.707106 * erf_nr_deriv(Z * 0.707106);
        if (acq == IBO_ACQ_PI) { *dmu = dcdf / s; *ds = -Z * dcdf / s; return; }
        const double pdf = exp(-(Z * Z / 2)) * 0.398942;
        const double dpdf = -Z * pdf;
        // v = ydiff cdf(Z) + s pdf(Z), ydiff = s Z
        *dmu = cdf + Z * dcdf + dpdf;
        *ds = pdf - Z * Z * dcdf - Z * dpdf;
        return;
    }
    const double pdf = exp(-(Z * Z / 2.)) / 2.5066282746310002;
    if (acq == IBO_ACQ_PI) { *dmu = pdf / s; *ds = -Z * pdf / s; return; }
    *dmu = 0.5 * (1. + erf(Z / 1.4142135623730951));
    *ds = pdf;
}

__device__ __forceinline__ double acq_value(int acq, int mode_py, double mu, double s2, double ymax, double parm) {
    double s = sqrt(s2);
    if (acq == IBO_ACQ_UCB) return mu + parm * s;
    if (mode_py) {
        if (acq == IBO_ACQ_EI) {
            double ydiff = mu - ymax - parm;                                   // acquisition/__init__.py:156
            double Z = ydiff / s;
            double cdf = 0.5 * (1 + erf_nr(Z * 0.707106));                     // gaussianprocess/__init__.py:73-74
            double pdf = exp(-(Z * Z / 2)) * 0.398942;                         // :76-77
            return ydiff * cdf + s * pdf;                                      // acquisition/__init__.py:160
        }
        double Z = (mu - (ymax + parm)) / s;                                   // acquisition/__init__.py:105,110
        return 0.5 * (1 + erf_nr(Z * 0.707106));
    }
    double ydiff = mu - ymax - parm;                                           // cpp/optimizeGP.cpp:200
    double Z = ydiff / s;
    double cdf = 0.5 * (1. + erf(Z / 1.4142135623730951));                     // :202
    if (acq == IBO_ACQ_PI) return cdf;                                         // :225-226
    double pdf = exp(-(Z * Z / 2.)) / 2.5066282746310002;                      // :203  sqrt(2*pi)
    return ydiff * cdf + s * pdf;                                              // :204
}

// RBF-network mean prior at one point, ego/gaussianprocess/prior.py:60-66 == cpp/optimizeGP.cpp:116-134
__device__ __forceinline__ double prior_mean(const double* __restrict__ x, int d, int npb, const double* __restrict__ pmeans,
                                             const double* __restrict__ pbeta, double ptheta, const double* __restrict__ plb,
                                             const double* __restrict__ pwidth) {
    double m0 = 0.0;
    for (int b = 0; b < npb; b++) {
        double dd = 0;
        for (int j = 0; j < d; j++) {
            double t = (x[j] - plb[j]) / pwidth[j] - pmeans[(size_t)b * d + j];
            dd += t * t;
        }
        m0 += pbeta[b] * exp(-ptheta * dd);
    }
    return m0;
}

struct ScoreReq {
    int acq;            // -1: posterior only
    double ymax, parm;
    int flags;
    bool want_score, want_mu, want_s2;
    bool want_argmax = true;
    ScoreForce force = ScoreForce::None;
};

}  // namespace ibo
