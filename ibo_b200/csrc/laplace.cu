// Laplace MAP fit of PrefGaussianProcess on the device (SURVEY 8f-2).
//
// Replaces (reference file:line): the functional S and its minimisation in PrefGaussianProcess.addPreferences
// (ego/gaussianprocess/__init__.py:355-386,441-442):
//     S(y) = - sum_p (deg_p + 1) log( CDF((y[v_p] - y[u_p]) / sqrt 2) + 1e-10 )  +  |inv(L) y|^2 / 2,   L = chol(R)
// with the reference's CDF (Chebyshev erf, constant 0.707106, :55-77).  The reference minimises S with BFGS on
// numerical gradients (N + 1 evaluations of an O(N^2) functional per step).  S is convex up to the 1e-10 guard, so
// here it is minimised by damped Newton steps in whitened coordinates y = L a:
//     grad_a = L^T g + a,   Hess_a = I + L^T Lambda L = I + G G^T,   G[:, p] = sqrt(w_p) (L[v_p, :] - L[u_p, :])^T
// (g, w: first / second derivatives of the preference terms).  B = I + G G^T is a rank-P update formed on the DMMA
// pipe, factorised with the blocked Cholesky of model.cu, and solved through its explicit triangular inverse.
#include "model.cuh"
#include <cmath>
#include <vector>

namespace ibo {
namespace {

__device__ __forceinline__ double erf_nr_d(double z) {      // ego/gaussianprocess/__init__.py:55-71
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

// per preference: the log term of S, dS/d(delta) and the curvature weight w >= 0
__global__ void pref_terms_kernel(const double* __restrict__ y, const int* __restrict__ v, const int* __restrict__ u,
                                  const double* __restrict__ deg, int P, double* __restrict__ logterm, double* __restrict__ gd,
                                  double* __restrict__ w) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const double eps = 1e-10;
    double z = (y[v[p]] - y[u[p]]) / 1.4142135623730951;                  // :384  (x[v]-x[u]) / (sqrt(2) sigma), sigma = 1
    double cdf = 0.5 * (1 + erf_nr_d(z * 0.707106));                       // :73-74
    double dp1 = deg[p] + 1.0;
    logterm[p] = dp1 * log(cdf + eps);                                     // :384
    double phi = exp(-0.5 * z * z) * 0.3989422804014327;
    double q = phi / (cdf + eps);
    gd[p] = -dp1 * q * 0.7071067811865476;                                 // d(-logterm)/d(delta), delta = y_v - y_u
    double ww = 0.5 * dp1 * (z * q + q * q);
    if (w) w[p] = ww > 0.0 ? ww : 0.0;
}

// gl[i] = sum over the preferences touching point i (CSR, fixed order) of +/- gd[p]
__global__ void pref_gather_kernel(const int* __restrict__ rowptr, const int* __restrict__ ent, const double* __restrict__ gd,
                                   double* __restrict__ gl, int N, int Np) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    double s = 0;
    if (i < N)
        for (int e = rowptr[i]; e < rowptr[i + 1]; e++) { int c = ent[e]; s += (c >= 0) ? gd[c] : -gd[~c]; }
    gl[i] = s;
}

// out[0] = -sum logterm + |a|^2 / 2, out[1] = |grad_a|_inf where grad_a = ltg + a (either may be skipped with NULL)
__global__ void __launch_bounds__(256) objective_kernel(const double* __restrict__ logterm, int P, const double* __restrict__ a,
                                                        const double* __restrict__ ltg, int N, double* __restrict__ out) {
    __shared__ double sh[8];
    double s = 0, q = 0, g = 0;
    for (int p = threadIdx.x; p < P; p += 256) s += logterm[p];
    for (int i = threadIdx.x; i < N; i += 256) {
        q = fma(a[i], a[i], q);
        if (ltg) g = fmax(g, fabs(ltg[i] + a[i]));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
        g = fmax(g, __shfl_xor_sync(0xffffffffu, g, o));
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    double S = 0;
    for (int w = 0; w < 8; w++) S += sh[w];
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = q;
    __syncthreads();
    double Q = 0;
    for (int w = 0; w < 8; w++) Q += sh[w];
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = g;
    __syncthreads();
    double Gm = 0;
    for (int w = 0; w < 8; w++) Gm = fmax(Gm, sh[w]);
    if (threadIdx.x == 0) { out[0] = -S + 0.5 * Q; out[1] = Gm; }
}

// G[i][p] = sqrt(w_p) (L[v_p][i] - L[u_p][i]); rows >= N and columns >= P are zero.  L is the lower triangle of `A`.
__global__ void build_G_kernel(const double* __restrict__ A, int Np, int N, const int* __restrict__ v, const int* __restrict__ u,
                               const double* __restrict__ w, int P, int K, double* __restrict__ G) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;      // row of G (fast: coalesced reads of L rows)
    int p = blockIdx.y;
    if (i >= Np) return;
    double val = 0.0;
    if (p < P && i < N) {
        int vp = v[p], up = u[p];
        double lv = i <= vp ? A[(size_t)vp * Np + i] : 0.0;
        double lu = i <= up ? A[(size_t)up * Np + i] : 0.0;
        val = sqrt(w[p]) * (lv - lu);
    }
    G[(size_t)i * K + p] = val;
}

__global__ void neg_sum_kernel(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out, int N, int Np) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < Np) out[i] = i < N ? -(a[i] + b[i]) : 0.0;
}
__global__ void axpy_kernel(const double* __restrict__ a, const double* __restrict__ d, double t, double* __restrict__ out, int N, int Np) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < Np) out[i] = i < N ? fma(t, d[i], a[i]) : 0.0;
}

struct Scratch {
    int *dV = nullptr, *dU = nullptr, *dRowptr = nullptr, *dEnt = nullptr;
    double* buf = nullptr;           // all double workspaces in one block
    ~Scratch() {
        if (dV) cudaFree(dV);
        if (dU) cudaFree(dU);
        if (dRowptr) cudaFree(dRowptr);
        if (dEnt) cudaFree(dEnt);
        if (buf) pool_free(buf);
    }
};

}  // namespace
}  // namespace ibo

using namespace ibo;

extern "C" int ibo_pref_fit(ibo_model* m, int P, const int* v, const int* u, const double* deg, double* y,
                            int maxit, double gtol, double* S_out, double* gnorm_out, int* iters_out) {
    if (!m || P < 1 || !v || !u || !deg || !y) { set_error("bad argument"); return IBO_E_BADARG; }
    if (m->cpp_prior || m->has_cinv) { set_error("ibo_pref_fit needs the plain R model of the preference points"); return IBO_E_BADARG; }
    const int N = m->N, Np = m->Np;
    for (int p = 0; p < P; p++)
        if (v[p] < 0 || v[p] >= N || u[p] < 0 || u[p] >= N) { set_error("preference index out of range"); return IBO_E_BADARG; }
    if (maxit <= 0) maxit = 100;
    if (!(gtol > 0)) gtol = 1e-9;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    const int K = ((P + BK - 1) / BK) * BK;
    Scratch sc;
#define TRYS(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { set_error(std::string(#expr) + ": " + cudaGetErrorString(e__)); cudaGetLastError(); return e__ == cudaErrorMemoryAllocation ? IBO_E_NOMEM : IBO_E_CUDA; } } while (0)
    // ---- B = I + G G^T, its factor and inverse factor: the model's scratch factor, factorised on the model's lanes ----
    int rc = chol_setup(m, N, true);
    if (rc) return rc;
    Factor& B = cand_work(m)->chol;
    // cleared here as well as by each factorisation: a start that already meets gtol runs none, and the pivot read after the
    // loop must see neither what a fresh allocation held nor the pivot an earlier failed factorisation on this model left there
    TRYS(cudaMemsetAsync(B.dInfo, 0, sizeof(int), st));
    // ---- preference index arrays + CSR (point -> its preferences, in preference order) ----
    std::vector<int> rowptr(N + 1, 0), ent(2 * (size_t)P);
    for (int p = 0; p < P; p++) { rowptr[v[p] + 1]++; rowptr[u[p] + 1]++; }
    for (int i = 0; i < N; i++) rowptr[i + 1] += rowptr[i];
    {
        std::vector<int> fill(rowptr.begin(), rowptr.end() - 1);
        for (int p = 0; p < P; p++) { ent[fill[v[p]]++] = p; ent[fill[u[p]]++] = ~p; }     // +gd for the winner, -gd for the loser
    }
    TRYS(cudaMalloc(&sc.dV, sizeof(int) * P));
    TRYS(cudaMalloc(&sc.dU, sizeof(int) * P));
    TRYS(cudaMalloc(&sc.dRowptr, sizeof(int) * (N + 1)));
    TRYS(cudaMalloc(&sc.dEnt, sizeof(int) * 2 * (size_t)P));
    TRYS(cudaMemcpyAsync(sc.dV, v, sizeof(int) * P, cudaMemcpyHostToDevice, st));
    TRYS(cudaMemcpyAsync(sc.dU, u, sizeof(int) * P, cudaMemcpyHostToDevice, st));
    TRYS(cudaMemcpyAsync(sc.dRowptr, rowptr.data(), sizeof(int) * (N + 1), cudaMemcpyHostToDevice, st));
    TRYS(cudaMemcpyAsync(sc.dEnt, ent.data(), sizeof(int) * ent.size(), cudaMemcpyHostToDevice, st));
    // ---- double workspaces ----
    const size_t nG = (size_t)Np * K;
    TRYS(pool_malloc((void**)&sc.buf, sizeof(double) * (nG + 4 * (size_t)P + 7 * (size_t)Np + 4)));
    double* G = sc.buf;
    double* dDeg = G + nG;
    double* logterm = dDeg + P;
    double* gd = logterm + P;
    double* w = gd + P;
    double* ya = w + P;          // y (original coordinates) of the current / trial point
    double* a = ya + Np;         // whitened coordinates
    double* at = a + Np;         // trial point
    double* gl = at + Np;        // gradient of the preference terms wrt y
    double* ltg = gl + Np;       // L^T gl
    double* da = ltg + Np;       // Newton direction
    double* tmp = da + Np;
    double* scal = tmp + Np;     // [S, |grad|_inf]
    TRYS(cudaMemcpyAsync(dDeg, deg, sizeof(double) * P, cudaMemcpyHostToDevice, st));
    TRYS(cudaMemsetAsync(ya, 0, sizeof(double) * Np, st));
    TRYS(cudaMemcpyAsync(ya, y, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    const int gp = (P + 255) / 256, gn = (Np + 255) / 256;
    launch_tri_matvec(m->dW, ya, a, Np, st);                        // a = inv(L) y

    double hs[2];
    // evaluates S and the gradient pieces at whitened point `pt`
    auto eval = [&](const double* pt, bool need_w) -> int {
        launch_tri_matvec(m->dA, pt, ya, Np, st);                   // y = L a
        pref_terms_kernel<<<gp, 256, 0, st>>>(ya, sc.dV, sc.dU, dDeg, P, logterm, gd, need_w ? w : nullptr);
        pref_gather_kernel<<<gn, 256, 0, st>>>(sc.dRowptr, sc.dEnt, gd, gl, N, Np);
        launch_tri_matvec_t(m->dA, gl, ltg, N, Np, st);             // L^T gl
        objective_kernel<<<1, 256, 0, st>>>(logterm, P, pt, ltg, N, scal);
        g_launches += 3;
        TRYS(cudaMemcpyAsync(hs, scal, sizeof(double) * 2, cudaMemcpyDeviceToHost, st));
        TRYS(cudaStreamSynchronize(st));
        return IBO_OK;
    };
    if ((rc = eval(a, true))) return rc;
    double S = hs[0], gn_inf = hs[1];
    int it = 0;
    for (; it < maxit && gn_inf > gtol; it++) {
        // B = I + G G^T, factorise, da = -inv(B) (L^T gl + a)
        build_G_kernel<<<dim3(gn, K), 256, 0, st>>>(m->dA, Np, N, sc.dV, sc.dU, w, P, K, G);
        g_launches++;
        if ((rc = launch_syrk_identity(B.dA, G, Np, K, st))) return rc;
        neg_sum_kernel<<<gn, 256, 0, st>>>(ltg, a, B.dY, N, Np);
        g_launches++;
        if ((rc = launch_factorize(*m, B, false, false, true))) return rc;   // B.dW = inv(chol(B)), B.dBetaY = dW * rhs
        TRYS(cudaMemsetAsync(da, 0, sizeof(double) * Np, st));
        launch_tri_matvec_t(B.dW, B.dBetaY, da, Np, Np, st);           // da = dW^T dW rhs
        // backtracking on S (convex: the full step is accepted except far from the optimum)
        double t = 1.0;
        bool ok = false;
        for (int ls = 0; ls < 30; ls++) {
            axpy_kernel<<<gn, 256, 0, st>>>(a, da, t, at, N, Np);
            g_launches++;
            if ((rc = eval(at, true))) return rc;
            if (std::isfinite(hs[0]) && hs[0] <= S + 1e-12 * fabs(S)) { ok = true; break; }
            t *= 0.5;
        }
        if (!ok) break;      // no decrease along the Newton direction: converged to rounding
        TRYS(cudaMemcpyAsync(a, at, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
        S = hs[0]; gn_inf = hs[1];
    }
    int hinfo = 0;
    TRYS(cudaMemcpy(&hinfo, B.dInfo, sizeof(int), cudaMemcpyDeviceToHost));
    // y = L a at the accepted point
    launch_tri_matvec(m->dA, a, ya, Np, st);
    TRYS(cudaMemcpyAsync(y, ya, sizeof(double) * N, cudaMemcpyDeviceToHost, st));
    TRYS(cudaStreamSynchronize(st));
    TRYS(cudaGetLastError());
#undef TRYS
    if (S_out) *S_out = S;
    if (gnorm_out) *gnorm_out = gn_inf;
    if (iters_out) *iters_out = it;
    if (hinfo) { set_error("Newton system of the Laplace fit is not positive definite"); return IBO_E_NOTSPD; }
    return IBO_OK;
}
