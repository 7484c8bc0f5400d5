// Pathwise posterior samples (Matheron's rule, Wilson et al. 2020): S posterior sample paths of one model as deterministic functions
//
//   f_s(x) = mu(x) + phi(x)^T w_s - k_g(x)^T c_s,   c_s = R_g^-1 (Phi_g w_s + E e_s)
//   phi_j(x) = sqrt(2 sf2 / F) cos(omega_j . x / theta + b_j)       (random Fourier features of the prior)
//   mu(x) = m0(x) + k_m(x)^T a - m0(x) k_m(x)^T b,  a = R_m^-1 Y, b = R_m^-1 1
//
// g is the variance model when one is attached, else the model.  Create does the O(N^2 S) work once: Phi_g w with the eval kernel on
// g's own training points, the noise draw, and c through the two W GEMMs of joint.cu.  Every candidate then costs one pass over the
// training rows and one over the features: no M x M matrix and no cap on M.
//
// Eval: one CTA per 64 candidates x 64 path columns.  The rows run in a fixed order over up to three segments (the model's training
// rows with coefficients a - c_s, or a and then g's rows with -c_s when a variance model is attached; then the F frequencies with w_s).
// Per stage of 32 rows the CTA computes the 32 x 64 feature values (kernel values from direct differences, or the cosine features)
// into shared memory and multiplies them with the 32 x 64 coefficient slice on the FP64 pipe; each value is one FMA chain over the
// rows in order, so a candidate's values do not depend on the other candidates of the call and ibo_paths_grad repeats the same chain
// to the bit.  A snapshot holds copies of everything it reads and runs on its own stream.
#include "model.cuh"
#include "scoremath.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace ibo {
namespace {

constexpr int PT = 64;     // candidates per CTA
constexpr int PC = 64;     // path columns per CTA
constexpr int PK = 32;     // rows per stage; every segment is padded to a multiple of it with zero coefficient rows
constexpr int MAXF = 65536, MAXS = 1024;

enum { SEG_KM = 0, SEG_KG = 1, SEG_FEAT = 2 };   // kernel rows with candidates scaled like the model's / g's points; features

struct PathsDev {
    const double* rows;    // [R][d]: scaled, centred training inputs, or frequencies omega
    const double* phase;   // [R]: folded phases b_j + omega_j . centre_g (feature rows), 0 elsewhere
    const double* coef;    // [R][ldc]
    int ldc, nseg, d, kindm, kindg;
    int segEnd[3], segKind[3];
    double sf2m, sf2g, amp;
};

// covariance from the scaled squared distance, cov_r2's formulas with every rounding explicit: the eval and gradient kernels compute
// the same bits whatever the compiler contracts around them
__device__ __forceinline__ double kern_val(int kind, double sf2, double r2) {
    if (kind <= IBO_KERNEL_SE_ISO) return __dmul_rn(sf2, exp(__dmul_rn(-0.5, r2)));
    const double r = sqrt(r2);
    if (kind == IBO_KERNEL_MATERN3) {
        const double z = __dmul_rn(1.7320508075688772, r);
        return __dmul_rn(__dmul_rn(sf2, __dadd_rn(1.0, z)), exp(-z));
    }
    const double z = __dmul_rn(2.23606797749979, r);
    const double p = __dadd_rn(__dadd_rn(1.0, z), __ddiv_rn(__dmul_rn(5.0, r2), 3.0));
    return __dmul_rn(__dmul_rn(sf2, p), exp(-z));
}

// one feature value of a candidate c (scaled like the segment wants) against row `r`; *aux = r^2 (kernel rows) or the cosine's argument
__device__ __forceinline__ double feature(const PathsDev& P, int sk, int r, const double* c, double* aux) {
    const double* x = P.rows + (size_t)r * P.d;
    if (sk == SEG_FEAT) {
        double a = 0.0;
        for (int t = 0; t < P.d; t++) a = fma(x[t], c[t], a);
        a = __dadd_rn(a, P.phase[r]);
        *aux = a;
        return __dmul_rn(P.amp, cos(a));
    }
    double r2 = 0.0;
    for (int t = 0; t < P.d; t++) { const double df = __dsub_rn(x[t], c[t]); r2 = fma(df, df, r2); }
    *aux = r2;
    return sk == SEG_KM ? kern_val(P.kindm, P.sf2m, r2) : kern_val(P.kindg, P.sf2g, r2);
}

// the RBF prior mean with explicit roundings (the gradient kernel repeats it)
struct PriorDev { int npb; double ptheta; const double *pmeans, *pbeta, *plb, *pwidth; };
__device__ __forceinline__ double prior_m0(const PriorDev& Q, const double* x, int d) {
    double m0 = 0.0;
    for (int b = 0; b < Q.npb; b++) {
        double dd = 0.0;
        for (int t = 0; t < d; t++) {
            const double q = __dsub_rn(__ddiv_rn(__dsub_rn(x[t], Q.plb[t]), Q.pwidth[t]), Q.pmeans[(size_t)b * d + t]);
            dd = fma(q, q, dd);
        }
        m0 = fma(Q.pbeta[b], exp(__dmul_rn(-Q.ptheta, dd)), m0);
    }
    return m0;
}

// C[j][t] = X[j][t] * inv_theta[t] - centre[t] for the two scalings (model, g)
__global__ void __launch_bounds__(256) paths_scale_kernel(double* __restrict__ Cm, double* __restrict__ Cg, const double* __restrict__ X,
                                                          const double* __restrict__ itm, const double* __restrict__ cm,
                                                          const double* __restrict__ itg, const double* __restrict__ cg, long n, int d) {
    const long idx = blockIdx.x * 256L + threadIdx.x;
    if (idx >= n * d) return;
    const int t = (int)(idx % d);
    Cm[idx] = __dsub_rn(__dmul_rn(X[idx], itm[t]), cm[t]);
    Cg[idx] = __dsub_rn(__dmul_rn(X[idx], itg[t]), cg[t]);
}

// prior only: m0[j] and kb[j] = sum over the model's rows of k_i b_i (column ldc - 1 of the coefficients), in row order
__global__ void __launch_bounds__(128) paths_prior_kernel(PathsDev P, PriorDev Q, const double* __restrict__ X, const double* __restrict__ Cm,
                                                          int n, double* __restrict__ m0, double* __restrict__ kb) {
    const int j = blockIdx.x * 128 + threadIdx.x;
    if (j >= n) return;
    double acc = 0.0, aux;
    for (int r = 0; r < P.segEnd[0]; r++) acc = fma(feature(P, SEG_KM, r, Cm + (size_t)j * P.d, &aux), P.coef[(size_t)r * P.ldc + P.ldc - 1], acc);
    kb[j] = acc;
    m0[j] = prior_m0(Q, X + (size_t)j * P.d, P.d);
}

// values of n candidates on path columns [64 blockIdx.y, +64) of S: out[j][s] (leading dimension ldo, may be null), and per CTA and
// column the argmax over its 64 candidates (lowest index wins, NaN never wins; -1 when all are NaN)
__global__ void __launch_bounds__(256) paths_eval_kernel(PathsDev P, const double* __restrict__ Cm, const double* __restrict__ Cg, int n,
                                                         int S, const double* __restrict__ m0, const double* __restrict__ kb,
                                                         double* __restrict__ out, int ldo, double* __restrict__ blkBest,
                                                         long long* __restrict__ blkIdx, long long idx0) {
    extern __shared__ double sm[];
    const int d = P.d, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    double* sFeat = sm;                  // [PK][PT]
    double* sCoef = sFeat + PK * PT;     // [PK][PC]
    double* sCm = sCoef + PK * PC;       // [PT][d]
    double* sCg = sCm + PT * d;          // [PT][d]
    const int j0 = blockIdx.x * PT, col0 = blockIdx.y * PC;
    for (int idx = tid; idx < PT * d; idx += 256) {
        const int j = idx / d;
        sCm[idx] = j0 + j < n ? Cm[(size_t)j0 * d + idx] : 0.0;
        sCg[idx] = j0 + j < n ? Cg[(size_t)j0 * d + idx] : 0.0;
    }
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[i][c] = 0.0;
    const int R = P.segEnd[P.nseg - 1];
    int seg = 0;
    for (int r0 = 0; r0 < R; r0 += PK) {
        while (r0 >= P.segEnd[seg]) seg++;
        const int sk = P.segKind[seg];
        const double* cs = sk == SEG_KM ? sCm : sCg;
        __syncthreads();
        for (int idx = tid; idx < PK * PC; idx += 256) {
            const int k = idx / PC, c = idx - k * PC;
            sCoef[idx] = P.coef[(size_t)(r0 + k) * P.ldc + col0 + c];
        }
        for (int idx = tid; idx < PK * PT; idx += 256) {
            const int k = idx / PT, j = idx - k * PT;
            double aux;
            sFeat[idx] = feature(P, sk, r0 + k, cs + j * d, &aux);
        }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < PK; k++) {
            double fa[4], cb[4];
#pragma unroll
            for (int i = 0; i < 4; i++) fa[i] = sFeat[k * PT + ty + 16 * i];
#pragma unroll
            for (int c = 0; c < 4; c++) cb[c] = sCoef[k * PC + tx + 16 * c];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int c = 0; c < 4; c++) acc[i][c] = fma(fa[i], cb[c], acc[i][c]);
        }
    }
    __syncthreads();
    double* sOut = sm;                   // [PT][PC]
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int j = ty + 16 * i;
        double a0 = 0.0, b0 = 0.0;
        if (m0 && j0 + j < n) { a0 = m0[j0 + j]; b0 = kb[j0 + j]; }
#pragma unroll
        for (int c = 0; c < 4; c++) sOut[j * PC + tx + 16 * c] = m0 ? fma(-a0, b0, __dadd_rn(a0, acc[i][c])) : acc[i][c];
    }
    __syncthreads();
    if (out)
        for (int idx = tid; idx < PT * PC; idx += 256) {
            const int j = idx / PC, c = idx - j * PC;
            if (j0 + j < n && col0 + c < S) out[(size_t)(j0 + j) * ldo + col0 + c] = sOut[idx];
        }
    if (blkBest && tid < PC && col0 + tid < S) {
        double bv = -INFINITY;
        long long bi = -1;
        for (int j = 0; j < PT && j0 + j < n; j++) {
            const double v = sOut[j * PC + tid];
            if (!isnan(v) && (bi < 0 || v > bv)) { bv = v; bi = idx0 + j0 + j; }
        }
        blkBest[(size_t)blockIdx.x * S + col0 + tid] = bv;
        blkIdx[(size_t)blockIdx.x * S + col0 + tid] = bi;
    }
}

// best[s] / idx[s] = the running argmax merged with the nblk per-CTA partials of this chunk in ascending order (first: no running value)
__global__ void __launch_bounds__(128) paths_argmax_kernel(const double* __restrict__ blkBest, const long long* __restrict__ blkIdx, int nblk,
                                                           int S, double* __restrict__ best, long long* __restrict__ idx, int first) {
    const int s = blockIdx.x * 128 + threadIdx.x;
    if (s >= S) return;
    double bv = first ? -INFINITY : best[s];
    long long bi = first ? -1 : idx[s];
    for (int b = 0; b < nblk; b++) {
        const double v = blkBest[(size_t)b * S + s];
        const long long i = blkIdx[(size_t)b * S + s];
        if (i >= 0 && (bi < 0 || v > bv || (v == bv && i < bi))) { bv = v; bi = i; }
    }
    best[s] = bv;
    idx[s] = bi;
}

// one thread per point j on path which[j]: the value by the eval kernel's FMA chain (the same bits) and the gradient with respect to x
__global__ void __launch_bounds__(128) paths_grad_kernel(PathsDev P, PriorDev Q, const double* __restrict__ X, const double* __restrict__ Cm,
                                                         const double* __restrict__ Cg, int n, const int* __restrict__ which,
                                                         const double* __restrict__ itm, const double* __restrict__ itg,
                                                         double* __restrict__ val, double* __restrict__ G) {
    const int j = blockIdx.x * 128 + threadIdx.x;
    if (j >= n) return;
    const int d = P.d, s = which[j];
    const double* cm = Cm + (size_t)j * d;
    const double* cg = Cg + (size_t)j * d;
    double* g = G + (size_t)j * d;
    for (int t = 0; t < d; t++) g[t] = 0.0;
    const bool prior = Q.npb > 0;
    double acc = 0.0, kb = 0.0;
    int seg = 0;
    const int R = P.segEnd[P.nseg - 1];
    for (int r = 0; r < R; r++) {
        while (r >= P.segEnd[seg]) seg++;
        const int sk = P.segKind[seg];
        const double* c = sk == SEG_KM ? cm : cg;
        double aux;
        const double f = feature(P, sk, r, c, &aux);
        const double w = P.coef[(size_t)r * P.ldc + s];
        acc = fma(f, w, acc);
        const double* x = P.rows + (size_t)r * d;
        if (sk == SEG_FEAT) {
            if (w == 0.0) continue;
            const double e = -w * P.amp * sin(aux);
            for (int t = 0; t < d; t++) g[t] += e * x[t] * itg[t];
            continue;
        }
        double wb = 0.0;
        if (prior && sk == SEG_KM) { wb = P.coef[(size_t)r * P.ldc + P.ldc - 1]; kb = fma(f, wb, kb); }
        double k;
        const double h = sk == SEG_KM ? cov_grad_h(P.kindm, P.sf2m, aux, &k) : cov_grad_h(P.kindg, P.sf2g, aux, &k);
        const double* it = sk == SEG_KM ? itm : itg;
        for (int t = 0; t < d; t++) g[t] += -w * h * (c[t] - x[t]) * it[t];
    }
    double v = acc;
    if (prior) {
        const double* xr = X + (size_t)j * d;
        const double m0 = prior_m0(Q, xr, d);
        v = fma(-m0, kb, __dadd_rn(m0, acc));
        // the prior's share: (1 - k^T b) dm0 - m0 sum_i b_i dk_i
        for (int b = 0; b < Q.npb; b++) {
            double dd = 0.0;
            for (int t = 0; t < d; t++) {
                const double q = (xr[t] - Q.plb[t]) / Q.pwidth[t] - Q.pmeans[(size_t)b * d + t];
                dd += q * q;
            }
            const double e = (1.0 - kb) * Q.pbeta[b] * exp(-Q.ptheta * dd) * (-2.0 * Q.ptheta);
            for (int t = 0; t < d; t++) g[t] += e * ((xr[t] - Q.plb[t]) / Q.pwidth[t] - Q.pmeans[(size_t)b * d + t]) / Q.pwidth[t];
        }
        for (int r = 0; r < P.segEnd[0]; r++) {
            const double wb = P.coef[(size_t)r * P.ldc + P.ldc - 1];
            if (wb == 0.0) continue;
            double aux;
            feature(P, SEG_KM, r, cm, &aux);
            double k;
            const double h = cov_grad_h(P.kindm, P.sf2m, aux, &k);
            const double* x = P.rows + (size_t)r * d;
            for (int t = 0; t < d; t++) g[t] += m0 * wb * h * (cm[t] - x[t]) * itm[t];
        }
    }
    val[j] = v;
}

// V[i][s] (leading dimension ldv) += scale e[i][s] for i < n
__global__ void __launch_bounds__(256) add_scaled_kernel(double* __restrict__ V, int ldv, const double* __restrict__ e, int n, int S, double scale) {
    const long idx = blockIdx.x * 256L + threadIdx.x;
    if (idx >= (long)n * S) return;
    const long i = idx / S, s = idx - i * S;
    V[i * ldv + s] = fma(scale, e[idx], V[i * ldv + s]);
}

// lower tiles of inv(C) + (1 + noise - sf2) I over g's N points (identity in the padding, zeros above the diagonal), from the device's
// inv(C) (fromA = 0: src = inv(C), c = 1 + noise - sf2) or from A = R + inv(C) (fromA = 1: A - K with k(x, x) = sf2 on the diagonal)
__global__ void __launch_bounds__(256) noise_matrix_kernel(double* __restrict__ Nm, int Np, const double* __restrict__ src, int fromA,
                                                           const double* __restrict__ Xt, int N, int d, int kind, double sf2, double c) {
    const int j = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (j >= Np || (j >> 7) > (i >> 7)) return;
    double v;
    if (i >= N || j >= N) v = i == j ? 1.0 : 0.0;
    else if (j > i) v = 0.0;
    else if (!fromA) v = src[(size_t)i * Np + j] + (i == j ? c : 0.0);
    else if (i == j) v = src[(size_t)i * Np + j] - sf2;
    else {
        double r2 = 0.0;
        for (int t = 0; t < d; t++) { const double df = Xt[(size_t)i * d + t] - Xt[(size_t)j * d + t]; r2 = fma(df, df, r2); }
        v = src[(size_t)i * Np + j] - cov_r2(kind, sf2, r2);
    }
    Nm[(size_t)i * Np + j] = v;
}

// V[i][s] (leading dimension ldv) += sum_{k <= i} L[i][k] e[k][s] for i < n: the noise draw through the factor L (lower, leading
// dimension ldl; entries above the diagonal are not read)
__global__ void __launch_bounds__(256) tri_noise_kernel(double* __restrict__ V, int ldv, const double* __restrict__ L, int ldl,
                                                        const double* __restrict__ e, int S) {
    const int s = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (s >= S) return;
    double acc = 0.0;
    for (int k = 0; k <= i; k++) acc = fma(L[(size_t)i * ldl + k], e[(size_t)k * S + s], acc);
    V[(size_t)i * ldv + s] += acc;
}

// coefficient rows: the model's rows (a_i - c_i,s, or a_i with a variance model; b_i in the last column with a prior), g's rows (-c_i,s)
__global__ void __launch_bounds__(256) build_coef_kernel(double* __restrict__ coef, int ldc, int Nm, int Ng, int rowG, const double* __restrict__ a,
                                                         const double* __restrict__ b, const double* __restrict__ c, int ldcc, int S, int merged) {
    const int s = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (s >= ldc) return;
    if (i < Nm) {
        double v = 0.0;
        if (s < S) v = merged ? a[i] - c[(size_t)i * ldcc + s] : a[i];
        else if (s == ldc - 1 && b) v = b[i];
        coef[(size_t)i * ldc + s] = v;
    }
    if (!merged && i < Ng && s < S) coef[(size_t)(rowG + i) * ldc + s] = -c[(size_t)i * ldcc + s];
}

long round_to(long x, long k) { return (x + k - 1) / k * k; }

size_t eval_smem(int d) { return sizeof(double) * ((size_t)PK * PT + (size_t)PK * PC + 2 * (size_t)PT * d); }

cudaError_t set_paths_attrs() {
    return cudaFuncSetAttribute(paths_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eval_smem(64));
}

}  // namespace
}  // namespace ibo

struct ibo_paths {
    int device = 0;
    cudaStream_t stream = nullptr;
    int d = 0, F = 0, S = 0, Nm = 0, Ng = 0;
    bool prior = false;
    ibo::PathsDev P{};
    ibo::PriorDev Q{};
    double* dRows = nullptr;    // [R][d]
    double* dPhase = nullptr;   // [R]
    double* dCoef = nullptr;    // [R][ldc]
    double* dScale = nullptr;   // inv_theta_m | centre_m | inv_theta_g | centre_g  [4][d]
    double* dPrior = nullptr;   // pmeans | pbeta | plb | pwidth
    // per-call workspace, grown on demand
    double* dWork = nullptr; size_t workCap = 0;
};

namespace ibo {
namespace {

void free_paths(ibo_paths* p) {
    if (!p) return;
    cudaSetDevice(p->device);
    if (p->stream) cudaStreamSynchronize(p->stream);   // blocks go back to the pool: nothing may still be using them
    for (double* q : {p->dRows, p->dPhase, p->dCoef, p->dScale, p->dPrior, p->dWork}) pool_free(q);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

// candidates per chunk of an eval call: the chunk's whole workspace (raw and scaled candidates, m0 / kb, values, argmax partials:
// 3 d + S + 2 doubles per candidate and 2 S per 64 candidates) stays within 256 MiB
long eval_chunk(int d, int S) { return std::max<long>(PT, ((256L << 20) / (8L * (3L * d + S + 2 + (S + 31) / 32))) / PT * PT); }

// Enqueues on p->stream the values of n device candidates X (raw, [n][d]) into out (leading dimension ldo, may be null) and, when best
// is not null, the running argmax merge; the workspace w holds the scaled candidates, m0 / kb and the per-CTA partials.
int eval_device(ibo_paths* p, const double* X, long n, double* out, int ldo, double* best, long long* bestIdx, long long idx0, bool first,
                double* w) {
    const int d = p->d, S = p->S;
    const long nb = (n + PT - 1) / PT;
    double* Cm = w;
    double* Cg = Cm + (size_t)n * d;
    double* m0 = Cg + (size_t)n * d;
    double* kb = m0 + n;
    double* blkBest = kb + n;
    long long* blkIdx = reinterpret_cast<long long*>(blkBest + (size_t)nb * S);
    const double* sc = p->dScale;
    paths_scale_kernel<<<(unsigned)((n * d + 255) / 256), 256, 0, p->stream>>>(Cm, Cg, X, sc, sc + d, sc + 2 * d, sc + 3 * d, n, d);
    g_launches++;
    if (p->prior) {
        paths_prior_kernel<<<(unsigned)((n + 127) / 128), 128, 0, p->stream>>>(p->P, p->Q, X, Cm, (int)n, m0, kb);
        g_launches++;
    }
    paths_eval_kernel<<<dim3((unsigned)nb, (S + PC - 1) / PC), 256, eval_smem(d), p->stream>>>(
        p->P, Cm, Cg, (int)n, S, p->prior ? m0 : nullptr, kb, out, ldo, best ? blkBest : nullptr, blkIdx, idx0);
    g_launches++;
    if (best) {
        paths_argmax_kernel<<<(S + 127) / 128, 128, 0, p->stream>>>(blkBest, blkIdx, (int)nb, S, best, bestIdx, first ? 1 : 0);
        g_launches++;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

size_t eval_work(int d, int S, long n) { return (size_t)n * (2 * d + 2) + 2 * (size_t)((n + PT - 1) / PT) * S; }

}  // namespace
}  // namespace ibo

using namespace ibo;

extern "C" int ibo_paths_create(ibo_model* m, int F, int S, const double* omega, const double* phase, const double* w, const double* e,
                                ibo_paths** out, int* info) {
    if (info) *info = 0;
    if (!m || !omega || !phase || !w || !e || !out || F < 1 || F > MAXF || S < 1 || S > MAXS) { set_error("bad argument"); return IBO_E_BADARG; }
    if (m->d > 64) { set_error("d > 64 not supported"); return IBO_E_BADARG; }
    ibo_model* g = m->var_model ? m->var_model : m;
    if (g->sf2 > 1.0 + g->noise) { set_error("sample paths need sf2 <= 1 + noise"); return IBO_E_BADARG; }
    // a Laplace term: the noise factor needs inv(C) on the device (formed there by ibo_model_create_pref / _laplace), or A = R + inv(C),
    // which the model keeps up to 4096 points
    if (g->has_cinv && !g->dCinv && !g->dAorig) {
        set_error("sample paths of a model with inv(C) need inv(C) or A on the device (N <= 4096 for a host-supplied inv(C))");
        return IBO_E_BADARG;
    }
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    int rc;
    if ((rc = ensure_joint_attrs(m->device))) return rc;
    IBO_CUDA_TRY(set_paths_attrs());
    const int d = m->d, Nm = m->N, Ng = g->N;
    const bool merged = (g == m), prior = m->npb > 0;
    ibo_paths* p = new ibo_paths();
    p->device = m->device; p->d = d; p->F = F; p->S = S; p->Nm = Nm; p->Ng = Ng; p->prior = prior;
    auto fail = [&](int r) { free_paths(p); return r; };
    if (cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking) != cudaSuccess) { set_error("cudaStreamCreate failed"); return fail(IBO_E_CUDA); }
    // row layout: the model's rows, g's rows (variance model only), the frequencies; each padded to a multiple of PK
    const int r1 = (int)round_to(Nm, PK), r2 = merged ? r1 : r1 + (int)round_to(Ng, PK), R = r2 + (int)round_to(F, PK);
    const int ldc = (int)round_to(S + 1, PC);
    cudaStream_t st = m->stream;     // create reads the model: it runs on the model's stream and ends in a synchronisation
    size_t cap = 0;
    if ((rc = grow(&p->dRows, &cap, (size_t)R * d))) return fail(rc);
    cap = 0; if ((rc = grow(&p->dPhase, &cap, (size_t)R))) return fail(rc);
    cap = 0; if ((rc = grow(&p->dCoef, &cap, (size_t)R * ldc))) return fail(rc);
    cap = 0; if ((rc = grow(&p->dScale, &cap, (size_t)4 * d))) return fail(rc);
    if (cudaMemsetAsync(p->dRows, 0, sizeof(double) * (size_t)R * d, st) || cudaMemsetAsync(p->dPhase, 0, sizeof(double) * R, st) ||
        cudaMemsetAsync(p->dCoef, 0, sizeof(double) * (size_t)R * ldc, st)) { set_error("cudaMemsetAsync failed"); return fail(IBO_E_CUDA); }
    auto d2d = [&](double* dst, const double* src, size_t nd) { return cudaMemcpyAsync(dst, src, sizeof(double) * nd, cudaMemcpyDeviceToDevice, st); };
    auto h2d = [&](double* dst, const double* src, size_t nd) { return cudaMemcpyAsync(dst, src, sizeof(double) * nd, cudaMemcpyHostToDevice, st); };
#define TRYP(expr) do { if ((expr) != cudaSuccess) { cudaStreamSynchronize(st); set_error("paths create: copy failed"); return fail(IBO_E_CUDA); } } while (0)
    // frequencies, and the phases with g's centre folded in: omega . (x / theta) + b = omega . (x / theta - centre) + (b + omega . centre)
    std::vector<double> ph(F);
    for (int j = 0; j < F; j++) {
        double a = phase[j];
        for (int t = 0; t < d; t++) a += omega[(size_t)j * d + t] * g->hCenter[t];
        ph[j] = a;
    }
    TRYP(d2d(p->dRows, m->dXt, (size_t)Nm * d));
    if (!merged) TRYP(d2d(p->dRows + (size_t)r1 * d, g->dXt, (size_t)Ng * d));
    TRYP(h2d(p->dRows + (size_t)r2 * d, omega, (size_t)F * d));
    TRYP(h2d(p->dPhase + r2, ph.data(), F));
    TRYP(cudaMemcpy2DAsync(p->dCoef + (size_t)r2 * ldc, sizeof(double) * ldc, w, sizeof(double) * S, sizeof(double) * S, F,
                                   cudaMemcpyHostToDevice, st));
    TRYP(d2d(p->dScale, m->dInvTheta, d));
    TRYP(d2d(p->dScale + d, m->dCenter, d));
    TRYP(d2d(p->dScale + 2 * d, g->dInvTheta, d));
    TRYP(d2d(p->dScale + 3 * d, g->dCenter, d));
    if (prior) {
        const int nb = m->npb;
        cap = 0; if ((rc = grow(&p->dPrior, &cap, (size_t)nb * d + nb + 2 * d))) return fail(rc);
        TRYP(d2d(p->dPrior, m->dPmeans, (size_t)nb * d));
        TRYP(d2d(p->dPrior + (size_t)nb * d, m->dPbeta, nb));
        TRYP(d2d(p->dPrior + (size_t)nb * d + nb, m->dPlb, d));
        TRYP(d2d(p->dPrior + (size_t)nb * d + nb + d, m->dPwidth, d));
        p->Q.npb = nb; p->Q.ptheta = m->ptheta;
        p->Q.pmeans = p->dPrior; p->Q.pbeta = p->dPrior + (size_t)nb * d; p->Q.plb = p->Q.pbeta + nb; p->Q.pwidth = p->Q.plb + d;
    }
#undef TRYP
    PathsDev& P = p->P;
    P.rows = p->dRows; P.phase = p->dPhase; P.coef = p->dCoef; P.ldc = ldc; P.d = d;
    P.kindm = m->kind; P.kindg = g->kind; P.sf2m = m->sf2; P.sf2g = g->sf2; P.amp = std::sqrt(2.0 * g->sf2 / F);
    // Phi_g w: the eval kernel over the feature segment alone, with g's training points as the candidates.  The intermediates live in
    // the model's workspace: V (Phi_g w + E e, then c), T = W_g V, the normals e and a | b
    const int Sp = (int)round128(S), Npg = g->Np;
    CandWork* cw = cand_work(m);
    auto failc = [&](int r) { cudaStreamSynchronize(st); return fail(r); };
    if ((rc = grow(&cw->dV, &cw->vCap, (size_t)Npg * Sp)) || (rc = grow(&cw->dKc, &cw->kcCap, (size_t)Npg * Sp)) ||
        (rc = grow(&cw->dNormals, &cw->normalsCap, (size_t)Ng * S)) || (rc = grow(&cw->dAB, &cw->abCap, 2 * (size_t)m->Np)))
        return failc(rc);
    double *dV = cw->dV, *dT = cw->dKc, *dE = cw->dNormals, *dAB = cw->dAB;
    if (cudaMemsetAsync(dV, 0, sizeof(double) * (size_t)Npg * Sp, st) || cudaMemsetAsync(dAB, 0, sizeof(double) * 2 * (size_t)m->Np, st) ||
        h2d(dE, e, (size_t)Ng * S)) { set_error("copy failed"); return failc(IBO_E_CUDA); }
    {
        PathsDev Pf = P;
        Pf.rows = p->dRows + (size_t)r2 * d; Pf.phase = p->dPhase + r2; Pf.coef = p->dCoef + (size_t)r2 * ldc;
        Pf.nseg = 1; Pf.segEnd[0] = R - r2; Pf.segKind[0] = SEG_FEAT;
        // g's training inputs are stored scaled and centred like its candidates: pass them as both scalings
        const long nb = (Ng + PT - 1) / PT;
        paths_eval_kernel<<<dim3((unsigned)nb, (S + PC - 1) / PC), 256, eval_smem(d), st>>>(Pf, g->dXt, g->dXt, Ng, S, nullptr, nullptr, dV, Sp,
                                                                                           nullptr, nullptr, 0);
        g_launches++;
    }
    // + E e: sqrt(1 + noise - sf2) e for a plain, legacy or appended model; chol(inv(C) + (1 + noise - sf2) I) e with a Laplace term,
    // factorised on the device in the model's scratch factor (as joint.cu factorises Sigma); then c = W_g^T W_g (.)
    if (!g->has_cinv) {
        const double escale = std::sqrt(std::max(0.0, 1.0 + g->noise - g->sf2));
        add_scaled_kernel<<<(unsigned)(((long)Ng * S + 255) / 256), 256, 0, st>>>(dV, Sp, dE, Ng, S, escale);
        g_launches++;
    } else {
        if ((rc = chol_setup(m, Ng, false))) return failc(rc);
        Factor& sc = cw->chol;
        const bool fromA = g->dCinv == nullptr;
        noise_matrix_kernel<<<dim3((Npg + 255) / 256, Npg), 256, 0, st>>>(sc.dA, Npg, fromA ? g->dAorig : g->dCinv, fromA ? 1 : 0, g->dXt, Ng, d,
                                                                          g->kind, g->sf2, 1.0 + g->noise - g->sf2);
        g_launches++;
        int hinfo = 0;
        if ((rc = launch_factorize(*m, sc, false, false, false)) ||
            (rc = cudaMemcpyAsync(&hinfo, sc.dInfo, sizeof(int), cudaMemcpyDeviceToHost, st) || cudaStreamSynchronize(st) ? IBO_E_CUDA : 0))
            return failc(rc);
        if (hinfo != 0) {
            if (info) *info = hinfo;
            set_error("inv(C) + (1 + noise - sf2) I is not positive definite (pivot " + std::to_string(hinfo) + ")");
            return failc(IBO_E_NOTSPD);
        }
        tri_noise_kernel<<<dim3((S + 255) / 256, Ng), 256, 0, st>>>(dV, Sp, sc.dA, Npg, dE, S);
        g_launches++;
    }
    launch_w_gemm_v(dT, g, dV, Sp, st);
    launch_w_gemm_z(dV, g, dT, Sp, st);
    double* dB = launch_ab(m, dAB, st);
    build_coef_kernel<<<dim3((ldc + 255) / 256, std::max(Nm, Ng)), 256, 0, st>>>(p->dCoef, ldc, Nm, Ng, r1, dAB, dB, dV, Sp, S, merged ? 1 : 0);
    g_launches++;
    if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { set_error("paths create failed"); return failc(IBO_E_CUDA); }
    P.nseg = 0;
    P.segEnd[P.nseg] = r1; P.segKind[P.nseg++] = SEG_KM;
    if (!merged) { P.segEnd[P.nseg] = r2; P.segKind[P.nseg++] = SEG_KG; }
    P.segEnd[P.nseg] = R; P.segKind[P.nseg++] = SEG_FEAT;
    *out = p;
    return IBO_OK;
}

extern "C" int ibo_paths_eval(ibo_paths* p, const double* Xs, long M, double* values, double* best, long* best_idx) {
    if (!p || !Xs || M < 1) { set_error("bad argument"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(p->device));
    const int d = p->d, S = p->S;
    const long chunk = std::min<long>(round_to(M, PT), eval_chunk(d, S));
    const size_t raw = (size_t)chunk * d, vals = (size_t)chunk * S, res = 2 * (size_t)S;
    int rc;
    if ((rc = grow(&p->dWork, &p->workCap, raw + vals + res + eval_work(d, S, chunk)))) return rc;
    double* dX = p->dWork;
    double* dVals = dX + raw;
    double* dBest = dVals + vals;
    long long* dBestIdx = reinterpret_cast<long long*>(dBest + S);
    double* w = dBest + res;
    const bool wantArg = best || best_idx;
    for (long c0 = 0; c0 < M; c0 += chunk) {
        const long n = std::min(chunk, M - c0);
        IBO_CUDA_TRY(cudaMemcpyAsync(dX, Xs + (size_t)c0 * d, sizeof(double) * (size_t)n * d, cudaMemcpyHostToDevice, p->stream));
        if ((rc = eval_device(p, dX, n, values ? dVals : nullptr, S, wantArg ? dBest : nullptr, dBestIdx, c0, c0 == 0, w))) return rc;
        if (values) IBO_CUDA_TRY(cudaMemcpyAsync(values + (size_t)c0 * S, dVals, sizeof(double) * (size_t)n * S, cudaMemcpyDeviceToHost, p->stream));
        IBO_CUDA_TRY(cudaStreamSynchronize(p->stream));
    }
    if (wantArg) {
        std::vector<double> hb(S);
        std::vector<long long> hi(S);
        IBO_CUDA_TRY(cudaMemcpyAsync(hb.data(), dBest, sizeof(double) * S, cudaMemcpyDeviceToHost, p->stream));
        IBO_CUDA_TRY(cudaMemcpyAsync(hi.data(), dBestIdx, sizeof(long long) * S, cudaMemcpyDeviceToHost, p->stream));
        IBO_CUDA_TRY(cudaStreamSynchronize(p->stream));
        for (int s = 0; s < S; s++) {
            if (best) best[s] = hb[s];
            if (best_idx) best_idx[s] = (long)hi[s];
        }
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

extern "C" int ibo_paths_grad(ibo_paths* p, const double* Xs, long M, const int* which, double* values, double* grad) {
    if (!p || !Xs || M < 1 || M > (1L << 30) || !which || !values || !grad) { set_error("bad argument"); return IBO_E_BADARG; }
    for (long j = 0; j < M; j++)
        if (which[j] < 0 || which[j] >= p->S) { set_error("which[j] outside [0, S)"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(p->device));
    const int d = p->d;
    const size_t n = (size_t)M;
    int rc;
    if ((rc = grow(&p->dWork, &p->workCap, n * (4 * d + 1) + (n + 1) / 2))) return rc;
    double* dX = p->dWork;
    double* Cm = dX + n * d;
    double* Cg = Cm + n * d;
    double* G = Cg + n * d;
    double* V = G + n * d;
    int* dWhich = reinterpret_cast<int*>(V + n);
    cudaStream_t st = p->stream;
    IBO_CUDA_TRY(cudaMemcpyAsync(dX, Xs, sizeof(double) * n * d, cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(dWhich, which, sizeof(int) * n, cudaMemcpyHostToDevice, st));
    const double* sc = p->dScale;
    paths_scale_kernel<<<(unsigned)((n * d + 255) / 256), 256, 0, st>>>(Cm, Cg, dX, sc, sc + d, sc + 2 * d, sc + 3 * d, (long)n, d);
    paths_grad_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(p->P, p->Q, dX, Cm, Cg, (int)n, dWhich, sc, sc + 2 * d, V, G);
    g_launches += 2;
    IBO_CUDA_TRY(cudaMemcpyAsync(values, V, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(grad, G, sizeof(double) * n * d, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

extern "C" int ibo_paths_destroy(ibo_paths* p) {
    if (!p) return IBO_E_BADARG;
    free_paths(p);
    return IBO_OK;
}
