// Hyper-parameter learning on the device (SURVEY 8f-4): negative log marginal likelihood and its gradient.
//
// Replaces (reference file:line): trainhyper.marginalLikelihood / nlml / dnlml (ego/gaussianprocess/trainhyper.py:47-136,
// the useCholesky branch) and Kernel.covMatrix / Kernel.derivative (ego/gaussianprocess/kernel.py:43-52,92-105,120-127,
// 152-166,181-188,212-228,250-266):
//     K = covMatrix(X) + noise I,  L = chol(K),  alpha = inv(K) Y
//     nlml    = Y.alpha / 2 + sum_i log L_ii + N log(2 pi) / 2
//     dnlml_h = sum_ij (inv(K) - alpha alpha^T)_ij (dK / d log hyper_h)_ij / 2
// The reference forms inv(K) with two dense solves against the identity and one N x N derivative matrix per hyper-
// parameter through O(N^2) interpreted cov calls.  Here L and W = inv(L) come from the blocked DMMA factorisation of
// model.cu, inv(K) = W^T W is one triangular tile GEMM on the DMMA pipe (lower tiles only), and all derivative
// matrices are recomputed on the fly from the scaled inputs inside one fused reduction over the lower triangle
// (fixed summation order => deterministic).
#include "model.cuh"
#include "scoremath.cuh"
#include "tilegemm.cuh"
#include <cmath>
#include <mutex>
#include <vector>

namespace ibo {
namespace {

struct KDesc {
    int kind;      // IBO_KERNEL_*
    int nlen;      // number of length-scale hyperparameters (d for the ARD kinds, else 1)
    int has_mag;   // a magnitude hyperparameter follows the length scales
    int exact3;    // Matern-3/2: analytic derivative instead of the reference's expression
    double sf2;
    double theta0; // isotropic kinds: the length scale (Matern-3/2 reference expression needs the unscaled distance)
};

// dK_ij / d log hyper_h from the scaled squared distance r2, the scaled squared difference dh2 along dimension h
// (ARD kinds) and K_ij itself.
__device__ __forceinline__ double dk_value(const KDesc& kd, int h, double r2, double dh2, double kv) {
    if (h == kd.nlen) return 2.0 * kv;                                  // kernel.py:124-127,186-188,224-225,263-264
    switch (kd.kind) {
    case IBO_KERNEL_SE_ARD: return kv * dh2;                            // kernel.py:152-162
    case IBO_KERNEL_SE_ISO: return kv * r2;                             // kernel.py:92-101
    case IBO_KERNEL_MATERN3: {
        if (kd.exact3) { double z = 1.7320508075688772 * sqrt(r2); return kd.sf2 * z * z * exp(-z); }
        double r = kd.theta0 * sqrt(r2);                                // kernel.py:217-222: r = |xi - xj|, not divided by theta
        return kd.sf2 * r * r * exp(-r);
    }
    case IBO_KERNEL_MATERN5: {                                          // kernel.py:255-261
        double s = 2.23606797749979 * sqrt(r2);
        return kd.sf2 * (s * s + s * s * s) * exp(-s) / 3.0;
    }
    default: {                                                          // Matern-5/2 ARD (no reference class): analytic
        double s = 2.23606797749979 * sqrt(r2);
        return kd.sf2 * (5.0 / 3.0) * (1.0 + s) * exp(-s) * dh2;
    }
    }
}

// out[i][j] (N x N row-major) = covMatrix(X) (which < 0) or derivative(X, which)
__global__ void kernel_matrix_kernel(double* __restrict__ out, const double* __restrict__ Xt, int N, int d, KDesc kd, int which) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= N) return;
    int a = i < j ? i : j, b = i < j ? j : i;
    double r2 = 0, dh2 = 0;
    for (int t = 0; t < d; t++) {
        double df = Xt[(size_t)a * d + t] - Xt[(size_t)b * d + t];
        r2 += df * df;
        if (t == which) dh2 = df * df;
    }
    double kv = (i == j) ? kd.sf2 : cov_r2(kd.kind, kd.sf2, r2);
    out[(size_t)i * N + j] = which < 0 ? kv : dk_value(kd, which, r2, dh2, kv);
}

// Kinv tile (i, j), j <= i:  sum_{k >= i} W_ki^T W_kj  (W lower triangular with exact zeros above the diagonal)
__global__ void __launch_bounds__(256, 1) gram_wtw_kernel(double* __restrict__ C, const double* __restrict__ W, int Np) {
    extern __shared__ double sm[];
    const int nb = Np / 128;
    // heaviest tiles first: block row i has K = Np - 128 i
    const int i = blockIdx.y, j = blockIdx.x;
    if (j > i || i >= nb) return;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    const double* Wi = W + (size_t)i * 128 * Np;
    tile_gemm_core<false, true>(Wi + (size_t)i * 128, Np, Wi + (size_t)j * 128, Np, Np - i * 128, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
    double* Ct = C + (size_t)i * 128 * Np + (size_t)j * 128;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            int r = wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            double2 v;
            v.x = acc[mt][nt][0]; v.y = acc[mt][nt][1];
            *reinterpret_cast<double2*>(Ct + (size_t)r * Np + c) = v;
        }
}

// Fused gradient reduction over the lower triangle in 64 x 64 element tiles:
//   part[tile][a] = sum_{(i,j) in tile, j <= i} w_ij (Kinv_ij - alpha_i alpha_j) dK_ij/dlog hyper_{h0+a},  w = 2 off the diagonal
constexpr int GH = 8;    // hyperparameters per pass
constexpr int GT = 64;   // tile edge
__global__ void __launch_bounds__(256) grad_reduce_kernel(const double* __restrict__ Kinv, const double* __restrict__ alpha,
                                                          const double* __restrict__ Xt, int N, int Np, int d, KDesc kd, int h0, int nh,
                                                          double* __restrict__ part) {
    extern __shared__ double sm[];
    const int ti = blockIdx.y, tj = blockIdx.x;
    const int ntile = (N + GT - 1) / GT;
    if (tj > ti) return;
    double* Xi = sm;                  // [GT][d]
    double* Xj = sm + GT * d;         // [GT][d]
    double* red = Xj + GT * d;        // [8 warps][GH]
    const int tid = threadIdx.x;
    for (int idx = tid; idx < GT * d; idx += 256) {
        int r = idx / d, t = idx - r * d;
        int gi = ti * GT + r, gj = tj * GT + r;
        Xi[idx] = gi < N ? Xt[(size_t)gi * d + t] : 0.0;
        Xj[idx] = gj < N ? Xt[(size_t)gj * d + t] : 0.0;
    }
    __syncthreads();
    double acc[GH];
#pragma unroll
    for (int a = 0; a < GH; a++) acc[a] = 0.0;
    const int c = tid & 63, rg = tid >> 6;
    const int gj = tj * GT + c;
    const double aj = gj < N ? alpha[gj] : 0.0;
    for (int rr = 0; rr < 16; rr++) {
        const int r = rg * 16 + rr, gi = ti * GT + r;
        if (gi >= N || gj >= N || gj > gi) continue;
        // (min, max) = (gj, gi) ordering of the difference as in build_A_kernel
        double r2 = 0;
        for (int t = 0; t < d; t++) { double df = Xj[c * d + t] - Xi[r * d + t]; r2 += df * df; }
        const double kv = (gi == gj) ? kd.sf2 : cov_r2(kd.kind, kd.sf2, r2);
        const double g = (Kinv[(size_t)gi * Np + gj] - alpha[gi] * aj) * (gi == gj ? 1.0 : 2.0);
#pragma unroll
        for (int a = 0; a < GH; a++) {
            const int h = h0 + a;
            if (a < nh) {
                double dh2 = 0;
                if (h < kd.nlen && h < d) { double df = Xj[c * d + h] - Xi[r * d + h]; dh2 = df * df; }
                acc[a] = fma(g, dk_value(kd, h, r2, dh2, kv), acc[a]);
            }
        }
    }
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int a = 0; a < GH; a++) {
        double v = acc[a];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp * GH + a] = v;
    }
    __syncthreads();
    if (tid < GH) {
        double s = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) s += red[w * GH + tid];
        part[((size_t)ti * ntile + tj) * GH + tid] = s;
    }
}

// out[h0 + a] = sum over the lower tiles (fixed order) / 2
__global__ void __launch_bounds__(256) grad_final_kernel(const double* __restrict__ part, int ntile, int h0, int nh, double* __restrict__ out) {
    __shared__ double sh[256];
    for (int a = 0; a < nh; a++) {
        double s = 0;
        for (int idx = threadIdx.x; idx < ntile * ntile; idx += 256) {
            int ti = idx / ntile, tj = idx - ti * ntile;
            if (tj <= ti) s += part[(size_t)idx * GH + a];
        }
        sh[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) out[h0 + a] = 0.5 * sh[0];
        __syncthreads();
    }
}

// out[0] = beta.beta / 2 + sum_{i<N} log L_ii + N log(2 pi) / 2
__global__ void __launch_bounds__(256) nlml_value_kernel(const double* __restrict__ L, const double* __restrict__ beta, int N, int Np,
                                                         double* __restrict__ out) {
    __shared__ double sh[256];
    double s = 0;
    for (int i = threadIdx.x; i < N; i += 256) s += log(L[(size_t)i * Np + i]) + 0.5 * beta[i] * beta[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0] + 0.5 * N * 1.8378770664093453;   // log(2 pi)
}


int describe(int kind, const double* hyper, int nhyper, int d, int flags, KDesc* kd, int* nh_total) {
    if (kind < 0 || kind > IBO_KERNEL_MATERN5_ARD || !hyper || nhyper < 1) { set_error("bad kernel description"); return IBO_E_BADARG; }
    const bool ard = (kind == IBO_KERNEL_SE_ARD || kind == IBO_KERNEL_MATERN5_ARD);
    kd->kind = kind;
    kd->nlen = ard ? d : 1;
    if (nhyper < kd->nlen) { set_error("ARD kernel needs at least d hyperparameters"); return IBO_E_BADARG; }
    kd->has_mag = (kind != IBO_KERNEL_SE_ISO && nhyper > kd->nlen) ? 1 : 0;
    kd->exact3 = (flags & IBO_FLAG_GRAD_EXACT) ? 1 : 0;
    kd->sf2 = kd->has_mag ? exp(2.0 * log(hyper[kd->nlen])) : 1.0;      // kernel.py:63
    kd->theta0 = hyper[0];
    *nh_total = kd->nlen + kd->has_mag;
    return IBO_OK;
}

}  // namespace

static cudaError_t set_gram_attrs() {
    return cudaFuncSetAttribute(gram_wtw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
}
// C (lower 128 x 128 tiles, incl. full diagonal tiles) = W^T W for the lower-triangular W of a factorised model: inv(A) of its matrix
int launch_gram_wtw(double* C, const ibo_model* m, cudaStream_t st) {
    cudaError_t e = ensure_attrs(m->device, ATTR_GRAM, set_gram_attrs);
    if (e != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e)); return IBO_E_CUDA; }
    gram_wtw_kernel<<<dim3(m->nb, m->nb), 256, TILE_SMEM_DOUBLES * 8, st>>>(C, m->dW, m->Np);
    g_launches++;
    return IBO_OK;
}

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_nlml(int device, int kerneltype, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
                        double noise, int flags, double* nlml, double* dnlml, int* info) {
    if (info) *info = 0;
    if (!X || !Y || !nlml || N < 1 || d < 1) { set_error("bad argument"); return IBO_E_BADARG; }
    KDesc kd; int nh = 0;
    int rc = describe(kerneltype, hyper, nhyper, d, flags, &kd, &nh);
    if (rc) return rc;
    if (dnlml && nhyper > nh) {
        set_error("kernel has no derivative for hyperparameter " + std::to_string(nh) + " (kernel.py raises ValueError)");
        return IBO_E_BADARG;
    }
    ibo_model* m = nullptr;
    rc = create_model_with_diag(device, kerneltype, hyper, nhyper, X, Y, N, d, noise, kd.sf2 + noise, &m, info);
    if (rc) return rc;
    cudaStream_t st = m->stream;
    const int Np = m->Np;
    double* work = nullptr;      // [nlml | grad (nh) | alpha (Np)]
    double* dKinv = nullptr;
    double* dPart = nullptr;
    auto cleanup = [&]() {
        if (work) pool_free(work);
        if (dKinv) pool_free(dKinv);
        if (dPart) pool_free(dPart);
        ibo_model_destroy(m);
    };
#define TRYH(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { set_error(std::string(#expr) + ": " + cudaGetErrorString(e__)); cudaGetLastError(); cleanup(); return e__ == cudaErrorMemoryAllocation ? IBO_E_NOMEM : IBO_E_CUDA; } } while (0)
    TRYH(pool_malloc((void**)&work, sizeof(double) * (1 + (size_t)nh + Np)));
    double* dVal = work;
    double* dGrad = work + 1;
    double* dAlpha = dGrad + nh;
    nlml_value_kernel<<<1, 256, 0, st>>>(m->dA, m->dBetaY, N, Np, dVal);
    g_launches++;
    std::vector<double> hout(1 + nh, 0.0);
    if (dnlml) {
        TRYH(ensure_attrs(m->device, ATTR_GRAM, set_gram_attrs));
        TRYH(pool_malloc((void**)&dKinv, sizeof(double) * (size_t)Np * Np));
        const int ntile = (N + GT - 1) / GT;
        TRYH(pool_malloc((void**)&dPart, sizeof(double) * (size_t)ntile * ntile * GH));
        TRYH(cudaMemsetAsync(dAlpha, 0, sizeof(double) * Np, st));
        launch_tri_matvec_t(m->dW, m->dBetaY, dAlpha, N, Np, st);                     // alpha = W^T (W Y)
        gram_wtw_kernel<<<dim3(m->nb, m->nb), 256, TILE_SMEM_DOUBLES * 8, st>>>(dKinv, m->dW, Np);
        g_launches++;
        const size_t gsm = sizeof(double) * (2 * (size_t)GT * d + 8 * GH);
        if (gsm > 200 * 1024) { set_error("dimension too large for the gradient kernel"); cleanup(); return IBO_E_BADARG; }
        if (gsm > 48 * 1024) TRYH(cudaFuncSetAttribute(grad_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm));
        for (int h0 = 0; h0 < nh; h0 += GH) {
            const int cnt = nh - h0 < GH ? nh - h0 : GH;
            grad_reduce_kernel<<<dim3(ntile, ntile), 256, gsm, st>>>(dKinv, dAlpha, m->dXt, N, Np, d, kd, h0, cnt, dPart);
            grad_final_kernel<<<1, 256, 0, st>>>(dPart, ntile, h0, cnt, dGrad);
            g_launches += 2;
        }
    }
    TRYH(cudaMemcpyAsync(hout.data(), work, sizeof(double) * (1 + (dnlml ? nh : 0)), cudaMemcpyDeviceToHost, st));
    TRYH(cudaStreamSynchronize(st));
    TRYH(cudaGetLastError());
#undef TRYH
    *nlml = hout[0];
    if (dnlml) for (int h = 0; h < nhyper && h < nh; h++) dnlml[h] = hout[1 + h];
    cleanup();
    return IBO_OK;
}

extern "C" int ibo_kernel_matrix(int device, int kerneltype, const double* hyper, int nhyper, const double* X, int N, int d,
                                 int which, int flags, double* out) {
    if (!X || !out || N < 1 || d < 1) { set_error("bad argument"); return IBO_E_BADARG; }
    KDesc kd; int nh = 0;
    int rc = describe(kerneltype, hyper, nhyper, d, flags, &kd, &nh);
    if (rc) return rc;
    if (which >= nh) { set_error("kernel has no hyperparameter " + std::to_string(which)); return IBO_E_BADARG; }
    int ndev = ibo_device_count();
    if (ndev <= 0) { set_error("no CUDA device available (libibo_b200 has no CPU fallback)"); return IBO_E_CUDA; }
    if (device < 0 || device >= ndev) { set_error("bad device ordinal"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(device));
    const bool ard = (kerneltype == IBO_KERNEL_SE_ARD || kerneltype == IBO_KERNEL_MATERN5_ARD);
    std::vector<double> xt((size_t)N * d);
    for (int i = 0; i < N; i++)
        for (int t = 0; t < d; t++) {
            double th = ard ? hyper[t] : hyper[0];
            if (kerneltype == IBO_KERNEL_SE_ARD) th = fmin(fmax(th, 1e-4), 1e4);     // kernel.py:141
            xt[(size_t)i * d + t] = X[(size_t)i * d + t] * (1.0 / th);
        }
    double *dX = nullptr, *dOut = nullptr;
    auto cleanup = [&]() { if (dX) pool_free(dX); if (dOut) pool_free(dOut); };
#define TRYK(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { set_error(std::string(#expr) + ": " + cudaGetErrorString(e__)); cudaGetLastError(); cleanup(); return e__ == cudaErrorMemoryAllocation ? IBO_E_NOMEM : IBO_E_CUDA; } } while (0)
    TRYK(pool_malloc((void**)&dX, sizeof(double) * xt.size()));
    TRYK(pool_malloc((void**)&dOut, sizeof(double) * (size_t)N * N));
    TRYK(cudaMemcpy(dX, xt.data(), sizeof(double) * xt.size(), cudaMemcpyHostToDevice));
    kernel_matrix_kernel<<<dim3((N + 255) / 256, N), 256>>>(dOut, dX, N, d, kd, which);
    g_launches++;
    TRYK(cudaGetLastError());
    TRYK(cudaMemcpy(out, dOut, sizeof(double) * (size_t)N * N, cudaMemcpyDeviceToHost));
#undef TRYK
    cleanup();
    return IBO_OK;
}
