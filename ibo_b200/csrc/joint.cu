// Joint posterior over a candidate set: the covariance between candidates, joint posterior samples and their per-sample argmax
// (Thompson batches).
//
//   V = W R(X, X*)               (Np x Mp, W = inv(L) of the model, exact zeros above its diagonal)
//   Sigma = R(X*, X*) - V^T V    (Mp x Mp, lower 128 x 128 tiles; identity in the padding)
//   F = mu 1^T + chol(Sigma + jitter I) Z
//
// R carries the model's own correlation function: k(x_i, x_j) off the diagonal, 1 + noise on it, so diag(Sigma) is the
// library's sigma^2 before clipping.  With a variance model attached (PrefGaussianProcess.addObservationPoint) Sigma comes
// from that model's X and W, as sigma^2 does; mu always comes from the scoring path (score.cu) on the FP64 kernels.
// Both GEMMs and the Cholesky of Sigma run on the FP64 tensor pipe (tile_gemm_core, launch_factorize).
// The candidate scaling, R(X, X*) and the two W GEMMs are launched through wrappers that grad.cu and qei.cu use as well.
#include "model.cuh"
#include "scoremath.cuh"
#include "tilegemm.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace ibo {

constexpr long JOINT_MAX_M = 16384;

namespace {

// Cs[j][t] = X[j][t] / theta_t - centre_t for j < M, 0 in the padding
__global__ void __launch_bounds__(256) scale_cands_kernel(double* __restrict__ Cs, const double* __restrict__ X, const double* __restrict__ inv_theta,
                                                          const double* __restrict__ center, long M, long Mp, int d) {
    const long idx = blockIdx.x * 256L + threadIdx.x;
    if (idx >= Mp * d) return;
    const long j = idx / d;
    const int t = (int)(idx - j * d);
    Cs[idx] = j < M ? X[idx] * inv_theta[t] - center[t] : 0.0;
}

// Kc[i][j] = k(x_i, x*_j) for i < N, j < M and exactly 0 elsewhere (W's padding rows are identity: any value there would reach V)
__global__ void __launch_bounds__(256) cross_cov_kernel(double* __restrict__ Kc, const double* __restrict__ Xt, const double* __restrict__ Cs,
                                                        int N, int M, int Mp, int d, int kind, double sf2) {
    const int j = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (j >= Mp) return;
    double v = 0.0;
    if (i < N && j < M) {
        double r2 = 0;
        for (int t = 0; t < d; t++) { double df = Xt[(size_t)i * d + t] - Cs[(size_t)j * d + t]; r2 = fma(df, df, r2); }
        v = cov_r2(kind, sf2, r2);
    }
    Kc[(size_t)i * Mp + j] = v;
}

// lower 128 x 128 tiles of R(X*, X*): k(x*_i, x*_j) off the diagonal ((min, max) order: exactly symmetric), `diag` on it, identity in
// the padding so that the padded matrix still factorises
__global__ void __launch_bounds__(256) prior_cov_kernel(double* __restrict__ S, const double* __restrict__ Cs, int M, int Mp, int d, int kind,
                                                        double sf2, double diag) {
    const int j = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (j >= Mp || (j >> 7) > (i >> 7)) return;
    double v;
    if (i >= M || j >= M) v = (i == j) ? 1.0 : 0.0;
    else if (i == j) v = diag;
    else {
        const int a = i < j ? i : j, b = i < j ? j : i;
        double r2 = 0;
        for (int t = 0; t < d; t++) { double df = Cs[(size_t)a * d + t] - Cs[(size_t)b * d + t]; r2 = fma(df, df, r2); }
        v = cov_r2(kind, sf2, r2);
    }
    S[(size_t)i * Mp + j] = v;
}

// C[I][J] = sum_{k <= I} T_Ik B_kJ (+ bias[row] for rows < nbias) over 128 x 128 blocks: T lower block-triangular with zeros above the
// diagonal inside its diagonal blocks, B dense.  K = (I + 1) 128, so the heaviest row blocks are scheduled first.
__global__ void __launch_bounds__(256, 1) trimm_kernel(double* __restrict__ C, int ldc, const double* __restrict__ T, int ldt,
                                                       const double* __restrict__ B, int ldb, int nbr, const double* __restrict__ bias, int nbias) {
    extern __shared__ double sm[];
    const int I = nbr - 1 - blockIdx.y, J = blockIdx.x;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    tile_gemm_core<false>(T + (size_t)I * 128 * ldt, ldt, B + (size_t)J * 128, ldb, (I + 1) * 128, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            const int row = I * 128 + wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            const double b = (bias && row < nbias) ? bias[row] : 0.0;
            *reinterpret_cast<double2*>(C + (size_t)row * ldc + (size_t)J * 128 + c) = make_double2(acc[mt][nt][0] + b, acc[mt][nt][1] + b);
        }
}

// The transposed twin of trimm_kernel: C[I][J] = sum_{k >= I} T_kI^T B_kJ, T as there (the transposed-A tile path).  K = (nbr - I) 128,
// so row block 0 is the heaviest and is scheduled first.  With T = W (identity padding rows) and B zero in its padding rows, C is
// zero in its padding rows.
__global__ void __launch_bounds__(256, 1) trimm_t_kernel(double* __restrict__ C, int ldc, const double* __restrict__ T, int ldt,
                                                         const double* __restrict__ B, int ldb, int nbr) {
    extern __shared__ double sm[];
    const int I = blockIdx.y, J = blockIdx.x;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    tile_gemm_core<false, true>(T + (size_t)I * 128 * ldt + (size_t)I * 128, ldt, B + (size_t)I * 128 * ldb + (size_t)J * 128, ldb,
                                (nbr - I) * 128, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            const int row = I * 128 + wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            *reinterpret_cast<double2*>(C + (size_t)row * ldc + (size_t)J * 128 + c) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
        }
}

// Dense tile GEMM C[I][J] = alpha op(A)_I B_J (+ C[I][J] when ACC), op(A) = A^T (A stored [K][rows]) with TRANSA, else A ([rows][K]);
// B [K][cols].  K is the full depth for every tile (a multiple of 16), so a column of C does not depend on the other columns.
// Padding rows and columns of C are zero when A and B are zero there (and C is, with ACC).
template <bool TRANSA, bool ACC>
__global__ void __launch_bounds__(256, 1) gemm_kernel(double* __restrict__ C, int ldc, const double* __restrict__ A, int lda,
                                                      const double* __restrict__ B, int ldb, int K, double alpha) {
    extern __shared__ double sm[];
    const int I = blockIdx.y, J = blockIdx.x;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    tile_gemm_core<false, TRANSA>(TRANSA ? A + (size_t)I * 128 : A + (size_t)I * 128 * lda, lda, B + (size_t)J * 128, ldb, K, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            const int row = I * 128 + wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            double2* p = reinterpret_cast<double2*>(C + (size_t)row * ldc + (size_t)J * 128 + c);
            double2 v;
            if (ACC) {
                v = *p;
                v.x = fma(alpha, acc[mt][nt][0], v.x);
                v.y = fma(alpha, acc[mt][nt][1], v.y);
            } else {
                v = make_double2(alpha * acc[mt][nt][0], alpha * acc[mt][nt][1]);
            }
            *p = v;
        }
}

// Sigma tile (I, J), J <= I, in place over R(X*, X*): S_IJ -= sum_k V_kI^T V_kJ (the transposed-A path of gram_wtw_kernel), + jitter on
// the diagonal of the real candidates
__global__ void __launch_bounds__(256, 1) sigma_kernel(double* __restrict__ S, const double* __restrict__ V, int Mp, int K, int M, double jitter) {
    extern __shared__ double sm[];
    const int I = blockIdx.y, J = blockIdx.x;
    if (J > I) return;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    tile_gemm_core<false, true>(V + (size_t)I * 128, Mp, V + (size_t)J * 128, Mp, K, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            const int r = I * 128 + wm * 64 + mt * 8 + (lane >> 2), c = J * 128 + wn * 32 + nt * 8 + 2 * (lane & 3);
            double2* p = reinterpret_cast<double2*>(S + (size_t)r * Mp + c);
            double2 v = *p;
            v.x -= acc[mt][nt][0];
            v.y -= acc[mt][nt][1];
            if (r < M) {
                if (r == c) v.x += jitter;
                if (r == c + 1) v.y += jitter;
            }
            *p = v;
        }
}

// the factor is left in the lower triangle; the upper triangle of each diagonal block still holds Sigma (potrf_diag_kernel writes
// the lower one only) and must read as zero in trimm_kernel
__global__ void __launch_bounds__(256) zero_diag_upper_kernel(double* __restrict__ A, int ld) {
    double* blk = A + (size_t)blockIdx.x * 128 * ld + (size_t)blockIdx.x * 128;
    for (int idx = threadIdx.x; idx < 128 * 128; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        if (c > r) blk[(size_t)r * ld + c] = 0.0;
    }
}

// arg[s] = argmax over the M rows of column s of F: lowest index wins ties, NaN never wins (-1 when every value is NaN).
// 32 columns per CTA, lane = column, warp w scans rows w, w + 8, ... in ascending order.
__device__ __forceinline__ bool better(double v, long long i, double bv, long long bi) {
    if (i < 0) return false;
    if (bi < 0) return true;
    return v > bv || (v == bv && i < bi);
}
// best (optional) receives the maximum itself (-inf when every value is NaN).
__global__ void __launch_bounds__(256) sample_argmax_kernel(const double* __restrict__ F, int ldf, int M, int S, long long* __restrict__ arg,
                                                            double* __restrict__ best) {
    __shared__ double sv[8][32];
    __shared__ long long si[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, s = blockIdx.x * 32 + lane;
    double bv = -INFINITY;
    long long bi = -1;
    if (s < S)
        for (int i = warp; i < M; i += 8) {
            const double v = F[(size_t)i * ldf + s];
            if (!isnan(v) && (bi < 0 || v > bv)) { bv = v; bi = i; }
        }
    sv[warp][lane] = bv; si[warp][lane] = bi;
    __syncthreads();
    if (warp == 0 && s < S) {
        for (int w = 1; w < 8; w++)
            if (better(sv[w][lane], si[w][lane], bv, bi)) { bv = sv[w][lane]; bi = si[w][lane]; }
        arg[s] = bi;
        if (best) best[s] = bv;
    }
}

cudaError_t set_joint_attrs() {
    cudaError_t e = cudaFuncSetAttribute(trimm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sigma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(trimm_t_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TILE_SMEM_DOUBLES * 8);
    return e;
}

// Enqueues on m->stream: the candidates Xs (host, M x d) to the device, mu of the scoring path into w->dPost + M (when wantMu),
// and Sigma + jitter I (lower tiles) into w->chol.dA.  S > 0: also grows the buffers of S samples.
int joint_sigma(ibo_model* m, const double* Xs, long M, double jitter, bool wantMu, int S) {
    int rc;
    if ((rc = ensure_joint_attrs(m->device))) return rc;
    CandWork* w = cand_work(m);
    ibo_model* g = m->var_model ? m->var_model : m;      // the model sigma^2 comes from
    cudaStream_t st = m->stream;
    const int d = m->d, Np = g->Np, Mp = (int)round128(M);
    const size_t Sp = (size_t)round128(S);
    if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * d))) return rc;
    if ((rc = grow(&w->dScaled, &w->scaledCap, (size_t)Mp * d))) return rc;
    if ((rc = grow(&w->dKc, &w->kcCap, (size_t)Np * Mp))) return rc;
    if ((rc = grow(&w->dV, &w->vCap, (size_t)Np * Mp))) return rc;
    if ((rc = grow(&w->dPost, &w->postCap, (size_t)3 * M + 2))) return rc;
    if ((rc = chol_setup(m, M, false))) return rc;
    if (S > 0) {
        if ((rc = grow(&w->dNormals, &w->normalsCap, (size_t)Mp * Sp))) return rc;
        if ((rc = grow(&w->dF, &w->fCap, (size_t)Mp * Sp))) return rc;
        if ((rc = grow(&w->dArg, &w->argCap, (size_t)S))) return rc;
    }
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * d, cudaMemcpyHostToDevice, st));
    if (wantMu && (rc = posterior_score_device(m, w->dRaw, M, -1, 0.0, 0.0, IBO_FLAG_FP64, w->dPost))) return rc;
    launch_scale_cands(w->dScaled, w->dRaw, g, M, Mp, st);
    launch_cross_cov(w->dKc, g, w->dScaled, (int)M, Mp, st);
    launch_w_gemm_v(w->dV, g, w->dKc, Mp, st);
    launch_joint_sigma(w->chol, w->dScaled, w->dV, g, 1.0 + g->noise, jitter, st);
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

}  // namespace

int chol_setup(ibo_model* m, long M, bool invert) {
    int rc;
    CandWork* w = cand_work(m);
    Factor& c = w->chol;
    if (!c.dInfo) IBO_CUDA_TRY(cudaMalloc(&c.dInfo, sizeof(int)));
    const int Mp = (int)round128(M), nbM = Mp / 128;
    if ((rc = grow(&c.dA, &w->cholACap, (size_t)Mp * Mp))) return rc;
    if ((rc = grow(&c.dD, &w->cholDCap, (size_t)nbM * 128 * 128))) return rc;
    if (invert) {
        if ((rc = grow(&c.dW, &w->cholWCap, (size_t)Mp * Mp))) return rc;
        if ((rc = grow(&c.dY, &w->cholYCap, (size_t)2 * Mp))) return rc;
        c.dBetaY = c.dY + Mp;
        IBO_CUDA_TRY(cudaMemsetAsync(c.dY, 0, sizeof(double) * Mp, m->stream));
    }
    c.N = (int)M; c.Np = Mp; c.nb = nbM;
    return IBO_OK;
}

void launch_joint_sigma(Factor& c, const double* Cs, const double* V, const ibo_model* g, double diag, double jitter, cudaStream_t st) {
    const int Mp = c.Np;
    prior_cov_kernel<<<dim3((Mp + 255) / 256, Mp), 256, 0, st>>>(c.dA, Cs, c.N, Mp, g->d, g->kind, g->sf2, diag);
    sigma_kernel<<<dim3(c.nb, c.nb), 256, TILE_SMEM_DOUBLES * 8, st>>>(c.dA, V, Mp, g->Np, c.N, jitter);
    g_launches += 2;
}

void launch_clear_diag_upper(Factor& c, cudaStream_t st) {
    zero_diag_upper_kernel<<<c.nb, 256, 0, st>>>(c.dA, c.Np);
    g_launches++;
}

void launch_sample_max(const double* F, int ldf, int M, int S, long long* arg, double* best, cudaStream_t st) {
    sample_argmax_kernel<<<(S + 31) / 32, 256, 0, st>>>(F, ldf, M, S, arg, best);
    g_launches++;
}

int check_cands(const ibo_model* m, const double* Xs, long M, bool extra_ok) {
    if (!m || !Xs || M < 1 || !extra_ok) { set_error("bad argument"); return IBO_E_BADARG; }
    if (m->d > 64) { set_error("d > 64 not supported"); return IBO_E_BADARG; }
    return IBO_OK;
}

int ensure_joint_attrs(int device) {
    cudaError_t ae = ensure_attrs(device, ATTR_JOINT, set_joint_attrs);
    if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); return IBO_E_CUDA; }
    return IBO_OK;
}

void launch_scale_cands(double* Cs, const double* X, const ibo_model* g, long M, long Mp, cudaStream_t st) {
    scale_cands_kernel<<<(unsigned)((Mp * g->d + 255) / 256), 256, 0, st>>>(Cs, X, g->dInvTheta, g->dCenter, M, Mp, g->d);
    g_launches++;
}
void launch_cross_cov(double* Kc, const ibo_model* g, const double* Cs, int M, int Mp, cudaStream_t st) {
    cross_cov_kernel<<<dim3((Mp + 255) / 256, g->Np), 256, 0, st>>>(Kc, g->dXt, Cs, g->N, M, Mp, g->d, g->kind, g->sf2);
    g_launches++;
}
void launch_w_gemm_v(double* V, const ibo_model* g, const double* Kc, int Mp, cudaStream_t st) {
    trimm_kernel<<<dim3(Mp / 128, g->nb), 256, TILE_SMEM_DOUBLES * 8, st>>>(V, Mp, g->dW, g->Np, Kc, Mp, g->nb, nullptr, 0);
    g_launches++;
}
void launch_w_gemm_z(double* Z, const ibo_model* g, const double* V, int Mp, cudaStream_t st) {
    trimm_t_kernel<<<dim3(Mp / 128, g->nb), 256, TILE_SMEM_DOUBLES * 8, st>>>(Z, Mp, g->dW, g->Np, V, Mp, g->nb);
    g_launches++;
}
void launch_cross_cov_pts(double* Kc, const double* Xa, int Na, int Nap, const ibo_model* g, const double* Cs, int M, int Mp, cudaStream_t st) {
    cross_cov_kernel<<<dim3((Mp + 255) / 256, Nap), 256, 0, st>>>(Kc, Xa, Cs, Na, M, Mp, g->d, g->kind, g->sf2);
    g_launches++;
}
void launch_trimm(double* C, int ldc, const double* T, int ldt, const double* B, int ldb, int nbr, int cols, const double* bias, int nbias,
                  cudaStream_t st) {
    trimm_kernel<<<dim3(cols / 128, nbr), 256, TILE_SMEM_DOUBLES * 8, st>>>(C, ldc, T, ldt, B, ldb, nbr, bias, nbias);
    g_launches++;
}
void launch_trimm_t(double* C, int ldc, const double* T, int ldt, const double* B, int ldb, int nbr, int cols, cudaStream_t st) {
    trimm_t_kernel<<<dim3(cols / 128, nbr), 256, TILE_SMEM_DOUBLES * 8, st>>>(C, ldc, T, ldt, B, ldb, nbr);
    g_launches++;
}
void launch_gemm(double* C, int ldc, const double* A, int lda, bool transA, const double* B, int ldb, int rows, int cols, int K,
                 double alpha, bool acc, cudaStream_t st) {
    const dim3 grid(cols / 128, rows / 128);
    const int sm = TILE_SMEM_DOUBLES * 8;
    if (transA) {
        if (acc) gemm_kernel<true, true><<<grid, 256, sm, st>>>(C, ldc, A, lda, B, ldb, K, alpha);
        else gemm_kernel<true, false><<<grid, 256, sm, st>>>(C, ldc, A, lda, B, ldb, K, alpha);
    } else {
        if (acc) gemm_kernel<false, true><<<grid, 256, sm, st>>>(C, ldc, A, lda, B, ldb, K, alpha);
        else gemm_kernel<false, false><<<grid, 256, sm, st>>>(C, ldc, A, lda, B, ldb, K, alpha);
    }
    g_launches++;
}

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_posterior_cov(ibo_model* m, const double* Xs, long M, double* mu, double* cov) {
    int rc = check_cands(m, Xs, M, M <= JOINT_MAX_M && cov != nullptr);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if ((rc = joint_sigma(m, Xs, M, 0.0, mu != nullptr, 0))) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    const size_t Mp = (size_t)round128(M);
    if (mu) IBO_CUDA_TRY(cudaMemcpyAsync(mu, w->dPost + M, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpy2DAsync(cov, sizeof(double) * M, w->chol.dA, sizeof(double) * Mp, sizeof(double) * M, M, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    // the device holds the lower tiles; mirror the lower triangle so that the result is exactly symmetric (64 x 64 blocks: the
    // column reads stay in cache)
    const long T = 64;
    for (long i0 = 0; i0 < M; i0 += T)
        for (long j0 = i0; j0 < M; j0 += T)
            for (long i = i0; i < std::min(i0 + T, M); i++)
                for (long j = std::max(j0, i + 1); j < std::min(j0 + T, M); j++) cov[i * M + j] = cov[j * M + i];
    return IBO_OK;
}

extern "C" int ibo_posterior_sample(ibo_model* m, const double* Xs, long M, const double* Z, int S, double jitter,
                                    double* F, long* argmax, int* info) {
    if (info) *info = 0;
    int rc = check_cands(m, Xs, M, M <= JOINT_MAX_M && Z && S >= 1 && jitter >= 0.0);      // NaN jitter fails the comparison
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if ((rc = joint_sigma(m, Xs, M, jitter, true, S))) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    const int Mp = (int)round128(M), nbM = Mp / 128, Sp = (int)round128(S);
    if ((rc = launch_factorize(*m, w->chol, false, false, false))) return rc;
    int hinfo = 0;
    IBO_CUDA_TRY(cudaMemcpyAsync(&hinfo, w->chol.dInfo, sizeof(int), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    if (hinfo != 0) {
        if (info) *info = hinfo;
        set_error("posterior covariance + jitter I is not positive definite (pivot " + std::to_string(hinfo) + ")");
        return IBO_E_NOTSPD;
    }
    launch_clear_diag_upper(w->chol, st);
    IBO_CUDA_TRY(cudaMemsetAsync(w->dNormals, 0, sizeof(double) * (size_t)Mp * Sp, st));
    IBO_CUDA_TRY(cudaMemcpy2DAsync(w->dNormals, sizeof(double) * Sp, Z, sizeof(double) * S, sizeof(double) * S, M, cudaMemcpyHostToDevice, st));
    trimm_kernel<<<dim3(Sp / 128, nbM), 256, TILE_SMEM_DOUBLES * 8, st>>>(w->dF, Sp, w->chol.dA, Mp, w->dNormals, Sp, nbM, w->dPost + M, (int)M);
    g_launches++;
    long long* dArg = reinterpret_cast<long long*>(w->dArg);
    std::vector<long long> harg(argmax ? S : 0);
    if (argmax) {
        launch_sample_max(w->dF, Sp, (int)M, S, dArg, nullptr, st);
        IBO_CUDA_TRY(cudaMemcpyAsync(harg.data(), dArg, sizeof(long long) * S, cudaMemcpyDeviceToHost, st));
    }
    if (F) IBO_CUDA_TRY(cudaMemcpy2DAsync(F, sizeof(double) * S, w->dF, sizeof(double) * Sp, sizeof(double) * S, M, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    for (int s = 0; s < (argmax ? S : 0); s++) argmax[s] = (long)harg[s];
    return IBO_OK;
}
