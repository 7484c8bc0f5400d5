// Max-value entropy search (Wang & Jegelka 2017): a Gumbel fit of the distribution of max f over a candidate set, and the MES
// values and gradients of candidates for samples y* of that maximum.
//
//   g_k = (y*_k - mu) / s,   psi = phi / Phi,   h(g) = g psi(g) / 2 - log Phi(g),   MES = (1 / K) sum_k h(g_k)
//   h'(g) = -(psi / 2) (1 + g (g + psi));   d MES / d mu = -(1 / (K s)) sum_k h'(g_k),   d MES / d s = -(1 / (K s)) sum_k g_k h'(g_k)
//
// mu and s2 come from the scoring path's kernels (posterior_score_device, ibo_posterior_batch's bits) or, with gradients, from
// grad_device (the FP64 kernels, with d mu and d s2 already clipped).  One thread per candidate evaluates h in ascending k.
// For t = -g / sqrt2 >= 1.5, where both g psi / 2 + g^2 / 2 and 1 + g (g + psi) cancel in the textbook form, h and h' come from
// the continued fraction of erfc:  sqrt(pi) erfcx(t) = 1 / (t + r_1),  r_k = (k / 2) / (t + r_(k+1)),  so that
//   psi = sqrt2 (t + r_1),  g psi / 2 + g^2 / 2 = (g / 2) sqrt2 r_1,  log Phi = -log(2 sqrt(pi) (t + r_1)) - g^2 / 2,
//   1 + g (g + psi) = r_2 / (t + r_2),
// with 12 + ceil(240 / t^2) terms (at most 119; enough for r_1 to the last bit over t >= 1.5).
#include "model.cuh"
#include <algorithm>
#include <cmath>

namespace ibo {

namespace {

constexpr int MES_MAX_K = 1024;     // y* staged in shared memory: 8 KiB
constexpr int GT = 15;              // Gumbel fit: trial points per bracket and pass (a pass narrows a bracket 16-fold)
constexpr int GPASS = 16;           // passes: 16 x 4 bits = 64 bits, past adjacent doubles from any bracket
constexpr int GS = 3 * GT;          // trial sums per block and pass
constexpr long GMAX_BLK = 1024;     // blocks of the fit's kernels: a function of M alone, so the summation order is too
constexpr int MES_FLAGS = IBO_FLAG_MODE_PY | IBO_FLAG_INT8 | IBO_FLAG_FP64;

__device__ __forceinline__ void mes_h(double g, double* h, double* dh) {
    const double t = -g * 0.70710678118654752440;
    if (t >= 1.5) {
        const int n = 12 + (int)ceil(240.0 / (t * t));
        double r = 0.0;
        for (int k = n; k >= 2; k--) r = (0.5 * k) / (t + r);
        const double r1 = 0.5 / (t + r);
        *h = (0.5 * g) * (1.41421356237309504880 * r1) + log(3.54490770181103205460 * (t + r1));     // 2 sqrt(pi)
        *dh = -(0.70710678118654752440 * (t + r1)) * (r / (t + r));
    } else {
        const double e = erfcx(t);
        const double psi = 0.79788456080286535588 / e;                                              // sqrt(2 / pi)
        const double lphi = g < 0.0 ? log(0.5 * e) - 0.5 * g * g : log1p(-0.5 * erfc(g * 0.70710678118654752440));
        *h = 0.5 * g * psi - lphi;
        *dh = -0.5 * psi * (1.0 + g * (g + psi));
    }
}

__device__ __forceinline__ double log_ncdf(double z) {
    return z < 0.0 ? log(0.5 * erfcx(-z * 0.70710678118654752440)) - 0.5 * z * z : log1p(-0.5 * erfc(z * 0.70710678118654752440));
}

// block argmax of the scoring path's K3: lowest index wins ties, NaN never wins
__device__ __forceinline__ void block_argmax(double sc, long long idx, double* blkBest, long long* blkIdx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double os = __shfl_xor_sync(0xffffffffu, sc, o);
        long long oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (os > sc || (os == sc && oi < idx)) { sc = os; idx = oi; }
    }
    __shared__ double ws[8];
    __shared__ long long wi[8];
    if ((threadIdx.x & 31) == 0) { ws[threadIdx.x >> 5] = sc; wi[threadIdx.x >> 5] = idx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++)
            if (ws[w] > sc || (ws[w] == sc && wi[w] < idx)) { sc = ws[w]; idx = wi[w]; }
        blkBest[blockIdx.x] = sc;
        blkIdx[blockIdx.x] = idx;
    }
}

// One thread per candidate: values[m] = MES at (mu[m], s2[m]); with dmu and ds, d MES / d mu and d MES / d s.  h and h' are
// evaluated on one code path whether or not the derivatives are written, so the values do not depend on it.
__global__ void __launch_bounds__(256) mes_value_kernel(const double* __restrict__ mu, const double* __restrict__ s2, long M,
                                                        const double* __restrict__ ystar, int K, double* __restrict__ values,
                                                        double* __restrict__ dmu, double* __restrict__ ds, double* __restrict__ blkBest,
                                                        long long* __restrict__ blkIdx) {
    __shared__ double ys[MES_MAX_K];
    for (int k = threadIdx.x; k < K; k += 256) ys[k] = ystar[k];
    __syncthreads();
    const long m = blockIdx.x * 256L + threadIdx.x;
    double sc = -INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    if (m < M) {
        const double u = mu[m], s = sqrt(s2[m]);
        double sh = 0.0, sdh = 0.0, sgdh = 0.0;
        for (int k = 0; k < K; k++) {
            const double g = (ys[k] - u) / s;
            double h, dh;
            mes_h(g, &h, &dh);
            sh += h;
            sdh += dh;
            sgdh = fma(g, dh, sgdh);
        }
        const double v = sh / K;
        values[m] = v;
        if (dmu) {
            const double f = -1.0 / (K * s);
            dmu[m] = f * sdh;
            ds[m] = f * sgdh;
        }
        if (v == v) sc = v;
        idx = m;
    }
    block_argmax(sc, idx, blkBest, blkIdx);
}

// One thread per candidate: plane 2 of G ([3][M][d]: ds2 | dmu | out) = d MES / d mu dmu + d MES / d s ds2 / (2 s); ds2 is already 0
// where s2 is clipped
__global__ void __launch_bounds__(256) mes_grad_epilogue_kernel(const double* __restrict__ post, const double* __restrict__ dmes, long M,
                                                                int d, double* __restrict__ G) {
    const long m = blockIdx.x * 256L + threadIdx.x;
    if (m >= M) return;
    const double a = dmes[m], b = dmes[M + m] * (0.5 / sqrt(post[2 * M + m]));
    const size_t plane = (size_t)M * d;
    double* g = G + (size_t)m * d;
    for (int t = 0; t < d; t++) g[2 * plane + t] = a * g[plane + t] + b * g[t];
}

// ---- Gumbel fit ----
// trial point j = 1 .. GT of the bracket [lo, hi]; the trial and the narrowing kernels compute it the same way
__device__ __forceinline__ double trial_point(double lo, double hi, int j) { return __fma_rn(hi - lo, j * (1.0 / (GT + 1)), lo); }

// per block: max_i (mu_i - s_i) and max_i (mu_i + c s_i) over a grid-stride share of the candidates -> ends[blk][2]
__global__ void __launch_bounds__(256) gumbel_bracket_kernel(const double* __restrict__ post, long M, double c, double* __restrict__ ends) {
    double lo = -INFINITY, hi = -INFINITY;
    for (long m = blockIdx.x * 256L + threadIdx.x; m < M; m += (long)gridDim.x * 256) {
        const double mu = post[M + m], s = sqrt(post[2 * M + m]);
        lo = fmax(lo, mu - s);
        hi = fmax(hi, fma(c, s, mu));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmax(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    __shared__ double sl[8], sh[8];
    if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = lo; sh[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) { lo = fmax(lo, sl[w]); hi = fmax(hi, sh[w]); }
        ends[2 * blockIdx.x] = lo;
        ends[2 * blockIdx.x + 1] = hi;
    }
}

// one CTA: every bracket starts as [max of the lower ends, max of the upper ends] -> state lo[3] | hi[3]
__global__ void __launch_bounds__(256) gumbel_init_kernel(const double* __restrict__ ends, long nblk, double* __restrict__ state) {
    double lo = -INFINITY, hi = -INFINITY;
    for (long b = threadIdx.x; b < nblk; b += 256) { lo = fmax(lo, ends[2 * b]); hi = fmax(hi, ends[2 * b + 1]); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmax(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    __shared__ double sl[8], sh[8];
    if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = lo; sh[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++) { lo = fmax(lo, sl[w]); hi = fmax(hi, sh[w]); }
        for (int b = 0; b < 3; b++) { state[b] = lo; state[3 + b] = hi; }
    }
}

// per block: sums[blk][b GT + j - 1] = sum_i log Phi((y_bj - mu_i) / s_i) over a grid-stride share of the candidates, for the GT
// trial points y_bj of each of the three brackets; each candidate's mu and s are loaded once.  Thread sums are added in candidate
// order, warps by a fixed shuffle tree, the eight warps in order.
__global__ void __launch_bounds__(256) gumbel_trial_kernel(const double* __restrict__ post, long M, const double* __restrict__ state,
                                                           double* __restrict__ sums) {
    __shared__ double ys[GS];
    __shared__ double part[8][GS];
    if (threadIdx.x < GS) {
        const int b = threadIdx.x / GT, j = threadIdx.x - b * GT + 1;
        ys[threadIdx.x] = trial_point(state[b], state[3 + b], j);
    }
    __syncthreads();
    double acc[GS];
#pragma unroll
    for (int u = 0; u < GS; u++) acc[u] = 0.0;
    for (long m = blockIdx.x * 256L + threadIdx.x; m < M; m += (long)gridDim.x * 256) {
        const double mu = post[M + m], inv_s = 1.0 / sqrt(post[2 * M + m]);
#pragma unroll
        for (int u = 0; u < GS; u++) acc[u] += log_ncdf((ys[u] - mu) * inv_s);
    }
#pragma unroll
    for (int u = 0; u < GS; u++) {
        double v = acc[u];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][u] = v;
    }
    __syncthreads();
    if (threadIdx.x < GS) {
        double v = part[0][threadIdx.x];
        for (int w = 1; w < 8; w++) v += part[w][threadIdx.x];
        sums[(size_t)blockIdx.x * GS + threadIdx.x] = v;
    }
}

// one CTA: adds the blocks' trial sums in ascending block order and narrows bracket b to the first trial point with
// log F >= logp[b] (its predecessor, or lo, becomes the new lower end); a bracket at adjacent doubles is left as it is
__global__ void __launch_bounds__(64) gumbel_narrow_kernel(const double* __restrict__ sums, long nblk, double* __restrict__ state,
                                                           double lp0, double lp1, double lp2) {
    __shared__ double tot[GS];
    if (threadIdx.x < GS) {
        double v = 0.0;
        for (long b = 0; b < nblk; b++) v += sums[(size_t)b * GS + threadIdx.x];
        tot[threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        const int b = threadIdx.x;
        const double lo = state[b], hi = state[3 + b], lp = b == 0 ? lp0 : (b == 1 ? lp1 : lp2);
        if (nextafter(lo, hi) < hi) {
            int j = 1;
            while (j <= GT && !(tot[b * GT + j - 1] >= lp)) j++;
            state[b] = j == 1 ? lo : trial_point(lo, hi, j - 1);
            state[3 + b] = j > GT ? hi : trial_point(lo, hi, j);
        }
    }
}

// Enqueues everything on m->stream: MES values in the score plane of w->dPost, the argmax at w->dPost[3 M], [3 M + 1] and, with
// wantGrad, the gradient in plane 2 of w->dG.
int mes_device(ibo_model* m, const double* Xs, long M, const double* ystar, int K, int flags, bool wantGrad) {
    int rc;
    CandWork* w = cand_work(m);
    cudaStream_t st = m->stream;
    const long nblk = (M + 255) / 256;
    if ((rc = grow(&w->dYstar, &w->ystarCap, (size_t)K))) return rc;
    if ((rc = grow(&w->dBlk, &w->blkCap, (size_t)2 * nblk))) return rc;
    if (wantGrad && (rc = grow(&w->dMesD, &w->mesDCap, (size_t)2 * M))) return rc;
    if (wantGrad) {
        if ((rc = grad_device(m, Xs, M, -1, 0.0, 0.0, flags, true))) return rc;
    } else {
        if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * m->d))) return rc;
        if ((rc = grow(&w->dPost, &w->postCap, (size_t)3 * M + 2))) return rc;
        IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * m->d, cudaMemcpyHostToDevice, st));
        if ((rc = posterior_score_device(m, w->dRaw, M, -1, 0.0, 0.0, flags, w->dPost))) return rc;
    }
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dYstar, ystar, sizeof(double) * K, cudaMemcpyHostToDevice, st));
    long long* blkIdx = reinterpret_cast<long long*>(w->dBlk + nblk);
    mes_value_kernel<<<(unsigned)nblk, 256, 0, st>>>(w->dPost + M, w->dPost + 2 * M, M, w->dYstar, K, w->dPost, wantGrad ? w->dMesD : nullptr,
                                                      wantGrad ? w->dMesD + M : nullptr, w->dBlk, blkIdx);
    g_launches++;
    launch_argmax_final(w->dBlk, blkIdx, nblk, w->dPost + 3 * M, reinterpret_cast<long long*>(w->dPost + 3 * M + 1), st);
    if (wantGrad) {
        mes_grad_epilogue_kernel<<<(unsigned)nblk, 256, 0, st>>>(w->dPost, w->dMesD, M, m->d, w->dG);
        g_launches++;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

}  // namespace

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_max_value_gumbel(ibo_model* m, const double* Xs, long M, int flags, double* q, double* loc, double* scale) {
    int rc = check_cands(m, Xs, M, (flags & ~MES_FLAGS) == 0);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    CandWork* w = cand_work(m);
    cudaStream_t st = m->stream;
    const long nblk = std::min((M + 255) / 256, GMAX_BLK);
    if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * m->d))) return rc;
    if ((rc = grow(&w->dPost, &w->postCap, (size_t)3 * M + 2))) return rc;
    if ((rc = grow(&w->dBlk, &w->blkCap, 8 + (size_t)nblk * (GS + 2)))) return rc;
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * m->d, cudaMemcpyHostToDevice, st));
    if ((rc = posterior_score_device(m, w->dRaw, M, -1, 0.0, 0.0, flags, w->dPost))) return rc;
    double* const state = w->dBlk;
    double* const sums = w->dBlk + 8;
    double* const ends = sums + (size_t)nblk * GS;
    // F(max(mu - s)) <= Phi(-1) < 0.25; with c = sqrt(2 ln 5M), -log F(max(mu + c s)) <= 1.04 / (5 c sqrt(2 pi)) < -log 0.75
    gumbel_bracket_kernel<<<(unsigned)nblk, 256, 0, st>>>(w->dPost, M, std::sqrt(2.0 * std::log(5.0 * (double)M)), ends);
    gumbel_init_kernel<<<1, 256, 0, st>>>(ends, nblk, state);
    g_launches += 2;
    for (int pass = 0; pass < GPASS; pass++) {
        gumbel_trial_kernel<<<(unsigned)nblk, 256, 0, st>>>(w->dPost, M, state, sums);
        gumbel_narrow_kernel<<<1, 64, 0, st>>>(sums, nblk, state, std::log(0.25), std::log(0.5), std::log(0.75));
        g_launches += 2;
    }
    double hs[6];
    IBO_CUDA_TRY(cudaMemcpyAsync(hs, state, sizeof(hs), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    const double* qq = hs + 3;
    const double sc = (qq[2] - qq[0]) / (std::log(-std::log(0.25)) - std::log(-std::log(0.75)));
    if (q) for (int b = 0; b < 3; b++) q[b] = qq[b];
    if (scale) *scale = sc;
    if (loc) *loc = qq[1] + sc * std::log(-std::log(0.5));
    return IBO_OK;
}

extern "C" int ibo_mes(ibo_model* m, const double* Xs, long M, const double* ystar, int K, int flags, double* values, double* dvalues,
                       double* best, long* best_idx) {
    bool ok = ystar && values && K >= 1 && K <= MES_MAX_K && (flags & ~MES_FLAGS) == 0 && !(dvalues && (flags & ~IBO_FLAG_MODE_PY));
    for (int k = 0; ok && k < K; k++) ok = std::isfinite(ystar[k]);
    int rc = check_cands(m, Xs, M, ok);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if ((rc = mes_device(m, Xs, M, ystar, K, flags, dvalues != nullptr))) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    double hb = 0.0;
    long long hi = -1;
    IBO_CUDA_TRY(cudaMemcpyAsync(values, w->dPost, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
    if (dvalues) IBO_CUDA_TRY(cudaMemcpyAsync(dvalues, w->dG + 2 * (size_t)M * m->d, sizeof(double) * (size_t)M * m->d, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(&hb, w->dPost + 3 * M, sizeof(double), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(&hi, w->dPost + 3 * M + 1, sizeof(long long), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    if (best) *best = hb;
    if (best_idx) *best_idx = (long)hi;
    return IBO_OK;
}
