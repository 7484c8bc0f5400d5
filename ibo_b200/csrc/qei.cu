// Batch expected improvement (q-EI) of B batches of q points and its gradient with respect to the points, by Monte Carlo with
// caller-supplied standard normals Z[q][S] (Ginsbourger et al. 2010; reparameterisation gradients, Wilson et al. 2018):
//
//   qEI(b) = (1 / S) sum_s max(0, max_j (mu_b + L_b z_s)_j - ymax - xi),   L_b = chol(Sigma_b + jitter I)
//
// mu is the posterior mean sum_i a_i k_i (a = R^-1 Y; with the prior's terms), summed in a fixed order per point: the scoring path's
// FP64 mean groups its sums by the size of the call, which would make a batch's value depend on the other batches.
// Sigma_b = R(X*_b, X*_b) - V_b^T V_b is ibo_posterior_cov's (of the variance model when one is attached).  Reverse mode with Z
// fixed: per sample with positive improvement and argmax j* (lowest index wins), mubar_j* += 1 / S and Lbar_j*,k += z_k,s / S
// (k <= j*); the reverse Cholesky (Murray 2016) turns Lbar into the symmetric Gbar = d qEI / d Sigma (sum over all ordered pairs), and
//
//   d qEI / dx_j = mubar_j dmu(x_j) + 2 sum_l Gbar_jl d1 k(x_j, x_l) - 2 sum_i y_j,i dk_i(x_j) / dx_j,   y_j = sum_l Gbar_jl z_l
//
// with z_l = R_g^-1 k(X_g, x_l) = column l of W_g^T W_g K*.  Per chunk of whole batches: K* and V = W_g K* on the DMMA tile GEMM
// (joint.cu), the q x q blocks of Sigma on CUDA cores, one CTA per batch for the Cholesky, the sample loop and the reverse
// pass; with gradients Z = W_g^T V, y into V's buffer, and grad.cu's reduction with y in place of z.  Every sum runs in a fixed
// order without atomics and touches one batch only, so a batch's value and gradient do not depend on the other batches.
#include "model.cuh"
#include "scoremath.cuh"
#include <algorithm>
#include <cmath>
#include <string>

namespace ibo {

namespace {

constexpr int QEI_MAX_Q = 32;
constexpr int SIG_SLICES = 8;                                        // training points i = s, s + 8, ... per partial sum
constexpr int SIG_ROWS = 32;                                         // rows of V staged per step (a multiple of SIG_SLICES)
constexpr int SIG_ITEMS = QEI_MAX_Q * (QEI_MAX_Q + 1) / 2 * SIG_SLICES;
constexpr int SIG_PER_THREAD = (SIG_ITEMS + 255) / 256;
constexpr int QW = 4;                                                // warps of the per-batch kernel

// One CTA per batch: Sigma_b[j][l] = k(x_j, x_l) (diag on the diagonal) - sum_i V_ij V_il over the batch's q columns of V.  Item
// (pair p, slice s) sums the rows i = s (mod 8) in ascending order and the eight slices are added in slice order, so the order of
// every entry is the same whatever q is: a batch's Sigma_00 is that of its first point alone.
__global__ void __launch_bounds__(256) qei_sigma_kernel(double* __restrict__ Sig, const double* __restrict__ V, int ldv,
                                                        const double* __restrict__ Cs, int N, int q, int d, int kind, double sf2,
                                                        double diag) {
    __shared__ double tile[SIG_ROWS][QEI_MAX_Q + 1];
    __shared__ double part[SIG_ITEMS];
    const int b = blockIdx.x, c0 = b * q, np = q * (q + 1) / 2, items = np * SIG_SLICES;
    int pj[SIG_PER_THREAD], pl[SIG_PER_THREAD];
    double acc[SIG_PER_THREAD];
#pragma unroll
    for (int u = 0; u < SIG_PER_THREAD; u++) {
        const int p = (threadIdx.x + 256 * u) / SIG_SLICES;
        int j = 0;
        while ((j + 1) * (j + 2) / 2 <= p) j++;                      // p = j (j + 1) / 2 + l, l <= j
        pj[u] = j; pl[u] = p - j * (j + 1) / 2; acc[u] = 0.0;
    }
    for (int i0 = 0; i0 < N; i0 += SIG_ROWS) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < SIG_ROWS * q; idx += 256) {
            const int r = idx / q, c = idx - r * q;
            tile[r][c] = i0 + r < N ? V[(size_t)(i0 + r) * ldv + c0 + c] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < SIG_PER_THREAD; u++) {
            const int it = threadIdx.x + 256 * u;
            if (it < items)
                for (int r = it % SIG_SLICES; r < SIG_ROWS; r += SIG_SLICES) acc[u] = fma(tile[r][pj[u]], tile[r][pl[u]], acc[u]);
        }
    }
#pragma unroll
    for (int u = 0; u < SIG_PER_THREAD; u++) {
        const int it = threadIdx.x + 256 * u;
        if (it < items) part[it] = acc[u];
    }
    __syncthreads();
    for (int p = threadIdx.x; p < np; p += 256) {
        int j = 0;
        while ((j + 1) * (j + 2) / 2 <= p) j++;
        const int l = p - j * (j + 1) / 2;
        double s = part[p * SIG_SLICES];
        for (int k = 1; k < SIG_SLICES; k++) s += part[p * SIG_SLICES + k];
        double v = diag;
        if (j != l) {
            const double* xa = Cs + (size_t)(c0 + l) * d;
            const double* xb = Cs + (size_t)(c0 + j) * d;
            double r2 = 0;
            for (int t = 0; t < d; t++) { const double df = xa[t] - xb[t]; r2 = fma(df, df, r2); }
            v = cov_r2(kind, sf2, r2);
        }
        v -= s;
        Sig[(size_t)b * q * q + j * q + l] = v;
        Sig[(size_t)b * q * q + l * q + j] = v;
    }
}

// One CTA of four warps per batch.  Warp 0 factorises Sigma_b + jitter I (lane = row); warp w takes the samples s = w, w + 4, ...
// (lane j computes (mu + L z_s)_j, a butterfly finds the maximum and its lowest index) and the four warps' sums are added in warp
// order.  GRAD: per warp, lane k adds z_k,s to Lbar[j*][k]; the warps' Lbar are added in warp order, and warp 0 runs the reverse
// Cholesky Gbar = sym(L^-T Phi(L^T Lbar) L^-1) (Phi: lower triangle, halved diagonal).  The value path is the same code with
// and without GRAD.  A batch whose factorisation fails gets NaN for its value, mubar and Gbar.
// NEI (q-NEI): F_s,j = (mu_j + H[s][b q + j]) + (L z_s)_j and the improvement is max_j F_s,j - mb[s]; GRAD then overwrites the batch's
// columns of H with the winner indicator E[s][b q + j] = 1 / S (improving sample s, j = j*), else 0, rows S .. Sp - 1 included.
template <bool GRAD, bool NEI = false>
__global__ void __launch_bounds__(QW * 32) qei_batch_kernel(const double* __restrict__ Sig, const double* __restrict__ mu,
                                                            const double* __restrict__ Z, int S, int q, double ymax, double xi,
                                                            double jitter, double* __restrict__ val, double* __restrict__ mubar,
                                                            double* __restrict__ Gbar, double* __restrict__ H = nullptr, int ldh = 0,
                                                            const double* __restrict__ mb = nullptr, int Sp = 0) {
    __shared__ double L[QEI_MAX_Q][QEI_MAX_Q + 1];
    __shared__ double Lb[GRAD ? QW : 1][QEI_MAX_Q][QEI_MAX_Q + 1];
    __shared__ double wacc[QW];
    __shared__ int cnt[QW][QEI_MAX_Q];
    __shared__ int bad;
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double* A = Sig + (size_t)b * q * q;
    for (int idx = threadIdx.x; idx < q * q; idx += QW * 32) {
        const int r = idx / q, c = idx - r * q;
        L[r][c] = r == c ? A[idx] + jitter : A[idx];
    }
    if (GRAD)
        for (int idx = threadIdx.x; idx < QW * QEI_MAX_Q * (QEI_MAX_Q + 1); idx += QW * 32) (&Lb[0][0][0])[idx] = 0.0;
    __syncthreads();
    if (warp == 0) {
        int ok = 1;
        for (int k = 0; k < q && ok; k++) {
            double s = lane >= k && lane < q ? L[lane][k] : 0.0;
            if (lane >= k && lane < q)
                for (int i = 0; i < k; i++) s = fma(-L[lane][i], L[k][i], s);
            const double dk = __shfl_sync(0xffffffffu, s, k);
            ok = dk > 0.0;                                           // NaN fails too
            if (ok) {
                const double lkk = sqrt(dk);
                if (lane == k) L[k][k] = lkk;
                else if (lane > k && lane < q) L[lane][k] = s / lkk;
            }
            __syncwarp();
        }
        if (lane == 0) bad = !ok;
    }
    __syncthreads();
    if (bad) {
        if (threadIdx.x == 0) val[b] = NAN;
        if (GRAD) {
            for (int j = threadIdx.x; j < q; j += QW * 32) mubar[(size_t)b * q + j] = NAN;
            for (int j = threadIdx.x; j < q * q; j += QW * 32) Gbar[(size_t)b * q * q + j] = NAN;
        }
        return;
    }
    const bool live = lane < q;
    const double muj = live ? mu[(size_t)b * q + lane] : 0.0;
    double acc = 0.0;
    int c = 0;
    for (int s = warp; s < S; s += QW) {
        const double zk = live ? Z[(size_t)lane * S + s] : 0.0;
        double f = muj;
        if (NEI && live) f = muj + H[(size_t)s * ldh + (size_t)b * q + lane];
        for (int k = 0; k < q; k++) {
            const double zz = __shfl_sync(0xffffffffu, zk, k);
            if (k <= lane && live) f = fma(L[lane][k], zz, f);
        }
        double v = live ? f : -INFINITY;
        int ix = lane;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, v, off);
            const int oi = __shfl_xor_sync(0xffffffffu, ix, off);
            if (ov > v || (ov == v && oi < ix)) { v = ov; ix = oi; }
        }
        const double imp = NEI ? __dsub_rn(v, mb[s]) : __dsub_rn(__dsub_rn(v, ymax), xi);
        acc = __dadd_rn(acc, imp > 0.0 ? imp : 0.0);
        if (GRAD && NEI && live) H[(size_t)s * ldh + (size_t)b * q + lane] = imp > 0.0 && lane == ix ? 1.0 / S : 0.0;
        if (GRAD && imp > 0.0) {
            if (lane <= ix) Lb[warp][ix][lane] += zk;
            if (lane == ix) c++;
        }
    }
    if (GRAD && NEI && live)
        for (int s = S + warp; s < Sp; s += QW) H[(size_t)s * ldh + (size_t)b * q + lane] = 0.0;
    if (lane == 0) wacc[warp] = acc;
    if (GRAD && live) cnt[warp][lane] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = wacc[0];
        for (int w = 1; w < QW; w++) t = __dadd_rn(t, wacc[w]);
        val[b] = t / S;
    }
    if (!GRAD) return;
    if (threadIdx.x < q) {
        int n = 0;
        for (int w = 0; w < QW; w++) n += cnt[w][threadIdx.x];
        mubar[(size_t)b * q + threadIdx.x] = (double)n / S;
    }
    for (int idx = threadIdx.x; idx < q * q; idx += QW * 32) {        // Lbar into Lb[0]
        const int r = idx / q, k = idx - r * q;
        double t = Lb[0][r][k];
        for (int w = 1; w < QW; w++) t += Lb[w][r][k];
        Lb[0][r][k] = k <= r ? t / S : 0.0;
    }
    __syncthreads();
    if (warp != 0) return;
    double (*Lbar)[QEI_MAX_Q + 1] = Lb[0];
    double (*P)[QEI_MAX_Q + 1] = Lb[1];
    double (*X)[QEI_MAX_Q + 1] = Lb[2];
    double (*Sm)[QEI_MAX_Q + 1] = Lb[3];
    if (live) {                                                       // P = Phi(L^T Lbar), lane = column
        for (int k = 0; k < q; k++) {
            double s = 0.0;
            for (int i = max(k, lane); i < q; i++) s = fma(L[i][k], Lbar[i][lane], s);
            P[k][lane] = k > lane ? s : (k == lane ? 0.5 * s : 0.0);
        }
    }
    __syncwarp();
    if (live) {                                                       // X = L^-T P, lane = column
        for (int k = q - 1; k >= 0; k--) {
            double s = P[k][lane];
            for (int i = k + 1; i < q; i++) s = fma(-L[i][k], X[i][lane], s);
            X[k][lane] = s / L[k][k];
        }
    }
    __syncwarp();
    if (live) {                                                       // S = X L^-1, lane = row: L^T S[r]^T = X[r]^T
        for (int k = q - 1; k >= 0; k--) {
            double s = X[lane][k];
            for (int i = k + 1; i < q; i++) s = fma(-L[i][k], Sm[lane][i], s);
            Sm[lane][k] = s / L[k][k];
        }
    }
    __syncwarp();
    if (live)
        for (int l = 0; l < q; l++) Gbar[(size_t)b * q * q + lane * q + l] = 0.5 * (Sm[lane][l] + Sm[l][lane]);
}

// mu of the chunk's points over the model's training points, mu = sum_i a_i k_i (a = R^-1 Y), with a prior m0 + sum_i a_i k_i -
// m0 sum_i b_i k_i (b = R^-1 1).  One CTA: 32 points (lane = point) x 8 warps striding the training points i = w, w + 8, ...; the
// warps' partial sums are added in warp order, so a point's mu does not depend on the other points of the call.
__global__ void __launch_bounds__(256) qei_mean_kernel(double* __restrict__ mu, const double* __restrict__ Xt, int N,
                                                       const double* __restrict__ Cs, const double* __restrict__ raw, int Mc, int d,
                                                       int kind, double sf2, const double* __restrict__ a, const double* __restrict__ b,
                                                       int npb, const double* __restrict__ pmeans, const double* __restrict__ pbeta,
                                                       double ptheta, const double* __restrict__ plb, const double* __restrict__ pwidth) {
    __shared__ double sh[32 * 65];
    __shared__ double pa[8][32], pb[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, j0 = blockIdx.x * 32, j = j0 + lane, ldc = d | 1;
    for (int idx = threadIdx.x; idx < 32 * d; idx += 256) {
        const int c = idx / d, t = idx - c * d;
        sh[c * ldc + t] = j0 + c < Mc ? Cs[(size_t)(j0 + c) * d + t] : 0.0;
    }
    __syncthreads();
    const double* cj = sh + lane * ldc;
    double sa = 0.0, sb = 0.0;
    for (int i = warp; i < N && j < Mc; i += 8) {
        const double* xi = Xt + (size_t)i * d;
        double r2 = 0;
        for (int t = 0; t < d; t++) { const double df = xi[t] - cj[t]; r2 = fma(df, df, r2); }
        const double k = cov_r2(kind, sf2, r2);
        sa = fma(a[i], k, sa);
        if (npb > 0) sb = fma(b[i], k, sb);
    }
    pa[warp][lane] = sa;
    pb[warp][lane] = sb;
    __syncthreads();
    if (warp != 0 || j >= Mc) return;
    double A = pa[0][lane], Bs = pb[0][lane];
    for (int w = 1; w < 8; w++) { A += pa[w][lane]; Bs += pb[w][lane]; }
    if (npb > 0) {
        const double m0 = prior_mean(raw + (size_t)j * d, d, npb, pmeans, pbeta, ptheta, plb, pwidth);
        A = m0 + A - m0 * Bs;
    }
    mu[j] = A;
}

// y[i][j] = sum_l Zm[i][b q + l] Gbar_b[j - b q][l] for the rows i < gridDim.y and the chunk's points j (b = j / q); SUB2 (q-NEI's
// Tbar): y[i][j] -= 2 (that) in place
template <bool SUB2 = false>
__global__ void __launch_bounds__(256) qei_y_kernel(double* __restrict__ Y, const double* __restrict__ Zm, int ld,
                                                    const double* __restrict__ Gbar, int Mc, int q) {
    const int j = blockIdx.x * 256 + threadIdx.x, i = blockIdx.y;
    if (j >= Mc) return;
    const int b = j / q, jj = j - b * q;
    const double* z = Zm + (size_t)i * ld + (size_t)b * q;
    const double* g = Gbar + (size_t)b * q * q + (size_t)jj * q;
    double s = 0.0;
    for (int l = 0; l < q; l++) s = fma(z[l], g[l], s);
    if (SUB2) Y[(size_t)i * ld + j] = fma(-2.0, s, Y[(size_t)i * ld + j]);
    else Y[(size_t)i * ld + j] = s;
}

// One thread per point of the chunk, in place over its row of plane 0 (sum_i y_i dk_i): -2 (that) + 2 sum_{l != j} Gbar_jl d1 k(x_j, x_l)
// with d1 k(x_j, x_l) / dx_t = -(1 / theta_t) h(r) (s_j,t - s_l,t) in g's scaled coordinates Cs.  BASE (q-NEI): then
// + sum_{i < P} Cbar[i][j] d1 k(x_j, xb_i) over the baseline Cb, scaled like Cs
template <bool BASE = false>
__global__ void __launch_bounds__(256) qei_pair_kernel(double* __restrict__ G, const double* __restrict__ Cs, const double* __restrict__ Gbar,
                                                       int Mc, int q, int d, int kind, double sf2, const double* __restrict__ inv_theta,
                                                       const double* __restrict__ Cb = nullptr, const double* __restrict__ Cbar = nullptr,
                                                       int ldcb = 0, int P = 0) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= Mc) return;
    const int b = j / q, jj = j - b * q;
    double* g = G + (size_t)j * d;
    const double* xj = Cs + (size_t)j * d;
    for (int t = 0; t < d; t++) g[t] *= -2.0;
    for (int l = 0; l < q; l++) {
        if (l == jj) continue;
        const double* xl = Cs + (size_t)(b * q + l) * d;
        double r2 = 0;
        for (int t = 0; t < d; t++) { const double df = xj[t] - xl[t]; r2 = fma(df, df, r2); }
        double k;
        const double w = 2.0 * Gbar[(size_t)b * q * q + (size_t)jj * q + l] * cov_grad_h(kind, sf2, r2, &k);
        for (int t = 0; t < d; t++) g[t] = fma(-inv_theta[t] * w, xj[t] - xl[t], g[t]);
    }
    if (BASE)
        for (int i = 0; i < P; i++) {
            const double* xb = Cb + (size_t)i * d;
            double r2 = 0;
            for (int t = 0; t < d; t++) { const double df = xj[t] - xb[t]; r2 = fma(df, df, r2); }
            double k;
            const double w = Cbar[(size_t)i * ldcb + j] * cov_grad_h(kind, sf2, r2, &k);
            for (int t = 0; t < d; t++) g[t] = fma(-inv_theta[t] * w, xj[t] - xb[t], g[t]);
        }
}

// One thread per point: plane 0 += mubar dmu, dmu = plane 1 (+ plane 2 with a prior)
__global__ void __launch_bounds__(256) qei_epilogue_kernel(double* __restrict__ G, long M, int d, const double* __restrict__ mubar, int prior) {
    const long m = blockIdx.x * 256L + threadIdx.x;
    if (m >= M) return;
    const size_t plane = (size_t)M * d;
    double* g = G + (size_t)m * d;
    for (int t = 0; t < d; t++) {
        const double dmu = prior ? g[plane + t] + g[2 * plane + t] : g[plane + t];
        g[t] = fma(mubar[m], dmu, g[t]);
    }
}

// Enqueues everything on m->stream and leaves the values in w->dQei and, with wantGrad, the gradient [M][d] in w->dG.
int qei_device(ibo_model* m, const double* Xs, long B, int q, const double* Z, int S, double ymax, double xi, double jitter, bool wantGrad) {
    int rc;
    if ((rc = ensure_joint_attrs(m->device))) return rc;
    CandWork* w = cand_work(m);
    ibo_model* vm = m->var_model;
    ibo_model* g = vm ? vm : m;                          // the model Sigma comes from
    cudaStream_t st = m->stream;
    const int d = m->d;
    const bool prior = m->npb > 0;
    const long M = B * q;
    const long Bc = cand_chunk(g) / q;                   // whole batches per chunk
    const long Bcap = std::min(B, Bc), Mcap = round128(Bcap * q);
    if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * d))) return rc;
    if ((rc = grow(&w->dNormals, &w->normalsCap, (size_t)q * S))) return rc;
    if ((rc = grow(&w->dPost, &w->postCap, (size_t)M))) return rc;
    if ((rc = grow(&w->dAB, &w->abCap, (size_t)2 * m->Np))) return rc;
    if (vm && (rc = grow(&w->dScaledM, &w->scaledMCap, (size_t)Mcap * d))) return rc;
    if ((rc = grow(&w->dQei, &w->qeiCap, (size_t)B))) return rc;
    if ((rc = grow(&w->dSig, &w->sigCap, (size_t)Bcap * q * q))) return rc;
    if ((rc = grow(&w->dScaled, &w->scaledCap, (size_t)Mcap * d))) return rc;
    if ((rc = grow(&w->dKc, &w->kcCap, (size_t)g->Np * Mcap))) return rc;
    if ((rc = grow(&w->dV, &w->vCap, (size_t)g->Np * Mcap))) return rc;
    if (wantGrad) {
        if ((rc = grow(&w->dMubar, &w->mubarCap, (size_t)M))) return rc;
        if ((rc = grow(&w->dG, &w->gCap, (size_t)3 * M * d))) return rc;
        if ((rc = grow(&w->dGbar, &w->gbarCap, (size_t)Bcap * q * q))) return rc;
        if (prior && (rc = grow(&w->dKb, &w->kbCap, (size_t)M))) return rc;
    }
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * d, cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dNormals, Z, sizeof(double) * (size_t)q * S, cudaMemcpyHostToDevice, st));
    double* const mu = w->dPost;
    double* const dA = w->dAB;
    double* const dB = launch_ab(m, w->dAB, st);
    const size_t plane = (size_t)M * d;
    for (long b0 = 0; b0 < B; b0 += Bc) {
        const int nbt = (int)std::min(Bc, B - b0), Mc = nbt * q, Mcp = (int)round128(Mc);
        const long c0 = b0 * q;
        const double* raw = w->dRaw + (size_t)c0 * d;
        launch_scale_cands(w->dScaled, raw, g, Mc, Mcp, st);
        if (vm) launch_scale_cands(w->dScaledM, raw, m, Mc, Mcp, st);
        const double* Cm = vm ? w->dScaledM : w->dScaled;          // the chunk scaled like the model's training inputs
        qei_mean_kernel<<<(Mc + 31) / 32, 256, 0, st>>>(mu + c0, m->dXt, m->N, Cm, raw, Mc, d, m->kind, m->sf2, dA, dB, m->npb,
                                                        m->dPmeans, m->dPbeta, m->ptheta, m->dPlb, m->dPwidth);
        g_launches++;
        launch_cross_cov(w->dKc, g, w->dScaled, Mc, Mcp, st);
        launch_w_gemm_v(w->dV, g, w->dKc, Mcp, st);
        qei_sigma_kernel<<<nbt, 256, 0, st>>>(w->dSig, w->dV, Mcp, w->dScaled, g->N, q, d, g->kind, g->sf2, 1.0 + g->noise);
        g_launches += 2;
        if (!wantGrad) {
            qei_batch_kernel<false><<<nbt, QW * 32, 0, st>>>(w->dSig, mu + c0, w->dNormals, S, q, ymax, xi, jitter, w->dQei + b0, nullptr, nullptr);
            continue;
        }
        qei_batch_kernel<true><<<nbt, QW * 32, 0, st>>>(w->dSig, mu + c0, w->dNormals, S, q, ymax, xi, jitter, w->dQei + b0, w->dMubar + c0, w->dGbar);
        launch_w_gemm_z(w->dKc, g, w->dV, Mcp, st);
        qei_y_kernel<<<dim3((Mc + 255) / 256, g->N), 256, 0, st>>>(w->dV, w->dKc, Mcp, w->dGbar, Mc, q);
        g_launches += 2;
        double* G = w->dG + (size_t)c0 * d;
        launch_grad_sums(m, w->dScaled, w->dScaledM, Mc, w->dV, Mcp, dA, dB, G, plane, prior ? w->dKb + c0 : nullptr, st);
        qei_pair_kernel<<<(Mc + 255) / 256, 256, 0, st>>>(G, w->dScaled, w->dGbar, Mc, q, d, g->kind, g->sf2, g->dInvTheta);
        g_launches++;
    }
    if (wantGrad) {
        if (prior) launch_grad_prior(m, w->dRaw, M, w->dKb, w->dG, st);
        qei_epilogue_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(w->dG, M, d, w->dMubar, prior ? 1 : 0);
        g_launches++;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

// q-NEI: points per chunk, the largest multiple of 128 whose K* and V (Np each), C and T (Pp each) and H (Sp) fit in 2^26 doubles
long qnei_chunk(const ibo_model* g, long P, int S) {
    return std::max(128L, (long)((1L << 26) / (2L * g->Np + 2 * round128(P) + round128(S))) / 128 * 128);
}

// Enqueues everything on m->stream and leaves the values in w->dQei, the incumbent draws m_s at the end of w->dBase and, with
// wantGrad, the gradient [M][d] in w->dG.  The baseline's factorisation is checked on the host: IBO_E_NOTSPD with *info = its pivot.
int qnei_device(ibo_model* m, const double* Xs, long B, int q, const double* Xbase, long P, const double* Z, int S, double jitter,
                bool wantGrad, int* info) {
    int rc;
    if ((rc = ensure_joint_attrs(m->device))) return rc;
    CandWork* w = cand_work(m);
    ibo_model* vm = m->var_model;
    ibo_model* g = vm ? vm : m;                          // the model Sigma comes from
    cudaStream_t st = m->stream;
    const int d = m->d, Np = g->Np, Pi = (int)P, Pp = (int)round128(P), Sp = (int)round128(S), nbP = Pp / 128;
    const bool prior = m->npb > 0;
    const long M = B * q;
    const long Bc = qnei_chunk(g, P, S) / q;             // whole batches per chunk
    const long Bcap = std::min(B, Bc), Mcap = round128(Bcap * q);
    if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * d))) return rc;
    if ((rc = grow(&w->dNormals, &w->normalsCap, (size_t)q * S))) return rc;
    if ((rc = grow(&w->dPost, &w->postCap, (size_t)M))) return rc;
    if ((rc = grow(&w->dAB, &w->abCap, (size_t)2 * m->Np))) return rc;
    if (vm && (rc = grow(&w->dScaledM, &w->scaledMCap, (size_t)std::max<long>(Mcap, Pp) * d))) return rc;
    if ((rc = grow(&w->dQei, &w->qeiCap, (size_t)B))) return rc;
    if ((rc = grow(&w->dSig, &w->sigCap, (size_t)Bcap * q * q))) return rc;
    if ((rc = grow(&w->dScaled, &w->scaledCap, (size_t)Mcap * d))) return rc;
    if ((rc = grow(&w->dKc, &w->kcCap, (size_t)Np * std::max<long>(Mcap, Pp)))) return rc;
    if ((rc = grow(&w->dV, &w->vCap, (size_t)(Np + Pp) * Mcap))) return rc;
    if ((rc = grow(&w->dBase, &w->baseCap, (size_t)P * d + (size_t)Pp * d + Pp + Sp))) return rc;
    if ((rc = grow(&w->dVb, &w->vbCap, (size_t)Np * Pp))) return rc;
    if ((rc = grow(&w->dZb, &w->zbCap, (size_t)Pp * Sp))) return rc;
    if ((rc = grow(&w->dFb, &w->fbCap, (size_t)Pp * Sp))) return rc;
    if ((rc = grow(&w->dCT, &w->ctCap, (size_t)Pp * Mcap))) return rc;
    if ((rc = grow(&w->dH, &w->hCap, (size_t)Sp * Mcap))) return rc;
    if ((rc = grow(&w->dArg, &w->argCap, (size_t)S))) return rc;
    if (wantGrad) {
        if ((rc = grow(&w->dZbase, &w->zbaseCap, (size_t)Np * Pp))) return rc;
        if ((rc = grow(&w->dMubar, &w->mubarCap, (size_t)M))) return rc;
        if ((rc = grow(&w->dG, &w->gCap, (size_t)3 * M * d))) return rc;
        if ((rc = grow(&w->dGbar, &w->gbarCap, (size_t)Bcap * q * q))) return rc;
        if (prior && (rc = grow(&w->dKb, &w->kbCap, (size_t)M))) return rc;
    }
    if ((rc = chol_setup(m, P, true))) return rc;
    Factor& c = w->chol;
    double* const baseRaw = w->dBase;
    double* const baseS = baseRaw + (size_t)P * d;
    double* const mub = baseS + (size_t)Pp * d;
    double* const mmax = mub + Pp;
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * d, cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(baseRaw, Xbase, sizeof(double) * (size_t)P * d, cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dNormals, Z + (size_t)P * S, sizeof(double) * (size_t)q * S, cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemsetAsync(w->dZb, 0, sizeof(double) * (size_t)Pp * Sp, st));
    IBO_CUDA_TRY(cudaMemcpy2DAsync(w->dZb, sizeof(double) * Sp, Z, sizeof(double) * S, sizeof(double) * S, P, cudaMemcpyHostToDevice, st));
    double* const mu = w->dPost;
    double* const dA = w->dAB;
    double* const dB = launch_ab(m, w->dAB, st);
    // once per call: the baseline's mean, V_b, Sigma_bb = L_bb L_bb^T, W_bb = inv(L_bb), F_b = mu_b 1^T + L_bb Z_b and m_s
    launch_scale_cands(baseS, baseRaw, g, P, Pp, st);
    if (vm) launch_scale_cands(w->dScaledM, baseRaw, m, P, Pp, st);
    qei_mean_kernel<<<(Pi + 31) / 32, 256, 0, st>>>(mub, m->dXt, m->N, vm ? w->dScaledM : baseS, baseRaw, Pi, d, m->kind, m->sf2, dA, dB,
                                                    m->npb, m->dPmeans, m->dPbeta, m->ptheta, m->dPlb, m->dPwidth);
    g_launches++;
    launch_cross_cov(w->dKc, g, baseS, Pi, Pp, st);
    launch_w_gemm_v(w->dVb, g, w->dKc, Pp, st);
    if (wantGrad) launch_w_gemm_z(w->dZbase, g, w->dVb, Pp, st);                                 // R_g^-1 K(X_g, X_b)
    launch_joint_sigma(c, baseS, w->dVb, g, g->sf2, jitter, st);
    if ((rc = launch_factorize(*m, c, false, false, true))) return rc;
    int hinfo = 0;
    IBO_CUDA_TRY(cudaMemcpyAsync(&hinfo, c.dInfo, sizeof(int), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    if (hinfo != 0) {
        if (info) *info = hinfo;
        set_error("baseline covariance + jitter I is not positive definite (pivot " + std::to_string(hinfo) + ")");
        return IBO_E_NOTSPD;
    }
    launch_clear_diag_upper(c, st);
    launch_trimm(w->dFb, Sp, c.dA, Pp, w->dZb, Sp, nbP, Sp, mub, Pi, st);
    launch_sample_max(w->dFb, Sp, Pi, S, reinterpret_cast<long long*>(w->dArg), mmax, st);
    const size_t plane = (size_t)M * d;
    for (long b0 = 0; b0 < B; b0 += Bc) {
        const int nbt = (int)std::min(Bc, B - b0), Mc = nbt * q, Mcp = (int)round128(Mc);
        const long c0 = b0 * q;
        const double* raw = w->dRaw + (size_t)c0 * d;
        double* const T = w->dV + (size_t)Np * Mcp;               // T = W_bb C below V_q, then Cbar
        launch_scale_cands(w->dScaled, raw, g, Mc, Mcp, st);
        if (vm) launch_scale_cands(w->dScaledM, raw, m, Mc, Mcp, st);
        const double* Cm = vm ? w->dScaledM : w->dScaled;
        qei_mean_kernel<<<(Mc + 31) / 32, 256, 0, st>>>(mu + c0, m->dXt, m->N, Cm, raw, Mc, d, m->kind, m->sf2, dA, dB, m->npb,
                                                        m->dPmeans, m->dPbeta, m->ptheta, m->dPlb, m->dPwidth);
        g_launches++;
        launch_cross_cov(w->dKc, g, w->dScaled, Mc, Mcp, st);
        launch_w_gemm_v(w->dV, g, w->dKc, Mcp, st);
        launch_cross_cov_pts(w->dCT, baseS, Pi, Pp, g, w->dScaled, Mc, Mcp, st);                  // C = K(X_b, X_q) - V_b^T V_q
        launch_gemm(w->dCT, Mcp, w->dVb, Pp, true, w->dV, Mcp, Pp, Mcp, Np, -1.0, true, st);
        launch_trimm(T, Mcp, c.dW, Pp, w->dCT, Mcp, nbP, Mcp, nullptr, 0, st);                    // T = W_bb C
        launch_gemm(w->dH, Mcp, w->dZb, Sp, true, T, Mcp, Sp, Mcp, Pp, 1.0, false, st);           // H = Z_b^T T
        // Schur complements Sigma_qq - T^T T: the rows of [V_q; T] (V_q's padding rows are zero)
        qei_sigma_kernel<<<nbt, 256, 0, st>>>(w->dSig, w->dV, Mcp, w->dScaled, Np + Pi, q, d, g->kind, g->sf2, g->sf2);
        g_launches++;
        if (!wantGrad) {
            qei_batch_kernel<false, true><<<nbt, QW * 32, 0, st>>>(w->dSig, mu + c0, w->dNormals, S, q, 0.0, 0.0, jitter, w->dQei + b0,
                                                                  nullptr, nullptr, w->dH, Mcp, mmax, Sp);
            g_launches++;
            continue;
        }
        qei_batch_kernel<true, true><<<nbt, QW * 32, 0, st>>>(w->dSig, mu + c0, w->dNormals, S, q, 0.0, 0.0, jitter, w->dQei + b0,
                                                             w->dMubar + c0, w->dGbar, w->dH, Mcp, mmax, Sp);
        g_launches++;
        launch_gemm(w->dCT, Mcp, w->dZb, Sp, false, w->dH, Mcp, Pp, Mcp, Sp, 1.0, false, st);     // Tbar = Z_b E - 2 T Gbar
        qei_y_kernel<true><<<dim3((Mc + 255) / 256, Pi), 256, 0, st>>>(w->dCT, T, Mcp, w->dGbar, Mc, q);
        g_launches++;
        launch_trimm_t(T, Mcp, c.dW, Pp, w->dCT, Mcp, nbP, Mcp, st);                              // Cbar = W_bb^T Tbar
        launch_w_gemm_z(w->dKc, g, w->dV, Mcp, st);                                               // y = Z_q Gbar + Z_b Cbar / 2
        qei_y_kernel<<<dim3((Mc + 255) / 256, g->N), 256, 0, st>>>(w->dV, w->dKc, Mcp, w->dGbar, Mc, q);
        g_launches++;
        launch_gemm(w->dV, Mcp, w->dZbase, Pp, false, T, Mcp, Np, Mcp, Pp, 0.5, true, st);
        double* G = w->dG + (size_t)c0 * d;
        launch_grad_sums(m, w->dScaled, w->dScaledM, Mc, w->dV, Mcp, dA, dB, G, plane, prior ? w->dKb + c0 : nullptr, st);
        qei_pair_kernel<true><<<(Mc + 255) / 256, 256, 0, st>>>(G, w->dScaled, w->dGbar, Mc, q, d, g->kind, g->sf2, g->dInvTheta, baseS, T,
                                                                Mcp, Pi);
        g_launches++;
    }
    if (wantGrad) {
        if (prior) launch_grad_prior(m, w->dRaw, M, w->dKb, w->dG, st);
        qei_epilogue_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(w->dG, M, d, w->dMubar, prior ? 1 : 0);
        g_launches++;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

}  // namespace

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_qei(ibo_model* m, const double* Xs, long B, int q, const double* Z, int S, double ymax, double xi, double jitter,
                       double* values, double* dvalues, int* nbad) {
    if (nbad) *nbad = 0;
    int rc = check_cands(m, Xs, B, Z && values && q >= 1 && q <= QEI_MAX_Q && S >= 1 && S <= 65536 && jitter >= 0.0);   // NaN jitter fails
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    rc = qei_device(m, Xs, B, q, Z, S, ymax, xi, jitter, dvalues != nullptr);
    if (rc) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    IBO_CUDA_TRY(cudaMemcpyAsync(values, w->dQei, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
    if (dvalues) IBO_CUDA_TRY(cudaMemcpyAsync(dvalues, w->dG, sizeof(double) * (size_t)B * q * m->d, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    if (nbad)
        for (long b = 0; b < B; b++) *nbad += std::isnan(values[b]) ? 1 : 0;
    return IBO_OK;
}

extern "C" int ibo_qnei(ibo_model* m, const double* Xs, long B, int q, const double* Xbase, long P, const double* Z, int S, double jitter,
                        double* values, double* dvalues, double* incumbent, int* nbad, int* info) {
    if (nbad) *nbad = 0;
    if (info) *info = 0;
    bool ok = Xbase && Z && values && q >= 1 && q <= QEI_MAX_Q && P >= 1 && P <= 8192 && S >= 1 && S <= 8192 && jitter >= 0.0;   // NaN jitter fails
    if (ok && m) {
        const ibo_model* g = m->var_model ? m->var_model : m;
        ok = g->sf2 <= 1.0 + g->noise;                   // the latent covariance is PSD only then
    }
    int rc = check_cands(m, Xs, B, ok);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    rc = qnei_device(m, Xs, B, q, Xbase, P, Z, S, jitter, dvalues != nullptr, info);
    if (rc) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    IBO_CUDA_TRY(cudaMemcpyAsync(values, w->dQei, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
    if (dvalues) IBO_CUDA_TRY(cudaMemcpyAsync(dvalues, w->dG, sizeof(double) * (size_t)B * q * m->d, cudaMemcpyDeviceToHost, st));
    if (incumbent) {
        const double* mmax = w->dBase + (size_t)P * m->d + (size_t)round128(P) * m->d + round128(P);
        IBO_CUDA_TRY(cudaMemcpyAsync(incumbent, mmax, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    }
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    if (nbad)
        for (long b = 0; b < B; b++) *nbad += std::isnan(values[b]) ? 1 : 0;
    return IBO_OK;
}
