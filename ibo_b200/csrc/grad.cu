// Gradients of the posterior and of the acquisition with respect to the candidate.
//
//   d mu / dx_t   = d m0 / dx_t (1 - k^T b) + sum_i (a_i - m0 b_i) dk_i / dx_t       a = W^T W Y, b = W^T W 1 (of the model)
//   d s2 / dx_t   = -2 sum_i z_i dk_i / dx_t,  z = W_g^T (W_g k)                      (g: the variance model, else the model)
//   dk_i / dx_t   = -(1 / theta_t) h(r_i) (s_t - s_i,t)                               (cov_grad_h)
//
// Per chunk of candidates: scale the candidates, K* = R(X_g, X*), V = W_g K* and Z = W_g^T V on the FP64 tensor pipe (joint.cu),
// then one reduction kernel that recomputes r and h(r) per (training point, candidate).  The values (scores, mu, s2) come from the
// scoring path's FP64 kernels, so they are ibo_score_batch's / ibo_posterior_batch's with IBO_FLAG_FP64 bit for bit; one epilogue
// adds the prior's gradient, zeroes the gradient of s2 where the scoring path clips s2, and applies the acquisition's chain rule.
// Every sum runs in a fixed order without atomics and the GEMM columns are independent, so a candidate's gradients do not
// depend on which other candidates share its call.
#include "model.cuh"
#include "scoremath.cuh"
#include <algorithm>
#include <cmath>

namespace ibo {

namespace {

constexpr int RC = 32;    // candidates per CTA (lane = candidate)
constexpr int RW = 8;     // warps per CTA: warp w takes the training points i = w, w + 8, ...
constexpr int RDS = 16;   // dimensions per CTA (grid.y slices d)

// G[q][j][t] = sum_i w_q,i dk_i(x*_j) / dx_t for the weights w_0 = Z[:, j], w_1 = a, w_2 = b (those the template enables), over the
// N training points of Xt; kb[j] = sum_i b_i k_i (slice 0).  One CTA: 32 candidates x 16 dimensions; the eight warps' partial
// sums are combined in warp order.
template <bool DZ, bool DA, bool DB>
__global__ void __launch_bounds__(256) grad_reduce_kernel(const double* __restrict__ Xt, int N, const double* __restrict__ Cs, int Mc,
                                                          int d, int kind, double sf2, const double* __restrict__ inv_theta,
                                                          const double* __restrict__ Z, int ldz, const double* __restrict__ a,
                                                          const double* __restrict__ b, double* __restrict__ G, size_t plane,
                                                          double* __restrict__ kb) {
    __shared__ double sh[RW * RDS * RC];               // candidate coordinates, then the partial sums of one quantity
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j0 = blockIdx.x * RC, j = j0 + lane, t0 = blockIdx.y * RDS, dn = min(RDS, d - t0);
    const int ldc = d | 1;                             // odd stride: lanes read distinct banks
    for (int idx = threadIdx.x; idx < RC * d; idx += 256) {
        const int c = idx / d, t = idx - c * d;
        sh[c * ldc + t] = j0 + c < Mc ? Cs[(size_t)(j0 + c) * d + t] : 0.0;
    }
    __syncthreads();
    const double* cj = sh + lane * ldc;
    double cs[RDS], gz[RDS], ga[RDS], gb[RDS];
#pragma unroll
    for (int u = 0; u < RDS; u++) { cs[u] = u < dn ? cj[t0 + u] : 0.0; gz[u] = ga[u] = gb[u] = 0.0; }
    double skb = 0.0;
    const bool live = j < Mc;
    for (int i = warp; i < N && live; i += RW) {
        const double* xi = Xt + (size_t)i * d;
        double r2 = 0;
        for (int t = 0; t < d; t++) { const double df = xi[t] - cj[t]; r2 = fma(df, df, r2); }
        double k;
        const double h = cov_grad_h(kind, sf2, r2, &k);
        const double hz = DZ ? h * Z[(size_t)i * ldz + j] : 0.0;
        const double ha = DA ? h * a[i] : 0.0;
        const double hb = DB ? h * b[i] : 0.0;
        if (DB) skb = fma(b[i], k, skb);
#pragma unroll
        for (int u = 0; u < RDS; u++)
            if (u < dn) {
                const double df = cs[u] - xi[t0 + u];
                if (DZ) gz[u] = fma(hz, df, gz[u]);
                if (DA) ga[u] = fma(ha, df, ga[u]);
                if (DB) gb[u] = fma(hb, df, gb[u]);
            }
    }
    // combine the warps in a fixed order; -1 / theta_t turns sum_i w_i h_i (s_t - s_i,t) into sum_i w_i dk_i / dx_t
    auto combine = [&](double (&acc)[RDS], double* out) {
        __syncthreads();
#pragma unroll
        for (int u = 0; u < RDS; u++) sh[(warp * RDS + u) * RC + lane] = acc[u];
        __syncthreads();
        for (int o = threadIdx.x; o < RDS * RC; o += 256) {
            const int u = o / RC, l = o - u * RC;
            double s = 0;
            for (int w = 0; w < RW; w++) s += sh[(w * RDS + u) * RC + l];
            if (u < dn && j0 + l < Mc) out[(size_t)(j0 + l) * d + t0 + u] = -inv_theta[t0 + u] * s;
        }
    };
    if (DZ) combine(gz, G);
    if (DA) combine(ga, G + plane);
    if (DB) {
        combine(gb, G + 2 * plane);
        if (blockIdx.y == 0) {
            __syncthreads();
            sh[warp * RC + lane] = skb;
            __syncthreads();
            if (warp == 0 && live) {
                double s = 0;
                for (int w = 0; w < RW; w++) s += sh[w * RC + lane];
                kb[j] = s;
            }
        }
    }
}

struct GradEpi {
    long M;
    int d, acq, mode_py, npb;
    double ymax, parm, ptheta;
    const double *vals, *cand, *kb, *pmeans, *pbeta, *plb, *pwidth;
    double* G;              // [3][M][d]: sums with z, a, b in; ds2, dmu, dscore out
};

// One thread per candidate: the prior's share of dmu, d m0 / dx_t (1 - k^T b) - m0 sum_i b_i dk_i / dx_t, in place over the b plane
// (m0 = sum_b beta_b exp(-ptheta |q_b|^2), q_b,t = (x_t - lb_t) / width_t - mean_b,t)
__global__ void __launch_bounds__(256) grad_prior_kernel(GradEpi P) {
    const long m = blockIdx.x * 256L + threadIdx.x;
    if (m >= P.M) return;
    const double* x = P.cand + (size_t)m * P.d;
    double* gb = P.G + 2 * (size_t)P.M * P.d + (size_t)m * P.d;
    const double m0 = prior_mean(x, P.d, P.npb, P.pmeans, P.pbeta, P.ptheta, P.plb, P.pwidth), f = -2.0 * P.ptheta * (1.0 - P.kb[m]);
    for (int t = 0; t < P.d; t++) gb[t] *= -m0;
    for (int b = 0; b < P.npb; b++) {
        const double* pm = P.pmeans + (size_t)b * P.d;
        double dd = 0;
        for (int t = 0; t < P.d; t++) {
            const double q = (x[t] - P.plb[t]) / P.pwidth[t] - pm[t];
            dd += q * q;
        }
        const double e = f * P.pbeta[b] * exp(-P.ptheta * dd);
        for (int t = 0; t < P.d; t++) gb[t] += e * ((x[t] - P.plb[t]) / P.pwidth[t] - pm[t]) / P.pwidth[t];
    }
}

// One thread per candidate: the clipping rule of the scoring path (ds2 = 0 where it clipped s2 to the mode's floor or to 10) and
// the acquisition's chain rule through (mu, s = sqrt(s2)).
__global__ void __launch_bounds__(256) grad_epilogue_kernel(GradEpi P) {
    const long m = blockIdx.x * 256L + threadIdx.x;
    if (m >= P.M) return;
    const double mu = P.vals[P.M + m], s2 = P.vals[2 * P.M + m];
    const double floor_ = P.mode_py ? 10e-8 : 1e-8;
    const bool clipped = s2 <= floor_ || s2 >= 10.0;
    double amu = 0.0, as = 0.0;
    if (P.acq >= 0) acq_partials(P.acq, P.mode_py, mu, s2, P.ymax, P.parm, &amu, &as);
    const double ds_ds2 = 0.5 / sqrt(s2);
    const size_t plane = (size_t)P.M * P.d;
    double* gz = P.G + (size_t)m * P.d;
    for (int t = 0; t < P.d; t++) {
        const double dmu = P.npb > 0 ? gz[plane + t] + gz[2 * plane + t] : gz[plane + t];
        const double ds2 = clipped ? 0.0 : -2.0 * gz[t];
        gz[t] = ds2;
        gz[plane + t] = dmu;
        gz[2 * plane + t] = amu * dmu + as * (ds2 * ds_ds2);
    }
}

template <bool DZ, bool DA, bool DB>
void launch_reduce(const ibo_model* src, const double* Cs, int Mc, const double* Z, int ldz, const double* a, const double* b,
                   double* G, size_t plane, double* kb, cudaStream_t st) {
    const dim3 grid((Mc + RC - 1) / RC, (src->d + RDS - 1) / RDS);
    grad_reduce_kernel<DZ, DA, DB><<<grid, 256, 0, st>>>(src->dXt, src->N, Cs, Mc, src->d, src->kind, src->sf2, src->dInvTheta, Z, ldz,
                                                          a, b, G, plane, kb);
    g_launches++;
}

}  // namespace

long cand_chunk(const ibo_model* g) { return std::max(128L, (long)((512L << 20) / (2L * 8 * g->Np)) / 128 * 128); }

double* launch_ab(const ibo_model* m, double* ab, cudaStream_t st) {
    launch_tri_matvec_t(m->dW, m->dBetaY, ab, m->N, m->Np, st);
    if (m->npb == 0) return nullptr;
    launch_tri_matvec_t(m->dW, m->dBeta1, ab + m->Np, m->N, m->Np, st);
    return ab + m->Np;
}

// with a variance model the weights of s2 and those of mu run over different training points: two launches
void launch_grad_sums(const ibo_model* m, const double* Cs, const double* Cm, int Mc, const double* Zw, int ldz, const double* a,
                      const double* b, double* G, size_t plane, double* kb, cudaStream_t st) {
    if (const ibo_model* vm = m->var_model) {
        launch_reduce<true, false, false>(vm, Cs, Mc, Zw, ldz, nullptr, nullptr, G, plane, nullptr, st);
        if (b) launch_reduce<false, true, true>(m, Cm, Mc, nullptr, 0, a, b, G, plane, kb, st);
        else launch_reduce<false, true, false>(m, Cm, Mc, nullptr, 0, a, nullptr, G, plane, nullptr, st);
    } else if (b) {
        launch_reduce<true, true, true>(m, Cs, Mc, Zw, ldz, a, b, G, plane, kb, st);
    } else {
        launch_reduce<true, true, false>(m, Cs, Mc, Zw, ldz, a, nullptr, G, plane, nullptr, st);
    }
}

void launch_grad_prior(const ibo_model* m, const double* cand, long M, const double* kb, double* G, cudaStream_t st) {
    GradEpi P{};
    P.M = M; P.d = m->d; P.npb = m->npb; P.ptheta = m->ptheta;
    P.cand = cand; P.kb = kb;
    P.pmeans = m->dPmeans; P.pbeta = m->dPbeta; P.plb = m->dPlb; P.pwidth = m->dPwidth;
    P.G = G;
    grad_prior_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(P);
    g_launches++;
}

// Enqueues everything on m->stream and leaves [score | mu | s2] in w->dPost and ds2, dmu, dscore ([M][d] each) in w->dG.
int grad_device(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags, bool wantGrad) {
    int rc;
    if ((rc = ensure_joint_attrs(m->device))) return rc;
    CandWork* w = cand_work(m);
    ibo_model* vm = m->var_model;
    ibo_model* g = vm ? vm : m;                          // the model sigma^2 comes from
    cudaStream_t st = m->stream;
    const int d = m->d;
    const bool prior = m->npb > 0;
    const long chunk = cand_chunk(g), Mcap = round128(std::min(M, chunk));
    if ((rc = grow(&w->dRaw, &w->rawCap, (size_t)M * d))) return rc;
    if ((rc = grow(&w->dPost, &w->postCap, (size_t)3 * M + 2))) return rc;
    if (wantGrad) {
        if ((rc = grow(&w->dG, &w->gCap, (size_t)3 * M * d))) return rc;
        if (prior && (rc = grow(&w->dKb, &w->kbCap, (size_t)M))) return rc;
        if ((rc = grow(&w->dScaled, &w->scaledCap, (size_t)Mcap * d))) return rc;
        if (vm && (rc = grow(&w->dScaledM, &w->scaledMCap, (size_t)Mcap * d))) return rc;
        if ((rc = grow(&w->dKc, &w->kcCap, (size_t)g->Np * Mcap))) return rc;
        if ((rc = grow(&w->dV, &w->vCap, (size_t)g->Np * Mcap))) return rc;
        if ((rc = grow(&w->dAB, &w->abCap, (size_t)2 * m->Np))) return rc;
    }
    IBO_CUDA_TRY(cudaMemcpyAsync(w->dRaw, Xs, sizeof(double) * (size_t)M * d, cudaMemcpyHostToDevice, st));
    if ((rc = posterior_score_device(m, w->dRaw, M, acq, ymax, parm, IBO_FLAG_FP64 | flags, w->dPost))) return rc;
    if (!wantGrad) return IBO_OK;
    double* const dA = w->dAB;
    double* const dB = launch_ab(m, w->dAB, st);
    const size_t plane = (size_t)M * d;
    for (long c0 = 0; c0 < M; c0 += chunk) {
        const int Mc = (int)std::min(chunk, M - c0), Mcp = (int)round128(Mc);
        const double* raw = w->dRaw + (size_t)c0 * d;
        launch_scale_cands(w->dScaled, raw, g, Mc, Mcp, st);
        launch_cross_cov(w->dKc, g, w->dScaled, Mc, Mcp, st);
        launch_w_gemm_v(w->dV, g, w->dKc, Mcp, st);
        launch_w_gemm_z(w->dKc, g, w->dV, Mcp, st);
        if (vm) launch_scale_cands(w->dScaledM, raw, m, Mc, Mcp, st);
        launch_grad_sums(m, w->dScaled, w->dScaledM, Mc, w->dKc, Mcp, dA, dB, w->dG + (size_t)c0 * d, plane, prior ? w->dKb + c0 : nullptr, st);
    }
    GradEpi P{};
    P.M = M; P.d = d; P.acq = acq; P.mode_py = (flags & IBO_FLAG_MODE_PY) ? 1 : 0; P.npb = m->npb;
    P.ymax = ymax; P.parm = parm;
    P.vals = w->dPost;
    P.G = w->dG;
    if (prior) launch_grad_prior(m, w->dRaw, M, w->dKb, w->dG, st);
    grad_epilogue_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(P);
    g_launches++;
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

namespace {

int copy_out(double* dst, const double* src, size_t n, cudaStream_t st) {
    if (dst) IBO_CUDA_TRY(cudaMemcpyAsync(dst, src, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    return IBO_OK;
}

}  // namespace

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_posterior_grad(ibo_model* m, const double* Xs, long M, int flags, double* mu, double* s2, double* dmu, double* ds2) {
    int rc = check_cands(m, Xs, M, (flags & ~IBO_FLAG_MODE_PY) == 0);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if ((rc = grad_device(m, Xs, M, -1, 0.0, 0.0, flags, dmu || ds2))) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    const size_t plane = (size_t)M * m->d;
    if ((rc = copy_out(mu, w->dPost + M, M, st)) || (rc = copy_out(s2, w->dPost + 2 * M, M, st)) ||
        (rc = copy_out(ds2, w->dG, plane, st)) || (rc = copy_out(dmu, w->dG + plane, plane, st)))
        return rc;
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

extern "C" int ibo_score_grad(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags,
                              double* scores, double* dscores) {
    int rc = check_cands(m, Xs, M, (flags & ~IBO_FLAG_MODE_PY) == 0 && acq >= 0 && acq <= 2);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if ((rc = grad_device(m, Xs, M, acq, ymax, parm, flags, dscores != nullptr))) return rc;
    CandWork* w = m->cand;
    cudaStream_t st = m->stream;
    if ((rc = copy_out(scores, w->dPost, M, st)) || (rc = copy_out(dscores, w->dG + 2 * (size_t)M * m->d, (size_t)M * m->d, st))) return rc;
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}
