// Fused scoring kernel for small models (N <= 128: one 128-row block) -- the reference's own operating point
// (demo.py, the unit tests and interactive galleries work with tens of observations, BASELINE.json config #1).
//
// Replaces, in one launch, GaussianProcess.posterior + EI/PI/UCB.negf per candidate (ego/gaussianprocess/__init__.py:169-228,
// ego/acquisition/__init__.py:60-164) / GP_Maximizer::posterior + negei/negpi/negucb (cpp/optimizeGP.cpp:57-236).
//
// For such models the general path (K1 -> K2 -> K3, score.cu) is pure latency: three dependent launches, an H2D DMA and
// a slab round trip for ~N^2/2 = a few thousand FMAs per candidate.  Here one CTA keeps W = inv(L) transposed in shared
// memory and walks tiles of 8 candidates: k* by direct differences (no expansion, no cancellation), v = W k* with one
// thread per training row (ascending-k FMA chains, 8 candidates in flight per thread), the three row reductions in a
// fixed order, then the epilogue.  For a DIRECT batch the candidates are read straight from mapped pinned host memory
// and the values are written straight back to it: one launch and one stream synchronisation per batch.
// A candidate's value is a function of (model, x) only (fixed summation orders), so DIRECT trajectories stay reproducible.
#include "model.cuh"
#include "scoremath.cuh"
#include <atomic>
#include <chrono>
#include <cstring>
#include <mutex>

namespace ibo {
namespace {

constexpr int TC = 8;        // candidates per tile
constexpr int WS = 129;      // row stride of W in shared memory: odd, so that thread r walking row r is conflict free

struct TinySide {            // one factor: the model itself, or the variance model of PrefGaussianProcess.addObservationPoint
    const double *W, *Xt, *center;
    int N;
};

struct TinyParams {
    TinySide side[2];        // [1].N == 0 when there is no variance model
    const double *betaY, *beta1, *invTheta, *cand;
    const double *pmeans, *pbeta, *plb, *pwidth;
    double *score, *mu, *s2;
    double* blkBest; long long* blkIdx;
    long M;
    int d, acq, mode_py, npb, want_argmax;
    double sf2, noise, ymax, parm, ptheta;
};

// Batch server (SERVER = true): for the length of one DIRECT query the kernel stays resident -- a handful of CTAs with the factors
// staged in shared memory once -- and takes its batches from a mailbox in mapped pinned host memory: the host writes the candidates
// and publishes (batch number, size) in one word, every CTA that owns a tile scores it, writes the values into the mailbox and
// releases its own `done` word.  A batch then costs three dependent PCIe round trips (control word, candidates, values) instead of
// a kernel launch, a re-staging of W and a stream synchronisation.  All mailbox traffic uses system-scope loads / stores (a resident kernel must not find
// stale host data in L2); an idle server gives up after two seconds so that nothing spins on the GPU if the host goes away.
struct TinyMailbox {
    long long ctrl;      // host -> device: (batch number << 24) | candidates in the batch; -1 = quit.  One word, one PCIe read per poll.
    long long pad[15];
    long long done[16];  // device -> host: done[c] = number of the last batch CTA c finished (only CTAs that own a tile report)
    double data[1];      // candidates [M][d], then the values [M]
};
constexpr size_t MAILBOX_DOUBLES = (1u << 17) - 32;     // one pinned staging buffer of the pool (1 MiB)
constexpr int SERVER_CTAS = 16;

__device__ __forceinline__ long long ld_relaxed_sys(const long long* p) {
    long long v; asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ double ld_relaxed_sys(const double* p) {
    double v; asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_release_sys(long long* p, long long v) {
    asm volatile("st.release.sys.global.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
}

__device__ __forceinline__ void cp_async8(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src));
}

template <int KC, bool SERVER>
__global__ void __launch_bounds__(128) tiny_fused_kernel(const __grid_constant__ TinyParams P, const __grid_constant__ CandInline I,
                                                         TinyMailbox* mb, unsigned long long* srv) {
    extern __shared__ double sm[];
    const double* cands = SERVER ? mb->data : (P.cand ? P.cand : I.x);
    long Mcur = SERVER ? 0 : P.M;
    double* scoreOut = P.score;
    auto ld_cand = [&](size_t i) -> double { return SERVER ? ld_relaxed_sys(cands + i) : cands[i]; };
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d = P.d, XS = d | 1;                   // odd row stride of the training inputs
    const int nside = P.side[1].N > 0 ? 2 : 1;
    // shared-memory carve-up: per side W [N][WS] (lower triangle) and X [N][XS]; then k* [TC][128], the raw candidates of
    // the tile [TC][d], 1/theta [d], and the reduction scratch [3][4][TC]
    double* sW[2]; double* sX[2];
    double* ptr = sm;
    for (int s = 0; s < nside; s++) { sW[s] = ptr; ptr += (size_t)P.side[s].N * WS; sX[s] = ptr; ptr += (size_t)P.side[s].N * XS; }
    double* sK = ptr;  ptr += TC * 128;
    double* sC = ptr;  ptr += TC * d;
    double* sT = ptr;  ptr += d;             // 1 / theta
    double* sCtr = ptr; ptr += 2 * d;        // centres of the two sides
    double* sR = ptr;
    // stage the factors with 8-byte async copies: every element is in flight at once (a register-staged copy of W costs one
    // L2 round trip per row and was most of the kernel's time)
    for (int s = 0; s < nside; s++) {
        const int N = P.side[s].N;
        for (int idx = tid; idx < N * 128; idx += 128) {
            const int r = idx >> 7, c = idx & 127;
            if (c <= r) cp_async8(sW[s] + r * WS + c, P.side[s].W + (size_t)r * 128 + c);
        }
        for (int idx = tid; idx < N * d; idx += 128) {
            const int r = idx / d, q = idx - r * d;
            cp_async8(sX[s] + r * XS + q, P.side[s].Xt + idx);
        }
    }
    for (int q = tid; q < d; q += 128) {
        cp_async8(sT + q, P.invTheta + q);
        for (int s = 0; s < nside; s++) cp_async8(sCtr + s * d + q, P.side[s].center + q);
    }
    asm volatile("cp.async.commit_group;");
    // The first tile's candidates are fetched while the copies above are in flight: for a DIRECT batch they come over PCIe
    // (mapped host memory), the longest latency in the kernel -- everything else hides behind it.
    if (!SERVER)
        for (int idx = tid; idx < TC * d; idx += 128) {
            const int j = idx / d, q = idx - j * d;
            long m = (long)blockIdx.x * TC + j; if (m >= Mcur) m = Mcur - 1;
            sC[idx] = cands[(size_t)m * d + q];
        }
    const int N0 = P.side[0].N;
    const double by = tid < N0 ? P.betaY[tid] : 0.0;
    const double b1 = (tid < N0 && P.npb > 0) ? P.beta1[tid] : 0.0;
    double best = -INFINITY;
    long long bestIdx = 0x7fffffffffffffffLL;
    asm volatile("cp.async.wait_group 0;");
    __shared__ long long sh_seq, sh_M;
    long long lastSeq = 0;
  next_batch:
    if (SERVER) {
        // CTA 0 watches the host's mailbox (one PCIe read per poll) and passes each new batch on through device memory, where
        // the other CTAs wait: sixteen CTAs polling host memory at once made a batch cost 78 us instead of 24
        if (tid == 0) {
            long long w;
            if (blockIdx.x == 0) {
                const unsigned long long t0 = global_timer_ns();
                while ((w = ld_relaxed_sys(&mb->ctrl)) >= 0 && (w >> 24) == lastSeq)
                    if (global_timer_ns() - t0 > 2000000000ull) { w = -2; break; }      // idle for 2 s: everybody leaves (the host restarts the server)
                asm volatile("fence.acq_rel.sys;" ::: "memory");                         // the candidates were written before the word
                asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(srv + 1), "l"((unsigned long long)w) : "memory");
            } else {
                unsigned long long v;
                do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(srv + 1) : "memory"); }
                while ((long long)v >= 0 && ((long long)v >> 24) == lastSeq);
                w = (long long)v;
            }
            sh_seq = w < 0 ? w : (w >> 24);
            sh_M = w < 0 ? 0 : (w & 0xffffff);
        }
        __syncthreads();
        if (sh_seq < 0) return;
        lastSeq = sh_seq;
        Mcur = (long)sh_M;
        scoreOut = mb->data + (size_t)Mcur * d;
    }
    for (long t = blockIdx.x; t < (Mcur + TC - 1) / TC; t += gridDim.x) {
        const long m0 = t * TC;
        if (SERVER || t != blockIdx.x) {
            __syncthreads();                 // previous tile's scratch is free
            for (int idx = tid; idx < TC * d; idx += 128) {
                const int j = idx / d, q = idx - j * d;
                long m = m0 + j; if (m >= Mcur) m = Mcur - 1;
                sC[idx] = ld_cand((size_t)m * d + q);
            }
        }
        double q_sum = 0, p_sum = 0, p1_sum = 0;           // of candidate m0 + tid (threads 0..7)
        for (int s = 0; s < nside; s++) {
            const int N = P.side[s].N;
            __syncthreads();
            // k*[j][c], thread c: direct differences between its training row and the scaled, centred candidates
            {
                double r2[TC];
#pragma unroll
                for (int j = 0; j < TC; j++) r2[j] = 0.0;
                if (tid < N) {
                    const double* x = sX[s] + tid * XS;
                    for (int q = 0; q < d; q++) {
                        const double xv = x[q], it = sT[q], ctr = sCtr[s * d + q];     // rows are stored scaled and centred
#pragma unroll
                        for (int j = 0; j < TC; j++) { const double df = xv - (sC[j * d + q] * it - ctr); r2[j] = fma(df, df, r2[j]); }
                    }
                }
#pragma unroll
                for (int j = 0; j < TC; j++) sK[j * 128 + tid] = tid < N ? cov_r2_t<KC>(P.sf2, r2[j]) : 0.0;
            }
            __syncthreads();
            // v_r[j] = sum_{c <= r} W[r][c] k*[j][c], thread r
            double v[TC];
#pragma unroll
            for (int j = 0; j < TC; j++) v[j] = 0.0;
            if (tid < N) {
                const double* w = sW[s] + tid * WS;
                for (int c = 0; c <= tid; c++) {
                    const double wv = w[c];
#pragma unroll
                    for (int j = 0; j < TC; j++) v[j] = fma(wv, sK[j * 128 + c], v[j]);
                }
            }
            // row reductions: xor tree inside the warp, then the four warps in ascending order
#pragma unroll
            for (int j = 0; j < TC; j++) {
                double q = v[j] * v[j], p = v[j] * by, p1 = v[j] * b1;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    q += __shfl_xor_sync(0xffffffffu, q, o);
                    p += __shfl_xor_sync(0xffffffffu, p, o);
                    p1 += __shfl_xor_sync(0xffffffffu, p1, o);
                }
                if (lane == 0) { sR[(0 * 4 + warp) * TC + j] = q; sR[(1 * 4 + warp) * TC + j] = p; sR[(2 * 4 + warp) * TC + j] = p1; }
            }
            __syncthreads();
            if (tid < TC) {
                double q = 0, p = 0, p1 = 0;
#pragma unroll
                for (int w = 0; w < 4; w++) { q += sR[(0 * 4 + w) * TC + tid]; p += sR[(1 * 4 + w) * TC + tid]; p1 += sR[(2 * 4 + w) * TC + tid]; }
                q_sum = q;                                  // the variance comes from the last side (the aug factor if there is one)
                if (s == 0) { p_sum = p; p1_sum = p1; }     // the mean always from the model itself (gaussianprocess/__init__.py:214-223)
            }
        }
        if (tid < TC && m0 + tid < Mcur) {
            const long m = m0 + tid;
            double mean0 = 0.0;
            if (P.npb > 0) mean0 = prior_mean(sC + tid * d, d, P.npb, P.pmeans, P.pbeta, P.ptheta, P.plb, P.pwidth);
            const double mu = mean0 + p_sum - mean0 * p1_sum;
            double s2 = (1.0 + P.noise) - q_sum;
            const double floor_ = P.mode_py ? 10e-8 : 1e-8;   // gaussianprocess/__init__.py:224 vs cpp/optimizeGP.cpp:150
            s2 = s2 < floor_ ? floor_ : (s2 > 10.0 ? 10.0 : s2);
            if (P.mu) P.mu[m] = mu;
            if (P.s2) P.s2[m] = s2;
            if (P.acq >= 0) {
                const double val = acq_value(P.acq, P.mode_py, mu, s2, P.ymax, P.parm);
                if (scoreOut) scoreOut[m] = val;
                if (val == val) { if (val > best || (val == best && m < bestIdx)) { best = val; bestIdx = m; } }
                else if (bestIdx == 0x7fffffffffffffffLL) bestIdx = m;      // NaN never wins, but an all-NaN set still names an index
            }
        }
    }
    if (SERVER) {
        __syncthreads();
        // a CTA that scored a tile releases its own done word (the release orders its value stores before it); the host waits for
        // exactly the CTAs that own tiles of this batch
        if (tid == 0 && (long)blockIdx.x < (Mcur + TC - 1) / TC) st_release_sys(&mb->done[blockIdx.x], lastSeq);
        goto next_batch;
    }
    if (P.acq < 0 || !P.want_argmax) return;
    // the tile owners (threads 0..7, all in warp 0) combine: lowest index wins ties
    if (warp == 0) {
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const double os = __shfl_xor_sync(0xffffffffu, best, o);
            const long long oi = __shfl_xor_sync(0xffffffffu, bestIdx, o);
            if (os > best || (os == best && oi < bestIdx)) { best = os; bestIdx = oi; }
        }
        if (lane == 0) { P.blkBest[blockIdx.x] = best; P.blkIdx[blockIdx.x] = bestIdx; }
    }
}

cudaError_t set_tiny_attrs() {
    const int maxsm = 200 * 1024;
    cudaError_t e = cudaFuncSetAttribute(tiny_fused_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tiny_fused_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tiny_fused_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tiny_fused_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tiny_fused_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tiny_fused_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm);
    return e;
}

size_t tiny_smem(int N, int Nvar, int d) {
    return sizeof(double) * ((size_t)(N + Nvar) * (WS + (d | 1)) + TC * 128 + (size_t)TC * d + 3 * d + 3 * 4 * TC);
}
constexpr size_t TINY_SMEM_MAX = 200 * 1024;

}  // namespace

// models the fused kernel serves: a single row-block (also for the variance model of PrefGP's aug factor, if any) that
// fits shared memory; IBO_TINY=0 disables
// Batches above TINY_MAX_M go through the general path, whose DMMA kernels have the higher throughput (2^20 candidates at
// N = 128: 1.7 ms vs 6.3 ms here); the two paths agree to rounding, and every DIRECT / gallery batch is far below the limit.
constexpr long TINY_MAX_M = 4096;

bool tiny_eligible(const ibo_model* m, long M) {
    if (M > TINY_MAX_M) return false;
    if (m->nb != 1 || m->d > 64) return false;
    const ibo_model* vm = m->var_model;
    if (vm && (vm->nb != 1 || vm->kind != m->kind || vm->sf2 != m->sf2)) return false;
    if (tiny_smem(m->N, vm ? vm->N : 0, m->d) > TINY_SMEM_MAX) return false;
    return get_option(OPT_TINY) != 0;            // option tiny = 0 disables (the tests compare both paths in one process)
}

// Scores M candidates at `cand` (device memory, or mapped pinned host memory) into out = [score | mu | s2][M] (+ the argmax
// pair at out[3M], out[3M+1]); everything is enqueued on m->stream.
// `inl`: the batch in the parameter buffer (the caller's plan put it there; cand is then null)
int score_tiny(ibo_model* m, const double* cand, long M, const ScoreReq& rq, double* out, const CandInline* inl) {
    const cudaError_t ae = ensure_attrs(m->device, ATTR_TINY, set_tiny_attrs);
    if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); return IBO_E_CUDA; }
    const int g_tiny_sms = dev_info(m->device).sms;
    cudaStream_t st = m->stream;
    const bool prof = (rq.flags & IBO_FLAG_PROFILE) != 0;
    const long ntile = (M + TC - 1) / TC;
    // one CTA per tile up to a few waves; beyond that CTAs walk tiles so that W is staged once per CTA
    const ibo_model* vm = m->var_model;
    const size_t smem = tiny_smem(m->N, vm ? vm->N : 0, m->d);
    const int perSM = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / smem));
    const int grid = (int)std::min<long>(ntile, (long)g_tiny_sms * perSM);
    int rc;
    if ((rc = grow_blk(m, (size_t)grid, (size_t)g_tiny_sms * 8))) return rc;
    TinyParams P;
    P.side[0] = TinySide{m->dW, m->dXt, m->dCenter, m->N};
    P.side[1] = vm ? TinySide{vm->dW, vm->dXt, vm->dCenter, vm->N} : TinySide{nullptr, nullptr, nullptr, 0};
    P.betaY = m->dBetaY; P.beta1 = m->dBeta1; P.invTheta = m->dInvTheta; P.cand = cand;
    P.pmeans = m->dPmeans; P.pbeta = m->dPbeta; P.plb = m->dPlb; P.pwidth = m->dPwidth;
    P.score = rq.want_score ? out : nullptr;
    P.mu = rq.want_mu ? out + M : nullptr;
    P.s2 = rq.want_s2 ? out + 2 * M : nullptr;
    P.blkBest = m->dBlkBest; P.blkIdx = m->dBlkIdx;
    P.M = M; P.d = m->d; P.acq = rq.acq; P.mode_py = (rq.flags & IBO_FLAG_MODE_PY) ? 1 : 0; P.npb = m->npb;
    P.want_argmax = (rq.acq >= 0 && rq.want_argmax) ? 1 : 0;
    P.sf2 = m->sf2; P.noise = m->noise; P.ymax = rq.ymax; P.parm = rq.parm; P.ptheta = m->ptheta;
    static CandInline none;
    const CandInline* Ip = inl ? inl : &none;
    if (prof) IBO_CUDA_TRY(cudaEventRecord(m->ev[0], st));
    if (m->kind <= IBO_KERNEL_SE_ISO) tiny_fused_kernel<0, false><<<grid, 128, smem, st>>>(P, *Ip, nullptr, nullptr);
    else if (m->kind == IBO_KERNEL_MATERN3) tiny_fused_kernel<1, false><<<grid, 128, smem, st>>>(P, *Ip, nullptr, nullptr);
    else tiny_fused_kernel<2, false><<<grid, 128, smem, st>>>(P, *Ip, nullptr, nullptr);
    g_launches++;
    long nlaunch = 1;
    if (P.want_argmax) {
        launch_argmax_final(m->dBlkBest, m->dBlkIdx, grid, out + 3 * M, reinterpret_cast<long long*>(out + 3 * M + 1), st);
        nlaunch++;
    }
    if (prof) {
        IBO_CUDA_TRY(cudaEventRecord(m->ev[5], st));
        IBO_CUDA_TRY(cudaEventSynchronize(m->ev[5]));
        float tot; cudaEventElapsedTime(&tot, m->ev[0], m->ev[5]);
        m->prof[0] = 0; m->prof[1] = tot; m->prof[2] = 0; m->prof[3] = tot; m->prof[4] = (double)nlaunch; m->prof[5] = 1;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

// ---- batch server (host side) ---------------------------------------------------------------------
// Resident kernels must all fit on the device at once (a CTA that never becomes resident never answers): at most four servers
// per device (64 CTAs of <= 200 KB shared memory on 148 SMs); further side-by-side queries (ibo_acqmax_many) launch per batch.
static std::mutex g_srv_mu;
static int g_srv_active[16] = {0};
constexpr int SERVERS_PER_DEVICE = 4;

bool tiny_server_fits(const ibo_model* m, long n) {
    if (!(n >= 1 && get_option(OPT_TINY_SERVER) != 0 && tiny_eligible(m, n) && (size_t)n * (m->d + 1) <= MAILBOX_DOUBLES)) return false;
    if (m->srvRunning) return true;
    std::lock_guard<std::mutex> lk(g_srv_mu);
    return g_srv_active[m->device & 15] < SERVERS_PER_DEVICE;
}

static void server_gone(ibo_model* m) {      // the kernel is no longer there (idle timeout, error)
    if (!m->srvRunning) return;
    m->srvRunning = false;
    std::lock_guard<std::mutex> lk(g_srv_mu);
    g_srv_active[m->device & 15]--;
}

static int tiny_server_start(ibo_model* m, int acq, double ymax, double parm, int flags) {
    const cudaError_t ae = ensure_attrs(m->device, ATTR_TINY, set_tiny_attrs);
    if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); return IBO_E_CUDA; }
    cudaStream_t st = m->stream;
    if (!m->hServer) IBO_CUDA_TRY(pinned_get(&m->hServer));
    if (!m->dSrvCount) IBO_CUDA_TRY(cudaMalloc(&m->dSrvCount, 4 * sizeof(unsigned long long)));
    TinyMailbox* mb = reinterpret_cast<TinyMailbox*>(m->hServer);
    mb->ctrl = 0;
    for (int c = 0; c < 16; c++) mb->done[c] = 0;
    m->srvSeq = 0;
    IBO_CUDA_TRY(cudaMemsetAsync(m->dSrvCount, 0, 4 * sizeof(unsigned long long), st));
    const ibo_model* vm = m->var_model;
    const size_t smem = tiny_smem(m->N, vm ? vm->N : 0, m->d);
    TinyParams P;
    P.side[0] = TinySide{m->dW, m->dXt, m->dCenter, m->N};
    P.side[1] = vm ? TinySide{vm->dW, vm->dXt, vm->dCenter, vm->N} : TinySide{nullptr, nullptr, nullptr, 0};
    P.betaY = m->dBetaY; P.beta1 = m->dBeta1; P.invTheta = m->dInvTheta; P.cand = nullptr;
    P.pmeans = m->dPmeans; P.pbeta = m->dPbeta; P.plb = m->dPlb; P.pwidth = m->dPwidth;
    P.score = nullptr; P.mu = nullptr; P.s2 = nullptr;
    P.blkBest = nullptr; P.blkIdx = nullptr;
    P.M = 0; P.d = m->d; P.acq = acq; P.mode_py = (flags & IBO_FLAG_MODE_PY) ? 1 : 0; P.npb = m->npb;
    P.want_argmax = 0;
    P.sf2 = m->sf2; P.noise = m->noise; P.ymax = ymax; P.parm = parm; P.ptheta = m->ptheta;
    static CandInline none;
    const int grid = std::min(SERVER_CTAS, dev_info(m->device).sms);
    m->srvCtas = grid;
    if (m->kind <= IBO_KERNEL_SE_ISO) tiny_fused_kernel<0, true><<<grid, 128, smem, st>>>(P, none, mb, m->dSrvCount);
    else if (m->kind == IBO_KERNEL_MATERN3) tiny_fused_kernel<1, true><<<grid, 128, smem, st>>>(P, none, mb, m->dSrvCount);
    else tiny_fused_kernel<2, true><<<grid, 128, smem, st>>>(P, none, mb, m->dSrvCount);
    IBO_CUDA_TRY(cudaGetLastError());
    g_launches++;
    { std::lock_guard<std::mutex> lk(g_srv_mu); g_srv_active[m->device & 15]++; }
    m->srvRunning = true;
    m->srvAcq = acq; m->srvYmax = ymax; m->srvParm = parm; m->srvFlags = flags;
    return IBO_OK;
}

void tiny_server_stop(ibo_model* m) {
    if (!m || !m->srvRunning) return;
    cudaSetDevice(m->device);
    TinyMailbox* mb = reinterpret_cast<TinyMailbox*>(m->hServer);
    std::atomic_thread_fence(std::memory_order_release);
    *reinterpret_cast<volatile long long*>(&mb->ctrl) = -1;
    cudaStreamSynchronize(m->stream);
    m->srvRunning = false;
    std::lock_guard<std::mutex> lk(g_srv_mu);
    g_srv_active[m->device & 15]--;
}

int tiny_server_eval(ibo_model* m, const double* X, long n, int acq, double ymax, double parm, int flags, double* y) {
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if (m->srvRunning && (acq != m->srvAcq || ymax != m->srvYmax || parm != m->srvParm || flags != m->srvFlags)) tiny_server_stop(m);
    for (int attempt = 0; attempt < 3; attempt++) {
        if (!m->srvRunning) { int rc = tiny_server_start(m, acq, ymax, parm, flags); if (rc) return rc; }
        TinyMailbox* mb = reinterpret_cast<TinyMailbox*>(m->hServer);
        const size_t nin = (size_t)n * m->d;
        std::memcpy(mb->data, X, sizeof(double) * nin);
        const long long seq = ++m->srvSeq;
        std::atomic_thread_fence(std::memory_order_release);
        *reinterpret_cast<volatile long long*>(&mb->ctrl) = (seq << 24) | (long long)n;
        // wait for the values: plain reads of host memory; every 2^16 spins make sure the kernel is still there
        const int nwait = (int)std::min<long>((n + TC - 1) / TC, m->srvCtas);
        const auto t0 = std::chrono::steady_clock::now();
        bool gone = false;
        int c = 0;
        for (unsigned long spins = 1; c < nwait; spins++) {
            if (*reinterpret_cast<volatile long long*>(&mb->done[c]) == seq) { c++; continue; }
            if ((spins & 0xffff) == 0) {
                const cudaError_t q = cudaStreamQuery(m->stream);
                if (q == cudaSuccess) { gone = true; break; }      // the kernel left (its idle timeout raced with this batch): once more
                if (q != cudaErrorNotReady) { server_gone(m); set_error(std::string("small-model batch server: ") + cudaGetErrorString(q)); cudaGetLastError(); return IBO_E_CUDA; }
                if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 20.0) {
                    set_error("small-model batch server: no answer for 20 s"); return IBO_E_CUDA;
                }
            }
        }
        if (gone) { server_gone(m); continue; }
        std::atomic_thread_fence(std::memory_order_acquire);
        const double* sc = mb->data + nin;
        for (long i = 0; i < n; i++) y[i] = -sc[i];
        return IBO_OK;
    }
    set_error("small-model batch server: the kernel keeps leaving");
    return IBO_E_CUDA;
}

}  // namespace ibo
