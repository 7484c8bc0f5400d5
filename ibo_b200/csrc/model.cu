// Model build on the GPU: A = K_offdiag + (1+noise) I [+ Cinv], blocked FP64 Cholesky A = L L^T,
// W = inv(L) by blocked right-looking substitution, fragment-packing of W for the scoring GEMM,
// beta = W Y.  All off-diagonal block updates run on the FP64 tensor pipe (DMMA.8x8x4).
//
// Replaces (reference file:line): GaussianProcess._computeCorrelations / addData
// (ego/gaussianprocess/__init__.py:134-149,267-308), linalg.cholesky(R + inv(C)) (:487-498) and
// the explicit linalg.inv(R) of cdirectGP (ego/acquisition/__init__.py:385-388).
#include "model.cuh"
#include "tilegemm.cuh"
#include <cmath>
#include <cstring>
#include <mutex>
#include <map>
#include <set>

namespace ibo {

long g_launches = 0;
static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }
const char* get_error() { return g_err.c_str(); }

// ---------------------------------------------------------------------------------------------
// Small caching allocator: sequential BO and fastUCBGallery rebuild the model after every addData, and
// cudaMalloc / cudaFree of the N x N buffers (plus their implicit device synchronisation) would otherwise dominate
// the rebuild.  Freed blocks are kept per device and handed back for requests of up to 2x smaller size.
// ---------------------------------------------------------------------------------------------
namespace {
struct Pool {
    std::mutex mu;
    std::multimap<size_t, void*> free_blocks[16];
    std::map<void*, size_t> live;
    size_t cached[16] = {0};
    static constexpr size_t LIMIT = (size_t)12 << 30;
} g_pool;
}

cudaError_t pool_malloc(void** p, size_t bytes) {
    int dev = 0; cudaGetDevice(&dev); dev &= 15;
    bytes = (bytes + 511) & ~(size_t)511;
    std::lock_guard<std::mutex> lk(g_pool.mu);
    auto& fb = g_pool.free_blocks[dev];
    auto it = fb.lower_bound(bytes);
    if (it != fb.end() && it->first <= 2 * bytes + (1 << 20)) {
        *p = it->second;
        g_pool.live[*p] = it->first;
        g_pool.cached[dev] -= it->first;
        fb.erase(it);
        return cudaSuccess;
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {     // give cached memory back to the driver and retry once
        cudaGetLastError();
        for (auto& kv : fb) cudaFree(kv.second);
        fb.clear(); g_pool.cached[dev] = 0;
        e = cudaMalloc(p, bytes);
    }
    if (e == cudaSuccess) g_pool.live[*p] = bytes;
    return e;
}

// pinned 1 MiB staging buffers (small-batch path of score_host) are recycled too
static std::vector<double*> g_pinned_free;
cudaError_t pinned_get(double** p) {
    {
        std::lock_guard<std::mutex> lk(g_pool.mu);
        if (!g_pinned_free.empty()) { *p = g_pinned_free.back(); g_pinned_free.pop_back(); return cudaSuccess; }
    }
    return cudaHostAlloc((void**)p, sizeof(double) * (1u << 17), cudaHostAllocMapped | cudaHostAllocPortable);
}
void pinned_put(double* p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_pool.mu);
    g_pinned_free.push_back(p);
}

void pool_free(void* p) {
    if (!p) return;
    int dev = 0; cudaGetDevice(&dev); dev &= 15;
    std::lock_guard<std::mutex> lk(g_pool.mu);
    auto it = g_pool.live.find(p);
    if (it == g_pool.live.end()) { cudaFree(p); return; }
    size_t bytes = it->second;
    g_pool.live.erase(it);
    if (g_pool.cached[dev] + bytes > Pool::LIMIT) { cudaFree(p); return; }
    g_pool.free_blocks[dev].insert(std::make_pair(bytes, p));
    g_pool.cached[dev] += bytes;
}

int grow(double** p, size_t* cap, size_t need) {
    if (*cap >= need) return IBO_OK;
    if (*p) pool_free(*p);
    *p = nullptr; *cap = 0;
    size_t want = need + need / 8;
    cudaError_t e = pool_malloc((void**)p, want * sizeof(double));
    if (e != cudaSuccess) {
        e = pool_malloc((void**)p, need * sizeof(double));
        want = need;
        if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); cudaGetLastError(); return IBO_E_NOMEM; }
    }
    *cap = want;
    return IBO_OK;
}

// ---------------------------------------------------------------------------------------------
// covariance function on the scaled squared distance r2 = sum_j ((x_j - y_j)/theta_j)^2
//   (ego/gaussianprocess/kernel.py:87-89,147-149,207-210,246-248; cpp/optimizeGP.cpp:70-112)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double cov_from_r2(int kind, double sf2, double r2) {
    if (kind <= IBO_KERNEL_SE_ISO) return sf2 * exp(-0.5 * r2);
    double r = sqrt(r2);
    if (kind == IBO_KERNEL_MATERN3) {
        double z = 1.7320508075688772 * r;   // sqrt(3)
        return sf2 * (1.0 + z) * exp(-z);
    }
    double z = 2.23606797749979 * r;         // sqrt(5)
    return sf2 * (1.0 + z + 5.0 * r2 / 3.0) * exp(-z);
}

// A[i][j] = k(x_i, x_j) (i != j), `diag` (1 + noise for the GP's R) on the diagonal, + Cinv; identity in the padding.
__global__ void build_A_kernel(double* __restrict__ A, const double* __restrict__ Xt, const double* __restrict__ Cinv,
                               int N, int Np, int d, int kind, double sf2, double diag) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= Np) return;
    double v;
    if (i >= N || j >= N) v = (i == j) ? 1.0 : 0.0;
    else if (i == j) v = diag;
    else {
        // evaluate with (min,max) ordering so that A is exactly symmetric
        int a = i < j ? i : j, b = i < j ? j : i;
        double r2 = 0;
        for (int t = 0; t < d; t++) { double df = Xt[(size_t)a * d + t] - Xt[(size_t)b * d + t]; r2 += df * df; }
        v = cov_from_r2(kind, sf2, r2);
    }
    if (Cinv && i < N && j < N) v += Cinv[(size_t)i * N + j];
    A[(size_t)i * Np + j] = v;
}

// C = cdiag I + sum_p w_p (e_a - e_b)(e_a - e_b)^T over the preference pairs (a_p, b_p): the Laplace term of PrefGaussianProcess
// (ego/gaussianprocess/__init__.py:461-486).  One thread per row walks the pairs in their given order, so every entry is summed
// in a fixed order (no atomics); identity in the padding.
__global__ void pref_build_C_kernel(double* __restrict__ C, int N, int Np, int P, const int* __restrict__ pa, const int* __restrict__ pb,
                                    const double* __restrict__ w, double cdiag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    double* row = C + (size_t)i * Np;
    for (int j = 0; j < Np; j++) row[j] = 0.0;
    if (i >= N) { row[i] = 1.0; return; }
    double dg = cdiag;
    for (int p = 0; p < P; p++) {
        const int a = pa[p], b = pb[p];
        if (a == b) continue;
        if (a == i) { dg += w[p]; row[b] -= w[p]; }
        else if (b == i) { dg += w[p]; row[a] -= w[p]; }
    }
    row[i] = dg;
}
// A[i][j] += S[max(i,j)][min(i,j)] for i, j < N: S holds the lower 128 x 128 tiles of a symmetric matrix (gram_wtw_kernel)
// A = [C 0; 0 I]: a dense N x N matrix padded to Np x Np
__global__ void pad_copy_kernel(double* __restrict__ A, const double* __restrict__ src, int N, int Np) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= Np) return;
    A[(size_t)i * Np + j] = (i < N && j < N) ? src[(size_t)i * N + j] : (i == j ? 1.0 : 0.0);
}
__global__ void add_symmetric_lower_kernel(double* __restrict__ A, const double* __restrict__ S, int N, int Np) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (i >= N || j >= N) return;
    const int hi = i > j ? i : j, lo = i > j ? j : i;
    // inside a diagonal tile both triangles were computed; take the lower one so that the sum is exactly symmetric
    A[(size_t)i * Np + j] += S[(size_t)hi * Np + lo];
}

// A_rev = J invR J (reversal of the leading N x N part), identity padding -- legacy acqmaxGP path.
__global__ void build_reversed_kernel(double* __restrict__ A, const double* __restrict__ invR, int N, int Np) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= Np) return;
    double v;
    if (i >= N || j >= N) v = (i == j) ? 1.0 : 0.0;
    else v = invR[(size_t)(N - 1 - i) * N + (N - 1 - j)];
    A[(size_t)i * Np + j] = v;
}

// W'[i][j] = G[N-1-j][N-1-i] for j <= i < N (G = chol(J invR J)), identity padding, zeros above.
__global__ void reverse_transpose_kernel(double* __restrict__ W, const double* __restrict__ G, int N, int Np) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= Np) return;
    double v = 0.0;
    if (i >= N || j >= N) v = (i == j) ? 1.0 : 0.0;
    else if (j <= i) v = G[(size_t)(N - 1 - j) * Np + (N - 1 - i)];
    W[(size_t)i * Np + j] = v;
}

__global__ void set_identity_kernel(double* __restrict__ W, int Np) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j < Np) W[(size_t)i * Np + j] = (i == j) ? 1.0 : 0.0;
}

// ---------------------------------------------------------------------------------------------
// Diagonal block: L_kk = chol(A_kk) in place (lower), D_k = inv(L_kk) (dense 128x128, zeros above).
// One CTA, 512 threads, the block lives in shared memory.  The kernel sits on the critical path of every block step of the
// factorisation (one launch per 128 columns, nothing else can run before it), so everything with more than 8 x 8 work in it
// goes through the FP64 tensor-core instruction (mma.sync m8n8k4), 16 warps at a time:
//   * Cholesky, right-looking over 16 panels of 8 columns: the threads of warps 0-3 factor the 8 x 8 diagonal block in
//     registers (all the same values, no broadcast through shared memory; rsqrt instead of sqrt + divide) and thread t solves
//     row t of the panel below it; the rank-8 update of the trailing triangle is one 8 x 8 tile = two MMAs per warp and turn.
//   * Inverse in place by doubling: the sixteen 8 x 8 diagonal blocks first (one thread per column), then for b = 8, 16, 32, 64
//     every pair of adjacent b x b inverses is merged, X21 = -X22 (L21 X11): two tile GEMMs that skip the zero blocks of the
//     triangular factors, with the b x b product parked in a side buffer.
// clock64 timeline of the debug build (tools/potrf_trace.py), before -> after this organisation: see DESIGN.md section 4.
// info gets the first failing global pivot (1-based) if A is not SPD.
// ---------------------------------------------------------------------------------------------
// One level of the in-place inversion of potrf_diag_kernel: every pair of adjacent B x B inverses on the diagonal of S becomes one
// 2B x 2B inverse, X21 = -X22 (L21 X11).  8 x 8 tiles, B tiles per level in all, dealt to the 16 warps; T = L21 X11 is parked in Tb.
template <int B>
__device__ __forceinline__ void potrf_merge_level(double* S, double* Tb, int warp, int lr, int lc) {
    constexpr int PS_ = 132, tb = B >> 3, ts = B + 4;      // PS_: row stride of S (= PS below)
    // T = L21 X11: X11 is lower triangular, so column tile nt needs k >= 8 nt only
    for (int t = warp; t < B; t += 16) {
        const int p = t / (tb * tb), tt = t % (tb * tb), nt = tt / tb, mt = tt % tb, base = 2 * p * B;
        const double* ap = S + (base + B + 8 * mt + lr) * PS_ + base + lc;
        const double* bp = S + (base + lc) * PS_ + base + 8 * nt + lr;
        double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll 2
        for (int k = 8 * nt; k < B; k += 8) {
            dmma884(c0, c1, ap[k], bp[k * PS_]);
            dmma884(d0, d1, ap[k + 4], bp[(k + 4) * PS_]);
        }
        *reinterpret_cast<double2*>(Tb + p * B * ts + (8 * mt + lr) * ts + 8 * nt + 2 * lc) = make_double2(c0 + d0, c1 + d1);
    }
    __syncthreads();
    // X21 = -X22 T: X22 is lower triangular, so row tile mt needs k < 8 (mt + 1) only; X21 replaces L21
    for (int t = warp; t < B; t += 16) {
        const int p = t / (tb * tb), tt = t % (tb * tb), mt = tt / tb, nt = tt % tb, base = 2 * p * B;
        const double* ap = S + (base + B + 8 * mt + lr) * PS_ + base + B + lc;
        const double* bp = Tb + p * B * ts + lc * ts + 8 * nt + lr;
        double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll 2
        for (int k = 0; k < 8 * (mt + 1); k += 8) {
            dmma884(c0, c1, ap[k], bp[k * ts]);
            dmma884(d0, d1, ap[k + 4], bp[(k + 4) * ts]);
        }
        *reinterpret_cast<double2*>(S + (base + B + 8 * mt + lr) * PS_ + base + 8 * nt + 2 * lc) = make_double2(-(c0 + d0), -(c1 + d1));
    }
    __syncthreads();
}

#ifdef IBO_I8_TRACE
__device__ long long g_potrf_stamp[72];
#define PSTAMP(i) do { if (threadIdx.x == 0) g_potrf_stamp[i] = clock64(); } while (0)
#else
#define PSTAMP(i) do { } while (0)
#endif
constexpr int PS = 132;    // smem row stride of the 128 x 128 block: 4 mod 16 keeps the MMA fragment loads conflict-free
constexpr int POTRF_SMEM = (128 * PS + 64 * 68 + 128) * 8;
static_assert(PS == 132, "potrf_merge_level carries the same stride");
__global__ void __launch_bounds__(512) potrf_diag_kernel(double* __restrict__ A, int ld, int kblk,
                                                         double* __restrict__ Dall, int* __restrict__ info) {
    extern __shared__ __align__(16) double sm[];
    double* S = sm;                            // [128][PS] the block: L, then X = inv(L) in place; zeros above the diagonal
    double* Tb = sm + 128 * PS;                // products L21 X11 of the merge step, one b x (b + 4) slab per pair
    double* Dinv = Tb + 64 * 68;               // 1 / L_jj
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lr = lane >> 2, lc = lane & 3;   // MMA fragment coordinates of this lane
    double* Ablk = A + (size_t)kblk * 128 * ld + (size_t)kblk * 128;
    for (int idx = tid; idx < 128 * 64; idx += 512) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        double2 v = make_double2(0.0, 0.0);
        if (c <= r) {
            v = *reinterpret_cast<const double2*>(Ablk + (size_t)r * ld + c);
            if (c + 1 > r) v.y = 0.0;
        }
        *reinterpret_cast<double2*>(S + r * PS + c) = v;
    }
    PSTAMP(0);
    __syncthreads();
    PSTAMP(1);
    // ---------------- Cholesky ----------------
#pragma unroll 1
    for (int c0 = 0; c0 < 128; c0 += 8) {
        const int nbelow = 120 - c0;
        double a[8][8], invd[8];
        if (tid < 128) {
            // (1) 8 x 8 diagonal block in registers, every thread the same (broadcast reads)
#pragma unroll
            for (int r = 0; r < 8; r++)
#pragma unroll
                for (int c = 0; c <= r; c++) a[r][c] = S[(c0 + r) * PS + c0 + c];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                double piv = a[j][j];
                if (!(piv > 0.0)) {   // also catches NaN
                    if (tid == 0) atomicCAS(info, 0, kblk * 128 + c0 + j + 1);
                    piv = 1.0;        // keep going with garbage; the host checks info
                }
                const double ij = rsqrt(piv);
                a[j][j] = piv * ij; invd[j] = ij;
#pragma unroll
                for (int i = j + 1; i < 8; i++) a[i][j] *= ij;
#pragma unroll
                for (int i = j + 1; i < 8; i++)
#pragma unroll
                    for (int c = j + 1; c <= i; c++) a[i][c] = fma(-a[i][j], a[c][j], a[i][c]);
            }
            PSTAMP(2 + 3 * (c0 >> 3));
            // (2) rows below: thread t solves row c0 + 8 + t of the panel, x L11^T = b
            if (tid < nbelow) {
                double2* row = reinterpret_cast<double2*>(S + (c0 + 8 + tid) * PS + c0);
                double x[8];
#pragma unroll
                for (int j = 0; j < 8; j += 2) { double2 v = row[j >> 1]; x[j] = v.x; x[j + 1] = v.y; }
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    double v = x[j];
#pragma unroll
                    for (int q = 0; q < j; q++) v = fma(-x[q], a[j][q], v);
                    x[j] = v * invd[j];
                }
#pragma unroll
                for (int j = 0; j < 8; j += 2) row[j >> 1] = make_double2(x[j], x[j + 1]);
            }
        }
        __syncthreads();
        PSTAMP(3 + 3 * (c0 >> 3));
        // L11 and its reciprocal diagonal go back to shared memory only now (before the barrier another warp may still be reading
        // the unfactored block), split over two threads with static register indices; the trailing update never touches these rows
        if (tid == 126) {
#pragma unroll
            for (int r = 0; r < 6; r++)
#pragma unroll
                for (int c = 0; c <= r; c++) S[(c0 + r) * PS + c0 + c] = a[r][c];
        } else if (tid == 127) {
#pragma unroll
            for (int r = 6; r < 8; r++)
#pragma unroll
                for (int c = 0; c <= r; c++) S[(c0 + r) * PS + c0 + c] = a[r][c];
#pragma unroll
            for (int r = 0; r < 8; r++) Dinv[c0 + r] = invd[r];
        }
        // (3) trailing triangle (rows / cols >= c0 + 8) -= P P^T, P = the panel just solved: 8 x 8 tiles, two MMAs each.
        // Tile rows i and n-1-i are folded into one run of n + 1 tiles, which enumerates the triangle without a square root.
        // (one tile and two chained MMAs per warp and turn measured fastest: batches of 2 or 4 tiles with independent accumulators
        // cost ~220 clk per MMA and warp however they were arranged)
        {
            const int n = nbelow >> 3, nfold = (n + 1) >> 1;
            for (int q = warp; q < nfold * (n + 1); q += 16) {
                const int pr = q / (n + 1), off = q - pr * (n + 1);
                int ti, tj;
                if (off <= pr) { ti = pr; tj = off; }
                else { ti = n - 1 - pr; tj = off - pr - 1; if (ti == pr) continue; }
                const int r0 = c0 + 8 + 8 * ti, q0 = c0 + 8 + 8 * tj;
                const double* ap = S + (r0 + lr) * PS + c0 + lc;
                const double* bp = S + (q0 + lr) * PS + c0 + lc;
                double2* cp = reinterpret_cast<double2*>(S + (r0 + lr) * PS + q0 + 2 * lc);
                const double a0 = -ap[0], a1 = -ap[4], b0 = bp[0], b1 = bp[4];
                double2 c = *cp;
                dmma884(c.x, c.y, a0, b0);
                dmma884(c.x, c.y, a1, b1);
                if (ti != tj) *cp = c;
                else {   // diagonal tile: the upper triangle stays zero
                    if (2 * lc <= lr) S[(r0 + lr) * PS + q0 + 2 * lc] = c.x;
                    if (2 * lc + 1 <= lr) S[(r0 + lr) * PS + q0 + 2 * lc + 1] = c.y;
                }
            }
        }
        __syncthreads();
        PSTAMP(4 + 3 * (c0 >> 3));
    }
    for (int idx = tid; idx < 128 * 64; idx += 512) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        if (c + 1 <= r) *reinterpret_cast<double2*>(Ablk + (size_t)r * ld + c) = *reinterpret_cast<const double2*>(S + r * PS + c);
        else if (c == r) Ablk[(size_t)r * ld + c] = S[r * PS + c];
    }
    __syncthreads();   // the inverse overwrites S
    PSTAMP(50);
    // ---------------- X = inv(L), in place ----------------
    if (tid < 128) {
        // X_jj = inv(L_jj): thread = (block j, column c); forward substitution down the column.  The eight threads of a block
        // share a warp: everyone reads L_jj before anyone overwrites it.
        const int j = tid >> 3, c = tid & 7, b0 = 8 * j;
        double l[8][8], x[8];
#pragma unroll
        for (int r = 0; r < 8; r++)
#pragma unroll
            for (int q = 0; q < r; q++) l[r][q] = S[(b0 + r) * PS + b0 + q];
#pragma unroll
        for (int r = 0; r < 8; r++) {
            double v = (r == c) ? 1.0 : 0.0;
#pragma unroll
            for (int q = 0; q < r; q++)
                if (q >= c) v = fma(-l[r][q], x[q], v);
            x[r] = (r >= c) ? v * Dinv[b0 + r] : 0.0;
        }
        __syncwarp();
#pragma unroll
        for (int r = 0; r < 8; r++)
            if (r >= c) S[(b0 + r) * PS + b0 + c] = x[r];
    }
    __syncthreads();
    PSTAMP(51);
    // merge pairs of b x b inverses: [X11 0; X21 X22] with X21 = -X22 (L21 X11)
    potrf_merge_level<8>(S, Tb, warp, lr, lc);   PSTAMP(52);
    potrf_merge_level<16>(S, Tb, warp, lr, lc);  PSTAMP(53);
    potrf_merge_level<32>(S, Tb, warp, lr, lc);  PSTAMP(54);
    potrf_merge_level<64>(S, Tb, warp, lr, lc);  PSTAMP(55);
    double* D = Dall + (size_t)kblk * 128 * 128;
    for (int idx = tid; idx < 128 * 64; idx += 512) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        double2 v = make_double2(0.0, 0.0);
        if (c <= r) { v = *reinterpret_cast<const double2*>(S + r * PS + c); if (c + 1 > r) v.y = 0.0; }
        *reinterpret_cast<double2*>(D + r * 128 + c) = v;
    }
    PSTAMP(67);
}

enum { MODE_CHOL_PANEL = 0, MODE_CHOL_TRAIL = 1, MODE_TRTRI_SCALE = 2, MODE_TRTRI_UPDATE = 3 };

// C_ij = [i == j] I + G_i G_j^T for the lower tiles j <= i; G is [Np][K] row-major (K a multiple of 16).
// Used by the Laplace fit (laplace.cu): B = I + L^T Lambda L as a rank-P update.
__global__ void __launch_bounds__(256, 1) syrk_identity_kernel(double* __restrict__ C, const double* __restrict__ G, int Np, int K) {
    extern __shared__ double sm[];
    const int i = blockIdx.y, j = blockIdx.x;
    if (j > i) return;
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    tile_gemm_core<true>(G + (size_t)i * 128 * K, K, G + (size_t)j * 128 * K, K, K, acc, sm);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
    double* Ct = C + (size_t)i * 128 * Np + (size_t)j * 128;
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            int r = wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            double2 v;
            v.x = acc[mt][nt][0] + ((i == j && r == c) ? 1.0 : 0.0);
            v.y = acc[mt][nt][1] + ((i == j && r == c + 1) ? 1.0 : 0.0);
            *reinterpret_cast<double2*>(Ct + (size_t)r * Np + c) = v;
        }
}


// the tile a CTA will read-modify-write at its end, requested into L2 at its start (the trailing matrix does not stay in L2 between
// two passes once N > ~3000)
template <int MROWS>
__device__ __forceinline__ void prefetch_tile_l2(const double* C, int Np) {
    for (int idx = threadIdx.x; idx < MROWS * 8; idx += 2 * MROWS)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(C + (size_t)(idx >> 3) * Np + (idx & 7) * 16));
}

// MROWS = 64: the tile is split into an upper and a lower half (blockIdx.z), one 4-warp CTA each, two CTAs per SM
template <int MODE, int MROWS = 128>
__global__ void __launch_bounds__(2 * MROWS, MROWS == 128 ? 1 : 2) block_step_kernel(double* __restrict__ A, double* __restrict__ W,
                                                            const double* __restrict__ D, int Np, int k, int jofs = 0,
                                                            int c0 = -1, int kspan = 128) {
    static_assert(MROWS == 128 || MODE != MODE_TRTRI_SCALE, "the in-place scaling reads all 128 rows of the block it overwrites");
    extern __shared__ double sm[];
    double acc[8][4][2];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
    const size_t half = MROWS == 128 ? 0 : (size_t)blockIdx.z * 64 * Np;      // offset of this CTA's rows inside the block row
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wm = warp >> 2, wn = warp & 3;
    double* C;
    bool subtract;
    if (MODE == MODE_CHOL_PANEL) {
        // A_ik <- A_ik * D_k^T, i = k+1+blockIdx.x
        int i = k + 1 + blockIdx.x;
        C = A + (size_t)i * 128 * Np + half + (size_t)k * 128;
        tile_gemm_core<true, false, MROWS>(C, Np, D + (size_t)k * 128 * 128, 128, 128, acc, sm);
        subtract = false;
    } else if (MODE == MODE_CHOL_TRAIL) {
        // A_ij -= sum over the block columns k .. k + kspan/128 - 1 of L_i. L_j.^T, for c0 <= j <= i: rows from block c0, columns from
        // block c0 + jofs (the look-ahead launches the nearest columns separately)
        if (c0 < 0) c0 = k + 1;
        int i = c0 + blockIdx.y, j = c0 + jofs + blockIdx.x;
        if (j > i) return;
        C = A + (size_t)i * 128 * Np + half + (size_t)j * 128;
        prefetch_tile_l2<MROWS>(C, Np);
        tile_gemm_core<true, false, MROWS>(A + (size_t)i * 128 * Np + half + (size_t)k * 128, Np, A + (size_t)j * 128 * Np + (size_t)k * 128, Np, kspan, acc, sm);
        subtract = true;
    } else if (MODE == MODE_TRTRI_SCALE) {
        // W_kj <- D_k * B_kj, j = blockIdx.x <= k   (B lives in W)
        int j = blockIdx.x;
        C = W + (size_t)k * 128 * Np + (size_t)j * 128;
        tile_gemm_core<false>(D + (size_t)k * 128 * 128, 128, C, Np, 128, acc, sm);
        subtract = false;
    } else {
        // B_ij -= sum over the block rows k .. k + kspan/128 - 1 of L_i. W_.j, for i >= c0 (default k + 1) and j = blockIdx.x
        if (c0 < 0) c0 = k + 1;
        int i = c0 + blockIdx.y, j = blockIdx.x;
        C = W + (size_t)i * 128 * Np + half + (size_t)j * 128;
        prefetch_tile_l2<MROWS>(C, Np);
        tile_gemm_core<false, false, MROWS>(A + (size_t)i * 128 * Np + half + (size_t)k * 128, Np, W + (size_t)k * 128 * Np + (size_t)j * 128, Np, kspan, acc, sm);
        subtract = true;
    }
    // all operand reads are complete (tile_gemm_core ends with __syncthreads) -> in-place write is safe
#pragma unroll
    for (int mt = 0; mt < 8; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++) {
            int r = wm * 64 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + 2 * (lane & 3);
            double2* p = reinterpret_cast<double2*>(C + (size_t)r * Np + c);
            double2 v;
            if (subtract) { v = *p; v.x -= acc[mt][nt][0]; v.y -= acc[mt][nt][1]; }
            else { v.x = acc[mt][nt][0]; v.y = acc[mt][nt][1]; }
            *p = v;
        }
}

// Pack W (row-major, lower) into fragment-major blobs for the scoring GEMM.
__global__ void pack_w_kernel(const double* __restrict__ W, double* __restrict__ Wpack, int Np, int nb) {
    // one CTA per (row-block i, k-blob kb <= (i+1)*8-1)
    int i = blockIdx.y, kb = blockIdx.x;
    if (kb >= (i + 1) * KB_PER_BLOCK) return;
    double* blob = Wpack + (wpack_base(i) + kb) * (size_t)BLOB;
    for (int idx = threadIdx.x; idx < BLOB; idx += blockDim.x) {
        int r = idx >> 4, kk = idx & 15;
        blob[blob_offset(r, kk)] = W[(size_t)(i * 128 + r) * Np + kb * BK + kk];
    }
}

// out[r] = sum_{c<=r} W[r][c] * v[c]  (one warp per row; fixed summation order)
__global__ void tri_matvec_kernel(const double* __restrict__ W, const double* __restrict__ v, double* __restrict__ out, int Np) {
    int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (r >= Np) return;
    double s = 0;
    for (int c = lane; c <= r; c += 32) s += W[(size_t)r * Np + c] * v[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[r] = s;
}


// ---------------------------------------------------------------------------------------------
// Rank-1 append of an observation (ego/gaussianprocess/__init__.py:300-308 with a one-row block):
//   k = k(X, x_p), l = W k (= inv(L) k), lambda = sqrt(1 + noise - l.l),
//   L <- [[L, 0], [l^T, lambda]],  W <- [[W, 0], [-(l^T W) / lambda, 1 / lambda]],  beta_p = W_p . Y
// O(N^2) instead of the O(N^3) rebuild; the new row lands in the identity padding of the 128-row block, so the
// scoring kernels see it without any re-layout (only row p's entries of the packed blobs are rewritten).
// Workspace: x_new[d] | kvec[Np] | l[Np] | u[Np] | lambda, 1/lambda.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) append_kvec_kernel(double* __restrict__ Xt, const double* __restrict__ xnew, double* __restrict__ kvec,
                                                          double* __restrict__ Aorig, int p, int Np, int d, int kind, double sf2, double noise) {
    int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= Np) return;
    double v = 0.0;
    if (c < p) {
        double r2 = 0;
        for (int t = 0; t < d; t++) { double df = Xt[(size_t)c * d + t] - xnew[t]; r2 += df * df; }   // (min, max) order as build_A_kernel
        v = cov_from_r2(kind, sf2, r2);
    }
    kvec[c] = v;
    if (Aorig) {
        if (c < p) { Aorig[(size_t)p * Np + c] = v; Aorig[(size_t)c * Np + p] = v; }
        else if (c == p) Aorig[(size_t)p * Np + p] = 1.0 + noise;
    }
    if (c < d) Xt[(size_t)p * d + c] = xnew[c];
}

// u[c] = sum_{r=c}^{p-1} l[r] W[r][c]: 16 columns x 16 row lanes per CTA, lanes summed in a fixed order
__global__ void __launch_bounds__(256) append_colsum_kernel(const double* __restrict__ W, const double* __restrict__ l, double* __restrict__ u,
                                                            int p, int Np) {
    __shared__ double red[16][17];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int c0 = blockIdx.x * 16, c = c0 + tx;
    double acc = 0;
    for (int r = c0 + ty; r < p; r += 16)
        if (r >= c) acc = fma(l[r], W[(size_t)r * Np + c], acc);   // lower triangle only (dA keeps stale values above it)
    red[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && c < p) {
        double s = 0;
#pragma unroll
        for (int t = 0; t < 16; t++) s += red[t][tx];
        u[c] = s;
    }
}

__device__ __forceinline__ double block_sum_256(double v, double* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) s += sh[w];
    __syncthreads();
    return s;
}

__global__ void __launch_bounds__(256) append_pivot_kernel(const double* __restrict__ l, double* __restrict__ lam, int* __restrict__ info,
                                                           int p, double diag) {
    __shared__ double sh[8];
    double s = 0;
    for (int r = threadIdx.x; r < p; r += 256) s = fma(l[r], l[r], s);
    s = block_sum_256(s, sh);
    if (threadIdx.x == 0) {
        double piv = diag - s;
        if (!(piv > 0.0)) { atomicCAS(info, 0, p + 1); piv = 1.0; }
        double lm = sqrt(piv);
        lam[0] = lm; lam[1] = 1.0 / lm;
    }
}

__global__ void __launch_bounds__(256) append_write_kernel(double* __restrict__ A, double* __restrict__ W, double* __restrict__ Wpack,
                                                           const double* __restrict__ l, const double* __restrict__ u,
                                                           const double* __restrict__ lam, int p, int Np) {
    int c = blockIdx.x * 256 + threadIdx.x;
    if (c > p) return;
    const double lm = lam[0], inv = lam[1];
    const double a = c < p ? l[c] : lm;
    const double w = c < p ? -u[c] * inv : inv;
    A[(size_t)p * Np + c] = a;
    W[(size_t)p * Np + c] = w;
    const int i = p >> 7, r = p & 127;
    Wpack[(wpack_base(i) + (c >> 4)) * (size_t)BLOB + blob_offset(r, c & 15)] = w;
}

// betaY[p] = W[p][:] . Y, beta1[p] = W[p][:] . 1 over the real rows c <= p
__global__ void __launch_bounds__(256) append_beta_kernel(const double* __restrict__ W, const double* __restrict__ Y,
                                                          double* __restrict__ betaY, double* __restrict__ beta1, int p, int Np) {
    __shared__ double sh[8];
    double sy = 0, s1 = 0;
    for (int c = threadIdx.x; c <= p; c += 256) { double w = W[(size_t)p * Np + c]; sy = fma(w, Y[c], sy); s1 += w; }
    sy = block_sum_256(sy, sh);
    s1 = block_sum_256(s1, sh);
    if (threadIdx.x == 0) { betaY[p] = sy; beta1[p] = s1; }
}

// Re-home the model in buffers of NpNew rows (a new 128-row block of identity padding).
static int grow_model_rows(ibo_model* m, int NpNew) {
    cudaStream_t st = m->stream;
    const int Np = m->Np, nbNew = NpNew / TM, d = m->d;
    double *nA = nullptr, *nW = nullptr, *nAo = nullptr, *nXt = nullptr, *nD = nullptr, *nWp = nullptr, *nBY = nullptr, *nB1 = nullptr, *nY = nullptr;
    double** fresh[] = {&nA, &nW, &nAo, &nXt, &nD, &nWp, &nBY, &nB1, &nY};
    auto fail = [&](cudaError_t e, const char* what) {
        set_error(std::string(what) + ": " + cudaGetErrorString(e)); cudaGetLastError();
        for (auto q : fresh) if (*q) pool_free(*q);
        return e == cudaErrorMemoryAllocation ? IBO_E_NOMEM : IBO_E_CUDA;
    };
#define TRYG(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return fail(e__, #expr); } while (0)
    const size_t sq = (size_t)NpNew * NpNew;
    const bool keepAo = m->dAorig && NpNew <= 4096;
    TRYG(pool_malloc((void**)&nA, sizeof(double) * sq));
    TRYG(pool_malloc((void**)&nW, sizeof(double) * sq));
    if (keepAo) TRYG(pool_malloc((void**)&nAo, sizeof(double) * sq));
    TRYG(pool_malloc((void**)&nXt, sizeof(double) * (size_t)NpNew * d));
    TRYG(pool_malloc((void**)&nD, sizeof(double) * (size_t)nbNew * 128 * 128));
    TRYG(pool_malloc((void**)&nWp, sizeof(double) * wpack_base(nbNew) * BLOB));
    TRYG(pool_malloc((void**)&nBY, sizeof(double) * NpNew));
    TRYG(pool_malloc((void**)&nB1, sizeof(double) * NpNew));
    TRYG(pool_malloc((void**)&nY, sizeof(double) * NpNew));
    dim3 g2((NpNew + 255) / 256, NpNew);
    set_identity_kernel<<<g2, 256, 0, st>>>(nA, NpNew);
    set_identity_kernel<<<g2, 256, 0, st>>>(nW, NpNew);
    g_launches += 2;
    const size_t rowB = sizeof(double) * Np, rowBn = sizeof(double) * NpNew;
    TRYG(cudaMemcpy2DAsync(nA, rowBn, m->dA, rowB, rowB, Np, cudaMemcpyDeviceToDevice, st));
    TRYG(cudaMemcpy2DAsync(nW, rowBn, m->dW, rowB, rowB, Np, cudaMemcpyDeviceToDevice, st));
    if (keepAo) {
        set_identity_kernel<<<g2, 256, 0, st>>>(nAo, NpNew);
        g_launches++;
        TRYG(cudaMemcpy2DAsync(nAo, rowBn, m->dAorig, rowB, rowB, Np, cudaMemcpyDeviceToDevice, st));
    }
    TRYG(cudaMemsetAsync(nXt, 0, sizeof(double) * (size_t)NpNew * d, st));
    TRYG(cudaMemcpyAsync(nXt, m->dXt, sizeof(double) * (size_t)Np * d, cudaMemcpyDeviceToDevice, st));
    TRYG(cudaMemsetAsync(nD, 0, sizeof(double) * (size_t)nbNew * 128 * 128, st));
    TRYG(cudaMemcpyAsync(nD, m->dD, sizeof(double) * (size_t)m->nb * 128 * 128, cudaMemcpyDeviceToDevice, st));
    double* vecs[3][2] = {{nBY, m->dBetaY}, {nB1, m->dBeta1}, {nY, m->dY}};
    for (auto& v : vecs) {
        TRYG(cudaMemsetAsync(v[0], 0, sizeof(double) * NpNew, st));
        TRYG(cudaMemcpyAsync(v[0], v[1], sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
    }
    pack_w_kernel<<<dim3(nbNew * KB_PER_BLOCK, nbNew), 256, 0, st>>>(nW, nWp, NpNew, nbNew);
    g_launches++;
    TRYG(cudaStreamSynchronize(st));      // the old blocks go back to the pool: nothing may still read them
    TRYG(cudaGetLastError());
#undef TRYG
    double** old[] = {&m->dA, &m->dW, &m->dAorig, &m->dXt, &m->dD, &m->dWpack, &m->dBetaY, &m->dBeta1, &m->dY};
    double* repl[] = {nA, nW, nAo, nXt, nD, nWp, nBY, nB1, nY};
    for (int q = 0; q < 9; q++) { if (*old[q]) pool_free(*old[q]); *old[q] = repl[q]; }
    m->Np = NpNew; m->nb = nbNew;
    for (auto& kv : m->unitTables) if (kv.second.first) cudaFree(kv.second.first);     // keyed on the old nb
    m->unitTables.clear();
    m->planCache.clear();
    return IBO_OK;
}

int append_rows(ibo_model* m, const double* X, const double* Y, int k, int* info) {
    m->i8Valid = false;      // W changes: the int8 slices are rebuilt on the next use
    const int d = m->d;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    if (m->N + k > m->Np) {
        int rc = grow_model_rows(m, ((m->N + k + TM - 1) / TM) * TM);
        if (rc) return rc;
    }
    const int Np = m->Np;
    int rc = grow(&m->dAppend, &m->appendCap, (size_t)k * d + 3 * (size_t)Np + 2);
    if (rc) return rc;
    double* dXn = m->dAppend;
    double* kvec = dXn + (size_t)k * d;
    double* lvec = kvec + Np;
    double* uvec = lvec + Np;
    double* lam = uvec + Np;
    std::vector<double> xs((size_t)k * d);
    for (int j = 0; j < k; j++)
        for (int t = 0; t < d; t++) xs[(size_t)j * d + t] = X[(size_t)j * d + t] * m->hInvTheta[t] - m->hCenter[t];
    IBO_CUDA_TRY(cudaMemsetAsync(m->dInfo, 0, sizeof(int), st));
    IBO_CUDA_TRY(cudaMemcpyAsync(dXn, xs.data(), sizeof(double) * xs.size(), cudaMemcpyHostToDevice, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(m->dY + m->N, Y, sizeof(double) * k, cudaMemcpyHostToDevice, st));
    const int nblk = (Np + 255) / 256;
    for (int j = 0; j < k; j++) {
        const int p = m->N + j;
        append_kvec_kernel<<<nblk, 256, 0, st>>>(m->dXt, dXn + (size_t)j * d, kvec, m->dAorig, p, Np, d, m->kind, m->sf2, m->noise);
        tri_matvec_kernel<<<(Np + 7) / 8, 256, 0, st>>>(m->dW, kvec, lvec, Np);      // l = W k (rows >= p: identity x 0)
        append_pivot_kernel<<<1, 256, 0, st>>>(lvec, lam, m->dInfo, p, 1.0 + m->noise);
        if (p > 0) append_colsum_kernel<<<(p + 15) / 16, 256, 0, st>>>(m->dW, lvec, uvec, p, Np);
        append_write_kernel<<<(p + 256) / 256, 256, 0, st>>>(m->dA, m->dW, m->dWpack, lvec, uvec, lam, p, Np);
        append_beta_kernel<<<1, 256, 0, st>>>(m->dW, m->dY, m->dBetaY, m->dBeta1, p, Np);
        g_launches += p > 0 ? 6 : 5;
    }
    int hinfo = 0;
    IBO_CUDA_TRY(cudaMemcpyAsync(&hinfo, m->dInfo, sizeof(int), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    IBO_CUDA_TRY(cudaGetLastError());
    m->N += k;
    if (info) *info = hinfo;
    if (hinfo != 0) {
        set_error("appended matrix is not positive definite (pivot " + std::to_string(hinfo) + "); the model is no longer valid");
        return IBO_E_NOTSPD;
    }
    return IBO_OK;
}

// dynamic shared-memory opt-ins of the factorisation kernels (per device: ensure_attrs)
static cudaError_t set_model_attrs() {
    const int tile_smem = TILE_SMEM_DOUBLES * 8;
    cudaError_t e = cudaFuncSetAttribute(block_step_kernel<MODE_TRTRI_SCALE>, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_smem);
    const int half_smem = TileCfg<64>::SMEM_DOUBLES * 8;
    if (e == cudaSuccess) e = cudaFuncSetAttribute(block_step_kernel<MODE_CHOL_PANEL, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, half_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(block_step_kernel<MODE_CHOL_TRAIL, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, half_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(block_step_kernel<MODE_TRTRI_UPDATE, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, half_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(syrk_identity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tile_smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POTRF_SMEM);
    return e;
}
static int set_kernel_attrs() {
    int dev = 0;
    IBO_CUDA_TRY(cudaGetDevice(&dev));
    IBO_CUDA_TRY(ensure_attrs(dev, ATTR_MODEL, set_model_attrs));
    return IBO_OK;
}

// Factorise m->dA in place, produce dW, dD, dWpack, dBetaY, dBeta1.
// from_inverse_reversed: dA holds J invR J; W' = reverse-transpose of its Cholesky factor.
int launch_factorize(ibo_model* m, bool from_inverse_reversed, bool pack) {
    int rc = set_kernel_attrs();
    if (rc) return rc;
    cudaStream_t st = m->stream;
    const int Np = m->Np, nb = m->nb;
    const int tile_smem = TILE_SMEM_DOUBLES * 8, half_smem = TileCfg<64>::SMEM_DOUBLES * 8;
    const int potrf_smem = POTRF_SMEM;
    IBO_CUDA_TRY(cudaMemsetAsync(m->dInfo, 0, sizeof(int), st));
    dim3 g2((Np + 255) / 256, Np);
    // Block columns go in groups of w = 1 or 2.  With w = 2 everything behind the pair (k, k+1) is updated with both columns at
    // once: one pass with a 256-deep product instead of two 128-deep ones halves the read-modify-write traffic of the trailing
    // matrix and the number of launches; it pays from ~48 block columns on (option chol_pair), below that the longer chain of
    // one-tile kernels between two diagonal factorisations costs more than the bulk saves.
    // Look-ahead: the update behind the group is split -- the w nearest block columns stay on the critical stream (they are all
    // the next group's diagonal factorisations and panels wait for), the rest goes to a low-priority bulk stream, so the one-CTA
    // diagonal kernels and thin panels of the next group run while the bulk update still fills the GPU.  Dependencies: bulk(k)
    // reads the panels of the group (evStep) and follows bulk(k-w) in stream order; ahead(k) updates columns bulk(k-w) wrote (evRest).
    // The inversion W = inv(L) is a forward substitution on B = I that follows the factorisation group by group on its own pair
    // of streams, split the same way: rows k..k+w-1 are scaled by D (W_kj = D_k B_kj), the next group's rows are updated on the
    // near stream, all later rows on the far stream (after evScale; near(k) waits for far(k-w) through evFar).
    cudaStream_t s2 = from_inverse_reversed ? st : m->stream2;
    cudaStream_t s4 = m->stream4;
    const bool trtri = !from_inverse_reversed;
    if (trtri) {
        IBO_CUDA_TRY(cudaEventRecord(m->evStep, st));            // orders s2 / s4 after whatever produced dA / dD users
        IBO_CUDA_TRY(cudaStreamWaitEvent(s2, m->evStep, 0));
        IBO_CUDA_TRY(cudaStreamWaitEvent(s4, m->evStep, 0));
        set_identity_kernel<<<g2, 256, 0, s2>>>(m->dW, Np);
        g_launches++;
        IBO_CUDA_TRY(cudaEventRecord(m->evFar, s2));
        IBO_CUDA_TRY(cudaStreamWaitEvent(s4, m->evFar, 0));
    }
    cudaStream_t sb = m->stream3;
    const long pair_opt = get_option(OPT_CHOL_PAIR);
    const int w = (pair_opt < 0 ? nb >= 48 : pair_opt != 0) ? 2 : 1;
#ifdef IBO_I8_TRACE
    struct TlEv { cudaEvent_t e; int k; const char* tag; };
    std::vector<TlEv> tl;
    const bool tl_on = get_option(OPT_DEBUG_PLAN) == 7;
    auto TL = [&](cudaStream_t s, int k, const char* tag) {
        if (!tl_on) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); tl.push_back({e, k, tag});
    };
    TL(st, -1, "start");
#else
#define TL(s, k, tag) do { } while (0)
#endif
    IBO_CUDA_TRY(cudaEventRecord(m->evRest, st));
    IBO_CUDA_TRY(cudaStreamWaitEvent(sb, m->evRest, 0));
    for (int k = 0; k < nb; k += w) {
        // ---- block column k
        potrf_diag_kernel<<<1, 512, potrf_smem, st>>>(m->dA, Np, k, m->dD, m->dInfo);
        g_launches++;
        TL(st, k, "potrf");
        int kl = k;                            // last block column of the group
        if (k + 1 < nb) {
            block_step_kernel<MODE_CHOL_PANEL, 64><<<dim3(nb - 1 - k, 1, 2), 128, half_smem, st>>>(m->dA, nullptr, m->dD, Np, k);
            g_launches++;
            TL(st, k, "panel");
            if (w == 2) {
                // ---- block column k+1: its update by column k, then the same two kernels
                kl = k + 1;
                block_step_kernel<MODE_CHOL_TRAIL, 64><<<dim3(1, nb - 1 - k, 2), 128, half_smem, st>>>(m->dA, nullptr, m->dD, Np, k, 0, k + 1, 128);
                TL(st, k, "first");
                potrf_diag_kernel<<<1, 512, potrf_smem, st>>>(m->dA, Np, kl, m->dD, m->dInfo);
                g_launches += 2;
                TL(st, kl, "potrf");
                if (kl + 1 < nb) {
                    block_step_kernel<MODE_CHOL_PANEL, 64><<<dim3(nb - 1 - kl, 1, 2), 128, half_smem, st>>>(m->dA, nullptr, m->dD, Np, kl);
                    g_launches++;
                    TL(st, kl, "panel");
                }
            }
        }
        const int gw = kl - k + 1;             // columns in this group (1 at the end of an odd count)
        const int nbehind = nb - 1 - kl;       // block rows / columns behind the group
        const int c0 = kl + 1, kspan = 128 * gw;
        IBO_CUDA_TRY(cudaEventRecord(m->evStep, st));
        if (trtri) {
            IBO_CUDA_TRY(cudaStreamWaitEvent(s2, m->evStep, 0));
            block_step_kernel<MODE_TRTRI_SCALE><<<k + 1, 256, tile_smem, s2>>>(m->dA, m->dW, m->dD, Np, k);
            g_launches++;
            if (gw == 2) {
                block_step_kernel<MODE_TRTRI_UPDATE, 64><<<dim3(k + 1, 1, 2), 128, half_smem, s2>>>(m->dA, m->dW, m->dD, Np, k, 0, k + 1, 128);
                block_step_kernel<MODE_TRTRI_SCALE><<<kl + 1, 256, tile_smem, s2>>>(m->dA, m->dW, m->dD, Np, kl);
                g_launches += 2;
            }
            if (nbehind > 0) {
                // rows behind the group take all its block rows in one pass (the block W_(k),(k+1) above the diagonal is zero)
                const int nnear = nbehind < w ? nbehind : w;
                if (nbehind > nnear) {
                    IBO_CUDA_TRY(cudaEventRecord(m->evScale, s2));
                    IBO_CUDA_TRY(cudaStreamWaitEvent(s4, m->evScale, 0));
                    block_step_kernel<MODE_TRTRI_UPDATE, 64><<<dim3(kl + 1, nbehind - nnear, 2), 128, half_smem, s4>>>(m->dA, m->dW, m->dD, Np, k, 0, c0 + nnear, kspan);
                    g_launches++;
                    TL(s4, k, "far");
                }
                IBO_CUDA_TRY(cudaStreamWaitEvent(s2, m->evFar, 0));        // far(k-w) wrote the near rows of this group
                block_step_kernel<MODE_TRTRI_UPDATE, 64><<<dim3(kl + 1, nnear, 2), 128, half_smem, s2>>>(m->dA, m->dW, m->dD, Np, k, 0, c0, kspan);
                g_launches++;
                if (nbehind > nnear) IBO_CUDA_TRY(cudaEventRecord(m->evFar, s4));
            }
            TL(s2, k, "near");
        }
        if (nbehind > 0) {
            // look-ahead columns (they carry the bulk update of the previous group), then the rest in the background
            if (k > 0) IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evRest, 0));
            const int nla = nbehind < w ? nbehind : w;
            block_step_kernel<MODE_CHOL_TRAIL, 64><<<dim3(nla, nbehind, 2), 128, half_smem, st>>>(m->dA, nullptr, m->dD, Np, k, 0, c0, kspan);
            g_launches++;
            TL(st, k, "ahead");
            if (nbehind > nla) {
                IBO_CUDA_TRY(cudaStreamWaitEvent(sb, m->evStep, 0));
                block_step_kernel<MODE_CHOL_TRAIL, 64><<<dim3(nbehind - nla, nbehind, 2), 128, half_smem, sb>>>(m->dA, nullptr, m->dD, Np, k, nla, c0, kspan);
                g_launches++;
                IBO_CUDA_TRY(cudaEventRecord(m->evRest, sb));
                TL(sb, k, "bulk");
            }
        }
    }
#ifdef IBO_I8_TRACE
    if (tl_on) {
        cudaStreamSynchronize(st); cudaStreamSynchronize(sb); cudaStreamSynchronize(s2); cudaStreamSynchronize(s4);
        for (auto& x : tl) {
            float ms = 0; cudaEventElapsedTime(&ms, tl[0].e, x.e);
            fprintf(stderr, "tl k=%d %s %.1f\n", x.k, x.tag, 1e3 * ms);
        }
        for (auto& x : tl) cudaEventDestroy(x.e);
    }
#else
#undef TL
#endif
    IBO_CUDA_TRY(cudaEventRecord(m->evRest, sb));
    IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evRest, 0));
    if (from_inverse_reversed) {
        reverse_transpose_kernel<<<g2, 256, 0, st>>>(m->dW, m->dA, m->N, Np);
        g_launches++;
    } else {
        IBO_CUDA_TRY(cudaEventRecord(m->evStep, s2));
        IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evStep, 0));
        IBO_CUDA_TRY(cudaEventRecord(m->evFar, s4));
        IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evFar, 0));
    }
    if (pack) { pack_w_kernel<<<dim3(nb * KB_PER_BLOCK, nb), 256, 0, st>>>(m->dW, m->dWpack, Np, nb); g_launches++; }
    tri_matvec_kernel<<<(Np + 7) / 8, 256, 0, st>>>(m->dW, m->dY, m->dBetaY, Np);
    g_launches++;
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

// launch wrappers for the other translation units (laplace.cu)
void launch_tri_matvec(const double* T, const double* v, double* out, int Np, cudaStream_t st) {
    tri_matvec_kernel<<<(Np + 7) / 8, 256, 0, st>>>(T, v, out, Np);
    g_launches++;
}
void launch_tri_matvec_t(const double* T, const double* v, double* out, int n, int Np, cudaStream_t st) {
    append_colsum_kernel<<<(n + 15) / 16, 256, 0, st>>>(T, v, out, n, Np);      // out[c] = sum_{r >= c} v[r] T[r][c], c < n
    g_launches++;
}
int launch_syrk_identity(double* C, const double* G, int Np, int K, cudaStream_t st) {
    int rc = set_kernel_attrs();
    if (rc) return rc;
    syrk_identity_kernel<<<dim3(Np / 128, Np / 128), 256, TILE_SMEM_DOUBLES * 8, st>>>(C, G, Np, K);
    g_launches++;
    return IBO_OK;
}

}  // namespace ibo

// =============================================================================================
// C ABI: model lifetime
// =============================================================================================
using namespace ibo;

extern "C" const char* ibo_last_error(void) { return ibo::get_error(); }
extern "C" const char* ibo_version(void) { return "ibo_b200 0.1 (sm_100a)"; }
extern "C" long ibo_launch_count(void) { return ibo::g_launches; }

extern "C" int ibo_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { set_error(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); cudaGetLastError(); return 0; }
    return n;
}

// live models: destroying one that is still attached as another model's variance model detaches it there first
static std::mutex g_live_mu;
static std::set<ibo_model*> g_live;

static void register_model(ibo_model* m) { std::lock_guard<std::mutex> lk(g_live_mu); g_live.insert(m); }

static void free_model(ibo_model* m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(g_live_mu);
        g_live.erase(m);
        for (ibo_model* o : g_live) if (o->var_model == m) o->var_model = nullptr;
    }
    cudaSetDevice(m->device);
    tiny_server_stop(m);
    if (m->hServer) pinned_put(m->hServer);
    if (m->dSrvCount) cudaFree(m->dSrvCount);
    if (m->stream2) cudaStreamSynchronize(m->stream2);
    if (m->stream3) cudaStreamSynchronize(m->stream3);
    if (m->stream4) cudaStreamSynchronize(m->stream4);
    if (m->stream) cudaStreamSynchronize(m->stream);   // blocks go back to the pool: nothing may still be using them
    double** ptrs[] = {&m->dXt, &m->dInvTheta, &m->dCenter, &m->dA, &m->dAorig, &m->dW, &m->dD, &m->dWpack, &m->dBetaY, &m->dBeta1, &m->dY,
                       &m->dPmeans, &m->dPbeta, &m->dPlb, &m->dPwidth, &m->dCand, &m->dSlab, &m->dPart, &m->dOut, &m->dBlkBest, &m->dBest, &m->dAppend,
                       &m->dWi8s, &m->dRowScale, &m->dAlphaY, &m->dAlpha1, &m->dGuard, &m->dGuardList, &m->dCinv};
    for (auto p : ptrs) if (*p) { pool_free(*p); *p = nullptr; }
    if (m->dInfo) cudaFree(m->dInfo);
    if (m->dBlkIdx) cudaFree(m->dBlkIdx);
    if (m->dBestIdx) cudaFree(m->dBestIdx);
    for (auto& kv : m->unitTables) if (kv.second.first) cudaFree(kv.second.first);
    m->unitTables.clear();
    if (m->hPinned) pinned_put(m->hPinned);
    for (auto& e : m->ev) if (e) cudaEventDestroy(e);
    if (m->evStep) cudaEventDestroy(m->evStep);
    if (m->evRest) cudaEventDestroy(m->evRest);
    if (m->stream3) cudaStreamDestroy(m->stream3);
    if (m->evScale) cudaEventDestroy(m->evScale);
    if (m->evFar) cudaEventDestroy(m->evFar);
    if (m->stream4) cudaStreamDestroy(m->stream4);
    for (auto& e : m->evI8) if (e) cudaEventDestroy(e);
    for (auto& e : m->evCopy) if (e) cudaEventDestroy(e);
    if (m->stream2) cudaStreamDestroy(m->stream2);
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
}

static int theta_and_sf2(int kind, const double* hyper, int nhyper, int d, bool clip_ard, std::vector<double>& theta, double* sf2) {
    theta.assign(d, 1.0);
    *sf2 = 1.0;
    bool ard = (kind == IBO_KERNEL_SE_ARD || kind == IBO_KERNEL_MATERN5_ARD);
    if (ard) {
        if (nhyper < d) { set_error("ARD kernel needs at least d hyperparameters"); return IBO_E_BADARG; }
        for (int j = 0; j < d; j++) {
            double t = hyper[j];
            if (kind == IBO_KERNEL_SE_ARD && clip_ard) t = fmin(fmax(t, 1e-4), 1e4);   // kernel.py:141
            theta[j] = t;
        }
        if (nhyper > d) *sf2 = exp(2.0 * log(hyper[d]));                                // kernel.py:63
    } else {
        if (nhyper < 1) { set_error("isotropic kernel needs theta"); return IBO_E_BADARG; }
        for (int j = 0; j < d; j++) theta[j] = hyper[0];
        if (kind != IBO_KERNEL_SE_ISO && nhyper > 1) *sf2 = exp(2.0 * log(hyper[1]));   // kernel.py:203-204,242-243
    }
    return IBO_OK;
}

// diag < 0: the GP's own diagonal 1 + noise; otherwise the value to put on the diagonal of A (marginal likelihood:
// covMatrix(X) + noise I has sf2 + noise there).
// the Laplace term given as preference pairs: inv(C) is formed on the device (Cholesky of C, triangular inverse, Gram product)
struct PrefPairs { int P; const int* a; const int* b; const double* w; double cdiag; const double* denseC; };   // denseC: C itself, N x N (host)

static int create_common(int device, int kind, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
                         double noise, double diag, const double* Cinv, const double* invR, double sf2_override, bool legacy,
                         int npb, const double* pmeans, const double* pbeta, double ptheta, const double* plb, const double* pwidth,
                         ibo_model** out, int* info, const PrefPairs* pref = nullptr) {
    if (info) *info = 0;
    if (!out || !X || !Y || !hyper || N < 1 || d < 1 || kind < 0 || kind > IBO_KERNEL_MATERN5_ARD) { set_error("bad argument"); return IBO_E_BADARG; }
    if (npb > 0 && (!pmeans || !pbeta || !plb || !pwidth)) { set_error("prior arrays missing"); return IBO_E_BADARG; }
    *out = nullptr;
    int ndev = ibo_device_count();
    if (ndev <= 0) { set_error("no CUDA device available (libibo_b200 has no CPU fallback)"); return IBO_E_CUDA; }
    if (device < 0 || device >= ndev) { set_error("bad device ordinal"); return IBO_E_BADARG; }
    std::vector<double> theta; double sf2;
    int rc = theta_and_sf2(kind, hyper, nhyper, d, !legacy, theta, &sf2);
    if (rc) return rc;
    if (legacy) sf2 = sf2_override;
    IBO_CUDA_TRY(cudaSetDevice(device));
    ibo_model* m = new ibo_model();
    m->device = device; m->N = N; m->d = d; m->kind = kind; m->noise = noise; m->sf2 = sf2;
    m->nb = (N + TM - 1) / TM; m->Np = m->nb * TM;
    m->npb = npb > 0 ? npb : 0; m->ptheta = ptheta; m->cpp_prior = legacy;
    const int Np = m->Np, nb = m->nb;
    auto fail = [&](int code) { free_model(m); return code; };
#define TRYM(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) { set_error(std::string(#expr) + ": " + cudaGetErrorString(e__)); cudaGetLastError(); return fail(e__ == cudaErrorMemoryAllocation ? IBO_E_NOMEM : IBO_E_CUDA); } } while (0)
    // main stream at the highest priority, the helper stream at the lowest: on the INT8 path K1 of the next chunk (stream2) fills
    // the SM resources the resident K2 CTAs (main stream) leave free, and must never keep a K2 CTA waiting for a slot
    int prLo = 0, prHi = 0;
    TRYM(cudaDeviceGetStreamPriorityRange(&prLo, &prHi));
    TRYM(cudaStreamCreateWithPriority(&m->stream, cudaStreamNonBlocking, prHi));
    TRYM(cudaStreamCreateWithPriority(&m->stream2, cudaStreamNonBlocking, prLo));
    TRYM(cudaStreamCreateWithPriority(&m->stream3, cudaStreamNonBlocking, prLo));
    TRYM(cudaStreamCreateWithPriority(&m->stream4, cudaStreamNonBlocking, prLo));
    TRYM(cudaEventCreateWithFlags(&m->evRest, cudaEventDisableTiming));
    TRYM(cudaEventCreateWithFlags(&m->evStep, cudaEventDisableTiming));
    TRYM(cudaEventCreateWithFlags(&m->evScale, cudaEventDisableTiming));
    TRYM(cudaEventCreateWithFlags(&m->evFar, cudaEventDisableTiming));
    for (auto& e : m->ev) TRYM(cudaEventCreate(&e));
    TRYM(pool_malloc((void**)&m->dXt, sizeof(double) * (size_t)Np * d));
    TRYM(pool_malloc((void**)&m->dInvTheta, sizeof(double) * d));
    TRYM(pool_malloc((void**)&m->dCenter, sizeof(double) * d));
    TRYM(pool_malloc((void**)&m->dA, sizeof(double) * (size_t)Np * Np));
    TRYM(pool_malloc((void**)&m->dW, sizeof(double) * (size_t)Np * Np));
    TRYM(pool_malloc((void**)&m->dD, sizeof(double) * (size_t)nb * 128 * 128));
    TRYM(pool_malloc((void**)&m->dWpack, sizeof(double) * wpack_base(nb) * BLOB));
    TRYM(pool_malloc((void**)&m->dBetaY, sizeof(double) * Np));
    TRYM(pool_malloc((void**)&m->dBeta1, sizeof(double) * Np));
    TRYM(pool_malloc((void**)&m->dY, sizeof(double) * Np));
    TRYM(cudaMalloc(&m->dInfo, sizeof(int)));
    TRYM(pool_malloc((void**)&m->dBest, sizeof(double)));
    TRYM(cudaMalloc(&m->dBestIdx, sizeof(long long)));
    cudaStream_t st = m->stream;
    // scaled inputs, zero padded
    std::vector<double> xt((size_t)Np * d, 0.0), it(d), yp(Np, 0.0), ones(Np, 0.0);
    // scaled inputs x * (1/theta), centred on their mean: distances are translation invariant, and centring keeps
    // |x|^2 small for the |x|^2 + |y|^2 - 2 x.y expansion of K1 (candidates get the same scale and shift there)
    std::vector<double> ctr(d, 0.0);
    for (int j = 0; j < d; j++) it[j] = 1.0 / theta[j];
    for (int i = 0; i < N; i++)
        for (int j = 0; j < d; j++) ctr[j] += X[(size_t)i * d + j] * it[j];
    for (int j = 0; j < d; j++) ctr[j] /= N;
    for (int i = 0; i < N; i++) {
        for (int j = 0; j < d; j++) xt[(size_t)i * d + j] = X[(size_t)i * d + j] * it[j] - ctr[j];
        yp[i] = Y[i]; ones[i] = 1.0;
    }
    m->hInvTheta = it; m->hCenter = ctr; m->has_cinv = (Cinv != nullptr || pref != nullptr); m->from_inverse = (invR != nullptr);
    TRYM(cudaMemcpyAsync(m->dXt, xt.data(), sizeof(double) * xt.size(), cudaMemcpyHostToDevice, st));
    TRYM(cudaMemcpyAsync(m->dInvTheta, it.data(), sizeof(double) * d, cudaMemcpyHostToDevice, st));
    TRYM(cudaMemcpyAsync(m->dCenter, ctr.data(), sizeof(double) * d, cudaMemcpyHostToDevice, st));
    TRYM(cudaMemcpyAsync(m->dY, yp.data(), sizeof(double) * Np, cudaMemcpyHostToDevice, st));
    if (m->npb > 0) {
        TRYM(pool_malloc((void**)&m->dPmeans, sizeof(double) * (size_t)npb * d));
        TRYM(pool_malloc((void**)&m->dPbeta, sizeof(double) * npb));
        TRYM(pool_malloc((void**)&m->dPlb, sizeof(double) * d));
        TRYM(pool_malloc((void**)&m->dPwidth, sizeof(double) * d));
        TRYM(cudaMemcpyAsync(m->dPmeans, pmeans, sizeof(double) * (size_t)npb * d, cudaMemcpyHostToDevice, st));
        TRYM(cudaMemcpyAsync(m->dPbeta, pbeta, sizeof(double) * npb, cudaMemcpyHostToDevice, st));
        TRYM(cudaMemcpyAsync(m->dPlb, plb, sizeof(double) * d, cudaMemcpyHostToDevice, st));
        TRYM(cudaMemcpyAsync(m->dPwidth, pwidth, sizeof(double) * d, cudaMemcpyHostToDevice, st));
    }
    dim3 g2((Np + 255) / 256, Np);
    double* dTmp = nullptr;
    if (invR) {
        TRYM(pool_malloc((void**)&dTmp, sizeof(double) * (size_t)N * N));
        TRYM(cudaMemcpyAsync(dTmp, invR, sizeof(double) * (size_t)N * N, cudaMemcpyHostToDevice, st));
        build_reversed_kernel<<<g2, 256, 0, st>>>(m->dA, dTmp, N, Np);
    } else {
        if (Cinv) {
            TRYM(pool_malloc((void**)&dTmp, sizeof(double) * (size_t)N * N));
            TRYM(cudaMemcpyAsync(dTmp, Cinv, sizeof(double) * (size_t)N * N, cudaMemcpyHostToDevice, st));
        }
        if (pref) {
            // inv(C) without leaving the device: C -> dA, C = Lc Lc^T, Wc = inv(Lc) (the model's own factorisation kernels),
            // inv(C) = Wc^T Wc (DMMA Gram product, lower tiles); then A = R + inv(C) is built in place and factorised as usual
            int* dPairs = nullptr; double* dWts = nullptr;
            if (pref->denseC) {
                TRYM(pool_malloc((void**)&dWts, sizeof(double) * (size_t)N * N));
                TRYM(cudaMemcpyAsync(dWts, pref->denseC, sizeof(double) * (size_t)N * N, cudaMemcpyHostToDevice, st));
                pad_copy_kernel<<<dim3((Np + 255) / 256, Np), 256, 0, st>>>(m->dA, dWts, N, Np);
            } else {
                TRYM(pool_malloc((void**)&dPairs, sizeof(int) * 2 * (size_t)std::max(pref->P, 1)));
                TRYM(pool_malloc((void**)&dWts, sizeof(double) * (size_t)std::max(pref->P, 1)));
                if (pref->P > 0) {
                    TRYM(cudaMemcpyAsync(dPairs, pref->a, sizeof(int) * pref->P, cudaMemcpyHostToDevice, st));
                    TRYM(cudaMemcpyAsync(dPairs + pref->P, pref->b, sizeof(int) * pref->P, cudaMemcpyHostToDevice, st));
                    TRYM(cudaMemcpyAsync(dWts, pref->w, sizeof(double) * pref->P, cudaMemcpyHostToDevice, st));
                }
                pref_build_C_kernel<<<(Np + 127) / 128, 128, 0, st>>>(m->dA, N, Np, pref->P, dPairs, dPairs + pref->P, dWts, pref->cdiag);
            }
            g_launches++;
            rc = launch_factorize(m, false, false);
            int cinfo = 0;
            if (!rc) {
                TRYM(cudaMemcpyAsync(&cinfo, m->dInfo, sizeof(int), cudaMemcpyDeviceToHost, st));
                TRYM(cudaStreamSynchronize(st));
            }
            if (dPairs) pool_free(dPairs);
            pool_free(dWts);
            if (rc) return fail(rc);
            if (cinfo != 0) {
                if (info) *info = cinfo;
                set_error("the Laplace matrix C is not positive definite (pivot " + std::to_string(cinfo) + ")");
                return fail(IBO_E_NOTSPD);
            }
            TRYM(pool_malloc((void**)&m->dCinv, sizeof(double) * (size_t)Np * Np));
            TRYM(cudaMemsetAsync(m->dCinv, 0, sizeof(double) * (size_t)Np * Np, st));
            if ((rc = launch_gram_wtw(m->dCinv, m, st))) return fail(rc);
            TRYM(cudaMemsetAsync(m->dInfo, 0, sizeof(int), st));
        }
        build_A_kernel<<<g2, 256, 0, st>>>(m->dA, m->dXt, dTmp, N, Np, d, kind, sf2, diag < 0 ? 1.0 + noise : diag);
        if (pref) { add_symmetric_lower_kernel<<<dim3((N + 255) / 256, N), 256, 0, st>>>(m->dA, m->dCinv, N, Np); g_launches++; }
    }
    g_launches++;
    if (Np <= 4096 && !invR) {   // keep A for get_matrix(0)
        TRYM(pool_malloc((void**)&m->dAorig, sizeof(double) * (size_t)Np * Np));
        TRYM(cudaMemcpyAsync(m->dAorig, m->dA, sizeof(double) * (size_t)Np * Np, cudaMemcpyDeviceToDevice, st));
    }
    rc = launch_factorize(m, invR != nullptr, true);
    if (rc) { if (dTmp) pool_free(dTmp); return fail(rc); }
    // beta1 = W 1 (prior-mean correction term)
    TRYM(cudaMemcpyAsync(m->dBeta1, ones.data(), sizeof(double) * Np, cudaMemcpyHostToDevice, st));
    {
        double* dOnes = nullptr;
        TRYM(pool_malloc((void**)&dOnes, sizeof(double) * Np));
        TRYM(cudaMemcpyAsync(dOnes, m->dBeta1, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
        tri_matvec_kernel<<<(Np + 7) / 8, 256, 0, st>>>(m->dW, dOnes, m->dBeta1, Np);
        g_launches++;
        TRYM(cudaStreamSynchronize(st));
        pool_free(dOnes);
    }
    int hinfo = 0;
    TRYM(cudaMemcpy(&hinfo, m->dInfo, sizeof(int), cudaMemcpyDeviceToHost));
    if (dTmp) pool_free(dTmp);
    TRYM(cudaGetLastError());
    if (hinfo != 0) {
        if (info) *info = hinfo;
        set_error("matrix is not positive definite (pivot " + std::to_string(hinfo) + ")");
        return fail(IBO_E_NOTSPD);
    }
#undef TRYM
    register_model(m);
    *out = m;
    return IBO_OK;
}

extern "C" int ibo_model_create(int device, int kerneltype, const double* hyper, int nhyper, const double* X, const double* Y,
                                int N, int d, double noise, const double* Cinv, int npbases, const double* pmeans,
                                const double* pbeta, double ptheta, const double* plowerb, const double* pwidth,
                                ibo_model** out, int* info) {
    return create_common(device, kerneltype, hyper, nhyper, X, Y, N, d, noise, -1.0, Cinv, nullptr, 1.0, false,
                         npbases, pmeans, pbeta, ptheta, plowerb, pwidth, out, info);
}

extern "C" int ibo_model_create_pref(int device, int kerneltype, const double* hyper, int nhyper, const double* X, const double* Y,
                                     int N, int d, double noise, int P, const int* pa, const int* pb, const double* w, double cdiag,
                                     ibo_model** out, int* info) {
    if (P < 0 || (P > 0 && (!pa || !pb || !w)) || !(cdiag > 0)) { set_error("bad argument"); return IBO_E_BADARG; }
    for (int p = 0; p < P; p++)
        if (pa[p] < 0 || pa[p] >= N || pb[p] < 0 || pb[p] >= N) { set_error("preference index out of range"); return IBO_E_BADARG; }
    PrefPairs pr{P, pa, pb, w, cdiag, nullptr};
    return create_common(device, kerneltype, hyper, nhyper, X, Y, N, d, noise, -1.0, nullptr, nullptr, 1.0, false,
                         0, nullptr, nullptr, 0.0, nullptr, nullptr, out, info, &pr);
}

extern "C" int ibo_model_create_laplace(int device, int kerneltype, const double* hyper, int nhyper, const double* X, const double* Y,
                                        int N, int d, double noise, const double* C, ibo_model** out, int* info) {
    if (!C) { set_error("C is NULL"); return IBO_E_BADARG; }
    PrefPairs pr{0, nullptr, nullptr, nullptr, 1.0, C};
    return create_common(device, kerneltype, hyper, nhyper, X, Y, N, d, noise, -1.0, nullptr, nullptr, 1.0, false,
                         0, nullptr, nullptr, 0.0, nullptr, nullptr, out, info, &pr);
}

extern "C" int ibo_model_create_from_inverse(int device, int kerneltype, const double* hyper, int nhyper, const double* X,
                                             const double* Y, int N, int d, double noise, const double* invR, double sf2,
                                             int npbases, const double* pmeans, const double* pbeta, double ptheta,
                                             const double* plowerb, const double* pwidth, ibo_model** out, int* info) {
    if (!invR) { set_error("invR is NULL"); return IBO_E_BADARG; }
    return create_common(device, kerneltype, hyper, nhyper, X, Y, N, d, noise, -1.0, nullptr, invR, sf2, true,
                         npbases, pmeans, pbeta, ptheta, plowerb, pwidth, out, info);
}

namespace ibo {
int create_model_with_diag(int device, int kind, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
                           double noise, double diag, ibo_model** out, int* info) {
    return create_common(device, kind, hyper, nhyper, X, Y, N, d, noise, diag, nullptr, nullptr, 1.0, false,
                         0, nullptr, nullptr, 0.0, nullptr, nullptr, out, info);
}
}  // namespace ibo

extern "C" int ibo_model_append(ibo_model* m, const double* X, const double* Y, int k, int* info) {
    if (info) *info = 0;
    if (!m || !X || !Y || k < 1) { set_error("bad argument"); return IBO_E_BADARG; }
    if (m->cpp_prior || m->has_cinv || m->var_model) {
        set_error("append needs a plain R model (no explicit inverse, no Laplace term, no variance model)");
        return IBO_E_BADARG;
    }
    return ibo::append_rows(m, X, Y, k, info);
}

extern "C" int ibo_model_destroy(ibo_model* m) { free_model(m); return IBO_OK; }
extern "C" int ibo_model_n(const ibo_model* m) { return m ? m->N : IBO_E_BADARG; }
extern "C" int ibo_model_last_guarded(const ibo_model* m) { return m ? m->lastGuarded : IBO_E_BADARG; }
extern "C" int ibo_model_dim(const ibo_model* m) { return m ? m->d : IBO_E_BADARG; }

extern "C" int ibo_model_set_variance_model(ibo_model* m, ibo_model* aug) {
    if (!m) { set_error("null model"); return IBO_E_BADARG; }
    if (aug && (aug->d != m->d || aug->device != m->device)) { set_error("variance model must share dim and device"); return IBO_E_BADARG; }
    m->var_model = aug;
    return IBO_OK;
}

extern "C" int ibo_model_get_matrix(ibo_model* m, int which, double* out) {
    if (!m || !out || which < 0 || which > 3) { set_error("bad argument"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    const double* src = which == 0 ? m->dAorig : (which == 1 ? m->dA : (which == 2 ? m->dW : m->dCinv));
    if (!src) { set_error("matrix not retained for this model"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaStreamSynchronize(m->stream));
    IBO_CUDA_TRY(cudaMemcpy2D(out, sizeof(double) * m->N, src, sizeof(double) * m->Np, sizeof(double) * m->N, m->N, cudaMemcpyDeviceToHost));
    if (which == 1)
        for (int i = 0; i < m->N; i++)
            for (int j = i + 1; j < m->N; j++) out[(size_t)i * m->N + j] = 0.0;
    if (which == 3)          // the device keeps the lower tiles of the symmetric inv(C)
        for (int i = 0; i < m->N; i++)
            for (int j = i + 1; j < m->N; j++) out[(size_t)i * m->N + j] = out[(size_t)j * m->N + i];
    return IBO_OK;
}

#ifdef IBO_I8_TRACE
// debug build only: the diagonal-block kernel alone on a 128 x 128 SPD block; us = min over 20 launches, stamps = clock64 timeline
extern "C" int ibo_debug_potrf(int device, long long* stamps72, double* us) {
    using namespace ibo;
    IBO_CUDA_TRY(cudaSetDevice(device));
    int rc = set_kernel_attrs();
    if (rc) return rc;
    std::vector<double> h(128 * 128);
    unsigned s = 12345u;
    for (int r = 0; r < 128; r++)
        for (int c = 0; c <= r; c++) {
            s = s * 1664525u + 1013904223u;
            double v = (double)(s >> 8) / (double)(1u << 24) - 0.5;
            h[r * 128 + c] = h[c * 128 + r] = (r == c) ? 40.0 + v : v;
        }
    double *dA0, *dA, *dD; int* dInfo;
    IBO_CUDA_TRY(cudaMalloc(&dA0, sizeof(double) * 128 * 128));
    IBO_CUDA_TRY(cudaMalloc(&dA, sizeof(double) * 128 * 128));
    IBO_CUDA_TRY(cudaMalloc(&dD, sizeof(double) * 128 * 128));
    IBO_CUDA_TRY(cudaMalloc(&dInfo, sizeof(int)));
    IBO_CUDA_TRY(cudaMemset(dInfo, 0, sizeof(int)));
    IBO_CUDA_TRY(cudaMemcpy(dA0, h.data(), sizeof(double) * 128 * 128, cudaMemcpyHostToDevice));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int it = 0; it < 20; it++) {
        IBO_CUDA_TRY(cudaMemcpy(dA, dA0, sizeof(double) * 128 * 128, cudaMemcpyDeviceToDevice));
        cudaEventRecord(e0);
        potrf_diag_kernel<<<1, 512, POTRF_SMEM>>>(dA, 128, 0, dD, dInfo);
        cudaEventRecord(e1);
        IBO_CUDA_TRY(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    *us = 1e3 * best;
    IBO_CUDA_TRY(cudaMemcpyFromSymbol(stamps72, g_potrf_stamp, sizeof(long long) * 72));
    cudaFree(dA0); cudaFree(dA); cudaFree(dD); cudaFree(dInfo);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return IBO_OK;
}
#endif
