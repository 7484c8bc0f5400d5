// The acquisition hot path on B200:
//   K1  kstar_kernel    fused cross-covariance K* = k(X, X*) written as fragment-packed blobs
//   K2  trigemm_kernel  V = W K* (W = inv(L), lower triangular) on the FP64 tensor pipe with
//                       1-D bulk-TMA (UBLKCP) staged operand blobs and an mbarrier pipeline; V is
//                       never stored -- each 128x128 block is reduced in registers to
//                       sum_i V_i^2, sum_i V_i betaY_i, sum_i V_i beta1_i per candidate
//   K3  epilogue_kernel mu, sigma^2 (clipped), EI / PI / UCB, block argmax
//   K4  argmax_final    lowest-index-wins reduction of the block winners
//
// Replaces (reference file:line): GaussianProcess.posterior (ego/gaussianprocess/__init__.py:169-228),
// EI/PI/UCB.negf (ego/acquisition/__init__.py:60-75,100-114,138-164), GP_Maximizer::posterior / aMb /
// negei / negpi / negucb (cpp/optimizeGP.cpp:57-236) and RBFNMeanPrior.mu (ego/gaussianprocess/prior.py:60-66).
//
// Determinism: the value computed for a candidate depends only on (model, x): every reduction has a
// fixed order that is independent of the batch size, of the candidate's position in the batch and of
// how row-blocks are grouped over CTAs (per-row-block partials are summed in ascending order by K3).
#include "model.cuh"
#include "scoremath.cuh"
#include <cmath>
#include <algorithm>
#include <mutex>
#include <queue>
#include <functional>
#include <cstdlib>
#include <cstring>

namespace ibo {

// n-tiles (8 candidates) of tile T that hold at least one real candidate: the last tile of a small batch computes only
// those (a 24-candidate DIRECT batch evaluates 3 of the 16 n-tiles); the rest of the slab tile keeps stale values that
// only reach the partial sums of candidates >= M, which K3 never reads (candidate columns are independent in K2).
__device__ __forceinline__ int valid_ntiles(long M, long m0, int T) {
    long left = M - m0 - (long)T * 128;
    return left >= 128 ? 16 : (int)((left + 7) >> 3);
}

// ---------------------------------------------------------------------------------------------
// K1: one CTA = (candidate tile T, training row-block i); warp w produces k-blob i*8+w.
// Thread (lane) owns candidate n8 = lane/4 of each 8-wide n-tile and training rows k4, k4+4 of each
// 8-row group -- exactly the two values of its 16-byte slot in the packed B-operand layout.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kstar_kernel(const double* __restrict__ Xt, const double* __restrict__ cand,
                                                    const double* __restrict__ inv_theta, const double* __restrict__ center,
                                                    double* __restrict__ slab,
                                                    int N, int d, int nb, long M, long m0, int kind, double sf2) {
    extern __shared__ double sm[];
    const int S = d | 1;
    double* sX = sm;              // [128][S] scaled training rows of block i
    double* sC = sm + 128 * S;    // [128][S] scaled candidates of tile T
    const int T = blockIdx.x, i = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    for (int idx = tid; idx < 128 * d; idx += 256) {
        int r = idx / d, j = idx - r * d;
        sX[r * S + j] = Xt[(size_t)(i * 128 + r) * d + j];
        long c = m0 + (long)T * 128 + r;
        if (c >= M) c = M - 1;
        sC[r * S + j] = cand[(size_t)c * d + j] * inv_theta[j] - center[j];
    }
    __syncthreads();
    const int n8 = lane >> 2, k4 = lane & 3;
    double* blob = slab + ((size_t)T * (nb * KB_PER_BLOCK) + (size_t)i * KB_PER_BLOCK + w) * BLOB;
    const int rowbase = i * 128 + w * 16;
    const int ntv = valid_ntiles(M, m0, T);
#pragma unroll 1
    for (int ks2 = 0; ks2 < 2; ks2++) {
        const int ka = w * 16 + ks2 * 8 + k4, kb = ka + 4;
        const double* xa = sX + ka * S;
        const double* xb = sX + kb * S;
        const bool va = (rowbase + ks2 * 8 + k4) < N, vb = (rowbase + ks2 * 8 + k4 + 4) < N;
#pragma unroll 2
        for (int nt = 0; nt < ntv; nt++) {
            const double* c = sC + (nt * 8 + n8) * S;
            double ra = 0, rb = 0;
            for (int j = 0; j < d; j++) {
                double cj = c[j];
                double da = xa[j] - cj, db = xb[j] - cj;
                ra = fma(da, da, ra);
                rb = fma(db, db, rb);
            }
            double2 v;
            v.x = va ? cov_r2(kind, sf2, ra) : 0.0;
            v.y = vb ? cov_r2(kind, sf2, rb) : 0.0;
            reinterpret_cast<double2*>(blob)[(nt * 2 + ks2) * 32 + lane] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K1 (tensor-pipe form): the squared distance through |x|^2 + |y|^2 - 2 x.y with the cross term X* X^T as
// DMMA.8x8x4 GEMMs over the (zero-padded, centred, 1/theta-scaled) input dimensions, exp / Matern epilogue in
// registers.  The MMA's column order is permuted (column c <-> training row (c>>1) + 4(c&1) of the 8-row group)
// so that the accumulator fragment a lane receives -- C[cand = lane/4][cols 2(lane%4), 2(lane%4)+1] -- is exactly
// the (k4, k4+4) pair of its 16-byte slot in the packed B-operand blob: no shuffle, no shared-memory transpose.
// Cancellation guard: the expansion's absolute error is ~6 eps (|x|^2 + |y|^2); inputs are centred on the training
// mean, and any pair with |x|^2 + |y|^2 > EXPAND_LIMIT is recomputed from direct differences in the same thread.
// ---------------------------------------------------------------------------------------------
constexpr double EXPAND_LIMIT = 256.0;    // => relative error of k below ~2e-13

template <int DP4, int KC>   // DP4: number of 4-wide dimension groups, d <= 4*DP4; KC: kernel class (cov_r2_t)
__global__ void __launch_bounds__(256) kstar_mma_kernel(const double* __restrict__ Xt, const double* __restrict__ cand_dev,
                                                        const double* __restrict__ inv_theta, const double* __restrict__ center,
                                                        double* __restrict__ slab, int N, int d, int nb, long M, long m0,
                                                        int kind, double sf2, const __grid_constant__ CandInline inl) {
    const double* __restrict__ cand = cand_dev ? cand_dev : inl.x;      // small batches ride in the parameter buffer
    constexpr int DP = 4 * DP4;
    constexpr int S = (DP % 16 == 4 || DP % 16 == 12) ? DP : DP + 4;   // (row*S + k) mod 16 distinct over a half-warp
    extern __shared__ double sm[];
    double* sX = sm;                  // [128][S] scaled, centred training rows of block i (zero padded dims)
    double* sC = sX + 128 * S;        // [128][S] scaled, centred candidates of tile T
    double* sXn = sC + 128 * S;       // [128] squared norms
    double* sCn = sXn + 128;
    const int T = blockIdx.x, i = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    for (int idx = tid; idx < 128 * DP; idx += 256) {
        int r = idx / DP, j = idx - r * DP;
        double xv = 0.0, cv = 0.0;
        if (j < d) {
            xv = Xt[(size_t)(i * 128 + r) * d + j];
            long c = m0 + (long)T * 128 + r;
            if (c >= M) c = M - 1;
            cv = cand[(size_t)c * d + j] * inv_theta[j] - center[j];
        }
        sX[r * S + j] = xv;
        sC[r * S + j] = cv;
    }
    __syncthreads();
    if (tid < 128) {
        double a = 0, b = 0;
        for (int j = 0; j < d; j++) { double x = sX[tid * S + j], c = sC[tid * S + j]; a = fma(x, x, a); b = fma(c, c, b); }
        sXn[tid] = a; sCn[tid] = b;
    }
    __syncthreads();
    const int n8 = lane >> 2, k4 = lane & 3;
    const int rowmap = (n8 >> 1) + 4 * (n8 & 1);           // training row (within an 8-row group) fed to MMA column n8
    double* blob = slab + ((size_t)T * (nb * KB_PER_BLOCK) + (size_t)i * KB_PER_BLOCK + w) * BLOB;
    const int rowbase = i * 128 + w * 16;
    double bfr[2][DP4], yn[2][2];
    bool valid[2][2];
#pragma unroll
    for (int ks2 = 0; ks2 < 2; ks2++) {
#pragma unroll
        for (int s4 = 0; s4 < DP4; s4++) bfr[ks2][s4] = sX[(w * 16 + ks2 * 8 + rowmap) * S + 4 * s4 + k4];
        yn[ks2][0] = sXn[w * 16 + ks2 * 8 + k4];
        yn[ks2][1] = sXn[w * 16 + ks2 * 8 + k4 + 4];
        valid[ks2][0] = (rowbase + ks2 * 8 + k4) < N;
        valid[ks2][1] = (rowbase + ks2 * 8 + k4 + 4) < N;
    }
    // small batches split the 16 n-tiles of a candidate tile over gridDim.z CTAs (4x the CTAs, a quarter of the dependent
    // exp chain each): K1 of a 162-point DIRECT batch at N = 4096 otherwise runs 64 CTAs of 64 exps per thread
    const int ntPer = 16 / (int)gridDim.z;
    const int ntv = min(valid_ntiles(M, m0, T), ((int)blockIdx.z + 1) * ntPer);
#pragma unroll 2
    for (int nt = (int)blockIdx.z * ntPer; nt < ntv; nt++) {
        double afr[DP4];
#pragma unroll
        for (int s4 = 0; s4 < DP4; s4++) afr[s4] = sC[(nt * 8 + n8) * S + 4 * s4 + k4];
        const double xn = sCn[nt * 8 + n8];
#pragma unroll
        for (int ks2 = 0; ks2 < 2; ks2++) {
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int s4 = 0; s4 < DP4; s4++) dmma884(c0, c1, afr[s4], bfr[ks2][s4]);
            double r0 = fma(-2.0, c0, xn + yn[ks2][0]);
            double r1 = fma(-2.0, c1, xn + yn[ks2][1]);
            if (xn + fmax(yn[ks2][0], yn[ks2][1]) > EXPAND_LIMIT) {
                // rare: badly scaled inputs -- direct differences for this pair
                const double* c = sC + (nt * 8 + n8) * S;
                const double* xa = sX + (w * 16 + ks2 * 8 + k4) * S;
                const double* xb = xa + 4 * S;
                r0 = 0; r1 = 0;
                for (int j = 0; j < d; j++) {
                    double da = xa[j] - c[j], db = xb[j] - c[j];
                    r0 = fma(da, da, r0); r1 = fma(db, db, r1);
                }
            }
            double2 v;
            v.x = valid[ks2][0] ? cov_r2_t<KC>(sf2, fmax(r0, 0.0)) : 0.0;
            v.y = valid[ks2][1] ? cov_r2_t<KC>(sf2, fmax(r1, 0.0)) : 0.0;
            reinterpret_cast<double2*>(blob)[(nt * 2 + ks2) * 32 + lane] = v;
        }
    }
    // Small batches launch K2 programmatically: it may be scheduled once every CTA of this grid is here.  (Triggering at the
    // top instead lets K2's CTAs occupy SMs this grid still needs -- measured: a 162-point batch at N = 4096 went 181 -> 274 us.)
    pdl_launch_dependents();
}

// ---------------------------------------------------------------------------------------------
// K2: triangular GEMM + fused reduction.
// ---------------------------------------------------------------------------------------------
constexpr int K2_STAGES = 6;
constexpr int K2_THREADS = 384;   // warpgroups 0,1: 8 DMMA warps; warpgroup 2: bulk-copy producer

// NT = n-tiles (8 candidates each) per warp, MT = m-tiles (8 rows each) per warp: a CTA covers 16*MT rows x 32*NT candidates.
//   <4, 8>  throughput shape: 128 rows x 128 candidates, 64 accumulators / thread (240 regs via setmaxnreg), 1 CTA / SM
//   <1, MT> small batches (DIRECT, gallery): 32 candidates per CTA and, for MT < 8, a 16*MT-row slice ("sub-block") of a
//           128-row block, so that a batch of a few dozen candidates still spreads over all SMs and the longest
//           dependent DMMA chain, not a 128-row block, bounds the latency.
// The work list of a CTA is a table built on the host (units[gstart[g] .. gstart[g+1]), unit = i * 8 + h: sub-block h of
// row-block i).  Every accumulator runs over k in ascending order whatever the shape or the grouping, so V is bit-identical
// across shapes; the row reduction is fixed per shape (results do not depend on the batch size, position or grouping
// within a shape; across shapes they differ by the association of the row sums only).
// DEEP: the small shapes with as many pipeline stages as shared memory allows (one CTA per SM).  A batch whose CTAs all fit
// side by side (grid <= number of SMs: a few dozen candidates) is bound by the bulk-copy round trip of its longest unit --
// 32 stages of 4 k-blobs for the last 16-row sub-block at N = 2048, three in flight -- not by the DMMA pipe.
template <int NT, int MT, bool DEEP = false> struct K2Cfg {
    static constexpr int SUBS = 8 / MT;                      // sub-blocks per 128-row block
    static constexpr int ADBL = MT * 2 * 128;                // doubles of one k-blob's A-operand slice: 2*MT m-tiles x 16 k
    static constexpr int BDBL = NT * 4 * 128;                // doubles of one k-blob's B-operand slice: 4*NT n-tiles x 16 k
    // A pipeline stage holds KS k-blobs: the small shapes would otherwise be bound by the bulk-copy round trip (a 6 KiB stage
    // is consumed in ~150 ns, the copy takes ~1 us) and by the per-stage mbarrier handshake.
    static constexpr int KS = (NT == 4 || MT == 8) ? 1 : (MT == 4 ? 2 : 4);
    static constexpr int NS = DEEP ? (MT == 8 ? 9 : (MT == 2 ? 6 : 8))
                                   : ((NT == 4 || MT == 8) ? K2_STAGES : (MT == 4 ? 4 : 3));
    static constexpr int SMEM = NS * KS * (ADBL + BDBL) * 8 + 2 * 3 * 128 * 8 + 2 * NS * 8;
    static constexpr int MINB = (DEEP || NT == 4) ? 1 : (MT == 8 ? 1 : (MT == 1 ? 3 : 2));
    static constexpr bool REGSPLIT = (NT == 4);              // setmaxnreg warp specialisation only where registers are tight
};

template <int NT, int MT, bool P1, bool DEEP = false>
__global__ void __launch_bounds__(K2_THREADS, (K2Cfg<NT, MT, DEEP>::MINB))
trigemm_kernel(const double* __restrict__ Wpack, const double* __restrict__ slab, const double* __restrict__ betaY,
               const double* __restrict__ beta1, double* __restrict__ part, const int* __restrict__ units,
               const int* __restrict__ gstart, int nb, long Mpad, long Mvalid) {
    using Cfg = K2Cfg<NT, MT, DEEP>;
    constexpr int ADBL = Cfg::ADBL, BDBL = Cfg::BDBL, SUBS = Cfg::SUBS, KS = Cfg::KS, NS = Cfg::NS;
    extern __shared__ __align__(128) unsigned char smraw[];
    double* sA = reinterpret_cast<double*>(smraw);
    double* sB = sA + NS * KS * ADBL;
    double* sRed = sB + NS * KS * BDBL;                         // [2][3][128]
    uint64_t* full = reinterpret_cast<uint64_t*>(sRed + 2 * 3 * 128);
    uint64_t* empty = full + NS;
    constexpr int SUB = 4 / NT;                 // CTAs per 128-candidate slab tile
    const int g = blockIdx.x;                   // group fastest: the G CTAs of one tile are co-resident and share its slab in L2
    const int T = blockIdx.y / SUB, sub = blockIdx.y % SUB;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u0 = gstart[g], u1 = gstart[g + 1];
    // The multi-blob stages of the small shapes are fed by KS producer lanes (one per producer warp, lane p moves blob p of
    // every stage): a single lane issuing the 2 KS small bulk copies of a stage was the floor of a small batch.
    constexpr int NPROD = KS;
    if (tid == 0) {
        for (int s = 0; s < NS; s++) { mbar_init(&full[s], NPROD); mbar_init(&empty[s], 8); }
        fence_barrier_init();
        fence_proxy_async();
    }
    __syncthreads();
    if (warp >= 8) {
        // ---------------- producer warpgroup: hands its registers to the DMMA warps ----------------
        if (Cfg::REGSPLIT) asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        // one lane per stage blob streams the operand slices with bulk TMA
        const int pk = warp - 8;
        if (pk < NPROD && lane == 0) {
            if (NT == 1) pdl_wait();             // the K* slab comes from K1 (programmatic launch: K1 may still be running)
            int s = 0; uint32_t ph = 0;
            const double* Bbase = slab + (size_t)T * (nb * KB_PER_BLOCK) * BLOB + sub * BDBL;
            for (int uu = u0; uu < u1; ++uu) {
                const int i = units[uu] >> 3, h = units[uu] & 7;
                // m-tiles are the slowest index of a blob: the sub-block's 2*MT m-tiles are one contiguous slice
                const double* Abase = Wpack + wpack_base(i) * BLOB + h * ADBL;
                const int nkb = i * KB_PER_BLOCK + (h + 1) * MT;     // k-blobs right of column 16 (h+1) MT of the diagonal block are zero
                for (int kb = 0; kb < nkb; kb += KS) {
                    mbar_wait(&empty[s], ph ^ 1);
                    if (kb + pk < nkb) {
                        mbar_arrive_expect_tx(&full[s], (ADBL + BDBL) * 8);
                        bulk_g2s(sA + (s * KS + pk) * ADBL, Abase + (size_t)(kb + pk) * BLOB, ADBL * 8, &full[s]);
                        // n-tiles are the slowest index of a blob, so this CTA's 4*NT n-tiles are one contiguous slice
                        bulk_g2s(sB + (s * KS + pk) * BDBL, Bbase + (size_t)(kb + pk) * BLOB, BDBL * 8, &full[s]);
                    } else {
                        mbar_arrive(&full[s]);   // short last stage: nothing to move for this lane
                    }
                    if (++s == NS) { s = 0; ph ^= 1; }
                }
            }
        }
        return;
    }
    // ---------------- consumers: 8 warps, warp tile 8*MT (rows) x 8*NT (candidates) ----------------
    if (Cfg::REGSPLIT) asm volatile("setmaxnreg.inc.sync.aligned.u32 240;");
    const int wm = warp >> 2, wn = warp & 3;
    // Small batches: a warp whose 8 candidates lie beyond the batch (a 9-point DIRECT batch fills 2 of the 4 n-tiles of its
    // 32-candidate CTA tile) issues no DMMAs -- it only keeps the pipeline handshake going -- so the SM's DMMA pipe serves
    // the warps that carry candidates; the longest unit of such a batch is bound by that pipe.
    const bool active = (NT != 1) || ((long)T * 128 + sub * 32 + wn * 8 < Mvalid);
    int s = 0; uint32_t ph = 0;
    int rbcount = 0;
    for (int uu = u0; uu < u1; ++uu) {
        const int i = units[uu] >> 3, h = units[uu] & 7;
        // SPLIT independent accumulator chains per (m-tile, n-tile): a warp of the smallest shapes owns one or two DMMA tiles,
        // and a single chain of dependent DMMAs (4 per k-blob, ~60 cycles each) was the floor of a small batch -- 16 us for the
        // last sub-block at N = 2048.  Chain c takes the k-steps with (2 ks2 + half) % SPLIT == c; the chains are summed once
        // at the end (in a fixed order: V is deterministic per shape).
        constexpr int SPLIT = (MT * NT >= 4) ? 1 : 4 / (MT * NT);
        double accs[SPLIT][MT][NT][2];
#pragma unroll
        for (int c = 0; c < SPLIT; c++)
#pragma unroll
            for (int a = 0; a < MT; a++)
#pragma unroll
                for (int b = 0; b < NT; b++) accs[c][a][b][0] = accs[c][a][b][1] = 0.0;
        const int nfull = i * KB_PER_BLOCK;     // k-blobs left of the diagonal block: dense
        const int nkb = nfull + (h + 1) * MT;
        for (int kb0 = 0; kb0 < nkb; kb0 += KS) {
            const int nk = (KS == 1) ? 1 : min(KS, nkb - kb0);
            mbar_wait(&full[s], ph);
#pragma unroll 1
            for (int kk = 0; kk < (active ? nk : 0); kk++) {
                const int kb = kb0 + kk;
                // warp wm owns the interleaved m-tiles 2*mt + wm of the sub-block so that the triangular skip below is balanced
                const double2* a2 = reinterpret_cast<const double2*>(sA + (s * KS + kk) * ADBL) + (wm * 2) * 32 + lane;
                const double2* b2 = reinterpret_cast<const double2*>(sB + (s * KS + kk) * BDBL) + (wn * NT * 2) * 32 + lane;
                if (kb < nfull) {
#pragma unroll
                    for (int ks2 = 0; ks2 < 2; ks2++) {
                        double2 af[MT], bf[NT];
#pragma unroll
                        for (int mt = 0; mt < MT; mt++) af[mt] = a2[(mt * 4 + ks2) * 32];
#pragma unroll
                        for (int nt = 0; nt < NT; nt++) bf[nt] = b2[(nt * 2 + ks2) * 32];
#pragma unroll
                        for (int mt = 0; mt < MT; mt++)
#pragma unroll
                            for (int nt = 0; nt < NT; nt++)
                                dmma884(accs[(2 * ks2) % SPLIT][mt][nt][0], accs[(2 * ks2) % SPLIT][mt][nt][1], af[mt].x, bf[nt].x);
#pragma unroll
                        for (int mt = 0; mt < MT; mt++)
#pragma unroll
                            for (int nt = 0; nt < NT; nt++)
                                dmma884(accs[(2 * ks2 + 1) % SPLIT][mt][nt][0], accs[(2 * ks2 + 1) % SPLIT][mt][nt][1], af[mt].y, bf[nt].y);
                    }
                } else {
                    // diagonal block of W (lower triangular): in its k-blob kbl the m-tiles 2*(h*MT+mt) + wm with h*MT+mt < kbl
                    // are identically zero (their rows end before column 16*kbl) and are skipped
                    const int kbl = kb - nfull - h * MT;
#pragma unroll
                    for (int ks2 = 0; ks2 < 2; ks2++) {
                        double2 bf[NT];
#pragma unroll
                        for (int nt = 0; nt < NT; nt++) bf[nt] = b2[(nt * 2 + ks2) * 32];
#pragma unroll
                        for (int mt = 0; mt < MT; mt++) {
                            if (mt >= kbl) {
                                const double2 af = a2[(mt * 4 + ks2) * 32];
#pragma unroll
                                for (int nt = 0; nt < NT; nt++)
                                    dmma884(accs[(2 * ks2) % SPLIT][mt][nt][0], accs[(2 * ks2) % SPLIT][mt][nt][1], af.x, bf[nt].x);
#pragma unroll
                                for (int nt = 0; nt < NT; nt++)
                                    dmma884(accs[(2 * ks2 + 1) % SPLIT][mt][nt][0], accs[(2 * ks2 + 1) % SPLIT][mt][nt][1], af.y, bf[nt].y);
                            }
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (++s == NS) { s = 0; ph ^= 1; }
        }
        double acc[MT][NT][2];
#pragma unroll
        for (int a = 0; a < MT; a++)
#pragma unroll
            for (int b = 0; b < NT; b++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    if (SPLIT == 1) acc[a][b][j] = accs[0][a][b][j];
                    else if (SPLIT == 2) acc[a][b][j] = accs[0][a][b][j] + accs[1 % SPLIT][a][b][j];
                    else acc[a][b][j] = (accs[0][a][b][j] + accs[1 % SPLIT][a][b][j]) + (accs[2 % SPLIT][a][b][j] + accs[3 % SPLIT][a][b][j]);
                }
        // ---- fused reduction of this (16 MT) x (32 NT) block of V over its rows ----
        double by[MT], b1[MT];
#pragma unroll
        for (int mt = 0; mt < MT; mt++) {
            int r = i * 128 + (2 * (h * MT + mt) + wm) * 8 + (lane >> 2);
            by[mt] = betaY[r];
            b1[mt] = P1 ? beta1[r] : 0.0;
        }
        double q[NT][2], p[NT][2], p1[NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; nt++)
#pragma unroll
            for (int j = 0; j < 2; j++) {
                double sq = 0, sp = 0, s1 = 0;
#pragma unroll
                for (int mt = 0; mt < MT; mt++) {
                    double v = acc[mt][nt][j];
                    sq = fma(v, v, sq);
                    sp = fma(v, by[mt], sp);
                    if (P1) s1 = fma(v, b1[mt], s1);
                }
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    sq += __shfl_xor_sync(0xffffffffu, sq, o);
                    sp += __shfl_xor_sync(0xffffffffu, sp, o);
                    if (P1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                }
                q[nt][j] = sq; p[nt][j] = sp; p1[nt][j] = s1;
            }
        double* red = sRed + (rbcount & 1) * 3 * 128;
        if (wm == 1 && lane < 4) {
#pragma unroll
            for (int nt = 0; nt < NT; nt++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    int c = (wn * NT + nt) * 8 + 2 * lane + j;
                    red[c] = q[nt][j]; red[128 + c] = p[nt][j]; if (P1) red[256 + c] = p1[nt][j];
                }
        }
        named_bar_sync(1, 256);
        if (wm == 0 && lane < 4) {
            const size_t plane = (size_t)nb * SUBS * Mpad;
            double* dst = part + (size_t)(i * SUBS + h) * Mpad + (size_t)T * 128 + sub * (32 * NT);
#pragma unroll
            for (int nt = 0; nt < NT; nt++)
#pragma unroll
                for (int j = 0; j < 2; j++) {
                    int c = (wn * NT + nt) * 8 + 2 * lane + j;
                    dst[c] = q[nt][j] + red[c];
                    dst[plane + c] = p[nt][j] + red[128 + c];
                    if (P1) dst[2 * plane + c] = p1[nt][j] + red[256 + c];
                }
        }
        rbcount++;
    }
    if (NT == 1) pdl_launch_dependents();        // small batches: K3 (programmatic launch) may be scheduled as this grid drains
}

// ---------------------------------------------------------------------------------------------
// K3: per-candidate epilogue.
// ---------------------------------------------------------------------------------------------
struct EpiParams {
    int nbPart, d, N, acq, mode_py, npb, want_p1, want_argmax, rowLanes;   // nbPart: rows of the partial-sum planes (nb * sub-blocks)
    long M, m0, chunkM, Mpad;
    double noise, ymax, parm, ptheta;
    const double *part, *partVar, *cand, *pmeans, *pbeta, *plb, *pwidth;
    int nbVarPart; long MpadVar;
    double *score, *mu, *s2;
    double* blkBest; long long* blkIdx; long blk0;
    double guard_s2; unsigned char* flag;       // INT8 path: candidates with sigma^2 < guard_s2 are flagged for the DMMA re-score
};

__global__ void __launch_bounds__(256) epilogue_kernel(EpiParams P) {
    // rowLanes = 1: one thread per candidate walks all partial rows (throughput shape: nb rows).
    // rowLanes = 8 / 32: small batches, whose latency shapes of K2 leave up to 8 nb partial rows: 256 / rowLanes candidates
    //               per block, rowLanes threads per candidate each sum every rowLanes-th row (loads batched four deep),
    //               combined in a fixed order through shared memory.
    __shared__ double shq[3][256];
    pdl_wait();                                                // programmatic launch behind K2 (small batches); no-op otherwise
    const int RL = P.rowLanes, CPB = 256 / RL;                 // candidates per block
    const int tl = threadIdx.x / CPB;                          // row lane
    const int cl = threadIdx.x - tl * CPB;
    const long lm = (long)blockIdx.x * CPB + cl;               // index within the chunk
    const long m = P.m0 + lm;
    double sc = -INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    const bool live = lm < P.chunkM && m < P.M;
    double q = 0, p = 0, p1 = 0;
    if (live) {
        const size_t plane = (size_t)P.nbPart * P.Mpad;
        const double* pq = P.partVar ? nullptr : P.part + lm;
        const double* pp = P.part + plane + lm;
        const double* p1p = P.want_p1 ? P.part + 2 * plane + lm : nullptr;
        int i = tl;
        for (; i + 3 * RL < P.nbPart; i += 4 * RL) {
            double a0 = pp[(size_t)i * P.Mpad], a1 = pp[(size_t)(i + RL) * P.Mpad], a2 = pp[(size_t)(i + 2 * RL) * P.Mpad], a3 = pp[(size_t)(i + 3 * RL) * P.Mpad];
            double b0 = 0, b1 = 0, b2 = 0, b3 = 0, c0 = 0, c1 = 0, c2 = 0, c3 = 0;
            if (pq) { b0 = pq[(size_t)i * P.Mpad]; b1 = pq[(size_t)(i + RL) * P.Mpad]; b2 = pq[(size_t)(i + 2 * RL) * P.Mpad]; b3 = pq[(size_t)(i + 3 * RL) * P.Mpad]; }
            if (p1p) { c0 = p1p[(size_t)i * P.Mpad]; c1 = p1p[(size_t)(i + RL) * P.Mpad]; c2 = p1p[(size_t)(i + 2 * RL) * P.Mpad]; c3 = p1p[(size_t)(i + 3 * RL) * P.Mpad]; }
            p += a0; p += a1; p += a2; p += a3;          // same ascending order as the scalar tail below
            q += b0; q += b1; q += b2; q += b3;
            p1 += c0; p1 += c1; p1 += c2; p1 += c3;
        }
        for (; i < P.nbPart; i += RL) {
            p += pp[(size_t)i * P.Mpad];
            if (pq) q += pq[(size_t)i * P.Mpad];
            if (p1p) p1 += p1p[(size_t)i * P.Mpad];
        }
        if (P.partVar) {
            const double* pv = P.partVar + lm;
            for (int iv = tl; iv < P.nbVarPart; iv += RL) q += pv[(size_t)iv * P.MpadVar];
        }
    }
    if (RL > 1) {
        shq[0][threadIdx.x] = q; shq[1][threadIdx.x] = p; shq[2][threadIdx.x] = p1;
        __syncthreads();
        if (tl == 0) {
            q = 0; p = 0; p1 = 0;
            for (int t = 0; t < RL; t++) { q += shq[0][t * CPB + cl]; p += shq[1][t * CPB + cl]; p1 += shq[2][t * CPB + cl]; }
        }
    }
    if (live && tl == 0) {
        double m0 = 0.0;
        if (P.npb > 0) m0 = prior_mean(P.cand + (size_t)m * P.d, P.d, P.npb, P.pmeans, P.pbeta, P.ptheta, P.plb, P.pwidth);
        double mu = m0 + p - m0 * p1;
        double s2 = (1.0 + P.noise) - q;
        // INT8 path only: too close to total cancellation for the integer scheme's absolute error -- the guard pass re-scores
        // this candidate with the DMMA kernels and merges it into the argmax; here it takes no part in it
        const bool guarded = P.flag != nullptr && s2 < P.guard_s2;
        if (P.flag) P.flag[m] = guarded ? 1 : 0;
        const double floor_ = P.mode_py ? 10e-8 : 1e-8;   // gaussianprocess/__init__.py:224 vs cpp/optimizeGP.cpp:150
        s2 = s2 < floor_ ? floor_ : (s2 > 10.0 ? 10.0 : s2);
        if (P.mu) P.mu[m] = mu;
        if (P.s2) P.s2[m] = s2;
        if (P.acq >= 0) {
            double v = acq_value(P.acq, P.mode_py, mu, s2, P.ymax, P.parm);
            if (P.score) P.score[m] = v;
            if (!guarded) {
                if (v == v) { sc = v; idx = m; }   // NaN never wins
                else idx = m;
            }
        }
    }
    if (P.acq < 0 || !P.want_argmax) return;
    // block argmax, lowest index wins ties
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
        P.blkBest[P.blk0 + blockIdx.x] = sc;
        P.blkIdx[P.blk0 + blockIdx.x] = idx;
    }
}

__global__ void __launch_bounds__(256) argmax_final_kernel(const double* __restrict__ blkBest, const long long* __restrict__ blkIdx,
                                                           long nblk, double* __restrict__ best, long long* __restrict__ bestIdx) {
    double sc = -INFINITY;
    long long idx = 0x7fffffffffffffffLL;
    for (long b = threadIdx.x; b < nblk; b += 256) {
        double os = blkBest[b]; long long oi = blkIdx[b];
        if (os > sc || (os == sc && oi < idx)) { sc = os; idx = oi; }
    }
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
        *best = sc; *bestIdx = idx;
    }
}


// ---------------------------------------------------------------------------------------------
// Guard pass of the INT8 path: ordered compaction of the flagged candidates (ascending index, so that "lowest index wins" keeps
// its meaning), their coordinates gathered for a DMMA re-score, the results scattered back and merged into the argmax.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) guard_count_kernel(const unsigned char* __restrict__ flag, long M, int* __restrict__ blkCount) {
    const long base = (long)blockIdx.x * 1024 + threadIdx.x * 4;
    int c = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) if (base + j < M && flag[base + j]) c++;
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ int ws[8];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; w++) t += ws[w]; blkCount[blockIdx.x] = t; }
}
// exclusive scan of the block counts in place (one block; nblk <= a few ten thousand); total -> *count
__global__ void __launch_bounds__(256) guard_scan_kernel(int* __restrict__ blkCount, int nblk, int* __restrict__ count) {
    __shared__ int part[256];
    const int per = (nblk + 255) / 256, b0 = threadIdx.x * per, b1 = min(nblk, b0 + per);
    int s = 0;
    for (int b = b0; b < b1; b++) s += blkCount[b];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) { int run = 0; for (int t = 0; t < 256; t++) { int v = part[t]; part[t] = run; run += v; } *count = run; }
    __syncthreads();
    int run = part[threadIdx.x];
    for (int b = b0; b < b1; b++) { int v = blkCount[b]; blkCount[b] = run; run += v; }
}
__global__ void __launch_bounds__(256) guard_gather_kernel(const unsigned char* __restrict__ flag, long M, const int* __restrict__ blkOff,
                                                           const double* __restrict__ cand, int d, long long* __restrict__ list,
                                                           double* __restrict__ gcand) {
    const long base = (long)blockIdx.x * 1024 + threadIdx.x * 4;
    int f[4], c = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) { f[j] = (base + j < M && flag[base + j]) ? 1 : 0; c += f[j]; }
    // exclusive prefix of c over the block: warp scan, then the warps in order
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if ((threadIdx.x & 31) >= o) incl += v; }
    __shared__ int ws[8];
    if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    int off = blkOff[blockIdx.x] + incl - c;
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) off += ws[w];
#pragma unroll
    for (int j = 0; j < 4; j++)
        if (f[j]) {
            list[off] = base + j;
            for (int t = 0; t < d; t++) gcand[(size_t)off * d + t] = cand[(size_t)(base + j) * d + t];
            off++;
        }
}
// out planes [score | mu | s2][M] <- the re-scored values; (best, index) merged with the re-scored set's own argmax
__global__ void __launch_bounds__(256) guard_scatter_kernel(const long long* __restrict__ list, int count, const double* __restrict__ gout,
                                                            double* __restrict__ out, long M, int wscore, int wmu, int ws2, int wargmax) {
    const int k = blockIdx.x * 256 + threadIdx.x;
    if (k < count) {
        const long long m = list[k];
        if (wscore) out[m] = gout[k];
        if (wmu) out[M + m] = gout[(size_t)count + k];
        if (ws2) out[2 * M + m] = gout[2 * (size_t)count + k];
    }
    if (wargmax && k == 0) {
        const double gs = gout[3 * (size_t)count];
        long long gi; memcpy(&gi, &gout[3 * (size_t)count + 1], 8);
        if (gi >= 0 && gi < count) {
            const long long gm = list[gi];
            double bs = out[3 * M];
            long long bi; memcpy(&bi, &out[3 * M + 1], 8);
            // the main pass left (-inf, sentinel) when every candidate was guarded; NaN scores never win on either side
            if (gs > bs || (gs == bs && gm < bi) || !(bs == bs)) { out[3 * M] = gs; memcpy(&out[3 * M + 1], &gm, 8); }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host-side orchestration
// ---------------------------------------------------------------------------------------------
template <int NT, int MT>
static cudaError_t set_k2_attr() {
    cudaError_t e = cudaFuncSetAttribute(trigemm_kernel<NT, MT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2Cfg<NT, MT>::SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(trigemm_kernel<NT, MT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2Cfg<NT, MT>::SMEM);
    if constexpr (NT == 1) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trigemm_kernel<NT, MT, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2Cfg<NT, MT, true>::SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(trigemm_kernel<NT, MT, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2Cfg<NT, MT, true>::SMEM);
    }
    return e;
}
// dynamic shared-memory opt-ins of the scoring kernels; cudaFuncSetAttribute is per device (ensure_attrs runs this once per device)
static cudaError_t set_score_attrs() {
    cudaError_t e = set_k2_attr<4, 8>();
    if (e == cudaSuccess) e = set_k2_attr<1, 8>();
    if (e == cudaSuccess) e = set_k2_attr<1, 4>();
    if (e == cudaSuccess) e = set_k2_attr<1, 2>();
    if (e == cudaSuccess) e = set_k2_attr<1, 1>();
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kstar_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 128 * 65 * 8);
    return e;
}

static long chunk_tiles_default(int sms) {
    const long v = get_option(OPT_CHUNK_TILES);     // tuning knob (tools/perf_sweep.sh)
    return v > 0 ? v : 2L * sms;
}

static long narrow_threshold() { return get_option(OPT_NARROW_MAX); }

// ---------------------------------------------------------------------------------------------
// K2 launch plans.  A plan fixes the CTA shape (MT), the number G of CTAs that share one candidate tile, and the table
// that deals the (row-block, sub-block) units of a tile to those G CTAs.
//   wide (NT = 4): G = nb/4 row-block groups in snake order (work ~ i+1; exactly balanced when 2G | nb).  (a) L2
//     residency: the G CTAs of a tile run side by side, so about num_sms / G slab tiles (Np KiB each) are live at once --
//     <= 148 * 4 * 128 KiB = 74 MiB of the 126 MiB L2 for every N; (b) small sets raise G until tiles * G >= num_sms.
//   narrow (NT = 1, M <= 2048): latency matters.  For each shape MT in {8, 4, 2, 1} and each G that fills whole "rounds" of
//     the SMs, the units are dealt longest-first to the least loaded CTA (LPT) and the makespan is estimated; the cheapest
//     (MT, G) wins.  Small MT = more, shorter CTAs (a 24-candidate DIRECT batch at N = 2048 runs as 128 CTAs of 16 rows
//     instead of 16 CTAs of 128 rows) at the price of less operand reuse (A: 2 MT KiB, B: 4 KiB per stage).
// ---------------------------------------------------------------------------------------------
struct UnitTable { int G = 0; int* dUnits = nullptr; int* dStart = nullptr; };   // device copies, owned by the model

static double lpt_deal(int nb, int MT, int G, std::vector<int>* units, std::vector<int>* start) {
    const int SUBS = 8 / MT;
    struct U { double c; int code; };
    std::vector<U> us;
    us.reserve((size_t)nb * SUBS);
    for (int i = nb - 1; i >= 0; --i)
        for (int h = SUBS - 1; h >= 0; --h)
            us.push_back({(double)((i * 8 + (h + 1) * MT) * MT + 6), i * 8 + h});     // stages x m-tiles per warp + epilogue
    std::stable_sort(us.begin(), us.end(), [](const U& a, const U& b) { return a.c > b.c; });
    std::vector<double> load(G, 0.0);
    std::vector<std::vector<int>> mine(units ? G : 0);
    typedef std::pair<double, int> LG;                                  // (load, group): least loaded first, lowest group on ties
    std::priority_queue<LG, std::vector<LG>, std::greater<LG>> heap;
    for (int gI = 0; gI < G; gI++) heap.push(LG(0.0, gI));
    for (const U& u : us) {
        LG top = heap.top(); heap.pop();
        top.first += u.c; load[top.second] = top.first;
        if (units) mine[top.second].push_back(u.code);
        heap.push(top);
    }
    double mk = 0;
    for (int gI = 0; gI < G; gI++) mk = std::max(mk, load[gI]);
    if (units) {
        units->clear(); start->assign(G + 1, 0);
        for (int gI = 0; gI < G; gI++) { for (int c : mine[gI]) units->push_back(c); (*start)[gI + 1] = (int)units->size(); }
    }
    return mk;
}

static void snake_deal(int nb, int G, std::vector<int>* units, std::vector<int>* start) {
    units->clear(); start->assign(G + 1, 0);
    for (int gI = 0; gI < G; gI++) {
        for (int i = nb - 1; i >= 0; --i) {
            int idx = nb - 1 - i, round = idx / G, pos = idx - round * G;
            if (((round & 1) ? (G - 1 - pos) : pos) == gI) units->push_back(i * 8);
        }
        (*start)[gI + 1] = (int)units->size();
    }
}

struct K2Plan { int MT; int G; };

static K2Plan plan_narrow(int nb, long ctaTiles, int g_num_sms) {
    const int forceMT = (int)get_option(OPT_NARROW_MT);
    const int mts[4] = {8, 4, 2, 1};
    const int resident[4] = {1, 2, 2, 3};
    const double eff[4] = {1.0, 0.95, 0.75, 0.5};        // achievable share of the DMMA rate (operand traffic per DMMA grows as MT shrinks)
    K2Plan best{8, 1};
    double bestT = 1e300;
    for (int q = 0; q < 4; q++) {
        const int MT = mts[q];
        if (forceMT > 0 && MT != forceMT) continue;
        const int nunits = nb * (8 / MT);
        const long bins = (long)g_num_sms * resident[q];
        long Gmax = std::min<long>(nunits, std::max<long>(1, bins / ctaTiles));
        // candidates: G that fill 1 .. resident rounds of the SMs, and the largest one
        long cand[6]; int nc = 0;
        for (int r = 1; r <= resident[q]; r++) { long Gc = (long)g_num_sms * r / ctaTiles; if (Gc >= 1 && Gc <= Gmax) cand[nc++] = Gc; }
        cand[nc++] = Gmax;
        if (Gmax > 1) cand[nc++] = 1;
        for (int c = 0; c < nc; c++) {
            const int G = (int)cand[c];
            const double mk = lpt_deal(nb, MT, G, nullptr, nullptr);
            const long perSM = (ctaTiles * G + g_num_sms - 1) / g_num_sms;     // CTAs sharing one SM's DMMA pipe
            const double t = perSM * (mk + 16.0) / eff[q];
            if (t < bestT) { bestT = t; best = K2Plan{MT, G}; }
        }
    }
    return best;
}

static K2Plan plan_narrow_cached(ibo_model* m, long ctaTiles) {
    auto it = m->planCache.find(ctaTiles);
    if (it == m->planCache.end()) {
        K2Plan pl = plan_narrow(m->nb, ctaTiles, dev_info(m->device).sms);
        if (get_option(OPT_DEBUG_PLAN)) fprintf(stderr, "[plan_narrow] nb=%d ctaTiles=%ld -> MT=%d G=%d (%ld CTAs)\n", m->nb, ctaTiles, pl.MT, pl.G, ctaTiles * pl.G);
        it = m->planCache.emplace(ctaTiles, std::make_pair(pl.MT, pl.G)).first;
    }
    return K2Plan{it->second.first, it->second.second};
}

static int pick_groups_wide(int nb, long tiles, int g_num_sms) {
    long G = std::max(1, nb / 4);
    if (tiles * G < g_num_sms) G = (g_num_sms + tiles - 1) / tiles;
    return (int)std::min<long>(G, nb);
}

// device table for (MT, G), cached on the model
static int get_unit_table(ibo_model* m, bool narrow, int MT, int G, const int** dUnits, const int** dStart) {
    const long key = ((long)(narrow ? 1 : 0) << 40) | ((long)MT << 32) | (long)G;
    auto it = m->unitTables.find(key);
    if (it == m->unitTables.end()) {
        std::vector<int> units, start;
        if (narrow) lpt_deal(m->nb, MT, G, &units, &start); else snake_deal(m->nb, G, &units, &start);
        int* d = nullptr;
        IBO_CUDA_TRY(cudaMalloc(&d, sizeof(int) * (units.size() + start.size())));
        IBO_CUDA_TRY(cudaMemcpyAsync(d, units.data(), sizeof(int) * units.size(), cudaMemcpyHostToDevice, m->stream));
        IBO_CUDA_TRY(cudaMemcpyAsync(d + units.size(), start.data(), sizeof(int) * start.size(), cudaMemcpyHostToDevice, m->stream));
        IBO_CUDA_TRY(cudaStreamSynchronize(m->stream));      // the host vectors go out of scope
        it = m->unitTables.emplace(key, std::make_pair(d, (int)units.size())).first;
    }
    *dUnits = it->second.first;
    *dStart = it->second.first + it->second.second;
    return IBO_OK;
}

// launch with (pdl) or without the programmatic-stream-serialization attribute
template <typename... KArgs, typename... Args>
static cudaError_t launch_ex(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

static bool pdl_enabled() { return get_option(OPT_PDL) != 0; }

// option k2_deep: 0 = never, 1 = whenever the shape is a small one, -1 (default) = when the grid fits the SMs
static int deep_mode() { return (int)get_option(OPT_K2_DEEP); }

template <int NT, int MT>
static void launch_k2_shape(const ibo_model* m, bool p1, dim3 grid, const int* dUnits, const int* dStart, long Mpad, long Mvalid, cudaStream_t st) {
    const bool pdl = (NT == 1) && pdl_enabled();     // small batches only: the throughput shape must not sit on SMs K1 is using
    if constexpr (NT == 1) {
        const int dm = deep_mode();
        if (dm == 1 || (dm < 0 && (long)grid.x * grid.y <= dev_info(m->device).sms)) {
            if (p1) launch_ex(trigemm_kernel<NT, MT, true, NT == 1>, grid, dim3(K2_THREADS), K2Cfg<NT, MT, NT == 1>::SMEM, st, pdl,
                              m->dWpack, m->dSlab, m->dBetaY, m->dBeta1, m->dPart, dUnits, dStart, m->nb, Mpad, Mvalid);
            else launch_ex(trigemm_kernel<NT, MT, false, NT == 1>, grid, dim3(K2_THREADS), K2Cfg<NT, MT, NT == 1>::SMEM, st, pdl,
                           m->dWpack, m->dSlab, m->dBetaY, m->dBeta1, m->dPart, dUnits, dStart, m->nb, Mpad, Mvalid);
            return;
        }
    }
    if (p1) launch_ex(trigemm_kernel<NT, MT, true>, grid, dim3(K2_THREADS), K2Cfg<NT, MT>::SMEM, st, pdl,
                      m->dWpack, m->dSlab, m->dBetaY, m->dBeta1, m->dPart, dUnits, dStart, m->nb, Mpad, Mvalid);
    else launch_ex(trigemm_kernel<NT, MT, false>, grid, dim3(K2_THREADS), K2Cfg<NT, MT>::SMEM, st, pdl,
                   m->dWpack, m->dSlab, m->dBetaY, m->dBeta1, m->dPart, dUnits, dStart, m->nb, Mpad, Mvalid);
}

// ytiles: CTAs along the candidate axis (128-candidate tiles when wide, 32-candidate tiles when narrow)
static int launch_trigemm(ibo_model* m, bool narrow, K2Plan pl, bool p1, long ytiles, long Mpad, long Mvalid, cudaStream_t st) {
    const int *dUnits, *dStart;
    int rc = get_unit_table(m, narrow, pl.MT, pl.G, &dUnits, &dStart);
    if (rc) return rc;
    dim3 grid(pl.G, (unsigned)ytiles);
    if (!narrow) launch_k2_shape<4, 8>(m, p1, grid, dUnits, dStart, Mpad, Mvalid, st);
    else if (pl.MT == 8) launch_k2_shape<1, 8>(m, p1, grid, dUnits, dStart, Mpad, Mvalid, st);
    else if (pl.MT == 4) launch_k2_shape<1, 4>(m, p1, grid, dUnits, dStart, Mpad, Mvalid, st);
    else if (pl.MT == 2) launch_k2_shape<1, 2>(m, p1, grid, dUnits, dStart, Mpad, Mvalid, st);
    else launch_k2_shape<1, 1>(m, p1, grid, dUnits, dStart, Mpad, Mvalid, st);
    return IBO_OK;
}

template <int DP4>
static void launch_kstar_mma(dim3 grid, cudaStream_t st, const ibo_model* m, const double* dCand, double* slab, long M, long m0,
                             const CandInline& inl) {
    constexpr int DP = 4 * DP4;
    constexpr int S = (DP % 16 == 4 || DP % 16 == 12) ? DP : DP + 4;
    const size_t smem = (2 * 128 * S + 256) * 8;
    if (m->kind <= IBO_KERNEL_SE_ISO)
        kstar_mma_kernel<DP4, 0><<<grid, 256, smem, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, slab, m->N, m->d, m->nb, M, m0, m->kind, m->sf2, inl);
    else if (m->kind == IBO_KERNEL_MATERN3)
        kstar_mma_kernel<DP4, 1><<<grid, 256, smem, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, slab, m->N, m->d, m->nb, M, m0, m->kind, m->sf2, inl);
    else
        kstar_mma_kernel<DP4, 2><<<grid, 256, smem, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, slab, m->N, m->d, m->nb, M, m0, m->kind, m->sf2, inl);
}

static bool kstar_uses_mma(const ibo_model* m) { return get_option(OPT_KSTAR_DIRECT) == 0 && (m->d + 3) / 4 <= 8; }

// cross-covariance of one chunk; expansion on the tensor pipe for d <= 32 unless IBO_KSTAR=direct
// inl != nullptr: the candidates are in *inl (host copy for the parameter buffer) and dCand is not valid
static void launch_kstar(const ibo_model* m, const double* dCand, double* slab, long tiles, long M, long m0, cudaStream_t st,
                         const CandInline* inl = nullptr) {
    static CandInline none;
    const CandInline& I = inl ? *inl : none;
    if (inl) dCand = nullptr;
    dim3 grid((unsigned)tiles, m->nb);
    const int dp4 = (m->d + 3) / 4;
    if (!kstar_uses_mma(m)) {
        const int kS = m->d | 1;
        kstar_kernel<<<grid, 256, 2 * 128 * kS * 8, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, slab, m->N, m->d, m->nb, M, m0, m->kind, m->sf2);
        return;
    }
    // few CTAs (DIRECT / gallery batches): split each candidate tile's n-tiles over grid.z until the grid covers the SMs
    unsigned z = 1;
    while (z < 16 && (long)tiles * m->nb * z < dev_info(m->device).sms) z *= 2;
    grid.z = z;
    switch (dp4) {
        case 1: launch_kstar_mma<1>(grid, st, m, dCand, slab, M, m0, I); break;
        case 2: launch_kstar_mma<2>(grid, st, m, dCand, slab, M, m0, I); break;
        case 3: launch_kstar_mma<3>(grid, st, m, dCand, slab, M, m0, I); break;
        case 4: launch_kstar_mma<4>(grid, st, m, dCand, slab, M, m0, I); break;
        case 5: launch_kstar_mma<5>(grid, st, m, dCand, slab, M, m0, I); break;
        case 6: launch_kstar_mma<6>(grid, st, m, dCand, slab, M, m0, I); break;
        case 7: launch_kstar_mma<7>(grid, st, m, dCand, slab, M, m0, I); break;
        default: launch_kstar_mma<8>(grid, st, m, dCand, slab, M, m0, I); break;
    }
}


}  // namespace ibo
#include "score_i8.cuh"
namespace ibo {

constexpr int FLAG_FORCE_WIDE = 0x40000000;     // internal: K2's throughput shape (and no fused small-model kernel) whatever the batch size
constexpr int FLAG_I8_ANY_SIZE = 0x20000000;    // internal (sharded DIRECT): the INT8 path whatever the size of this slice -- the
                                                // arithmetic of a candidate is chosen from the size of the FULL batch on every rank

static cudaError_t set_i8_attrs() {
    return cudaFuncSetAttribute(trigemm_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, I8_SMEM);
}

// Which arithmetic scores this batch.  Wide batches (more than `narrow_max` candidates) of a plain model go through the INT8
// tensor-core path unless the caller forces FP64 (IBO_FLAG_FP64, option int8 = 0); small batches, models with a variance model
// (PrefGP aug), d > 32 and N > 16384 (INT32 head-room of the 8-bit digits) always take the DMMA kernels.
static bool i8_eligible(const ibo_model* m, int flags) {
    if (m->var_model || m->d > 32 || m->Np > 16384 || (flags & IBO_FLAG_FP64)) return false;
    return (flags & IBO_FLAG_INT8) || get_option(OPT_INT8) != 0;
}
// Mid-size batches (DIRECT's, up to narrow_max candidates) on a model of more than one row-block: the FP64 latency shapes need
// N^2 flops per candidate at 37 TF/s, the INT8 kernels finish a large enough batch several times sooner.  Where "large enough"
// starts was measured (tools/i8_crossover.py, host candidates in, scores out, d = 6 and 20): the INT8 call costs ~50 us + N / 60 us
// up to ~256 candidates, the FP64 call ~40 us + 3.5e-8 us x M N^2; they cross at M = 735 / 300 / 133 / 62 for N = 1024 / 2048 /
// 4096 / 8192.  Option i8_min_batch: -1 this rule, 0 never, > 0 a fixed batch size.
static bool i8_for_small_batch(const ibo_model* m, long M, int flags) {
    if (!i8_eligible(m, flags) || m->nb < 2) return false;
    if (flags & FLAG_I8_ANY_SIZE) return true;
    const long lo = get_option(OPT_I8_MIN_BATCH);
    if (lo >= 0) return lo > 0 && M >= lo;
    const double n = (double)m->Np;
    return (double)M * 3.5e-8 * n * n >= 10.0 + n / 60.0;
}

// Runs K1..K4 for M candidates resident at dCand; results land in m->dOut ([score|mu|s2][M]) and
// the (best score, best index) pair at m->dOut[3M], [3M+1].  Everything is enqueued on m->stream; the only host
// synchronisation is the 4-byte read of the guard count on the INT8 path of a small-noise model.
// `hostWide`: the candidates are still in host memory (all M of them, destined for dCand): every chunk is copied on a separate
// stream two chunks ahead of the kernels that read it, so that a call from host buffers pays for the first chunk's copy only.
static int score_device(ibo_model* m, const double* dCand, long M, const ScoreReq& rq, double* outBase = nullptr,
                        const double* hostCand = nullptr, const double* hostWide = nullptr) {
    cudaError_t ae = ensure_attrs(m->device, ATTR_SCORE, set_score_attrs);
    if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); return IBO_E_CUDA; }
    if (m->d > 64) { set_error("d > 64 not supported"); return IBO_E_BADARG; }
    const bool forceWide = (rq.flags & FLAG_FORCE_WIDE) != 0;
    if (!forceWide && tiny_eligible(m, M)) {       // N <= 128, small batch: one fused launch (tiny.cu)
        int rc0;
        if (!outBase && (rc0 = grow(&m->dOut, &m->outCap, (size_t)3 * M + 2))) return rc0;
        if (hostWide) IBO_CUDA_TRY(cudaMemcpyAsync(const_cast<double*>(dCand), hostWide, sizeof(double) * (size_t)M * m->d, cudaMemcpyHostToDevice, m->stream));
        return score_tiny(m, dCand, M, rq, outBase ? outBase : m->dOut, hostCand);
    }
    cudaStream_t st = m->stream;
    const int sms = dev_info(m->device).sms;
    const bool prof = (rq.flags & IBO_FLAG_PROFILE) != 0;
    ibo_model* vm = m->var_model;
    const int nb = m->nb;
    // hostCand given and dCand null: the batch is small enough to ride in K1's parameter buffer (score_host decided)
    CandInline inlBuf;
    const CandInline* inl = nullptr;
    if (hostCand && !dCand) {
        std::memcpy(inlBuf.x, hostCand, sizeof(double) * (size_t)M * m->d);
        inl = &inlBuf;
    }
    const long tilesTotal = (M + TN - 1) / TN;
    long chunkTiles = std::min<long>(tilesTotal, chunk_tiles_default(sms));
    const bool i8small = !forceWide && M <= narrow_threshold() && i8_for_small_batch(m, M, rq.flags);
    const bool narrow = !forceWide && !i8small && M <= narrow_threshold();
    const bool i8 = !narrow && i8_eligible(m, rq.flags);
    // keep the slab below ~6 GiB (FP64: 8 N bytes per candidate; INT8: 7 N bytes, double buffered)
    while (chunkTiles > 1 && (double)chunkTiles * nb * KB_PER_BLOCK * BLOB * (i8 ? 14.0 : 8.0) > 6.0e9) chunkTiles = (chunkTiles + 1) / 2;
    const long Mpad = chunkTiles * TN;
    int rc;
    const long ctaTilesAll = narrow ? (std::min<long>(M, Mpad) + 31) / 32 : chunkTiles;      // K2 CTAs along the candidate axis
    const K2Plan plan = narrow ? plan_narrow_cached(m, ctaTilesAll) : K2Plan{8, pick_groups_wide(nb, chunkTiles, sms)};
    const int subs = 8 / plan.MT;
    if (i8) {
        ae = ensure_attrs(m->device, ATTR_I8, set_i8_attrs);
        if (ae != cudaSuccess) { set_error(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(ae)); return IBO_E_CUDA; }
        if ((rc = ensure_i8(m))) return rc;
    }
    // int8 path: K1 of chunk c+1 (FP64 / integer pipes, low-priority stream2) runs under K2 of chunk c (tensor pipe, main stream);
    // slab and partial-sum planes are double buffered.  With IBO_FLAG_PROFILE the chunks run back to back so that K1 / K2 can be timed.
    const bool i8pipe = i8 && !prof && get_option(OPT_I8_PIPE) != 0 && tilesTotal > chunkTiles;     // a single chunk has nothing to overlap
    const size_t i8SlabBytes = (size_t)chunkTiles * 2 * nb * 4 * I8_B_STAGE, i8PartDbl = (size_t)3 * nb * Mpad;
    // guard pass: only a model whose sigma^2 can get below the threshold needs it (sigma^2 >= noise for a model built from R)
    const bool guard = i8 && get_option(OPT_I8_GUARD) != 0 && (m->noise < I8_GUARD_S2 || m->from_inverse);
    if (i8) {
        if ((rc = grow(&m->dSlab, &m->slabCap, 2 * ((i8SlabBytes + 7) / 8)))) return rc;
        if ((rc = grow(&m->dPart, &m->partCap, 2 * i8PartDbl))) return rc;
        if (guard && (rc = grow(&m->dGuard, &m->guardCap, (size_t)(M + 7) / 8 + (size_t)(M + 1023) / 1024 / 2 + 4))) return rc;
        if (i8pipe) {
            IBO_CUDA_TRY(cudaEventRecord(m->evI8[4], st));
            IBO_CUDA_TRY(cudaStreamWaitEvent(m->stream2, m->evI8[4], 0));
        }
    } else {
        if ((rc = grow(&m->dSlab, &m->slabCap, (size_t)chunkTiles * nb * KB_PER_BLOCK * BLOB))) return rc;
    }
    unsigned char* const dFlag = guard ? reinterpret_cast<unsigned char*>(m->dGuard) : nullptr;
    long ci = 0;
    if ((rc = grow(&m->dPart, &m->partCap, (size_t)3 * nb * subs * Mpad))) return rc;
    if ((rc = grow(&m->dOut, &m->outCap, (size_t)3 * M + 2))) return rc;
    double* const out = outBase ? outBase : m->dOut;     // outBase: device-visible pinned host memory (zero-copy results)
    if (vm) {
        if ((rc = grow(&vm->dSlab, &vm->slabCap, (size_t)chunkTiles * vm->nb * KB_PER_BLOCK * BLOB))) return rc;
    }
    K2Plan planV{8, 1};
    if (vm) {
        planV = narrow ? plan_narrow_cached(vm, ctaTilesAll) : K2Plan{8, pick_groups_wide(vm->nb, chunkTiles, sms)};
        if ((rc = grow(&vm->dPart, &vm->partCap, (size_t)3 * vm->nb * (8 / planV.MT) * Mpad))) return rc;
    }
    const long nblkTotal = (M + 7) / 8 + tilesTotal;       // generous upper bound (chunk boundaries, 8-candidate blocks of small batches)
    if (m->blkCap < (size_t)nblkTotal) {
        if (m->dBlkBest) cudaFree(m->dBlkBest);
        if (m->dBlkIdx) cudaFree(m->dBlkIdx);
        m->dBlkBest = nullptr; m->dBlkIdx = nullptr; m->blkCap = 0;
        IBO_CUDA_TRY(cudaMalloc(&m->dBlkBest, sizeof(double) * nblkTotal));
        IBO_CUDA_TRY(cudaMalloc(&m->dBlkIdx, sizeof(long long) * nblkTotal));
        m->blkCap = nblkTotal;
    }
    double tK1 = 0, tK2 = 0, tK3 = 0;
    long nlaunch = 0, nK2 = 0;
    if (prof) IBO_CUDA_TRY(cudaEventRecord(m->ev[0], st));
    long blk0 = 0;
    const long nchunks = (tilesTotal + chunkTiles - 1) / chunkTiles;
    long copied = 0;                                    // chunks whose host -> device copy has been issued
    cudaStream_t cs = m->stream3;                       // idle outside the model build; the copies run on the DMA engines
    if (hostWide) {
        for (auto& e : m->evCopy) if (!e) IBO_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        IBO_CUDA_TRY(cudaEventRecord(m->evCopy[4], st));                 // whatever still reads dCand from an earlier call
        IBO_CUDA_TRY(cudaStreamWaitEvent(cs, m->evCopy[4], 0));
    }
    for (long t0 = 0; t0 < tilesTotal; t0 += chunkTiles) {
        const long tiles = std::min(chunkTiles, tilesTotal - t0);
        const long m0 = t0 * TN;
        const long chunkM = std::min<long>(tiles * TN, M - m0);
        if (hostWide) {
            for (; copied < nchunks && copied <= ci + 2; copied++) {
                const long c0 = copied * Mpad, cn = std::min<long>(Mpad, M - c0);
                IBO_CUDA_TRY(cudaMemcpyAsync(const_cast<double*>(dCand) + (size_t)c0 * m->d, hostWide + (size_t)c0 * m->d,
                                             sizeof(double) * (size_t)cn * m->d, cudaMemcpyHostToDevice, cs));
                IBO_CUDA_TRY(cudaEventRecord(m->evCopy[copied & 3], cs));
            }
            // slot ci & 3 is re-recorded for chunk ci + 4 only two iterations from now, after these waits have been enqueued
            IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evCopy[ci & 3], 0));
            if (i8pipe) IBO_CUDA_TRY(cudaStreamWaitEvent(m->stream2, m->evCopy[ci & 3], 0));
        }
        const long ctaTiles = narrow ? (chunkM + 31) / 32 : tiles;      // K2 CTAs along the candidate axis
        K2Plan pl = plan;
        if (!narrow && tiles != chunkTiles) pl.G = pick_groups_wide(nb, tiles, sms);      // last, shorter chunk
        if (prof) IBO_CUDA_TRY(cudaEventRecord(m->ev[1], st));
        const int buf = (int)(ci & 1);
        uint8_t* const i8Slab = reinterpret_cast<uint8_t*>(m->dSlab) + (size_t)buf * (((i8SlabBytes + 7) / 8) * 8);
        double* const chunkPart = i8 ? m->dPart + (size_t)buf * i8PartDbl : m->dPart;
        if (i8pipe) {
            if (ci >= 2) IBO_CUDA_TRY(cudaStreamWaitEvent(m->stream2, m->evI8[2 + buf], 0));     // chunk ci-2 is done with this buffer
            launch_kstar_i8(m, dCand, tiles, M, m0, Mpad, i8Slab, chunkPart, m->stream2);
            IBO_CUDA_TRY(cudaEventRecord(m->evI8[buf], m->stream2));
            IBO_CUDA_TRY(cudaStreamWaitEvent(st, m->evI8[buf], 0));
        }
        else if (i8) launch_kstar_i8(m, dCand, tiles, M, m0, Mpad, i8Slab, chunkPart, st);
        else launch_kstar(m, dCand, m->dSlab, tiles, M, m0, st, inl);
        nlaunch++;
        if (vm) {
            launch_kstar(vm, dCand, vm->dSlab, tiles, M, m0, st, inl);
            nlaunch++;
        }
        if (prof) IBO_CUDA_TRY(cudaEventRecord(m->ev[2], st));
        if (i8) launch_trigemm_i8(m, tiles, Mpad, i8Slab, chunkPart, st);
        else if ((rc = launch_trigemm(m, narrow, pl, m->npb > 0, ctaTiles, Mpad, chunkM, st))) return rc;
        nlaunch++; nK2++;
        if (vm) {
            K2Plan plv = planV;
            if (!narrow && tiles != chunkTiles) plv.G = pick_groups_wide(vm->nb, tiles, sms);
            if ((rc = launch_trigemm(vm, narrow, plv, false, ctaTiles, Mpad, chunkM, st))) return rc;
            nlaunch++; nK2++;
        }
        if (prof) IBO_CUDA_TRY(cudaEventRecord(m->ev[3], st));
        EpiParams P;
        P.nbPart = nb * subs; P.d = m->d; P.N = m->N; P.acq = rq.acq; P.mode_py = (rq.flags & IBO_FLAG_MODE_PY) ? 1 : 0;
        P.npb = m->npb; P.want_p1 = m->npb > 0;
        P.M = M; P.m0 = m0; P.chunkM = chunkM; P.Mpad = Mpad;
        P.noise = m->noise; P.ymax = rq.ymax; P.parm = rq.parm; P.ptheta = m->ptheta;
        P.part = chunkPart; P.partVar = vm ? vm->dPart : nullptr; P.nbVarPart = vm ? vm->nb * (8 / planV.MT) : 0; P.MpadVar = Mpad;
        P.cand = dCand; P.pmeans = m->dPmeans; P.pbeta = m->dPbeta; P.plb = m->dPlb; P.pwidth = m->dPwidth;
        P.score = rq.want_score ? out : nullptr;
        P.mu = rq.want_mu ? out + M : nullptr;
        P.s2 = rq.want_s2 ? out + 2 * M : nullptr;
        P.want_argmax = rq.want_argmax ? 1 : 0;
        P.blkBest = m->dBlkBest; P.blkIdx = m->dBlkIdx; P.blk0 = blk0;
        P.guard_s2 = I8_GUARD_S2; P.flag = dFlag;
        P.rowLanes = !narrow ? 1 : (std::max(P.nbPart, P.nbVarPart) >= 64 ? 32 : (P.nbPart > 16 ? 8 : 1));
        const int cpb = 256 / P.rowLanes;
        const unsigned nblk = (unsigned)((chunkM + cpb - 1) / cpb);
        launch_ex(epilogue_kernel, dim3(nblk), dim3(256), 0, st, narrow && pdl_enabled() && !prof, P);
        nlaunch++;
        blk0 += nblk;
        if (i8pipe) IBO_CUDA_TRY(cudaEventRecord(m->evI8[2 + buf], st));
        ci++;
        if (prof) {
            IBO_CUDA_TRY(cudaEventRecord(m->ev[4], st));
            IBO_CUDA_TRY(cudaEventSynchronize(m->ev[4]));
            float a, b, c;
            cudaEventElapsedTime(&a, m->ev[1], m->ev[2]);
            cudaEventElapsedTime(&b, m->ev[2], m->ev[3]);
            cudaEventElapsedTime(&c, m->ev[3], m->ev[4]);
            tK1 += a; tK2 += b; tK3 += c;
        }
    }
    if (rq.acq >= 0 && rq.want_argmax) {
        argmax_final_kernel<<<1, 256, 0, st>>>(m->dBlkBest, m->dBlkIdx, blk0, out + 3 * M, reinterpret_cast<long long*>(out + 3 * M + 1));
        nlaunch++;
    }
    g_launches += nlaunch;
    int guarded = 0;
    if (guard) {
        // ---- guard pass: the flagged candidates (ascending index) are re-scored by the DMMA kernels and merged ----
        const int nblkG = (int)((M + 1023) / 1024);
        int* blkCnt = reinterpret_cast<int*>(dFlag + (((size_t)M + 7) / 8) * 8);
        int* dCount = blkCnt + nblkG;
        guard_count_kernel<<<nblkG, 256, 0, st>>>(dFlag, M, blkCnt);
        guard_scan_kernel<<<1, 256, 0, st>>>(blkCnt, nblkG, dCount);
        int count = 0;
        IBO_CUDA_TRY(cudaMemcpyAsync(&count, dCount, sizeof(int), cudaMemcpyDeviceToHost, st));
        IBO_CUDA_TRY(cudaStreamSynchronize(st));
        g_launches += 2;
        guarded = count;
        if (count > 0) {
            if ((rc = grow(&m->dGuardList, &m->guardListCap, (size_t)count * (1 + m->d) + 3 * (size_t)count + 2))) return rc;
            long long* list = reinterpret_cast<long long*>(m->dGuardList);
            double* gcand = m->dGuardList + count;
            double* gout = gcand + (size_t)count * m->d;
            guard_gather_kernel<<<nblkG, 256, 0, st>>>(dFlag, M, blkCnt, dCand, m->d, list, gcand);
            ScoreReq r2 = rq;
            // the throughput shape whatever the count: a guarded candidate then gets exactly the value the FP64 path gives it in any
            // wide batch -- its score stays a function of (model, x) only
            r2.flags = (rq.flags | IBO_FLAG_FP64 | FLAG_FORCE_WIDE) & ~(IBO_FLAG_INT8 | IBO_FLAG_PROFILE);
            if ((rc = score_device(m, gcand, count, r2, gout))) return rc;
            guard_scatter_kernel<<<(count + 255) / 256, 256, 0, st>>>(list, count, gout, out, M, rq.want_score ? 1 : 0, rq.want_mu ? 1 : 0,
                                                                       rq.want_s2 ? 1 : 0, (rq.acq >= 0 && rq.want_argmax) ? 1 : 0);
            g_launches += 2;
        }
    }
    m->lastGuarded = guarded;
    if (prof) {
        IBO_CUDA_TRY(cudaEventRecord(m->ev[5], st));
        IBO_CUDA_TRY(cudaEventSynchronize(m->ev[5]));
        float tot; cudaEventElapsedTime(&tot, m->ev[0], m->ev[5]);
        m->prof[0] = tK1; m->prof[1] = tK2; m->prof[2] = tK3; m->prof[3] = tot; m->prof[4] = (double)nlaunch; m->prof[5] = (double)nK2;
    }
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}

static int score_host(ibo_model* m, const double* Xs, long M, const ScoreReq& rq, double* scores, double* mu, double* s2,
                      double* best_score, long* best_idx) {
    if (!m || !Xs || M < 0) { set_error("bad argument"); return IBO_E_BADARG; }
    if (M == 0) { if (best_score) *best_score = -INFINITY; if (best_idx) *best_idx = -1; return IBO_OK; }
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    int rc;
    if ((rc = grow(&m->dCand, &m->candCap, (size_t)M * m->d))) return rc;
    cudaStream_t st = m->stream;
    // Small batches (DIRECT, gallery) are latency bound: stage through one pinned buffer so that the H2D and the
    // single D2H are plain DMA transfers instead of pageable copies (each of which costs a staging round trip).
    const size_t nin = (size_t)M * m->d, nout = 3 * (size_t)M + 2;
    const bool staged = (nin + nout) <= (1u << 17);
    double hb = 0; long long hi = -1;
    if (staged) {
        // Zero-copy results: the pinned buffer is mapped into the device address space and K3 / K4 write the results
        // straight into it (posted PCIe writes), so a call is: memcpy into pinned memory, one H2D DMA, 3-4 launches,
        // one stream synchronisation.
        if (m->pinnedCap < nin + nout) {
            IBO_CUDA_TRY(pinned_get(&m->hPinned));
            m->pinnedCap = 1u << 17;
        }
        std::memcpy(m->hPinned, Xs, sizeof(double) * nin);
        // candidates go to device memory with one small DMA (K1 reading them over PCIe costs ~15 us of dependent round trips);
        // the fused small-model kernel stages its tile with one parallel load and reads the mapped buffer directly
        const double* cand = m->dCand;
        const ibo_model* vmh = m->var_model;
        if (tiny_eligible(m, M)) cand = m->hPinned;
        else if (nin <= (size_t)CAND_INLINE && m->npb == 0 && kstar_uses_mma(m) && (!vmh || kstar_uses_mma(vmh)) &&
                 !i8_for_small_batch(m, M, rq.flags))
            cand = nullptr;          // the FP64 K1 takes the batch from its parameter buffer (K3 reads candidates only for a prior mean)
        else IBO_CUDA_TRY(cudaMemcpyAsync(m->dCand, m->hPinned, sizeof(double) * nin, cudaMemcpyHostToDevice, st));
        double* ho = m->hPinned + nin;
        if ((rc = score_device(m, cand, M, rq, ho, m->hPinned))) return rc;
        IBO_CUDA_TRY(cudaStreamSynchronize(st));
        if (scores) std::memcpy(scores, ho, sizeof(double) * M);
        if (mu) std::memcpy(mu, ho + M, sizeof(double) * M);
        if (s2) std::memcpy(s2, ho + 2 * M, sizeof(double) * M);
        if (rq.acq >= 0 && rq.want_argmax) { hb = ho[3 * M]; std::memcpy(&hi, &ho[3 * M + 1], 8); }
    } else {
        if ((rc = score_device(m, m->dCand, M, rq, nullptr, nullptr, Xs))) return rc;
        if (scores) IBO_CUDA_TRY(cudaMemcpyAsync(scores, m->dOut, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
        if (mu) IBO_CUDA_TRY(cudaMemcpyAsync(mu, m->dOut + M, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
        if (s2) IBO_CUDA_TRY(cudaMemcpyAsync(s2, m->dOut + 2 * M, sizeof(double) * M, cudaMemcpyDeviceToHost, st));
        if (rq.acq >= 0 && rq.want_argmax) {
            IBO_CUDA_TRY(cudaMemcpyAsync(&hb, m->dOut + 3 * M, sizeof(double), cudaMemcpyDeviceToHost, st));
            IBO_CUDA_TRY(cudaMemcpyAsync(&hi, m->dOut + 3 * M + 1, sizeof(long long), cudaMemcpyDeviceToHost, st));
        }
        IBO_CUDA_TRY(cudaStreamSynchronize(st));
    }
    if (best_score) *best_score = hb;
    if (best_idx) *best_idx = (long)hi;
    return IBO_OK;
}

__global__ void debug_exp_kernel(const double* __restrict__ x, long n, double* __restrict__ fast, double* __restrict__ ref) {
    long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
    if (i < n) { fast[i] = exp_nonpos(x[i]); ref[i] = exp(x[i]); }
}

// used by the DIRECT objective (direct.cpp): negated acquisition for n points
// the arithmetic a DIRECT batch of n points gets (sharded DIRECT asks with the size of the full batch and forces the answer on
// every rank's slice): 1 = INT8 path, 0 = FP64 kernels
int batch_uses_i8(ibo_model* m, long n, int flags) {
    if (n > narrow_threshold()) return i8_eligible(m, flags) ? 1 : 0;
    return i8_for_small_batch(m, n, flags) ? 1 : 0;
}
int eval_neg_acq(ibo_model* m, const double* Xs, long n, int acq, double ymax, double parm, int flags, double* y) {
    ScoreReq rq{acq, ymax, parm, flags, true, false, false};
    rq.want_argmax = false;      // DIRECT consumes every value; the argmax kernels would be wasted launches
    int rc = score_host(m, Xs, n, rq, y, nullptr, nullptr, nullptr, nullptr);
    if (rc) return rc;
    for (long i = 0; i < n; i++) y[i] = -y[i];
    return IBO_OK;
}

}  // namespace ibo

using namespace ibo;

extern "C" int ibo_posterior_batch(ibo_model* m, const double* Xs, long M, int flags, double* mu, double* s2) {
    ScoreReq rq{-1, 0.0, 0.0, flags, false, mu != nullptr, s2 != nullptr};
    return score_host(m, Xs, M, rq, nullptr, mu, s2, nullptr, nullptr);
}

extern "C" int ibo_score_batch(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags,
                               double* scores, double* mu, double* s2, double* best_score, long* best_idx) {
    if (acq < 0 || acq > 2) { set_error("unknown acquisition function"); return IBO_E_BADARG; }
    ScoreReq rq{acq, ymax, parm, flags, scores != nullptr, mu != nullptr, s2 != nullptr};
    return score_host(m, Xs, M, rq, scores, mu, s2, best_score, best_idx);
}

extern "C" int ibo_cands_create(ibo_model* m, const double* Xs, long M, ibo_cands** out) {
    if (!m || !Xs || M < 1 || !out) { set_error("bad argument"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    ibo_cands* c = new ibo_cands();
    c->owner = m; c->M = M;
    cudaError_t e = cudaMalloc(&c->dX, sizeof(double) * (size_t)M * m->d);
    if (e != cudaSuccess) { delete c; set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); cudaGetLastError(); return IBO_E_NOMEM; }
    e = cudaMemcpy(c->dX, Xs, sizeof(double) * (size_t)M * m->d, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(c->dX); delete c; set_error(std::string("cudaMemcpy: ") + cudaGetErrorString(e)); return IBO_E_CUDA; }
    *out = c;
    return IBO_OK;
}

extern "C" int ibo_cands_destroy(ibo_cands* c) {
    if (!c) return IBO_OK;
    if (c->owner) cudaSetDevice(c->owner->device);
    if (c->dX) cudaFree(c->dX);
    delete c;
    return IBO_OK;
}

extern "C" int ibo_score_resident(ibo_model* m, ibo_cands* c, int acq, double ymax, double parm, int flags,
                                  double* scores_host, double* best_score, long* best_idx, float* ms_device) {
    if (!m || !c || c->owner != m || acq < 0 || acq > 2) { set_error("bad argument"); return IBO_E_BADARG; }
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    ScoreReq rq{acq, ymax, parm, flags, true, false, false};
    IBO_CUDA_TRY(cudaEventRecord(m->ev[6], st));
    int rc = score_device(m, c->dX, c->M, rq);
    if (rc) return rc;
    IBO_CUDA_TRY(cudaEventRecord(m->ev[7], st));
    double hb = 0; long long hi = -1;
    if (scores_host) IBO_CUDA_TRY(cudaMemcpyAsync(scores_host, m->dOut, sizeof(double) * c->M, cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(&hb, m->dOut + 3 * c->M, sizeof(double), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaMemcpyAsync(&hi, m->dOut + 3 * c->M + 1, sizeof(long long), cudaMemcpyDeviceToHost, st));
    IBO_CUDA_TRY(cudaStreamSynchronize(st));
    if (ms_device) { float ms = 0; cudaEventElapsedTime(&ms, m->ev[6], m->ev[7]); *ms_device = ms; }
    if (best_score) *best_score = hb;
    if (best_idx) *best_idx = (long)hi;
    return IBO_OK;
}

extern "C" int ibo_get_profile(ibo_model* m, double* out6) {
    if (!m || !out6) { set_error("bad argument"); return IBO_E_BADARG; }
    for (int i = 0; i < 6; i++) out6[i] = m->prof[i];
    return IBO_OK;
}

// live INT8 tensor-pipe peaks of `device` in TOP/s (int8 multiply-adds x 2), tcgen05.mma kind::i8 issue rate:
//   burst      best of a few ~2 ms launches with near-constant operand bytes -- the pipe's ceiling at the full SM clock
//   sustained  pseudo-random operand bytes, launches back to back for `seconds`; the rate over the second half of that time --
//              what the power cap lets a dense INT8 kernel with real data sustain (the denominator for a kernel timed inside a long step)
extern "C" int ibo_i8_peak2(int device, double seconds, double* burst_tops, double* sustained_tops) {
    if (ibo_device_count() <= 0) { set_error("no CUDA device available (libibo_b200 has no CPU fallback)"); return IBO_E_CUDA; }
    IBO_CUDA_TRY(cudaSetDevice(device));
    const int sms = dev_info(device).sms, iters = 4000, smem = (128 + 256) * 128;
    IBO_CUDA_TRY(cudaFuncSetAttribute(i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int* sink = nullptr;
    IBO_CUDA_TRY(cudaMalloc(&sink, sizeof(int) * 128 * sms));
    cudaEvent_t e0, e1;
    IBO_CUDA_TRY(cudaEventCreate(&e0));
    IBO_CUDA_TRY(cudaEventCreate(&e1));
    const double ops = 2.0 * 128 * 256 * 128 * (double)iters * sms;
    if (burst_tops) {
        double best = 0;
        for (int r = 0; r < 5; r++) {
            IBO_CUDA_TRY(cudaEventRecord(e0));
            i8_peak_kernel<<<sms, 128, smem>>>(iters, 0, sink);
            IBO_CUDA_TRY(cudaEventRecord(e1));
            IBO_CUDA_TRY(cudaEventSynchronize(e1));
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (r >= 1) best = std::max(best, ops / (ms * 1e-3) / 1e12);
            g_launches++;
        }
        *burst_tops = best;
    }
    if (sustained_tops) {
        // launches of 10 x iters (~20 ms) back to back; timed over the second half of the run
        const int big = 10 * iters;
        int nl = 0, nhalf = 0;
        float elapsed = 0;
        IBO_CUDA_TRY(cudaEventRecord(e0));
        while (elapsed < 500.0f * seconds) {             // first half: reach the steady clock
            i8_peak_kernel<<<sms, 128, smem>>>(big, 1, sink);
            IBO_CUDA_TRY(cudaEventRecord(e1));
            IBO_CUDA_TRY(cudaEventSynchronize(e1));
            cudaEventElapsedTime(&elapsed, e0, e1);
            nl++;
        }
        nhalf = std::max(nl, 1);
        IBO_CUDA_TRY(cudaEventRecord(e0));
        for (int r = 0; r < nhalf; r++) i8_peak_kernel<<<sms, 128, smem>>>(big, 1, sink);
        IBO_CUDA_TRY(cudaEventRecord(e1));
        IBO_CUDA_TRY(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&elapsed, e0, e1);
        *sustained_tops = 10.0 * ops * nhalf / (elapsed * 1e-3) / 1e12;
        g_launches += nl + nhalf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(sink);
    IBO_CUDA_TRY(cudaGetLastError());
    return IBO_OK;
}
extern "C" int ibo_i8_peak(int device, double* tops) {
    if (!tops) { set_error("bad argument"); return IBO_E_BADARG; }
    return ibo_i8_peak2(device, 0.0, tops, nullptr);
}

// test hook: K1's exp_nonpos next to libdevice exp for n arguments <= 0 (host arrays)
extern "C" int ibo_debug_exp(int device, const double* x, long n, double* out_fast, double* out_ref) {
    if (!x || !out_fast || !out_ref || n < 1) { set_error("bad argument"); return IBO_E_BADARG; }
    if (ibo_device_count() <= 0) { set_error("no CUDA device available (libibo_b200 has no CPU fallback)"); return IBO_E_CUDA; }
    IBO_CUDA_TRY(cudaSetDevice(device));
    double* d = nullptr;
    IBO_CUDA_TRY(cudaMalloc(&d, sizeof(double) * 3 * (size_t)n));
    cudaError_t e = cudaMemcpy(d, x, sizeof(double) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        debug_exp_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d, n, d + n, d + 2 * n);
        g_launches++;
        e = cudaMemcpy(out_fast, d + n, sizeof(double) * n, cudaMemcpyDeviceToHost);
    }
    if (e == cudaSuccess) e = cudaMemcpy(out_ref, d + 2 * n, sizeof(double) * n, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) { set_error(std::string("ibo_debug_exp: ") + cudaGetErrorString(e)); return IBO_E_CUDA; }
    return IBO_OK;
}
