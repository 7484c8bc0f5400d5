// The wide-batch scoring path: K2's FP64 triangular GEMM V = W K* evaluated on the INT8 tensor cores (tcgen05.mma kind::i8,
// INT32 accumulators in TMEM) through an Ozaki-style split of both operands into base-256 digits, and the K1 / model-side
// kernels that feed it.  tcgen05 has no f64 kind, so the DMMA path (score.cu) is pinned at 37 TF/s; the INT8 pipe issues
// 4.5 POP/s, and 28 exact digit products per FP64 product leave a ~4x higher ceiling at the accuracy of the FP64 path:
// against an extended-precision evaluation of sum_r V_r^2 with the same W, the FP64 GEMM is off by ~2e-15 and this scheme by
// ~4e-15 (oracle/int8_model.py, tests/test_int8_model.py; device: tests/test_gpu_int8.py).
//
//   W  (row r) = 2^e_r sum_{t=1..7} 2^(-8t) A_t     A_t balanced base-256 digits of rint(w 2^(56 - e_r)),  |w| 2^-e_r < 1/4
//   K*         = 1/2 + 2 sum_{u=1..7} 2^(-8u) B_u   B_u balanced base-256 digits of rint((k / sf2 - 1/2) 2^55)
//   V          = 2 sf2 2^e_r sum_{g=2..8} 2^(-8g) D_g + sf2/2 sum_k W[r, k],     D_g = sum_{t+u=g} A_t B_u^T   (exact in INT32)
//
// Pairs with t + u > 8 are dropped (below 2^-64 of the row scale); pairs with equal t + u share an accumulator: seven groups
// of 128 x 64 INT32 = 448 of the 512 TMEM columns.  The B digits of a candidate tile are consecutive 64-row blocks of one
// K-major operand, so A_t x [B_u0 .. B_u0+n-1] is ONE 128 x 64n x 32 instruction whose 64-column output blocks land on the
// accumulators of groups t+u0 .. t+u0+n-1: 10 instructions per 32-deep k-step instead of 28.
//
// Operand feed.  Every operand is in shared memory: per 32-deep k-step the producer issues two contiguous bulk copies into a
// 4-stage ring, the seven W digits of the row-block (28 KiB) and the seven K* digits of the candidate tile (14 KiB), and the ten
// MMAs read both through shared-memory descriptors.  A k-step moves 138 KiB through the SM's 128 B/clk shared-memory pipe (10 A
// reads of 4 KiB, 28 B reads of 2 KiB, 42 KiB of bulk-copy fill) against 896 clk of tensor work, but under the 1 kW power cap
// the lowered SM clock bounds the kernel (0.93 of the sustained INT8 peak).  A TMEM feed for W digits 1..4 was built, measured
// 6-13 % slower under the power cap, and removed (profiles/r02_int8_k2.md).
//
// sigma^2 only needs sum_r V_r^2 per candidate; the posterior mean is k* . alpha (alpha = W^T W Y, plain FP64 dot products
// inside K1, written to the partial-sum planes K2 would fill with V . beta), so K3 is the DMMA path's.
#pragma once

namespace ibo {

constexpr int I8_S = 7;                          // digits per operand
constexpr int I8_NT = 64;                        // candidates per tile
constexpr int I8_A_SLICE = 128 * 32;             // bytes of one W digit of a k-step: 128 rows x 32 k
constexpr int I8_B_SLICE = I8_NT * 32;           // bytes of one K* digit of a k-step: 64 candidates x 32 k
constexpr int I8_A_STAGE = I8_S * I8_A_SLICE;                // 28672
constexpr int I8_B_STAGE = I8_S * I8_B_SLICE;                // 14336
constexpr int I8_STAGES = 4;
constexpr int I8_SMEM = I8_STAGES * (I8_A_STAGE + I8_B_STAGE) + 4 * 64 * 8 + 32 * 8;
constexpr int I8_THREADS = 320;                  // 10 warps, 31 K registers: leaves room for two K1 CTAs of the next chunk beside a
                                                 // resident K2 CTA
// warp 0: bulk-copy producer, warp 1: TMEM owner + MMA issuer, warps 2-9: epilogue (warp w drains TMEM lanes 32 (w % 4) .. + 31
// for candidates 32 ((w - 2) / 4) .. + 31 of the tile)
constexpr int I8_EPI_WARP0 = 2;
// sigma^2 below this value is not taken from the integer path: the candidate is re-scored by the DMMA kernels in the same
// call (score.cu: guard pass).  The scheme's absolute error on sum v^2 is ~1e-14 (1 + noise), so above the threshold its
// relative effect on sigma^2 stays below 1e-11; a model with noise >= 2^-10 never gets there (sigma^2 >= noise).
constexpr double I8_GUARD_S2 = 0.0009765625;

// byte offset of element (row r, k) in a [rows x 32] canonical tile (no-swizzle K-major: 8 x 16-byte core matrices, the two
// k chunks of a row group 128 B apart, row groups 256 B apart)
__host__ __device__ inline uint32_t i8_canon(int r, int k) { return (uint32_t)((((r >> 3) * 2 + (k >> 4)) << 7) + ((r & 7) << 4) + (k & 15)); }
// k-steps that precede row-block i in the packed W digits (row-block i owns 4 (i + 1) steps)
__host__ __device__ inline size_t i8_steps_before(int i) { return (size_t)4 * ((size_t)i * (i + 1) / 2); }

// ---- tcgen05 / TMEM primitives (encodings checked on the device by tools/research/umma_i8_probe.cu) ----------------------
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t addr) {        // LBO = 128 B, SBO = 256 B, version 1, no swizzle
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ constexpr uint32_t umma_idesc_i8(int M, int N) { // S32 accumulator, signed 8-bit A / B, K-major
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {               // arrives on `bar` once every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_nowait(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// One lane of a converged warp (CUTLASS's elect_one_sync).  tcgen05.mma / tcgen05.commit / bulk copies run on the warp-uniform
// datapath: under a plain `lane == 0` test the compiler cannot prove that a single thread is active and wraps EVERY such
// instruction in an elect / vote loop (~150 issue slots per k-step: the MMA issuer, not the tensor pipe, was the bound of the
// first versions of this kernel); under elect.sync it emits them back to back.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------------------------------------
// model side: per-row power-of-two scale of W and its seven digits
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) i8_rowscale_kernel(const double* __restrict__ W, int Np, int N, double sf2,
                                                          double* __restrict__ rowScale) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= Np) return;
    double mx = 0.0, sum = 0.0;
    for (int k = lane; k <= row; k += 32) {
        const double w = W[(size_t)row * Np + k];
        mx = fmax(mx, fabs(w));
        if (k < N) sum += w;
    }
    for (int o = 16; o; o >>= 1) { mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o)); sum += __shfl_xor_sync(0xffffffffu, sum, o); }
    // 2^e with |w| / 2^e < 1/4 for the whole row: the top balanced digit stays within [-64, 64].
    // slot 0: slicing scale 2^e; slot 1: 2 * 2^e * sf2, the factor that turns the assembled integer sum into v (K* is sliced as
    // (k / sf2 - 1/2) / 2); slot 2: sf2 / 2 * sum_{k < N} W[row][k], the constant the shift by 1/2 leaves behind
    if (lane == 0) {
        const double sc = mx > 0.0 ? scalbn(1.0, ilogb(mx) + 3) : 1.0;
        rowScale[row] = sc;
        rowScale[Np + row] = 2.0 * sc * sf2;
        rowScale[2 * Np + row] = 0.5 * sf2 * sum;
    }
}

// digits 1..7 -> Ws: per k-step [digit][canonical 128 x 32 tile] (one contiguous bulk copy per stage)
__global__ void __launch_bounds__(256) i8_slice_w_kernel(const double* __restrict__ W, const double* __restrict__ rowScale, int Np,
                                                         uint8_t* __restrict__ Ws) {
    const int j = blockIdx.x, i = blockIdx.y;                 // k-step, row-block
    if (j >= (i + 1) * 4) return;
    const int r = threadIdx.x & 127, c16 = threadIdx.x >> 7;  // row of the block, 16-byte k chunk of the step
    const int row = i * 128 + r, k0 = j * 32 + c16 * 16;
    const double inv = 1.0 / rowScale[row];                   // power of two: exact
    long long q[16];
#pragma unroll
    for (int kk = 0; kk < 16; kk++) {
        const double w = W[(size_t)row * Np + k0 + kk];        // exact zeros above the diagonal
        q[kk] = __double2ll_rn(w * inv * 72057594037927936.0); // 2^56, round to nearest; |w| * inv < 1/4
    }
    const size_t step = i8_steps_before(i) + j;
    // balanced digits, least significant first: d_t in [-128, 127] for t = 7 .. 2, what is left (|d_1| <= 64) is the top digit.
    // Zero-mean digits make the dropped pairs (t + u > 8) a zero-mean error that grows like sqrt(N), not N.
#pragma unroll
    for (int t = I8_S; t >= 1; t--) {
        uint32_t w4[4];
#pragma unroll
        for (int v = 0; v < 4; v++) {
            uint32_t word = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int kk = v * 4 + b;
                long long dgt;
                if (t > 1) { dgt = ((q[kk] + 128) & 255) - 128; q[kk] = (q[kk] - dgt) >> 8; }
                else dgt = q[kk];
                word |= ((uint32_t)(int)dgt & 0xffu) << (8 * b);
            }
            w4[v] = word;
        }
        uint8_t* dst = Ws + step * I8_A_STAGE + (size_t)(t - 1) * I8_A_SLICE + i8_canon(r, c16 * 16);
        *reinterpret_cast<uint4*>(dst) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    }
}

// ---------------------------------------------------------------------------------------------
// K1 (int8): one CTA = (64-candidate tile T, row-block i); thread = (candidate c, k-step of the block).  Kernel values from
// direct differences, (k - 1/2) sliced from a 55-bit fixed-point image, 16 bytes (one core-matrix row) per store; the partial
// dot products k* . alphaY / k* . alpha1 of the block go to planes 1 / 2 of `part` (what the DMMA K2 writes as V . beta).
// ---------------------------------------------------------------------------------------------
template <int KC, int DMAX>
__global__ void __launch_bounds__(256, (DMAX <= 8 ? 4 : (DMAX <= 16 ? 3 : 2))) kstar_i8_kernel(const double* __restrict__ Xt, const double* __restrict__ cand,
                                                       const double* __restrict__ inv_theta, const double* __restrict__ center,
                                                       const double* __restrict__ alphaY, const double* __restrict__ alpha1,
                                                       uint8_t* __restrict__ Ki8, double* __restrict__ part,
                                                       int N, int d, int nb, long M, long m0, long Mpad, double sf2, int want_p1) {
    // DMAX >= d (even): the dimension loops have a compile-time length, the thread's candidate lives in registers and the
    // training rows (zero padded to DMAX) are read with 16-byte broadcast loads
    __shared__ __align__(16) double sX[128 * DMAX];
    __shared__ double sAy[128], sA1[128], red[512];
    const int T = blockIdx.x, i = blockIdx.y, tid = threadIdx.x;
    for (int idx = tid; idx < 128 * DMAX; idx += 256) {
        const int r = idx / DMAX, j = idx - r * DMAX;
        sX[idx] = j < d ? Xt[(size_t)(i * 128 + r) * d + j] : 0.0;
    }
    if (tid < 128) { sAy[tid] = alphaY[i * 128 + tid]; sA1[tid] = alpha1[i * 128 + tid]; }
    const int c = tid & 63, kg = tid >> 6;
    double xc[DMAX];
    {
        long cg = m0 + (long)T * 64 + c;
        if (cg >= M) cg = M - 1;
#pragma unroll
        for (int j = 0; j < DMAX; j++) xc[j] = j < d ? cand[(size_t)cg * d + j] * inv_theta[j] - center[j] : 0.0;
    }
    __syncthreads();
    double sy = 0.0, s1 = 0.0;
    uint8_t* dst0 = Ki8 + ((size_t)T * (nb * 4) + (size_t)i * 4 + kg) * I8_B_STAGE;
#pragma unroll 1
    for (int c16 = 0; c16 < 2; c16++) {
        // Balanced base-256 digits of (v - 1/2) 2^55, four values at a time: adding 128 to each of the six low bytes (one 64-bit add,
        // carries included) turns every byte into digit + 128, the xor takes the 128 off again in two's complement; byte 6 is then
        // the signed top digit (|q| <= 2^54, so it fits).  Digit t is byte 7 - t.  A 4 x 4 byte transpose (8 PRMT per four values
        // and word half) lines the bytes of one digit up: sixteen values give the 16-byte store of one core-matrix row per digit.
        uint32_t wd[7][4];
#pragma unroll
        for (int v = 0; v < 4; v++) {
            uint32_t lo[4], hi[4];
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int k = kg * 32 + c16 * 16 + v * 4 + b;
                const double2* xr = reinterpret_cast<const double2*>(sX + k * DMAX);
                double r2a = 0.0, r2b = 0.0;
#pragma unroll
                for (int j2 = 0; j2 < DMAX / 2; j2++) {
                    const double2 x2 = xr[j2];
                    const double da = x2.x - xc[2 * j2], db = x2.y - xc[2 * j2 + 1];
                    r2a = fma(da, da, r2a);
                    r2b = fma(db, db, r2b);
                }
                const bool live = (i * 128 + k) < N;
                const double val = live ? cov_r2_t<KC>(1.0, r2a + r2b) : 0.0;   // in [0, 1]
                sy = fma(val, sAy[k], sy);
                s1 = fma(val, sA1[k], s1);
                // (v - 1/2) / 2 in [-1/4, 1/4] at 56 fractional bits, signed; rows beyond N contribute nothing (W is zero there)
                const long long q = live ? __double2ll_rn((val - 0.5) * 36028797018963968.0) : 0ll;     // 2^55
                const unsigned long long u = ((unsigned long long)q + 0x0000808080808080ull) ^ 0x0000808080808080ull;
                lo[b] = (uint32_t)u; hi[b] = (uint32_t)(u >> 32);
            }
            const uint32_t l01 = __byte_perm(lo[0], lo[1], 0x5140), l23 = __byte_perm(lo[2], lo[3], 0x5140);
            const uint32_t m01 = __byte_perm(lo[0], lo[1], 0x7362), m23 = __byte_perm(lo[2], lo[3], 0x7362);
            const uint32_t h01 = __byte_perm(hi[0], hi[1], 0x5140), h23 = __byte_perm(hi[2], hi[3], 0x5140);
            const uint32_t g01 = __byte_perm(hi[0], hi[1], 0x7362), g23 = __byte_perm(hi[2], hi[3], 0x7362);
            wd[6][v] = __byte_perm(l01, l23, 0x5410);      // byte 0: digit 7 (least significant)
            wd[5][v] = __byte_perm(l01, l23, 0x7632);      // byte 1: digit 6
            wd[4][v] = __byte_perm(m01, m23, 0x5410);      // byte 2: digit 5
            wd[3][v] = __byte_perm(m01, m23, 0x7632);      // byte 3: digit 4
            wd[2][v] = __byte_perm(h01, h23, 0x5410);      // byte 4: digit 3
            wd[1][v] = __byte_perm(h01, h23, 0x7632);      // byte 5: digit 2
            wd[0][v] = __byte_perm(g01, g23, 0x5410);      // byte 6: digit 1 (most significant, takes the rest)
        }
        uint8_t* dst = dst0 + i8_canon(c, c16 * 16);
#pragma unroll
        for (int t = I8_S; t >= 1; t--)
            *reinterpret_cast<uint4*>(dst + (size_t)(t - 1) * I8_B_SLICE) = make_uint4(wd[t - 1][0], wd[t - 1][1], wd[t - 1][2], wd[t - 1][3]);
    }
    red[kg * 64 + c] = sy;
    red[256 + kg * 64 + c] = s1;
    __syncthreads();
    if (tid < 64) {
        const size_t plane = (size_t)nb * Mpad;
        const size_t o = (size_t)i * Mpad + (size_t)T * 64 + tid;
        part[plane + o] = sf2 * (((red[tid] + red[64 + tid]) + red[128 + tid]) + red[192 + tid]);
        if (want_p1) part[2 * plane + o] = sf2 * (((red[256 + tid] + red[320 + tid]) + red[384 + tid]) + red[448 + tid]);
    }
}

// ---------------------------------------------------------------------------------------------
// K2 (int8): CTA = (row-block group g of G, 64-candidate tile T).  Each row-block is a full sweep over its 4 (i + 1) k-steps
// into the seven group accumulators, then the epilogue warps assemble V in FP64 and reduce sum_r V_r^2 per candidate in a
// fixed order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(I8_THREADS, 2) trigemm_i8_kernel(const uint8_t* __restrict__ Ws, const uint8_t* __restrict__ Ki8,
                                                                   const double* __restrict__ rowScaleSf, double* __restrict__ part,
                                                                   int nb, long Mpad) {
    // rowScaleSf[row]: the factor that turns the assembled integer sum into v; rowScaleSf[Np + row]: the additive constant
    constexpr int STAGES = I8_STAGES;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sA = smem;                                          // [stage][7][128 x 32]   W digits 1..7
    uint8_t* sB = smem + STAGES * I8_A_STAGE;                    // [stage][7][64 x 32]    K* digits 1..7
    double* red = reinterpret_cast<double*>(smem + STAGES * (I8_A_STAGE + I8_B_STAGE));     // [4][64]
    uint64_t* full = reinterpret_cast<uint64_t*>(red + 4 * 64);
    uint64_t* empty = full + STAGES;
    uint64_t* tfull = empty + STAGES;
    uint64_t* tempty = tfull + 1;
    uint32_t* tbase = reinterpret_cast<uint32_t*>(tempty + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = blockIdx.x, G = gridDim.x, T = blockIdx.y;
    if (tid == 0) {
        // full[s]: the producer's expect-tx arrival (+ the bytes of its two bulk copies); empty[s]: one tcgen05.commit -- the MMAs
        // of the k-step have read the stage
        for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(tfull, 1);
        mbar_init(tempty, 8);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 1) {
        // 512 columns: the smallest allocation that holds the 448 accumulator columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tbase)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tb = *tbase;

    const int rounds = (nb + G - 1) / G;
    if (warp == 0) {
        // ---------------- producer (one elected lane): two contiguous bulk copies per k-step ----------------
        if (elect_one()) {
            int s = 0; uint32_t ph = 0;
            const uint8_t* Bb = Ki8 + (size_t)T * (nb * 4) * I8_B_STAGE;
            for (int r = 0; r < rounds; r++) {
                const int idx = r * G + ((r & 1) ? (G - 1 - g) : g);
                if (idx >= nb) continue;
                const int i = nb - 1 - idx, nk = (i + 1) * 4;
                const uint8_t* Ab = Ws + i8_steps_before(i) * I8_A_STAGE;
                for (int j = 0; j < nk; j++) {
                    mbar_wait(&empty[s], ph ^ 1);
                    mbar_arrive_expect_tx(&full[s], I8_A_STAGE + I8_B_STAGE);
                    bulk_g2s(sA + s * I8_A_STAGE, Ab + (size_t)j * I8_A_STAGE, I8_A_STAGE, &full[s]);
                    bulk_g2s(sB + s * I8_B_STAGE, Bb + (size_t)j * I8_B_STAGE, I8_B_STAGE, &full[s]);
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer (one elected lane): the loop is its whole critical path -- one barrier wait, ten MMAs and
        // one commit per k-step and nothing else ----------------
        if (elect_one()) {
            int s = 0; uint32_t ph = 0; int rb = 0;
            for (int r = 0; r < rounds; r++) {
                const int idx = r * G + ((r & 1) ? (G - 1 - g) : g);
                if (idx >= nb) continue;
                const int nk = (nb - idx) * 4;
                mbar_wait(tempty, (uint32_t)(rb & 1) ^ 1);          // the epilogue has drained the previous row-block's accumulators
                for (int j = 0; j < nk; j++) {
                    mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint64_t da = umma_smem_desc(smem_u32(sA + s * I8_A_STAGE)), db = umma_smem_desc(smem_u32(sB + s * I8_B_STAGE));
                    const uint32_t first = j == 0 ? 0u : 1u;
                    // digit t of W against K* digits u0 .. u0+n-1: accumulator columns 64 (t + u0 - 2), N = 64 n
                    // (descriptor + (bytes >> 4): the start-address field counts 16-byte units and cannot carry here)
#define I8_MMA(t, u0, n, acc) umma_i8(tb + 64u * ((t) + (u0) - 2), da + (uint64_t)((((t) - 1) * I8_A_SLICE) >> 4), \
                                      db + (uint64_t)((((u0) - 1) * I8_B_SLICE) >> 4), umma_idesc_i8(128, 64 * (n)), acc)
                    I8_MMA(1, 1, 4, first); I8_MMA(1, 5, 3, first);          // the two t = 1 instructions touch groups 2..8 first
                    I8_MMA(2, 1, 4, 1u);    I8_MMA(2, 5, 2, 1u);
                    I8_MMA(3, 1, 4, 1u);    I8_MMA(3, 5, 1, 1u);
                    I8_MMA(4, 1, 4, 1u);
                    I8_MMA(5, 1, 3, 1u);
                    I8_MMA(6, 1, 2, 1u);
                    I8_MMA(7, 1, 1, 1u);
#undef I8_MMA
                    umma_commit(&empty[s]);                          // the stage is free once these MMAs have read it
                    if (++s == STAGES) { s = 0; ph ^= 1; }
                }
                umma_commit(tfull);                                  // accumulators of this row-block complete
                rb++;
            }
        }
    } else {
        // ---------------- epilogue: warp w drains TMEM lanes 32 (w % 4) .. + 31 (rows) x candidates 32 h .. + 31, h = (w - 2) / 4 ----------------
        const int qd = warp & 3, hf = (warp - I8_EPI_WARP0) >> 2, et = (warp - I8_EPI_WARP0) * 32 + lane;
        const uint32_t tq = tb + ((uint32_t)(qd * 32) << 16) + 32u * hf;
        int rb = 0;
        for (int r = 0; r < rounds; r++) {
            const int idx = r * G + ((r & 1) ? (G - 1 - g) : g);
            if (idx >= nb) continue;
            const int i = nb - 1 - idx;
            const double rs = rowScaleSf[i * 128 + qd * 32 + lane];
            const double rc = rowScaleSf[(size_t)nb * 128 + i * 128 + qd * 32 + lane];
            mbar_wait_warp(tfull, (uint32_t)(rb & 1));
            tc_fence_after();
#pragma unroll 1
            for (int c16 = 0; c16 < 2; c16++) {
                double sq[16];
#pragma unroll
                for (int c4 = 0; c4 < 4; c4++) {
                    uint32_t D[I8_S][4];
#pragma unroll
                    for (int gq = 0; gq < I8_S; gq++) tmem_ld4_nowait(tq + 64u * gq + 16u * c16 + 4u * c4, D[gq]);
                    tmem_ld_wait();
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        // groups 2..4 at 2^-32, 5..7 at 2^-56, 8 at 2^-64: two exact INT64 partial sums, three roundings
                        const long long hi = (long long)(int)D[0][e] * 65536 + (long long)(int)D[1][e] * 256 + (long long)(int)D[2][e];
                        const long long mid = (long long)(int)D[3][e] * 65536 + (long long)(int)D[4][e] * 256 + (long long)(int)D[5][e];
                        const double lo = (double)(int)D[6][e] * 5.42101086242752217003726400434970855712890625e-20;    // 2^-64
                        double v = fma((double)hi, 2.3283064365386962890625e-10,                                        // 2^-32
                                       fma((double)mid, 1.387778780781445675529539585113525390625e-17, lo));           // 2^-56
                        v = fma(v, rs, rc);
                        sq[c4 * 4 + e] = v * v;
                    }
                }
                // Sum over the warp's 32 rows by recursive halving: at distance o a lane keeps the candidates whose index bit matches its
                // lane bit and hands the others to its partner -- 15 exchanges + one butterfly step for 16 candidates instead of 80.
                // Every partial sum is x_self + x_partner of the SAME balanced tree as a full xor butterfly (addition commutes), so the
                // result is bit-identical to reducing each candidate with five shuffles.
#pragma unroll
                for (int lv = 0; lv < 4; lv++) {
                    const int o = 16 >> lv, cnt = 8 >> lv;              // lane bit o selects which half of the remaining candidates it keeps
                    const bool up = (lane & o) != 0;
#pragma unroll
                    for (int x = 0; x < cnt; x++) {
                        const double mine = up ? sq[x + cnt] : sq[x], theirs = up ? sq[x] : sq[x + cnt];
                        sq[x] = mine + __shfl_xor_sync(0xffffffffu, theirs, o);
                    }
                }
                sq[0] += __shfl_xor_sync(0xffffffffu, sq[0], 1);
                // lane bits (16, 8, 4, 2) = candidate bits (8, 4, 2, 1) of this batch of 16
                if (!(lane & 1)) red[qd * 64 + hf * 32 + c16 * 16 + (lane >> 1)] = sq[0];
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);                      // 8 arrivals: the accumulators may be overwritten
            named_bar_sync(1, 256);
            if (et < 64) {
                // TMEM lane quarter q holds rows 32 q .. 32 q + 31: ascending row order
                part[(size_t)i * Mpad + (size_t)T * 64 + et] = ((red[et] + red[64 + et]) + red[128 + et]) + red[192 + et];
            }
            named_bar_sync(1, 256);
            rb++;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tb), "r"(512u) : "memory");
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// builds (once per model state) the packed digits of W, the row scales / constants and alpha
static int ensure_i8(ibo_model* m) {
    if (m->i8Valid) return IBO_OK;
    const int Np = m->Np, nb = m->nb;
    cudaStream_t st = m->stream;
    for (double** p : {&m->dAlphaY, &m->dAlpha1, &m->dWi8s, &m->dRowScale}) if (*p) { pool_free(*p); *p = nullptr; }
    IBO_CUDA_TRY(pool_malloc((void**)&m->dAlphaY, sizeof(double) * Np));
    IBO_CUDA_TRY(pool_malloc((void**)&m->dAlpha1, sizeof(double) * Np));
    launch_tri_matvec_t(m->dW, m->dBetaY, m->dAlphaY, Np, Np, st);       // alpha = W^T (W Y)
    launch_tri_matvec_t(m->dW, m->dBeta1, m->dAlpha1, Np, Np, st);
    for (auto& e : m->evI8) if (!e) IBO_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    IBO_CUDA_TRY(pool_malloc((void**)&m->dWi8s, i8_steps_before(nb) * (size_t)I8_A_STAGE));
    IBO_CUDA_TRY(pool_malloc((void**)&m->dRowScale, sizeof(double) * 3 * Np));
    i8_rowscale_kernel<<<(Np + 7) / 8, 256, 0, st>>>(m->dW, Np, m->N, m->sf2, m->dRowScale);
    i8_slice_w_kernel<<<dim3(nb * 4, nb), 256, 0, st>>>(m->dW, m->dRowScale, Np, reinterpret_cast<uint8_t*>(m->dWi8s));
    g_launches += 4;
    IBO_CUDA_TRY(cudaGetLastError());
    m->i8Valid = true;
    return IBO_OK;
}

template <int DMAX>
static void launch_kstar_i8_d(ibo_model* m, const double* dCand, dim3 g1, long M, long m0, long Mpad, uint8_t* Ki8, double* part, cudaStream_t st) {
    const int p1 = m->npb > 0 ? 1 : 0;
    if (m->kind <= IBO_KERNEL_SE_ISO)
        kstar_i8_kernel<0, DMAX><<<g1, 256, 0, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, m->dAlphaY, m->dAlpha1, Ki8, part, m->N, m->d, m->nb, M, m0, Mpad, m->sf2, p1);
    else if (m->kind == IBO_KERNEL_MATERN3)
        kstar_i8_kernel<1, DMAX><<<g1, 256, 0, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, m->dAlphaY, m->dAlpha1, Ki8, part, m->N, m->d, m->nb, M, m0, Mpad, m->sf2, p1);
    else
        kstar_i8_kernel<2, DMAX><<<g1, 256, 0, st>>>(m->dXt, dCand, m->dInvTheta, m->dCenter, m->dAlphaY, m->dAlpha1, Ki8, part, m->N, m->d, m->nb, M, m0, Mpad, m->sf2, p1);
}

// K1 of one chunk on the int8 path; tiles = 128-candidate tiles of the chunk (the slab holds 2 * tiles 64-candidate tiles)
static void launch_kstar_i8(ibo_model* m, const double* dCand, long tiles, long M, long m0, long Mpad, uint8_t* Ki8, double* part, cudaStream_t st) {
    dim3 g1((unsigned)(tiles * 2), m->nb);
    const int d = m->d;
    if (d <= 2) launch_kstar_i8_d<2>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 4) launch_kstar_i8_d<4>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 6) launch_kstar_i8_d<6>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 8) launch_kstar_i8_d<8>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 12) launch_kstar_i8_d<12>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 16) launch_kstar_i8_d<16>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else if (d <= 24) launch_kstar_i8_d<24>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
    else launch_kstar_i8_d<32>(m, dCand, g1, M, m0, Mpad, Ki8, part, st);
}

// K2 of one chunk on the int8 path
static void launch_trigemm_i8(ibo_model* m, long tiles, long Mpad, const uint8_t* Ki8, double* part, cudaStream_t st) {
    const int sms = dev_info(m->device).sms;
    // Row-block groups G (a CTA walks nb / G row-blocks of its candidate tile, dealt in snake order).  Fewer groups = fewer CTA
    // prologues per unit of work and, above all, fewer passes over the tile's K* digits: the G CTAs of a tile share them through L2
    // only while they walk in step, and at N = 8192 the digits of W (235 MB) push them out between passes.  Measured (one B200,
    // tools/i8_bench.py): G = 4 is the best or within 1 % of it at every size -- N = 2048: 24.0 M evals/s (G = 2: 23.9, G = 1: 22.1),
    // N = 4096: 5.96 M (G = 8: 5.92, G = 2: 5.79), N = 8192: 1.58 M (G = 16: 1.35, G = 8: 1.53, G = 2: 1.52).
    // Option i8_rb_per_cta > 0 fixes the row-blocks per CTA instead (G = nb / value).
    const long per = get_option(OPT_I8_RB_PER_CTA);
    int G = per > 0 ? (int)std::max<long>(1, m->nb / per) : std::min(m->nb, 4);
    if (tiles * 2 * G < sms) G = (int)std::min<long>(m->nb, (sms + tiles * 2 - 1) / (tiles * 2));
    const dim3 grid(G, (unsigned)(tiles * 2));
    trigemm_i8_kernel<<<grid, I8_THREADS, I8_SMEM, st>>>(reinterpret_cast<const uint8_t*>(m->dWi8s), Ki8, m->dRowScale + m->Np, part, m->nb, Mpad);
}

// ---- live INT8 tensor peak (bench.py): back-to-back 128 x 256 x 32 MMAs from resident operands, one CTA per SM -------------
// rnd = 0: operand bytes in {0..3} (almost no switching activity: the burst ceiling of the pipe at full clock);
// rnd = 1: pseudo-random bytes -- the rate a kernel with real operands can reach; run for seconds it shows what the 1 kW power
// cap sustains (the SM clock drops from 1965 to ~1650 MHz under a dense INT8 load with random operands).
__global__ void __launch_bounds__(128) i8_peak_kernel(int iters, int rnd, int* __restrict__ sink) {
    extern __shared__ __align__(1024) uint8_t smem[];      // A: 128 x 128 B, B: 256 x 128 B (four k-steps of 32)
    __shared__ uint64_t bar;
    __shared__ uint32_t tbase;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < (128 + 256) * 128; i += 128)
        smem[i] = rnd ? (uint8_t)((((unsigned)i + 977u * blockIdx.x) * 2654435761u) >> 13) : (uint8_t)((i * 7 + 3) & 3);
    if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&tbase)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t td = tbase;
    if (warp == 0 && elect_one()) {
        // 128-byte-deep tiles: the k chunks of a row group are 128 B apart, row groups 8 * 128 B apart
        auto desc = [](uint32_t addr) {
            return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46);
        };
        const uint32_t a0 = smem_u32(smem), b0 = smem_u32(smem + 128 * 128);
        for (int it = 0; it < iters; it++)
#pragma unroll
            for (int kk = 0; kk < 4; kk++) umma_i8(td + (uint32_t)(it & 1) * 256u, desc(a0 + kk * 256), desc(b0 + kk * 256), umma_idesc_i8(128, 256), (it >> 1) & 1);
        umma_commit(&bar);
    }
    mbar_wait(&bar, 0);
    tc_fence_after();
    uint32_t v[8];
    tmem_ld8_nowait(td + ((uint32_t)(warp * 32) << 16), v);
    tmem_ld_wait();
    if (v[0] == 0x7fffffffu) sink[blockIdx.x * 128 + tid] = (int)v[1];
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(td), "r"(512u) : "memory");
}

}  // namespace ibo
