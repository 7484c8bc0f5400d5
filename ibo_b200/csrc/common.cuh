// Shared device/host helpers for libibo_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <string>

namespace ibo {

// ---------------------------------------------------------------------------------------------
// tile geometry shared by every kernel
// ---------------------------------------------------------------------------------------------
constexpr int TM = 128;          // training rows per row-block (M dimension of the DMMA GEMMs)
constexpr int TN = 128;          // candidates per tile         (N dimension)
constexpr int BK = 16;           // contraction depth of one pipeline stage
constexpr int BLOB = TM * BK;    // doubles in one packed operand blob (16 KiB)
constexpr int KB_PER_BLOCK = TM / BK;   // 8 k-blobs per 128-wide block

// Packed ("fragment-major") operand blob layout, identical for the A operand (W: rows x k) and
// the B operand (K*: k x candidates).  For element (r in [0,128), k in [0,16)):
//   tile = r / 8, lane = (r % 8) * 4 + (k % 4), ks = k / 4, ks2 = ks / 2, par = ks % 2
//   offset = ((tile * 2 + ks2) * 32 + lane) * 2 + par
// so that one LDS.128 per lane yields the DMMA.8x8x4 fragments of two consecutive k-steps and a
// whole warp reads 512 contiguous bytes (bank-conflict free by construction).
__host__ __device__ inline int blob_offset(int r, int k) {
    int tile = r >> 3, lane = ((r & 7) << 2) | (k & 3), ks = k >> 2;
    return (((tile * 2 + (ks >> 1)) * 32 + lane) << 1) | (ks & 1);
}

// first blob of row-block i in the packed W array (row-block i owns (i+1)*8 blobs)
__host__ __device__ inline size_t wpack_base(int i) { return (size_t)KB_PER_BLOCK * ((size_t)i * (i + 1) / 2); }

// x rounded up to whole 128-wide tiles
inline long round128(long x) { return (x + 127) / 128 * 128; }

// ---------------------------------------------------------------------------------------------
// error handling
// ---------------------------------------------------------------------------------------------
void set_error(const std::string& s);
#define IBO_CUDA_TRY(expr)                                                                        \
    do {                                                                                          \
        cudaError_t e__ = (expr);                                                                 \
        if (e__ != cudaSuccess) {                                                                 \
            ::ibo::set_error(std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
            return IBO_E_CUDA;                                                                    \
        }                                                                                         \
    } while (0)

extern long g_launches;   // kernels launched by this library (bench.py's gpu_launches)

// ---------------------------------------------------------------------------------------------
// per-device state and tuning options (util.cu)
// ---------------------------------------------------------------------------------------------
// cudaFuncSetAttribute is per device: every kernel family records, per device ordinal, that its attributes are set.
enum { ATTR_MODEL = 0, ATTR_SCORE, ATTR_TINY, ATTR_I8, ATTR_GRAM, ATTR_JOINT, ATTR_COUNT };
struct DevInfo { int sms = 148; bool known = false; bool attrs[ATTR_COUNT] = {false, false, false, false, false, false}; };
DevInfo& dev_info(int device);            // SM count filled on first use
// Runs `setter` once per (device, family) with `device` current; returns the CUDA error of the first failing call.
cudaError_t ensure_attrs(int device, int family, cudaError_t (*setter)());

}  // namespace ibo
#include "options.h"
namespace ibo {

// A small candidate batch can travel in a kernel's parameter buffer: the launch itself delivers it, no H2D DMA and no PCIe
// read inside the kernel.  448 doubles keep the parameter block inside the classic 4 KiB limit.
constexpr int CAND_INLINE = 448;
struct CandInline { double x[CAND_INLINE]; };

// ---------------------------------------------------------------------------------------------
// device primitives
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
// D(8x8) += A(8x4) * B(4x8), FP64, SASS: DMMA.8x8x4.
//   a: A[row = lane/4][k = lane%4]      b: B[k = lane%4][col = lane/4]
//   c0,c1: C[row = lane/4][col = 2*(lane%4) + {0,1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// Warp-level wait: one lane polls, the others park on the warp barrier.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
    if ((threadIdx.x & 31) == 0) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "WAITW_%=:\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
            "@p bra DONEW_%=;\n\t"
            "bra WAITW_%=;\n\t"
            "DONEW_%=:\n\t}"
            ::"r"(smem_u32(bar)), "r"(parity) : "memory");
    }
    __syncwarp();
}
// 1-D bulk async copy global -> shared (TMA engine, SASS: UBLKCP), completion on an mbarrier.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// Programmatic dependent launch (sm_90+): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may be
// scheduled while its predecessor in the stream is still running; pdl_wait() blocks until that predecessor has completed and
// its writes are visible (a no-op for a normal launch), pdl_launch_dependents() lets the successor be scheduled early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
#endif  // __CUDACC__

}  // namespace ibo
