// Measurement helpers exported through the C ABI (used by bench.py only):
//   ibo_fp64_peak      live DMMA.8x8x4 issue-rate microbenchmark = the FP64 tensor-pipe roofline
//                      denominator on the GPU the bench runs on (MEASURED_PEAKS.json has no FP64 entry)
//   ibo_host_register  pin a caller-owned NumPy buffer so H2D/D2H copies of the e2e leg are DMA'd directly
#include "model.cuh"
#include <cctype>
#include <cstdlib>
#include <cstring>
#include <mutex>

namespace ibo {

static std::mutex g_dev_mu;
static DevInfo g_dev[64];

DevInfo& dev_info(int device) {
    if (device < 0 || device >= 64) device = 0;
    DevInfo& D = g_dev[device];
    if (!D.known) {
        std::lock_guard<std::mutex> lk(g_dev_mu);
        if (!D.known) {
            cudaDeviceProp pr;
            if (cudaGetDeviceProperties(&pr, device) == cudaSuccess) D.sms = pr.multiProcessorCount;
            else cudaGetLastError();
            D.known = true;
        }
    }
    return D;
}

cudaError_t ensure_attrs(int device, int family, cudaError_t (*setter)()) {
    DevInfo& D = dev_info(device);
    if (D.attrs[family]) return cudaSuccess;
    std::lock_guard<std::mutex> lk(g_dev_mu);
    if (D.attrs[family]) return cudaSuccess;
    int cur = 0;
    cudaError_t e = cudaGetDevice(&cur);
    if (e == cudaSuccess && cur != device) e = cudaSetDevice(device);
    if (e == cudaSuccess) e = setter();
    if (cur != device) cudaSetDevice(cur);
    if (e == cudaSuccess) D.attrs[family] = true;
    return e;
}

struct OptDef { const char* name; long def; };
static const OptDef g_optdef[OPT_COUNT] = {
    {"int8", 1}, {"i8_pipe", 1}, {"chunk_tiles", 0}, {"narrow_max", 2048}, {"narrow_mt", 0}, {"k2_deep", -1}, {"pdl", 1},
    {"kstar_direct", 0}, {"debug_plan", 0}, {"tiny", -1}, {"direct_timing", 0}, {"shard_min", 0}, {"i8_guard", 1}, {"i8_min_batch", -1}, {"i8_rb_per_cta", 0}, {"chol_pair", -1}, {"tiny_server", 1}};
static long g_opt[OPT_COUNT];
static std::once_flag g_opt_once;
static void init_options() {
    for (int i = 0; i < OPT_COUNT; i++) {
        g_opt[i] = g_optdef[i].def;
        std::string env = "IBO_";
        for (const char* c = g_optdef[i].name; *c; c++) env += (char)toupper(*c);
        const char* e = getenv(env.c_str());
        if (e && *e) g_opt[i] = atol(e);
    }
    // spelling of round 1: IBO_KSTAR=direct
    const char* e = getenv("IBO_KSTAR");
    if (e && !strcmp(e, "direct")) g_opt[OPT_KSTAR_DIRECT] = 1;
}
long get_option(int id) {
    std::call_once(g_opt_once, init_options);
    return (id >= 0 && id < OPT_COUNT) ? g_opt[id] : 0;
}
static int find_option(const char* name) {
    if (!name) return -1;
    for (int i = 0; i < OPT_COUNT; i++) if (!strcmp(name, g_optdef[i].name)) return i;
    return -1;
}

}  // namespace ibo

extern "C" int ibo_set_option(const char* name, long value) {
    const int id = ibo::find_option(name);
    if (id < 0) { ibo::set_error(std::string("unknown option: ") + (name ? name : "(null)")); return IBO_E_BADARG; }
    ibo::get_option(id);          // make sure the defaults / environment presets are in place
    ibo::g_opt[id] = value;
    return IBO_OK;
}
extern "C" int ibo_get_option(const char* name, long* value) {
    const int id = ibo::find_option(name);
    if (id < 0 || !value) { ibo::set_error(std::string("unknown option: ") + (name ? name : "(null)")); return IBO_E_BADARG; }
    *value = ibo::get_option(id);
    return IBO_OK;
}

namespace {
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double a0, double b0) {
    double c0[8], c1[8];
    double a = a0 + threadIdx.x * 1e-9, b = b0 + threadIdx.x * 1e-9;
#pragma unroll
    for (int i = 0; i < 8; i++) { c0[i] = i; c1[i] = -i; }
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) ibo::dmma884(c0[i], c1[i], a, b);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s += c0[i] + c1[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace

extern "C" int ibo_fp64_peak(int device, double* tflops) {
    if (!tflops) return IBO_E_BADARG;
    IBO_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp p;
    IBO_CUDA_TRY(cudaGetDeviceProperties(&p, device));
    const int sms = p.multiProcessorCount, bps = 4, iters = 8000;
    double* out = nullptr;
    IBO_CUDA_TRY(cudaMalloc(&out, sizeof(double) * sms * bps * 256));
    cudaEvent_t e0, e1;
    IBO_CUDA_TRY(cudaEventCreate(&e0));
    IBO_CUDA_TRY(cudaEventCreate(&e1));
    double best = 0;
    for (int r = 0; r < 6; r++) {
        IBO_CUDA_TRY(cudaEventRecord(e0));
        dmma_peak_kernel<<<sms * bps, 256>>>(out, iters, 1.0000001, 1e-9);
        IBO_CUDA_TRY(cudaEventRecord(e1));
        IBO_CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        double tf = 512.0 * 8 * iters * 8.0 * sms * bps / (ms * 1e-3) / 1e12;   // 512 flop per warp-level DMMA.8x8x4
        if (r >= 2 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    IBO_CUDA_TRY(cudaGetLastError());
    *tflops = best;
    return IBO_OK;
}

extern "C" int ibo_host_register(void* p, unsigned long bytes) {
    if (!p || !bytes) return IBO_E_BADARG;
    IBO_CUDA_TRY(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
    return IBO_OK;
}

extern "C" int ibo_host_unregister(void* p) {
    if (!p) return IBO_E_BADARG;
    IBO_CUDA_TRY(cudaHostUnregister(p));
    return IBO_OK;
}

// CUDA events on the model's stream: slot 0/1 of a private pair (bench.py brackets its timed region with them)
static cudaEvent_t g_marks[2] = {nullptr, nullptr};
extern "C" int ibo_stream_mark(ibo_model* m, int slot) {
    if (!m || slot < 0 || slot > 1) return IBO_E_BADARG;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    if (!g_marks[slot]) IBO_CUDA_TRY(cudaEventCreate(&g_marks[slot]));
    IBO_CUDA_TRY(cudaEventRecord(g_marks[slot], m->stream));
    return IBO_OK;
}
extern "C" int ibo_stream_elapsed_ms(ibo_model* m, float* ms) {
    if (!m || !ms || !g_marks[0] || !g_marks[1]) return IBO_E_BADARG;
    IBO_CUDA_TRY(cudaSetDevice(m->device));
    IBO_CUDA_TRY(cudaEventSynchronize(g_marks[1]));
    IBO_CUDA_TRY(cudaEventElapsedTime(ms, g_marks[0], g_marks[1]));
    return IBO_OK;
}
extern "C" int ibo_device_synchronize(int device) {
    IBO_CUDA_TRY(cudaSetDevice(device));
    IBO_CUDA_TRY(cudaDeviceSynchronize());
    return IBO_OK;
}
