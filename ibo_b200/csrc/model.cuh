// Internal model/state structs of libibo_b200.
#pragma once
#include "common.cuh"
#include "../../include/ibo_b200.h"
#include <map>
#include <utility>
#include <vector>

struct ibo_model {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;   // inversion pipeline of the model build; K1 of the next chunk on the INT8 path
    cudaStream_t stream3 = nullptr;   // bulk trailing updates of the look-ahead Cholesky
    cudaStream_t stream4 = nullptr;   // bulk row updates of the inversion that follows it
    cudaEvent_t evStep = nullptr, evRest = nullptr, evScale = nullptr, evFar = nullptr;
    int N = 0, d = 0, kind = 0;
    int nb = 0;          // 128-row blocks
    int Np = 0;          // nb * 128 (identity padded)
    double noise = 0, sf2 = 1;
    bool cpp_prior = false;
    bool has_cinv = false;            // A = R + inv(C): no rank-1 append
    double* dCinv = nullptr;          // [Np][Np] lower tiles of inv(C) when it was formed on the device (ibo_model_create_pref)
    std::vector<double> hInvTheta, hCenter;   // host copies (append scales new points the same way)
    double* dAppend = nullptr; size_t appendCap = 0;   // append workspace: [x_new (d) | kvec (Np) | l (Np) | u (Np) | lambda]
    // device arrays
    double* dXt = nullptr;      // scaled training inputs x/theta, [Np][d], rows >= N are zero
    double* dInvTheta = nullptr;// [d]
    double* dCenter = nullptr;  // [d] mean of the scaled training inputs (dXt is stored centred)
    double* dA = nullptr;       // [Np][Np] row-major: A = R (+Cinv), overwritten by L (lower)
    double* dAorig = nullptr;   // optional copy of A (kept for get_matrix(0)); N<=4096 only
    double* dW = nullptr;       // [Np][Np] row-major: W = inv(L), exact zeros above the diagonal
    double* dD = nullptr;       // [nb][128][128] inverses of the diagonal blocks of L
    double* dWpack = nullptr;   // packed blobs, wpack_base(nb) * BLOB doubles
    double* dBetaY = nullptr;   // [Np]  W Y
    double* dBeta1 = nullptr;   // [Np]  W 1
    double* dY = nullptr;       // [Np]
    int* dInfo = nullptr;
    bool from_inverse = false;        // built from a caller-supplied inverse (legacy acqmaxGP): sigma^2 >= noise is not guaranteed
    // INT8 path of wide batches (score_i8.cuh), built on first use: the seven base-256 digits of W packed for shared memory
    // (dWi8s), per-row scales ([Np] slicing scale, [Np] 2 scale sf2, [Np] shift constant), alpha = W^T W Y and W^T W 1
    double* dWi8s = nullptr; double* dRowScale = nullptr; double* dAlphaY = nullptr; double* dAlpha1 = nullptr;
    bool i8Valid = false;
    cudaEvent_t evI8[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // K1 done [2], K2+K3 done [2], fork
    cudaEvent_t evCopy[5] = {nullptr, nullptr, nullptr, nullptr, nullptr}; // host candidates: chunk copy done [4], fork
    // guard pass of the INT8 path: per-candidate flags + block counts; index list, gathered candidates and their re-scored values
    double* dGuard = nullptr; size_t guardCap = 0;
    double* dGuardList = nullptr; size_t guardListCap = 0;
    int lastGuarded = 0;              // candidates the last scoring call re-scored on the DMMA path
    // prior (RBF network), device copies
    int npb = 0;
    double ptheta = 0;
    double* dPmeans = nullptr;  // [npb][d]
    double* dPbeta = nullptr;   // [npb]
    double* dPlb = nullptr;     // [d]
    double* dPwidth = nullptr;  // [d]
    // variance model (PrefGP aug): not owned
    ibo_model* var_model = nullptr;
    // scoring workspace (grown on demand)
    double* dCand = nullptr;  size_t candCap = 0;     // candidates of the current call [M][d]
    double* dSlab = nullptr;  size_t slabCap = 0;     // packed K* of the current chunk
    double* dPart = nullptr;  size_t partCap = 0;     // [3][nb][chunkM] partial reductions
    double* dOut = nullptr;   size_t outCap = 0;      // [3][M]: score, mu, s2
    double* dBlkBest = nullptr; long long* dBlkIdx = nullptr; size_t blkCap = 0;
    double* dBest = nullptr;  long long* dBestIdx = nullptr;      // final argmax
    double* hPinned = nullptr; size_t pinnedCap = 0;              // pinned staging for small batches
    // batch server of the fused small-model kernel (tiny.cu): mailbox in mapped pinned memory, resident kernel on `stream`
    double* hServer = nullptr; unsigned long long* dSrvCount = nullptr; bool srvRunning = false; long long srvSeq = 0;
    int srvAcq = 0, srvFlags = 0, srvCtas = 0; double srvYmax = 0, srvParm = 0;
    std::map<long, std::pair<int*, int>> unitTables;              // K2 work tables (device), keyed by shape and group count
    std::map<long, std::pair<int, int>> planCache;                // K2 launch plan (MT, G) per number of 32-candidate CTA tiles
    // profile of the last call
    double prof[6] = {0, 0, 0, 0, 0, 0};
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

struct ibo_cands {
    ibo_model* owner = nullptr;
    double* dX = nullptr;   // [M][d] raw coordinates in HBM
    long M = 0;
};

namespace ibo {
struct ScoreReq;
// fused single-launch path for models of one row-block (tiny.cu)
bool tiny_eligible(const ibo_model* m, long M);
int score_tiny(ibo_model* m, const double* cand, long M, const ScoreReq& rq, double* out, const double* host_cand);
// batch server for one DIRECT query on such a model: y[i] = -acq(X[i]); the first call starts the resident kernel, stop ends it
bool tiny_server_fits(const ibo_model* m, long n);
int tiny_server_eval(ibo_model* m, const double* X, long n, int acq, double ymax, double parm, int flags, double* y);
void tiny_server_stop(ibo_model* m);
int grow(double** p, size_t* cap, size_t need);
cudaError_t pool_malloc(void** p, size_t bytes);
void pool_free(void* p);
cudaError_t pinned_get(double** p);
void pinned_put(double* p);
// launches (all on m->stream)
int launch_factorize(ibo_model* m, bool from_inverse_reversed, bool pack);
void launch_tri_matvec(const double* T, const double* v, double* out, int Np, cudaStream_t st);              // out = T v, T lower [Np][Np]
void launch_tri_matvec_t(const double* T, const double* v, double* out, int n, int Np, cudaStream_t st);     // out = T^T v over the leading n x n
int launch_syrk_identity(double* C, const double* G, int Np, int K, cudaStream_t st);                        // C = I + G G^T (lower tiles)
// model whose A carries `diag` on the diagonal instead of 1 + noise (hyper.cu: K = covMatrix(X) + noise I)
int create_model_with_diag(int device, int kind, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
                           double noise, double diag, ibo_model** out, int* info);
int launch_gram_wtw(double* C, const ibo_model* m, cudaStream_t st);      // hyper.cu: C (lower tiles) = W^T W = inv(A)
const char* get_error();
}  // namespace ibo
