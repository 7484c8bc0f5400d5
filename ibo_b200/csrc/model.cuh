// Internal model/state structs of libibo_b200.
#pragma once
#include "common.cuh"
#include "../../include/ibo_b200.h"
#include <map>
#include <utility>
#include <vector>

namespace ibo {
struct CandWork;

// the streams and events launch_factorize runs on: the model's own, whatever it factorises
struct Lanes {
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;   // inversion pipeline of the model build; K1 of the next chunk on the INT8 path
    cudaStream_t stream3 = nullptr;   // bulk trailing updates of the look-ahead Cholesky
    cudaStream_t stream4 = nullptr;   // bulk row updates of the inversion that follows it
    cudaEvent_t evStep = nullptr, evRest = nullptr, evScale = nullptr, evFar = nullptr;
};

// the matrices launch_factorize reads and writes: the model's, or a scratch factor of the candidate workspace
struct Factor {
    int N = 0;
    int Np = 0;                 // nb * 128 (identity padded)
    int nb = 0;                 // 128-row blocks
    double* dA = nullptr;       // [Np][Np] row-major: A (the model's R (+Cinv)), overwritten by L (lower)
    double* dD = nullptr;       // [nb][128][128] inverses of the diagonal blocks of L
    double* dW = nullptr;       // [Np][Np] row-major: W = inv(L), exact zeros above the diagonal
    double* dWpack = nullptr;   // packed blobs, wpack_base(nb) * BLOB doubles
    double* dY = nullptr;       // [Np]
    double* dBetaY = nullptr;   // [Np]  W Y
    int* dInfo = nullptr;       // 0, or the pivot at which A is not positive definite
};
}  // namespace ibo

struct ibo_model : ibo::Lanes, ibo::Factor {
    int device = 0;
    int d = 0, kind = 0;
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
    double* dAorig = nullptr;   // optional copy of A (kept for get_matrix(0)); N<=4096 only
    double* dBeta1 = nullptr;   // [Np]  W 1
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
    std::map<std::pair<long, int>, std::pair<int, int>> planCache;   // K2 launch plan (MT, G) per (32-candidate CTA tiles, option narrow_mt)
    // profile of the last call
    double prof[6] = {0, 0, 0, 0, 0, 0};
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // workspace of the joint posterior, the candidate gradients, q-EI and MES (joint.cu, grad.cu, qei.cu, mes.cu), built on first use
    ibo::CandWork* cand = nullptr;
};

namespace ibo {
// Workspace of the candidate-side entry points (joint.cu, grad.cu, qei.cu, mes.cu), of sample-path creation (paths.cu) and of the
// Laplace fit (laplace.cu), kept with the model that owns the call and grown on demand.  One call at a time runs on a model, so they
// share one set of buffers, one per role; g is the variance model when one is attached and the model otherwise.  Within a call no two live roles share a buffer: Z overwrites K* and y overwrites V
// once K* and V are dead.  A call grows every buffer it uses before it takes a pointer into the workspace.
struct CandWork {
    double* dRaw = nullptr;     size_t rawCap = 0;     // candidates as given [M][d]
    double* dScaled = nullptr;  size_t scaledCap = 0;  // candidates (of the chunk) scaled and centred like g's training inputs [Mcp][d]
    double* dScaledM = nullptr; size_t scaledMCap = 0; // the same scaled like the model's (variance model attached) [Mcp][d]
    double* dKc = nullptr;      size_t kcCap = 0;      // K* = R(X_g, X*), then Z = W_g^T V [Np][Mcp]; T = W_g V (paths) [Np][Sp]
    double* dV = nullptr;       size_t vCap = 0;       // V = W_g K*, then y (q-EI) [Np][Mcp]; Phi_g w + E e, then c (paths) [Np][Sp]
    double* dAB = nullptr;      size_t abCap = 0;      // a | b [2][Np]
    double* dKb = nullptr;      size_t kbCap = 0;      // k^T b [M] (prior only)
    double* dG = nullptr;       size_t gCap = 0;       // three [M][d] gradient planes
    double* dNormals = nullptr; size_t normalsCap = 0; // standard normals: [Mp][Sp] zero padded (samples), [q][S] (q-EI), e [Ng][S] (paths)
    double* dPost = nullptr;    size_t postCap = 0;    // [score | mu | s2] of the scoring path, 3 M + 2 (joint, gradients; MES values in
                                                       // the score plane, best value and index at 3 M); mu [M] (q-EI)
    // scratch factor of the joint posterior, q-NEI, the Laplace fit and the noise factor of sample paths, on the owner's lanes
    Factor chol;                                       // Sigma in chol.dA (Mp x Mp), factorised in place (q-NEI: Sigma of the baseline,
                                                       // with W = inv(L) in chol.dW; Laplace fit: B = I + G G^T and its inverse factor)
    size_t cholACap = 0, cholDCap = 0;                 // chol.dA, chol.dD
    size_t cholWCap = 0, cholYCap = 0;                 // chol.dW; chol.dY (zeros) | chol.dBetaY [2][Mp], when inverted
    double* dF = nullptr;       size_t fCap = 0;       // samples [Mp][Sp]
    double* dArg = nullptr;     size_t argCap = 0;     // per-sample argmax (long long)
    // q-EI only
    double* dQei = nullptr;     size_t qeiCap = 0;     // values [B]
    double* dMubar = nullptr;   size_t mubarCap = 0;   // d qEI / d mu [M]
    double* dSig = nullptr;     size_t sigCap = 0;     // Sigma of the chunk's batches [Bc][q][q]
    double* dGbar = nullptr;    size_t gbarCap = 0;    // Gbar of the chunk's batches [Bc][q][q]
    // q-NEI only (the per-batch buffers of q-EI above too; V grows to [Np + Pp][Mcp]: T below V, then Cbar in T's place)
    double* dBase = nullptr;    size_t baseCap = 0;    // baseline raw [P][d] | scaled like g [Pp][d] | mu_b [Pp] | incumbent m [Sp]
    double* dVb = nullptr;      size_t vbCap = 0;      // V_b = W_g K(X_g, X_b) [Np][Pp]
    double* dZbase = nullptr;   size_t zbaseCap = 0;   // Z_b = W_g^T V_b [Np][Pp] (gradient only)
    double* dZb = nullptr;      size_t zbCap = 0;      // baseline normals Z_b [Pp][Sp] zero padded
    double* dFb = nullptr;      size_t fbCap = 0;      // baseline draws F_b [Pp][Sp]
    double* dCT = nullptr;      size_t ctCap = 0;      // C = Sigma_bq, then Tbar [Pp][Mcp]
    double* dH = nullptr;       size_t hCap = 0;       // H = Z_b^T T, then the winner indicator E [Sp][Mcp]
    // max-value entropy search only
    double* dYstar = nullptr;   size_t ystarCap = 0;   // y* samples [K]
    double* dMesD = nullptr;    size_t mesDCap = 0;    // d MES / d mu | d MES / d s [2][M]
    double* dBlk = nullptr;     size_t blkCap = 0;     // per-block partials: argmax values | indices (long long) [2][nblk]; Gumbel fit:
                                                       // bracket state lo[3] | hi[3], then trial sums [nblk][3 T] | bracket ends [nblk][2]
};
CandWork* cand_work(ibo_model* m);                     // model.cu: the model's workspace, created empty on first use
}  // namespace ibo

struct ibo_cands {
    ibo_model* owner = nullptr;
    double* dX = nullptr;   // [M][d] raw coordinates in HBM
    long M = 0;
};

namespace ibo {
struct ScoreReq;
// fused single-launch path for models of one row-block (tiny.cu)
bool tiny_eligible(const ibo_model* m, long M);
int score_tiny(ibo_model* m, const double* cand, long M, const ScoreReq& rq, double* out, const CandInline* inl);
// the scoring path's block-argmax pair (dBlkBest, dBlkIdx) holds at least `need` blocks; a smaller pair is freed and `cap` blocks allocated
int grow_blk(ibo_model* m, size_t need, size_t cap);
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
// f.dA = L L^T in place on the streams and events of `ln` (the model build passes the model as both: launch_factorize(*m, *m, ..)).
// invert = false: the Cholesky factor only (no W = inv(L), no beta = W Y); dW, dWpack and the beta vectors are not touched
int launch_factorize(const Lanes& ln, Factor& f, bool from_inverse_reversed, bool pack, bool invert);
void launch_tri_matvec(const double* T, const double* v, double* out, int Np, cudaStream_t st);              // out = T v, T lower [Np][Np]
void launch_tri_matvec_t(const double* T, const double* v, double* out, int n, int Np, cudaStream_t st);     // out = T^T v over the leading n x n
int launch_syrk_identity(double* C, const double* G, int Np, int K, cudaStream_t st);                        // C = I + G G^T (lower tiles)
// model whose A carries `diag` on the diagonal instead of 1 + noise (hyper.cu: K = covMatrix(X) + noise I)
int create_model_with_diag(int device, int kind, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
                           double noise, double diag, ibo_model** out, int* info);
int launch_gram_wtw(double* C, const ibo_model* m, cudaStream_t st);      // hyper.cu: C (lower tiles) = W^T W = inv(A)
const char* get_error();
// score.cu: [score | mu | s2] of M device-resident candidates at out, what ibo_score_batch (acq >= 0) or ibo_posterior_batch
// (acq < 0) returns with flags; out holds 3 M + 2 doubles
int posterior_score_device(ibo_model* m, const double* dCand, long M, int acq, double ymax, double parm, int flags, double* out);
// joint.cu: the argument checks of the candidate-side entry points (Xs, M >= 1, d <= 64); extra_ok carries the entry point's own
// bounds, computed before the model is read
int check_cands(const ibo_model* m, const double* Xs, long M, bool extra_ok);
// joint.cu: the dynamic shared memory of the W GEMMs below, once per call before them
int ensure_joint_attrs(int device);
// joint.cu, on st: candidates scaled and centred like g's training inputs ([Mp][d], zero padded); R(X_g, X*) with exact
// zeros in the padding ([Np][Mp]); V = W_g Kc and Z = W_g^T V ([Np][Mp] each, Z may overwrite Kc)
void launch_scale_cands(double* Cs, const double* X, const ibo_model* g, long M, long Mp, cudaStream_t st);
void launch_cross_cov(double* Kc, const ibo_model* g, const double* Cs, int M, int Mp, cudaStream_t st);
void launch_w_gemm_v(double* V, const ibo_model* g, const double* Kc, int Mp, cudaStream_t st);
void launch_w_gemm_z(double* Z, const ibo_model* g, const double* V, int Mp, cudaStream_t st);
// joint.cu: the workspace's scratch factor (chol) sized for an M x M matrix; it is factorised on the model's lanes
// (launch_factorize(*m, w->chol, ..)); invert: also chol.dW and the vectors launch_factorize(.., invert = true) reads and writes
int chol_setup(ibo_model* m, long M, bool invert);
// joint.cu, on st: c.dA (lower tiles) = R(X*, X*) with `diag` on the diagonal, kernel of g elsewhere, - V^T V (K = g->Np) + jitter I
void launch_joint_sigma(Factor& c, const double* Cs, const double* V, const ibo_model* g, double diag, double jitter, cudaStream_t st);
// joint.cu, on st: zeros above the diagonal inside the diagonal blocks of a factorised c.dA
void launch_clear_diag_upper(Factor& c, cudaStream_t st);
// joint.cu, on st: per column s < S of F ([M][ldf]) the argmax (lowest index wins, NaN never wins) and, when best is non-null, the max
void launch_sample_max(const double* F, int ldf, int M, int S, long long* arg, double* best, cudaStream_t st);
// joint.cu, on st: Kc[i][j] = k(xa_i, x*_j) with g's kernel for the Na points Xa scaled like g, exact zeros in the padding ([Nap][Mp])
void launch_cross_cov_pts(double* Kc, const double* Xa, int Na, int Nap, const ibo_model* g, const double* Cs, int M, int Mp, cudaStream_t st);
// joint.cu, on st: the DMMA triangular GEMMs with explicit operands: C = T B (T lower block-triangular, nbr block rows, + bias[row]
// for rows < nbias) and C = T^T B; cols a multiple of 128
void launch_trimm(double* C, int ldc, const double* T, int ldt, const double* B, int ldb, int nbr, int cols, const double* bias, int nbias,
                  cudaStream_t st);
void launch_trimm_t(double* C, int ldc, const double* T, int ldt, const double* B, int ldb, int nbr, int cols, cudaStream_t st);
// joint.cu, on st: dense DMMA GEMM C = alpha op(A) B (+ C with acc), op(A) = A^T (A [K][rows]) with transA, else A [rows][K]; B [K][cols];
// rows, cols multiples of 128, K of 16; every column of C runs over the full K in the same order
void launch_gemm(double* C, int ldc, const double* A, int lda, bool transA, const double* B, int ldb, int rows, int cols, int K,
                 double alpha, bool acc, cudaStream_t st);
// grad.cu: candidates per chunk of the gradient and q-EI paths, the largest multiple of 128 whose K* / Z and V over g's training
// points (2 Np doubles per candidate) fit in 512 MiB
long cand_chunk(const ibo_model* g);
// grad.cu, on st: a = W^T (W Y) and, with a prior, b = W^T (W 1) of the model into ab ([2][Np]), recomputed every call (an appended
// model needs no invalidation); returns b, or nullptr without a prior
double* launch_ab(const ibo_model* m, double* ab, cudaStream_t st);
// grad.cu, on st: G[q][j][t] = sum_i w_q,i dk_i(x*_j) / dx_t for the Mc candidates of a chunk (planes `plane` doubles apart): w_0 =
// Zw[:, j] (leading dimension ldz) over g's training points with Cs scaled like them, w_1 = a and w_2 = b over the model's with Cm
// scaled like them (Cm is read with a variance model attached only); b and kb[j] = sum_i b_i k_i with a prior only (b non-null)
void launch_grad_sums(const ibo_model* m, const double* Cs, const double* Cm, int Mc, const double* Zw, int ldz, const double* a,
                      const double* b, double* G, size_t plane, double* kb, cudaStream_t st);
// grad.cu, on st: the prior's share of dmu in place over plane 2 of G ([3][M][d]) for the M candidates `cand` (original coordinates)
void launch_grad_prior(const ibo_model* m, const double* cand, long M, const double* kb, double* G, cudaStream_t st);
// grad.cu: enqueues everything on m->stream and leaves [score | mu | s2] (the FP64 kernels' with flags) in the workspace's dPost and,
// with wantGrad, ds2, dmu and dscore ([M][d] each; ds2 = 0 where s2 is clipped; dscore = 0 for acq < 0) in its dG
int grad_device(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags, bool wantGrad);
// score.cu, on st: the final argmax over nblk per-block (best, index) pairs of the scoring path's block argmax (lowest index wins
// ties, NaN never wins)
void launch_argmax_final(const double* blkBest, const long long* blkIdx, long nblk, double* best, long long* bestIdx, cudaStream_t st);
}  // namespace ibo
