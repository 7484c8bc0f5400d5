/*
 * ibo_b200.h -- C ABI of libibo_b200.so, the B200 (sm_100a) implementation of IBO's acquisition
 * hot path: batched GP posterior mean/variance + EI/PI/UCB scoring, and the DIRECT driver
 * (maximizeEI / fastUCBGallery inner loop).
 *
 * This is the drop-in boundary.  Plain pointers and sizes only; all arrays are C-contiguous
 * FP64 in HOST memory unless a name ends in `_dev`.  Citations are file:line in the reference
 * (misterwindupbird/IBO):
 *
 *   acqmaxGP      replaces  cpp/optimizeGP.cpp:262-349 (bound by ego/acquisition/__init__.py:343-436)
 *   direct        replaces  cpp/direct.cpp:329-581, cpp/direct.h:57 (bound by ego/utils/optimize.py:310-343)
 *   ibo_model_*   replaces  GaussianProcess._computeCorrelations/addData (ibo_model_append: the block append)
 *                           (ego/gaussianprocess/__init__.py:134-149,267-308), the Laplace
 *                           L = chol(R + inv(C)) of PrefGaussianProcess (:487-498), and the explicit
 *                           inv(R) of cdirectGP (ego/acquisition/__init__.py:385-388)
 *   ibo_posterior_batch / ibo_score_batch
 *                 replace   GaussianProcess.posterior/posteriors (ego/gaussianprocess/__init__.py:169-244),
 *                           EI/PI/UCB.negf (ego/acquisition/__init__.py:60-75,100-114,138-164) and
 *                           GP_Maximizer::posterior/negei/negpi/negucb (cpp/optimizeGP.cpp:57-236)
 *   ibo_acqmax    replaces  cdirectGP + acqmaxGP without the explicit inverse
 *   ibo_nlml / ibo_kernel_matrix
 *                 replace   trainhyper.marginalLikelihood/nlml/dnlml (ego/gaussianprocess/trainhyper.py:47-136) and
 *                           Kernel.covMatrix / Kernel.derivative (ego/gaussianprocess/kernel.py:43-52,92-266)
 *
 * Return convention of the ibo_* functions: 0 = ok, <0 = error (see IBO_E_*); the legacy symbols
 * keep the reference's convention (malloc'd double[ndim+1], NULL on failure; caller frees with
 * libc free(), ego/acquisition/__init__.py:443-447).
 * There is no CPU fallback: every compute entry point fails with IBO_E_CUDA when no device is usable.
 */
#ifndef IBO_B200_H
#define IBO_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* kernel types: 0..3 as in ego/acquisition/__init__.py:323-333; 4 is the ARD form config #4 names */
#define IBO_KERNEL_SE_ARD       0   /* hyper = theta[d] (+ optional magnitude)          kernel.py:130-149 */
#define IBO_KERNEL_SE_ISO       1   /* hyper = theta (+ unused)                         kernel.py:71-89   */
#define IBO_KERNEL_MATERN3      2   /* hyper = theta, magnitude                         kernel.py:191-210 */
#define IBO_KERNEL_MATERN5      3   /* hyper = theta, magnitude (intended formula)      kernel.py:230-248 */
#define IBO_KERNEL_MATERN5_ARD  4   /* hyper = theta[d], magnitude                      (no reference class) */

/* acquisition ids (ego/acquisition/__init__.py:309-321) */
#define IBO_ACQ_EI   0
#define IBO_ACQ_PI   1
#define IBO_ACQ_UCB  2

/* flag word of the scoring entry points */
#define IBO_FLAG_MODE_CPP      0x0  /* libm erf, exact constants, sigma^2 floor 1e-8  (cpp/optimizeGP.cpp:150-215) */
#define IBO_FLAG_MODE_PY       0x1  /* Chebyshev erf, 0.707106/0.398942, floor 10e-8  (gaussianprocess/__init__.py:55-77,224) */
#define IBO_FLAG_KSTAR_EXPAND  0x2  /* cross-covariance through |x|^2+|y|^2-2x.y on the DMMA pipe (default: direct differences) */
#define IBO_FLAG_DIRECT_SEQ    0x4  /* DIRECT: evaluate rectangle by rectangle in the reference's call order */
#define IBO_FLAG_PROFILE       0x8  /* record per-kernel CUDA-event times (ibo_get_profile) */
#define IBO_FLAG_SHARD         0x20 /* ibo_acqmax: cut every DIRECT batch into one slice per rank of the communicator
                                       (ibo_comm_init) and all-gather the values; all ranks must make the same call */
#define IBO_FLAG_DIRECT_SPECULATE 0x40 /* DIRECT over a PURE batch objective: where a child centre depends on the division order
                                       only in its last bit, evaluate its (<= 4) possible values together with the probe points
                                       instead of in a second batch.  The callback then sees a few points the reference never
                                       samples; their values are discarded, so FMIN/XMIN/nsamples and the trajectory are unchanged.
                                       ibo_acqmax sets it (the GPU objective is pure). */
#define IBO_FLAG_INT8          0x80 /* scoring calls: take the INT8 tensor-core path even when the option "int8" is 0.  It is the DEFAULT for
                                       batches of more than 2048 candidates on models without a variance model, d <= 32, N <= 16384:
                                       sigma^2 through an exact-integer emulation of the FP64 triangular GEMM (7 x 7 base-256 digits,
                                       28 digit products in INT32 on tcgen05.mma kind::i8, FP64 assembly; ibo_b200/csrc/score_i8.cuh) and
                                       mu as k* . alpha.  Its error on sum v^2 is that of the FP64 GEMM (~4e-15 vs ~2e-15); candidates
                                       whose sigma^2 comes out below 2^-10 are re-scored by the FP64 DMMA kernels in the same call. */
#define IBO_FLAG_FP64          0x100 /* scoring calls: FP64 DMMA kernels for every candidate (no INT8 path) */
#define IBO_FLAG_GRAD_EXACT    0x10 /* ibo_nlml / ibo_kernel_matrix: analytic Matern-3/2 length-scale derivative instead of
                                       the reference's expression with the unscaled distance (kernel.py:217-222) */

/* error codes */
#define IBO_OK            0
#define IBO_E_BADARG     -1
#define IBO_E_CUDA       -2   /* no device / CUDA runtime error (ibo_last_error() has the text) */
#define IBO_E_NOTSPD     -3   /* Cholesky failed; *info = 1-based index of the first bad pivot */
#define IBO_E_NOMEM      -4
#define IBO_E_COMM       -5
#define IBO_E_OBJECTIVE  -6   /* DIRECT: the batch objective reported a failed evaluation (a NaN value); the run was stopped */

typedef struct ibo_model ibo_model;   /* opaque: owns device memory + one CUDA stream */
typedef struct ibo_cands ibo_cands;   /* opaque: a candidate set resident in HBM */

const char* ibo_last_error(void);
const char* ibo_version(void);
int  ibo_device_count(void);

/* ---- model ---------------------------------------------------------------------------------
 * A = K_offdiag(X) + (1+noise) I [+ Cinv], L = chol(A), W = inv(L), beta = W Y  on `device`.
 * X: N x d row-major.  hyper: the kernel's hyperparams array as-is (length nhyper).
 * Cinv: NULL or N x N row-major (PrefGP Laplace term, inv(C)).
 * prior: npbases==0 for none; else RBF-network mean prior (ego/gaussianprocess/prior.py:60-66):
 *        pmeans npbases x d row-major, pbeta[npbases], ptheta, plowerb[d], pwidth[d].
 * info:  receives 0, or the 1-based failing pivot when IBO_E_NOTSPD is returned (model is not created).
 */
int ibo_model_create(int device, int kerneltype, const double* hyper, int nhyper,
                     const double* X, const double* Y, int N, int d, double noise,
                     const double* Cinv,
                     int npbases, const double* pmeans, const double* pbeta, double ptheta,
                     const double* plowerb, const double* pwidth,
                     ibo_model** out, int* info);

/* PrefGaussianProcess after the Laplace fit (ego/gaussianprocess/__init__.py:461-498) without any explicit inverse on the host:
 *   C = cdiag I + sum_p w[p] (e_a - e_b)(e_a - e_b)^T  over the P preference pairs (a[p], b[p]) (indices into X; the reference's
 *   triple loop adds +w to C[a,a], C[b,b] and -w to C[a,b], C[b,a], starting from 5 I),
 *   A = K_offdiag(X) + (1+noise) I + inv(C),  L = chol(A), ...  -- C is assembled, factorised and inverted (Cholesky, triangular
 * inverse, Gram product) on the device.  IBO_E_NOTSPD with *info = pivot when C or A is not positive definite (the caller retries
 * with cdiag + 1 as the reference does with C += I, :487-498).  ibo_model_get_matrix(m, 3, out) returns inv(C). */
int ibo_model_create_pref(int device, int kerneltype, const double* hyper, int nhyper,
                          const double* X, const double* Y, int N, int d, double noise,
                          int P, const int* a, const int* b, const double* w, double cdiag,
                          ibo_model** out, int* info);

/* the same with C given as a dense symmetric N x N matrix (a Laplace fit made elsewhere): inv(C) is still formed on the device */
int ibo_model_create_laplace(int device, int kerneltype, const double* hyper, int nhyper,
                             const double* X, const double* Y, int N, int d, double noise, const double* C,
                             ibo_model** out, int* info);

/* Same model from an explicit inverse (legacy acqmaxGP layout, N x N row-major): factors invR = W'W. */
int ibo_model_create_from_inverse(int device, int kerneltype, const double* hyper, int nhyper,
                                  const double* X, const double* Y, int N, int d, double noise,
                                  const double* invR, double sf2,
                                  int npbases, const double* pmeans, const double* pbeta, double ptheta,
                                  const double* plowerb, const double* pwidth,
                                  ibo_model** out, int* info);

/* Rank-1 append of k observations (X: k x d row-major, Y[k]) to a plain model (no Cinv, not from_inverse, no variance
 * model): the block append of GaussianProcess.addData (ego/gaussianprocess/__init__.py:300-308) one row at a time on
 * the device -- l = W k, lambda = sqrt(1+noise - l.l), new rows of L and W = inv(L), beta -- O(k N^2) instead of the
 * O(N^3) rebuild; buffers are re-homed when N crosses a multiple of 128.  On IBO_E_NOTSPD (*info = 1-based pivot)
 * the model is no longer valid and must be destroyed. */
int ibo_model_append(ibo_model* m, const double* X, const double* Y, int k, int* info);
int ibo_model_destroy(ibo_model* m);
int ibo_model_n(const ibo_model* m);
int ibo_model_dim(const ibo_model* m);
/* copy back N x N row-major matrices: which = 0 -> A (=R [+Cinv]), 1 -> L (lower, zeros above), 2 -> W = inv(L),
 * 3 -> inv(C) of a model made by ibo_model_create_pref */
int ibo_model_get_matrix(ibo_model* m, int which, double* out);
/* secondary ("aug") factor used for the variance only (PrefGaussianProcess.addObservationPoint,
 * ego/gaussianprocess/__init__.py:214-223,502-519): sigma^2 comes from `aug`, mu from `m`. */
int ibo_model_set_variance_model(ibo_model* m, ibo_model* aug);

/* ---- PrefGaussianProcess: Laplace MAP fit (SURVEY 8f-2) -----------------------------------------
 * Minimises the reference's functional (ego/gaussianprocess/__init__.py:355-386)
 *     S(y) = - sum_p (deg[p]+1) log(CDF((y[v[p]] - y[u[p]]) / sqrt 2) + 1e-10) + |inv(L) y|^2 / 2
 * (v[p] preferred to u[p]; indices into the model's points; the reference's Chebyshev-erf CDF) by damped Newton steps
 * on the device instead of the reference's BFGS on numerical gradients (:441-442).  `m` is the plain R model of the N
 * distinct preference points.  y[N]: in = starting latents (:410-430), out = minimiser.  maxit <= 0 -> 100, gtol <= 0 ->
 * 1e-9 (sup-norm of the whitened gradient).  S_out / gnorm_out / iters_out may be NULL. */
int ibo_pref_fit(ibo_model* m, int P, const int* v, const int* u, const double* deg, double* y,
                 int maxit, double gtol, double* S_out, double* gnorm_out, int* iters_out);

/* ---- hyper-parameter learning (SURVEY 8f-4) --------------------------------------------------------
 * Negative log marginal likelihood of trainhyper.marginalLikelihood (useCholesky branch, trainhyper.py:47-76):
 *     K = covMatrix(X) + noise I (diagonal sf2 + noise), nlml = Y.inv(K).Y/2 + sum log diag chol(K) + N log(2 pi)/2
 * and, when dnlml != NULL, dnlml[h] = sum((inv(K) - alpha alpha^T) o dK/dlog hyper[h]) / 2 for every entry of `hyper`
 * (length scales first, then the magnitude when the kernel has one: SE-ARD/Matern-5/2-ARD with nhyper == d+1,
 * Matern-3/2, Matern-5/2 with nhyper == 2).  The derivative matrices are the reference's Kernel.derivative
 * (kernel.py:92-105,152-166,212-228,250-266) including its Matern-3/2 expression unless IBO_FLAG_GRAD_EXACT.
 * IBO_E_NOTSPD (*info = failing pivot) when K is not positive definite (the reference catches LinAlgError, :61-67).
 * X: N x d row-major; nothing stays resident. */
int ibo_nlml(int device, int kerneltype, const double* hyper, int nhyper, const double* X, const double* Y, int N, int d,
             double noise, int flags, double* nlml, double* dnlml, int* info);
/* out (N x N row-major) = Kernel.covMatrix(X) when which < 0 (kernel.py:43-52), else Kernel.derivative(X, which) */
int ibo_kernel_matrix(int device, int kerneltype, const double* hyper, int nhyper, const double* X, int N, int d,
                      int which, int flags, double* out);

/* ---- batched posterior / scoring -------------------------------------------------------------
 * Xs: M x d row-major candidates (original coordinates).  Outputs may be NULL when not wanted.
 * mu[M], s2[M]: posterior mean and *clipped* variance (floor by mode, ceiling 10).
 * scores[M]: acquisition value being maximised (EI, PI or UCB; i.e. minus the reference's negf).
 * best_score/best_idx: argmax over the batch, lowest index wins ties; NaN scores never win.
 * ymax = max(Y) (EI/PI incumbent, ego/acquisition/__init__.py:143), parm = xi (EI/PI) or the UCB multiplier.
 */
int ibo_posterior_batch(ibo_model* m, const double* Xs, long M, int flags, double* mu, double* s2);
int ibo_score_batch(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags,
                    double* scores, double* mu, double* s2, double* best_score, long* best_idx);

/* Candidates kept resident in HBM (the bench's device-resident leg; also used for sharded sets). */
int ibo_cands_create(ibo_model* m, const double* Xs, long M, ibo_cands** out);
int ibo_cands_destroy(ibo_cands* c);
/* Scores a resident set; scores_host may be NULL (then only best_* cross PCIe).  ms_device, if not NULL,
 * receives the CUDA-event time of the launch sequence on the model's stream. */
int ibo_score_resident(ibo_model* m, ibo_cands* c, int acq, double ymax, double parm, int flags,
                       double* scores_host, double* best_score, long* best_idx, float* ms_device);

/* Per-kernel CUDA-event times (ms) and launch counts of the last scoring call made with
 * IBO_FLAG_PROFILE: out[0]=K1 cross-covariance, out[1]=K2 triangular GEMM + reduce,
 * out[2]=K3 epilogue/argmax, out[3]=total, out[4]=#launches, out[5]=K2 launches. */
int ibo_get_profile(ibo_model* m, double* out6);
/* cumulative count of kernels this library launched in this process */
long ibo_launch_count(void);
/* measurement helpers (bench.py): live FP64 tensor-pipe peak of `device` in TFLOP/s (DMMA.8x8x4 issue rate);
 * page-lock / unlock a caller-owned host buffer so the copies of the end-to-end leg run from pinned memory */
int ibo_fp64_peak(int device, double* tflops);
/* live INT8 tensor-pipe peak in TOP/s (tcgen05.mma kind::i8 issue rate): the roofline of the INT8 path of wide batches */
int ibo_i8_peak(int device, double* tops);
/* the same pipe measured two ways: burst (a few ~2 ms launches, near-constant operand bytes: full SM clock) and sustained
 * (pseudo-random operand bytes, back to back for `seconds`, rate over the second half: what the power cap lets a dense INT8 kernel
 * with real data hold).  Either pointer may be NULL. */
int ibo_i8_peak2(int device, double seconds, double* burst_tops, double* sustained_tops);
int ibo_host_register(void* p, unsigned long bytes);
int ibo_host_unregister(void* p);
/* CUDA events on the model's stream (slot 0 = start, 1 = stop) and their elapsed device time */
int ibo_stream_mark(ibo_model* m, int slot);
int ibo_stream_elapsed_ms(ibo_model* m, float* ms);
int ibo_device_synchronize(int device);
/* test hook: the cross-covariance kernel's own exp (x <= 0) next to libdevice exp, host arrays of n values */
int ibo_debug_exp(int device, const double* x, long n, double* out_fast, double* out_ref);

/* ---- options -----------------------------------------------------------------------------------
 * Process-wide tuning / debugging switches, visible at the boundary (no hidden environment reads in the launch paths; an
 * environment variable IBO_<NAME IN CAPITALS> presets the option when the library is loaded).  Names:
 *   int8 (1)          wide batches take the INT8 tensor-core path (0: FP64 DMMA everywhere; per call: IBO_FLAG_INT8 / IBO_FLAG_FP64)
 *   i8_min_batch (-1) batches of this many .. narrow_max candidates take the INT8 path too (DIRECT's mid-size batches); -1: from the
 *                     measured break-even with the FP64 latency shapes on (735 / 300 / 133 / 62 candidates at N = 1024 / 2048 /
 *                     4096 / 8192), 0: wide batches only
 *   i8_guard (1)      INT8 path: re-score candidates with sigma^2 < 2^-10 on the DMMA path
 *   i8_pipe (1)       INT8 path: cross-covariance of chunk c+1 on a low-priority stream under the GEMM of chunk c
 *   i8_rb_per_cta (0) INT8 GEMM: row-blocks per CTA (0: four row-block groups whatever the size)
 *   chunk_tiles (0)   128-candidate tiles per chunk (0: 2 x number of SMs)
 *   narrow_max (2048) batches up to this size use the latency shapes of the FP64 GEMM
 *   narrow_mt (0), k2_deep (-1), pdl (1), kstar_direct (0), tiny (-1)   shape / launch switches of the small-batch path
 *   debug_plan (0), direct_timing (0)   diagnostics on stderr
 *   shard_min (0)     sharded DIRECT: batches below this many points are not sharded (0: 64 x ranks)
 *   tiny_server (1)   DIRECT on a model of <= 128 observations: the fused kernel stays resident for the query and takes its batches
 *                     from a mailbox in mapped host memory (0: one launch per batch)
 *   chol_pair (-1)    model build: block columns in pairs (256-deep trailing updates); -1: from 48 block columns on, 0 / 1 forced
 * Unknown names return IBO_E_BADARG. */
int ibo_set_option(const char* name, long value);
int ibo_get_option(const char* name, long* value);
/* candidates the last scoring call on `m` re-scored on the DMMA path (guard of the INT8 path); 0 when the path was not taken */
int ibo_model_last_guarded(const ibo_model* m);

/* ---- DIRECT ----------------------------------------------------------------------------------
 * Batched DIRECT following the reference's rectangle rules (cpp/direct.cpp:146-235,372-498).
 * The callback receives n points (n x ndim row-major, original box coordinates) and fills y[n]
 * with the objective being MINIMISED.  One call per iteration carries every probe point and every child centre that does not
 * depend on the division order; a second, small call follows only for rectangles whose child centres do (see
 * IBO_FLAG_DIRECT_SPECULATE).  The set of points evaluated without that flag is exactly the reference's.
 * A NaN value means "this evaluation failed": the driver stops at once and returns IBO_E_OBJECTIVE (the reference has no error
 * channel -- an exception in its Python callback aborts the C call through ctypes).
 */
typedef void (*ibo_batch_objective_t)(void* user, long n, int ndim, const double* X, double* y);
int ibo_direct_batched(ibo_batch_objective_t f, void* user, int ndim, const double* lb, const double* ub,
                       int maxiter, int maxtime, int maxsample, int flags,
                       double* fmin, double* xmin, long* nsamples, int* iterations);

/* maximise an acquisition over a box with the GPU objective; opt = max value, optx[ndim] */
int ibo_acqmax(ibo_model* m, const double* lb, const double* ub, int acq, double ymax, double parm, int flags,
               int maxiter, int maxtime, int maxsample,
               double* opt, double* optx, long* nsamples, int* iterations);

/* nq independent queries at once, one host thread each: query q maximises over the same box on models[q] (distinct handles, any
 * devices) with incumbent ymax[q] and parameter parm[q].  opt[nq], optx[nq x ndim]; nsamples / iterations / status (per-query
 * return codes) may be NULL.  Returns the first non-zero status.  This is how several GPUs serve DIRECT: throughput across
 * queries -- one query is a chain of dependent small batches. */
int ibo_acqmax_many(int nq, ibo_model* const* models, const double* lb, const double* ub, int acq, const double* ymax,
                    const double* parm, int flags, int maxiter, int maxtime, int maxsample,
                    double* opt, double* optx, long* nsamples, int* iterations, int* status);

/* ---- legacy drop-in symbols (same names, same ABI as libego) ---------------------------------- */
typedef double (*objective_t)(int, double*);                                    /* cpp/direct.h:14 */
const double* direct(objective_t objective, int ndim, double* lb, double* ub,
                     int maxiter, int maxtime, int maxsample);                   /* cpp/direct.h:57 */
const double* acqmaxGP(int ndim, double* lb, double* ub, double* invR, double* X, double* Y, int nx,
                       int acqfunc, int kerneltype, double* hyperparams,
                       int npbases, double* pbasismeans, double* pbasisbeta, double pbasistheta,
                       double* pbasislowerb, double* pbasiswidth,
                       double parm, double noise, int maxiter, int maxtime, int maxsample);
                                                                                 /* cpp/optimizeGP.cpp:262-283 */

/* ---- multi-GPU (one process per GPU; NCCL is dlopen'ed on first use) -------------------------- */
int ibo_comm_unique_id(unsigned char* id128);                 /* rank 0: 128-byte ncclUniqueId */
int ibo_comm_init(int device, int rank, int nranks, const unsigned char* id128);
int ibo_comm_destroy(void);
/* all-reduce of a (score, global index) pair: max score, lowest index wins ties */
int ibo_comm_argmax(double* score, long* index);
/* broadcast `count` doubles in HOST memory from root through device buffers over NVLink */
int ibo_comm_bcast(double* buf, long count, int root);
int ibo_comm_barrier(void);
int ibo_comm_rank(void);                                       /* 0 when no communicator */
int ibo_comm_size(void);                                       /* 1 when no communicator */
/* all[r * count + i] = rank r's mine[i] (host buffers, same count on every rank) */
int ibo_comm_allgather(const double* mine, long count, double* all);

#ifdef __cplusplus
}
#endif
#endif /* IBO_B200_H */
