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
#define IBO_FLAG_KSTAR_EXPAND  0x2  /* no effect, value kept for ABI compatibility: the cross-covariance of the FP64 kernels always goes
                                       through |x|^2+|y|^2-2x.y on the DMMA pipe for d <= 32 (pairs with large scaled norms are
                                       recomputed from direct differences); option "kstar_direct" = 1 selects direct differences */
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

/* ---- joint posterior over a candidate set --------------------------------------------------------
 * Xs: M x d row-major candidates (original coordinates), 1 <= M <= 16384, d <= 64.  With R the model's correlation function
 * (k off the diagonal, 1 + noise on it) and W = inv(L) of the model (of its variance model when one is attached):
 *     V = W R(X, Xs),  Sigma = R(Xs, Xs) - V^T V     (diag(Sigma) = the unclipped sigma^2 of ibo_posterior_batch)
 * mu = the posterior mean exactly as ibo_posterior_batch returns it with IBO_FLAG_FP64.  GEMMs and the Cholesky on the FP64
 * tensor pipe; workspace stays with the model (M x M and N x M doubles).
 * mu[M] (may be NULL) and cov[M x M] row-major, full symmetric; 1 <= M <= 16384, d <= 64 */
int ibo_posterior_cov(ibo_model* m, const double* Xs, long M, double* mu, double* cov);
/* F[M x S] row-major = mu + chol(Sigma + jitter I) Z for caller-supplied standard normals Z[M x S] (row-major);
 * argmax[S] = per-sample argmax over the M candidates (a Thompson batch).  F or argmax may be NULL.
 * IBO_E_NOTSPD with *info = 1-based failing pivot when Sigma + jitter I is not positive definite.
 * jitter is added for the factorisation only.  Ties go to the lowest index, NaN never wins.  IBO_E_BADARG for a NULL model,
 * Xs or Z, M outside [1, 16384], S < 1, or jitter < 0 or NaN. */
int ibo_posterior_sample(ibo_model* m, const double* Xs, long M, const double* Z, int S, double jitter,
                         double* F, long* argmax, int* info);

/* ---- gradients with respect to the candidate ----------------------------------------------------
 * Xs: M x d row-major candidates (original coordinates), M >= 1, d <= 64.  flags: 0 (IBO_FLAG_MODE_CPP) or IBO_FLAG_MODE_PY.
 * Values (mu, s2, scores) are those of the FP64 kernels (IBO_FLAG_FP64) bit for bit.  With s = x / theta - centre,
 *     dk_i / dx_t = -(1 / theta_t) h(r_i) (s_t - s_i,t),   d mu = d m0 (1 - k^T b) + sum_i (a_i - m0 b_i) dk_i,
 *     d s2 = -2 sum_i z_i dk_i,  z = R^-1 k         (a = R^-1 Y, b = R^-1 1; R of the variance model for s2 when one is attached)
 * z comes from two DMMA triangular GEMMs (W K*, W^T V) per chunk of candidates; workspace stays with the model.
 * dmu, ds2: M x d row-major; ds2 = 0 where sigma^2 is clipped (floor by mode, ceiling 10).  Any output may be NULL.
 * IBO_E_BADARG for a NULL model or Xs, M < 1, d > 64, acq outside 0..2, or a flag bit other than IBO_FLAG_MODE_PY. */
int ibo_posterior_grad(ibo_model* m, const double* Xs, long M, int flags, double* mu, double* s2, double* dmu, double* ds2);
/* scores[M] as ibo_score_batch returns them with IBO_FLAG_FP64; dscores[M x d] row-major = the chain rule through (mu, sqrt(s2)):
 * EI d/dmu = Phi(Z), d/ds = phi(Z); PI phi(Z) / s, -Z phi(Z) / s; UCB 1, parm.  In IBO_FLAG_MODE_PY Phi and phi are the derivatives
 * of that mode's own formula (the Chebyshev erf with 0.707106 / 0.398942), so that dscores match finite differences of its values. */
int ibo_score_grad(ibo_model* m, const double* Xs, long M, int acq, double ymax, double parm, int flags,
                   double* scores, double* dscores);

/* ---- batch expected improvement (q-EI) -----------------------------------------------------------
 * Xs: B x q x d row-major, batch b = (x_b1 .. x_bq) contiguous (original coordinates).  With mu_b, Sigma_b the joint posterior of
 * batch b as ibo_posterior_cov defines it (Sigma = R(Xs, Xs) - V^T V, 1 + noise on the diagonal, unclipped; from the variance model
 * when one is attached; mu = the posterior mean, summed in a fixed order per point, so it agrees with ibo_posterior_batch's to
 * rounding but does not depend on the other points of the call), L_b = chol(Sigma_b + jitter I) and caller-supplied standard
 * normals Z[q x S] (row-major, the layout of ibo_posterior_sample):
 *     values[b] = (1 / S) sum_s max(0, max_j (mu_b + L_b z_s)_j - ymax - xi)
 * (at q = 1 the Monte-Carlo estimate of EI in libm arithmetic with the unclipped sigma^2).  dvalues[B x q x d] (may be NULL) is its
 * exact gradient with respect to the points for the fixed Z: per sample with positive improvement and argmax j* (lowest index wins
 * ties) mubar_j* += 1 / S, Lbar_j*,k += z_k,s / S (k <= j*); Gbar = d qEI / d Sigma by the reverse Cholesky (Murray 2016), summed
 * over all ordered pairs; then
 *     d qEI / dx_j = mubar_j dmu(x_j) + 2 sum_l Gbar_jl d1 k(x_j, x_l) - 2 sum_i y_j,i dk_i(x_j) / dx_j,   y_j = sum_l Gbar_jl R^-1 k(X, x_l)
 * Without dvalues the gradient work is skipped; the values are the same bits either way, and a batch's value and gradient do not
 * depend on the other batches of the call.  A batch whose Sigma_b + jitter I is not positive definite gets NaN for its value and
 * its gradient rows; *nbad (may be NULL) receives the number of such batches and the call still returns IBO_OK.
 * IBO_E_BADARG for a NULL model, Xs, Z or values, B < 1, q outside [1, 32], S outside [1, 65536], d > 64, or jitter < 0 or NaN. */
int ibo_qei(ibo_model* m, const double* Xs, long B, int q, const double* Z, int S,
            double ymax, double xi, double jitter, double* values, double* dvalues, int* nbad);

/* ---- noisy batch expected improvement (q-NEI) ------------------------------------------------------
 * Xs: B x q x d as for ibo_qei; Xbase: P x d row-major, the points already evaluated (original coordinates); Z[(P + q) x S]
 * row-major standard normals, the P baseline rows first, then the q batch rows.  For each batch the LATENT joint posterior of the
 * P + q points [Xbase; batch] is taken (Letham et al. 2019):
 *     Sigma = K(., .) - V^T V,  V = W_g K(X_g, .)    (the kernel itself, sf2 on the diagonal; g the variance model when one is
 *                                                     attached, else the model),
 * mu the posterior mean of ibo_qei (fixed order per point), L = chol(Sigma + jitter I) and
 *     F_s = mu + L z_s,   m_s = max_{i < P} F_s,i (the incumbent of sample s),
 *     values[b] = (1 / S) sum_s max(0, max_{j >= P} F_s,j - m_s).
 * The incumbent is the best true value among the evaluated points, drawn jointly with the batch: no observation noise is added
 * to points already measured (the convention of ibo_paths_*), which needs sf2 <= 1 + noise.  L is formed blockwise with the
 * baseline first: L_bb = chol(Sigma_bb + jitter I), m_s and W_bb = inv(L_bb) once per call, then per batch T = W_bb Sigma_bq,
 * F_s,q = mu_q + T^T z_b + chol(Sigma_qq + jitter I - T^T T) z_q.  incumbent[S] (may be NULL) receives m_s.  dvalues[B x q x d]
 * (may be NULL) is the exact gradient for the fixed Z in reverse mode (the baseline does not depend on the batch): per improving
 * sample with winner j*, mubar_j* += 1 / S, Lbar_j*,k += z_q,k / S, Tbar[:, j*] += z_b / S; Gbar by the reverse Cholesky,
 * Tbar -= 2 T Gbar, Cbar = W_bb^T Tbar, and
 *     d qNEI / dx_j = mubar_j dmu(x_j) + 2 sum_l Gbar_jl d1 k(x_j, x_l) + sum_i Cbar_ij d1 k(x_j, xb_i) - 2 sum_i y_j,i dk_i(x_j) / dx_j,
 *     y_j = R_g^-1 (K(X_g, X_q) Gbar + K(X_g, X_b) Cbar / 2)_j.
 * Every sum runs in a fixed order without atomics: a batch's value and gradient do not depend on the other batches of the call,
 * the values are the same bits with and without dvalues, and repeated calls give the same bits.  Points per chunk =
 * max(128, floor(2^26 / (2 Np + 2 Pp + Sp) / 128) 128) (Np, Pp, Sp: g's training points, P and S rounded up to 128), whole
 * batches per chunk.  If Sigma_bb + jitter I is not positive definite the call returns IBO_E_NOTSPD with *info (may be NULL) = the
 * 1-based baseline pivot; a batch whose Schur complement is not gets NaN for its value and gradient rows and is counted in *nbad
 * (may be NULL), and the call returns IBO_OK.
 * IBO_E_BADARG, before the device is touched, for a NULL model, Xs, Xbase, Z or values, B < 1, q outside [1, 32], P outside
 * [1, 8192], S outside [1, 8192], d > 64, jitter < 0 or NaN, or sf2 > 1 + noise (of g). */
int ibo_qnei(ibo_model* m, const double* Xs, long B, int q, const double* Xbase, long P, const double* Z, int S, double jitter,
             double* values, double* dvalues, double* incumbent, int* nbad, int* info);

/* ---- max-value entropy search (MES) -------------------------------------------------------------
 * Xs: M x d row-major candidates (original coordinates), M >= 1, d <= 64.  mu and s2 are what ibo_posterior_batch returns with the
 * same flags: s2 is the library's clipped variance (floor 1e-8, 1e-7 under IBO_FLAG_MODE_PY, ceiling 10), which like EI's carries
 * the 1 + noise diagonal of R, so MES measures the information about max y of a noisy observation.  For samples y*[K] of the maximum
 *     g_k = (y*_k - mu) / s,  s = sqrt(s2),  psi = phi / Phi,  h(g) = g psi(g) / 2 - log Phi(g) >= 0,  MES = (1 / K) sum_k h(g_k)
 * summed in ascending k.  h'(g) = -(psi / 2)(1 + g (g + psi)) < 0: raising a y* lowers every value.  For g <= -1.5 sqrt2, h and h'
 * come from the continued fraction of erfc, which does not cancel.  The gradient is the chain rule
 *     d MES = d MES / d mu  d mu + d MES / d s  d s2 / (2 s),  d MES / d mu = -(1 / (K s)) sum h'(g_k),  d MES / d s = -(1 / (K s)) sum g_k h'(g_k)
 * with d s2 = 0 where s2 is clipped (ibo_posterior_grad's).
 *
 * Gumbel fit of the distribution of max f over the candidate set Xs (M x d, M >= 1): with mu_i, s_i = sqrt(s2_i) as
 * ibo_posterior_batch returns them with `flags` (0, IBO_FLAG_MODE_PY, IBO_FLAG_INT8, IBO_FLAG_FP64), q[0..2] solve
 * sum_i log Phi((q - mu_i) / s_i) = log 0.25, log 0.5, log 0.75; scale = (q[2] - q[0]) / (log(-log .25) - log(-log .75)),
 * loc = q[1] + scale log(-log .5).  Any output may be NULL.  Deterministic: the same set gives the same bits.
 * Samples of the maximum are then y* = loc - scale log(-log u) for uniforms u in (0, 1) the caller draws.  The three roots are
 * bracketed by max(mu_i - s_i) and max(mu_i + c s_i), c = sqrt(2 ln 5M), and found by 16 passes of multisection with 15 trial
 * points per bracket (64 bits), each pass one kernel over all candidates and one that adds the blocks' sums in a fixed order: q[b]
 * is the upper end of the final bracket.  The grid is a function of M alone.
 * IBO_E_BADARG for a NULL model or Xs, M < 1, d > 64, or a flag bit other than those listed. */
int ibo_max_value_gumbel(ibo_model* m, const double* Xs, long M, int flags, double* q, double* loc, double* scale);

/* values[M] = (1/K) sum_k h((ystar[k] - mu) / s), h(g) = g psi(g) / 2 - log Phi(g), psi = phi / Phi; 1 <= K <= 1024, every ystar
 * finite.  Without dvalues: mu, s2 as ibo_posterior_batch with `flags`.  With dvalues (M x d, d <= 64): flags 0 or IBO_FLAG_MODE_PY
 * only, mu and s2 of the FP64 kernels (as ibo_score_grad), and values the same bits as the dvalues = NULL call with IBO_FLAG_FP64.
 * best / best_idx: argmax, lowest index wins, NaN never wins; any output may be NULL.
 * IBO_E_BADARG for a NULL model, Xs, ystar or values, M < 1, d > 64, K outside [1, 1024], a non-finite ystar, a flag bit other
 * than IBO_FLAG_MODE_PY, IBO_FLAG_INT8 and IBO_FLAG_FP64, or dvalues with a flag other than IBO_FLAG_MODE_PY. */
int ibo_mes(ibo_model* m, const double* Xs, long M, const double* ystar, int K, int flags,
            double* values, double* dvalues, double* best, long* best_idx);

/* ---- pathwise posterior samples (Matheron's rule, Wilson et al. 2020) -------------------------------
 * S posterior sample paths drawn from one model, each a deterministic function of x that can be evaluated at any number of points.
 * g is the model Sigma comes from: the attached variance model if there is one, otherwise m (ibo_posterior_cov's rule); Ng is g's N.
 * The caller supplies every random number, so the same draws reproduce the same bits:
 *   omega[F x d]  frequencies in unit-length-scale coordinates, drawn from the kernel's spectral density (SE: N(0, I); Matern-nu:
 *                 multivariate Student-t with 2 nu degrees of freedom, z sqrt(2 nu / u), u ~ chi^2(2 nu));
 *   phase[F]      b_j ~ U(0, 2 pi);   w[F x S], e[Ng x S]  standard normals (row-major).
 * With s(x) = x / theta (g's length scales, no centring; g's centre is folded into the phases on the device):
 *   phi_j(x) = sqrt(2 sf2 / F) cos(omega_j . s(x) + b_j)
 *   mu(x)    = m0(x) + k_m(x)^T a - m0(x) k_m(x)^T b,  a = R_m^-1 Y, b = R_m^-1 1, m0 the prior mean as ibo_posterior_batch applies it
 *              (the mean whose derivative ibo_posterior_grad uses; it agrees with ibo_posterior_batch's mu to rounding, not bit for bit)
 *   f_s(x)   = mu(x) + phi(x)^T w_s - k_g(x)^T R_g^-1 (Phi_g w_s + E e_s),  Phi_g = phi at g's training points, with the training
 *              noise E e_s = sqrt(1 + noise - sf2) e_s (plain, legacy or appended g) or chol(inv(C) + (1 + noise - sf2) I) e_s (g with a
 *              Laplace term, R_g = R + inv(C); factorised on the device at create time: the noise that R_g implies, as k(x, x) = sf2)
 * These are samples of the LATENT function: their covariance approximates Sigma - (1 + noise - sf2) I with Sigma from
 * ibo_posterior_cov, whereas the draws of ibo_posterior_sample carry the 1 + noise diagonal of an observation.
 * A paths object is a snapshot: it holds copies of everything it reads (scaled training inputs of m and g, a, b, c_s, the folded
 * phases, w, omega, the prior) and gives the same bits after ibo_model_append or ibo_model_destroy on m.  It has its own stream on m's
 * device and does not use the model's workspace.
 * Limits: 1 <= F <= 65536, 1 <= S <= 1024, d <= 64, M >= 1.  IBO_E_BADARG for NULL pointers, sizes out of range, sf2 > 1 + noise, or
 * a g with a host-supplied inv(C) (ibo_model_create with Cinv) of more than 4096 points, whose inv(C) the device no longer holds.
 * IBO_E_NOTSPD with *info = 1-based pivot when inv(C) + (1 + noise - sf2) I is not positive definite. */
typedef struct ibo_paths ibo_paths;
int ibo_paths_create(ibo_model* m, int F, int S, const double* omega, const double* phase, const double* w, const double* e,
                     ibo_paths** out, int* info);
/* values[M x S] row-major (may be NULL) at the M x d points Xs (original coordinates); best[S] / best_idx[S] (may be NULL): per path the
 * argmax over the M points, lowest index wins ties, NaN never wins.  Each value is one fixed-order sum over the rows, so a point's values
 * do not depend on the other points of the call and two calls give the same bits. */
int ibo_paths_eval(ibo_paths* p, const double* Xs, long M, double* values, double* best, long* best_idx);
/* point j on path which[j] (0 <= which[j] < S): values[M] (the same bits as ibo_paths_eval's) and the exact gradient with respect to x,
 * grad[M x d] = d mu - sqrt(2 sf2 / F) sum_j w_j,s sin(omega_j . s + b_j) omega_j / theta - sum_i c_i,s dk_i.  Meant for few points
 * (one thread per point).  IBO_E_BADARG for NULL pointers, M < 1 or a which outside [0, S). */
int ibo_paths_grad(ibo_paths* p, const double* Xs, long M, const int* which, double* values, double* grad);
int ibo_paths_destroy(ibo_paths* p);

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
 *   debug_plan (0), direct_timing (0)   diagnostics on stderr (debug_plan: each new latency-shape plan, "[plan_narrow] ...",
 *                     and the instance of every FP64 GEMM launch, "[k2] ... MT=.. P1=.. DEEP=..")
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
