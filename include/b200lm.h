/* b200lm -- C ABI of the B200-native batched Levenberg-Marquardt engine.
 *
 * This is the drop-in boundary for ONE hot path of gplepage/lsqfit (v13.3.1):
 *   whiten  ->  residual + Jacobian  ->  trust-region LM fit  ->  covariance propagation
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference tree).  The reference is Python; a maintainer binds these symbols with
 * ctypes (see INTEGRATION.md).  No torch / C++ types cross this boundary: plain
 * pointers and sizes only.
 *
 * Conventions
 *   - all matrices are row-major IEEE fp64; index arrays are int32
 *   - pointers named d_* are CUDA DEVICE pointers on the handle's device;
 *     pointers named h_* are HOST pointers
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream)
 *   - every function returns 0 on success, a negative B200LM_E* code otherwise and
 *     never throws; b200lm_last_error() gives the message.  Non-convergence of a
 *     fit is data (status[] / stopping criterion), not an error -- the reference's
 *     convention (src/lsqfit/_gsl.pyx:686-717, src/lsqfit/_scipy.py:177-181)
 *   - a handle is thread-compatible: one handle per host thread, and ONE batch in flight per handle (its work queue and
 *     statistics buffers belong to the launch in progress: use one handle per stream for concurrent batches)
 */
#ifndef B200LM_H
#define B200LM_H

#ifdef __cplusplus
extern "C" {
#endif

#define B200LM_VERSION 100          /* 0.1.0 */

#define B200LM_OK          0
#define B200LM_EINVAL     -1        /* bad argument */
#define B200LM_ENOFUNCTOR -2        /* (family, np) not in the device functor registry */
#define B200LM_ECUDA      -3        /* CUDA runtime error */
#define B200LM_ENOMEM     -4
#define B200LM_ESIZE      -5        /* problem does not fit the kernel's shared-memory plan */

typedef struct b200lm_handle_s* b200lm_handle;
typedef struct b200lm_comm_s* b200lm_comm;

/* ---- library ------------------------------------------------------------------------ */
int b200lm_version(void);
/* message of the last failing call on `h` (or of the last failing call without a handle
 * when h == NULL).  Mirrors the reference's fit.error convention. */
const char* b200lm_last_error(b200lm_handle h);
/* number of visible CUDA devices (0 if none / driver missing) */
int b200lm_device_count(void);

/* ---- device functor registry ---------------------------------------------------------
 * The reference receives the fit function as an opaque Python callable
 * (src/lsqfit/__init__.py:566, 1997-2042: flatfcn).  Here the model is one of a registry
 * of CUDA device functors, selected by family name + number of parameters.
 * The registry lists the built-in functors first (families 0 ... 30, always at the same
 * indices), then the entries of run-time plug-ins in load order.  The registry only grows;
 * reading and appending are thread-safe. */
int b200lm_functor_count(void);
int b200lm_functor_info(int i, int* family, int* np, int* nx, const char** name);
int b200lm_functor_family(const char* name);            /* family id, or B200LM_ENOFUNCTOR */

/* Add the functors of a plug-in to the registry: a shared object compiled from the library's
 * own headers with its flags (lsqfit_b200.cuda_functor generates and builds one from a model
 * body) that exports b200lm_plugin_entries (csrc/registry.h).  The plug-in is dlopen'ed and
 * its ABI record checked against the library (version, sizeof(FitParams),
 * sizeof(FunctorEntry), digest of the headers and flags): a mismatch is B200LM_EINVAL with
 * the field named.  All entries of one plug-in share one model name, np in 1..25, nx in 1..8;
 * they get the family *family_out, numbered from B200LM_USER_FAMILY0 upward in load order.
 * A name that a built-in functor or another plug-in already uses is B200LM_EINVAL; loading
 * the same name from the same model source again returns its family.  Plug-ins are never
 * unloaded (plans hold their launchers).  Needs no GPU. */
#define B200LM_USER_FAMILY0 1000
#define B200LM_USER_MAX_NP 25
#define B200LM_USER_MAX_NX 8
int b200lm_load_functors(const char* path, int* family_out);

/* ---- plan ---------------------------------------------------------------------------
 * One handle per (functor, ny, np, device).  noprior != 0 means fits without a prior
 * (src/lsqfit/_utilities.pyx:74-75): the mean vector then has ny entries, otherwise
 * N = ny + np entries (data means followed by prior means, :76-77). */
int b200lm_create(int family, int ny, int np, int nx, int noprior, int device, b200lm_handle* out);
void b200lm_destroy(b200lm_handle h);

/* model constants: the x array of flatfcn.keywords['x'] (src/lsqfit/__init__.py:1997-2012),
 * row-major [ny][nx].  Host pointer; copied once. */
int b200lm_set_const(b200lm_handle h, const double* h_x, int n);

/* whitening description == the reference's yp_pdf.i_invwgts
 * (consumed at src/lsqfit/_utilities.pyx:59-61, 85-93):
 *   entry 0 : ndiag 1x1 blocks, (diag_idx[i], diag_w[i] = 1/sigma)
 *   entry k : block k with blk_nin[k] input indices blk_idx[...] and a
 *             blk_nout[k] x blk_nin[k] row-major weight matrix W_k in blk_w[...]
 *             (sum_i outer(W_k[i], W_k[i]) = inverse covariance of the block)
 * Indices address the concatenated y(+)prior vector.  Host pointers; copied once.
 * Residual order (chiv) = diag entries in the given order, then block rows. */
int b200lm_set_weights(b200lm_handle h, int ndiag, const int* h_diag_idx, const double* h_diag_w,
                       int nblk, const int* h_blk_nin, const int* h_blk_nout,
                       const int* h_blk_idx, const double* h_blk_w);
int b200lm_nchiv(b200lm_handle h);

/* ---- the fit --------------------------------------------------------------------------
 * Replaces   fit = FITTERS[fitter](p0, nf, chiv, tol=tol, maxit=maxit, **fitterargs)
 * (src/lsqfit/__init__.py:662-664) and the plugin behind it (src/lsqfit/_scipy.py:115-181,
 * src/lsqfit/_gsl.pyx:563-723) for a whole batch of B independent fits that share the
 * model, x and whitening:
 *   d_mean   [B][N] means of y(+)prior per fit (mean_stride = N) or one shared vector
 *            (mean_stride = 0)  -- what bootstrapped_fit_iter / simulated_fit_iter vary
 *            (src/lsqfit/__init__.py:1619-1623, 545-552)
 *   d_p0     [B][np] starting points (p0_stride = np) or one shared start (p0_stride = 0); with bounds
 *            (b200lm_set_bounds) every start is projected into the box as scipy's make_strictly_feasible does
 *   xtol, gtol, ftol, maxit   as normalised at src/lsqfit/_scipy.py:124-132
 *   scaler   1 = More' column scaling (GSL scaler='more', scipy x_scale='jac'); 0 = none
 *   polish   max number of undamped Gauss-Newton refinement steps taken after the trust-region
 *            loop has stopped (0 = none; they count in d_nit)
 * Outputs (device): d_x [B][np], d_chi2 [B] (= sum f^2, __init__.py:667),
 *   d_cov [B][np][np] (= inv(J^T J), __init__.py:668), d_logdet [B] (= log det J^T J,
 *   __init__.py:712-719), d_nit [B] (function evaluations, _scipy.py:167),
 *   d_status [B] solver status 0 maxit / 1 gtol / 2 ftol / 3 xtol / 4 ftol+xtol /
 *   -1 non-finite start (map to stopping_criterion with {0:0,1:2,2:3,3:1,4:1},
 *   _scipy.py:178-181); optional d_f [B][nchiv], d_J [B][nchiv][np] (NULL to skip). */
int b200lm_fit_batch(b200lm_handle h, int B,
                     const double* d_mean, long long mean_stride,
                     const double* d_p0, long long p0_stride,
                     double xtol, double gtol, double ftol, int maxit, int scaler, int polish,
                     double* d_x, double* d_chi2, double* d_cov, double* d_logdet,
                     int* d_nit, int* d_status, double* d_f, double* d_J, void* stream);

/* Same call with HOST buffers: copies inputs to the device, runs the batch, copies the
 * results back and synchronises.  This is the call the Python plugin makes for users
 * whose data live in numpy arrays (and the path bench.py reports as `e2e`). */
int b200lm_fit_batch_host(b200lm_handle h, int B,
                          const double* h_mean, long long mean_stride,
                          const double* h_p0, long long p0_stride,
                          double xtol, double gtol, double ftol, int maxit, int scaler, int polish,
                          double* h_x, double* h_chi2, double* h_cov, double* h_logdet,
                          int* h_nit, int* h_status, double* h_f, double* h_J);

/* totals of the last fit_batch on this handle: out[0] function evaluations, out[1] Jacobian
 * evaluations, out[2] Cholesky factorisations.  Synchronises the handle's last stream. */
int b200lm_last_stats(b200lm_handle h, unsigned long long out[3]);
/* diagnostics: the first n (<= 16) counters of the last fit_batch.  [0..2] as above; [3..5] SM cycles the
 * driving warps spent in evaluations / in the trust-region sub-problem / in total; [6..10] leader cycles of the
 * team kernel's evaluation phases (prior + 1x1 rows, model rows, W.G, normal equations, reduction). */
int b200lm_last_stats_ex(b200lm_handle h, unsigned long long* out, int n);
/* warps per fit used by the last fit_batch launch: 1 (one warp per fit), 2 or 4 (team kernel) */
int b200lm_last_team(b200lm_handle h);
/* choose the kernel: 0 = default policy (by problem shape only, never by batch size -- a fit's bits must not depend on
 * the batch it is in: two warps per fit where one trial point is expensive -- np >= 12 and a correlated block of >= 32
 * points -- else one), 1 = one warp per fit, 2 / 4 = team kernel (4: lowest latency per trial point, best for batches
 * of a few hundred fits), 32 = wave kernel (highest throughput on saturated batches).  The kernels sum in a different
 * order: results agree to rounding, not bit for bit. */
int b200lm_set_team(b200lm_handle h, int team);
/* order of the work queue: -1 / 0 = input order (default), 1 = fits with the largest chi2 at their start point first
 * (one extra evaluation per fit + a device ranking pass; B <= 40000).  A batch is bounded by its slowest fits, and handing
 * out the fits expected to run longest first CAN shorten it (one C3 batch of 10^4 copies: 12.3 -> 11.6 ms) -- but the
 * start-point chi2 predicts the evaluation count only weakly, and over eight different batches the mean gain is zero
 * (tools/order_seeds.py), so it is off unless asked for.  Scheduling only: every fit is computed exactly as in input
 * order (the reference's iterators, src/lsqfit/__init__.py:1548-1642, run the copies one after the other).
 * b200lm_last_order: 1 if the last fit_batch used an ordered queue. */
int b200lm_set_order(b200lm_handle h, int mode);
int b200lm_last_order(b200lm_handle h);
/* trust-region decisions of the following fit_batch calls on this handle:
 *   0 = those of the solver behind lsqfit.scipy_least_squares (scipy trf, src/lsqfit/_scipy.py:156-161) -- default;
 *   1 = those of lsqfit.gsl_multifit with alg='lm' (src/lsqfit/_gsl.pyx:563-723: GSL's gsl_multifit_nlinear trust
 *       driver with the Levenberg-Marquardt sub-problem): Nielsen's update of the LM parameter, accept iff rho > 0,
 *       GSL's xtol / gtol tests.  With this policy d_nit counts ITERATIONS (gsl_multifit_nlinear_niter, _gsl.pyx:713),
 *       maxit limits iterations, scaler may also be 2 (= 'marquardt'), and d_status is 0 (maxit), 11 (info 1: xtol),
 *       12 (info 2: gtol) or 14 (info 27: no progress in the first iteration) -- stopping_criterion = status - 10
 *       (_gsl.pyx:689-701). */
int b200lm_set_policy(b200lm_handle h, int policy);
/* bound constraints of the following fit_batch calls on this handle: scipy's ``bounds`` (lsqfit.scipy_least_squares(
 * bounds=...), src/lsqfit/_scipy.py:77).  h_lb, h_ub: HOST arrays of np entries in device parameter order, -inf / +inf
 * for "no bound"; one box for every fit of a batch.  NULL, NULL clears the bounds, and so do bounds that are all
 * infinite (scipy then runs its unbounded trf: the results are those of an unbounded batch, bit for bit).
 * B200LM_EINVAL for lb >= ub in any entry or a NaN.  A bounded batch runs scipy's trf_bounds decisions (Coleman-Li
 * scaling, reflective select_step) in the one-warp kernel: team and wave requests are overridden (b200lm_last_team
 * reports 1), polish is skipped (undamped steps would leave the box), and the GSL policy is refused (EINVAL at
 * fit_batch).  b200lm_fit_batch projects every start into the box (scipy's make_strictly_feasible with rstep=1e-10);
 * b200lm_fit_batch_host refuses a host p0 outside the box ("`x0` is infeasible.", as scipy does).  Every returned x
 * lies in the box. */
int b200lm_set_bounds(b200lm_handle h, const double* h_lb, const double* h_ub);
/* number of kernel launches issued through this handle so far */
long long b200lm_launch_count(b200lm_handle h);

/* ---- residual / Jacobian test hook ----------------------------------------------------
 * chiv(p) and its Jacobian at B parameter vectors (src/lsqfit/_utilities.pyx:65-94 called
 * with floats and with valder+p, src/lsqfit/_scipy.py:146-154).  d_f [B][nchiv],
 * d_J [B][nchiv][np], d_chi2 [B]; any may be NULL. */
int b200lm_residual_jacobian(b200lm_handle h, int B, const double* d_p, long long p_stride,
                             const double* d_mean, long long mean_stride,
                             double* d_f, double* d_J, double* d_chi2, void* stream);

/* ---- whitening (svdcut / eps) ----------------------------------------------------------
 * Replaces gvar.PDF(concat(y, prior), svdcut=, eps=) for the correlated blocks
 * (call sites src/lsqfit/__init__.py:1895,1898; semantics doc/source/overview.rst:1546-1611).
 * Batched over nblk blocks on `device`; block k is n[k] x n[k], stored contiguously one
 * after another in d_cov (row-major).  Per block: D = diag^-1/2, corr = D cov D,
 * eigen-decomposition by parallel Jacobi (n <= 112: one CTA per block in shared memory; larger blocks:
 * pivoted Cholesky + one-sided block Jacobi over the whole GPU, two-sided block Jacobi as fallback), then
 *   svdcut > 0 : eigenvalues < svdcut*max are replaced by svdcut*max (nmod counts them)
 *   svdcut < 0 : those modes are dropped (nout[k] < n[k])
 *   use_eps    : corr += eps*norm_inf(corr) I and inverse-Cholesky instead; a non-positive pivot (block not positive
 *                definite after the shift) is reported as d_nmod[k] = -(pivot index + 1)
 * Outputs: d_w (same layout as d_cov) rows W[i] = val_i^-1/2 vec_i D, largest eigenvalue
 * first, unused rows zero (for blocks > 112 the rows of the clamped null space are an arbitrary
 * orthonormal basis of it -- W^T W, i.e. the inverse of the corrected covariance, is the same); d_cov_out the corrected covariance; d_nout, d_nmod [nblk];
 * d_logdet [nblk] (log det of the corrected block).  h_n is a host array. */
int b200lm_whiten(int device, int nblk, const int* h_n, const double* d_cov,
                  double svdcut, double eps, int use_eps,
                  double* d_w, double* d_cov_out, int* d_nout, int* d_nmod, double* d_logdet,
                  void* stream);

/* ---- covariance propagation -----------------------------------------------------------
 * Replaces nonlinear_fit._getp (src/lsqfit/__init__.py:897-922) with its chivw call
 * (src/lsqfit/_utilities.pyx:110-139):  D = cov . G^T . C^-1  (np x N, derivative of the
 * best-fit parameters with respect to y(+)prior) and  cov(p) = D . C . D^T  with C the
 * (svd-corrected) covariance of y(+)prior given densely in d_C [N][N] (shared by the batch).
 * d_x, d_cov [B][...] are the fit results; outputs d_D [B][np][N], d_covp [B][np][np]. */
int b200lm_propagate(b200lm_handle h, int B, const double* d_x, const double* d_cov,
                     const double* d_C, double* d_D, double* d_covp, void* stream);

/* ---- dense FP64 GEMM on the DMMA path ---------------------------------------------------
 * C[b] (M x N) = alpha * op(A[b]) . op(B[b]) + beta * C[b], all row-major fp64, batch strides in
 * elements (0 = operand shared by the batch).  transA: A is stored [K][M]; transB: B is stored
 * [N][K].  This is the building block of the dense side of the path -- W.[G|delta] and J^T J of
 * src/lsqfit/_utilities.pyx:20-36, 90-93 at config-5 sizes, and the D / D C D^T products of
 * nonlinear_fit._getp (src/lsqfit/__init__.py:897-922); exported for tests and for host drivers. */
int b200lm_dgemm(int device, int transA, int transB, int batch, int M, int N, int K, double alpha,
                 const double* d_A, long long sA, int lda, const double* d_B, long long sB, int ldb,
                 double beta, double* d_C, long long sC, int ldc, void* stream);

/* ---- single-fit row kernels: ONE fit, parallel over its data rows ----------------------------
 * Un-whitened model rows of the handle's functor at d_p[np]:  d_G (ny x np, leading dimension ld >= np; NULL for a
 * residual-only evaluation) = df/dp,  d_delta[ny] = f(p) - d_y.  Replaces fcn(x, p) on GVars and the delta of
 * src/lsqfit/_utilities.pyx:76-77 for any registered functor; the dense path multiplies by the whitening with
 * b200lm_dgemm.  Needs b200lm_set_const only. */
int b200lm_model_rows(b200lm_handle h, const double* d_p, const double* d_y, double* d_G, int ld, double* d_delta,
                      void* stream);
/* Uncorrelated data (1x1 weights d_w[ny] = 1/sigma, src/lsqfit/_utilities.pyx:85-89), np <= 8: one pass over the rows
 * gives d_out = [ packed upper triangle of J^T J (row-major, i <= j) | J^T r (np) | r^T r ] for r = w (f(p) - y) --
 * the normal equations of a fit with millions of points and a handful of parameters (examples/uncorrelated.py:30-41).
 * HBM bound (x, y, w are read once); deterministic (fixed-order reduction). */
int b200lm_normal_diag(b200lm_handle h, const double* d_p, const double* d_y, const double* d_w, double* d_out,
                       void* stream);

/* ---- dense single-fit path (config 5: np in the thousands) ------------------------------
 * Multi-exponential correlator with K exponentials: un-whitened model rows at parameters
 * d_p = [a_0..a_K-1, E_0..E_K-1]:  d_G (ny x 2K, leading dimension ld >= 2K; may be NULL for a
 * residual-only evaluation) = df/dp,  d_delta[ny] = f(p) - y.  Feeds b200lm_dgemm with the
 * whitening matrix; replaces fcn(x, p) on GVar object arrays + the delta of
 * src/lsqfit/_utilities.pyx:76-77. */
int b200lm_multiexp_dense(int device, int ny, int K, const double* d_t, const double* d_p,
                          const double* d_y, double* d_G, int ld, double* d_delta, void* stream);

/* Blocked Cholesky  L L^T = A + shift*I  (lower, row-major; d_L may equal d_A).  d_linv receives
 * the inverted 64 x 64 diagonal blocks (ceil(n/64) * 4096 doubles) used by b200lm_trsm.  *d_info
 * (device int) = 0 or the 1-based index of the first non-positive pivot.  Stands in for the
 * per-iteration LAPACK SVD of scipy's trf behind src/lsqfit/_scipy.py:156-161. */
int b200lm_potrf(int device, int n, const double* d_A, int lda, double shift, double* d_L, int ldl,
                 double* d_linv, int* d_info, void* stream);

/* Triangular solve with the factor of b200lm_potrf: trans = 0: L X = B, trans = 1: L^T X = B.
 * B (n x nrhs, row-major) is workspace and is destroyed; X must not alias B.  With B = I twice
 * this gives the parameter covariance (J^T J)^-1 of src/lsqfit/_scipy.py:171-175. */
int b200lm_trsm(int device, int n, int nrhs, const double* d_L, int ldl, const double* d_linv, int trans,
                double* d_B, int ldb, double* d_X, int ldx, void* stream);

/* ---- bootstrap / simulated copies of the means (SURVEY 8f-1) ------------------------------
 * d_z[count] <- standard normals number first .. first+count-1 of the stream keyed by `seed`
 * (Philox4x32-10, counter = pair index, Box-Muller on 53-bit uniforms); any sub-range is
 * bit-identical to the same elements of a larger call.  d_raw (may be NULL) receives the four raw
 * Philox words of every pair touched (known-answer testing). */
int b200lm_normals(int device, long long first, long long count, unsigned long long seed, double* d_z,
                   unsigned int* d_raw, void* stream);

/* d_out[b][0..N) = d_mean + L z_b for copies first .. first+B-1, z_b = normals [(first+b)*M, +M) of
 * the stream, L row-major N x M (L L^T = covariance of y (+) prior after the svd correction); d_z is
 * a B*M workspace that returns the normals.  Replaces gvar.bootstrap_iter / raniter as driven by
 * src/lsqfit/__init__.py:1532-1535 and 1615-1624 (one Python iteration per copy there). */
int b200lm_bootstrap_means(int device, long long B, long long first, int N, int M, const double* d_mean,
                           const double* d_L, int ldl, unsigned long long seed, double* d_z,
                           double* d_out, long long out_stride, void* stream);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink / NVSwitch (SURVEY 8(b), 8(e)) ----------------------------
 * Batches shard over the ranks by fit index and are fitted without any exchange; afterwards the packed per-fit results
 * are gathered and moment buffers summed.  The reference has no counterpart (its iterators run copy by copy in one
 * process, src/lsqfit/__init__.py:1612-1624); these calls are what a multi-process driver binds.
 *   b200lm_comm_unique_id  rank 0 creates the 128-byte NCCL id; the caller ships it to the other ranks (any host channel)
 *   b200lm_comm_init       every rank, with the same id
 *   b200lm_gather          d_recv[world * count] = concatenation in rank order of every rank's d_send[count]
 *   b200lm_allreduce_sum   d_buf[count] <- sum over ranks, in place
 * Device pointers, fp64, asynchronous on `stream`.  NCCL is bound at run time (libnccl.so.2). */
int b200lm_comm_unique_id(char* out128);
int b200lm_comm_init(int device, int rank, int world, const char* id128, b200lm_comm* out);
void b200lm_comm_destroy(b200lm_comm c);
int b200lm_comm_rank(b200lm_comm c);
int b200lm_comm_world(b200lm_comm c);
int b200lm_gather(b200lm_comm c, const double* d_send, double* d_recv, long long count_per_rank, void* stream);
int b200lm_allreduce_sum(b200lm_comm c, double* d_buf, long long count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200LM_H */
