// Internal plan / argument structures shared by the kernels and the C-ABI layer.
#pragma once
#include <cuda_runtime.h>

namespace b200lm {

// One correlated block of the whitening (entry k>=1 of the reference's
// yp_pdf.i_invwgts, reference src/lsqfit/_utilities.pyx:90-93).
struct BlockDesc {
    int n_in;        // number of y(+)prior entries in the block
    int n_out;       // number of residuals it produces (rows of W_k; < n_in if svdcut<0 dropped modes)
    int ldw;         // row stride of the zero-padded, row-major weight matrix (== 4 mod 16, >= n_in)
    int idx_off;     // offset into blk_idx[]  (n_in entries: index into y(+)prior)
    int wt_off;      // offset into blk_wt[]   (W[r*ldw + k], n_out rounded up to 8 rows)
    int chiv_off;    // first residual slot of this block in chiv
    int ldw2;        // team kernel copy: row stride (== 8 mod 16, >= n_in rounded up to 8)
    int wt2_off;     // offset into blk_wt2[]
};

// One window of a window scan (b200lm_set_windows): its part of the concatenated row tables of FitParams.
// BlockDesc::idx_off and wt_off address the concatenated blk_idx / blk_wt, chiv_off the window's own residual vector.
struct WinDesc {
    int nd_fn, nd_pr, nblk, nchiv;
    int dfn_off, dpr_off, blk_off;
};

// normal_diag_kernel (lm_rows.cuh): rows of the per-CTA partial buffer that b200lm_normal_diag allocates per SM
constexpr int ND_MAX_PARTS_PER_SM = 8;

struct FitParams {
    // ---- problem description (shared by every fit of the batch) ----------
    int ny, np, N, nchiv, nx, noprior;
    const double* x;            // [ny][nx] functor constants
    int nd_fn;                  // 1x1 blocks that are data rows
    const int* dfn_idx;         //   data row index (< ny)
    const double* dfn_w;        //   1/sigma
    int nd_pr;                  // 1x1 blocks that are prior rows
    const int* dpr_idx;         //   index into y(+)prior (>= ny)
    const double* dpr_w;
    int nblk;
    const BlockDesc* blk;
    const int* blk_idx;
    const double* blk_wt;
    int wt_total;               // doubles in blk_wt
    const double* blk_wt2;      // the same weights in the team kernel's layout (BlockDesc::ldw2)
    int wt2_total;
    int wt_in_smem;             // stage blk_wt in shared memory
    int rb;                     // rows of the per-warp row buffer
    int dual_from;              // from this evaluation count on, the secular equation is evaluated at two
                                // values of alpha per factorisation round (np <= 16); < 0: never
    int warps;                  // warps per CTA
    int nblk_idx;               // entries of blk_idx (sum of n_in)
    int staged;                 // team kernel: weights AND the index / x tables are staged in shared memory
    int team_stride;            // team kernel: doubles of shared memory per team
    int team;                   // warps per fit: 0/1 = one warp per fit (fit_kernel), 2 or 4 = fit_team_kernel
    // ---- batch ------------------------------------------------------------
    int B;
    const double* mean;         // [B][N] (mean_stride = N) or shared (mean_stride = 0)
    long long mean_stride;
    const double* p0;           // [B][np] or shared (p0_stride = 0)
    long long p0_stride;
    double xtol, gtol, ftol;
    int maxit;
    int scaler;                 // 0: none (scipy x_scale=1), 1: More' (scipy 'jac', GSL 'more')
    int polish;                 // max Gauss-Newton refinement steps after the trust-region loop stops
    int finalize_only;          // 1: the fits are done (d_x = solutions, status given): only covariance, log det, f / J, polish
    int policy;                 // 0: scipy TRF decisions (src/lsqfit/_scipy.py:156-161); 1: GSL trust/lm decisions
                                // (gsl_multifit_nlinear behind src/lsqfit/_gsl.pyx:563-723; scaler 2 = marquardt)
    // ---- outputs (any of f_out, J_out, cov, logdet may be null) ----------------
    double* x_out;              // [B][np]
    double* chi2;               // [B]
    double* cov;                // [B][np][np]
    double* logdet;             // [B]  log det(J^T J)
    int* nit;                   // [B]  function evaluations (scipy nfev); policy 1: iterations (gsl niter)
    int* status;                // [B]  scipy status: 0 maxit, 1 gtol, 2 ftol, 3 xtol, 4 both, -1 non-finite start;
                                //      policy 1: 0 maxit, 11 xtol (info 1), 12 gtol (info 2), 14 no progress (info 27)
    double* f_out;              // [B][nchiv]
    double* J_out;              // [B][nchiv][np]
    int* counter;               // work-queue head (zeroed before launch)
    double* wave_A;             // optional [B][np(np+1)/2]: packed J^T J at the solution, written by the wave kernel for its
                                // finalisation pass (which then needs no evaluation of its own)
    const int* order;           // optional: the queue hands out fit order[i] instead of fit i (longest-expected first)
    unsigned long long* stats;  // [0] total nfev, [1] total jacobian evals, [2] total factorisations
    // ---- bound constraints (last: the offsets of every field above are those of the kernels without bounds) ----
    const double* lb;           // [np] lower bounds (-inf: none), device parameter order
    const double* ub;           // [np] upper bounds (+inf: none)
    int bounded;                // 1: scipy's trf_bounds decisions (fit_kernel<F, 3>); lb / ub are set
    // ---- fit windows (last, for the same reason; b200lm_set_windows) ----
    int nwin;                   // > 0: fit b is copy b % win_copies of window b / win_copies (fit_kernel<F, 4>); the
                                // tables above (dfn_*, dpr_*, blk, blk_idx, blk_wt) hold every window, one after the other
    int win_copies;
    const WinDesc* win;         // [nwin]
};

}  // namespace b200lm
