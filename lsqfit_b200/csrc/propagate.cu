// Post-fit covariance propagation for fit.p as dense fp64 GEMMs (DMMA kernel of csrc/dgemm.cuh).
//
// Replaces nonlinear_fit._getp (reference src/lsqfit/__init__.py:897-922) and the chivw
// call inside it (src/lsqfit/_utilities.pyx:110-139):
//     D      = cov . G^T . C^-1 = (cov . J^T) . W        (np x N)   W = whitening operator
//     cov(p) = D . C . D^T                                (np x np)
// where J = W [G; I] is the whitened Jacobian at the solution (recomputed by the
// residual/Jacobian kernel), W is the dense [nchiv][N] form of yp_pdf.i_invwgts and C is
// the (svd-corrected) covariance of y(+)prior.  The reference builds D column by column in
// a Python loop over N GVars (:907-911) and each p[a] with wsum_der (:914-918).
#include <cuda_runtime.h>
#include <vector>
#include "../../include/b200lm.h"
#include "handle.h"
#include "dgemm.cuh"

using namespace b200lm;

// at least `need` bytes of h->d_scratch
static cudaError_t scratch(b200lm_handle h, size_t need) {
    if (need > h->scratch_bytes) {
        if (h->d_scratch) cudaFree(h->d_scratch);
        h->d_scratch = nullptr; h->scratch_bytes = 0;
        cudaError_t e = cudaMalloc((void**)&h->d_scratch, need);
        if (e != cudaSuccess) return e;
        h->scratch_bytes = need;
    }
    h->scratch_counter_clean = false;          // (b200lm_normal_diag keeps an arrival counter in this buffer)
    return cudaSuccess;
}

extern "C" int b200lm_propagate(b200lm_handle h, int B, const double* d_x, const double* d_cov,
                                const double* d_C, double* d_D, double* d_covp, void* stream) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (!h->have_weights || !h->have_const) return set_error(h, B200LM_EINVAL, "plan is not complete");
    if (h->nwin > 0) return set_error(h, B200LM_EINVAL, "propagate is not built for window scans");
    if (B < 0 || !d_x || !d_cov || !d_D) return set_error(h, B200LM_EINVAL, "NULL required argument");
    if (d_covp && !d_C) return set_error(h, B200LM_EINVAL, "d_C is required for cov(p)");
    if (B == 0) return B200LM_OK;
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return cuda_fail(h, e, "cudaSetDevice");
    cudaStream_t s = (cudaStream_t)stream;
    const int np = h->np, N = h->N, nchiv = h->nchiv;
    // dense whitening operator W [nchiv][N], built once per weight set
    if (!h->d_wfull) {
        const WeightTables& t = h->rows.host;
        std::vector<double> W((size_t)nchiv * N, 0.0);
        const int nfn = (int)t.fn_idx.size();      // 1x1 rows: data rows first, then prior rows
        for (int i = 0; i < nfn; ++i) W[(size_t)i * N + t.fn_idx[i]] = t.fn_w[i];
        for (size_t i = 0; i < t.pr_idx.size(); ++i) W[(nfn + i) * N + t.pr_idx[i]] = t.pr_w[i];
        for (auto& b : t.blk)
            for (int r = 0; r < b.n_out; ++r)
                for (int j = 0; j < b.n_in; ++j)
                    W[(size_t)(b.chiv_off + r) * N + t.blk_idx[b.idx_off + j]] = t.wt[b.wt_off + (size_t)r * b.ldw + j];
        e = cudaMalloc((void**)&h->d_wfull, W.size() * sizeof(double));
        if (e == cudaSuccess) e = cudaMemcpy(h->d_wfull, W.data(), W.size() * sizeof(double), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) return cuda_fail(h, e, "upload dense whitening operator");
    }
    // scratch: J [B][nchiv][np], M [B][np][nchiv], T [B][np][N]
    const size_t nJ = (size_t)B * nchiv * np, nM = nJ, nT = (size_t)B * np * N;
    e = scratch(h, (nJ + nM + nT) * sizeof(double));
    if (e != cudaSuccess) return cuda_fail(h, e, "scratch allocation");
    double* dJ = h->d_scratch;
    double* dM = dJ + nJ;
    double* dT = dM + nM;
    // J at the solution.  The residual/Jacobian kernel needs a mean vector only for the
    // residuals, which are not used here: the zeroed head of the D buffer serves as a dummy.
    e = cudaMemsetAsync(d_D, 0, (size_t)N * sizeof(double), s);
    if (e != cudaSuccess) return cuda_fail(h, e, "memset");
    int rc = b200lm_residual_jacobian(h, B, d_x, np, d_D, 0, nullptr, dJ, nullptr, stream);
    if (rc) return rc;
    // M = cov . J^T      (np x nchiv)
    e = dgemm(false, true, B, np, nchiv, np, 1.0, d_cov, (long long)np * np, np, dJ, (long long)nchiv * np, np,
              0.0, dM, (long long)np * nchiv, nchiv, s);
    // D = M . W          (np x N)
    if (e == cudaSuccess)
        e = dgemm(false, false, B, np, N, nchiv, 1.0, dM, (long long)np * nchiv, nchiv, h->d_wfull, 0, N,
                  0.0, d_D, (long long)np * N, N, s);
    if (e == cudaSuccess && d_covp) {
        // T = D . C ; cov(p) = T . D^T
        e = dgemm(false, false, B, np, N, N, 1.0, d_D, (long long)np * N, N, d_C, 0, N, 0.0, dT, (long long)np * N, N, s);
        if (e == cudaSuccess)
            e = dgemm(false, true, B, np, np, N, 1.0, dT, (long long)np * N, N, d_D, (long long)np * N, N,
                      0.0, d_covp, (long long)np * np, np, s);
    }
    if (e != cudaSuccess) return cuda_fail(h, e, "propagate");
    h->launches += d_covp ? 4 : 2;
    h->last_stream = s;
    return B200LM_OK;
}

// ---- fit.p of a fit-window scan -----------------------------------------------------------------------------------
// Window w is its own nonlinear_fit of the rows of the shared y(+)prior that it lists, so its parameters depend on
// y(+)prior through  D_w = cov_w . J_w^T . W_w  [np][N]  (W_w: the window's whitening, zero columns outside it), and
//     cov(p_w, p_v) = D_w . C . D_v^T     (w != v: the windows share the data and prior, C their input covariance)
//     cov(p_w, p_w) = D_w . C_w . D_w^T   (C_w = C + Delta_w: each window's svd cut adds its own, independent, part)
// M_w = cov_w J_w^T and the joint product are DMMA GEMMs; W_w is applied from the window row tables
// (window_dcols_kernel), and the diagonal blocks get D_w Delta_w D_w^T over the window's correlated blocks
// (window_covp_finish_kernel).  Every output element is written by one thread in a fixed order: no atomics.

struct WinPropArgs {
    int nwin, np, N, nchiv;
    const WinDesc* win;
    const int* fn_idx; const double* fn_w;
    const int* pr_idx; const double* pr_w;
    const BlockDesc* blk; const int* blk_idx; const double* wt;
    const double* M;            // [nwin][np][nchiv]
    double* D;                  // [nwin][np][N], zero outside the window (cleared before)
    const double* dC;           // svd corrections, n_in x n_in per block in set_windows order, or null
    double* covp;               // [nwin*np][nwin*np]
};

// D_w[:, i] = sum_r M_w[:, r] W_w[r, i].  CTA w < nwin: window w's 1x1 data and prior rows; CTA nwin + g: correlated
// block g of the concatenated tables, in the window whose blk_off is the last one <= g (windows without blocks share
// their blk_off with the next window).  b200lm_set_windows checked that each column of a window has exactly one row
// source.
__global__ void __launch_bounds__(256) window_dcols_kernel(const __grid_constant__ WinPropArgs a) {
    const int np = a.np;
    const bool rows1 = (int)blockIdx.x < a.nwin;
    const int g = (int)blockIdx.x - a.nwin;
    int w = blockIdx.x;
    if (!rows1) {
        int lo = 0, hi = a.nwin - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) / 2;
            if (a.win[mid].blk_off <= g) lo = mid; else hi = mid - 1;
        }
        w = lo;
    }
    const WinDesc d = a.win[w];
    const double* M = a.M + (size_t)w * np * a.nchiv;
    double* D = a.D + (size_t)w * np * a.N;
    if (rows1) {
        // chiv rows: data rows first, then prior rows
        const int n1 = d.nd_fn + d.nd_pr;
        for (int e = threadIdx.x; e < np * n1; e += blockDim.x) {
            const int p = e / n1, r = e % n1;
            const bool fn = r < d.nd_fn;
            const int col = fn ? a.fn_idx[d.dfn_off + r] : a.pr_idx[d.dpr_off + r - d.nd_fn];
            const double wr = fn ? a.fn_w[d.dfn_off + r] : a.pr_w[d.dpr_off + r - d.nd_fn];
            D[(size_t)p * a.N + col] = M[(size_t)p * a.nchiv + r] * wr;
        }
        return;
    }
    const BlockDesc b = a.blk[g];
    for (int e = threadIdx.x; e < np * b.n_in; e += blockDim.x) {
        const int p = e / b.n_in, j = e % b.n_in;
        const double* m = M + (size_t)p * a.nchiv + b.chiv_off;
        const double* wj = a.wt + b.wt_off + j;
        double s = 0.0;
        for (int r = 0; r < b.n_out; ++r) s = fma(m[r], wj[(size_t)r * b.ldw], s);
        D[(size_t)p * a.N + a.blk_idx[b.idx_off + j]] = s;
    }
}

// Blocks (w, v), v <= w, of the joint covariance: (S + S^T) / 2 for v < w; for v == w also + D_w Delta_w D_w^T, in
// row chunks of 32 of each correlated block (t = Delta rows . D^T in shared memory, then D . t).
constexpr int WP_CHUNK = 32;
__global__ void __launch_bounds__(256) window_covp_finish_kernel(const __grid_constant__ WinPropArgs a) {
    const int w = blockIdx.y, v = blockIdx.x, np = a.np, nn = np * np;
    if (v > w) return;
    const size_t ld = (size_t)a.nwin * np;
    double* S = a.covp;
    if (v < w) {
        for (int e = threadIdx.x; e < nn; e += blockDim.x) {
            const int i = e / np, j = e % np;
            double* x = S + (w * (size_t)np + i) * ld + v * (size_t)np + j;
            double* y = S + (v * (size_t)np + j) * ld + w * (size_t)np + i;
            const double s = 0.5 * (*x + *y);
            *x = s; *y = s;
        }
        return;
    }
    extern __shared__ double wp_smem[];
    double* corr = wp_smem;                 // [np][np]
    double* t = wp_smem + nn;               // [WP_CHUNK][np]
    for (int e = threadIdx.x; e < nn; e += blockDim.x) corr[e] = 0.0;
    if (a.dC) {
        const WinDesc d = a.win[w];
        const double* D = a.D + (size_t)w * np * a.N;
        size_t off = 0;
        for (int g = 0; g < d.blk_off; ++g) off += (size_t)a.blk[g].n_in * a.blk[g].n_in;
        for (int k = 0; k < d.nblk; ++k) {
            const BlockDesc b = a.blk[d.blk_off + k];
            const int n = b.n_in;
            const int* idx = a.blk_idx + b.idx_off;
            const double* dc = a.dC + off;
            for (int i0 = 0; i0 < n; i0 += WP_CHUNK) {
                const int m = n - i0 < WP_CHUNK ? n - i0 : WP_CHUNK;
                __syncthreads();
                for (int e = threadIdx.x; e < m * np; e += blockDim.x) {
                    const int ii = e / np, c = e % np;
                    const double* row = dc + (size_t)(i0 + ii) * n;
                    const double* Dc = D + (size_t)c * a.N;
                    double s = 0.0;
                    for (int j = 0; j < n; ++j) s = fma(row[j], Dc[idx[j]], s);
                    t[e] = s;
                }
                __syncthreads();
                for (int e = threadIdx.x; e < nn; e += blockDim.x) {
                    const int r = e / np, c = e % np;
                    const double* Dr = D + (size_t)r * a.N;
                    double s = corr[e];
                    for (int ii = 0; ii < m; ++ii) s = fma(Dr[idx[i0 + ii]], t[ii * np + c], s);
                    corr[e] = s;
                }
            }
            off += (size_t)n * n;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nn; e += blockDim.x) {
        const int i = e / np, j = e % np;
        if (j > i) continue;
        double* x = S + (w * (size_t)np + i) * ld + w * (size_t)np + j;
        double* y = S + (w * (size_t)np + j) * ld + w * (size_t)np + i;
        const double s = 0.5 * (*x + *y) + 0.5 * (corr[i * np + j] + corr[j * np + i]);
        *x = s; *y = s;
    }
}

extern "C" int b200lm_window_propagate(b200lm_handle h, const double* d_cov, const double* d_J, const double* d_C,
                                       const double* d_dC, double* d_D, double* d_covp, void* stream) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (h->nwin == 0) return set_error(h, B200LM_EINVAL, "no windows set (b200lm_set_windows)");
    if (!d_cov || !d_J || !d_D) return set_error(h, B200LM_EINVAL, "NULL required argument");
    if (d_covp && !d_C) return set_error(h, B200LM_EINVAL, "d_C is required for cov(p)");
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return cuda_fail(h, e, "cudaSetDevice");
    cudaStream_t s = (cudaStream_t)stream;
    const int nwin = h->nwin, np = h->np, N = h->N, nchiv = h->nchiv;
    const long long R = (long long)nwin * np;            // rows of D_all = [D_0; D_1; ...]
    // scratch: M [nwin][np][nchiv], T = D_all . C [nwin*np][N]
    const size_t nM = (size_t)R * nchiv, nT = d_covp ? (size_t)R * N : 0;
    e = scratch(h, (nM + nT) * sizeof(double));
    if (e != cudaSuccess) return cuda_fail(h, e, "scratch allocation");
    double* dM = h->d_scratch;
    double* dT = dM + nM;
    const RowTables& t = h->win_rows;
    WinPropArgs a;
    a.nwin = nwin; a.np = np; a.N = N; a.nchiv = nchiv; a.win = h->d_win;
    a.fn_idx = t.d_fn_idx; a.fn_w = t.d_fn_w; a.pr_idx = t.d_pr_idx; a.pr_w = t.d_pr_w;
    a.blk = t.d_blk; a.blk_idx = t.d_blk_idx; a.wt = t.d_wt;
    a.M = dM; a.D = d_D; a.dC = d_dC; a.covp = d_covp;
    const int nblk = (int)t.host.blk.size();
    int launches = 0;
    // M_w = cov_w . J_w^T      (np x nchiv; rows of J beyond the window's nchiv are 0)
    e = dgemm(false, true, nwin, np, nchiv, np, 1.0, d_cov, (long long)np * np, np, d_J, (long long)nchiv * np, np,
              0.0, dM, (long long)np * nchiv, nchiv, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_D, 0, (size_t)R * N * sizeof(double), s);
    if (e == cudaSuccess) {
        window_dcols_kernel<<<nwin + nblk, 256, 0, s>>>(a);
        e = cudaGetLastError();
    }
    launches += 2;
    if (e == cudaSuccess && d_covp) {
        // T = D_all . C ; S = T . D_all^T      ([nwin*np] x [nwin*np])
        e = dgemm(false, false, 1, (int)R, N, N, 1.0, d_D, 0, N, d_C, 0, N, 0.0, dT, 0, N, s);
        if (e == cudaSuccess) e = dgemm(false, true, 1, (int)R, (int)R, N, 1.0, dT, 0, N, d_D, 0, N, 0.0, d_covp, 0, (int)R, s);
        if (e == cudaSuccess) {
            window_covp_finish_kernel<<<dim3(nwin, nwin), 256, (size_t)(np * np + WP_CHUNK * np) * sizeof(double), s>>>(a);
            e = cudaGetLastError();
        }
        launches += 3;
    }
    if (e != cudaSuccess) return cuda_fail(h, e, "window propagate");
    h->launches += launches;
    h->last_stream = s;
    return B200LM_OK;
}
