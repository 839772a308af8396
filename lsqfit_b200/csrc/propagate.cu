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
    const size_t need = (nJ + nM + nT) * sizeof(double);
    if (need > h->scratch_bytes) {
        if (h->d_scratch) cudaFree(h->d_scratch);
        h->d_scratch = nullptr; h->scratch_bytes = 0;
        e = cudaMalloc((void**)&h->d_scratch, need);
        if (e != cudaSuccess) return cuda_fail(h, e, "scratch allocation");
        h->scratch_bytes = need;
    }
    h->scratch_counter_clean = false;          // (b200lm_normal_diag keeps an arrival counter in this buffer)
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
