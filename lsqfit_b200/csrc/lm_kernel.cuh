// Batched trust-region Levenberg-Marquardt: one warp per fit, persistent CTAs
// pulling fits from a device work queue, every decision kept on the device.
//
// What it replaces in the reference (paths relative to the reference tree):
//   * chiv.__call__            src/lsqfit/_utilities.pyx:65-94   (whiten + residual)
//   * Dfun / valder Jacobian   src/lsqfit/_scipy.py:144-154
//   * the fitter plugin        src/lsqfit/_scipy.py:156-181 / src/lsqfit/_gsl.pyx:563-723
//   * chi2 / logdet(J^T J)     src/lsqfit/__init__.py:665-682, 706-725
//
// Algorithm (host model: tests/lm_model.py).  The trust-region *decisions* are those
// of the solver behind the reference's scipy plugin (unbounded TRF: radius update
// 0.25/0.75, Delta0 = |x0*scale|, accept iff cost decreases, ftol/xtol/gtol tests),
// with More' column scaling (GSL `scaler='more'`, scipy x_scale='jac') by default.
// The Levenberg parameter is found by Newton iteration on the secular equation,
// evaluated with a Cholesky factorisation of the scaled normal matrix
//       d (J^T J) d + alpha I
// held in shared memory -- not by an SVD/QR of J.
//
// Data layout per warp (shared memory):
//   R[rb][LDR]   row buffer: rows of [G | delta] before whitening, [J | r] after
//   A[NP][LDA]   J^T J (unscaled)        L[NP][LDA]   Cholesky factor
//   p, pn, g, sinv, dsc, idg   NP-vectors
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include "lm_types.h"

namespace b200lm {

#define B200LM_FULL 0xffffffffu

// the counters cost a few hundred cycles per trial point: compiled in only with -DB200LM_PHASE_TICKS
// (python lsqfit_b200/build.py with B200LM_EXTRA_CFLAGS=-DB200LM_PHASE_TICKS; tools/phase_probe.py)
#ifdef B200LM_PHASE_TICKS
#define B200LM_CLOCK() clock64()
#else
#define B200LM_CLOCK() 0ll
#endif

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(B200LM_FULL, v, o);
    return v;
}
// several sums at once: the butterflies interleave, so the latency is that of ONE reduction
// (a 64-bit shuffle + add costs ~35 cycles per step on B200, and a trial point needs several norms)
__device__ __forceinline__ void warp_sum3(double& a, double& b, double& c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ta = __shfl_xor_sync(B200LM_FULL, a, o);
        const double tb = __shfl_xor_sync(B200LM_FULL, b, o);
        const double tc = __shfl_xor_sync(B200LM_FULL, c, o);
        a += ta; b += tb; c += tc;
    }
}
// sum of a and max of m in one pass
__device__ __forceinline__ void warp_sum_max(double& a, double& m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ta = __shfl_xor_sync(B200LM_FULL, a, o);
        const double tm = __shfl_xor_sync(B200LM_FULL, m, o);
        a += ta; m = fmax(m, tm);
    }
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(B200LM_FULL, v, o));
    return v;
}

// number of lanes a functor can spread one row's value_grad over (value_grad_part); specialised in functors.cuh
template <class F> struct SplitOf { static constexpr int value = 1; };

template <class F>
struct FitLayout {
    static constexpr int NP = F::NP;
    static constexpr int NP1 = NP + 1;
    // Row buffer columns: [ G or J (NP) | delta or r (1) | zero padding ].  The FP64 tensor
    // instruction (DMMA m8n8k4) consumes 8-column tiles:
    //   NTA tiles cover the NP Jacobian columns (J^T J),
    //   if NP is not a multiple of 8 the residual column rides in the padding of the last tile
    //   (DELTA_IN_TILE) and J^T r / r^T r fall out of the same tiles; otherwise the residual
    //   column is handled by plain DFMA (a ninth column would cost a whole extra tile).
    static constexpr int NTA = (NP + 7) / 8;
    static constexpr bool DELTA_IN_TILE = (NP % 8) != 0;
    static constexpr int NT = NTA;                         // tiles in the W.[G|delta] product
    static constexpr int NCOL = 8 * NT > NP1 ? 8 * NT : NP1;
    // leading dimension == 4 (mod 8): fragment loads (row = 4s + lane%4, col = 8t + lane/4)
    // then hit every shared-memory bank pair exactly twice (the minimum for 256 B)
    static constexpr int LDR = ((NCOL + 3) / 8) * 8 + 4;
    static constexpr int LDA = NP | 1;
    static constexpr int NVEC = 6;
    static constexpr int NTRI = NT * (NT + 1) / 2;         // upper-triangular tile pairs
    // register budget: 16 warps/CTA leave 128 registers per thread, 12 warps leave 168.  Measured on
    // C3 (NP=16): 12 warps beat 16 (19.1 vs 22.6 ms per 10k fits) -- per-warp latency and
    // instruction-cache pressure matter more than occupancy for this kernel.
    static constexpr int MAX_WARPS = NP > 10 ? 12 : 16;
    __host__ __device__ static int per_warp_doubles(int rb) {
        // R | dvec | A0 | A1 | L | vectors (+ second gradient).  A0/A1, g0/g1: the Jacobian is
        // evaluated speculatively at every trial point, so the normal equations of the current
        // point must survive a rejected trial.
        int n = rb * LDR + rb + 3 * NP * LDA + (NVEC + 1) * NP + 64;      // + column broadcast buffers
        return (n + 1) & ~1;
    }
};

template <class F>
struct WarpCtx {
    typedef FitLayout<F> Lay;
    const FitParams& P;
    const double* wt;       // whitening matrices (shared or global)
    const double* mean;     // this fit's y(+)prior means
    double *R, *dvec, *A, *L, *p, *pn, *g, *sinv, *dsc, *idg, *colb;
    double *Abuf[2], *gbuf[2];      // c.A / c.g point at the buffer the next evaluation writes
    int lane;
    __device__ WarpCtx(const FitParams& P_) : P(P_) {}
    // select buffer k (0 or 1) without indexing Abuf / gbuf at run time: a dynamic index would keep the whole
    // context in local memory
    __device__ __forceinline__ void use_buf(int k) {
        A = k ? Abuf[1] : Abuf[0];
        g = k ? gbuf[1] : gbuf[0];
    }
};

// D(8x8) += A(8x4) . B(4x8) on the FP64 tensor path.  Fragment ownership (PTX m8n8k4):
//   a = A[lane/4][lane%4]      b = B[lane%4][lane/4]      c0,c1 = C[lane/4][2*(lane%4) + {0,1}]
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------
// normal-equation accumulators in DMMA C-fragment layout (registers)
// ---------------------------------------------------------------------------
template <class F>
struct NormalAcc {
    typedef FitLayout<F> Lay;
    double t[Lay::NTRI][2];     // tiles (ta <= tb) of S^T S
    double g;                   // partial of J^T r for column (lane % 16 or lane) when !DELTA_IN_TILE
    double cost;                // partial of r^T r when !DELTA_IN_TILE
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int q = 0; q < Lay::NTRI; ++q) { t[q][0] = 0.0; t[q][1] = 0.0; }
        g = 0.0; cost = 0.0;
    }
};

// acc += S^T S over `nrows4` rows (multiple of 4; rows beyond the data are zero) of the row
// buffer S = [J | r | 0].  A-operand J^T and B-operand J are the same fragment.
template <class F>
__device__ __forceinline__ void mma_accumulate(WarpCtx<F>& c, const double* S, int nrows4, NormalAcc<F>& na) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, NT = Lay::NT, LDR = Lay::LDR;
    const int lane = c.lane;
    const double* base = S + (lane & 3) * LDR + (lane >> 2);
    for (int s4 = 0; s4 < nrows4; s4 += 4) {
        double f[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) f[t] = base[s4 * LDR + 8 * t];
        int q = 0;
#pragma unroll
        for (int ta = 0; ta < NT; ++ta)
#pragma unroll
            for (int tb = ta; tb < NT; ++tb) { dmma(na.t[q][0], na.t[q][1], f[ta], f[tb]); ++q; }
    }
    if (!Lay::DELTA_IN_TILE) {
        // J^T r by DFMA: lane (a + 16h) sums rows of half h for column a (NP <= 16), else lane a
        if (NP <= 16) {
            const int a = lane & 15, h = lane >> 4;
            if (a < NP) {
                const int half = nrows4 >> 1;
                for (int i = h * half; i < (h + 1) * half; ++i) na.g = fma(S[i * LDR + a], S[i * LDR + NP], na.g);
            }
        } else {
            if (lane < NP)
                for (int i = 0; i < nrows4; ++i) na.g = fma(S[i * LDR + lane], S[i * LDR + NP], na.g);
        }
        for (int i = lane; i < nrows4; i += 32) { const double r = S[i * LDR + NP]; na.cost = fma(r, r, na.cost); }
    }
}

// add the register tiles into shared A (J^T J), g (J^T r); returns this lane's share of r^T r
template <class F>
__device__ __forceinline__ double flush_normal(WarpCtx<F>& c, NormalAcc<F>& na) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, NT = Lay::NT, LDA = Lay::LDA;
    const int lane = c.lane;
    double cost = na.cost;
    int q = 0;
#pragma unroll
    for (int ta = 0; ta < NT; ++ta)
#pragma unroll
        for (int tb = ta; tb < NT; ++tb) {
            const int row = 8 * ta + (lane >> 2);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int col = 8 * tb + 2 * (lane & 3) + e;
                const double v = na.t[q][e];
                if (row < NP && col < NP) {
                    c.A[row * LDA + col] += v;
                    if (ta != tb) c.A[col * LDA + row] += v;
                } else if (Lay::DELTA_IN_TILE && col == NP && row < NP) {
                    c.g[row] += v;
                } else if (Lay::DELTA_IN_TILE && col == NP && row == NP) {
                    cost += v;
                }
            }
            ++q;
        }
    if (!Lay::DELTA_IN_TILE) {
        if (NP <= 16) {
            const double other = __shfl_xor_sync(B200LM_FULL, na.g, 16);
            if (lane < NP) c.g[lane] += na.g + other;
        } else if (lane < NP) {
            c.g[lane] += na.g;
        }
    }
    __syncwarp();
    return cost;
}

template <class F>
__device__ __forceinline__ void emit_rows(const double* S, int nrows, int slot0, int lane,
                                          double* fout, double* Jout) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDR = Lay::LDR;
    for (int i = lane; i < nrows; i += 32) {
        if (fout) fout[slot0 + i] = S[i * LDR + NP];
        if (Jout) {
#pragma unroll
            for (int j = 0; j < NP; ++j) Jout[(size_t)(slot0 + i) * NP + j] = S[i * LDR + j];
        }
    }
}

// Householder update of the triangular factor Rt (in c.A) with `nrows` rows of S, columns
// scaled by c.dsc:  Rt <- R of qr([Rt ; S.diag(dsc)]).  Rows are owned by lanes (i mod 32);
// S is destroyed.  Used for the final covariance: (J^T J)^-1 = dsc Rt^-1 Rt^-T dsc has a
// relative error ~kappa(J)*eps instead of kappa^2*eps for the normal equations.
template <class F>
__device__ __forceinline__ void qr_update(double* A, const double* dsc, double* S, int nrows, int lane) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDR = Lay::LDR, LDA = Lay::LDA;
    for (int i = lane; i < nrows; i += 32) {
#pragma unroll
        for (int j = 0; j < NP; ++j) S[i * LDR + j] *= dsc[j];
    }
    __syncwarp();
    for (int j = 0; j < NP; ++j) {
        double ss = 0.0;
        for (int i = lane; i < nrows; i += 32) { const double v = S[i * LDR + j]; ss = fma(v, v, ss); }
        ss = warp_sum(ss);
        if (ss == 0.0) continue;                             // uniform across the warp
        const double rjj = A[j * LDA + j];
        const double nrm = sqrt(fma(rjj, rjj, ss));
        const double alpha = rjj > 0.0 ? -nrm : nrm;
        const double v0 = rjj - alpha;
        const double beta = 1.0 / (nrm * fabs(v0));
        double t[NP];
#pragma unroll
        for (int q = 0; q < NP; ++q) t[q] = 0.0;
        for (int i = lane; i < nrows; i += 32) {
            const double sj = S[i * LDR + j];
#pragma unroll
            for (int q = 0; q < NP; ++q) if (q > j) t[q] = fma(sj, S[i * LDR + q], t[q]);
        }
#pragma unroll
        for (int q = 0; q < NP; ++q) if (q > j) t[q] = (fma(v0, A[j * LDA + q], warp_sum(t[q]))) * beta;
        __syncwarp();
        for (int i = lane; i < nrows; i += 32) {
            const double sj = S[i * LDR + j];
#pragma unroll
            for (int q = 0; q < NP; ++q) if (q > j) S[i * LDR + q] = fma(-t[q], sj, S[i * LDR + q]);
        }
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < NP; ++q) if (q > j) A[j * LDA + q] = fma(-t[q], v0, A[j * LDA + q]);
            A[j * LDA + j] = alpha;
        }
        __syncwarp();
    }
}

// scipy's robust losses (least_squares loss= / f_scale=, P.loss codes as lsqfit_b200.dense.LOSSES), one residual r at a
// time: z = (r / C)^2 (divide, then square, as construct_loss_function does), rho, rho', rho'' of the loss, and the row
// scale of scale_for_robust_loss_function, s = sqrt(max(rho' + 2 rho'' r^2 / C^2, EPS)): the row [J | r] becomes
// [s J | r rho' / s].  Returns C^2 rho(z), the row's share of twice the robust cost.  `loss` is warp-uniform.
__device__ __forceinline__ double robust_row(int loss, double C, double r, double& s, double& rs) {
    const double u = r / C;
    const double z = u * u;
    double rho0, rho1, rho2;
    switch (loss) {
    case 1:                                                  // huber
        if (z <= 1.0) {
            rho0 = z; rho1 = 1.0; rho2 = 0.0;
        } else {
            const double sz = sqrt(z);
            rho0 = 2.0 * sz - 1.0; rho1 = 1.0 / sz; rho2 = -0.5 * rho1 / z;
        }
        break;
    case 2: {                                                // soft_l1
        const double t = 1.0 + z, st = sqrt(t);
        rho0 = 2.0 * (st - 1.0); rho1 = 1.0 / st; rho2 = -0.5 * rho1 / t;
        break;
    }
    case 3: {                                                // cauchy
        rho0 = log1p(z); rho1 = 1.0 / (1.0 + z); rho2 = -rho1 * rho1;
        break;
    }
    case 4: {                                                // arctan
        rho0 = atan(z); rho1 = 1.0 / fma(z, z, 1.0); rho2 = -2.0 * z * rho1 * rho1;
        break;
    }
    default:
        rho0 = z; rho1 = 1.0; rho2 = 0.0;
    }
    const double C2 = C * C;
    double js = rho1 + 2.0 * (rho2 / C2) * (r * r);
    // scipy clips J_scale < EPS to EPS; for cauchy and arctan that is every row with z > 1 (rho' + 2 z rho'' < 0)
    if (js < 2.220446049250313e-16) js = 2.220446049250313e-16;
    s = sqrt(js);
    rs = r * (rho1 / s);
    return C2 * rho0;
}

// rows of the buffer are finished [J | r]: emit / fold them into the normal equations or the QR factor.
// ROBUST (fit_kernel<F, 6>): after the (true) rows are emitted, each is rescaled by the loss (robust_row) and its
// C^2 rho is added to `rcost`; without it, rcost is untouched.
template <class F, int MODE, bool ROBUST = false>
__device__ __forceinline__ void consume_rows(WarpCtx<F>& c, int nrows, int slot0, double* fout, double* Jout,
                                             NormalAcc<F>& na, double& rcost) {
    if (fout || Jout) emit_rows<F>(c.R, nrows, slot0, c.lane, fout, Jout);
    if constexpr (ROBUST) {
        constexpr int NP = FitLayout<F>::NP;
        if (c.lane < nrows) {
            double* row = c.R + c.lane * FitLayout<F>::LDR;
            double s, rs;
            rcost += robust_row(c.P.loss, c.P.f_scale, row[NP], s, rs);
#pragma unroll
            for (int j = 0; j < NP; ++j) row[j] *= s;
            row[NP] = rs;
        }
        __syncwarp();
    }
    if (MODE == 0) {
        mma_accumulate<F>(c, c.R, (nrows + 3) & ~3, na);
    } else {
        __syncwarp();
        qr_update<F>(c.A, c.dsc, c.R, nrows, c.lane);
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------
// residual + Jacobian + normal equations at pv: fills c.A (J^T J), c.g (J^T r),
// returns cost.  Optionally writes the residual vector and J to global memory.
// MODE 0: normal equations (A = J^T J, g = J^T r).  MODE 1: QR factor of J.diag(dsc) in c.A.
// ---------------------------------------------------------------------------
// the row tables of one window (P.win[w]), in the names eval_rows reads
struct WinRows {
    int nd_fn, nd_pr, nblk, pr_base;
    const int* dfn_idx;
    const double* dfn_w;
    const int* dpr_idx;
    const double* dpr_w;
    const BlockDesc* blk;
};

// the entry of y(+)prior that holds prior entry 0 (parameter j sits at prior_base + j): the plan's one prior follows
// its ny data rows; a window's is its own slot (every data row of a fit set precedes every slot)
__device__ __forceinline__ int prior_base(const FitParams& P) { return P.ny; }
__device__ __forceinline__ int prior_base(const WinRows& T) { return T.pr_base; }

// T: the row tables (nd_fn, dfn_idx, dfn_w, nd_pr, dpr_idx, dpr_w, nblk, blk) -- the FitParams themselves, or those of
// one window (WinRows)
// TRANS (parameter distributions, fit_kernel<F, 5>): the data rows see the model at qv = T(pv), and their Jacobian
// columns are scaled by tp = T'(pv); the prior rows stay in pv
// ROBUST (robust loss, fit_kernel<F, 6>): every row is rescaled by the loss before it enters A / g or the QR factor,
// and the returned cost is 1/2 sum C^2 rho; emitted rows (fout, Jout) are the true ones
template <class F, int MODE, bool WSMEM, class RS, bool TRANS = false, bool ROBUST = false>
__device__ __forceinline__ double eval_rows(WarpCtx<F>& c, const RS& T, const double* pv, double* fout, double* Jout,
                                            const double* qv = nullptr, const double* tp = nullptr) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, NT = Lay::NT, LDR = Lay::LDR, LDA = Lay::LDA, NCOL = Lay::NCOL;
    const FitParams& P = c.P;
    const int lane = c.lane;
    const double* mv = pv;                  // the parameters the model sees
    if constexpr (TRANS) mv = qv;
    for (int e = lane; e < NP * LDA; e += 32) c.A[e] = 0.0;
    if (MODE == 0 && lane < NP) c.g[lane] = 0.0;
    __syncwarp();
    double acc = 0.0;
    NormalAcc<F> na;
    na.clear();
    // 1x1 prior rows: J row = w e_j, analytic contribution
    for (int i = lane; i < T.nd_pr; i += 32) {
        const int idx = T.dpr_idx[i];
        const int j = idx - prior_base(T);
        const double w = T.dpr_w[i];
        const double r = w * (pv[j] - c.mean[idx]);
        double ws = w, rs = r;                               // the row as it enters A / g (ROBUST: rescaled)
        if constexpr (ROBUST) {
            double s;
            acc += robust_row(P.loss, P.f_scale, r, s, rs);
            ws = s * w;
        }
        if (MODE == 0) {
            c.A[j * LDA + j] += ws * ws;
            c.g[j] += ws * rs;
        } else {
            c.A[j * LDA + j] = ws * c.dsc[j];                // a diagonal matrix is triangular
        }
        if constexpr (!ROBUST) acc = fma(r, r, acc);
        if (fout) fout[T.nd_fn + i] = r;
        if (Jout) {
            for (int q = 0; q < NP; ++q) Jout[(size_t)(T.nd_fn + i) * NP + q] = (q == j) ? w : 0.0;
        }
    }
    __syncwarp();
    // 1x1 data rows, staged through the row buffer 32 at a time (one row per lane)
    for (int c0 = 0; c0 < T.nd_fn; c0 += 32) {
        const int nrows = min(32, T.nd_fn - c0);
        double* row_ = c.R + lane * LDR;
        if (lane < nrows) {
            const int row = T.dfn_idx[c0 + lane];
            const double w = T.dfn_w[c0 + lane];
            const double f = F::value_grad(P.x + (size_t)row * P.nx, row, mv, w, row_);
            if constexpr (TRANS) {
#pragma unroll
                for (int j = 0; j < NP; ++j) row_[j] *= tp[j];
            }
            row_[NP] = w * (f - c.mean[row]);
#pragma unroll
            for (int j = NP + 1; j < NCOL; ++j) row_[j] = 0.0;
        } else {
#pragma unroll
            for (int j = 0; j < NCOL; ++j) row_[j] = 0.0;
        }
        __syncwarp();
        consume_rows<F, MODE, ROBUST>(c, nrows, c0, fout, Jout, na, acc);
    }
    // correlated blocks: J_blk = W.[G | delta] on the FP64 tensor path.  The C fragments of a
    // 64-row output group stay in registers while the input rows stream through the row buffer
    // 32 at a time; the finished rows then pass through the same buffer into J^T J.
    for (int b = 0; b < T.nblk; ++b) {
        const BlockDesc bd = T.blk[b];
        const double* W = c.wt + bd.wt_off;
        if constexpr (WSMEM) __builtin_assume(__isShared(W));
        for (int g0 = 0; g0 < bd.n_out; g0 += 64) {
            const int mtiles = min(8, (bd.n_out - g0 + 7) >> 3);
            double pc[8][NT][2];
#pragma unroll
            for (int m = 0; m < 8; ++m)
#pragma unroll
                for (int t = 0; t < NT; ++t) { pc[m][t][0] = 0.0; pc[m][t][1] = 0.0; }
            // when the residual column does not ride in a tile (np % 8 == 0) it gets a tile of its
            // own in which only column 0 is populated: r = W.delta as 8 more DMMA per k-step
            double pr[Lay::DELTA_IN_TILE ? 1 : 8][2];
#pragma unroll
            for (int m = 0; m < (Lay::DELTA_IN_TILE ? 1 : 8); ++m) { pr[m][0] = 0.0; pr[m][1] = 0.0; }
            for (int k0 = 0; k0 < bd.n_in; k0 += 32) {
                const int nk = min(32, bd.n_in - k0);
                const int nk4 = (nk + 3) & ~3;
                double* row_ = c.R + lane * LDR;
                if (lane < nk) {
                    const int idx = P.blk_idx[bd.idx_off + k0 + lane];
                    double dlt;
                    if (idx < P.ny) {
                        const double f = F::value_grad(P.x + (size_t)idx * P.nx, idx, mv, 1.0, row_);
                        if constexpr (TRANS) {
#pragma unroll
                            for (int j = 0; j < NP; ++j) row_[j] *= tp[j];
                        }
                        dlt = f - c.mean[idx];
                    } else {
                        const int j0 = idx - prior_base(T);
#pragma unroll
                        for (int j = 0; j < NP; ++j) row_[j] = (j == j0) ? 1.0 : 0.0;
                        dlt = pv[j0] - c.mean[idx];
                    }
                    row_[NP] = dlt;
#pragma unroll
                    for (int j = NP + 1; j < NCOL; ++j) row_[j] = 0.0;
                    if (!Lay::DELTA_IN_TILE) c.dvec[lane] = dlt;
                } else if (lane < nk4) {
#pragma unroll
                    for (int j = 0; j < NCOL; ++j) row_[j] = 0.0;
                    if (!Lay::DELTA_IN_TILE) c.dvec[lane] = 0.0;
                }
                __syncwarp();
                // A fragment: W[g0 + 8m + lane/4][k0 + 4s + lane%4];  B fragment: R[4s + lane%4][8t + lane/4]
                const double* wa = W + (g0 + (lane >> 2)) * bd.ldw + k0 + (lane & 3);
                const double* rb_ = c.R + (lane & 3) * LDR + (lane >> 2);
                const int ldw8 = 8 * bd.ldw;
#pragma unroll 2
                for (int s4 = 0; s4 < nk4; s4 += 4) {
                    double bf[NT];
#pragma unroll
                    for (int t = 0; t < NT; ++t) bf[t] = rb_[s4 * LDR + 8 * t];
                    double bd_ = 0.0;
                    if constexpr (!Lay::DELTA_IN_TILE) bd_ = (lane >> 2) == 0 ? c.dvec[s4 + (lane & 3)] : 0.0;
#pragma unroll
                    for (int m = 0; m < 8; ++m) {
                        if (m < mtiles) {
                            const double af = wa[m * ldw8 + s4];
#pragma unroll
                            for (int t = 0; t < NT; ++t) dmma(pc[m][t][0], pc[m][t][1], af, bf[t]);
                            if constexpr (!Lay::DELTA_IN_TILE) dmma(pr[m][0], pr[m][1], af, bd_);
                        }
                    }
                }
                __syncwarp();                      // everyone has finished reading this chunk
            }
            // finished rows: two passes of (up to) 32 rows = 4 m-tiles each.  The loop is rolled
            // (code size); the second pass first moves tiles 4..7 down into registers 0..3.
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                const int nrows = min(32, bd.n_out - g0 - 32 * half);
                if (nrows <= 0) break;
                const int mt_here = min(4, mtiles - 4 * half);
#pragma unroll
                for (int m4 = 0; m4 < 4; ++m4) {
                    if (m4 < mt_here) {
                        double* dst = c.R + (8 * m4 + (lane >> 2)) * LDR + 2 * (lane & 3);
#pragma unroll
                        for (int t = 0; t < NT; ++t) {
                            dst[8 * t] = pc[m4][t][0];
                            dst[8 * t + 1] = pc[m4][t][1];
                        }
                    }
                }
                if constexpr (!Lay::DELTA_IN_TILE) {
                    // column 0 of the residual tile lives in c0 of the lanes with lane % 4 == 0
#pragma unroll
                    for (int m4 = 0; m4 < 4; ++m4)
                        if (m4 < mt_here && (lane & 3) == 0) c.R[(8 * m4 + (lane >> 2)) * LDR + NP] = pr[m4][0];
                }
                __syncwarp();
                consume_rows<F, MODE, ROBUST>(c, nrows, bd.chiv_off + g0 + 32 * half, fout, Jout, na, acc);
#pragma unroll
                for (int m4 = 0; m4 < 4; ++m4) {
#pragma unroll
                    for (int t = 0; t < NT; ++t) { pc[m4][t][0] = pc[m4 + 4][t][0]; pc[m4][t][1] = pc[m4 + 4][t][1]; }
                    if constexpr (!Lay::DELTA_IN_TILE) pr[m4][0] = pr[m4 + 4][0];
                }
            }
        }
    }
    if (MODE == 0) {
        const double rr = flush_normal<F>(c, na);
        if constexpr (!ROBUST) acc += rr;                   // ROBUST: r^T r of the rescaled rows is not the cost
    }
    return 0.5 * warp_sum(acc);
}

template <class F, int MODE, bool WSMEM>
__device__ __noinline__ double eval_full_impl(const WarpCtx<F>& c_in, const double* pv, double* fout, double* Jout) {
    WarpCtx<F> c = c_in;                // local copy: the address-space assumptions below attach to SSA values
    // per-warp state lives in shared memory: say so, or the out-of-line code uses generic LD/ST
    __builtin_assume(__isShared(c.R));
    __builtin_assume(__isShared(c.dvec));
    __builtin_assume(__isShared(c.A));
    __builtin_assume(__isShared(c.g));
    __builtin_assume(__isShared(c.dsc));
    __builtin_assume(__isShared(pv));
    return eval_rows<F, MODE, WSMEM>(c, c.P, pv, fout, Jout);
}

// the block weights are staged in shared memory whenever they fit (P.wt_in_smem, uniform)
template <class F, int MODE = 0>
__device__ __forceinline__ double eval_full(WarpCtx<F>& c, const double* pv, double* fout, double* Jout) {
    return c.P.wt_in_smem ? eval_full_impl<F, MODE, true>(c, pv, fout, Jout)
                          : eval_full_impl<F, MODE, false>(c, pv, fout, Jout);
}

// window evaluation: the weights stay in global memory (a scan's windows together are too large to stage, and the
// fits of one window are contiguous in the batch, so the warps in flight share a few windows' weights in L2)
template <class F, int MODE>
__device__ __noinline__ double eval_win_impl(const WarpCtx<F>& c_in, int w, const double* pv, double* fout, double* Jout) {
    WarpCtx<F> c = c_in;
    __builtin_assume(__isShared(c.R));
    __builtin_assume(__isShared(c.dvec));
    __builtin_assume(__isShared(c.A));
    __builtin_assume(__isShared(c.g));
    __builtin_assume(__isShared(c.dsc));
    __builtin_assume(__isShared(pv));
    const FitParams& P = c.P;
    const WinDesc wd = P.win[w];
    WinRows T;
    T.nd_fn = wd.nd_fn; T.nd_pr = wd.nd_pr; T.nblk = wd.nblk; T.pr_base = wd.pr_base;
    T.dfn_idx = P.dfn_idx + wd.dfn_off; T.dfn_w = P.dfn_w + wd.dfn_off;
    T.dpr_idx = P.dpr_idx + wd.dpr_off; T.dpr_w = P.dpr_w + wd.dpr_off;
    T.blk = P.blk + wd.blk_off;
    const double cost = eval_rows<F, MODE, false>(c, T, pv, fout, Jout);
    // f / J rows have the stride of the largest window: zero beyond this window's own residuals
    for (int i = wd.nchiv + c.lane; i < P.nchiv; i += 32) {
        if (fout) fout[i] = 0.0;
        if (Jout)
            for (int q = 0; q < F::NP; ++q) Jout[(size_t)i * F::NP + q] = 0.0;
    }
    return cost;
}

// q = T(p) and dq/dp of one parameter with distribution code `code` (FitParams::pd_code; the uniform form is
// written with erfc, which keeps q - lo accurate in the lower tail; host mirror: lsqfit_b200/pdist.py)
__device__ __forceinline__ void param_transform(int code, double lo, double hi, double p, double& q, double& dq) {
    if (code == 1) {
        q = exp(p); dq = q;
    } else if (code == 2) {
        q = p * p; dq = 2.0 * p;
    } else if (code == 3) {
        const double w = hi - lo;
        q = fma(w, 0.5 * erfc(-0.7071067811865476 * p), lo);
        dq = w * 0.3989422804014327 * exp(-0.5 * p * p);                 // (hi - lo) exp(-p^2/2) / sqrt(2 pi)
    } else {
        q = p; dq = 1.0;
    }
}

// evaluation with parameter distributions: lane j < NP puts q_j = T(p_j) and T'(p_j) into the warp's qt buffer
// (q [NP] | T' [NP], behind the per-warp layout of FitLayout), then the rows as in eval_full with TRANS set
template <class F, int MODE, bool WSMEM>
__device__ __noinline__ double eval_trans_impl(const WarpCtx<F>& c_in, double* qt, const double* pv, double* fout,
                                               double* Jout) {
    WarpCtx<F> c = c_in;
    __builtin_assume(__isShared(c.R));
    __builtin_assume(__isShared(c.dvec));
    __builtin_assume(__isShared(c.A));
    __builtin_assume(__isShared(c.g));
    __builtin_assume(__isShared(c.dsc));
    __builtin_assume(__isShared(pv));
    __builtin_assume(__isShared(qt));
    constexpr int NP = F::NP;
    const FitParams& P = c.P;
    if (c.lane < NP) {
        double q, dq;
        param_transform(P.pd_code[c.lane], P.pd_lo[c.lane], P.pd_hi[c.lane], pv[c.lane], q, dq);
        qt[c.lane] = q;
        qt[NP + c.lane] = dq;
    }
    __syncwarp();
    return eval_rows<F, MODE, WSMEM, FitParams, true>(c, P, pv, fout, Jout, qt, qt + NP);
}

// evaluation with a robust loss (fit_kernel<F, 6>): the rows of eval_full, rescaled by the loss; returns the robust cost
template <class F, int MODE, bool WSMEM>
__device__ __noinline__ double eval_robust_impl(const WarpCtx<F>& c_in, const double* pv, double* fout, double* Jout) {
    WarpCtx<F> c = c_in;
    __builtin_assume(__isShared(c.R));
    __builtin_assume(__isShared(c.dvec));
    __builtin_assume(__isShared(c.A));
    __builtin_assume(__isShared(c.g));
    __builtin_assume(__isShared(c.dsc));
    __builtin_assume(__isShared(pv));
    return eval_rows<F, MODE, WSMEM, FitParams, false, true>(c, c.P, pv, fout, Jout);
}

// ---------------------------------------------------------------------------
// small dense kernels on the warp: lane i owns row i, everything in registers
// ---------------------------------------------------------------------------
#ifndef B200LM_LDL_VARIANT
#define B200LM_LDL_VARIANT 1
#endif

// 1/x for a positive, normal x: MUFU.RCP64H seed (about 20 bits) + two Newton steps.  No slow path
// (the pivots handed to it are tested separately), four dependent FMAs after the seed.
__device__ __forceinline__ double fast_rcp(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    return fma(y, e, y);
}

// One factorisation + the solves every caller needs, written for LATENCY: a fit spends most of its
// life in this dependency chain (measured on B200: DFMA 8.5, 64-bit shuffle 26, shared-memory round
// trip 42, fp64 divide 71 cycles).
//     L D L^T = d_i A_ij d_j + alpha delta_ij      (unit lower L, D = pivots; no square roots)
//     p = -(L D L^T)^-1 gh ,  res[0] = |p| ,  res[1] = p^T (L D L^T)^-1 p ,  res[2] = min_j pivot_j / diag_j
// Lane i owns row i of the trailing matrix in registers r[0..NP); the loop over columns is fully
// unrolled so that every register index is static, only live columns are updated, and all
// lane == column tests are predicates -- no divergent branch anywhere.  Per column j the chain is
//     pivot = shfl(r[j], j) + alpha  ->  1/pivot  ->  l_ij = r[j]/pivot  ->  r[j+1] -= l_ij * a_(j+1)j
// The UNSCALED column a_kj goes to shared memory (double-buffered, one __syncwarp per column) while
// the reciprocal is still being computed, so the broadcast is off the critical path.  The forward
// substitution y = L^-1 (-gh) rides along.  Finished columns are stored as rows of L^T
// (LT[j][i] = L[i][j], LT[j][j] = pivot_j) with the reciprocal pivots in idg for the covariance.
// HALF: two systems per warp (np <= 16): lanes 0..15 use alpha_lo, lanes 16..31 alpha_hi, each half
// with its own L^T (LT0 / LT1) -- the same instructions factor both (16-wide shuffles).
// Per-lane outputs refer to the lane's own system; `ok` false = not numerically positive definite.
// EXTRA: the factored matrix is  d_i A_ij d_j + (alpha + ex_i) delta_ij  with a per-lane extra diagonal ex (the
// Coleman-Li term of the bounded driver); it enters where alpha does, at the pivot.
template <int NP, int LDA, bool HALF, bool EXTRA = false>
__device__ __forceinline__ void ldl_solve(const double* A, const double* dsc, double* LT0, double* LT1, double* idg,
                                          double* colb, int lane, double alpha_lo, double alpha_hi, double gh_in,
                                          bool want_ratio, double& p_out, double& pn_out, double& w2_out,
                                          double& minr_out, bool& ok_out, double ex = 0.0) {
    static_assert(!HALF || NP <= 16, "two systems per warp need np <= 16");
    static_assert(NP <= 32, "one lane per row");
    constexpr int W = HALF ? 16 : 32;
    const int hi = HALF ? (lane >> 4) : 0;
    const int i = lane & (W - 1);
    const bool act = i < NP;
    const int ii = act ? i : NP - 1;    // idle lanes shadow the last row (same values, same addresses)
    const double alpha = hi ? alpha_hi : alpha_lo;
    double* LT = hi ? LT1 : LT0;
    double* cb0 = colb + hi * 16;       // column broadcast buffers: [2][32] doubles
    const double gh = HALF ? __shfl_sync(B200LM_FULL, gh_in, i) : gh_in;      // both halves solve for the same gradient
    double r[NP];
    const double di = dsc[ii];
#pragma unroll
    for (int k = 0; k < NP; ++k) r[k] = A[ii * LDA + k] * di * dsc[k];
    double mdiag = fma(A[ii * LDA + ii] * di, di, alpha);                     // diagonal entry of this lane's row
    if constexpr (EXTRA) mdiag += ex;
    double myrcp = 1.0, mypiv = 1.0;
    bool ok = true;
    double b = act ? -gh : 0.0;
    double pivsrc = r[0];                   // lane j holds the raw pivot of column j here when its turn comes
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        const double cj = r[j];                                              // a_ij of the trailing matrix
        double* cb = cb0 + (j & 1) * 32;
        cb[ii] = cj;
        double piv;
        if (B200LM_LDL_VARIANT & 4) {
            __syncwarp();
            piv = cb[j] + alpha;
            if constexpr (EXTRA) piv += __shfl_sync(B200LM_FULL, ex, j, W);
        } else if constexpr (EXTRA) {
            piv = __shfl_sync(B200LM_FULL, ((B200LM_LDL_VARIANT & 1) ? pivsrc : cj) + ex, j, W) + alpha;
            __syncwarp();
        } else {
            piv = __shfl_sync(B200LM_FULL, (B200LM_LDL_VARIANT & 1) ? pivsrc : cj, j, W) + alpha;
            __syncwarp();
        }
        const double rcp = fast_rcp(piv);
        const double l = cj * rcp;                                           // L[i][j]  (i > j)
        // the next pivot from registers only (lane j+1: its own column entry is a_(j+1)j): keeps the
        // shared-memory broadcast of the column off the pivot -> reciprocal -> pivot chain
        if (j + 1 < NP) pivsrc = fma(-l, cj, r[j + 1 < NP ? j + 1 : j]);
        const bool me = (ii == j);            // (idle lanes shadow row NP-1: they must store what its owner stores)
        myrcp = me ? rcp : myrcp;
        mypiv = me ? piv : mypiv;
        ok = ok && (!me || ((piv > 8.0 * NP * 2.220446049250313e-16 * mdiag) && (piv < 1e300)));
        LT[j * LDA + ii] = me ? piv : l;
        if (!(B200LM_LDL_VARIANT & 2)) {
            const double yj = __shfl_sync(B200LM_FULL, b, j, W);             // y_j = b_j (unit diagonal)
            b = (i > j) ? fma(-l, yj, b) : b;
        }
#pragma unroll
        for (int k = j + 1; k < NP; ++k) r[k] = fma(-l, cb[k], r[k]);
    }
    if (B200LM_LDL_VARIANT & 2) {
        __syncwarp();
#pragma unroll
        for (int j = 0; j < NP; ++j) {
            const double yj = __shfl_sync(B200LM_FULL, b, j, W);
            const double lij = LT[j * LDA + ii];
            b = (i > j) ? fma(-lij, yj, b) : b;
        }
    }
    if (!HALF && act) idg[i] = myrcp;
    if (HALF) {
        const unsigned okm = __ballot_sync(B200LM_FULL, ok);
        ok = ((okm >> (16 * hi)) & 0xffffu) == 0xffffu;
    } else {
        ok = __all_sync(B200LM_FULL, ok);
    }
    __syncwarp();
    // z = D^-1 y ;  p = L^-T z  (a system whose factorisation failed computes junk that is never used)
    b *= myrcp;
#pragma unroll
    for (int j = NP - 1; j >= 0; --j) {
        const double xj = __shfl_sync(B200LM_FULL, b, j, W);
        const double lji = LT[ii * LDA + j];                                 // L[j][i]
        b = (i < j) ? fma(-lji, xj, b) : b;
    }
    const double p = act ? b : 0.0;
    // w = L^-1 p ;  p^T (L D L^T)^-1 p = sum_i w_i^2 / d_i
    double w = p;
#pragma unroll
    for (int j = 0; j < NP; ++j) {
        const double wj = __shfl_sync(B200LM_FULL, w, j, W);
        const double lij = LT[j * LDA + ii];                                 // L[i][j]
        w = (i > j) ? fma(-lij, wj, w) : w;
    }
    double s = p * p, w2 = act ? w * w * myrcp : 0.0;
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) {
        s += __shfl_xor_sync(B200LM_FULL, s, o);
        w2 += __shfl_xor_sync(B200LM_FULL, w2, o);
    }
    double minr = 0.0;
    if (want_ratio) {
        double q = act ? mypiv / mdiag : 1.0;
#pragma unroll
        for (int o = W / 2; o > 0; o >>= 1) q = fmin(q, __shfl_xor_sync(B200LM_FULL, q, o));
        minr = q;
    }
    __syncwarp();
    p_out = p; pn_out = sqrt(s); w2_out = w2; minr_out = minr; ok_out = ok;
}

// out-of-line entry points (ONE copy of the unrolled code per kernel)
template <int NP, int LDA>
__device__ __noinline__ bool factor_solve(const double* A, const double* dsc, double* LT, double* idg, double* colb,
                                          int lane, double alpha, double gh, bool want_ratio,
                                          double* p_out, double* res) {
    // the matrices live in shared memory: tell the compiler, or it emits generic LD/ST
    __builtin_assume(__isShared(A));
    __builtin_assume(__isShared(dsc));
    __builtin_assume(__isShared(LT));
    __builtin_assume(__isShared(idg));
    __builtin_assume(__isShared(colb));
    double p, pn, w2, minr;
    bool ok;
    ldl_solve<NP, LDA, false>(A, dsc, LT, LT, idg, colb, lane, alpha, alpha, gh, want_ratio, p, pn, w2, minr, ok);
    *p_out = ok ? p : 0.0;
    res[0] = ok ? pn : 0.0; res[1] = ok ? w2 : 0.0; res[2] = ok ? minr : 0.0;
    return ok;
}

// the same with the per-lane extra diagonal ex (bounded driver)
template <int NP, int LDA>
__device__ __noinline__ bool factor_solve_ex(const double* A, const double* dsc, double* LT, double* idg, double* colb,
                                             int lane, double alpha, double gh, double ex, double* p_out, double* res) {
    __builtin_assume(__isShared(A));
    __builtin_assume(__isShared(dsc));
    __builtin_assume(__isShared(LT));
    __builtin_assume(__isShared(idg));
    __builtin_assume(__isShared(colb));
    double p, pn, w2, minr;
    bool ok;
    ldl_solve<NP, LDA, false, true>(A, dsc, LT, LT, idg, colb, lane, alpha, alpha, gh, false, p, pn, w2, minr, ok, ex);
    *p_out = ok ? p : 0.0;
    res[0] = ok ? pn : 0.0; res[1] = ok ? w2 : 0.0; res[2] = 0.0;
    return ok;
}

// Gauss-Newton step of the current outer iteration (alpha = 0), cached across rejected trials
struct GNCache {
    bool valid, full_rank;
    double p, pn, w2;
};

// Trust-region sub-problem in scaled variables: min 1/2 s^T Ah s + gh^T s, |s| <= Delta.
// gh: lane-distributed scaled gradient.  Returns lane-distributed step; updates alpha.
// (cf. scipy/optimize/_lsq/common.py: solve_lsq_trust_region, with the secular equation
// evaluated through Cholesky factors instead of singular values.)
// EXTRA: Ah = d A d + diag(ex) (bounded driver: scipy's Coleman-Li augmented normal matrix).
template <class F, bool EXTRA>
__device__ __forceinline__ double solve_tr_impl(WarpCtx<F>& c, double gh, double Delta, double& alpha, int& nfac,
                                                GNCache& gn, long long& fclk, double ex) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    const int lane = c.lane;
    const bool act = lane < NP;
    auto factor = [&](double a, double* p_out, double* r) -> bool {
        if constexpr (EXTRA) return factor_solve_ex<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, a, gh, ex, p_out, r);
        else return factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, a, gh, false, p_out, r);
    };
    double res[3];
    double p = 0.0, pn = 0.0;
    bool have_p = false;
    // |p(alpha)| decreases with alpha.  If the warm-started alpha > 0 already gives a step longer
    // than Delta, the Gauss-Newton step (alpha = 0) is longer still: its factorisation is skipped.
    bool tried_warm = false, warm_ok = false;
    double warm_phi = 0.0, warm_w2 = 0.0, warm_pn = 0.0, warm_p = 0.0;
    if (!gn.valid && alpha > 0.0) {
        ++nfac;
        tried_warm = true;
        const long long tq = B200LM_CLOCK();
        warm_ok = factor(alpha, &warm_p, res);
        fclk += B200LM_CLOCK() - tq;
        if (warm_ok) { warm_pn = res[0]; warm_w2 = res[1]; warm_phi = warm_pn - Delta; }
    }
    const bool need_gn = !(tried_warm && warm_ok && warm_phi > 0.0);
    if (!gn.valid && need_gn) {
        ++nfac;
        const long long tq = B200LM_CLOCK();
        gn.full_rank = factor(0.0, &p, res);
        fclk += B200LM_CLOCK() - tq;
        gn.p = p; gn.pn = res[0]; gn.w2 = res[1];
        gn.valid = true;
    }
    const bool full_rank = gn.valid && gn.full_rank;
    if (full_rank && gn.pn <= Delta) { alpha = 0.0; return gn.p; }
    double alpha_upper = sqrt(warp_sum(act ? gh * gh : 0.0)) / Delta;
    double alpha_lower = 0.0;
    if (full_rank) {
        const double phi = gn.pn - Delta;
        const double phi_prime = -gn.w2 / gn.pn;
        alpha_lower = -phi / phi_prime;
        p = gn.p; have_p = true;
    }
    if (!full_rank && alpha == 0.0)
        alpha = fmax(0.001 * alpha_upper, sqrt(alpha_lower * alpha_upper));
    // Newton iteration on the secular equation phi(alpha) = |p(alpha)| - Delta (More' 1978; the
    // same safeguarded update as scipy's solve_lsq_trust_region).  The step of the last iterate is
    // kept (it is rescaled to the boundary below) instead of being recomputed at the updated
    // alpha, and the iteration stops at |phi| < 0.1 Delta (MINPACK's lmpar tolerance).
    for (int it = 0; it < 10; ++it) {
        bool ok;
        double pt;
        if (it == 0 && tried_warm) {
            ok = warm_ok; pt = warm_p; res[0] = warm_pn; res[1] = warm_w2;
        } else {
            if (alpha < alpha_lower || alpha > alpha_upper)
                alpha = fmax(0.001 * alpha_upper, sqrt(alpha_lower * alpha_upper));
            ++nfac;
            const long long tq = B200LM_CLOCK();
            ok = factor(alpha, &pt, res);
            fclk += B200LM_CLOCK() - tq;
        }
        if (!ok) {
            alpha_lower = fmax(alpha_lower, alpha);
            alpha = fmax(2.0 * alpha, 0.001 * alpha_upper);
            if (alpha > alpha_upper) alpha_upper = 2.0 * alpha;
            continue;
        }
        p = pt;
        have_p = true;
        pn = res[0];
        const double phi = pn - Delta;
        const double phi_prime = -res[1] / pn;
        if (phi < 0.0) alpha_upper = alpha;
        const double ratio = phi / phi_prime;
        alpha_lower = fmax(alpha_lower, alpha - ratio);
        alpha -= (phi + Delta) * ratio / Delta;
        if (fabs(phi) < 0.1 * Delta) break;
    }
    if (!have_p) p = act ? -gh : 0.0;             // steepest descent fallback
    pn = sqrt(warp_sum(act ? p * p : 0.0));
    if (pn > 0.0) p *= Delta / pn;
    return p;
}

template <class F>
__device__ double solve_tr(WarpCtx<F>& c, double gh, double Delta, double& alpha, int& nfac, GNCache& gn, long long& fclk) {
    return solve_tr_impl<F, false>(c, gh, Delta, alpha, nfac, gn, fclk, 0.0);
}

// ---------------------------------------------------------------------------
// Two shifts per factorisation round (np <= 16): lanes 0..15 factor d A d + alpha_lo I, lanes 16..31
// d A d + alpha_hi I in the same instructions (ldl_solve<HALF>).  Used by solve_tr_dual.
// Per lane outputs refer to the lane's own half: p (entry lane%16 of the step), |p|, p^T M^-1 p, ok.
// ---------------------------------------------------------------------------
template <int NP, int LDA>
__device__ __noinline__ void factor_solve2(const double* A, const double* dsc, double* LT0, double* LT1, double* colb,
                                           int lane, double alpha_lo, double alpha_hi, double gh_lo,
                                           double* p_out, double* pn_out, double* w2_out, bool* ok_out) {
    __builtin_assume(__isShared(A));
    __builtin_assume(__isShared(dsc));
    __builtin_assume(__isShared(LT0));
    __builtin_assume(__isShared(LT1));
    __builtin_assume(__isShared(colb));
    double p, pn, w2, minr;
    bool ok;
    ldl_solve<NP, LDA, true>(A, dsc, LT0, LT1, nullptr, colb, lane, alpha_lo, alpha_hi, gh_lo, false, p, pn, w2, minr, ok);
    *p_out = p; *pn_out = pn; *w2_out = w2; *ok_out = ok;
}

// 1/|p(alpha)| is close to linear in alpha; its fit from the previous trial predicts the Levenberg
// parameter of the next one (the matrix changes little between consecutive trials of a slow fit)
struct LinModel {
    bool valid;
    double a, b;
};

struct TRCand {
    bool ok;
    double a, pn, w2, p;        // shift, |p|, |L^-1 p|^2, lane-distributed step (lanes 0..15)
};

// Trust-region sub-problem with TWO shifts per factorisation round: the warm-started alpha and the
// prediction of the linear model (or the Gauss-Newton shift 0 when it is still needed), then Newton and
// secant iterates side by side.  Same acceptance rule as solve_tr (|phi| < 0.1 Delta, step rescaled to the
// boundary).  On the slow C3 copies this needs 1.3 rounds per trial instead of 1.8 factorisations
// (numpy model tests/lm_model.py: solve_tr_dual; DESIGN.md section 3.1).  Falls back to solve_tr if no shift could be factorised.
template <class F>
__device__ double solve_tr_dual(WarpCtx<F>& c, double gh, double Delta, double& alpha, int& nfac, GNCache& gn,
                                LinModel& lm, long long& fclk) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    constexpr int NPD = NP <= 16 ? NP : 16;          // (never instantiated for np > 16; keeps the template legal)
    const int lane = c.lane;
    const bool act = lane < NP;
    double* LT1 = c.R;                                 // the row buffer is idle between evaluations
    TRCand best, second;
    best.ok = false; second.ok = false;
    auto insert = [&](const TRCand& t) {
        if (!t.ok || !(t.a > 0.0)) return;
        const double d = fabs(t.pn - Delta);
        if (!best.ok || d < fabs(best.pn - Delta)) { second = best; best = t; }
        else if (!second.ok || d < fabs(second.pn - Delta)) second = t;
    };
    auto dual = [&](double a_lo, double a_hi, TRCand& lo, TRCand& hi) {
        double p, pn, w2;
        bool ok;
        const long long tq = B200LM_CLOCK();
        factor_solve2<NPD, LDA>(c.A, c.dsc, c.L, LT1, c.colb, lane, a_lo, a_hi, gh, &p, &pn, &w2, &ok);
        fclk += B200LM_CLOCK() - tq;
        nfac += 2;
        lo.a = a_lo; hi.a = a_hi;
        lo.p = p;
        hi.p = __shfl_down_sync(B200LM_FULL, p, 16);
        lo.pn = __shfl_sync(B200LM_FULL, pn, 0);  hi.pn = __shfl_sync(B200LM_FULL, pn, 16);
        lo.w2 = __shfl_sync(B200LM_FULL, w2, 0);  hi.w2 = __shfl_sync(B200LM_FULL, w2, 16);
        const unsigned m = __ballot_sync(B200LM_FULL, ok);
        lo.ok = (m & 1u) != 0u; hi.ok = (m & 0x10000u) != 0u;
    };
    auto take_gn = [&](const TRCand& t) {
        gn.valid = true; gn.full_rank = t.ok; gn.p = t.p; gn.pn = t.pn; gn.w2 = t.w2;
    };
    double alpha_upper = sqrt(warp_sum(act ? gh * gh : 0.0)) / Delta;
    double alpha_lower = 0.0;
    auto bounds = [&](const TRCand& t) {
        if (!t.ok) return;
        if (t.pn < Delta) alpha_upper = fmin(alpha_upper, t.a); else alpha_lower = fmax(alpha_lower, t.a);
    };
    auto predict = [&]() -> double {
        if (!lm.valid) return -1.0;
        const double pr = (1.0 / Delta - lm.a) / lm.b;
        return (pr > 0.0 && pr < 1e300) ? pr : -1.0;
    };
    // ---- first round ----
    if (!gn.valid && !(alpha > 0.0)) {
        double res[3], p0;
        ++nfac;
        const long long tq = B200LM_CLOCK();
        gn.full_rank = factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, 0.0, gh, false, &p0, res);
        fclk += B200LM_CLOCK() - tq;
        gn.p = p0; gn.pn = res[0]; gn.w2 = res[1];
        gn.valid = true;
    } else {
        double x1 = alpha > 0.0 ? alpha : -1.0;
        double x2 = predict();
        TRCand lo, hi;
        if (x1 < 0.0) {                                  // Gauss-Newton step known and too long, no warm start
            const double nl = (gn.valid && gn.full_rank) ? (gn.pn - Delta) * gn.pn / gn.w2 : 0.0;
            x1 = x2 > 0.0 ? x2 : fmax(nl, 0.001 * alpha_upper);
            x2 = -1.0;
        }
        if (x2 < 0.0 || fabs(x2 - x1) < 1e-3 * x1) x2 = gn.valid ? 1.5 * x1 : 0.0;   // Gauss-Newton rides along if still unknown
        dual(x1, x2, lo, hi);
        if (x2 == 0.0) take_gn(hi); else insert(hi);
        insert(lo);
    }
    if (gn.valid && gn.full_rank && gn.pn <= Delta) { alpha = 0.0; return gn.p; }
    for (int it = 0; it < 5; ++it) {
        if (gn.valid && gn.full_rank) alpha_lower = fmax(alpha_lower, (gn.pn - Delta) * gn.pn / gn.w2);
        bounds(best); bounds(second);
        // a step shorter than Delta at alpha > 0 does not exclude an interior Gauss-Newton step: only accept it
        // once the Gauss-Newton step is known (and known to be outside)
        if (best.ok && fabs(best.pn - Delta) < 0.1 * Delta && (gn.valid || best.pn >= Delta)) break;
        double an, as;
        if (best.ok) {
            const double phi = best.pn - Delta;
            const double ratio = -phi * best.pn / best.w2;            // phi / phi'
            an = best.a - (phi + Delta) * ratio / Delta;
        } else {
            an = alpha > 0.0 ? 2.0 * alpha : 0.0;
        }
        if (!(an > alpha_lower && an < alpha_upper)) an = fmax(0.001 * alpha_upper, sqrt(alpha_lower * alpha_upper));
        if (!gn.valid && best.ok && best.pn < Delta) {
            as = 0.0;                                                // the step may be interior: Gauss-Newton is needed
        } else {
            as = -1.0;
            if (best.ok && second.ok && second.a != best.a) {
                const double y0 = 1.0 / best.pn, y1 = 1.0 / second.pn;
                if (y1 != y0) as = best.a + (1.0 / Delta - y0) * (second.a - best.a) / (y1 - y0);
            }
            if (!(as > alpha_lower && as < alpha_upper) || fabs(as - an) < 1e-3 * an)
                as = (best.ok && best.pn < Delta) ? 0.5 * (an + alpha_lower) : fmin(1.5 * an, 0.5 * (an + alpha_upper));
            if (!(as > 0.0)) as = 1.5 * an;
        }
        TRCand lo, hi;
        dual(an, as, lo, hi);
        if (as == 0.0) {
            take_gn(hi);
            if (gn.full_rank && gn.pn <= Delta) { alpha = 0.0; return gn.p; }
        } else {
            insert(hi);
        }
        insert(lo);
        if (!lo.ok && (as == 0.0 || !hi.ok)) {                       // not positive definite at these shifts: push up
            alpha_lower = fmax(alpha_lower, fmax(an, as));
            alpha = fmax(2.0 * fmax(an, as), 0.001 * alpha_upper);
            if (alpha > alpha_upper) alpha_upper = 2.0 * alpha;
        }
    }
    if (!best.ok) return solve_tr<F>(c, gh, Delta, alpha, nfac, gn, fclk);
    // model of 1/|p(alpha)| for the next trial
    if (second.ok && second.a != best.a) {
        const double b = (1.0 / second.pn - 1.0 / best.pn) / (second.a - best.a);
        lm.valid = b > 0.0; lm.b = b; lm.a = 1.0 / best.pn - b * best.a;
    } else {
        const double b = best.w2 / (best.pn * best.pn * best.pn);   // d(1/|p|)/d alpha from the factorisation
        lm.valid = b > 0.0; lm.b = b; lm.a = 1.0 / best.pn - b * best.a;
    }
    {   // warm start of the next trial: the Newton update of the accepted shift (as in solve_tr)
        const double phi = best.pn - Delta;
        const double ratio = -phi * best.pn / best.w2;
        const double an = best.a - (phi + Delta) * ratio / Delta;
        alpha = an > 0.0 ? an : best.a;
    }
    double p = act ? best.p : 0.0;
    if (best.pn > 0.0) p *= Delta / best.pn;
    return p;
}

// covariance (J^T J)^-1 = d (L D L^T)^-1 d from the factor of the scaled matrix at alpha=0
// (c.L holds L^T with the pivots on the diagonal: c.L[k*LDA + j] = L[j][k], c.L[j*LDA + j] = D_j; c.idg = 1/D).
// Uses c.A as scratch for L^-1 (column a computed by lane a).  Returns log det(J^T J).
template <class F>
__device__ double covariance_from_chol(WarpCtx<F>& c, double* cov_out) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    const int a = c.lane;
    double ld = 0.0;
    if (a < NP) ld = log(c.L[a * LDA + a]) - 2.0 * log(c.dsc[a]);
    ld = warp_sum(ld);
    __syncwarp();
    if (a < NP) {
        // column a of Linv (unit lower): x_j = delta_ja - sum_{a<=k<j} L[j][k] x_k , j >= a
        for (int j = 0; j < NP; ++j) {
            double s = (j == a) ? 1.0 : 0.0;
            if (j < a) { c.A[j * LDA + a] = 0.0; continue; }
            for (int k = a; k < j; ++k) s = fma(-c.L[k * LDA + j], c.A[k * LDA + a], s);
            c.A[j * LDA + a] = s;
        }
    }
    __syncwarp();
    if (a < NP && cov_out) {
        for (int b = 0; b < NP; ++b) {
            double s = 0.0;
            const int k0 = a > b ? a : b;
            for (int k = k0; k < NP; ++k) s = fma(c.A[k * LDA + a] * c.idg[k], c.A[k * LDA + b], s);
            // element (a, b) goes to its mirror position (b, a): for a fixed b the lanes write one contiguous row
            // (the matrix is symmetric; stride-NP stores would be 16 partial sectors per instruction -- and the output
            // may be pinned HOST memory written over PCIe, b200lm_fit_batch_host)
            cov_out[b * NP + a] = s * c.dsc[a] * c.dsc[b];
        }
    }
    __syncwarp();
    return ld;
}

// covariance from the triangular factor Rt (c.A) of J.diag(dsc): (J^T J)^-1 =
// dsc Rt^-1 Rt^-T dsc.  Uses c.L as scratch for Rt^-1.  Returns log det(J^T J) (nan if singular).
template <class F>
__device__ double covariance_from_qr(WarpCtx<F>& c, double* cov_out) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    const int a = c.lane;
    double ld = 0.0;
    if (a < NP) ld = 2.0 * (log(fabs(c.A[a * LDA + a])) - log(c.dsc[a]));
    ld = warp_sum(ld);
    if (a < NP) {
        // column a of Rt^-1 (upper triangular): back substitution from row a up to row 0
        for (int j = NP - 1; j > a; --j) c.L[j * LDA + a] = 0.0;
        for (int j = a; j >= 0; --j) {
            double s = (j == a) ? 1.0 : 0.0;
            for (int k = j + 1; k <= a; ++k) s = fma(-c.A[j * LDA + k], c.L[k * LDA + a], s);
            c.L[j * LDA + a] = s / c.A[j * LDA + j];
        }
    }
    __syncwarp();
    if (a < NP && cov_out) {
        for (int b = 0; b < NP; ++b) {
            double s = 0.0;
            const int k0 = a > b ? a : b;
            for (int k = k0; k < NP; ++k) s = fma(c.L[a * LDA + k], c.L[b * LDA + k], s);
            cov_out[b * NP + a] = s * c.dsc[a] * c.dsc[b];               // (mirror position: contiguous rows, as above)
        }
    }
    __syncwarp();
    return ld;
}

// ---------------------------------------------------------------------------
// bound constraints: scipy's trf_bounds restated on the warp (numpy model: tests/lm_model_bounded.py).
// scipy/optimize/_lsq/trf.py: trf_bounds, select_step; common.py: CL_scaling_vector, step_size_to_bound,
// intersect_trust_region, minimize_quadratic_1d, make_strictly_feasible.  One lane per parameter; idle lanes carry
// x = s = 0 and an unbounded box.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(B200LM_FULL, v, o));
    return v;
}

// CL_scaling_vector: v = distance to the bound the anti-gradient points at (1 if none), dv = its derivative
__device__ __forceinline__ void cl_scaling(double x, double g, double lb, double ub, double& v, double& dv) {
    v = 1.0; dv = 0.0;
    if (g < 0.0 && isfinite(ub)) { v = ub - x; dv = -1.0; }
    if (g > 0.0 && isfinite(lb)) { v = x - lb; dv = 1.0; }
}

// make_strictly_feasible(x, lb, ub, rstep=1e-10): the start point of a bounded fit
__device__ __forceinline__ double feasible_start(double x, double lb, double ub) {
    const double lt = 1e-10 * fmax(1.0, fabs(lb)), ut = 1e-10 * fmax(1.0, fabs(ub));
    const double ld = x - lb, ud = ub - x;
    double xn = x;
    if (isfinite(lb) && ld <= fmin(ud, lt)) xn = lb + lt;
    if (isfinite(ub) && ud <= fmin(ld, ut)) xn = ub - ut;
    if (xn < lb || xn > ub) xn = 0.5 * (lb + ub);
    return xn;
}

// make_strictly_feasible(x, lb, ub, rstep=0): every trial point
__device__ __forceinline__ double feasible_trial(double x, double lb, double ub) {
    double xn = x;
    if (x <= lb) xn = nextafter(lb, ub);
    if (x >= ub) xn = nextafter(ub, lb);
    if (xn < lb || xn > ub) xn = 0.5 * (lb + ub);
    return xn;
}

// step_size_to_bound: the largest t with x + t s in the box (min over s_i != 0); hit = this lane reaches it
__device__ __forceinline__ double step_to_bound(bool act, double x, double s, double lb, double ub, bool& hit) {
    const bool nz = act && s != 0.0;
    const double st = nz ? fmax((lb - x) / s, (ub - x) / s) : INFINITY;
    const double m = warp_min(st);
    hit = nz && st == m;
    return m;
}

// minimize_quadratic_1d: argmin of a t^2 + b t + c over [lo, hi] -> (t, value)
__device__ __forceinline__ double min_quad_1d(double a, double b, double lo, double hi, double c, double& val) {
    double t = lo, y = lo * (a * lo + b) + c;
    const double yh = hi * (a * hi + b) + c;
    if (yh < y) { t = hi; y = yh; }
    if (a != 0.0) {
        const double e = -0.5 * b / a;
        const double ye = e * (a * e + b) + c;
        if (lo < e && e < hi && ye < y) { t = e; y = ye; }
    }
    val = y;
    return t;
}

// select_step: the trust-region step p_h (scaled space, x = d x_h) if x + d p_h stays in the box; otherwise the best of
// that step cut back to the box (times theta), its reflection off the box minimised along the reflected direction,
// and the cut-back anti-gradient step, on q(s) = 1/2 s^T Ah s + gh^T s with Ah = d A d + diag(ex).  Returns the step
// in x space; s_h becomes the step in scaled space, `predicted` = -q(s_h).  Scratch: c.idg.
template <class F>
__device__ double select_step(WarpCtx<F>& c, double x, double gh, double& s_h, double d, double ex, double Delta,
                              double theta, double lb, double ub, double& predicted) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    const int lane = c.lane;
    const bool act = lane < NP;
    auto Ah = [&](double s) -> double {            // (Ah s)_lane
        if (act) c.idg[lane] = d * s;
        __syncwarp();
        double t = 0.0;
        if (act) {
            const double* Ar = c.A + lane * LDA;
#pragma unroll
            for (int j = 0; j < NP; ++j) t = fma(Ar[j], c.idg[j], t);
        }
        __syncwarp();
        return act ? fma(d, t, ex * s) : 0.0;
    };
    double p_h = act ? s_h : 0.0;
    double p = d * p_h;
    double qa = p_h * Ah(p_h), qb = gh * p_h;
    double xo = (act && !(x + p >= lb && x + p <= ub)) ? 1.0 : 0.0;       // lanes whose step leaves the box
    warp_sum3(qa, qb, xo);
    if (xo == 0.0) { predicted = -(0.5 * qa + qb); return p; }
    bool hit;
    const double p_stride = step_to_bound(act, x, p, lb, ub, hit);
    double r_h = hit ? -p_h : p_h;
    const double r = d * r_h;
    p *= p_stride; p_h *= p_stride;
    qa *= p_stride * p_stride; qb *= p_stride;            // p_h^T Ah p_h and gh^T p_h of the cut-back step
    double r_value = INFINITY, r_step = 0.0, r_hs = 0.0;
    {
        double ra = r_h * r_h, rb = p_h * r_h, pp = p_h * p_h;       // intersect_trust_region(p_h, r_h, Delta)
        warp_sum3(ra, rb, pp);
        const double cc = pp - Delta * Delta;
        const double disc = sqrt(fmax(rb * rb - ra * cc, 0.0));
        const double q = -(rb + copysign(disc, rb));
        const double to_tr = fmax(q / ra, cc / q);
        bool h2;
        const double to_bound = step_to_bound(act, x + p, r, lb, ub, h2);
        const double r_stride = fmin(to_bound, to_tr);
        double lo = 0.0, hi = -1.0;
        if (r_stride > 0.0) {
            lo = (1.0 - theta) * p_stride / r_stride;
            hi = r_stride == to_bound ? theta * to_bound : to_tr;
        }
        if (lo <= hi) {
            const double Ar = Ah(r_h);
            double a = r_h * Ar, b = gh * r_h + p_h * Ar, z = 0.0;
            warp_sum3(a, b, z);
            const double t = min_quad_1d(0.5 * a, b, lo, hi, 0.5 * qa + qb, r_value);
            r_hs = fma(r_h, t, p_h);
            r_step = d * r_hs;
        }
    }
    const double p_value = 0.5 * theta * theta * qa + theta * qb;
    double ag_h = act ? -gh : 0.0;
    double ag_value, ag_stride;
    {
        const double Aag = Ah(ag_h);
        double a = ag_h * Aag, b = gh * ag_h, gg = ag_h * ag_h;
        warp_sum3(a, b, gg);
        const double to_tr = Delta / sqrt(gg);
        bool h3;
        const double to_bound = step_to_bound(act, x, d * ag_h, lb, ub, h3);
        const double hi = to_bound < to_tr ? theta * to_bound : to_tr;
        ag_stride = min_quad_1d(0.5 * a, b, 0.0, hi, 0.0, ag_value);
    }
    if (p_value < r_value && p_value < ag_value) { s_h = theta * p_h; predicted = -p_value; return theta * p; }
    if (r_value < p_value && r_value < ag_value) { s_h = r_hs; predicted = -r_value; return r_step; }
    s_h = ag_h * ag_stride; predicted = -ag_value;
    return d * ag_h * ag_stride;
}

// ---------------------------------------------------------------------------
// the fit kernel
// ---------------------------------------------------------------------------
// EXTRA: doubles per warp behind the layout of FitLayout (the q | T' buffer of TransEval)
template <class F, int EXTRA = 0>
__device__ __forceinline__ void setup_ctx(WarpCtx<F>& c, double* smem, const FitParams& P) {
    typedef FitLayout<F> Lay;
    const int warp = threadIdx.x >> 5;
    c.lane = threadIdx.x & 31;
    const int wt_region = P.wt_in_smem ? ((P.wt_total + 1) & ~1) : 0;
    if (P.wt_in_smem) {
        for (int i = threadIdx.x; i < P.wt_total; i += blockDim.x) smem[i] = P.blk_wt[i];
        c.wt = smem;
    } else {
        c.wt = P.blk_wt;
    }
    double* base = smem + wt_region + (size_t)warp * (Lay::per_warp_doubles(P.rb) + EXTRA);
    c.R = base;
    c.dvec = c.R + (size_t)P.rb * Lay::LDR;
    c.Abuf[0] = c.dvec + P.rb;
    c.Abuf[1] = c.Abuf[0] + Lay::NP * Lay::LDA;
    c.A = c.Abuf[0];
    c.L = c.Abuf[1] + Lay::NP * Lay::LDA;
    c.p = c.L + Lay::NP * Lay::LDA;
    c.pn = c.p + Lay::NP;
    c.g = c.pn + Lay::NP;
    c.sinv = c.g + Lay::NP;
    c.dsc = c.sinv + Lay::NP;
    c.idg = c.dsc + Lay::NP;
    c.gbuf[0] = c.g;
    c.gbuf[1] = c.idg + Lay::NP;
    c.colb = c.gbuf[1] + Lay::NP;
    __syncthreads();
}

// Robust loss (fit_kernel<F, 6>): the covariance of the rescaled normal matrix in c.A at the solution, by the rule of
// fit_one's results block -- columns scaled by their norms; the Cholesky factor when well conditioned, else the QR
// pass over the rescaled rows (EV::run mode 1); NaN at a non-finite point.  fit_one then evaluates the true rows.
template <class F, class EV>
__device__ __forceinline__ void robust_covariance(WarpCtx<F>& c, bool finite, double* cov_out, int& nfac, int& njev,
                                                  EV& ev) {
    constexpr int NP = FitLayout<F>::NP, LDA = FitLayout<F>::LDA;
    const int lane = c.lane;
    const bool act = lane < NP;
    if (act) {
        const double s = sqrt(c.A[lane * LDA + lane]);
        c.dsc[lane] = s > 0.0 ? 1.0 / s : 1.0;
    }
    __syncwarp();
    ++nfac;
    double pdummy, fres[3];
    const bool okc = factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, 0.0, 0.0, true, &pdummy, fres);
    if (okc && fres[2] > 1e-6) {
        covariance_from_chol<F>(c, cov_out);
    } else if (finite) {
        ev.run(c, c.p, nullptr, nullptr, 1);
        ++njev;
        covariance_from_qr<F>(c, cov_out);
    } else if (cov_out && act) {
        for (int j = 0; j < NP; ++j) cov_out[lane * NP + j] = nan("");
    }
}

// Evaluator of the one-warp-per-fit kernel: the warp evaluates all rows itself.
template <class F>
struct WarpEval {
    // the means of fit b (global memory)
    __device__ __forceinline__ const double* begin(WarpCtx<F>&, const FitParams& P, int b) {
        return P.mean + (size_t)b * P.mean_stride;
    }
    __device__ __forceinline__ double run(WarpCtx<F>& c, const double* pv, double* fout, double* Jout, int mode) {
        return mode == 0 ? eval_full<F, 0>(c, pv, fout, Jout) : eval_full<F, 1>(c, pv, fout, Jout);
    }
};

// Evaluator of the window kernel (fit_kernel<F, 4>): one warp per fit, fit b is copy b % win_copies of window
// b / win_copies, with that window's rows and weights
template <class F>
struct WinEval {
    int w;
    __device__ __forceinline__ const double* begin(WarpCtx<F>&, const FitParams& P, int b) {
        w = b / P.win_copies;
        return P.mean + (size_t)(b % P.win_copies) * P.mean_stride;
    }
    __device__ __forceinline__ double run(WarpCtx<F>& c, const double* pv, double* fout, double* Jout, int mode) {
        return mode == 0 ? eval_win_impl<F, 0>(c, w, pv, fout, Jout) : eval_win_impl<F, 1>(c, w, pv, fout, Jout);
    }
};

// Evaluator of the kernels with parameter distributions (fit_kernel<F, 5>, resjac_trans_kernel): as WarpEval, with the
// model evaluated at q = T(p) (eval_trans_impl)
template <class F>
struct TransEval {
    static constexpr int EXTRA = 2 * F::NP;         // doubles per warp: q | T'
    double* qt;
    __device__ __forceinline__ const double* begin(WarpCtx<F>& c, const FitParams& P, int b) {
        qt = c.R + FitLayout<F>::per_warp_doubles(P.rb);
        return P.mean + (size_t)b * P.mean_stride;
    }
    __device__ __forceinline__ double run(WarpCtx<F>& c, const double* pv, double* fout, double* Jout, int mode) {
        if (c.P.wt_in_smem)
            return mode == 0 ? eval_trans_impl<F, 0, true>(c, qt, pv, fout, Jout)
                             : eval_trans_impl<F, 1, true>(c, qt, pv, fout, Jout);
        return mode == 0 ? eval_trans_impl<F, 0, false>(c, qt, pv, fout, Jout)
                         : eval_trans_impl<F, 1, false>(c, qt, pv, fout, Jout);
    }
};

// Evaluator of the robust-loss kernel (fit_kernel<F, 6>): as WarpEval, with every row rescaled by the loss and the
// robust cost returned (eval_robust_impl).  The true rows at the solution come from eval_full (fit_one, MODE 6).
template <class F>
struct RobustEval {
    __device__ __forceinline__ const double* begin(WarpCtx<F>&, const FitParams& P, int b) {
        return P.mean + (size_t)b * P.mean_stride;
    }
    __device__ __forceinline__ double run(WarpCtx<F>& c, const double* pv, double* fout, double* Jout, int mode) {
        if (c.P.wt_in_smem)
            return mode == 0 ? eval_robust_impl<F, 0, true>(c, pv, fout, Jout) : eval_robust_impl<F, 1, true>(c, pv, fout, Jout);
        return mode == 0 ? eval_robust_impl<F, 0, false>(c, pv, fout, Jout) : eval_robust_impl<F, 1, false>(c, pv, fout, Jout);
    }
};

template <class F, int MODE> struct EvalOf { typedef WarpEval<F> type; static constexpr int EXTRA = 0; };
template <class F> struct EvalOf<F, 6> { typedef RobustEval<F> type; static constexpr int EXTRA = 0; };
template <class F> struct EvalOf<F, 4> { typedef WinEval<F> type; static constexpr int EXTRA = 0; };
template <class F> struct EvalOf<F, 5> { typedef TransEval<F> type; static constexpr int EXTRA = TransEval<F>::EXTRA; };

// One complete fit (number b of the batch) driven by the warp that owns `c`: trust-region loop, optional
// polish, covariance, results.  EV::run evaluates residual + Jacobian + normal equations at a point -- by
// this warp alone (WarpEval) or by the warps of a team (lm_team.cuh: TeamEval); everything else is the
// same code for both kernels.
// cycle counters of the warp that drives a fit (diagnostics: b200lm_last_stats entries 3..)
struct PhaseClock {
    long long eval, solve, total, fact;
    __device__ __forceinline__ void clear() { eval = 0; solve = 0; total = 0; fact = 0; }
};


// MODE selects what is COMPILED into a kernel (the trust-region loop is the hot code: every policy it does not run
// would only cost registers and instruction cache):  0 = scipy TRF decisions (the default kernels),  1 = GSL trust/lm
// decisions (b200lm_set_policy),  2 = no loop at all: finalisation of fits the wave kernel has already converged,
// 3 = scipy TRF with bound constraints (trf_bounds: Coleman-Li scaling, select_step; b200lm_set_bounds),
// 4 = scipy TRF on fit windows (the loop of MODE 0; EV = WinEval: rows, weights and means per window, b200lm_set_windows),
// 5 = scipy TRF with parameter distributions (the loop of MODE 0; EV = TransEval: the model at q = T(p),
// b200lm_set_param_dist),
// 6 = scipy TRF with a robust loss (trf_no_bounds with loss_function: the loop of MODE 0 on the rows rescaled by the
// loss and the robust cost, EV = RobustEval; no polish; b200lm_set_loss).
template <class F, class EV, int MODE = 0>
__device__ __forceinline__ void fit_one(WarpCtx<F>& c, EV& ev, const FitParams& P, int b,
                                        unsigned long long& tot_nfev, unsigned long long& tot_njev,
                                        unsigned long long& tot_nfac, PhaseClock& pk) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    const int lane = c.lane;
    const bool act = lane < NP;
    {
        c.mean = ev.begin(c, P, b);
        const double* p0 = P.p0 + (size_t)(MODE == 4 ? b / P.win_copies : b) * P.p0_stride;     // MODE 4: per window
        if (act) c.p[lane] = p0[lane];
        double lbi = -INFINITY, ubi = INFINITY;             // this lane's bounds (MODE 3)
        if constexpr (MODE == 3) {
            if (act) {
                lbi = P.lb[lane]; ubi = P.ub[lane];
                c.p[lane] = feasible_start(c.p[lane], lbi, ubi);
            }
        }
        __syncwarp();

        int cur = 0;                              // buffer holding J^T J, J^T r of the current point
        c.use_buf(0);
        const long long t_fit0 = B200LM_CLOCK();
        double cost = 0.0;
        bool have_A = false;
        if constexpr (MODE == 2) {
            // finalisation after the wave kernel: J^T J at the solution comes from the wave kernel (packed lower
            // triangle, row-major) and chi2 is known -- no evaluation, unless a polish step needs the gradient
            if (P.wave_A && P.polish == 0 && P.status[b] != -1) {
                if (act) {
                    const double* Ap = P.wave_A + (size_t)b * (NP * (NP + 1) / 2) + lane * (lane + 1) / 2;
                    for (int j = 0; j <= lane; ++j) {
                        const double v = Ap[j];
                        c.A[lane * LDA + j] = v;
                        c.A[j * LDA + lane] = v;
                    }
                }
                cost = 0.5 * P.chi2[b];
                have_A = true;
                __syncwarp();
            }
        }
        if (!have_A) cost = ev.run(c, c.p, nullptr, nullptr, 0);
        pk.eval += B200LM_CLOCK() - t_fit0;
        int nfev = 1, njev = 1, nfac = 0;
        int status = -2;                         // -2: running
        if (!isfinite(cost)) status = -1;
        else if (MODE == 2) status = P.status[b];            // the wave kernel has done the trust-region loop (lm_wave.cuh)
        // scale_inv_j = |J_j| = sqrt(A_jj)   (More': running max; scaler 0: 1)
        double sinv = 1.0;
        if (act && P.scaler == 1) {
            sinv = sqrt(c.A[lane * LDA + lane]);
            if (sinv == 0.0) sinv = 1.0;
        }
        double t = act ? c.p[lane] * sinv : 0.0;
        if constexpr (MODE == 3) {
            // Delta0 = |x0 scale_inv / sqrt(v)|, v of the Coleman-Li scaling (scaled by scale_inv where it varies)
            double v, dv;
            cl_scaling(act ? c.p[lane] : 0.0, act ? c.g[lane] : 0.0, lbi, ubi, v, dv);
            if (dv != 0.0) v *= sinv;
            t = act ? t / sqrt(v) : 0.0;
        }
        double Delta = sqrt(warp_sum(t * t));
        if (Delta == 0.0) Delta = 1.0;
        double alpha = 0.0;
        LinModel lm;
        lm.valid = false; lm.a = 0.0; lm.b = 0.0;

        int nit_report = -1;                      // what P.nit reports when it is not nfev (GSL policy: iterations)
        if (MODE == 1 && status == -2) {
            // ---- GSL trust-region driver with the Levenberg-Marquardt sub-problem (gsl_multifit_nlinear: trust.c,
            // lm.c, nielsen.c, scaling.c, convergence.c, fdf.c as called by the reference's src/lsqfit/_gsl.pyx:563-723;
            // CPU restatement: oracle/gsl_lm.py).  One factorisation per trial: (D^-1 J^T J D^-1 + mu I) (D dx) = -D^-1 g.
            const double cn0 = act ? sqrt(c.A[lane * LDA + lane]) : 0.0;          // |J_j|
            double diag = 1.0;                                                    // D_j: levenberg 1, more / marquardt |J_j|
            if (P.scaler != 0) diag = cn0 == 0.0 ? 1.0 : cn0;
            double mu;
            {
                const double m = warp_max(act ? cn0 / diag : 0.0);
                mu = 1.0e-3 * m * m;                                              // nielsen_init
            }
            double nu = 2.0;
            int iter = 0;
            while (status == -2) {
                const double gi = act ? c.g[lane] : 0.0;
                const double d = 1.0 / diag;
                if (act) c.dsc[lane] = d;
                __syncwarp();
                const double gh = d * gi;
                int bad = 0;
                bool found = false;
                double step = 0.0;
                while (!found) {
                    double sh, res[3];
                    ++nfac;
                    const long long t_s0 = B200LM_CLOCK();
                    const bool ok = factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, mu, gh, false, &sh, res);
                    pk.solve += B200LM_CLOCK() - t_s0;
                    double rho = -1.0;
                    double cost_new = cost;
                    step = (act && ok) ? d * sh : 0.0;
                    if (ok) {
                        if (act) { c.pn[lane] = c.p[lane] + step; c.idg[lane] = step; }
                        __syncwarp();
                        double As = 0.0;
                        if (act) {
                            const double* Ar = c.A + lane * LDA;
#pragma unroll
                            for (int j = 0; j < NP; ++j) As = fma(Ar[j], c.idg[j], As);
                        }
                        // quadratic_preduction * |f|^2 / 2 = -(1/2 dx^T A dx + g^T dx)
                        const double predicted = warp_sum(act ? -step * (0.5 * As + gi) : 0.0);
                        __syncwarp();
                        c.use_buf(cur ^ 1);
                        const long long t_e0 = B200LM_CLOCK();
                        cost_new = ev.run(c, c.pn, nullptr, nullptr, 0);
                        pk.eval += B200LM_CLOCK() - t_e0;
                        c.use_buf(cur);
                        ++nfev; ++njev;
                        // trust_calc_rho: |f_trial| >= |f| (or NaN) rejects; rho = (1 - u^2) / pred
                        if (cost_new < cost && predicted > 0.0) rho = (cost - cost_new) / predicted;
                    }
                    if (rho > 0.0) {
                        if (act) c.p[lane] = c.pn[lane];
                        cur ^= 1;
                        c.use_buf(cur);
                        cost = cost_new;
                        __syncwarp();
                        if (P.scaler != 0) {
                            const double cn = act ? sqrt(c.A[lane * LDA + lane]) : 0.0;
                            if (P.scaler == 1) diag = fmax(diag, cn);                 // more
                            else diag = cn == 0.0 ? 1.0 : cn;                         // marquardt
                        }
                        __syncwarp();
                        const double bq = 2.0 * rho - 1.0;                            // nielsen_accept
                        mu *= fmax(0.333333333333333, 1.0 - bq * bq * bq);
                        nu = 2.0;
                        found = true;
                    } else {
                        mu *= nu;                                                     // nielsen_reject
                        nu *= 2.0;
                        if (++bad > 15) break;                                        // GSL_ENOPROG
                    }
                }
                if (!found && iter == 0) { status = 14; iter = 1; break; }            // fdf.c: no progress in the first iteration
                ++iter;
                // gsl_multifit_nlinear_test: dx of the last trial, x, g, f of the current point
                const double xi = act ? c.p[lane] : 0.0;
                const bool small = !act || fabs(step) < P.xtol * P.xtol + P.xtol * fabs(xi) || step == 0.0;
                const double gnorm = warp_max(act ? fabs(c.g[lane] * fmax(xi, 1.0)) : 0.0);
                if (__all_sync(B200LM_FULL, small)) status = 11;
                else if (gnorm <= P.gtol * fmax(cost, 1.0)) status = 12;
                else if (iter >= P.maxit) status = 0;
            }
            nit_report = iter;
            // the scale of the covariance / polish code below
            sinv = diag;
        }

        // MODE 3 (bounds) is the same loop with scipy's trf_bounds changes: the gtol test on |g v|_inf, the scaling
        // d = sqrt(v) / scale_inv, the Coleman-Li diagonal in the sub-problem, select_step, strictly feasible trials
        while ((MODE == 0 || MODE == 3 || MODE == 4 || MODE == 5 || MODE == 6) && status == -2) {
            const double gi = act ? c.g[lane] : 0.0;
            double v = 1.0, dv = 0.0;                              // Coleman-Li scaling (MODE 3)
            const double xi = act ? c.p[lane] : 0.0;
            if constexpr (MODE == 3) cl_scaling(xi, gi, lbi, ubi, v, dv);
            // |g|_inf and |x|^2 of the current point in one reduction (x does not change until a step is accepted)
            double xx = 0.0, g_norm = fabs(gi);
            if constexpr (MODE == 3) g_norm = fabs(gi * v);
            {
                const double pi_ = act ? c.p[lane] : 0.0;
                xx = pi_ * pi_;
                warp_sum_max(xx, g_norm);
            }
            if (g_norm < P.gtol) { status = 1; break; }
            if (nfev >= P.maxit) { status = 0; break; }
            const double xthr = P.xtol * (P.xtol + sqrt(xx));      // xtol test: |step| < xtol (xtol + |x|)
            double d = 1.0 / sinv;
            double ex = 0.0, theta = 0.0;                          // Coleman-Li diagonal, select_step's theta (MODE 3)
            if constexpr (MODE == 3) {
                if (dv != 0.0) v *= sinv;
                ex = act ? gi * dv * d : 0.0;
                d = act ? sqrt(v) * d : 0.0;
                theta = fmax(0.995, 1.0 - g_norm);
            }
            if (act) c.dsc[lane] = d;
            __syncwarp();
            const double gh = d * gi;
            double actual_reduction = -1.0, cost_new = cost;
            int term = -2;
            GNCache gn;
            gn.valid = false;
            while (actual_reduction <= 0.0 && nfev < P.maxit) {
                double sh;
                const long long t_s0 = B200LM_CLOCK();
                // two shifts per round pay off where the factorisation dominates a trial (np = 12..16: +8 % on
                // C3); for small np the extra control flow and code size cost more than they save (C4, np = 6:
                // -10 %), so those kernels do not even contain the dual path
                if constexpr (MODE == 3) {
                    sh = solve_tr_impl<F, true>(c, gh, Delta, alpha, nfac, gn, pk.fact, ex);
                } else if constexpr (NP >= 12 && NP <= 16) {
                    sh = (P.dual_from >= 0 && nfev >= P.dual_from) ? solve_tr_dual<F>(c, gh, Delta, alpha, nfac, gn, lm, pk.fact)
                                                                   : solve_tr<F>(c, gh, Delta, alpha, nfac, gn, pk.fact);
                } else {
                    sh = solve_tr<F>(c, gh, Delta, alpha, nfac, gn, pk.fact);
                }
                pk.solve += B200LM_CLOCK() - t_s0;
                double predicted, step2, sh2;
                if constexpr (MODE == 3) {
                    const double step = select_step<F>(c, xi, gh, sh, d, ex, Delta, theta, lbi, ubi, predicted);
                    if (act) c.pn[lane] = feasible_trial(xi + step, lbi, ubi);
                    step2 = step * step;
                    sh2 = act ? sh * sh : 0.0;
                    double z = 0.0;
                    warp_sum3(step2, sh2, z);
                } else {
                const double step = act ? d * sh : 0.0;
                if (act) { c.pn[lane] = c.p[lane] + step; c.idg[lane] = step; }
                __syncwarp();
                // predicted reduction = -(1/2 step^T A step + g^T step)   (unscaled == scaled); the row sum runs
                // in four independent chains
                double As = 0.0;
                if (act) {
                    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
                    const double* Ar = c.A + lane * LDA;
#pragma unroll
                    for (int j = 0; j + 3 < NP; j += 4) {
                        a0 = fma(Ar[j], c.idg[j], a0);
                        a1 = fma(Ar[j + 1], c.idg[j + 1], a1);
                        a2 = fma(Ar[j + 2], c.idg[j + 2], a2);
                        a3 = fma(Ar[j + 3], c.idg[j + 3], a3);
                    }
#pragma unroll
                    for (int j = NP & ~3; j < NP; ++j) a0 = fma(Ar[j], c.idg[j], a0);
                    As = (a0 + a1) + (a2 + a3);
                }
                // predicted reduction, |step|^2 and |sh|^2 in ONE reduction
                predicted = act ? -step * (0.5 * As + gi) : 0.0;
                step2 = step * step;
                sh2 = act ? sh * sh : 0.0;
                warp_sum3(predicted, step2, sh2);
                }
                __syncwarp();
                // Speculative evaluation: residual AND Jacobian / normal equations at the trial
                // point, into the other buffer.  ~87 % of the trials are accepted, and then no
                // second pass over the rows is needed; a rejected trial leaves the current
                // buffers untouched.
                c.use_buf(cur ^ 1);
                const long long t_e0 = B200LM_CLOCK();
                cost_new = ev.run(c, c.pn, nullptr, nullptr, 0);
                pk.eval += B200LM_CLOCK() - t_e0;
                c.use_buf(cur);
                ++nfev; ++njev;
                if (!isfinite(cost_new)) { Delta = 0.25 * sqrt(sh2); continue; }
                actual_reduction = cost - cost_new;
                // ratio = actual / predicted enters only through comparisons with 1/4 and 3/4: no division
                bool lt25, gt25, gt75;
                if (predicted > 0.0) {
                    lt25 = actual_reduction < 0.25 * predicted;
                    gt25 = actual_reduction > 0.25 * predicted;
                    gt75 = actual_reduction > 0.75 * predicted;
                } else if (predicted == 0.0 && actual_reduction == 0.0) {
                    lt25 = false; gt25 = true; gt75 = true;             // ratio = 1
                } else {
                    lt25 = true; gt25 = false; gt75 = false;            // ratio = 0
                }
                const bool ft = actual_reduction < P.ftol * cost && gt25;
                const bool xt = step2 < xthr * xthr;
                if (ft && xt) term = 4; else if (ft) term = 2; else if (xt) term = 3;
                if (term != -2) break;
                if (lt25) {
                    const double Delta_new = 0.25 * sqrt(sh2);
                    alpha *= Delta / Delta_new;
                    Delta = Delta_new;
                } else if (gt75 && sh2 > (0.95 * 0.95) * Delta * Delta) {
                    alpha *= 0.5;
                    Delta = 2.0 * Delta;
                }
            }
            if (actual_reduction > 0.0) {
                // accept: the trial buffers become the current ones
                if (act) c.p[lane] = c.pn[lane];
                cur ^= 1;
                c.use_buf(cur);
                cost = cost_new;
                __syncwarp();
                if (act && P.scaler == 1) sinv = fmax(sinv, sqrt(c.A[lane * LDA + lane]));
                __syncwarp();      // the diagonal has been read before anything (polish, QR pass) reuses this buffer
            }
            if (term != -2) {
                // the solver behind the reference re-tests gtol before leaving (trf.py loop head)
                double gl = act ? fabs(c.g[lane]) : 0.0;
                if constexpr (MODE == 3) {
                    double v2, dv2;
                    cl_scaling(act ? c.p[lane] : 0.0, act ? c.g[lane] : 0.0, lbi, ubi, v2, dv2);
                    gl *= v2;
                }
                const double gf = warp_max(gl);
                status = gf < P.gtol ? 1 : term;
            }
        }

        // ---- optional Gauss-Newton polish (P.polish > 0; off by default) ----------------
        // The trust-region loop accepts a step only if the cost decreases, and cost differences
        // below eps*cost cannot be resolved in fp64: it stalls ~sqrt(eps*chi2) standard deviations
        // from the stationary point (so does the reference's solver).  Undamped Gauss-Newton
        // steps, accepted on the decrease of the Newton decrement instead of the cost, take the
        // solution on to the gradient's rounding level.
        // (not with bounds: undamped steps would leave the box; not with a loss, as on the single-fit path)
        if (MODE != 3 && MODE != 6 && status >= 1 && P.polish > 0) {
            // Newton decrement dec = g^T (J^T J)^-1 g = predicted decrease of chi2; sqrt(dec) is
            // the distance to the stationary point in standard deviations.
            const double d = 1.0 / sinv;
            if (act) c.dsc[lane] = d;
            __syncwarp();
            double dec_prev = 1e300;
            for (int it = 0; it <= P.polish; ++it) {
                ++nfac;
                const double gh = act ? d * c.g[lane] : 0.0;
                double sh, pres[3];
                if (!factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, 0.0, gh, false, &sh, pres)) break;
                const double dec = -warp_sum(act ? gh * sh : 0.0);
                if (it > 0) {
                    if (!(dec < dec_prev)) {                        // the last step did not help: undo it
                        if (act) { const double t = c.p[lane]; c.p[lane] = c.pn[lane]; c.pn[lane] = t; }
                        __syncwarp();
                        cost = ev.run(c, c.p, nullptr, nullptr, 0);
                        ++njev;
                        break;
                    }
                }
                if (!(dec > 1e-22) || it == P.polish) break;        // < 1e-11 sdev from stationarity
                dec_prev = dec;
                // keep the old point in pn, step to the new one
                if (act) { const double t = c.p[lane]; c.pn[lane] = t; c.p[lane] = t + d * sh; }
                __syncwarp();
                const double cost_try = ev.run(c, c.p, nullptr, nullptr, 0);
                ++nfev; ++njev;
                if (!isfinite(cost_try)) {
                    if (act) c.p[lane] = c.pn[lane];
                    __syncwarp();
                    cost = ev.run(c, c.p, nullptr, nullptr, 0);
                    ++njev;
                    break;
                }
                cost = cost_try;
            }
        }

        // ---- results -----------------------------------------------------------
        if constexpr (MODE == 6) {
            // robust loss: cov from the rescaled normal matrix of the solution (scipy's fit.jac); then the true rows at
            // the solution: f / J, chi2 and the J^T J whose log det the block below takes
            robust_covariance<F>(c, isfinite(cost), P.cov ? P.cov + (size_t)b * NP * NP : nullptr, nfac, njev, ev);
            cost = eval_full<F, 0>(c, c.p, P.f_out ? P.f_out + (size_t)b * P.nchiv : nullptr,
                                   P.J_out ? P.J_out + (size_t)b * P.nchiv * NP : nullptr);
            ++njev;
        } else if (P.f_out || P.J_out) {
            cost = ev.run(c, c.p, P.f_out ? P.f_out + (size_t)b * P.nchiv : nullptr,
                          P.J_out ? P.J_out + (size_t)b * P.nchiv * NP : nullptr, 0);
        }
        // covariance at the solution, scaled by the current column norms for conditioning (MODE 6: the log det of the
        // true J^T J only, its QR pass on the true rows)
        double dfin = 1.0;
        if (act) {
            const double s = sqrt(c.A[lane * LDA + lane]);
            dfin = s > 0.0 ? 1.0 / s : 1.0;
            c.dsc[lane] = dfin;
        }
        __syncwarp();
        ++nfac;
        double pdummy, fres[3];
        const bool okc = factor_solve<NP, LDA>(c.A, c.dsc, c.L, c.idg, c.colb, lane, 0.0, 0.0, true, &pdummy, fres);
        const double pivr = fres[2];
        double* cov_out = (MODE != 6 && P.cov) ? P.cov + (size_t)b * NP * NP : nullptr;
        double ld = nan("");
        if (okc && pivr > 1e-6) {
            // well conditioned: kappa^2 * eps < ~2e-10, the normal-equation factor is accurate enough
            ld = covariance_from_chol<F>(c, cov_out);
        } else if (isfinite(cost)) {
            // ill conditioned: one more pass over the rows, Householder QR of J.diag(dsc)
            if constexpr (MODE == 6) eval_full<F, 1>(c, c.p, nullptr, nullptr);
            else ev.run(c, c.p, nullptr, nullptr, 1);
            ++njev;
            ld = covariance_from_qr<F>(c, cov_out);
        } else if (cov_out && act) {
            for (int j = 0; j < NP; ++j) cov_out[lane * NP + j] = nan("");
        }
        if (act) P.x_out[(size_t)b * NP + lane] = c.p[lane];
        if (lane == 0) {
            P.chi2[b] = 2.0 * cost;
            if (MODE != 2) {
                P.nit[b] = nit_report >= 0 ? nit_report : nfev;
                P.status[b] = status;
            } else if (nfev > 1) {
                P.nit[b] += nfev - 1;                        // polish steps
            }
            if (P.logdet) P.logdet[b] = ld;
        }
        if (MODE == 2) { --nfev; --njev; }
        tot_nfev += nfev; tot_njev += njev; tot_nfac += nfac;
        pk.total += B200LM_CLOCK() - t_fit0;
        __syncwarp();
    }
}

template <class F, int MODE = 0>
__global__ void __launch_bounds__(FitLayout<F>::MAX_WARPS * 32, 1) fit_kernel(const __grid_constant__ FitParams P) {
    typedef FitLayout<F> Lay;
    static_assert(Lay::NP <= 32, "one lane per parameter");
    extern __shared__ double smem[];
    WarpCtx<F> c(P);
    setup_ctx<F, EvalOf<F, MODE>::EXTRA>(c, smem, P);
    const int lane = c.lane;
    unsigned long long tot_nfev = 0, tot_njev = 0, tot_nfac = 0;
    typename EvalOf<F, MODE>::type ev;
    PhaseClock pk;
    pk.clear();

    for (;;) {
        int b = 0;
        if (lane == 0) {
            b = atomicAdd(P.counter, 1);
            if (P.order && b < P.B) b = P.order[b];
        }
        b = __shfl_sync(B200LM_FULL, b, 0);
        if (b >= P.B) break;
        fit_one<F, typename EvalOf<F, MODE>::type, MODE>(c, ev, P, b, tot_nfev, tot_njev, tot_nfac, pk);
    }
    if (lane == 0 && P.stats) {
        atomicAdd(&P.stats[0], tot_nfev);
        atomicAdd(&P.stats[1], tot_njev);
        atomicAdd(&P.stats[2], tot_nfac);
        atomicAdd(&P.stats[3], (unsigned long long)pk.eval);
        atomicAdd(&P.stats[4], (unsigned long long)pk.solve);
        atomicAdd(&P.stats[5], (unsigned long long)pk.total);
        atomicAdd(&P.stats[11], (unsigned long long)pk.fact);
    }
}

// residual + Jacobian at given parameter vectors (test hook for the chiv parity of
// reference src/lsqfit/_utilities.pyx:65-94); P.p0 holds the B parameter vectors.
template <class F>
__global__ void __launch_bounds__(FitLayout<F>::MAX_WARPS * 32, 1) resjac_kernel(const __grid_constant__ FitParams P) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP;
    extern __shared__ double smem[];
    WarpCtx<F> c(P);
    setup_ctx<F>(c, smem, P);
    const int lane = c.lane;
    const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int nwarps = gridDim.x * (blockDim.x >> 5);
    for (int b = warp_global; b < P.B; b += nwarps) {
        c.mean = P.mean + (size_t)b * P.mean_stride;
        const double* p0 = P.p0 + (size_t)b * P.p0_stride;
        if (lane < NP) c.p[lane] = p0[lane];
        __syncwarp();
        const double cost = eval_full<F>(c, c.p, P.f_out ? P.f_out + (size_t)b * P.nchiv : nullptr,
                                         P.J_out ? P.J_out + (size_t)b * P.nchiv * NP : nullptr);
        if (lane == 0 && P.chi2) P.chi2[b] = 2.0 * cost;
        __syncwarp();
    }
}

// the same with parameter distributions (P.ntrans > 0): f and J in fit space, J = dchiv/dp
template <class F>
__global__ void __launch_bounds__(FitLayout<F>::MAX_WARPS * 32, 1) resjac_trans_kernel(const __grid_constant__ FitParams P) {
    constexpr int NP = F::NP;
    extern __shared__ double smem[];
    WarpCtx<F> c(P);
    setup_ctx<F, TransEval<F>::EXTRA>(c, smem, P);
    const int lane = c.lane;
    TransEval<F> ev;
    const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int nwarps = gridDim.x * (blockDim.x >> 5);
    for (int b = warp_global; b < P.B; b += nwarps) {
        c.mean = ev.begin(c, P, b);
        const double* p0 = P.p0 + (size_t)b * P.p0_stride;
        if (lane < NP) c.p[lane] = p0[lane];
        __syncwarp();
        const double cost = ev.run(c, c.p, P.f_out ? P.f_out + (size_t)b * P.nchiv : nullptr,
                                   P.J_out ? P.J_out + (size_t)b * P.nchiv * NP : nullptr, 0);
        if (lane == 0 && P.chi2) P.chi2[b] = 2.0 * cost;
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------
struct LaunchInfo {
    int grid, block;
    size_t smem;
};

// extra: doubles per warp behind the FitLayout (EvalOf<F, MODE>::EXTRA of the kernel launched)
template <class F>
inline cudaError_t plan_launch(FitParams& P, int sm_count, size_t smem_budget, LaunchInfo& li, int extra = 0) {
    typedef FitLayout<F> Lay;
    const size_t wt_bytes = ((size_t)(P.wt_total + 1) & ~(size_t)1) * sizeof(double);
    const size_t per_warp = (size_t)(Lay::per_warp_doubles(P.rb) + extra) * sizeof(double);
    P.wt_in_smem = (P.nwin == 0 && P.wt_total > 0 && wt_bytes + 4 * per_warp <= smem_budget) ? 1 : 0;
    const size_t avail = smem_budget - (P.wt_in_smem ? wt_bytes : 0);
    int warps = (int)(avail / per_warp);
    if (warps < 1) return cudaErrorInvalidConfiguration;
    if (warps > Lay::MAX_WARPS) warps = Lay::MAX_WARPS;
    if (const char* env = getenv("B200LM_WARPS")) {          // tuning knob (profiling only)
        const int w = atoi(env);
        if (w >= 1 && w < warps) warps = w;
    }
    P.warps = warps;
    li.block = warps * 32;
    li.smem = (P.wt_in_smem ? wt_bytes : 0) + warps * per_warp;
    // one persistent CTA per SM; a batch smaller than the machine is SPREAD over the SMs (a fit is latency
    // bound: 7 fits on each of 148 SMs finish sooner than 12 on each of 84)
    int grid = P.B < sm_count ? P.B : sm_count;
    if (grid < 1) grid = 1;
    li.grid = grid;
    return cudaSuccess;
}

template <class F, int MODE>
cudaError_t launch_fit_mode(const FitParams& P, const LaunchInfo& li, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(fit_kernel<F, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)li.smem);
    if (e != cudaSuccess) return e;
    fit_kernel<F, MODE><<<li.grid, li.block, li.smem, stream>>>(P);
    return cudaGetLastError();
}

template <class F>
cudaError_t launch_fit(FitParams P, int sm_count, size_t smem_budget, cudaStream_t stream) {
    LaunchInfo li;
    // parameter distributions: b200lm_set_param_dist refuses windows, bounds and the GSL policy, and the wave kernel
    // (the only user of finalize_only) does not run with them
    const bool trans = P.ntrans > 0;
    cudaError_t e = plan_launch<F>(P, sm_count, smem_budget, li, trans ? EvalOf<F, 5>::EXTRA : 0);
    if (e != cudaSuccess) return e;
    if (trans) return launch_fit_mode<F, 5>(P, li, stream);
    // a robust loss: b200lm_set_loss refuses windows, bounds, distributions and the GSL policy, and the batch runs
    // one warp per fit (no wave kernel, so no finalize_only)
    if (P.loss > 0) return launch_fit_mode<F, 6>(P, li, stream);
    if (P.nwin > 0) return launch_fit_mode<F, 4>(P, li, stream);
    if (P.finalize_only) return launch_fit_mode<F, 2>(P, li, stream);
    if (P.bounded) return launch_fit_mode<F, 3>(P, li, stream);
    if (P.policy == 1) return launch_fit_mode<F, 1>(P, li, stream);
    return launch_fit_mode<F, 0>(P, li, stream);
}

template <class F>
cudaError_t launch_resjac(FitParams P, int sm_count, size_t smem_budget, cudaStream_t stream) {
    LaunchInfo li;
    if (P.ntrans > 0) {
        cudaError_t e = plan_launch<F>(P, sm_count, smem_budget, li, TransEval<F>::EXTRA);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(resjac_trans_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)li.smem);
        if (e != cudaSuccess) return e;
        resjac_trans_kernel<F><<<li.grid, li.block, li.smem, stream>>>(P);
        return cudaGetLastError();
    }
    cudaError_t e = plan_launch<F>(P, sm_count, smem_budget, li);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(resjac_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)li.smem);
    if (e != cudaSuccess) return e;
    resjac_kernel<F><<<li.grid, li.block, li.smem, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace b200lm
