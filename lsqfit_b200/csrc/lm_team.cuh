// Team variant of the batched LM kernel: TW warps (2 or 4) cooperate on ONE fit.
//
// Why: a batch of correlator fits is bounded by its slowest copies (the reference solver itself needs
// up to ~400 trial points on 1 % of the bootstrap copies) and by the LATENCY of one trial -- not by
// FP64 throughput (measured on B200: DFMA 8.5, DMMA 26, 64-bit shuffle 26, shared-memory round trip 42,
// L2 hit > 500 cycles; tools/micro/lat_probe.cu).  Here the evaluation of residual + Jacobian + normal
// equations (the reference's chiv, src/lsqfit/_utilities.pyx:65-94, plus J^T J) is split over the warps
// of a team and everything a trial touches lives in shared memory:
//   once per CTA   block weights W, x, the index tables of the whitening        (staged)
//   once per fit   the means of y (+) prior                                      (TeamEval::begin)
//   P1  the team fills a 64-row chunk of [G | delta]: one model row per lane, or per PAIR of lanes where
//       the functor can split its terms (value_grad_part), stored TRANSPOSED (T[col][row]) so that the
//       stores are conflict free and every DMMA fragment is one 16-byte load
//   P2  warp w multiplies ITS 64/TW rows of W with the chunk on the FP64 tensor path (C fragments stay
//       in registers across chunks)
//   P3  the finished rows [J | r] go through shared memory once (row-major, own rows only) into the
//       warp's partial J^T J and J^T r tiles (DMMA); the leader adds the partials in a fixed order,
//       stores A, g and adds the 1x1 prior rows.
// The trust-region logic (fit_one, shared with the one-warp kernel) runs on the team's leader warp,
// which posts "evaluate at p" commands to its helpers; teams synchronise with named barriers, so
// several teams share one CTA and one staged copy of the weights.
#pragma once
#include <cstdio>
#include "lm_kernel.cuh"

#ifndef B200LM_P2_PIPE
#define B200LM_P2_PIPE 1
#endif

namespace b200lm {

template <class F, int TW>
struct TeamLayout {
    typedef FitLayout<F> Lay;
    static constexpr int NP = Lay::NP, NT = Lay::NT, LDR = Lay::LDR, LDA = Lay::LDA, NCOL = Lay::NCOL;
    static constexpr int CH = 64;                 // rows per input chunk / output group
    static constexpr int MT = 8 / TW;             // 8-row output tiles per warp and group
    static constexpr int RW = CH / TW;            // rows of a chunk / group owned by one warp
    static constexpr int LPR = (RW <= 16 && SplitOf<F>::value >= 2) ? 2 : 1;   // lanes per model row in P1
    static constexpr int LDT = 72;                // row stride of the transposed chunk (== 8 mod 16, >= CH)
    static constexpr int TROWS = 8 * NT > NP + 1 ? 8 * NT : NP + 1;
    static constexpr int UNION = TROWS * LDT > CH * LDR ? TROWS * LDT : CH * LDR;
    // partial sums of one warp: upper tiles of J^T J (2 doubles per lane each), J^T r tiles, r^T r
    static constexpr int NGT = Lay::DELTA_IN_TILE ? 0 : Lay::NTA;
    static constexpr int NACC = 2 * Lay::NTRI + NGT + 1;
    static constexpr bool STAGE_OWN = NACC * 32 <= RW * LDR;       // partials fit into the warp's own rows
    static constexpr int CMD = 8;                                  // scratch (4 doubles) + command block (8 ints)
    static constexpr int MAX_THREADS = 512;      // 4 teams of 4 or 8 teams of 2 (measured best on C3), 128 registers per thread
    static constexpr int MAX_TEAMS = MAX_THREADS / (32 * TW) > 15 ? 15 : MAX_THREADS / (32 * TW);
    // doubles per team, without the staged means
    static constexpr int FIXED = (UNION + 3 * NP * LDA + (Lay::NVEC + 1) * NP + 64 + CMD + 1) & ~1;
    __host__ __device__ static int per_team_doubles(int N) { return FIXED + ((N + 1) & ~1); }
};

template <class F, int TW>
struct TeamCtx {
    WarpCtx<F> c;
    int* cmd;
    double* mean_s;           // this fit's means, staged by the leader
    const double *xs, *fw, *pw;       // x rows, 1x1 data weights, 1x1 prior weights
    const int *bidx, *fidx, *pidx;    // block / 1x1 data / 1x1 prior index tables
    int tw;        // warp index inside the team (0 = leader)
    int bar;       // named barrier of the team
    __device__ TeamCtx(const FitParams& P) : c(P) {}
};

template <int TW>
__device__ __forceinline__ void team_sync(int bar) {
    asm volatile("bar.sync %0, %1;" ::"r"(bar), "n"(TW * 32) : "memory");
}

// strided view of one column position of the transposed chunk: g[j] = T[j][kk]
template <int LD>
struct ColOut {
    double* p;
    __device__ __forceinline__ double& operator[](int j) const { return p[j * LD]; }
};

// shared memory of the CTA: [ block weights | x, 1x1 weights | index tables | team 0 | team 1 | ... ]
struct TeamStage {
    int wt, x, fw, pw, ints, total;     // offsets in doubles (ints: start of the int tables), total doubles
};
__host__ __device__ inline TeamStage team_stage(const FitParams& P) {
    TeamStage s;
    s.wt = 0;
    s.x = (P.wt2_total + 1) & ~1;
    s.fw = s.x + P.ny * P.nx;
    s.pw = s.fw + P.nd_fn;
    s.ints = (s.pw + P.nd_pr + 1) & ~1;
    const int nints = P.nblk_idx + P.nd_fn + P.nd_pr;
    s.total = (s.ints + (nints + 1) / 2 + 1) & ~1;
    return s;
}

// every pointer of a team's context from its base address (cheap to recompute: the offsets are
// compile-time constants or kernel parameters, so nothing has to travel through local memory)
template <class F, int TW>
__device__ __forceinline__ void team_pointers(TeamCtx<F, TW>& tc, const FitParams& P, double* base, const double* stage) {
    typedef FitLayout<F> Lay;
    typedef TeamLayout<F, TW> TL;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    WarpCtx<F>& c = tc.c;
    if (P.staged) {
        const TeamStage st = team_stage(P);
        const int* si = reinterpret_cast<const int*>(stage + st.ints);
        c.wt = stage + st.wt;
        tc.xs = stage + st.x; tc.fw = stage + st.fw; tc.pw = stage + st.pw;
        tc.bidx = si; tc.fidx = si + P.nblk_idx; tc.pidx = si + P.nblk_idx + P.nd_fn;
    } else {
        c.wt = P.blk_wt2;
        tc.xs = P.x; tc.fw = P.dfn_w; tc.pw = P.dpr_w;
        tc.bidx = P.blk_idx; tc.fidx = P.dfn_idx; tc.pidx = P.dpr_idx;
    }
    c.R = base;
    c.Abuf[0] = c.R + TL::UNION;
    c.Abuf[1] = c.Abuf[0] + NP * LDA;
    c.A = c.Abuf[0];
    c.L = c.Abuf[1] + NP * LDA;
    c.p = c.L + NP * LDA;
    c.pn = c.p + NP;
    c.g = c.pn + NP;
    c.sinv = c.g + NP;
    c.dsc = c.sinv + NP;
    c.idg = c.dsc + NP;
    c.gbuf[0] = c.g;
    c.gbuf[1] = c.idg + NP;
    c.colb = c.gbuf[1] + NP;                       // column broadcast buffers of the factorisation
    c.dvec = c.colb + 64;                          // CMD doubles: scratch (4) + command ints
    tc.cmd = reinterpret_cast<int*>(c.dvec + 4);
    tc.mean_s = base + TL::FIXED;
    c.mean = tc.mean_s;
}

__device__ __forceinline__ double* shared_ptr(unsigned s) { return reinterpret_cast<double*>(__cvta_shared_to_generic(s)); }
__device__ __forceinline__ unsigned shared_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// the operands arrive as shared-memory addresses: a context passed by reference would have to sit in local memory
template <class F>
__device__ __noinline__ void qr_update_rows(unsigned A_s, unsigned dsc_s, unsigned S_s, int nrows, int lane) {
    qr_update<F>(shared_ptr(A_s), shared_ptr(dsc_s), shared_ptr(S_s), nrows, lane);
}

// partial normal equations of one warp in DMMA C-fragment layout
template <class F, int TW>
struct TeamAcc {
    typedef FitLayout<F> Lay;
    typedef TeamLayout<F, TW> TL;
    double t[Lay::NTRI][2];                     // tiles (ta <= tb) of S^T S, S = [J | r | 0]
    double g[TL::NGT > 0 ? TL::NGT : 1][2];     // J^T r tiles (np % 8 == 0: the residual column has no tile of its own)
    double cost;                                // partial of r^T r (same case)
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int q = 0; q < Lay::NTRI; ++q) { t[q][0] = 0.0; t[q][1] = 0.0; }
#pragma unroll
        for (int q = 0; q < (TL::NGT > 0 ? TL::NGT : 1); ++q) { g[q][0] = 0.0; g[q][1] = 0.0; }
        cost = 0.0;
    }
};

// acc += S^T S (and S^T r, r^T r) over nrows4 rows (multiple of 4, rows beyond the data are zero) of the
// row-major buffer S = [J | r | 0].  Everything but r^T r runs on the tensor path.
template <class F, int TW>
__device__ __forceinline__ void team_accumulate(const double* S, int nrows4, int lane, TeamAcc<F, TW>& na) {
    typedef FitLayout<F> Lay;
    constexpr int NP = Lay::NP, NT = Lay::NT, LDR = Lay::LDR;
    const double* base = S + (lane & 3) * LDR + (lane >> 2);
    const bool col0 = (lane >> 2) == 0;
#pragma unroll 4
    for (int s4 = 0; s4 < nrows4; s4 += 4) {
        double f[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) f[t] = base[s4 * LDR + 8 * t];
        int q = 0;
#pragma unroll
        for (int ta = 0; ta < NT; ++ta)
#pragma unroll
            for (int tb = ta; tb < NT; ++tb) { dmma(na.t[q][0], na.t[q][1], f[ta], f[tb]); ++q; }
        if constexpr (!Lay::DELTA_IN_TILE) {
            // B tile with r in column 0: C[i][0] = sum_k J[k][8 ta + i] r[k]
            const double rk = S[(s4 + (lane & 3)) * LDR + NP];
            const double fr = col0 ? rk : 0.0;
#pragma unroll
            for (int ta = 0; ta < NT; ++ta) dmma(na.g[ta][0], na.g[ta][1], f[ta], fr);
            na.cost = fma(fr, fr, na.cost);          // lanes 0..3 cover the four rows of the step
        }
    }
}

// leader: STORE the summed tiles as A = J^T J, g = J^T r (every entry of A is covered by a tile);
// returns this lane's share of r^T r
template <class F, int TW>
__device__ __forceinline__ double team_flush(WarpCtx<F>& c, TeamAcc<F, TW>& na) {
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
                    c.A[row * LDA + col] = v;
                    if (ta != tb) c.A[col * LDA + row] = v;
                } else if (Lay::DELTA_IN_TILE && col == NP && row < NP) {
                    c.g[row] = v;
                } else if (Lay::DELTA_IN_TILE && col == NP && row == NP) {
                    cost += v;
                }
            }
            ++q;
        }
    if constexpr (!Lay::DELTA_IN_TILE) {
        if ((lane & 3) == 0) {
#pragma unroll
            for (int ta = 0; ta < NT; ++ta) {
                const int row = 8 * ta + (lane >> 2);
                if (row < NP) c.g[row] = na.g[ta][0];
            }
        }
    }
    __syncwarp();
    return cost;
}

// residual + Jacobian + normal equations at pv by the whole team; the leader (tw == 0) receives
// A = J^T J, g = J^T r in c.A / c.g and the cost as return value.  mode 1: the leader instead folds
// all rows into the Householder factor of J.diag(dsc) (final covariance of ill-conditioned fits).
template <class F, int TW, bool STAGED>
__device__ __noinline__ double team_eval_impl(const FitParams& P, unsigned base_s, unsigned stage_s, int ids, int flags,
                                              double* fout, double* Jout) {
    // the context arrives as two shared-memory OFFSETS: every pointer is rebuilt from them (constants and
    // kernel parameters only), so nothing is copied through local memory and the compiler knows the
    // address space of everything it derives (LDS/STS without __builtin_assume)
    double* base = shared_ptr(base_s);
    const double* stage = shared_ptr(stage_s);
    typedef FitLayout<F> Lay;
    typedef TeamLayout<F, TW> TL;
    constexpr int NP = Lay::NP, NT = Lay::NT, LDR = Lay::LDR, LDA = Lay::LDA, NCOL = Lay::NCOL;
    constexpr int CH = TL::CH, MT = TL::MT, RW = TL::RW, LDT = TL::LDT, TROWS = TL::TROWS, LPR = TL::LPR;
    // ids = lane | tw << 8 | bar << 16 ;  flags = mode | pv_sel << 1 | cur << 2
    TeamCtx<F, TW> tc(P);
    WarpCtx<F>& c = tc.c;
    team_pointers<F, TW>(tc, P, base, stage);
    c.lane = ids & 31; tc.tw = (ids >> 8) & 7; tc.bar = ids >> 16;
    const int mode = flags & 1;
    c.use_buf((flags >> 2) & 1);
    const double* pv = (flags & 2) ? c.pn : c.p;
    const int lane = c.lane, tw = tc.tw, bar = tc.bar;
    double* Jb = c.R;                       // row-major view  [CH][LDR]  of finished rows [J | r]
    double* T = c.R;                        // transposed view [TROWS][LDT] of a chunk of [G | delta]
    double* Jown = Jb + tw * RW * LDR;      // the rows this warp owns
    TeamAcc<F, TW> na;
    na.clear();
    bool dirty = false;                     // the buffer may still be read by another warp of the team
#ifdef B200LM_PHASE_TICKS
    long long tk0 = B200LM_CLOCK(), tk[5] = {0, 0, 0, 0, 0};
#define B200LM_TICK(i) do { const long long t_ = B200LM_CLOCK(); tk[i] += t_ - tk0; tk0 = t_; } while (0)
#else
#define B200LM_TICK(i) do { } while (0)
#endif

    // 1x1 prior rows (leader): J row = w e_j, analytic contribution.  mode 0: added on top of the stored
    // tiles at the end; mode 1: the diagonal matrix that starts the triangular factor.
    auto prior_rows = [&]() -> double {
        double a = 0.0;
        for (int i = lane; i < P.nd_pr; i += 32) {
            const int idx = tc.pidx[i];
            const int j = idx - P.ny;
            const double w = tc.pw[i];
            const double rr = w * (pv[j] - c.mean[idx]);
            if (mode == 0) {
                c.A[j * LDA + j] += w * w;
                c.g[j] += w * rr;
            } else {
                c.A[j * LDA + j] = w * c.dsc[j];
            }
            a = fma(rr, rr, a);
            if (fout) fout[P.nd_fn + i] = rr;
            if (Jout) {
                for (int u = 0; u < NP; ++u) Jout[(size_t)(P.nd_fn + i) * NP + u] = (u == j) ? w : 0.0;
            }
        }
        __syncwarp();
        return a;
    };
    double acc = 0.0;
    if (mode != 0 && tw == 0) {
        for (int e = lane; e < NP * LDA; e += 32) c.A[e] = 0.0;
        __syncwarp();
        acc += prior_rows();
    }
    // 1x1 data rows: CH rows per pass, RW of them per warp (one row per lane), consumed by the same warp
    for (int c0 = 0; c0 < P.nd_fn; c0 += CH) {
        const int my0 = c0 + tw * RW;
        const int nrows = max(0, min(RW, P.nd_fn - my0));
        if (dirty) team_sync<TW>(bar);
        for (int rr = lane; rr < RW; rr += 32) {
            double* row_ = Jown + rr * LDR;
            if (rr < nrows) {
                const int row = tc.fidx[my0 + rr];
                const double w = tc.fw[my0 + rr];
                const double f = F::value_grad(tc.xs + (size_t)row * P.nx, row, pv, w, row_);
                row_[NP] = w * (f - c.mean[row]);
#pragma unroll
                for (int j = NP + 1; j < NCOL; ++j) row_[j] = 0.0;
            } else {
#pragma unroll
                for (int j = 0; j < NCOL; ++j) row_[j] = 0.0;
            }
        }
        __syncwarp();
        if (mode == 0) {
            if (nrows > 0) {
                if (fout || Jout) emit_rows<F>(Jown, nrows, my0, lane, fout, Jout);
                team_accumulate<F, TW>(Jown, (nrows + 3) & ~3, lane, na);
            }
            __syncwarp();
            dirty = false;                  // only this warp reads its rows
        } else {
            team_sync<TW>(bar);
            if (tw == 0) {
                const int nall = min(CH, P.nd_fn - c0);
                if (fout || Jout) emit_rows<F>(Jb, nall, c0, lane, fout, Jout);
                __syncwarp();
                qr_update_rows<F>(shared_addr(c.A), shared_addr(c.dsc), shared_addr(Jb), nall, lane);
            }
            dirty = true;
        }
    }
    B200LM_TICK(0);
    if (P.nd_fn > 0) dirty = true;          // the chunk buffer aliases the rows the other warps are still reading
    // correlated blocks: J_blk = W . [G | delta]
    const int q = lane & 3, r = lane >> 2;
    for (int b = 0; b < P.nblk; ++b) {
        const BlockDesc bd = P.blk[b];
        const double* W = c.wt + bd.wt2_off;
        const int ldw = bd.ldw2;
        for (int g0 = 0; g0 < bd.n_out; g0 += CH) {
            double pc[MT][NT][2];
            double pr[MT];
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                pr[m] = 0.0;
#pragma unroll
                for (int t = 0; t < NT; ++t) { pc[m][t][0] = 0.0; pc[m][t][1] = 0.0; }
            }
            for (int k0 = 0; k0 < bd.n_in; k0 += CH) {
                const int nk = min(CH, bd.n_in - k0);
                const int nk8 = (nk + 7) & ~7;
                if (dirty) team_sync<TW>(bar);
                // ---- P1: the chunk of [G | delta], transposed; LPR lanes share one model row ----------
                for (int u = lane; u < RW * LPR; u += 32) {
                    const int kk = tw * RW + (LPR == 2 ? (u & (RW - 1)) : u);
                    const int part = LPR == 2 ? u / RW : 0;
                    int idx = 0;
                    bool model = false;
                    double f = 0.0;
                    if (kk < nk) {
                        idx = tc.bidx[bd.idx_off + k0 + kk];
                        model = idx < P.ny;
                        if (model) {
                            if constexpr (LPR == 2)
                                f = F::value_grad_part(tc.xs + (size_t)idx * P.nx, idx, pv, 1.0, ColOut<LDT>{T + kk}, part);
                            else
                                f = F::value_grad(tc.xs + (size_t)idx * P.nx, idx, pv, 1.0, ColOut<LDT>{T + kk});
                        }
                    }
                    if constexpr (LPR == 2) f += __shfl_xor_sync(B200LM_FULL, f, RW);    // the two halves of the row
                    if (part == 0) {
                        if (kk < nk) {
                            double dlt;
                            if (model) {
                                dlt = f - c.mean[idx];
                            } else {                       // a prior entry inside a correlated block: unit row
                                const int j0 = idx - P.ny;
#pragma unroll
                                for (int j = 0; j < NP; ++j) T[j * LDT + kk] = (j == j0) ? 1.0 : 0.0;
                                dlt = pv[j0] - c.mean[idx];
                            }
                            T[NP * LDT + kk] = dlt;
#pragma unroll
                            for (int j = NP + 1; j < TROWS; ++j) T[j * LDT + kk] = 0.0;
                        } else if (kk < nk8) {
#pragma unroll
                            for (int j = 0; j < TROWS; ++j) T[j * LDT + kk] = 0.0;
                        }
                    }
                }
                team_sync<TW>(bar);
                B200LM_TICK(1);
                // ---- P2: own rows of W times the chunk.  k-slot q of the two DMMA steps of an
                // 8-wide slab holds k = S + 2q and S + 2q + 1: both fragments are one 16-byte load.
                // (W is zero padded to whole 64-row groups: no row guards.)
                const double* wa = W + (size_t)(g0 + 8 * (tw * MT) + r) * ldw + k0 + 2 * q;
                const double* tb = T + r * LDT + 2 * q;
#if B200LM_P2_PIPE
                const double* td = T + NP * LDT + 2 * q;
                double2 bf[NT], af[MT], dl = make_double2(0.0, 0.0);
#pragma unroll
                for (int t = 0; t < NT; ++t) bf[t] = *reinterpret_cast<const double2*>(tb + 8 * t * LDT);
#pragma unroll
                for (int m = 0; m < MT; ++m) af[m] = *reinterpret_cast<const double2*>(wa + (size_t)m * 8 * ldw);
                if constexpr (!Lay::DELTA_IN_TILE) dl = *reinterpret_cast<const double2*>(td);
#pragma unroll 2
                for (int S = 0; S < nk8; S += 8) {
                    // software pipeline: the fragments of the next slab are in flight while this one is multiplied
                    // (the last iteration re-reads the current slab: in bounds, unused)
                    const int Sn = S + 8 < nk8 ? S + 8 : S;
                    double2 bfn[NT], afn[MT], dln = make_double2(0.0, 0.0);
#pragma unroll
                    for (int t = 0; t < NT; ++t) bfn[t] = *reinterpret_cast<const double2*>(tb + 8 * t * LDT + Sn);
#pragma unroll
                    for (int m = 0; m < MT; ++m) afn[m] = *reinterpret_cast<const double2*>(wa + (size_t)m * 8 * ldw + Sn);
                    if constexpr (!Lay::DELTA_IN_TILE) dln = *reinterpret_cast<const double2*>(td + Sn);
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
#pragma unroll
                        for (int t = 0; t < NT; ++t) dmma(pc[m][t][0], pc[m][t][1], af[m].x, bf[t].x);
                    }
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
#pragma unroll
                        for (int t = 0; t < NT; ++t) dmma(pc[m][t][0], pc[m][t][1], af[m].y, bf[t].y);
                        if constexpr (!Lay::DELTA_IN_TILE) pr[m] = fma(af[m].x, dl.x, fma(af[m].y, dl.y, pr[m]));
                    }
#pragma unroll
                    for (int t = 0; t < NT; ++t) bf[t] = bfn[t];
#pragma unroll
                    for (int m = 0; m < MT; ++m) af[m] = afn[m];
                    dl = dln;
                }
#else
#pragma unroll 4
                for (int S = 0; S < nk8; S += 8) {
                    double2 bf[NT];
#pragma unroll
                    for (int t = 0; t < NT; ++t) bf[t] = *reinterpret_cast<const double2*>(tb + 8 * t * LDT + S);
                    double2 dl = make_double2(0.0, 0.0);
                    if constexpr (!Lay::DELTA_IN_TILE) dl = *reinterpret_cast<const double2*>(T + NP * LDT + S + 2 * q);
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        const double2 af = *reinterpret_cast<const double2*>(wa + (size_t)m * 8 * ldw + S);
#pragma unroll
                        for (int t = 0; t < NT; ++t) {
                            dmma(pc[m][t][0], pc[m][t][1], af.x, bf[t].x);
                            dmma(pc[m][t][0], pc[m][t][1], af.y, bf[t].y);
                        }
                        if constexpr (!Lay::DELTA_IN_TILE) pr[m] = fma(af.x, dl.x, fma(af.y, dl.y, pr[m]));
                    }
                }
#endif
                dirty = true;
            }
            team_sync<TW>(bar);                 // every warp has finished reading the chunk
            B200LM_TICK(2);
            // ---- P3: own finished rows [J | r] -> shared (row-major) -> partial normal equations
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                const int mg = tw * MT + m;
                double* dst = Jb + (8 * mg + r) * LDR + 2 * q;
#pragma unroll
                for (int t = 0; t < NT; ++t)
                    *reinterpret_cast<double2*>(dst + 8 * t) = make_double2(pc[m][t][0], pc[m][t][1]);
                if constexpr (!Lay::DELTA_IN_TILE) {
                    double s = pr[m];
                    s += __shfl_xor_sync(B200LM_FULL, s, 1);
                    s += __shfl_xor_sync(B200LM_FULL, s, 2);
                    if (q == 0) Jb[(8 * mg + r) * LDR + NP] = s;
                }
            }
            __syncwarp();
            const int own0 = g0 + tw * RW;
            const int nrows = max(0, min(RW, bd.n_out - own0));
            if (mode == 0) {
                if (nrows > 0) {
                    if (fout || Jout) emit_rows<F>(Jown, nrows, bd.chiv_off + own0, lane, fout, Jout);
                    team_accumulate<F, TW>(Jown, (nrows + 3) & ~3, lane, na);
                }
                __syncwarp();
            } else {
                team_sync<TW>(bar);
                if (tw == 0) {
                    const int nall = min(CH, bd.n_out - g0);
                    if (fout || Jout) emit_rows<F>(Jb, nall, bd.chiv_off + g0, lane, fout, Jout);
                    __syncwarp();
                    qr_update_rows<F>(shared_addr(c.A), shared_addr(c.dsc), shared_addr(Jb), nall, lane);
                }
            }
            dirty = true;
            B200LM_TICK(3);
        }
    }
    if (mode == 0) {
        if constexpr (TL::STAGE_OWN) {
            // the warp's own rows are read by nobody else: they carry its partial sums to the leader
            if (tw != 0) {
                int s = 0;
#pragma unroll
                for (int u = 0; u < Lay::NTRI; ++u) {
                    Jown[(s++) * 32 + lane] = na.t[u][0];
                    Jown[(s++) * 32 + lane] = na.t[u][1];
                }
#pragma unroll
                for (int u = 0; u < TL::NGT; ++u) Jown[(s++) * 32 + lane] = na.g[u][0];
                Jown[(s++) * 32 + lane] = na.cost;
            }
            team_sync<TW>(bar);
            if (tw == 0) {
#pragma unroll
                for (int w = 1; w < TW; ++w) {
                    const double* st = Jb + w * RW * LDR;
                    int s = 0;
#pragma unroll
                    for (int u = 0; u < Lay::NTRI; ++u) {
                        na.t[u][0] += st[(s++) * 32 + lane];
                        na.t[u][1] += st[(s++) * 32 + lane];
                    }
#pragma unroll
                    for (int u = 0; u < TL::NGT; ++u) na.g[u][0] += st[(s++) * 32 + lane];
                    na.cost += st[(s++) * 32 + lane];
                }
                acc += team_flush<F, TW>(c, na);
            }
        } else {
            // partials too large for the staging rows: the leader stores, the others add in turn
#pragma unroll 1
            for (int w = 0; w < TW; ++w) {
                if (tw == w) {
                    if (w == 0) {
                        acc += team_flush<F, TW>(c, na);
                    } else {
                        NormalAcc<F> nb;
                        nb.clear();
#pragma unroll
                        for (int u = 0; u < Lay::NTRI; ++u) { nb.t[u][0] = na.t[u][0]; nb.t[u][1] = na.t[u][1]; }
                        double cw = flush_normal<F>(c, nb) + na.cost;
                        if constexpr (!Lay::DELTA_IN_TILE) {
                            if ((lane & 3) == 0) {
#pragma unroll
                                for (int ta = 0; ta < NT; ++ta) {
                                    const int row = 8 * ta + (lane >> 2);
                                    if (row < NP) c.g[row] += na.g[ta][0];
                                }
                            }
                        }
                        cw = warp_sum(cw);
                        if (lane == 0) c.dvec[w] = cw;
                    }
                }
                team_sync<TW>(bar);
            }
            if (tw == 0 && lane == 0) {
                for (int w = 1; w < TW; ++w) acc += c.dvec[w];
            }
        }
    }
    if (tw == 0 && mode == 0) acc += prior_rows();
    B200LM_TICK(4);
#ifdef B200LM_PHASE_TICKS
    if (tw == 0 && lane == 0 && P.stats) {
#pragma unroll
        for (int i = 0; i < 5; ++i) atomicAdd(&P.stats[6 + i], (unsigned long long)tk[i]);
    }
#endif
#undef B200LM_TICK
#ifdef B200LM_DEBUG_PRINT
    if (lane == 0 && blockIdx.x == 0) printf("eval warp %d tw %d mode %d flags %d ids %x acc %g A00 %g g0 %g base %p A %p\n", threadIdx.x >> 5, tw, mode, flags, ids, acc, c.A[0], c.g[0], (void*)base, (void*)c.A);
#endif
    return tw == 0 ? 0.5 * warp_sum(acc) : 0.0;
}

template <class F, int TW>
__device__ __forceinline__ double team_eval(const WarpCtx<F>& c, int tw, int bar, const double* pv, int mode,
                                            double* fout, double* Jout) {
    const int ids = c.lane | (tw << 8) | (bar << 16);
    const int flags = (mode & 1) | ((pv == c.pn) ? 2 : 0) | ((c.A == c.Abuf[1]) ? 4 : 0);
    const unsigned base_s = shared_addr(c.R);
    const unsigned stage_s = c.P.staged ? shared_addr(c.wt) : 0u;
    return c.P.staged ? team_eval_impl<F, TW, true>(c.P, base_s, stage_s, ids, flags, fout, Jout)
                      : team_eval_impl<F, TW, false>(c.P, base_s, stage_s, ids, flags, fout, Jout);
}

// leader side of fit_one's evaluator: post the command, then take part in the evaluation.  It holds the
// team's command block, means and barrier by value: a pointer to the team context would keep that
// context, and every pointer of the leader's WarpCtx, in local memory.
template <class F, int TW>
struct TeamEval {
    int* cmd;
    double* mean_s;
    int bar;
    int b;
    // stage the means of fit b in the team's shared memory (read by every warp of the team)
    __device__ __forceinline__ const double* begin(WarpCtx<F>& c, const FitParams& P, int b_) {
        b = b_;
        const double* src = P.mean + (size_t)b_ * P.mean_stride;
        for (int i = c.lane; i < P.N; i += 32) mean_s[i] = src[i];
        __syncwarp();
        return mean_s;
    }
    __device__ __forceinline__ double run(WarpCtx<F>& c, const double* pv, double* fout, double* Jout, int mode) {
        if (c.lane == 0) {
            cmd[0] = 1;
            cmd[1] = b;
            cmd[2] = (pv == c.pn) ? 1 : 0;
            cmd[3] = mode;
            cmd[4] = (fout ? 1 : 0) | (Jout ? 2 : 0);
            cmd[5] = (c.A == c.Abuf[1]) ? 1 : 0;
        }
        __syncwarp();
        team_sync<TW>(bar);
        return team_eval<F, TW>(c, 0, bar, pv, mode, fout, Jout);
    }
};

template <class F, int TW>
__global__ void __launch_bounds__(TeamLayout<F, TW>::MAX_THREADS, 1)
fit_team_kernel(const __grid_constant__ FitParams P) {
    typedef FitLayout<F> Lay;
    typedef TeamLayout<F, TW> TL;
    constexpr int NP = Lay::NP, LDA = Lay::LDA;
    static_assert(NP <= 32, "one lane per parameter");
    static_assert(TW == 2 || TW == 4, "team of 2 or 4 warps");
    extern __shared__ __align__(16) double smem[];
    const int warp = threadIdx.x >> 5;
    const int team = warp / TW;
    // leaders run the serial trust-region code: spread them over the four warp schedulers
    constexpr int TEAMS_PER_QUAD = TW >= 4 ? 1 : 4 / TW;
    const int tw = (warp + team / TEAMS_PER_QUAD) % TW;
    TeamCtx<F, TW> tc(P);
    WarpCtx<F>& c = tc.c;
    c.lane = threadIdx.x & 31;
    tc.tw = tw;
    tc.bar = 1 + team;
    int region = 0;
    if (P.staged) {
        const TeamStage st = team_stage(P);
        int* si = reinterpret_cast<int*>(smem + st.ints);
        for (int i = threadIdx.x; i < P.wt2_total; i += blockDim.x) smem[st.wt + i] = P.blk_wt2[i];
        for (int i = threadIdx.x; i < P.ny * P.nx; i += blockDim.x) smem[st.x + i] = P.x[i];
        for (int i = threadIdx.x; i < P.nd_fn; i += blockDim.x) { smem[st.fw + i] = P.dfn_w[i]; si[P.nblk_idx + i] = P.dfn_idx[i]; }
        for (int i = threadIdx.x; i < P.nd_pr; i += blockDim.x) { smem[st.pw + i] = P.dpr_w[i]; si[P.nblk_idx + P.nd_fn + i] = P.dpr_idx[i]; }
        for (int i = threadIdx.x; i < P.nblk_idx; i += blockDim.x) si[i] = P.blk_idx[i];
        region = st.total;
    }
    team_pointers<F, TW>(tc, P, smem + region + (size_t)team * P.team_stride, smem);
    __syncthreads();
    const int lane = c.lane;

    if (tw == 0) {
        unsigned long long tot_nfev = 0, tot_njev = 0, tot_nfac = 0;
        PhaseClock pk;
        pk.clear();
        TeamEval<F, TW> ev;
        ev.cmd = tc.cmd;
        ev.mean_s = tc.mean_s;
        ev.bar = tc.bar;
        for (;;) {
            int b = 0;
            if (lane == 0) {
                b = atomicAdd(P.counter, 1);
                if (P.order && b < P.B) b = P.order[b];
            }
            b = __shfl_sync(B200LM_FULL, b, 0);
            if (b >= P.B) break;
            fit_one<F>(c, ev, P, b, tot_nfev, tot_njev, tot_nfac, pk);
        }
        if (lane == 0) tc.cmd[0] = 0;
        __syncwarp();
        team_sync<TW>(tc.bar);
        if (lane == 0 && P.stats) {
            atomicAdd(&P.stats[0], tot_nfev);
            atomicAdd(&P.stats[1], tot_njev);
            atomicAdd(&P.stats[2], tot_nfac);
            atomicAdd(&P.stats[3], (unsigned long long)pk.eval);
            atomicAdd(&P.stats[4], (unsigned long long)pk.solve);
            atomicAdd(&P.stats[5], (unsigned long long)pk.total);
            atomicAdd(&P.stats[11], (unsigned long long)pk.fact);
        }
    } else {
        for (;;) {
            team_sync<TW>(tc.bar);
            const int op = tc.cmd[0], b = tc.cmd[1], sel = tc.cmd[2], mode = tc.cmd[3], flags = tc.cmd[4];
            const int cur = tc.cmd[5];
            if (op == 0) break;
            c.use_buf(cur);
            double* fout = (flags & 1) ? P.f_out + (size_t)b * P.nchiv : nullptr;
            double* Jout = (flags & 2) ? P.J_out + (size_t)b * P.nchiv * NP : nullptr;
            team_eval<F, TW>(c, tw, tc.bar, sel ? c.pn : c.p, mode, fout, Jout);
        }
    }
}

template <class F, int TW>
size_t team_bytes_of(int N) { return (size_t)TeamLayout<F, TW>::per_team_doubles(N) * sizeof(double); }

template <class F, int TW>
cudaError_t launch_fit_team(FitParams P, int sm_count, size_t smem_budget, cudaStream_t stream) {
    typedef TeamLayout<F, TW> TL;
    const size_t per_team = team_bytes_of<F, TW>(P.N);
    P.team_stride = TL::per_team_doubles(P.N);
    P.staged = 1;
    const size_t stage_bytes = (size_t)team_stage(P).total * sizeof(double);
    if (stage_bytes + 2 * per_team > smem_budget) P.staged = 0;
    const size_t avail = smem_budget - (P.staged ? stage_bytes : 0);
    int teams = (int)(avail / per_team);
    if (teams < 1) return cudaErrorInvalidConfiguration;
    if (teams > TL::MAX_TEAMS) teams = TL::MAX_TEAMS;
    if (const char* env = getenv("B200LM_TEAMS")) {          // tuning knob (profiling only)
        const int t = atoi(env);
        if (t >= 1 && t < teams) teams = t;
    }
    P.warps = teams * TW;
    const size_t smem = (P.staged ? stage_bytes : 0) + teams * per_team;
    int grid = P.B < sm_count ? P.B : sm_count;         // spread small batches over all SMs
    if (grid < 1) grid = 1;
    cudaError_t e = cudaFuncSetAttribute(fit_team_kernel<F, TW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    fit_team_kernel<F, TW><<<grid, teams * TW * 32, smem, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace b200lm
