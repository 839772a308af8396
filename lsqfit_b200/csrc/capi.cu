// C-ABI layer of libb200lm.so: plan objects, functor dispatch, launches.
// Declarations and the reference interfaces they replace: include/b200lm.h.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <deque>
#include <map>
#include <mutex>
#include <algorithm>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdlib.h>
#include "../../include/b200lm.h"
#include "handle.h"

using namespace b200lm;

static thread_local std::string g_err;

namespace b200lm {
int set_error(b200lm_handle_s* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    g_err = msg;
    return code;
}
int cuda_fail(b200lm_handle_s* h, cudaError_t e, const char* what) {
    return set_error(h, B200LM_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
void fill_params(b200lm_handle_s* h, FitParams& P) {
    memset(&P, 0, sizeof(P));
    P.ny = h->ny; P.np = h->np; P.N = h->N; P.nchiv = h->nchiv; P.nx = h->nx; P.noprior = h->noprior;
    P.x = h->d_x;
    if (h->nwin > 0) {
        // the window kernel (fit_kernel<F, 4>) reads each window's counts and offsets from P.win
        h->win_rows.fill(P);
        P.nwin = h->nwin; P.win = h->d_win;
    } else {
        h->rows.fill(P);
    }
    P.rb = h->rb;
    {
        const char* e = getenv("B200LM_DUAL_FROM");
        P.dual_from = e ? atoi(e) : 0;        // measured on C3: 0 -> 700 k fits/s, 12 -> 669 k, never -> 646 k
    }
    P.counter = h->d_counter;
    P.stats = h->d_stats;
    P.policy = h->policy;
}
}  // namespace b200lm

template <class T>
static cudaError_t upload(T** dst, const T* src, size_t n) {
    if (*dst) { cudaFree(*dst); *dst = nullptr; }
    if (n == 0) return cudaSuccess;
    cudaError_t e = cudaMalloc((void**)dst, n * sizeof(T));
    if (e != cudaSuccess) return e;
    return cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
}

namespace b200lm {
void WeightTables::append(const WeightTables& t) {
    for (BlockDesc b : t.blk) {
        b.idx_off += (int)blk_idx.size();
        b.wt_off += (int)wt.size();
        blk.push_back(b);
    }
    fn_idx.insert(fn_idx.end(), t.fn_idx.begin(), t.fn_idx.end());
    fn_w.insert(fn_w.end(), t.fn_w.begin(), t.fn_w.end());
    pr_idx.insert(pr_idx.end(), t.pr_idx.begin(), t.pr_idx.end());
    pr_w.insert(pr_w.end(), t.pr_w.begin(), t.pr_w.end());
    blk_idx.insert(blk_idx.end(), t.blk_idx.begin(), t.blk_idx.end());
    wt.insert(wt.end(), t.wt.begin(), t.wt.end());
}

cudaError_t RowTables::upload() {
    cudaError_t e = cudaSuccess;
    auto put = [&e](auto** dst, const auto& v) { if (e == cudaSuccess) e = ::upload(dst, v.data(), v.size()); };
    put(&d_fn_idx, host.fn_idx); put(&d_fn_w, host.fn_w);
    put(&d_pr_idx, host.pr_idx); put(&d_pr_w, host.pr_w);
    put(&d_blk, host.blk); put(&d_blk_idx, host.blk_idx);
    put(&d_wt, host.wt); put(&d_wt2, host.wt2);
    return e;
}

void RowTables::free() {
    cudaFree(d_fn_idx); cudaFree(d_fn_w); cudaFree(d_pr_idx); cudaFree(d_pr_w);
    cudaFree(d_blk); cudaFree(d_blk_idx); cudaFree(d_wt); cudaFree(d_wt2);
}

void RowTables::fill(FitParams& P) const {
    P.nd_fn = (int)host.fn_idx.size(); P.dfn_idx = d_fn_idx; P.dfn_w = d_fn_w;
    P.nd_pr = (int)host.pr_idx.size(); P.dpr_idx = d_pr_idx; P.dpr_w = d_pr_w;
    P.nblk = (int)host.blk.size(); P.blk = d_blk;
    P.blk_idx = d_blk_idx; P.nblk_idx = (int)host.blk_idx.size();
    P.blk_wt = d_wt; P.wt_total = (int)host.wt.size();
    P.blk_wt2 = d_wt2; P.wt2_total = (int)host.wt2.size();
}
}  // namespace b200lm


// The registry: the built-in tables in a fixed order, then the entries of run-time plug-ins (b200lm_load_functors) in
// load order.  A deque: handles keep pointers to their entry, and appending must not move the others.  Every read
// and every append holds g_registry_mu.
static std::mutex g_registry_mu;

static std::deque<FunctorEntry>& registry() {
    static std::deque<FunctorEntry> r = [] {
        std::deque<FunctorEntry> d;
        const FunctorEntry* (*tables[])(int*) = {registry_multiexp, registry_multiexp_b, registry_nist_a,
                                                  registry_nist_b, registry_misc, registry_misc_b, registry_poly_b};
        for (auto t : tables) {
            int n = 0;
            const FunctorEntry* e = t(&n);
            d.insert(d.end(), e, e + n);
        }
        return d;
    }();
    return r;
}

// default number of warps per fit.  The choice depends on the problem's shape only, never on the batch
// size: a fit's result must not depend on how many other fits share its launch (the kernels sum in a different
// order), so that a bootstrap copy gives the same bits in a batch of 500, of 10^4, or in the shard of a multi-GPU job.
// Measured on C3 (np = 16, one 64 x 64 block), ms per batch for one warp / team of 2 / team of 4 / wave kernel
// (tools/team_order_sweep.py, and the mean over eight different batches of tools/order_seeds.py at B = 10^4):
//     B = 1000:  8.0 /  5.6 /  5.1 / 11.7        B = 10^4:   13.2 / 11.7 / 12.7 /  -
//     B = 2048:  8.4 /  6.2 /  5.5 / 11.7        B = 4 10^4: 37.0 / 36.8 / 42.8 / 34.7
//     B = 5000: 10.0 /  8.3 /  8.6 / 12.3        B = 1.6 10^5: 125 /  -  / 160  / 87
// Four warps give the shortest trial point (batches of a few fits per team), one warp the most fits in flight
// (saturated batches); TWO warps per fit are within 10 % of the best warp-per-fit choice everywhere and the best from
// ~5000 fits up to saturation, which is where the reference's bootstrap sizes sit (10^3 ... 10^4 copies) -- the default.
// For small np (C4: np = 6) the evaluation is too short to split.  b200lm_set_team overrides (32 = wave kernel).
static int default_team(b200lm_handle_s* h) {
    if (h->team_request > 0) return h->team_request;
    int big = 0;
    for (const auto& b : h->rows.host.blk) big = b.n_in > big ? b.n_in : big;
    if (big >= 32 && h->np >= 12) return h->fe->fit_team[0] ? 2 : 4;
    return 1;
}

// ---- queue order ------------------------------------------------------------------------------------------------
// A batch whose fits need very different numbers of trial points (C3: median 19, 1 % above 117, longest 379) ends when
// its slowest fit ends, and with the queue in input order that fit may START late.  Measured on the C3 batch of 10^4
// copies (tools/order_probe.py, team of four warps): input order 12.34 ms, longest fit first with the evaluation counts
// known in advance 9.39 ms (the best any order can do), ordered by chi2 at the start point -- the one thing known
// before the fit, at the price of one evaluation per fit -- 11.58 ms ON THAT BATCH (see order_wanted below for the
// average over batches).  The order is a permutation of the work queue only: every fit is computed exactly as before.
//   rank[b] = #{ j : key[j] > key[b]  or  key[j] == key[b] and j < b },  order[rank[b]] = b      (O(B^2), B <= 40000)
static const int ORDER_MAX_B = 40000;
__global__ void __launch_bounds__(256) queue_order_kernel(int B, const double* __restrict__ key, int* __restrict__ order) {
    __shared__ double tile[1024];
    const int b = blockIdx.x * 256 + threadIdx.x;
    double kb = b < B ? key[b] : 0.0;
    if (!(kb == kb) || kb > 1e300) kb = 1e300;                 // non-finite start: first (it ends at once)
    int rank = 0;
    for (int j0 = 0; j0 < B; j0 += 1024) {
        __syncthreads();
        for (int t = threadIdx.x; t < 1024; t += 256) {
            double k = j0 + t < B ? key[j0 + t] : 0.0;
            if (!(k == k) || k > 1e300) k = 1e300;
            tile[t] = k;
        }
        __syncthreads();
        const int n = B - j0 < 1024 ? B - j0 : 1024;
        for (int t = 0; t < n; ++t) {
            const double k = tile[t];
            rank += (k > kb || (k == kb && j0 + t < b)) ? 1 : 0;
        }
    }
    if (b < B) order[rank] = b;
}

// OFF by default: over eight different C3 batches of 10^4 copies (tools/order_seeds.py) the ordered queue changes the
// mean batch time by +0.6 % (team of four), +2.3 % (team of two), +2.3 % (one warp) -- single batches move by -10 % ...
// +11 % depending on where their long fits happen to sit in the input order, and the start-point chi2 is too weak a
// predictor (rank correlation 0.18 with the evaluation count) to pay for its own pass on average.  On request:
// b200lm_set_order(h, 1) or B200LM_ORDER=1.
static bool order_wanted(b200lm_handle_s* h, int B) {
    if (h->nwin > 0 || B > ORDER_MAX_B || B < 2) return false;
    if (const char* env = getenv("B200LM_ORDER")) return atoi(env) != 0;
    return h->order_request == 1;
}

// shapes the wave kernel takes (lm_wave.cuh): one correlated block of <= 64 points, every other entry a 1x1 prior
// row, np <= 16, the scipy policy
static bool wave_ok(b200lm_handle_s* h) {
    const WeightTables& t = h->rows.host;
    if (!h->fe->fit_wave || h->policy != 0 || h->np > 16 || t.blk.size() != 1 || !t.fn_idx.empty()) return false;
    const auto& b = t.blk[0];
    if (b.n_in > 64 || b.n_out > 64 || b.n_out < 1) return false;
    return h->fe->wave_bytes((int)t.wt.size()) <= h->smem_budget;
}

// The warps per fit of a batch: 1 (fit_kernel), 2 or 4 (fit_team_kernel) or 32 (the wave kernel).  Windows run in
// the one-warp kernel (fit_kernel<F, 4>), and so do the GSL decisions and the bounded scipy decisions (fit_kernel<F, 1>
// and <F, 3>).  Otherwise B200LM_TEAM = 0/1, 2, 4, 32 overrides default_team, and a team that the functor or the
// shapes do not allow falls back to one warp.
static int kernel_team(b200lm_handle_s* h) {
    if (h->nwin > 0 || h->policy == 1 || h->bounded) return 1;
    int team = default_team(h);
    if (const char* env = getenv("B200LM_TEAM")) team = atoi(env);
    if (team == 32) return wave_ok(h) ? 32 : 1;
    const int ti = team == 4 ? 1 : (team == 2 ? 0 : -1);
    return ti >= 0 && h->fe->fit_team[ti] && h->fe->team_bytes[ti](h->N) <= h->smem_budget ? team : 1;
}

#define CUDA_TRY(h, call, what) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(h, e_, what); } while (0)

// One whitening description (the arguments of b200lm_set_weights), checked and laid out for the kernels.
// allowed[i]: 0 = entry i of y(+)prior must not appear, 1 = may appear, 2 = must appear; each appears at most once.
// Returns "" or the error ("size": a block too large for the shared-memory plan).

static std::string parse_weights(b200lm_handle_s* h, const std::vector<char>& allowed, int ndiag, const int* diag_idx,
                                 const double* diag_w, int nblk, const int* blk_nin, const int* blk_nout,
                                 const int* blk_idx, const double* blk_w, WeightTables& t) {
    if (ndiag < 0 || nblk < 0 || (ndiag > 0 && (!diag_idx || !diag_w)) ||
        (nblk > 0 && (!blk_nin || !blk_nout || !blk_idx || !blk_w)))
        return "bad weight description";
    const int N = h->N;
    std::vector<char> seen(N, 0);
    auto take = [&](int idx) {
        if (idx < 0 || idx >= N || seen[idx] || !allowed[idx]) return false;
        seen[idx] = 1;
        if (idx < h->ny) ++t.ndata;
        return true;
    };
    // 1x1 blocks: data rows first (in the given order), then prior rows -- this is the
    // reference's chiv order because gvar lists 1x1 indices in ascending order.
    bool prior_seen = false;
    for (int i = 0; i < ndiag; ++i) {
        const int idx = diag_idx[i];
        if (!take(idx)) return "diag index out of range or repeated";
        if (idx < h->ny) {
            if (prior_seen) return "diag indices must list data rows before prior rows";
            t.fn_idx.push_back(idx); t.fn_w.push_back(diag_w[i]);
        } else { prior_seen = true; t.pr_idx.push_back(idx); t.pr_w.push_back(diag_w[i]); }
    }
    t.blk.resize(nblk);
    int idx_off = 0, chiv_off = ndiag;
    for (int k = 0; k < nblk; ++k) {
        const int nin = blk_nin[k], nout = blk_nout[k];
        if (nin <= 0 || nout < 0 || nout > nin) return "bad block shape";
        for (int j = 0; j < nin; ++j)
            if (!take(blk_idx[idx_off + j])) return "block index out of range or repeated";
        BlockDesc& b = t.blk[k];
        b.n_in = nin; b.n_out = nout;
        // row-major [n_out padded to 8][ldw], zero padded; ldw == 4 (mod 16) >= n_in rounded to 4
        // keeps the DMMA A-fragment loads at the minimum of two shared-memory wavefronts
        int ldw = (nin + 3) & ~3;
        while ((ldw & 15) != 4) ldw += 4;
        b.ldw = ldw;
        const int nout8 = ((nout + 7) & ~7) > 0 ? ((nout + 7) & ~7) : 8;
        b.idx_off = idx_off; b.wt_off = (int)t.wt.size(); b.chiv_off = chiv_off;
        t.wt.resize(t.wt.size() + (size_t)nout8 * ldw, 0.0);
        for (int r = 0; r < nout; ++r)
            for (int j = 0; j < nin; ++j)
                t.wt[b.wt_off + (size_t)r * ldw + j] = blk_w[t.nw + (size_t)r * nin + j];
        // team-kernel copy: 16-byte fragment loads want a row stride == 8 (mod 16) >= n_in rounded to 8
        int ldw2 = (nin + 7) & ~7;
        while ((ldw2 & 15) != 8) ldw2 += 8;
        b.ldw2 = ldw2; b.wt2_off = (int)t.wt2.size();
        const int nout64 = ((nout + 63) & ~63) > 0 ? ((nout + 63) & ~63) : 64;     // whole 64-row groups: no row guards
        t.wt2.resize(t.wt2.size() + (size_t)nout64 * ldw2, 0.0);
        for (int r = 0; r < nout; ++r)
            for (int j = 0; j < nin; ++j)
                t.wt2[b.wt2_off + (size_t)r * ldw2 + j] = blk_w[t.nw + (size_t)r * nin + j];
        idx_off += nin; t.nw += (long long)nin * nout; chiv_off += nout;
    }
    t.blk_idx.assign(blk_idx, blk_idx + idx_off);
    for (int i = 0; i < N; ++i)
        if (allowed[i] == 2 && !seen[i])
            return i >= h->ny ? "every prior entry must appear in exactly one block"
                              : "every y(+)prior entry must appear in exactly one block";
    // does at least one warp fit?
    if (h->fe->per_warp_bytes(32) + (size_t)(chiv_off - ndiag + 2) * sizeof(double) > h->smem_budget) return "size";
    t.nchiv = chiv_off;
    return "";
}

extern "C" {

int b200lm_version(void) { return B200LM_VERSION; }

const char* b200lm_last_error(b200lm_handle h) { return h ? h->err.c_str() : g_err.c_str(); }

int b200lm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int b200lm_functor_count(void) {
    std::lock_guard<std::mutex> lock(g_registry_mu);
    return (int)registry().size();
}

int b200lm_functor_info(int i, int* family, int* np, int* nx, const char** name) {
    std::lock_guard<std::mutex> lock(g_registry_mu);
    auto& r = registry();
    if (i < 0 || i >= (int)r.size()) return set_error(nullptr, B200LM_EINVAL, "functor index out of range");
    if (family) *family = r[i].family;
    if (np) *np = r[i].np;
    if (nx) *nx = r[i].nx;
    if (name) *name = r[i].name;
    return B200LM_OK;
}

int b200lm_functor_family(const char* name) {
    if (!name) return B200LM_EINVAL;
    std::lock_guard<std::mutex> lock(g_registry_mu);
    for (auto& e : registry()) if (strcmp(e.name, name) == 0) return e.family;
    return set_error(nullptr, B200LM_ENOFUNCTOR, std::string("unknown functor family: ") + name);
}

#ifndef B200LM_HEADERS_DIGEST
#error "B200LM_HEADERS_DIGEST must be defined (lsqfit_b200/build.py passes the digest of the headers and flags)"
#endif

int b200lm_load_functors(const char* path, int* family_out) {
    if (!path || !family_out) return set_error(nullptr, B200LM_EINVAL, "NULL argument");
    const std::string where = std::string("functor plug-in ") + path + ": ";
    // never dlclose'd: plans created on its entries hold its launchers
    void* so = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!so) {
        const char* m = dlerror();
        return set_error(nullptr, B200LM_EINVAL, where + (m ? m : "dlopen failed"));
    }
    auto entries_fn = (b200lm_plugin_entries_fn)dlsym(so, "b200lm_plugin_entries");
    if (!entries_fn) return set_error(nullptr, B200LM_EINVAL, where + "no symbol b200lm_plugin_entries");
    b200lm_plugin_abi abi;
    memset(&abi, 0, sizeof abi);
    const FunctorEntry* e = nullptr;
    int n = 0;
    if (entries_fn(&e, &n, &abi) != 0 || !e || n < 1) return set_error(nullptr, B200LM_EINVAL, where + "no entries");
    abi.headers[sizeof abi.headers - 1] = 0;
    abi.model[sizeof abi.model - 1] = 0;
    auto mismatch = [&](const char* field, const std::string& got, const std::string& want) {
        return set_error(nullptr, B200LM_EINVAL, where + "ABI mismatch in " + field + ": plug-in " + got +
                                                 ", library " + want + " (rebuild the plug-in)");
    };
    if (abi.version != B200LM_VERSION)
        return mismatch("version", std::to_string(abi.version), std::to_string(B200LM_VERSION));
    if (abi.fitparams_size != (int)sizeof(FitParams))
        return mismatch("fitparams_size", std::to_string(abi.fitparams_size), std::to_string(sizeof(FitParams)));
    if (abi.entry_size != (int)sizeof(FunctorEntry))
        return mismatch("entry_size", std::to_string(abi.entry_size), std::to_string(sizeof(FunctorEntry)));
    if (strcmp(abi.headers, B200LM_HEADERS_DIGEST) != 0) return mismatch("headers", abi.headers, B200LM_HEADERS_DIGEST);
    if (!e[0].name || !e[0].name[0] || strlen(e[0].name) > 64)
        return set_error(nullptr, B200LM_EINVAL, where + "bad model name");
    const std::string name = e[0].name;
    for (int i = 0; i < n; ++i) {
        const FunctorEntry& f = e[i];
        char buf[160];
        snprintf(buf, sizeof buf, "entry %d (np=%d, nx=%d): ", i, f.np, f.nx);
        if (!f.name || name != f.name) return set_error(nullptr, B200LM_EINVAL, where + buf + "one model name per plug-in");
        if (f.np < 1 || f.np > B200LM_USER_MAX_NP || f.nx < 1 || f.nx > B200LM_USER_MAX_NX)
            return set_error(nullptr, B200LM_EINVAL, where + buf + "np must be in 1..25 and nx in 1..8");
        if (!f.fit || !f.resjac || !f.per_warp_bytes || !f.model_rows)
            return set_error(nullptr, B200LM_EINVAL, where + buf + "missing launcher");
        for (int j = 0; j < i; ++j)
            if (e[j].np == f.np) return set_error(nullptr, B200LM_EINVAL, where + buf + "np listed twice");
    }
    // name -> (family, model digest) of every plug-in loaded so far; names of plug-in entries are owned here
    static std::map<std::string, std::pair<int, std::string>> loaded;
    static std::deque<std::string> names;
    std::lock_guard<std::mutex> lock(g_registry_mu);
    auto& r = registry();
    auto it = loaded.find(name);
    if (it != loaded.end()) {
        if (it->second.second != abi.model)
            return set_error(nullptr, B200LM_EINVAL, where + "the name '" + name + "' is used by a different plug-in");
        *family_out = it->second.first;
        return B200LM_OK;
    }
    for (const auto& f : r)
        if (name == f.name) return set_error(nullptr, B200LM_EINVAL, where + "the name '" + name + "' is a built-in functor");
    const int family = B200LM_USER_FAMILY0 + (int)loaded.size();
    names.push_back(name);
    for (int i = 0; i < n; ++i) {
        FunctorEntry f = e[i];
        f.family = family;
        f.name = names.back().c_str();
        r.push_back(f);
    }
    loaded[name] = std::make_pair(family, std::string(abi.model));
    *family_out = family;
    return B200LM_OK;
}

int b200lm_create(int family, int ny, int np, int nx, int noprior, int device, b200lm_handle* out) {
    if (!out) return set_error(nullptr, B200LM_EINVAL, "out is NULL");
    *out = nullptr;
    if (ny <= 0 || np <= 0) return set_error(nullptr, B200LM_EINVAL, "ny and np must be positive");
    const FunctorEntry* fe = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_registry_mu);
        for (auto& e : registry()) if (e.family == family && e.np == np) { fe = &e; break; }
    }
    if (!fe) {
        char buf[128];
        snprintf(buf, sizeof buf, "no device functor for family %d with np=%d", family, np);
        return set_error(nullptr, B200LM_ENOFUNCTOR, buf);
    }
    if (nx != fe->nx) return set_error(nullptr, B200LM_EINVAL, "nx does not match the functor");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(nullptr, B200LM_ECUDA, "no CUDA device available (this engine has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return set_error(nullptr, B200LM_EINVAL, "bad device index");
    CUDA_TRY(nullptr, cudaSetDevice(device), "cudaSetDevice");
    b200lm_handle_s* h = new b200lm_handle_s();
    h->device = device; h->fe = fe; h->ny = ny; h->np = np; h->nx = nx; h->noprior = noprior ? 1 : 0;
    h->N = noprior ? ny : ny + np;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { delete h; return cuda_fail(nullptr, e, "cudaGetDeviceProperties"); }
    h->sm_count = prop.multiProcessorCount;
    h->smem_budget = prop.sharedMemPerBlockOptin;
    e = cudaMalloc((void**)&h->d_counter, sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void**)&h->d_stats, 16 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { b200lm_destroy(h); return cuda_fail(nullptr, e, "handle allocation"); }
    *out = h;
    return B200LM_OK;
}

void b200lm_destroy(b200lm_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaFree(h->d_x);
    h->rows.free(); h->win_rows.free(); cudaFree(h->d_win); cudaFree(h->d_wfull);
    cudaFree(h->d_counter); cudaFree(h->d_stats); cudaFree(h->d_stage); cudaFree(h->d_scratch);
    cudaFree(h->d_order_key); cudaFree(h->d_order); cudaFree(h->d_wave_A);
    cudaFree(h->d_lb); cudaFree(h->d_ub);
    if (h->h_pinned) cudaFreeHost(h->h_pinned);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
}

int b200lm_set_const(b200lm_handle h, const double* h_x, int n) {
    if (!h || !h_x) return set_error(h, B200LM_EINVAL, "NULL argument");
    if (n != h->ny * h->nx) return set_error(h, B200LM_EINVAL, "x must have ny*nx entries");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    CUDA_TRY(h, upload(&h->d_x, h_x, (size_t)n), "upload x");
    h->have_const = true;
    return B200LM_OK;
}

int b200lm_set_weights(b200lm_handle h, int ndiag, const int* diag_idx, const double* diag_w,
                       int nblk, const int* blk_nin, const int* blk_nout,
                       const int* blk_idx, const double* blk_w) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    WeightTables t;
    const std::string err = parse_weights(h, std::vector<char>(h->N, 2), ndiag, diag_idx, diag_w, nblk, blk_nin,
                                          blk_nout, blk_idx, blk_w, t);
    if (!err.empty()) return set_error(h, err == "size" ? B200LM_ESIZE : B200LM_EINVAL,
                                       err == "size" ? "correlated block too large for the per-warp shared-memory plan"
                                                     : err);
    h->rows.host = std::move(t);
    CUDA_TRY(h, h->rows.upload(), "upload weights");
    h->rb = 32; h->nchiv = h->rows.host.nchiv;
    if (h->d_wfull) { cudaFree(h->d_wfull); h->d_wfull = nullptr; }
    h->have_weights = true;
    h->nwin = 0;
    return B200LM_OK;
}

int b200lm_set_windows(b200lm_handle h, int nwin, const int* ndiag, const int* diag_idx, const double* diag_w,
                       const int* nblk, const int* blk_nin, const int* blk_nout, const int* blk_idx,
                       const double* blk_w) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (nwin < 1 || !ndiag || !nblk) return set_error(h, B200LM_EINVAL, "bad window description");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    // a window lists every prior entry and its own data rows exactly once
    std::vector<char> allowed(h->N, 2);
    for (int i = 0; i < h->ny; ++i) allowed[i] = 1;
    WeightTables all;
    std::vector<WinDesc> win(nwin);
    std::vector<int> nchiv(nwin);
    long long o_diag = 0, o_blk = 0, o_idx = 0, o_w = 0;
    for (int w = 0; w < nwin; ++w) {
        const std::string where = "window " + std::to_string(w) + ": ";
        WeightTables t;
        const std::string err = parse_weights(h, allowed, ndiag[w], diag_idx ? diag_idx + o_diag : nullptr,
                                              diag_w ? diag_w + o_diag : nullptr, nblk[w],
                                              blk_nin ? blk_nin + o_blk : nullptr, blk_nout ? blk_nout + o_blk : nullptr,
                                              blk_idx ? blk_idx + o_idx : nullptr, blk_w ? blk_w + o_w : nullptr, t);
        if (!err.empty()) return set_error(h, err == "size" ? B200LM_ESIZE : B200LM_EINVAL,
                                           where + (err == "size" ? "correlated block too large for the per-warp "
                                                                    "shared-memory plan" : err));
        if (t.ndata == 0) return set_error(h, B200LM_EINVAL, where + "no data row");
        WinDesc& d = win[w];
        d.nd_fn = (int)t.fn_idx.size(); d.nd_pr = (int)t.pr_idx.size(); d.nblk = nblk[w]; d.nchiv = t.nchiv;
        d.dfn_off = (int)all.fn_idx.size(); d.dpr_off = (int)all.pr_idx.size(); d.blk_off = (int)all.blk.size();
        all.append(t);
        nchiv[w] = t.nchiv;
        o_diag += ndiag[w]; o_blk += nblk[w]; o_idx += (long long)t.blk_idx.size(); o_w += t.nw;
    }
    CUDA_TRY(h, upload(&h->d_win, win.data(), win.size()), "upload windows");
    h->win_rows.host = std::move(all);
    CUDA_TRY(h, h->win_rows.upload(), "upload windows");
    h->nwin = nwin;
    h->win_nchiv = nchiv;
    h->nchiv = *std::max_element(nchiv.begin(), nchiv.end());
    h->rb = 32;
    return B200LM_OK;
}

int b200lm_window_nchiv(b200lm_handle h, int* h_nchiv) {
    if (!h || !h_nchiv) return set_error(h, B200LM_EINVAL, "NULL argument");
    if (h->nwin == 0) return set_error(h, B200LM_EINVAL, "no windows set (b200lm_set_windows)");
    for (int w = 0; w < h->nwin; ++w) h_nchiv[w] = h->win_nchiv[w];
    return B200LM_OK;
}

int b200lm_nchiv(b200lm_handle h) { return h ? h->nchiv : B200LM_EINVAL; }

// what a batch on fit windows does not combine with
static int window_refusal(b200lm_handle h, int B) {
    if (h->nwin == 0) return B200LM_OK;
    if (B % h->nwin != 0)
        return set_error(h, B200LM_EINVAL, "with windows set, B must be a multiple of the number of windows");
    if (h->policy == 1) return set_error(h, B200LM_EINVAL, "the GSL policy is not built for window scans");
    if (h->bounded) return set_error(h, B200LM_EINVAL, "bounds are not built for window scans");
    return B200LM_OK;
}

static int check_ready(b200lm_handle h) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (!h->have_weights && h->nwin == 0) return set_error(h, B200LM_EINVAL, "b200lm_set_weights has not been called");
    if (!h->have_const) return set_error(h, B200LM_EINVAL, "b200lm_set_const has not been called");
    return B200LM_OK;
}

int b200lm_fit_batch(b200lm_handle h, int B,
                     const double* d_mean, long long mean_stride,
                     const double* d_p0, long long p0_stride,
                     double xtol, double gtol, double ftol, int maxit, int scaler, int polish,
                     double* d_x, double* d_chi2, double* d_cov, double* d_logdet,
                     int* d_nit, int* d_status, double* d_f, double* d_J, void* stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (B == 0) return B200LM_OK;                 // empty batch: nothing to read or write
    if (B < 0 || !d_mean || !d_p0 || !d_x || !d_chi2 || !d_nit || !d_status)
        return set_error(h, B200LM_EINVAL, "NULL required argument");
    if ((mean_stride != 0 && mean_stride < h->N) || (p0_stride != 0 && p0_stride < h->np))
        return set_error(h, B200LM_EINVAL, "bad stride");
    if (scaler != 0 && scaler != 1 && !(scaler == 2 && h->policy == 1))
        return set_error(h, B200LM_EINVAL, "scaler must be 0 (levenberg), 1 (more) or, with the GSL policy, 2 (marquardt)");
    if (maxit < 1) return set_error(h, B200LM_EINVAL, "maxit must be >= 1");
    if (h->bounded && h->policy == 1)
        return set_error(h, B200LM_EINVAL, "bounds need the scipy trf policy (GSL's lm has no bound constraints)");
    rc = window_refusal(h, B);
    if (rc) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    cudaStream_t s = (cudaStream_t)stream;
    FitParams P;
    fill_params(h, P);
    P.B = B; P.mean = d_mean; P.mean_stride = mean_stride; P.p0 = d_p0; P.p0_stride = p0_stride;
    P.xtol = xtol; P.gtol = gtol; P.ftol = ftol; P.maxit = maxit; P.scaler = scaler; P.polish = polish < 0 ? 0 : polish;
    P.x_out = d_x; P.chi2 = d_chi2; P.cov = d_cov; P.logdet = d_logdet; P.nit = d_nit; P.status = d_status;
    P.f_out = d_f; P.J_out = d_J;
    if (h->bounded) { P.bounded = 1; P.lb = h->d_lb; P.ub = h->d_ub; }
    if (h->nwin > 0) P.win_copies = B / h->nwin;
    CUDA_TRY(h, cudaMemsetAsync(h->d_counter, 0, sizeof(int), s), "reset work queue");
    CUDA_TRY(h, cudaMemsetAsync(h->d_stats, 0, 16 * sizeof(unsigned long long), s), "reset stats");
    // queue order: chi2 at the start point of every fit (one evaluation each, resjac kernel without f / J outputs),
    // ranked on the device
    h->last_order = 0;
    if (order_wanted(h, B)) {
        if (B > h->order_cap) {
            if (h->d_order_key) cudaFree(h->d_order_key);
            if (h->d_order) cudaFree(h->d_order);
            h->d_order_key = nullptr; h->d_order = nullptr; h->order_cap = 0;
            CUDA_TRY(h, cudaMalloc((void**)&h->d_order_key, (size_t)B * sizeof(double)), "queue order buffers");
            CUDA_TRY(h, cudaMalloc((void**)&h->d_order, (size_t)B * sizeof(int)), "queue order buffers");
            h->order_cap = B;
        }
        FitParams R = P;
        R.f_out = nullptr; R.J_out = nullptr; R.chi2 = h->d_order_key; R.x_out = nullptr; R.cov = nullptr;
        CUDA_TRY(h, h->fe->resjac(R, h->sm_count, h->smem_budget, s), "start-point chi2 launch");
        queue_order_kernel<<<(B + 255) / 256, 256, 0, s>>>(B, h->d_order_key, h->d_order);
        CUDA_TRY(h, cudaGetLastError(), "queue order launch");
        P.order = h->d_order;
        h->last_order = 1;
        h->launches += 2;
    }
    P.team = kernel_team(h);
    if (P.team == 32) {
        // wave kernel: the trust-region loops of 32 fits per CTA in lock step, then covariance / log det / f / J
        // (and polish) of every fit by the one-warp kernel in finalize_only mode.
        // J^T J at every solution goes to the finalisation pass (np(np+1)/2 doubles per fit; skipped above 2 GB,
        // the pass then evaluates the model once more as it did before)
        const size_t need = (size_t)B * (size_t)(h->np * (h->np + 1) / 2);
        if (need * sizeof(double) <= ((size_t)2 << 30) && !getenv("B200LM_WAVE_REEVAL")) {
            if (need > h->wave_A_cap) {
                if (h->d_wave_A) cudaFree(h->d_wave_A);
                h->d_wave_A = nullptr; h->wave_A_cap = 0;
                if (cudaMalloc((void**)&h->d_wave_A, need * sizeof(double)) == cudaSuccess) h->wave_A_cap = need;
                else cudaGetLastError();
            }
            P.wave_A = h->wave_A_cap >= need ? h->d_wave_A : nullptr;
        }
        CUDA_TRY(h, h->fe->fit_wave(P, h->sm_count, h->smem_budget, s), "wave kernel launch");
        CUDA_TRY(h, cudaMemsetAsync(h->d_counter, 0, sizeof(int), s), "reset work queue");
        FitParams Q = P;
        Q.finalize_only = 1; Q.p0 = d_x; Q.p0_stride = h->np; Q.team = 1; Q.order = nullptr;
        CUDA_TRY(h, h->fe->fit(Q, h->sm_count, h->smem_budget, s), "finalize kernel launch");
        h->launches += 1;
    } else if (P.team > 1) {
        CUDA_TRY(h, h->fe->fit_team[P.team == 4 ? 1 : 0](P, h->sm_count, h->smem_budget, s), "fit kernel launch");
    } else {
        CUDA_TRY(h, h->fe->fit(P, h->sm_count, h->smem_budget, s), h->nwin ? "window fit kernel launch" : "fit kernel launch");
    }
    h->last_team = P.team;
    h->last_stream = s;
    h->launches += 1;
    return B200LM_OK;
}

int b200lm_last_stats(b200lm_handle h, unsigned long long out[3]) {
    if (!h || !out) return set_error(h, B200LM_EINVAL, "NULL argument");
    unsigned long long tmp[16];
    int rc = b200lm_last_stats_ex(h, tmp, 16);
    if (rc) return rc;
    out[0] = tmp[0]; out[1] = tmp[1]; out[2] = tmp[2];
    return B200LM_OK;
}

int b200lm_last_stats_ex(b200lm_handle h, unsigned long long* out, int n) {
    if (!h || !out || n < 1 || n > 16) return set_error(h, B200LM_EINVAL, "bad argument");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    CUDA_TRY(h, cudaStreamSynchronize(h->last_stream), "stream sync");
    unsigned long long tmp[16];
    CUDA_TRY(h, cudaMemcpy(tmp, h->d_stats, sizeof tmp, cudaMemcpyDeviceToHost), "read stats");
    for (int i = 0; i < n; ++i) out[i] = tmp[i];
    return B200LM_OK;
}

int b200lm_last_team(b200lm_handle h) { return h ? h->last_team : B200LM_EINVAL; }

int b200lm_set_team(b200lm_handle h, int team) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (team != 0 && team != 1 && team != 2 && team != 4 && team != 32)
        return set_error(h, B200LM_EINVAL, "team must be 0 (default), 1, 2, 4 or 32 (wave kernel)");
    h->team_request = team;
    return B200LM_OK;
}

int b200lm_set_order(b200lm_handle h, int mode) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (mode < -1 || mode > 1) return set_error(h, B200LM_EINVAL, "order must be -1 (default), 0 (input order) or 1 (by start-point chi2)");
    h->order_request = mode;
    return B200LM_OK;
}

int b200lm_last_order(b200lm_handle h) { return h ? h->last_order : B200LM_EINVAL; }

int b200lm_set_bounds(b200lm_handle h, const double* h_lb, const double* h_ub) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (!h_lb != !h_ub) return set_error(h, B200LM_EINVAL, "give both bounds or neither");
    bool finite = false;
    if (h_lb) {
        for (int j = 0; j < h->np; ++j) {
            if (h_lb[j] != h_lb[j] || h_ub[j] != h_ub[j]) return set_error(h, B200LM_EINVAL, "bounds must not be NaN");
            if (!(h_lb[j] < h_ub[j]))
                return set_error(h, B200LM_EINVAL, "Each lower bound must be strictly less than each upper bound.");
            finite = finite || h_lb[j] > -INFINITY || h_ub[j] < INFINITY;
        }
    }
    if (!finite) {                               // no bounds, or all infinite: scipy's unbounded trf
        h->bounded = false;
        h->h_lb.clear(); h->h_ub.clear();
        return B200LM_OK;
    }
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    CUDA_TRY(h, upload(&h->d_lb, h_lb, (size_t)h->np), "upload bounds");
    CUDA_TRY(h, upload(&h->d_ub, h_ub, (size_t)h->np), "upload bounds");
    h->h_lb.assign(h_lb, h_lb + h->np); h->h_ub.assign(h_ub, h_ub + h->np);
    h->bounded = true;
    return B200LM_OK;
}

int b200lm_set_policy(b200lm_handle h, int policy) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (policy != 0 && policy != 1) return set_error(h, B200LM_EINVAL, "policy must be 0 (scipy trf) or 1 (gsl lm)");
    h->policy = policy;
    return B200LM_OK;
}

// ---- single-fit row kernels (lm_rows.cuh) -------------------------------------------------------------------
int b200lm_model_rows(b200lm_handle h, const double* d_p, const double* d_y, double* d_G, int ld, double* d_delta,
                      void* stream) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (!h->have_const) return set_error(h, B200LM_EINVAL, "b200lm_set_const has not been called");
    if (!d_p || !d_y || !d_delta || (d_G && ld < h->np)) return set_error(h, B200LM_EINVAL, "bad model_rows argument");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    CUDA_TRY(h, h->fe->model_rows(h->ny, h->nx, h->d_x, d_p, d_y, d_G, ld, d_delta, h->sm_count, (cudaStream_t)stream),
             "model_rows kernel launch");
    h->last_stream = (cudaStream_t)stream;
    h->launches += 1;
    return B200LM_OK;
}

int b200lm_normal_diag(b200lm_handle h, const double* d_p, const double* d_y, const double* d_w, double* d_out,
                       void* stream) {
    if (!h) return set_error(h, B200LM_EINVAL, "NULL handle");
    if (!h->have_const) return set_error(h, B200LM_EINVAL, "b200lm_set_const has not been called");
    if (!d_p || !d_y || !d_w || !d_out) return set_error(h, B200LM_EINVAL, "NULL argument");
    if (!h->fe->normal_diag) return set_error(h, B200LM_ESIZE, "normal_diag needs np <= 8 (use b200lm_model_rows + b200lm_dgemm)");
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    const int nacc = h->np * (h->np + 1) / 2 + h->np + 1;
    const int max_parts = b200lm::ND_MAX_PARTS_PER_SM * h->sm_count;
    // per-CTA partial rows + the arrival counter of the in-kernel reduction (zero between launches: the kernel resets it;
    // b200lm_propagate shares this buffer as plain scratch, so it is cleared again whenever the two calls alternate)
    const size_t need = (size_t)max_parts * nacc * sizeof(double) + sizeof(double);
    if (need > h->scratch_bytes) {
        if (h->d_scratch) cudaFree(h->d_scratch);
        h->d_scratch = nullptr; h->scratch_bytes = 0;
        CUDA_TRY(h, cudaMalloc((void**)&h->d_scratch, need), "scratch allocation");
        h->scratch_bytes = need;
        h->scratch_counter_clean = false;
    }
    if (!h->scratch_counter_clean) {
        CUDA_TRY(h, cudaMemsetAsync((char*)h->d_scratch + (size_t)max_parts * nacc * sizeof(double), 0, sizeof(double),
                                    (cudaStream_t)stream), "reset arrival counter");
        h->scratch_counter_clean = true;
    }
    CUDA_TRY(h, h->fe->normal_diag(h->ny, h->nx, h->d_x, d_p, d_y, d_w, h->d_scratch, max_parts, d_out, h->sm_count,
                                   (cudaStream_t)stream), "normal_diag kernel launch");
    h->last_stream = (cudaStream_t)stream;
    h->launches += 1;
    return B200LM_OK;
}

long long b200lm_launch_count(b200lm_handle h) { return h ? h->launches : 0; }

int b200lm_residual_jacobian(b200lm_handle h, int B, const double* d_p, long long p_stride,
                             const double* d_mean, long long mean_stride,
                             double* d_f, double* d_J, double* d_chi2, void* stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (B < 0 || !d_p || !d_mean) return set_error(h, B200LM_EINVAL, "NULL required argument");
    if (h->nwin > 0) return set_error(h, B200LM_EINVAL, "residual_jacobian is not built for window scans");
    if (B == 0) return B200LM_OK;
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    FitParams P;
    fill_params(h, P);
    P.B = B; P.mean = d_mean; P.mean_stride = mean_stride; P.p0 = d_p; P.p0_stride = p_stride;
    P.f_out = d_f; P.J_out = d_J; P.chi2 = d_chi2;
    CUDA_TRY(h, h->fe->resjac(P, h->sm_count, h->smem_budget, (cudaStream_t)stream), "resjac kernel launch");
    h->last_stream = (cudaStream_t)stream;
    h->launches += 1;
    return B200LM_OK;
}

// ---- host-pointer variant ------------------------------------------------------------
static int ensure_stage(b200lm_handle h, size_t dev_bytes, size_t pin_bytes) {
    if (dev_bytes > h->stage_bytes) {
        if (h->d_stage) cudaFree(h->d_stage);
        h->d_stage = nullptr; h->stage_bytes = 0;
        CUDA_TRY(h, cudaMalloc(&h->d_stage, dev_bytes), "staging allocation");
        h->stage_bytes = dev_bytes;
    }
    if (pin_bytes > h->pinned_bytes) {
        if (h->h_pinned) cudaFreeHost(h->h_pinned);
        h->h_pinned = nullptr; h->pinned_bytes = 0;
        CUDA_TRY(h, cudaMallocHost(&h->h_pinned, pin_bytes), "pinned allocation");
        h->pinned_bytes = pin_bytes;
    }
    return B200LM_OK;
}

int b200lm_fit_batch_host(b200lm_handle h, int B,
                          const double* h_mean, long long mean_stride,
                          const double* h_p0, long long p0_stride,
                          double xtol, double gtol, double ftol, int maxit, int scaler, int polish,
                          double* h_x, double* h_chi2, double* h_cov, double* h_logdet,
                          int* h_nit, int* h_status, double* h_f, double* h_J) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (B == 0) return B200LM_OK;                 // empty batch
    if (B < 0 || !h_mean || !h_p0 || !h_x || !h_chi2 || !h_nit || !h_status)
        return set_error(h, B200LM_EINVAL, "NULL required argument");
    rc = window_refusal(h, B);
    if (rc) return rc;
    if (h->bounded) {                             // scipy refuses a start outside the box (least_squares: "`x0` is infeasible.")
        const long long nst = p0_stride ? (long long)B : 1;
        for (long long b = 0; b < nst; ++b)
            for (int j = 0; j < h->np; ++j) {
                const double x = h_p0[b * p0_stride + j];
                if (!(x >= h->h_lb[j] && x <= h->h_ub[j])) return set_error(h, B200LM_EINVAL, "`x0` is infeasible.");
            }
    }
    CUDA_TRY(h, cudaSetDevice(h->device), "cudaSetDevice");
    const size_t np = h->np, N = h->N, nchiv = h->nchiv;
    // with windows: a row of means per copy, a start per window
    const size_t n_mean = mean_stride ? (size_t)(h->nwin ? B / h->nwin : B) * mean_stride : N;
    const size_t n_p0 = p0_stride ? (size_t)(h->nwin ? h->nwin : B) * p0_stride : np;
    // device layout (doubles): mean | p0 | x | chi2 | logdet | cov | f | J | nit,status (ints)
    size_t off = 0;
    auto take = [&](size_t n) { size_t o = off; off += (n + 1) & ~(size_t)1; return o; };
    const size_t o_mean = take(n_mean), o_p0 = take(n_p0), o_x = take(B * np), o_chi2 = take(B),
                 o_ld = take(B), o_cov = take(h_cov ? B * np * np : 0), o_f = take(h_f ? B * nchiv : 0),
                 o_J = take(h_J ? B * nchiv * np : 0), o_int = take(B);   // 2 ints per double slot
    rc = ensure_stage(h, off * sizeof(double), 0);
    if (rc) return rc;
    double* d = (double*)h->d_stage;
    cudaStream_t s = h->own_stream;
    CUDA_TRY(h, cudaMemcpyAsync(d + o_mean, h_mean, n_mean * sizeof(double), cudaMemcpyHostToDevice, s), "H2D mean");
    CUDA_TRY(h, cudaMemcpyAsync(d + o_p0, h_p0, n_p0 * sizeof(double), cudaMemcpyHostToDevice, s), "H2D p0");
    int* d_nit = (int*)(d + o_int);
    int* d_status = d_nit + B;
    // The large write-only outputs (cov, f, J) go STRAIGHT to the caller's buffer when that is pinned, mapped host
    // memory: the kernels' stores travel over PCIe while other fits are still running, instead of a device copy
    // followed by a D2H transfer after the last fit (C3, 10^4 fits: 20 MB of covariances).  x, chi2, nit and status
    // stay on the device (the finalisation pass of the wave kernel reads x back) and are copied as before.
    auto alias = [](void* hp) -> double* {
        if (!hp || getenv("B200LM_NO_ZEROCOPY")) return nullptr;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, hp) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        return (at.type == cudaMemoryTypeHost && at.devicePointer) ? (double*)at.devicePointer : nullptr;
    };
    double* z_cov = alias(h_cov);
    double* z_f = alias(h_f);
    double* z_J = alias(h_J);
    rc = b200lm_fit_batch(h, B, d + o_mean, mean_stride, d + o_p0, p0_stride, xtol, gtol, ftol, maxit, scaler, polish,
                          d + o_x, d + o_chi2, h_cov ? (z_cov ? z_cov : d + o_cov) : nullptr, d + o_ld, d_nit, d_status,
                          h_f ? (z_f ? z_f : d + o_f) : nullptr, h_J ? (z_J ? z_J : d + o_J) : nullptr, (void*)s);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h_x, d + o_x, B * np * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H x");
    CUDA_TRY(h, cudaMemcpyAsync(h_chi2, d + o_chi2, B * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H chi2");
    if (h_logdet) CUDA_TRY(h, cudaMemcpyAsync(h_logdet, d + o_ld, B * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H logdet");
    if (h_cov && !z_cov) CUDA_TRY(h, cudaMemcpyAsync(h_cov, d + o_cov, B * np * np * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H cov");
    if (h_f && !z_f) CUDA_TRY(h, cudaMemcpyAsync(h_f, d + o_f, B * nchiv * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H f");
    if (h_J && !z_J) CUDA_TRY(h, cudaMemcpyAsync(h_J, d + o_J, B * nchiv * np * sizeof(double), cudaMemcpyDeviceToHost, s), "D2H J");
    CUDA_TRY(h, cudaMemcpyAsync(h_nit, d_nit, B * sizeof(int), cudaMemcpyDeviceToHost, s), "D2H nit");
    CUDA_TRY(h, cudaMemcpyAsync(h_status, d_status, B * sizeof(int), cudaMemcpyDeviceToHost, s), "D2H status");
    CUDA_TRY(h, cudaStreamSynchronize(s), "stream sync");
    return B200LM_OK;
}

}  // extern "C"
