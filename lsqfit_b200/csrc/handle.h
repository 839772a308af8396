// The plan object behind b200lm_handle (internal).
#pragma once
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "registry.h"

namespace b200lm {

// One whitening laid out for the kernels (parse_weights in capi.cu).
struct WeightTables {
    std::vector<int> fn_idx, pr_idx, blk_idx;
    std::vector<double> fn_w, pr_w, wt, wt2;
    std::vector<BlockDesc> blk;
    int nchiv = 0, ndata = 0;
    long long nw = 0;              // doubles of blk_w read
    // t's rows after these (a window scan's windows, one after the other); not wt2: windows run in the one-warp kernel
    void append(const WeightTables& t);
};

// Row tables on the host and their device copies.
struct RowTables {
    WeightTables host;
    int* d_fn_idx = nullptr; double* d_fn_w = nullptr;
    int* d_pr_idx = nullptr; double* d_pr_w = nullptr;
    BlockDesc* d_blk = nullptr; int* d_blk_idx = nullptr;
    double* d_wt = nullptr; double* d_wt2 = nullptr;
    cudaError_t upload();                   // host -> device (wt2 where the host tables have it)
    void free();
    void fill(FitParams& P) const;          // the row-table fields of P
};

}  // namespace b200lm

struct b200lm_handle_s {
    int device = 0;
    int sm_count = 0;
    size_t smem_budget = 0;
    const b200lm::FunctorEntry* fe = nullptr;
    int ny = 0, np = 0, nx = 0, noprior = 0, N = 0, nchiv = 0;
    // device-resident problem description
    double* d_x = nullptr;
    b200lm::RowTables rows;     // the plan's whitening (b200lm_set_weights)
    int rb = 64;
    bool have_weights = false, have_const = false;
    // whole whitening operator, dense [nchiv][N] (built lazily for propagate)
    double* d_wfull = nullptr;
    // work queue + statistics
    int* d_counter = nullptr;
    unsigned long long* d_stats = nullptr;
    cudaStream_t last_stream = nullptr;
    long long launches = 0;
    int team_request = 0;       // 0: default policy; 1, 2, 4: warps per fit asked for by b200lm_set_team
    int policy = 0;             // trust-region decisions: 0 scipy TRF, 1 GSL trust/lm (b200lm_set_policy)
    int last_team = 1;          // warps per fit of the last fit_batch launch
    // bound constraints (b200lm_set_bounds): device copies [np] and the host copies the host-buffer call checks p0 against
    double* d_lb = nullptr; double* d_ub = nullptr;
    std::vector<double> h_lb, h_ub;
    bool bounded = false;
    // fit windows (b200lm_set_windows): concatenated row tables of every window, used instead of the plan's weights
    // while nwin > 0; b200lm_set_weights sets nwin back to 0 (and nchiv back to the plan's)
    int nwin = 0;
    std::vector<int> win_nchiv;
    b200lm::WinDesc* d_win = nullptr;
    b200lm::RowTables win_rows;
    // queue order (longest-expected fits first): key = chi2 at the start point, one evaluation per fit
    int order_request = -1;     // -1: default policy (by problem shape and batch size); 0: off; 1: on  (b200lm_set_order)
    int last_order = 0;         // 1 if the last fit_batch launch used an ordered queue
    double* d_wave_A = nullptr; size_t wave_A_cap = 0;    // packed J^T J per fit, wave kernel -> finalisation pass
    double* d_order_key = nullptr; int* d_order = nullptr; int order_cap = 0;
    // staging for the host-pointer API
    void* d_stage = nullptr; size_t stage_bytes = 0;
    void* h_pinned = nullptr; size_t pinned_bytes = 0;
    cudaStream_t own_stream = nullptr;
    // scratch for propagate
    double* d_scratch = nullptr; size_t scratch_bytes = 0;
    bool scratch_counter_clean = false;       // normal_diag's arrival counter (behind its partial rows) is zero
    std::string err;
};

namespace b200lm {
int set_error(b200lm_handle_s* h, int code, const std::string& msg);
int cuda_fail(b200lm_handle_s* h, cudaError_t e, const char* what);
void fill_params(b200lm_handle_s* h, FitParams& P);
}
