// The plan object behind b200lm_handle (internal).
#pragma once
#include <string>
#include <vector>
#include <cuda_runtime.h>
#include "registry.h"

struct b200lm_handle_s {
    int device = 0;
    int sm_count = 0;
    size_t smem_budget = 0;
    const b200lm::FunctorEntry* fe = nullptr;
    int ny = 0, np = 0, nx = 0, noprior = 0, N = 0, nchiv = 0;
    // device-resident problem description
    double* d_x = nullptr;
    int* d_dfn_idx = nullptr; double* d_dfn_w = nullptr; int nd_fn = 0;
    int* d_dpr_idx = nullptr; double* d_dpr_w = nullptr; int nd_pr = 0;
    b200lm::BlockDesc* d_blk = nullptr; int nblk = 0;
    int* d_blk_idx = nullptr; double* d_blk_wt = nullptr; int wt_total = 0;
    double* d_blk_wt2 = nullptr; int wt2_total = 0;      // team-kernel layout of the same weights
    int rb = 64;
    bool have_weights = false, have_const = false;
    // host copies (used by propagate)
    std::vector<int> h_diag_idx; std::vector<double> h_diag_w;
    std::vector<b200lm::BlockDesc> h_blk; std::vector<int> h_blk_idx;
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
    int* d_win_dfn_idx = nullptr; double* d_win_dfn_w = nullptr;
    int* d_win_dpr_idx = nullptr; double* d_win_dpr_w = nullptr;
    b200lm::BlockDesc* d_win_blk = nullptr; int* d_win_blk_idx = nullptr; double* d_win_blk_wt = nullptr;
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
