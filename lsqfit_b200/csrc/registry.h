// Functor registry: (family, np) -> kernel launchers.  Each inst_*.cu contributes a
// table; capi.cu concatenates them.
#pragma once
#include "lm_types.h"

namespace b200lm {

struct FunctorEntry {
    int family;
    int np;
    int nx;
    const char* name;
    cudaError_t (*fit)(FitParams, int sm_count, size_t smem_budget, cudaStream_t);
    cudaError_t (*resjac)(FitParams, int sm_count, size_t smem_budget, cudaStream_t);
    size_t (*per_warp_bytes)(int rb);
    // team kernels (lm_team.cuh), indexed by log2(warps per fit) - 1: [0] two warps, [1] four warps;
    // NULL where the functor has no team instantiation
    cudaError_t (*fit_team[2])(FitParams, int sm_count, size_t smem_budget, cudaStream_t);
    size_t (*team_bytes[2])(int N);
    // wave kernel (lm_wave.cuh: 32 fits per CTA in lock-step phases); NULL where the functor has none
    cudaError_t (*fit_wave)(FitParams, int sm_count, size_t smem_budget, cudaStream_t);
    size_t (*wave_bytes)(int wt_total);
    // single-fit row kernels (lm_rows.cuh); normal_diag is NULL for np > 8 (its accumulators live in registers)
    cudaError_t (*model_rows)(int ny, int nx, const double* x, const double* p, const double* y, double* G, int ld,
                              double* delta, int sm_count, cudaStream_t);
    cudaError_t (*normal_diag)(int ny, int nx, const double* x, const double* p, const double* y, const double* w,
                               double* partial, int max_parts, double* out, int sm_count, cudaStream_t);
};

const FunctorEntry* registry_multiexp(int* n);
const FunctorEntry* registry_multiexp_b(int* n);
const FunctorEntry* registry_nist_a(int* n);
const FunctorEntry* registry_nist_b(int* n);
const FunctorEntry* registry_misc(int* n);
const FunctorEntry* registry_misc_b(int* n);
const FunctorEntry* registry_poly_b(int* n);

}  // namespace b200lm

// Run-time plug-ins (b200lm_load_functors, lsqfit_b200/user_functor.py): a shared object built from the same headers
// and flags as the library exports
//     extern "C" int b200lm_plugin_entries(const b200lm::FunctorEntry** out, int* n, b200lm_plugin_abi* abi);
// which fills the record below and returns 0.  The library copies the entries only when every field of the record
// matches its own: the entries hold launchers that take FitParams by value.
struct b200lm_plugin_abi {
    int version;               // B200LM_VERSION
    int fitparams_size;        // sizeof(b200lm::FitParams)
    int entry_size;            // sizeof(b200lm::FunctorEntry)
    char headers[72];          // B200LM_HEADERS_DIGEST: sha256 of the headers and compiler flags (build.py)
    char model[72];            // digest of the plug-in's model source: the same name from the same source is one family
};
typedef int (*b200lm_plugin_entries_fn)(const b200lm::FunctorEntry** out, int* n, b200lm_plugin_abi* abi);

#ifdef B200LM_DEFINE_ENTRIES
#include "lm_kernel.cuh"
#include "lm_team.cuh"
#include "lm_wave.cuh"
#include "lm_rows.cuh"
#include "functors.cuh"
namespace b200lm {
template <class F>
size_t per_warp_bytes_of(int rb) { return (size_t)FitLayout<F>::per_warp_doubles(rb) * sizeof(double); }
template <class F, bool SMALL = (F::NP <= 8)> struct NormalDiagOf {
    static constexpr decltype(&launch_normal_diag<F>) ptr = &launch_normal_diag<F>;
};
template <class F> struct NormalDiagOf<F, false> {
    static constexpr decltype(FunctorEntry::normal_diag) ptr = nullptr;
};
#define B200LM_ROWS(...) &launch_model_rows<__VA_ARGS__>, NormalDiagOf<__VA_ARGS__>::ptr
#define B200LM_ENTRY(family, name, ...) \
    { family, __VA_ARGS__::NP, __VA_ARGS__::NX, name, &launch_fit<__VA_ARGS__>, &launch_resjac<__VA_ARGS__>, \
      &per_warp_bytes_of<__VA_ARGS__>, {nullptr, nullptr}, {nullptr, nullptr}, nullptr, nullptr, B200LM_ROWS(__VA_ARGS__) }
// entry with team kernels (2 and 4 warps per fit)
#define B200LM_ENTRY_TEAM(family, name, ...) \
    { family, __VA_ARGS__::NP, __VA_ARGS__::NX, name, &launch_fit<__VA_ARGS__>, &launch_resjac<__VA_ARGS__>, \
      &per_warp_bytes_of<__VA_ARGS__>, {&launch_fit_team<__VA_ARGS__, 2>, &launch_fit_team<__VA_ARGS__, 4>}, \
      {&team_bytes_of<__VA_ARGS__, 2>, &team_bytes_of<__VA_ARGS__, 4>}, &launch_fit_wave<__VA_ARGS__>, \
      &wave_bytes_of<__VA_ARGS__>, B200LM_ROWS(__VA_ARGS__) }
}  // namespace b200lm
#endif
