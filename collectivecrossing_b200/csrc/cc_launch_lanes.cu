// cc_launch_lanes.cu — instantiations and launcher of ccb::cc_kernel (one lane per agent, cc_kernels.cuh) and of the
// numpy-exact seeded reset kernel.  Host-side plumbing only.
#define CCB_WITH_RESET_SEEDED 1
#include <cstdio>

#include "cc_internal.h"
#include "cc_kernels.cuh"

namespace {

using ccb::KParams;

template <int LPE, int APL, int OBS, int MODE>
int launch_t(cc_handle *h, const KParams &p, cudaStream_t s) {
    auto kern = ccb::cc_kernel<LPE, APL, OBS, MODE>;
    const int smem = p.smem_total;
    if (smem > 218 * 1024) return cc_fail(CC_ERR_UNSUPPORTED, "configuration needs %d bytes of shared memory", smem);
    int per_sm = 0;
    int rc = cc_cached_occupancy(h, reinterpret_cast<const void *>(kern), ccb::kThreads, smem, &per_sm);
    if (rc != CC_OK) return rc;
    // persistent grid: a whole number of waves of resident CTAs, never more CTAs than work
    long long want = (p.n_groups + ccb::kWarpsPerCta - 1) / ccb::kWarpsPerCta;
    long long cap = (long long)h->sm_count * per_sm;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, ccb::kThreads, smem, s>>>(p);
    CC_CUDA(cudaGetLastError());
    if (MODE == ccb::kModeStep) snprintf(h->last_kernel, sizeof h->last_kernel, "ccb::cc_kernel<%d,%d,%d,step>", LPE, APL, OBS);   // (OBS | 256: numpy placements)
    h->launches += 1;
    return CC_OK;
}

// F: 0, or ccb::kNpReset for the numpy-mode step / reset instantiations (KParams::gen set)
template <int LPE, int APL, int MODE, int F>
int launch_obs_f(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    if constexpr (MODE == ccb::kModePolicy) {
        return launch_t<LPE, APL, CC_OBS_NONE, MODE>(h, p, s);
    } else {
        switch (obs_dtype) {
        case CC_OBS_NONE:
            if constexpr (MODE == ccb::kModeObserve) return cc_fail(CC_ERR_INVALID_ARG, "observe needs an observation dtype");
            else return launch_t<LPE, APL, CC_OBS_NONE | F, MODE>(h, p, s);
        case CC_OBS_INT8: return launch_t<LPE, APL, CC_OBS_INT8 | F, MODE>(h, p, s);
        case CC_OBS_FP32: return launch_t<LPE, APL, CC_OBS_FP32 | F, MODE>(h, p, s);
        case CC_OBS_TABLE: return launch_t<LPE, APL, CC_OBS_TABLE | F, MODE>(h, p, s);
        }
        return cc_fail(CC_ERR_INVALID_ARG, "unknown obs_dtype %d", obs_dtype);
    }
}
template <int LPE, int APL, int MODE>
int launch_obs(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    if constexpr (MODE == ccb::kModeStep || MODE == ccb::kModeReset)
        if (p.gen) return launch_obs_f<LPE, APL, MODE, ccb::kNpReset>(h, p, obs_dtype, s);
    return launch_obs_f<LPE, APL, MODE, 0>(h, p, obs_dtype, s);
}

template <int MODE>
int launch(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    if (MODE == ccb::kModePolicy) obs_dtype = CC_OBS_NONE;
    switch (h->lpe * 8 + h->apl) {
    case 4 * 8 + 1: return launch_obs<4, 1, MODE>(h, p, obs_dtype, s);
    case 8 * 8 + 1: return launch_obs<8, 1, MODE>(h, p, obs_dtype, s);
    case 16 * 8 + 1: return launch_obs<16, 1, MODE>(h, p, obs_dtype, s);
    case 32 * 8 + 1: return launch_obs<32, 1, MODE>(h, p, obs_dtype, s);
    case 32 * 8 + 2: return launch_obs<32, 2, MODE>(h, p, obs_dtype, s);
    case 32 * 8 + 4: return launch_obs<32, 4, MODE>(h, p, obs_dtype, s);
    }
    return cc_fail(CC_ERR_UNSUPPORTED, "no kernel for %d agents", h->A);
}

}  // namespace

int cc_launch_lanes(cc_handle *h, const KParams &p, int mode, int obs_dtype, cudaStream_t s) {
    switch (mode) {
    case ccb::kModeStep: return launch<ccb::kModeStep>(h, p, obs_dtype, s);
    case ccb::kModeReset: return launch<ccb::kModeReset>(h, p, obs_dtype, s);
    case ccb::kModePolicy: return launch<ccb::kModePolicy>(h, p, obs_dtype, s);
    case ccb::kModeObserve: return launch<ccb::kModeObserve>(h, p, obs_dtype, s);
    }
    return cc_fail(CC_ERR_INVALID_ARG, "unknown kernel mode %d", mode);
}

int cc_launch_reset_seeded(cc_handle *h, const KParams &p, const int64_t *seeds, cudaStream_t s) {
    const int threads = 128;
    const long long blocks = (p.n_envs + threads - 1) / threads;
    ccb::cc_reset_seeded_kernel<<<(unsigned)blocks, threads, 0, s>>>(p, reinterpret_cast<const long long *>(seeds), h->gen);
    CC_CUDA(cudaGetLastError());
    h->launches += 1;
    return CC_OK;
}

size_t cc_rng_state_bytes(void) { return sizeof(ccb::Pcg64State); }
