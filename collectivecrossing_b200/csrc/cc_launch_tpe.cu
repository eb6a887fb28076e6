// cc_launch_tpe.cu — instantiations and launcher of ccb::cc_step_tpe_kernel (one thread per env, cc_kernel_tpe.cuh).
// Host-side plumbing only.  CCB_TPE_PART (0 / 1) splits the crews over two objects so that they compile in parallel.
#include <cstdio>
#include <cstdlib>

#if CCB_TPE_PART == 1
#define CCB_WITH_T2_TABLES 1
#endif
#include "cc_internal.h"
#include "cc_kernel_tpe2.cuh"

#ifndef CCB_TPE_PART
#error "compile with -DCCB_TPE_PART=0 (crews 1-4 and 8-agent int8 rows) or 1 (crews 5-8)"
#endif

namespace {

using ccb::KParams;

template <int A, int OBS>
int launch_tpe_t(cc_handle *h, KParams p, cudaStream_t s) {
    using L = ccb::TpeLayout<A, OBS & ~ccb::kNpReset>;
    auto kern = ccb::cc_step_tpe_kernel<A, OBS>;
    p.n_groups = (p.n_envs + 31) / 32;
    // greedy / waiting: a private lattice bitmap per thread while the lattice is small (README: 6 words)
    const bool on_device_policy = p.policy == CC_POLICY_GREEDY || p.policy == CC_POLICY_WAITING;
    // (with TMA rows the bitmap aliases the warp's image ring: 128 bytes per word)
    const int bm_cap = L::kTma ? (L::kImgRing * L::kImgBytes / 128 < ccb::kTpeMaxBitmapWords ? L::kImgRing * L::kImgBytes / 128 : ccb::kTpeMaxBitmapWords)
                               : ccb::kTpeMaxBitmapWords;
    p.tpe_bm_words = (on_device_policy && p.walk_words <= bm_cap) ? p.walk_words : 0;
    // one word per lattice row where the padded lattice has at most 32 columns and its rows fit the bitmap (README: 11 rows)
    if (on_device_policy && p.W + 3 <= 32 && p.H + 3 <= bm_cap) { p.tpe_bm_words = p.H + 3; p.tpe_bm_rows = 1; }
    // launch k counts its groups in counter k & 1 and zeroes the other one for launch k + 1 (launches of
    // one handle are stream-ordered by contract)
    if (p.n_steps < 1) p.n_steps = 1;
    p.tpe_counter = h->tpe_counters + (h->tpe_launches & 1);
    p.tpe_counter_next = h->tpe_counters + ((h->tpe_launches + 1) & 1);
    // (with TMA rows the bitmap aliases the warp's image ring)
    const int smem = L::kStageBytes + (L::kTma ? 0 : p.tpe_bm_words * ccb::kTpeThreads * 4);
    int per_sm = 0;
    int rc = cc_cached_occupancy(h, reinterpret_cast<const void *>(kern), ccb::kTpeThreads, smem, &per_sm);
    if (rc != CC_OK) return rc;
    long long want = (p.n_groups + ccb::kTpeWarps - 1) / ccb::kTpeWarps;
    long long cap = (long long)h->sm_count * per_sm;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, ccb::kTpeThreads, smem, s>>>(p);
    CC_CUDA(cudaGetLastError());
    snprintf(h->last_kernel, sizeof h->last_kernel, "ccb::cc_step_tpe_kernel<%d,%d>", A, OBS);
    h->launches += 1;
    h->tpe_launches += 1;
    return CC_OK;
}

// cc_step_tpe2_kernel: small lattices, compact output modes (cc_kernel_tpe2.cuh)
template <int A, int OBS, int BT = -1>
int launch_tpe2_t(cc_handle *h, KParams p, cudaStream_t s) {
    using L = ccb::T2Layout<A, OBS & ~ccb::kNpReset>;
    auto kern = ccb::cc_step_tpe2_kernel<A, OBS, BT>;
    int rc0 = cc_t2_ensure_tables(h, p, s);
    if (rc0 != CC_OK) return rc0;
    p.t2_tables = h->t2_tables;
    p.n_groups = (p.n_envs + 31) / 32;
    if (p.n_steps < 1) p.n_steps = 1;
    p.tpe_counter = h->tpe_counters + (h->tpe_launches & 1);
    p.tpe_counter_next = h->tpe_counters + ((h->tpe_launches + 1) & 1);
    // 4 warps per CTA; a batch that fits in one wave of those runs 2-warp CTAs: with about one group per warp the time is
    // set by the SM that got the most CTAs, and finer CTAs spread 2,048 groups over 148 SMs as 14 / 13 instead of 16 / 12
    int warps = ccb::kT2Warps;
    int per_sm = 0;
    int rc = cc_cached_occupancy(h, reinterpret_cast<const void *>(kern), warps * 32, warps * L::kBytesPerWarp, &per_sm);
    if (rc != CC_OK) return rc;
    if (p.n_groups <= (long long)h->sm_count * per_sm * warps) {
        warps = 2;
        rc = cc_cached_occupancy(h, reinterpret_cast<const void *>(kern), warps * 32, warps * L::kBytesPerWarp, &per_sm);
        if (rc != CC_OK) return rc;
    }
    const int smem = warps * L::kBytesPerWarp;
    long long want = (p.n_groups + warps - 1) / warps;
    long long cap = (long long)h->sm_count * per_sm;
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    kern<<<grid, warps * 32, smem, s>>>(p);
    CC_CUDA(cudaGetLastError());
    snprintf(h->last_kernel, sizeof h->last_kernel, "ccb::cc_step_tpe2_kernel<%d,%d>", A, OBS);
    h->launches += 1;
    h->tpe_launches += 1;
    return CC_OK;
}

// the small-lattice kernel serves: padded lattice of at most 256 cells, 32 columns, 16 rows; no float32 rows.
// CCB200_TPE2=0 in the environment switches it off (A/B measurements).
bool tpe2_eligible(const KParams &p, int obs_dtype) {
    static const bool enabled = [] { const char *v = std::getenv("CCB200_TPE2"); return !(v && v[0] == '0'); }();
    const int PW = p.W + 3, PH = p.H + 3;
    static const bool rows32 = [] { const char *v = std::getenv("CCB200_TPE2_FP32"); return !(v && v[0] == '0'); }();   // (A/B switch)
    if (obs_dtype == CC_OBS_FP32 && (!rows32 || p.A % 2 != 0)) return false;   // float32 rows of odd crews: cc_step_tpe_kernel
    return enabled && PW <= ccb::kT2MaxCols && PH <= ccb::kT2MaxRows && PW * PH <= ccb::kT2MaxCells;
}

}  // namespace

// F: 0, or ccb::kNpReset for the numpy-mode instantiations (KParams::gen set)
#define CCB_TPE2_CASES(A_, F)                                                               \
    case A_ * 32 + CC_OBS_NONE: return launch_tpe2_t<A_, CC_OBS_NONE | F>(h, p, s);             \
    case A_ * 32 + CC_OBS_TABLE: return launch_tpe2_t<A_, CC_OBS_TABLE | F>(h, p, s);
#define CCB_TPE2_CASES_EVEN(A_, F)                                                          \
    CCB_TPE2_CASES(A_, F)                                                                   \
    case A_ * 32 + CC_OBS_FP32: return launch_tpe2_t<A_, CC_OBS_FP32 | F>(h, p, s);
#define CCB_TPE_CASES(A_, F)                                                                \
    case A_ * 32 + CC_OBS_NONE: return launch_tpe_t<A_, CC_OBS_NONE | F>(h, p, s);              \
    case A_ * 32 + CC_OBS_TABLE: return launch_tpe_t<A_, CC_OBS_TABLE | F>(h, p, s);            \
    case A_ * 32 + CC_OBS_FP32: return launch_tpe_t<A_, CC_OBS_FP32 | F>(h, p, s);

#if CCB_TPE_PART == 0
template <int F>
int launch_tpe_part0(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    if (tpe2_eligible(p, obs_dtype)) {
        switch (p.A * 32 + obs_dtype) { CCB_TPE2_CASES(1, F) CCB_TPE2_CASES_EVEN(2, F) CCB_TPE2_CASES(3, F) CCB_TPE2_CASES_EVEN(4, F) }
    }
    switch (p.A * 32 + obs_dtype) {
        CCB_TPE_CASES(1, F) CCB_TPE_CASES(2, F) CCB_TPE_CASES(3, F) CCB_TPE_CASES(4, F)
    case 8 * 32 + CC_OBS_INT8: return launch_tpe_t<8, CC_OBS_INT8 | F>(h, p, s);
    }
    return cc_fail(CC_ERR_UNSUPPORTED, "no thread-per-env kernel for %d agents, obs_dtype %d", p.A, obs_dtype);
}
int cc_launch_tpe_part0(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    return p.gen ? launch_tpe_part0<ccb::kNpReset>(h, p, obs_dtype, s) : launch_tpe_part0<0>(h, p, obs_dtype, s);
}
#else
int cc_launch_tpe_part0(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s);
int cc_t2_ensure_tables(cc_handle *h, const KParams &p, cudaStream_t s) {
    if (h->t2_tables) return CC_OK;
    void *buf = nullptr;
    cudaError_t e = cudaMalloc(&buf, sizeof(ccb::T2Tables));
    if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaMalloc for the small-lattice tables: %s", cudaGetErrorString(e));
    ccb::cc_t2_tables_kernel<<<1, 256, 0, s>>>(p, static_cast<ccb::T2Tables *>(buf));
    e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(buf); return cc_fail(CC_ERR_CUDA, "cc_t2_tables_kernel: %s", cudaGetErrorString(e)); }
    h->t2_tables = buf;   // (a one-time set-up launch: not counted in cc_launch_count)
    return CC_OK;
}

template <int F>
int launch_tpe_part1(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    if (tpe2_eligible(p, obs_dtype)) {
        if (F == 0 && p.A == 8 && p.B == 5) {   // the README crew: boarding / exiting split known at compile time (Philox placements)
            switch (obs_dtype) {
            case CC_OBS_NONE: return launch_tpe2_t<8, CC_OBS_NONE, 5>(h, p, s);
            case CC_OBS_TABLE: return launch_tpe2_t<8, CC_OBS_TABLE, 5>(h, p, s);
            case CC_OBS_INT8: return launch_tpe2_t<8, CC_OBS_INT8, 5>(h, p, s);
            case CC_OBS_FP32: return launch_tpe2_t<8, CC_OBS_FP32, 5>(h, p, s);
            }
        }
        switch (p.A * 32 + obs_dtype) {
            CCB_TPE2_CASES(5, F) CCB_TPE2_CASES_EVEN(6, F) CCB_TPE2_CASES(7, F) CCB_TPE2_CASES_EVEN(8, F)
        case 8 * 32 + CC_OBS_INT8: return launch_tpe2_t<8, CC_OBS_INT8 | F>(h, p, s);
        }
    }
    switch (p.A * 32 + obs_dtype) {
        CCB_TPE_CASES(5, F) CCB_TPE_CASES(6, F) CCB_TPE_CASES(7, F) CCB_TPE_CASES(8, F)
    }
    return cc_launch_tpe_part0(h, p, obs_dtype, s);
}
int cc_launch_tpe(cc_handle *h, const KParams &p, int obs_dtype, cudaStream_t s) {
    return p.gen ? launch_tpe_part1<ccb::kNpReset>(h, p, obs_dtype, s) : launch_tpe_part1<0>(h, p, obs_dtype, s);
}
#endif
