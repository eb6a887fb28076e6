// cc_api.cu — the extern "C" boundary declared in include/ccb200.h.
// Host-side plumbing only: handle, kernel dispatch, host<->device staging, statistics.  The kernels are
// instantiated in cc_launch_lanes.cu / cc_launch_tpe.cu; the host-side row expansion is cc_expand.cpp.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include <cuda.h>   // driver types of cc_device_alloc (the functions are resolved at run time)

#include "cc_internal.h"
#include "cc_workers.h"
#include "cc_kernel_tpe.cuh"   // KParams, layout constants (no kernel is instantiated in this file)

#ifndef CCB_TPE_ALTERNATE
#define CCB_TPE_ALTERNATE 1   // single-step launches alternate the direction in which groups are handed out (L2 hits on the state)
#endif

namespace {

thread_local char g_err[512] = "";

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int round_up(int v, int m) { return (v + m - 1) / m * m; }
size_t align256(size_t v) { return (v + 255) / 256 * 256; }
bool aligned_to(const void *q, uintptr_t a) { return (reinterpret_cast<uintptr_t>(q) & (a - 1)) == 0; }
bool is_rows(int obs_dtype) { return obs_dtype == CC_OBS_INT8 || obs_dtype == CC_OBS_FP32; }
// bytes of one env's block of the `obs` output
size_t obs_env_bytes(int A, int obs_dtype) {
    if (obs_dtype == CC_OBS_TABLE) return 4 * (size_t)A;
    return is_rows(obs_dtype) ? (size_t)A * (6 + 4 * (size_t)A) * (size_t)obs_dtype : 0;
}

// Driver entry points of cc_device_alloc, resolved through the runtime: the library links the static runtime, not libcuda.
struct DriverApi {
    bool ok = false;
    decltype(&::cuDeviceGetAttribute) cuDeviceGetAttribute = nullptr;
    decltype(&::cuMemGetAllocationGranularity) cuMemGetAllocationGranularity = nullptr;
    decltype(&::cuMemCreate) cuMemCreate = nullptr;
    decltype(&::cuMemGetAllocationPropertiesFromHandle) cuMemGetAllocationPropertiesFromHandle = nullptr;
    decltype(&::cuMemAddressReserve) cuMemAddressReserve = nullptr;
    decltype(&::cuMemMap) cuMemMap = nullptr;
    decltype(&::cuMemSetAccess) cuMemSetAccess = nullptr;
    decltype(&::cuMemUnmap) cuMemUnmap = nullptr;
    decltype(&::cuMemAddressFree) cuMemAddressFree = nullptr;
    decltype(&::cuMemRelease) cuMemRelease = nullptr;
};

template <typename F>
bool driver_entry(const char *name, F &fn) {
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    void *p = nullptr;
    if (cudaGetDriverEntryPointByVersion(name, &p, 12000, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return false;
    fn = reinterpret_cast<F>(p);
    return true;
}

const DriverApi &driver_api() {
    static const DriverApi api = [] {
        DriverApi d;
        d.ok = driver_entry("cuDeviceGetAttribute", d.cuDeviceGetAttribute) && driver_entry("cuMemGetAllocationGranularity", d.cuMemGetAllocationGranularity) &&
               driver_entry("cuMemCreate", d.cuMemCreate) && driver_entry("cuMemGetAllocationPropertiesFromHandle", d.cuMemGetAllocationPropertiesFromHandle) &&
               driver_entry("cuMemAddressReserve", d.cuMemAddressReserve) && driver_entry("cuMemMap", d.cuMemMap) &&
               driver_entry("cuMemSetAccess", d.cuMemSetAccess) && driver_entry("cuMemUnmap", d.cuMemUnmap) &&
               driver_entry("cuMemAddressFree", d.cuMemAddressFree) && driver_entry("cuMemRelease", d.cuMemRelease);
        return d;
    }();
    return api;
}

// live allocations of cc_device_alloc; mapped = 0: plain cudaMalloc memory
struct DeviceAlloc { void *ptr; size_t mapped; unsigned long long handle; int device; };
std::mutex g_alloc_mu;
std::vector<DeviceAlloc> g_allocs;

}  // namespace

int cc_fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

int cc_cached_occupancy(cc_handle *h, const void *fn, int threads, int smem, int *per_sm) {
    for (const cc_launch_cfg &c : h->launch_cfgs)
        if (c.fn == fn && c.threads == threads && c.smem == smem) { *per_sm = c.per_sm; return CC_OK; }
    // the kernels also hold up to ~21 KB of static shared memory: always opt in to the dynamic size.  The attribute belongs to
    // the FUNCTION (per device), not to a handle, and one instantiation is launched with different sizes (4- and 2-warp CTAs,
    // different handles): it is only ever raised.
    {
        static std::mutex mu;
        static std::vector<std::pair<std::pair<const void *, int>, int>> raised;   // (function, device) -> largest size opted in to
        std::lock_guard<std::mutex> lock(mu);
        int *cur = nullptr;
        for (auto &r : raised)
            if (r.first.first == fn && r.first.second == h->device) cur = &r.second;
        if (!cur) { raised.push_back({{fn, h->device}, 0}); cur = &raised.back().second; }
        if (smem > *cur) {
            CC_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            *cur = smem;
        }
    }
    int n = 0;
    CC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, fn, threads, smem));
    if (n < 1) return cc_fail(CC_ERR_UNSUPPORTED, "kernel does not fit on an SM (%d bytes of dynamic shared memory)", smem);
    h->launch_cfgs.push_back(cc_launch_cfg{fn, threads, smem, n});
    *per_sm = n;
    return CC_OK;
}

namespace {

using ccb::KParams;

// lowered config + shard + shared-memory layout for the envs [first, first + count) of the handle
void fill_params(const cc_handle *h, KParams &p, int obs_dtype, bool needs_bitmap, long long first, long long count) {
    const cc_config &c = h->cfg;
    const int A = h->A;
    memset(&p, 0, sizeof p);
    p.W = c.width; p.H = c.height; p.D = c.division_y; p.TL = c.tram_left; p.TR = c.tram_right;
    p.DL = c.door_left; p.DR = c.door_right; p.DC = (c.door_left + c.door_right) / 2;
    p.YB = c.boarding_dest_y; p.YE = c.exiting_dest_y; p.B = c.num_boarding; p.A = A;
    p.max_steps = c.max_steps; p.reward_kind = c.reward_kind; p.terminated_kind = c.terminated_kind;
    for (int i = 0; i < 4; ++i) { p.rp[i] = c.reward_params[i]; p.rpf[i] = (float)c.reward_params[i]; }
    p.reward_category_mask = c.reward_kind == CC_REWARD_DEFAULT ? 0xFu : 0u;
    p.n_envs = count; p.genv_offset = (unsigned long long)(h->genv_offset + first); p.seed = h->seed; p.t = (unsigned)h->t;
    p.x = h->x + first * A; p.y = h->y + first * A; p.flags = h->flags + first * A; p.step = h->step + first; p.ep_ret = h->ep_ret + first;
    p.stats = h->stats; p.err = h->err;
    p.R = 3 + 2 * A;
    p.pairs_per_env = A * p.R;
    const bool rows = is_rows(obs_dtype);
    // int8 rows of big crews (one env per warp) whose env block is whole 16-byte vectors: shifted template copies, vector
    // lists, a LUT for the special vectors only and a ring of chunk images that leave through bulk copies (cc_kernels.cuh)
    const int env_bytes = A * (6 + 4 * A);
    const bool shifted = obs_dtype == CC_OBS_INT8 && h->lpe == 32 && h->epw == 1 && env_bytes % 16 == 0 && env_bytes / 16 < 65536;
    p.lut_entries = (rows && !shifted) ? h->epw * p.pairs_per_env : 0;
    p.stage_pairs = rows ? round_up(h->epw * (2 * A + 4), 8) : 0;  // one row template per env
    p.walk_words = ((c.width + 3) * (c.height + 3) + 31) / 32;
    const int pair_bytes = obs_dtype == CC_OBS_FP32 ? 8 : 2;
    int off = round_up(p.lut_entries * 2, 16);
    p.off_stage = off;
    off += round_up(ccb::kWarpsPerCta * p.stage_pairs * pair_bytes, 16);
    p.off_bitmap = off;
    off += needs_bitmap ? round_up(ccb::kWarpsPerCta * h->epw * p.walk_words * 4, 16) : 0;
    p.off_desc = off;
    off += (rows && h->lpe <= 16) ? ccb::kDescWords * 4 * ccb::kThreads : 0;
    if (shifted) {
        p.nvec_env = env_bytes / 16;
        p.shift_tst = round_up(14 + (6 + 4 * A) + 18, 16);   // shift + row template + its first 16 bytes again (+ agent 2's block)
        p.off_shift = off;
        off += ccb::kWarpsPerCta * 8 * p.shift_tst;
        // a row is 6 + 4A = 2 x odd bytes: 8 rows are the smallest run of rows that is a whole number of 16-byte vectors
        // (env_bytes % 16 == 0 <=> A % 8 == 0); chunks of 8 m rows, about 2.5 KB: small chunks pay a fence and three warp syncs each
        const int bytes8 = 8 * (6 + 4 * A);
        int m = (2560 + bytes8 / 2) / bytes8;
        if (m < 1) m = 1;
        if (8 * m > 32) m = 4;                    // one lane patches one row
        if (8 * m > A) m = A / 8;
        p.img_rows = 8 * m;
        p.img_vecs = m * bytes8 / 16;
        p.n_chunks = (A + p.img_rows - 1) / p.img_rows;
        p.max_special = 0;
        p.off_vlist = off;                        // source offsets of a chunk's vectors (uint32)
        off += round_up(p.img_vecs * 4, 16);
        p.off_img = off;
        off += ccb::kWarpsPerCta * ccb::kLaneImgRing * p.img_vecs * 16;
    }
    // one env per warp (crews above 16): byte maps of the padded lattice for the parallel resolution of the ordered moves
    // (cc_kernels.cuh); lattices whose maps would not fit keep the sequential turns
    const int cells = round_up((c.width + 3) * (c.height + 3), 16);
    static const bool cellmaps = [] { const char *v = getenv("CCB200_CELLMAP"); return !(v && v[0] == '0'); }();   // (A/B switch)
    if (cellmaps && h->lpe == 32 && h->epw == 1 && cells <= 3072) {
        off = round_up(off, 16);
        p.off_cellmap = off;
        p.cellmap_cells = cells;
        off += ccb::kWarpsPerCta * (2 * cells + 128);
    }
    p.smem_total = off;
    p.n_groups = (count + h->epw - 1) / h->epw;
    p.n_steps = 1;
    p.slice_envs = count; p.slice_agents = count * A; p.slice_obs_bytes = (long long)(count * obs_env_bytes(A, obs_dtype));
}

// which step launches the thread-per-env kernel can serve (io: DEVICE pointers of the sub-range's first env)
bool tpe_eligible(const cc_handle *h, const cc_step_io *io, long long first) {
    const int A = h->A;
    if (A < 1 || A > 8) return false;
    if (io->order || io->reward_dtype != CC_REWARD_F32) return false;      // dict order / float64 rewards: lane-group kernel
    if (io->obs_dtype == CC_OBS_INT8 && A != 8) return false;              // an env's int8 block must be whole 16-byte vectors
    if (A == 8 || A == 4) {                                                // rows are moved as one aligned word
        const void *rows[] = {h->x + first * A, h->y + first * A, h->flags + first * A, io->actions, io->actions_out, io->agent_flags, io->agent_info};
        for (const void *q : rows)
            if (q && !aligned_to(q, (uintptr_t)A)) return false;
    }
    return aligned_to(io->reward, A % 4 == 0 ? 16 : 4) && aligned_to(h->step, 4) && aligned_to(h->ep_ret, 4);
}

// a call that may place envs in CC_RESET_RNG_NUMPY mode needs seeded generators (like cc_reset_seeded(NULL))
int check_reset_rng(const cc_handle *h, bool places) {
    if (places && h->reset_rng == CC_RESET_RNG_NUMPY && !h->gen_seeded)
        return cc_fail(CC_ERR_INVALID_ARG, "CC_RESET_RNG_NUMPY places envs from the generators cc_reset_seeded(seeds) or cc_set_rng_state seed: seed them first");
    return CC_OK;
}

int check_io(const cc_handle *h, const cc_step_io *io) {
    if (!h || !io) return cc_fail(CC_ERR_INVALID_ARG, "null handle or io");
    if (io->policy < CC_POLICY_EXTERNAL || io->policy > CC_POLICY_WAITING) return cc_fail(CC_ERR_INVALID_ARG, "unknown policy %d", io->policy);
    if (io->policy == CC_POLICY_EXTERNAL && !io->actions) return cc_fail(CC_ERR_INVALID_ARG, "policy EXTERNAL needs io->actions");
    if (io->obs_dtype != CC_OBS_NONE && io->obs_dtype != CC_OBS_INT8 && io->obs_dtype != CC_OBS_FP32 && io->obs_dtype != CC_OBS_TABLE)
        return cc_fail(CC_ERR_INVALID_ARG, "unknown obs_dtype %d", io->obs_dtype);
    if (io->obs_dtype != CC_OBS_NONE && !io->obs) return cc_fail(CC_ERR_INVALID_ARG, "obs_dtype set but io->obs is null");
    if (io->reward_dtype != CC_REWARD_F32 && io->reward_dtype != CC_REWARD_F64) return cc_fail(CC_ERR_INVALID_ARG, "unknown reward_dtype %d", io->reward_dtype);
    if (!io->reward || !io->agent_flags || !io->env_flags) return cc_fail(CC_ERR_INVALID_ARG, "reward, agent_flags and env_flags are required");
    return check_reset_rng(h, io->auto_reset != 0);
}
int check_obs_alignment(const cc_step_io *io) {
    if (io->obs && (reinterpret_cast<uintptr_t>(io->obs) & 15)) return cc_fail(CC_ERR_INVALID_ARG, "io->obs must be 16-byte aligned");
    return CC_OK;
}

// every stream-taking call leaves an event behind; the host path waits for it (header: "Stream order")
int mark_order(cc_handle *h, cudaStream_t s) {
    CC_CUDA(cudaEventRecord(h->ev_order, s));
    h->order_pending = true;
    return CC_OK;
}

struct StepArgs {
    int n_steps = 1;               // > 1: one fused launch of the thread-per-env kernel (the caller has checked eligibility)
    long long first = 0, count = 0;   // envs [first, first + count) of the handle; io points at env `first` of time slice 0
    long long stride_envs = 0;     // envs between two time slices of the outputs (fused launches)
    long long obs_env_offset = 0;  // lane-group kernel: row block offset into io->obs (time slices whose byte offset is not 16-aligned)
    uint64_t t = 0;                // RNG counter word of the (first) step
    bool alternate = false;        // alternate the direction in which groups are handed out
};

// One launch.  Does not advance h->t (the callers do: a chunked host step is ONE step for the RNG).
int step_on(cc_handle *h, const cc_step_io *io, cudaStream_t s, const StepArgs &a) {
    KParams p;
    fill_params(h, p, io->obs_dtype, io->policy == CC_POLICY_GREEDY || io->policy == CC_POLICY_WAITING, a.first, a.count);
    p.t = (unsigned)a.t;
    p.n_steps = a.n_steps;
    p.obs_env_offset = a.obs_env_offset;
    const long long stride = a.stride_envs > 0 ? a.stride_envs : a.count;
    p.slice_envs = stride; p.slice_agents = stride * h->A; p.slice_obs_bytes = (long long)(stride * obs_env_bytes(h->A, io->obs_dtype));
    p.actions = io->actions; p.order = io->order; p.actions_out = io->actions_out;
    p.obs = io->obs; p.reward = io->reward; p.agent_flags = io->agent_flags; p.agent_info = io->agent_info; p.env_flags = io->env_flags;
    p.policy = io->policy; p.auto_reset = io->auto_reset != 0; p.reward_f64 = io->reward_dtype == CC_REWARD_F64;
    if (h->reset_rng == CC_RESET_RNG_NUMPY && p.auto_reset) p.gen = h->gen + a.first;   // (env n of the launch: generator first + n)
    const bool can_tpe = a.obs_env_offset == 0 && tpe_eligible(h, io, a.first);
    if (h->variant == CC_KERNEL_THREADS && !can_tpe)
        return cc_fail(CC_ERR_UNSUPPORTED, "CC_KERNEL_THREADS was requested but this step is not eligible (needs at most 8 agents, agent order, "
                                           "float32 rewards, int8 rows only for 8 agents, word-aligned rows for 4 or 8 agents)");
    const bool use_tpe = can_tpe && h->variant != CC_KERNEL_LANES;
    if (a.n_steps > 1 && !use_tpe) return cc_fail(CC_ERR_UNSUPPORTED, "fused multi-step launches need the thread-per-env kernel");
    if (use_tpe) p.tpe_reverse = (CCB_TPE_ALTERNATE && a.alternate && a.n_steps == 1) ? (int)(h->tpe_launches & 1) : 0;
    else p.tpe_reverse = (CCB_TPE_ALTERNATE && a.alternate) ? (int)(a.t & 1) : 0;
    int rc = use_tpe ? cc_launch_tpe(h, p, io->obs_dtype, s) : cc_launch_lanes(h, p, ccb::kModeStep, io->obs_dtype, s);
    if (rc == CC_OK) h->last_variant = use_tpe ? CC_KERNEL_THREADS : CC_KERNEL_LANES;
    return rc;
}

// n_steps env-steps of the envs [first, first + count) into time-major outputs (slice stride `stride_envs` envs):
// one fused launch where the thread-per-env kernel applies, else one launch per step.  io: DEVICE pointers of env `first`,
// slice 0.  Does not advance h->t.
int rollout_on(cc_handle *h, const cc_step_io *io, cudaStream_t s, int n_steps, long long first, long long count, long long stride_envs, uint64_t t0) {
    StepArgs a;
    a.first = first; a.count = count; a.stride_envs = stride_envs; a.t = t0;
    if (n_steps == 1) { a.alternate = (first == 0 && count == h->n_envs); return step_on(h, io, s, a); }
    if (tpe_eligible(h, io, first) && h->variant != CC_KERNEL_LANES) { a.n_steps = n_steps; return step_on(h, io, s, a); }   // state stays in registers
    if (h->variant == CC_KERNEL_THREADS) return cc_fail(CC_ERR_UNSUPPORTED, "CC_KERNEL_THREADS was requested but this rollout is not eligible");
    // any other crew / dtype: one launch per step into the time slices
    const size_t sa = (size_t)stride_envs * h->A, se = (size_t)stride_envs;
    for (int t = 0; t < n_steps; ++t) {
        cc_step_io d = *io;
        if (io->actions) d.actions = io->actions + t * sa;
        if (io->actions_out) d.actions_out = io->actions_out + t * sa;
        // (the observation slice is addressed through an env offset: t * slice bytes need not be 16-byte aligned)
        d.reward = static_cast<char *>(io->reward) + t * sa * (size_t)io->reward_dtype;
        d.agent_flags = io->agent_flags + t * sa;
        if (io->agent_info) d.agent_info = io->agent_info + t * sa;
        d.env_flags = io->env_flags + t * se;
        a.obs_env_offset = (long long)t * stride_envs;
        a.t = t0 + (uint64_t)t;
        int rc = step_on(h, &d, s, a);
        if (rc != CC_OK) return rc;
    }
    return CC_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// host path: HOST buffers in, HOST buffers out.  The envs are cut into chunks; chunk c+1's host->device copy and
// kernel overlap chunk c's device->host copies (three streams, a ring of kRing staging sets).
// ---------------------------------------------------------------------------------------------------------------
int ensure_host_path(cc_handle *h, size_t bytes) {
    if (!h->s_in) {
        CC_CUDA(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
        CC_CUDA(cudaStreamCreateWithFlags(&h->s_k, cudaStreamNonBlocking));
        CC_CUDA(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < cc_handle::kRing; ++i) {
            CC_CUDA(cudaEventCreateWithFlags(&h->ev_in[i], cudaEventDisableTiming));
            CC_CUDA(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
            CC_CUDA(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
        }
    }
    if (bytes > h->stage_bytes) {
        if (h->stage_block) CC_CUDA(cudaFree(h->stage_block));
        h->stage_block = nullptr; h->stage_bytes = 0;
        cudaError_t e = cudaMalloc(&h->stage_block, bytes);
        if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaMalloc(%zu) for host staging: %s", bytes, cudaGetErrorString(e));
        h->stage_bytes = bytes;
    }
    return CC_OK;
}

// rows of `row_bytes` bytes: device [T][c] (compact) <-> host [T][N], the chunk starting at env `first`
thread_local int64_t *g_copy_bytes = nullptr;   // host_pipeline's {h2d, d2h} byte counters of the call in progress

int copy_slices(void *dst, const void *src, size_t row_bytes, int T, long long c, long long N, long long first, bool to_device, cudaStream_t s) {
    if (T > 1 && (size_t)N * row_bytes >= (size_t)1 << 31) {   // pitch beyond what 2D copies accept: slice by slice
        for (int t = 0; t < T; ++t) {
            void *d = static_cast<char *>(dst) + (to_device ? (size_t)t * c : (size_t)t * N) * row_bytes;
            const void *q = static_cast<const char *>(src) + (to_device ? (size_t)t * N : (size_t)t * c) * row_bytes;
            int rc = copy_slices(d, q, row_bytes, 1, c, N, first, to_device, s);
            if (rc != CC_OK) return rc;
        }
        return CC_OK;
    }
    if (g_copy_bytes) g_copy_bytes[to_device ? 0 : 1] += (int64_t)((size_t)T * (size_t)c * row_bytes);
    if (to_device) {
        const char *hsrc = static_cast<const char *>(src) + (size_t)first * row_bytes;
        if (T == 1) CC_CUDA(cudaMemcpyAsync(dst, hsrc, (size_t)c * row_bytes, cudaMemcpyHostToDevice, s));
        else CC_CUDA(cudaMemcpy2DAsync(dst, (size_t)c * row_bytes, hsrc, (size_t)N * row_bytes, (size_t)c * row_bytes, T, cudaMemcpyHostToDevice, s));
    } else {
        char *hdst = static_cast<char *>(dst) + (size_t)first * row_bytes;
        if (T == 1) CC_CUDA(cudaMemcpyAsync(hdst, src, (size_t)c * row_bytes, cudaMemcpyDeviceToHost, s));
        else CC_CUDA(cudaMemcpy2DAsync(hdst, (size_t)N * row_bytes, src, (size_t)c * row_bytes, (size_t)c * row_bytes, T, cudaMemcpyDeviceToHost, s));
    }
    return CC_OK;
}

// ordinary (malloc / numpy) memory: copies to and from it are staged by the driver inside the calling thread
bool is_pageable(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeUnregistered;
}

int grow_pinned(void **block, size_t *have, size_t need, const char *what) {
    if (need <= *have) return CC_OK;
    if (*block) CC_CUDA(cudaFreeHost(*block));
    *block = nullptr; *have = 0;
    cudaError_t e = cudaHostAlloc(block, need, cudaHostAllocDefault);
    if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaHostAlloc(%zu) for %s: %s", need, what, cudaGetErrorString(e));
    *have = need;
    return CC_OK;
}

int host_pipeline(cc_handle *h, const cc_step_io *io, int T) {
    int rc = check_io(h, io);
    if (rc != CC_OK) return rc;
    if (T < 1) return cc_fail(CC_ERR_INVALID_ARG, "n_steps must be positive");
    if (T > 1 && io->order) return cc_fail(CC_ERR_INVALID_ARG, "multi-step rollouts move agents in agent order (io->order must be NULL)");
    DeviceGuard guard(h->device);
    const int A = h->A;
    const long long N = h->n_envs;
    // rows rebuilt on the host (cc_set_host_expand): the kernel writes the table, the table crosses PCIe
    bool expand = false;
    int expand_threads = 0;   // 0 = every hardware thread
    if (is_rows(io->obs_dtype) && h->host_expand != CC_HOST_EXPAND_OFF) {
        if (h->host_expand == CC_HOST_EXPAND_AUTO)
            expand = cc_expand_beats_pcie(&h->cfg, io->obs_dtype) && cc_host_threads() >= 8 &&
                     (size_t)T * (size_t)N * obs_env_bytes(A, io->obs_dtype) >= ((size_t)16 << 20);
        else { expand = true; expand_threads = h->host_expand > 0 ? h->host_expand : 0; }
    }
    const int k_obs = expand ? CC_OBS_TABLE : io->obs_dtype;
    const size_t obs_b = obs_env_bytes(A, k_obs), rew_b = (size_t)A * (size_t)io->reward_dtype;
    const size_t per_env_step = obs_b + rew_b + 5 * (size_t)A + 1;
    // chunk: about N/8 envs (enough chunks to hide the first kernel and the last copy, few enough to keep the
    // per-chunk API cost small), a multiple of 32, at least 16,384 envs, at most ~2 GB of staging per set
    long long chunk = h->host_chunk > 0 ? h->host_chunk : (N + 7) / 8;
    if (h->host_chunk <= 0 && chunk < 16384) chunk = 16384;
    const long long cap = (long long)((2ull << 30) / (per_env_step * (size_t)T));
    if (chunk > cap) chunk = cap;
    chunk = (chunk + 31) / 32 * 32;
    if (chunk < 32) chunk = 32;
    if (chunk > N) chunk = N;
    const long long n_chunks = (N + chunk - 1) / chunk;
    const int ring = n_chunks < cc_handle::kRing ? (int)n_chunks : cc_handle::kRing;
    // staging layout of one set (compact [T][chunk] arrays)
    const size_t ca = (size_t)chunk * A, tca = ca * (size_t)T;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = align256(off + bytes); return o; };
    const size_t o_act = take(tca), o_ord = take(ca), o_ao = take(tca), o_obs = take((size_t)T * chunk * obs_b), o_rew = take(tca * (size_t)io->reward_dtype),
                 o_af = take(tca), o_ai = take(tca), o_ef = take((size_t)T * chunk);
    const size_t set_bytes = off;
    rc = ensure_host_path(h, set_bytes * ring);
    if (rc != CC_OK) return rc;
    if (expand) {
        rc = grow_pinned(&h->host_table, &h->host_table_bytes, (size_t)T * N * obs_b, "the observation tables");
        if (rc != CC_OK) return rc;
    }
    // Pageable caller buffers (malloc, numpy): a copy to or from them is staged by the driver inside the calling thread (~15 GB/s and
    // the pipeline stands still meanwhile).  With host threads at hand such arrays go through pinned mirrors [T][N] of the handle:
    // the copies run at link speed and the threads move the bytes between mirror and caller, slice by slice.
    struct Mirror { char *user, *pinned; size_t row_b; };
    Mirror mir[6];
    int n_mir = 0;
    char *act_src = const_cast<char *>(reinterpret_cast<const char *>(io->actions));   // where the H2D copies of the actions read
    const bool crew_ok = h->host_expand > 0 || h->host_expand == CC_HOST_EXPAND_ALL || (h->host_expand == CC_HOST_EXPAND_AUTO && cc_host_threads() >= 8);
    {
        struct Out { void *p; size_t row_b; };
        const Out outs[6] = {{expand ? nullptr : io->obs, obs_b}, {io->reward, rew_b}, {io->agent_flags, (size_t)A}, {io->agent_info, (size_t)A},
                             {io->actions_out, (size_t)A}, {io->env_flags, 1}};
        size_t total = 0, mirrored = 0;
        for (const Out &o : outs) total += o.p ? (size_t)T * N * o.row_b : 0;
        if (crew_ok && total >= ((size_t)4 << 20)) {
            size_t moff = 0;
            for (const Out &o : outs) {
                const size_t bytes = (size_t)T * N * o.row_b;
                if (!o.p || !bytes || bytes > ((size_t)512 << 20) || !is_pageable(o.p)) continue;   // (huge arrays: no second copy of them)
                mir[n_mir++] = Mirror{static_cast<char *>(o.p), reinterpret_cast<char *>(moff), o.row_b};
                moff = align256(moff + bytes);
            }
            size_t act_off = 0;
            const bool mirror_actions = io->actions && (size_t)T * N * A >= ((size_t)1 << 20) && is_pageable(io->actions);
            if (mirror_actions) { act_off = moff; moff = align256(moff + (size_t)T * N * A); }
            mirrored = moff;
            if (mirrored) {
                rc = grow_pinned(&h->host_mirror, &h->host_mirror_bytes, mirrored, "the mirrors of pageable buffers");
                if (rc != CC_OK) return rc;
                for (int k = 0; k < n_mir; ++k) mir[k].pinned = static_cast<char *>(h->host_mirror) + reinterpret_cast<size_t>(mir[k].pinned);
                if (mirror_actions) act_src = static_cast<char *>(h->host_mirror) + act_off;
            }
        }
    }
    auto dst_of = [&](void *user) -> void * {   // where the D2H copies of this output land
        for (int k = 0; k < n_mir; ++k)
            if (mir[k].user == user) return mir[k].pinned;
        return user;
    };
    const int crew = (expand || n_mir || act_src != reinterpret_cast<const char *>(io->actions)) ? cc_expand_thread_count(expand_threads, chunk) : 1;
    if (crew > 1 && !h->workers) h->workers = new cc_worker_pool();
    auto run_crew = [&](const std::function<void(int)> &fn) {
        if (crew > 1) h->workers->run(crew, fn);
        else fn(0);
    };
    if (expand || n_mir) {
        for (std::vector<cudaEvent_t> *evs : {&h->ev_chunk, &h->ev_done})
            while ((long long)evs->size() < n_chunks) {
                cudaEvent_t ev;
                CC_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                evs->push_back(ev);
            }
    }
    if (act_src != reinterpret_cast<const char *>(io->actions)) {   // the caller's actions into the pinned mirror, all threads at once
        const size_t bytes = (size_t)T * N * A, per = (bytes / crew + 4095) & ~(size_t)4095;
        run_crew([&](int w) {
            const size_t a = std::min(bytes, (size_t)w * per), b = std::min(bytes, (size_t)(w + 1) * per);
            if (a < b) memcpy(act_src + a, reinterpret_cast<const char *>(io->actions) + a, b - a);
        });
    }
    if (h->order_pending) {   // everything enqueued on the caller's streams so far happens before this call
        CC_CUDA(cudaStreamWaitEvent(h->s_in, h->ev_order, 0));
        CC_CUDA(cudaStreamWaitEvent(h->s_k, h->ev_order, 0));
    }
    h->last_host[0] = n_chunks; h->last_host[1] = chunk; h->last_host[2] = 0; h->last_host[3] = h->last_host[4] = 0;
    struct CountCopies {
        explicit CountCopies(int64_t *c) { g_copy_bytes = c; }
        ~CountCopies() { g_copy_bytes = nullptr; }
    } count_copies(h->last_host + 3);
    const uint64_t t0 = h->t;
    // (a failure part-way leaves copies in flight that still write the caller's buffers: every exit drains the three streams)
    auto enqueue_all = [&]() -> int {
    for (long long c = 0; c < n_chunks; ++c) {
        const int set = (int)(c % ring);
        const long long first = c * chunk, cnt = (N - first < chunk) ? N - first : chunk;
        char *b = static_cast<char *>(h->stage_block) + (size_t)set * set_bytes;
        cc_step_io d = *io;
        d.obs_dtype = k_obs;
        d.actions = io->actions ? reinterpret_cast<int8_t *>(b + o_act) : nullptr;
        d.order = io->order ? reinterpret_cast<int8_t *>(b + o_ord) : nullptr;
        d.actions_out = io->actions_out ? reinterpret_cast<int8_t *>(b + o_ao) : nullptr;
        d.obs = obs_b ? b + o_obs : nullptr;
        d.reward = b + o_rew;
        d.agent_flags = reinterpret_cast<uint8_t *>(b + o_af);
        d.agent_info = io->agent_info ? reinterpret_cast<uint8_t *>(b + o_ai) : nullptr;
        d.env_flags = reinterpret_cast<uint8_t *>(b + o_ef);
        const bool reuse = c >= ring;
        if (io->actions || io->order) {
            if (reuse) CC_CUDA(cudaStreamWaitEvent(h->s_in, h->ev_k[set], 0));   // the kernel that read this set's actions is done
            if (io->actions) { rc = copy_slices(b + o_act, act_src, A, T, cnt, N, first, true, h->s_in); if (rc != CC_OK) return rc; }
            if (io->order) { rc = copy_slices(b + o_ord, io->order, A, 1, cnt, N, first, true, h->s_in); if (rc != CC_OK) return rc; }
            CC_CUDA(cudaEventRecord(h->ev_in[set], h->s_in));
            CC_CUDA(cudaStreamWaitEvent(h->s_k, h->ev_in[set], 0));
        }
        if (reuse) CC_CUDA(cudaStreamWaitEvent(h->s_k, h->ev_out[set], 0));      // this set's previous outputs have left
        rc = rollout_on(h, &d, h->s_k, T, first, cnt, cnt, t0);
        if (rc != CC_OK) return rc;
        CC_CUDA(cudaEventRecord(h->ev_k[set], h->s_k));
        CC_CUDA(cudaStreamWaitEvent(h->s_out, h->ev_k[set], 0));
        // the biggest output first, the per-env flags last
        if (obs_b) {
            rc = copy_slices(expand ? h->host_table : dst_of(io->obs), d.obs, obs_b, T, cnt, N, first, false, h->s_out);
            if (rc != CC_OK) return rc;
            if (expand) CC_CUDA(cudaEventRecord(h->ev_chunk[c], h->s_out));
        }
        rc = copy_slices(dst_of(io->reward), d.reward, rew_b, T, cnt, N, first, false, h->s_out); if (rc != CC_OK) return rc;
        rc = copy_slices(dst_of(io->agent_flags), d.agent_flags, A, T, cnt, N, first, false, h->s_out); if (rc != CC_OK) return rc;
        if (io->agent_info) { rc = copy_slices(dst_of(io->agent_info), d.agent_info, A, T, cnt, N, first, false, h->s_out); if (rc != CC_OK) return rc; }
        if (io->actions_out) { rc = copy_slices(dst_of(io->actions_out), d.actions_out, A, T, cnt, N, first, false, h->s_out); if (rc != CC_OK) return rc; }
        rc = copy_slices(dst_of(io->env_flags), d.env_flags, 1, T, cnt, N, first, false, h->s_out); if (rc != CC_OK) return rc;
        CC_CUDA(cudaEventRecord(h->ev_out[set], h->s_out));
        if (n_mir) CC_CUDA(cudaEventRecord(h->ev_done[c], h->s_out));
    }
    return CC_OK;
    };
    rc = enqueue_all();
    if (rc != CC_OK) {
        cudaStreamSynchronize(h->s_in); cudaStreamSynchronize(h->s_k); cudaStreamSynchronize(h->s_out);
        return rc;
    }
    h->t = t0 + (uint64_t)T;
    if (expand || n_mir) {
        // The chunks are cut into slices of 4,096 envs that the threads take in order from one counter (a thread that was held up
        // does not hold up a chunk).  Pass 1: the rows of a slice are rebuilt once the chunk's table has arrived (later chunks are
        // still in flight); pass 2: the mirrored outputs of a slice are copied out once all of the chunk's copies have completed.
        const size_t row_b = obs_env_bytes(A, io->obs_dtype);
        h->last_host[2] = expand ? crew : 0;
        std::atomic<int> cuda_err{(int)cudaSuccess};
        constexpr long long kSlice = 4096;
        const long long slices_per_chunk = (chunk + kSlice - 1) / kSlice, n_slices = slices_per_chunk * n_chunks;
        std::atomic<long long> next_rows{0}, next_out{0};
        run_crew([&](int) {
            cudaSetDevice(h->device);
            for (int pass = expand ? 0 : 1; pass < (n_mir ? 2 : 1); ++pass) {
                std::atomic<long long> &next = pass == 0 ? next_rows : next_out;
                const std::vector<cudaEvent_t> &evs = pass == 0 ? h->ev_chunk : h->ev_done;
                long long synced = -1;   // chunks up to here are known to have arrived (the events complete in order: one stream)
                for (;;) {
                    const long long idx = next.fetch_add(1, std::memory_order_relaxed);
                    if (idx >= n_slices) break;
                    const long long c = idx / slices_per_chunk, first = c * chunk, cnt = (N - first < chunk) ? N - first : chunk;
                    if (c > synced) {
                        const cudaError_t e = cudaEventSynchronize(evs[c]);
                        if (e != cudaSuccess) { cuda_err.store((int)e); return; }
                        synced = c;
                    }
                    const long long a = (idx % slices_per_chunk) * kSlice, b = std::min<long long>(cnt, a + kSlice);
                    if (a >= b) continue;
                    for (int t = 0; t < T; ++t) {
                        const size_t e0 = (size_t)t * N + (size_t)first;
                        if (pass == 0)
                            cc_expand_rows_range(&h->cfg, a, b, static_cast<const int8_t *>(h->host_table) + e0 * obs_b,
                                                 static_cast<char *>(io->obs) + e0 * row_b, io->obs_dtype);
                        else
                            for (int k = 0; k < n_mir; ++k)
                                memcpy(mir[k].user + (e0 + (size_t)a) * mir[k].row_b, mir[k].pinned + (e0 + (size_t)a) * mir[k].row_b, (size_t)(b - a) * mir[k].row_b);
                    }
                }
            }
        });
        if (cuda_err.load() != (int)cudaSuccess) {
            cudaStreamSynchronize(h->s_out);
            return cc_fail(CC_ERR_CUDA, "cudaEventSynchronize(chunk): %s", cudaGetErrorString((cudaError_t)cuda_err.load()));
        }
    }
    CC_CUDA(cudaStreamSynchronize(h->s_out));
    h->order_pending = false;   // the caller's earlier work and this call's are complete
    return CC_OK;
}

int launch_aux(cc_handle *h, int mode, int obs_dtype, bool bitmap, const uint8_t *mask, void *obs, int policy, int8_t *actions_out, cudaStream_t s) {
    KParams p;
    fill_params(h, p, obs_dtype, bitmap, 0, h->n_envs);
    p.mask = mask; p.obs = obs; p.policy = policy; p.actions_out = actions_out;
    if (mode == ccb::kModeReset && h->reset_rng == CC_RESET_RNG_NUMPY) p.gen = h->gen;
    return cc_launch_lanes(h, p, mode, obs_dtype, s);
}

}  // namespace

extern "C" {

const char *cc_last_error(void) { return g_err; }
int cc_abi_version(void) { return CCB200_ABI_VERSION; }

int cc_create(const cc_config *cfg, int64_t n_envs, int device, int64_t global_env_offset, uint64_t seed, cc_handle **out) {
    if (!cfg || !out) return cc_fail(CC_ERR_INVALID_ARG, "null config or out pointer");
    *out = nullptr;
    const int A = cfg->num_boarding + cfg->num_exiting;
    if (cfg->num_boarding < 0 || cfg->num_exiting < 0 || A < 1 || A > CC_MAX_AGENTS)
        return cc_fail(CC_ERR_UNSUPPORTED, "agents per env must be in 1..%d, got %d", CC_MAX_AGENTS, A);
    if (n_envs < 1) return cc_fail(CC_ERR_INVALID_ARG, "n_envs must be positive");
    if (n_envs * (int64_t)A >= (int64_t)1 << 31) return cc_fail(CC_ERR_UNSUPPORTED, "n_envs * agents must stay below 2^31 per handle (32-bit slot indices)");
    const int32_t geo[] = {cfg->width, cfg->height, cfg->division_y, cfg->tram_left, cfg->tram_right, cfg->door_left, cfg->door_right, cfg->boarding_dest_y, cfg->exiting_dest_y};
    for (int32_t v : geo)
        if (v < -1 || v > ccb::kMaxGeom) return cc_fail(CC_ERR_UNSUPPORTED, "geometry value %d is outside the supported lattice (0..%d)", v, ccb::kMaxGeom);
    if (cfg->width < 1 || cfg->height < 1) return cc_fail(CC_ERR_INVALID_ARG, "width and height must be positive");
    if (cfg->reward_kind < 0 || cfg->reward_kind > CC_REWARD_CONSTANT_NEGATIVE) return cc_fail(CC_ERR_INVALID_ARG, "unknown reward_kind %d", cfg->reward_kind);
    if (cfg->terminated_kind < 0 || cfg->terminated_kind > CC_TERM_ALL_AT_DESTINATION) return cc_fail(CC_ERR_INVALID_ARG, "unknown terminated_kind %d", cfg->terminated_kind);
    int count = 0;
    CC_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return cc_fail(CC_ERR_INVALID_ARG, "device %d out of range (%d visible)", device, count);
    DeviceGuard guard(device);

    cc_handle *h = new (std::nothrow) cc_handle();
    if (!h) return cc_fail(CC_ERR_NOMEM, "out of host memory");
    h->cfg = *cfg; h->n_envs = n_envs; h->device = device; h->genv_offset = global_env_offset; h->seed = seed; h->A = A;
    h->lpe = 4; while (h->lpe < A && h->lpe < 32) h->lpe <<= 1;
    h->apl = A <= 32 ? 1 : (A <= 64 ? 2 : 4);
    h->epw = 32 / h->lpe;
    cudaError_t e = cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) { delete h; return cc_fail(CC_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e)); }

    const size_t na = (size_t)n_envs * A;
    const size_t o_x = 0, o_y = align256(o_x + na), o_f = align256(o_y + na), o_s = align256(o_f + na),
                 o_r = align256(o_s + (size_t)n_envs * 4), o_st = align256(o_r + (size_t)n_envs * 4),
                 o_e = align256(o_st + ccb::kStCount * 8), o_c = align256(o_e + 4), total = align256(o_c + 8);
    e = cudaMalloc(&h->own_block, total);
    if (e != cudaSuccess) { delete h; return cc_fail(CC_ERR_NOMEM, "cudaMalloc(%zu): %s", total, cudaGetErrorString(e)); }
    // (synchronous on the legacy stream, followed by a device-wide wait: the zeroed block is visible to whatever
    // stream — blocking or not — the first call runs on)
    e = cudaMemset(h->own_block, 0, total);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        const int rc = cc_fail(CC_ERR_CUDA, "cc_create: %s", cudaGetErrorString(e));
        cc_destroy(h);
        return rc;
    }
    char *b = static_cast<char *>(h->own_block);
    h->x = reinterpret_cast<int8_t *>(b + o_x); h->y = reinterpret_cast<int8_t *>(b + o_y);
    h->flags = reinterpret_cast<uint8_t *>(b + o_f); h->step = reinterpret_cast<int32_t *>(b + o_s);
    h->ep_ret = reinterpret_cast<float *>(b + o_r); h->stats = reinterpret_cast<unsigned long long *>(b + o_st);
    h->err = reinterpret_cast<int *>(b + o_e);
    h->tpe_counters = reinterpret_cast<unsigned *>(b + o_c);
    h->owns_state = true;
    *out = h;
    return CC_OK;
}

void cc_destroy(cc_handle *h) {
    if (!h) return;
    DeviceGuard guard(h->device);
    cudaDeviceSynchronize();
    if (h->own_block) cudaFree(h->own_block);
    if (h->stage_block) cudaFree(h->stage_block);
    delete h->workers;
    if (h->host_table) cudaFreeHost(h->host_table);
    if (h->host_mirror) cudaFreeHost(h->host_mirror);
    for (cudaEvent_t ev : h->ev_done) cudaEventDestroy(ev);
    for (cudaEvent_t ev : h->ev_chunk) cudaEventDestroy(ev);
    if (h->gen) cudaFree(h->gen);
    if (h->t2_tables) cudaFree(h->t2_tables);
    for (cudaStream_t s : {h->s_in, h->s_k, h->s_out})
        if (s) cudaStreamDestroy(s);
    for (int i = 0; i < cc_handle::kRing; ++i)
        for (cudaEvent_t ev : {h->ev_in[i], h->ev_k[i], h->ev_out[i]})
            if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : {h->ev0, h->ev1, h->ev_order})
        if (ev) cudaEventDestroy(ev);
    delete h;
}

int cc_attach_state(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step, float *episode_return) {
    if (!h || !x || !y || !flags || !step || !episode_return) return cc_fail(CC_ERR_INVALID_ARG, "cc_attach_state: null pointer");
    h->x = x; h->y = y; h->flags = flags; h->step = step; h->ep_ret = episode_return;
    h->owns_state = false;
    return CC_OK;
}

static int copy_state(cc_handle *h, int8_t *x, int8_t *y, uint8_t *f, int32_t *st, bool to_device, cudaMemcpyKind kind, cudaStream_t s, bool sync) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    DeviceGuard guard(h->device);
    const size_t na = (size_t)h->n_envs * h->A;
    struct Item { void *dev; void *other; size_t bytes; } items[] = {
        {h->x, x, na}, {h->y, y, na}, {h->flags, f, na}, {h->step, st, (size_t)h->n_envs * 4}};
    if (sync && h->order_pending) CC_CUDA(cudaStreamWaitEvent(s, h->ev_order, 0));   // host variants run on the legacy stream
    for (auto &it : items) {
        if (!it.other) continue;
        if (to_device) CC_CUDA(cudaMemcpyAsync(it.dev, it.other, it.bytes, kind, s));
        else CC_CUDA(cudaMemcpyAsync(it.other, it.dev, it.bytes, kind, s));
    }
    if (to_device) CC_CUDA(cudaMemsetAsync(h->ep_ret, 0, (size_t)h->n_envs * 4, s));
    if (sync) CC_CUDA(cudaStreamSynchronize(s));
    return mark_order(h, s);
}
int cc_set_state(cc_handle *h, const int8_t *x, const int8_t *y, const uint8_t *flags, const int32_t *step, void *stream) {
    return copy_state(h, const_cast<int8_t *>(x), const_cast<int8_t *>(y), const_cast<uint8_t *>(flags), const_cast<int32_t *>(step), true,
                      cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream), false);
}
int cc_get_state(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step, void *stream) {
    return copy_state(h, x, y, flags, step, false, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream), false);
}
int cc_set_state_host(cc_handle *h, const int8_t *x, const int8_t *y, const uint8_t *flags, const int32_t *step) {
    return copy_state(h, const_cast<int8_t *>(x), const_cast<int8_t *>(y), const_cast<uint8_t *>(flags), const_cast<int32_t *>(step), true,
                      cudaMemcpyHostToDevice, nullptr, true);
}
int cc_get_state_host(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step) {
    return copy_state(h, x, y, flags, step, false, cudaMemcpyDeviceToHost, nullptr, true);
}

int cc_order_after(cc_handle *h, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    DeviceGuard guard(h->device);
    return mark_order(h, static_cast<cudaStream_t>(stream));
}

int cc_step(cc_handle *h, const cc_step_io *io, void *stream) {
    int rc = check_io(h, io);
    if (rc == CC_OK) rc = check_obs_alignment(io);
    if (rc != CC_OK) return rc;
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    rc = rollout_on(h, io, s, 1, 0, h->n_envs, h->n_envs, h->t);
    if (rc != CC_OK) return rc;
    h->t += 1;
    return mark_order(h, s);
}

int cc_rollout(cc_handle *h, const cc_step_io *io, int32_t n_steps, void *stream) {
    int rc = check_io(h, io);
    if (rc == CC_OK) rc = check_obs_alignment(io);
    if (rc != CC_OK) return rc;
    if (n_steps < 0) return cc_fail(CC_ERR_INVALID_ARG, "n_steps must be non-negative");
    if (io->policy == CC_POLICY_EXTERNAL) return cc_fail(CC_ERR_INVALID_ARG, "cc_rollout needs an on-device policy");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (int i = 0; i < n_steps; ++i) {
        rc = rollout_on(h, io, s, 1, 0, h->n_envs, h->n_envs, h->t);
        if (rc != CC_OK) return rc;
        h->t += 1;
    }
    return mark_order(h, s);
}

int cc_rollout_fused(cc_handle *h, const cc_step_io *io, int32_t n_steps, void *stream) {
    int rc = check_io(h, io);
    if (rc == CC_OK) rc = check_obs_alignment(io);
    if (rc != CC_OK) return rc;
    if (n_steps < 1) return cc_fail(CC_ERR_INVALID_ARG, "n_steps must be positive");
    if (io->order) return cc_fail(CC_ERR_INVALID_ARG, "cc_rollout_fused moves agents in agent order (io->order must be NULL)");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    rc = rollout_on(h, io, s, n_steps, 0, h->n_envs, h->n_envs, h->t);
    if (rc != CC_OK) return rc;
    h->t += (uint64_t)n_steps;
    return mark_order(h, s);
}

int cc_step_host(cc_handle *h, const cc_step_io *io) { return host_pipeline(h, io, 1); }
int cc_rollout_host(cc_handle *h, const cc_step_io *io, int32_t n_steps) { return host_pipeline(h, io, n_steps); }
int cc_set_host_expand(cc_handle *h, int32_t n_threads) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    if (n_threads < CC_HOST_EXPAND_AUTO) return cc_fail(CC_ERR_INVALID_ARG, "cc_set_host_expand: n_threads must be >= 0, CC_HOST_EXPAND_ALL or CC_HOST_EXPAND_AUTO, got %d", n_threads);
    h->host_expand = n_threads;
    return CC_OK;
}
int cc_set_host_chunk(cc_handle *h, int64_t chunk_envs) {
    if (!h || chunk_envs < 0) return cc_fail(CC_ERR_INVALID_ARG, "cc_set_host_chunk: null handle or negative chunk");
    h->host_chunk = chunk_envs;
    return CC_OK;
}

int cc_reset(cc_handle *h, const uint8_t *mask, void *obs, int32_t obs_dtype, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    if (obs_dtype != CC_OBS_NONE && !obs) return cc_fail(CC_ERR_INVALID_ARG, "obs_dtype set but obs is null");
    if (!obs) obs_dtype = CC_OBS_NONE;
    if (obs && (reinterpret_cast<uintptr_t>(obs) & 15)) return cc_fail(CC_ERR_INVALID_ARG, "obs must be 16-byte aligned");
    int rc = check_reset_rng(h, true);
    if (rc != CC_OK) return rc;
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    rc = launch_aux(h, ccb::kModeReset, obs_dtype, false, mask, obs, CC_POLICY_EXTERNAL, nullptr, s);
    if (rc != CC_OK) return rc;
    h->t += 1;
    return mark_order(h, s);
}

int cc_observe(cc_handle *h, void *obs, int32_t obs_dtype, void *stream) {
    if (!h || !obs) return cc_fail(CC_ERR_INVALID_ARG, "null handle or obs");
    if (reinterpret_cast<uintptr_t>(obs) & 15) return cc_fail(CC_ERR_INVALID_ARG, "obs must be 16-byte aligned");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = launch_aux(h, ccb::kModeObserve, obs_dtype, false, nullptr, obs, CC_POLICY_EXTERNAL, nullptr, s);
    return rc != CC_OK ? rc : mark_order(h, s);
}

int cc_policy_actions(cc_handle *h, int32_t policy, int8_t *actions_out, void *stream) {
    if (!h || !actions_out) return cc_fail(CC_ERR_INVALID_ARG, "null handle or actions_out");
    if (policy < CC_POLICY_RANDOM || policy > CC_POLICY_WAITING) return cc_fail(CC_ERR_INVALID_ARG, "cc_policy_actions needs an on-device policy");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = launch_aux(h, ccb::kModePolicy, CC_OBS_NONE, policy != CC_POLICY_RANDOM, nullptr, nullptr, policy, actions_out, s);
    return rc != CC_OK ? rc : mark_order(h, s);
}

int cc_reset_seeded(cc_handle *h, const int64_t *seeds, void *obs, int32_t obs_dtype, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    if (!seeds && !h->gen_seeded) return cc_fail(CC_ERR_INVALID_ARG, "cc_reset_seeded(seeds = NULL) continues the stored generators: seed them first");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!h->gen) {
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->gen), (size_t)h->n_envs * cc_rng_state_bytes());
        if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaMalloc for generator states: %s", cudaGetErrorString(e));
    }
    KParams p;
    fill_params(h, p, CC_OBS_NONE, false, 0, h->n_envs);
    int rc = cc_launch_reset_seeded(h, p, seeds, s);
    if (rc != CC_OK) return rc;
    h->gen_seeded = true;
    if (obs && obs_dtype != CC_OBS_NONE) return cc_observe(h, obs, obs_dtype, stream);
    return mark_order(h, s);
}

int cc_get_rng_state(cc_handle *h, uint64_t *out, void *stream) {
    if (!h || !out) return cc_fail(CC_ERR_INVALID_ARG, "null handle or out");
    if (!h->gen || !h->gen_seeded) return cc_fail(CC_ERR_INVALID_ARG, "cc_get_rng_state: the generators were never seeded (cc_reset_seeded with seeds, or cc_set_rng_state)");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CC_CUDA(cudaMemcpyAsync(out, h->gen, (size_t)h->n_envs * cc_rng_state_bytes(), cudaMemcpyDeviceToDevice, s));
    return mark_order(h, s);
}
int cc_set_rng_state(cc_handle *h, const uint64_t *in, void *stream) {
    if (!h || !in) return cc_fail(CC_ERR_INVALID_ARG, "null handle or in");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!h->gen) {
        cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->gen), (size_t)h->n_envs * cc_rng_state_bytes());
        if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaMalloc for generator states: %s", cudaGetErrorString(e));
    }
    CC_CUDA(cudaMemcpyAsync(h->gen, in, (size_t)h->n_envs * cc_rng_state_bytes(), cudaMemcpyDeviceToDevice, s));
    h->gen_seeded = true;
    return mark_order(h, s);
}
int32_t cc_rng_seeded(const cc_handle *h) { return (h && h->gen_seeded) ? 1 : 0; }
int cc_set_reset_rng(cc_handle *h, int32_t source) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    if (source != CC_RESET_RNG_PHILOX && source != CC_RESET_RNG_NUMPY) return cc_fail(CC_ERR_INVALID_ARG, "unknown reset generator %d", source);
    h->reset_rng = source;
    return CC_OK;
}
int32_t cc_reset_rng(const cc_handle *h) { return h ? h->reset_rng : CC_RESET_RNG_PHILOX; }

int cc_stats_read(cc_handle *h, cc_stats *out, void *stream) {
    if (!h || !out) return cc_fail(CC_ERR_INVALID_ARG, "null handle or out");
    DeviceGuard guard(h->device);
    static_assert(sizeof(cc_stats) == ccb::kStCount * 8, "cc_stats layout");
    CC_CUDA(cudaMemcpyAsync(out, h->stats, sizeof(cc_stats), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    CC_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    return CC_OK;
}
int cc_stats_copy(cc_handle *h, void *out_device, void *stream) {
    if (!h || !out_device) return cc_fail(CC_ERR_INVALID_ARG, "null handle or out");
    DeviceGuard guard(h->device);
    CC_CUDA(cudaMemcpyAsync(out_device, h->stats, sizeof(cc_stats), cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream)));
    return CC_OK;
}
int cc_stats_reset(cc_handle *h, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    DeviceGuard guard(h->device);
    CC_CUDA(cudaMemsetAsync(h->stats, 0, ccb::kStCount * 8, static_cast<cudaStream_t>(stream)));
    return mark_order(h, static_cast<cudaStream_t>(stream));
}
int cc_check_error(cc_handle *h, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    DeviceGuard guard(h->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int bits = 0;
    CC_CUDA(cudaMemcpyAsync(&bits, h->err, sizeof bits, cudaMemcpyDeviceToHost, s));
    CC_CUDA(cudaStreamSynchronize(s));
    if (!bits) return CC_OK;
    CC_CUDA(cudaMemsetAsync(h->err, 0, sizeof bits, s));
    if (bits & ccb::kErrInvalidAction)
        return cc_fail(CC_ERR_INVALID_ACTION, "Invalid action: some action is outside the valid actions [0, 1, 2, 3, 4] (or an order entry names an unknown agent)");
    return cc_fail(CC_ERR_RESET_STUCK, "reset(): no free valid cell found within %d attempts for some agent", ccb::kResetAttemptCap);
}

int64_t cc_num_envs(const cc_handle *h) { return h ? h->n_envs : 0; }
int32_t cc_num_agents(const cc_handle *h) { return h ? h->A : 0; }
int32_t cc_obs_len(const cc_handle *h) { return h ? 6 + 4 * h->A : 0; }
uint64_t cc_step_counter(const cc_handle *h) { return h ? h->t : 0; }
int cc_set_step_counter(cc_handle *h, uint64_t t) { if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle"); h->t = t; return CC_OK; }
int64_t cc_launch_count(const cc_handle *h) { return h ? h->launches : 0; }
int cc_set_kernel_variant(cc_handle *h, int32_t variant) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    if (variant != CC_KERNEL_AUTO && variant != CC_KERNEL_LANES && variant != CC_KERNEL_THREADS) return cc_fail(CC_ERR_INVALID_ARG, "unknown kernel variant %d", variant);
    h->variant = variant;
    return CC_OK;
}
int32_t cc_last_kernel_variant(const cc_handle *h) { return h ? h->last_variant : 0; }
const char *cc_last_kernel_name(const cc_handle *h) { return h ? h->last_kernel : ""; }
int cc_last_host_call(const cc_handle *h, int64_t out[5]) {
    if (!h || !out) return cc_fail(CC_ERR_INVALID_ARG, "cc_last_host_call: null pointer");
    for (int k = 0; k < 5; ++k) out[k] = h->last_host[k];
    return CC_OK;
}

int cc_timing_begin(cc_handle *h, void *stream) {
    if (!h) return cc_fail(CC_ERR_INVALID_ARG, "null handle");
    DeviceGuard guard(h->device);
    CC_CUDA(cudaEventRecord(h->ev0, static_cast<cudaStream_t>(stream)));
    return CC_OK;
}
int cc_timing_end(cc_handle *h, void *stream, float *total_ms) {
    if (!h || !total_ms) return cc_fail(CC_ERR_INVALID_ARG, "null handle or out");
    DeviceGuard guard(h->device);
    CC_CUDA(cudaEventRecord(h->ev1, static_cast<cudaStream_t>(stream)));
    CC_CUDA(cudaEventSynchronize(h->ev1));
    CC_CUDA(cudaEventElapsedTime(total_ms, h->ev0, h->ev1));
    return CC_OK;
}

int cc_device_alloc(int device, size_t bytes, void **ptr, int32_t *compressed) {
    if (!ptr || !compressed) return cc_fail(CC_ERR_INVALID_ARG, "cc_device_alloc: null pointer");
    if (bytes == 0) return cc_fail(CC_ERR_INVALID_ARG, "cc_device_alloc: bytes must be positive");
    *ptr = nullptr;
    *compressed = 0;
    int count = 0;
    CC_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return cc_fail(CC_ERR_INVALID_ARG, "device %d out of range (%d visible)", device, count);
    DeviceGuard guard(device);
    const DriverApi &d = driver_api();
    void *p = nullptr;
    size_t mapped = 0;
    unsigned long long handle = 0;
    int supported = 0;
    if (d.ok && d.cuDeviceGetAttribute(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, device) == CUDA_SUCCESS && supported) {
        CUmemAllocationProp prop = {};
        prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
        prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        prop.location.id = device;
        prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
        size_t gran = 0;
        CUmemGenericAllocationHandle h = 0;
        CUmemAllocationProp got = {};
        if (d.cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) == CUDA_SUCCESS && gran) {
            const size_t size = (bytes + gran - 1) / gran * gran;
            // the driver may grant plain memory (or none) instead: then this buffer comes from cudaMalloc
            if (d.cuMemCreate(&h, size, &prop, 0) == CUDA_SUCCESS) {
                CUdeviceptr va = 0;
                CUmemAccessDesc acc = {};
                acc.location = prop.location;
                acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
                if (d.cuMemGetAllocationPropertiesFromHandle(&got, h) == CUDA_SUCCESS && got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC &&
                    d.cuMemAddressReserve(&va, size, gran, 0, 0) == CUDA_SUCCESS) {
                    if (d.cuMemMap(va, size, 0, h, 0) == CUDA_SUCCESS) {
                        if (d.cuMemSetAccess(va, size, &acc, 1) == CUDA_SUCCESS) {
                            p = reinterpret_cast<void *>(va);
                            mapped = size;
                            handle = h;
                        } else {
                            d.cuMemUnmap(va, size);
                        }
                    }
                    if (!p) d.cuMemAddressFree(va, size);
                }
                if (!p) d.cuMemRelease(h);
            }
        }
    }
    if (!p) {
        const cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cc_fail(CC_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    }
    // Zero-initialised, like the tensors this memory replaces.  The fill goes to the legacy default stream, which a
    // non-blocking caller stream (torch.cuda.Stream()) does not wait for: it must be complete before this returns, or a
    // kernel launched right after on such a stream could race with it and have its outputs zeroed.
    cudaError_t e = cudaMemsetAsync(p, 0, bytes, cudaStreamLegacy);
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    if (e == cudaSuccess) {
        std::lock_guard<std::mutex> lock(g_alloc_mu);
        g_allocs.push_back({p, mapped, handle, device});
    } else {
        if (mapped) {
            d.cuMemUnmap(reinterpret_cast<CUdeviceptr>(p), mapped);
            d.cuMemAddressFree(reinterpret_cast<CUdeviceptr>(p), mapped);
            d.cuMemRelease(handle);
        } else {
            cudaFree(p);
        }
        return cc_fail(CC_ERR_CUDA, "zero fill of %zu bytes: %s", bytes, cudaGetErrorString(e));
    }
    *ptr = p;
    *compressed = mapped ? 1 : 0;
    return CC_OK;
}

int cc_device_free(void *ptr) {
    if (!ptr) return CC_OK;
    DeviceAlloc a = {};
    {
        std::lock_guard<std::mutex> lock(g_alloc_mu);
        auto it = std::find_if(g_allocs.begin(), g_allocs.end(), [&](const DeviceAlloc &x) { return x.ptr == ptr; });
        if (it == g_allocs.end()) return cc_fail(CC_ERR_INVALID_ARG, "cc_device_free: %p was not allocated by cc_device_alloc", ptr);
        a = *it;
    }
    DeviceGuard guard(a.device);
    if (!a.mapped) {
        CC_CUDA(cudaFree(ptr));
    } else {
        // cudaFree waits for the device before it releases memory; unmapping must too (a launch queued on any stream
        // may still write here).  The library does not know which streams used the buffer, so it waits for all of them.
        CC_CUDA(cudaDeviceSynchronize());
        const DriverApi &d = driver_api();
        const CUdeviceptr va = reinterpret_cast<CUdeviceptr>(ptr);
        if (d.cuMemUnmap(va, a.mapped) != CUDA_SUCCESS || d.cuMemAddressFree(va, a.mapped) != CUDA_SUCCESS || d.cuMemRelease(a.handle) != CUDA_SUCCESS)
            return cc_fail(CC_ERR_CUDA, "cc_device_free: releasing the compressible allocation at %p failed", ptr);
    }
    // forgotten only once released: a failed free (e.g. during stream capture) can be repeated
    std::lock_guard<std::mutex> lock(g_alloc_mu);
    auto it = std::find_if(g_allocs.begin(), g_allocs.end(), [&](const DeviceAlloc &x) { return x.ptr == ptr; });
    if (it != g_allocs.end()) g_allocs.erase(it);
    return CC_OK;
}

}  // extern "C"
