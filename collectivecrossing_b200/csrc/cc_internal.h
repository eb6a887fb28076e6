// cc_internal.h — what the translation units of libccb200.so share: the handle, the error helper and the
// launchers of the two kernel families (each family is compiled in its own .cu so that `make -j` builds
// them in parallel).  Nothing here is part of the ABI (include/ccb200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "../../include/ccb200.h"

class cc_worker_pool;   // cc_workers.h
namespace ccb {
struct KParams;
struct Pcg64State;
}  // namespace ccb

int cc_fail(int code, const char *fmt, ...);   // stores the thread-local message, returns `code`
#define CC_CUDA(expr)                                                                                \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess) return cc_fail(CC_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

// launch configuration of one kernel instantiation at one dynamic shared-memory size: queried once per handle
// (cudaFuncSetAttribute + cudaOccupancyMaxActiveBlocksPerMultiprocessor cost more than a 65,536-env step)
struct cc_launch_cfg {
    const void *fn;
    int threads, smem;
    int per_sm;
};

struct cc_handle {
    cc_config cfg;
    int64_t n_envs = 0;
    int device = 0;
    int64_t genv_offset = 0;
    uint64_t seed = 0;
    uint64_t t = 0;  // launches of step/reset so far: the RNG counter word
    int A = 0, lpe = 0, apl = 0, epw = 0, sm_count = 0;
    // persistent state (owned unless attached)
    int8_t *x = nullptr, *y = nullptr;
    uint8_t *flags = nullptr;
    int32_t *step = nullptr;
    float *ep_ret = nullptr;
    bool owns_state = false;
    void *own_block = nullptr;
    unsigned long long *stats = nullptr;
    int *err = nullptr;
    ccb::Pcg64State *gen = nullptr;  // per-env numpy-compatible generators (allocated on first seeded reset)
    bool gen_seeded = false;
    int reset_rng = CC_RESET_RNG_PHILOX;   // cc_set_reset_rng: where the unseeded placements come from
    int64_t launches = 0;
    unsigned *tpe_counters = nullptr;   // two work counters of the thread-per-env kernel (launch parity)
    int64_t tpe_launches = 0;
    int variant = CC_KERNEL_AUTO;   // cc_set_kernel_variant
    int last_variant = 0;           // mapping of the last step launch (CC_KERNEL_LANES / CC_KERNEL_THREADS)
    char last_kernel[64] = "";      // name of the last step kernel launched (cc_last_kernel_name)
    std::vector<cc_launch_cfg> launch_cfgs;
    void *t2_tables = nullptr;      // tables of the small-lattice kernel (built on first use; the config is immutable)
    // stream order (header, "Stream order"): recorded behind every stream-taking call, awaited by the host path
    cudaEvent_t ev_order = nullptr;
    bool order_pending = false;
    // host path: three streams, a ring of staging sets, events per set
    static constexpr int kRing = 3;
    void *stage_block = nullptr;
    size_t stage_bytes = 0;
    cudaStream_t s_in = nullptr, s_k = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[kRing] = {}, ev_k[kRing] = {}, ev_out[kRing] = {};
    int64_t host_chunk = 0;   // cc_set_host_chunk (0 = automatic)
    int host_expand = CC_HOST_EXPAND_AUTO;   // cc_set_host_expand: threads that rebuild observation rows on the host (0 = rows cross PCIe)
    void *host_table = nullptr;          // pinned scratch of the tables the host expands
    size_t host_table_bytes = 0;
    void *host_mirror = nullptr;         // pinned mirrors of the caller's pageable buffers
    size_t host_mirror_bytes = 0;
    std::vector<cudaEvent_t> ev_chunk;   // one event per chunk: its observation table is complete in host memory
    std::vector<cudaEvent_t> ev_done;    // one event per chunk: all its outputs are complete in host memory
    int64_t last_host[5] = {};           // cc_last_host_call: chunks, envs per chunk, expanding threads, H2D bytes, D2H bytes
    cc_worker_pool *workers = nullptr;   // the threads that expand (created by the first call that needs them)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // cc_timing_*
};

// cc_expand.cpp: rows of envs [e0, e1) of `table` into `obs` on the calling thread; threads a job of n_envs is worth
void cc_expand_rows_range(const cc_config *cfg, int64_t e0, int64_t e1, const int8_t *table, void *obs, int32_t obs_dtype);
int cc_host_threads(void);
int cc_expand_thread_count(int32_t requested, int64_t n_envs);
bool cc_expand_beats_pcie(const cc_config *cfg, int32_t obs_dtype);

// `per_sm` resident CTAs of kernel `fn` with `threads` threads and `smem` bytes of dynamic shared memory (cached);
// opts the kernel in to `smem` when it exceeds what the default limit leaves beside the static tables
int cc_cached_occupancy(cc_handle *h, const void *fn, int threads, int smem, int *per_sm);

// cc_launch_lanes.cu: one lane per agent (any crew up to CC_MAX_AGENTS); mode is a ccb::Mode
int cc_launch_lanes(cc_handle *h, const ccb::KParams &p, int mode, int obs_dtype, cudaStream_t s);
// cc_launch_tpe.cu: one thread per env (crews of at most 8); n_steps >= 1
int cc_launch_tpe(cc_handle *h, const ccb::KParams &p, int obs_dtype, cudaStream_t s);
// cc_reset_seeded_kernel (numpy-exact PCG64 placement), in cc_launch_lanes.cu
int cc_launch_reset_seeded(cc_handle *h, const ccb::KParams &p, const int64_t *seeds, cudaStream_t s);
size_t cc_rng_state_bytes(void);   // sizeof(ccb::Pcg64State)
// cc_launch_tpe.cu (part 1): h->t2_tables, built by one block on stream s the first time
int cc_t2_ensure_tables(cc_handle *h, const ccb::KParams &p, cudaStream_t s);
