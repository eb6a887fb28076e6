/*
 * ccb200.h — C ABI of the B200-native batched CollectiveCrossing step/reset path.
 *
 * The reference (nima-siboni/collectivecrossing, pure Python) has no FFI; its
 * boundary for this path is the Python class CollectiveCrossingEnv
 * (src/collectivecrossing/collectivecrossing.py:30-261).  Each entry point
 * below names the reference interface it replaces.  Plain pointers and sizes
 * only; no torch / C++ types cross this boundary.  Every function returns
 * CC_OK (0) or a negative cc_status; the message is available through
 * cc_last_error() (thread-local).  No C++ exception crosses the ABI.
 *
 * Threading: one handle is bound to one CUDA device.  Calls on one handle must
 * be serialised by the caller (stream order); distinct handles may be driven
 * from distinct threads / processes (one process per GPU under torchrun).
 *
 * Buffers: unless stated otherwise every pointer is a DEVICE pointer on the
 * handle's device, borrowed for the duration of the call.  The *_host entry
 * points take HOST pointers (pinned or pageable) and perform the copies.
 *
 * Stream order: every call that takes a `stream` enqueues its work there and
 * returns without waiting; calls on one handle must be issued in the order
 * they are meant to run.  The handle records an event behind each of them, and
 * the *_host entry points (which use the handle's own copy / compute streams)
 * wait for that event first and return only when their outputs are complete —
 * so step() / reset() on a caller stream followed by step_host() needs no
 * synchronisation by the caller.  A caller that switches from one stream to
 * another between two calls orders the two streams itself.
 */
#ifndef CCB200_H
#define CCB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCB200_ABI_VERSION 2
#define CC_MAX_AGENTS 128 /* num_boarding + num_exiting supported by the kernels */

typedef enum cc_status {
    CC_OK = 0,
    CC_ERR_INVALID_ARG = -1,
    CC_ERR_CUDA = -2,
    CC_ERR_UNSUPPORTED = -3,
    CC_ERR_INVALID_ACTION = -4, /* some action outside {0..4}: reference raises ValueError
                                   (collectivecrossing.py:707-711) */
    CC_ERR_RESET_STUCK = -5,    /* rejection sampling of reset() hit the attempt cap */
    CC_ERR_NOMEM = -6
} cc_status;

/* rewards.py:186-191 (REWARD_FUNCTIONS registry) */
typedef enum cc_reward_kind {
    CC_REWARD_DEFAULT = 0,           /* rewards.py:41-99   */
    CC_REWARD_SIMPLE_DISTANCE = 1,   /* rewards.py:102-129 */
    CC_REWARD_BINARY = 2,            /* rewards.py:132-159 */
    CC_REWARD_CONSTANT_NEGATIVE = 3  /* rewards.py:162-182 */
} cc_reward_kind;

/* terminateds.py:86-89 (TERMINATED_FUNCTIONS registry) */
typedef enum cc_terminated_kind {
    CC_TERM_INDIVIDUAL_AT_DESTINATION = 0, /* terminateds.py:63-82 */
    CC_TERM_ALL_AT_DESTINATION = 1         /* terminateds.py:37-60 */
} cc_terminated_kind;

/* what `obs` receives.  INT8 / FP32: the reference's observation tensor [N,A,6+4A] (the value is the
 * element size, s_obs in SURVEY.md §8d).  TABLE: the compact form of the same information (s_obs = 0
 * of SURVEY.md §8d): per env the int8 table [A][4] = (x_j, y_j, type_j, active_j) of
 * observations.py:80-91; every row of observations.py:62-94 is this table with block i replaced by
 * -1, preceded by (x_i, y_i) and four per-config constants — cc_expand_obs_host rebuilds the rows. */
typedef enum cc_obs_dtype {
    CC_OBS_NONE = 0, /* observations not materialised */
    CC_OBS_INT8 = 1,
    CC_OBS_FP32 = 4, /* the reference's dtype (observations.py:94) */
    CC_OBS_TABLE = 16 /* int8 [N,A,4] */
} cc_obs_dtype;

typedef enum cc_reward_dtype {
    CC_REWARD_F32 = 4,
    CC_REWARD_F64 = 8 /* the reference's dtype; used by the single-env facade */
} cc_reward_dtype;

/* where the per-agent actions of a step come from */
typedef enum cc_policy {
    CC_POLICY_EXTERNAL = 0, /* read io->actions (the reference's step(action_dict)) */
    CC_POLICY_RANDOM = 1,   /* uniform {0..4}, Philox4x32-10 keyed (seed, global env, t, agent) */
    CC_POLICY_GREEDY = 2,   /* baseline_policies/greedy_policy.py at randomness_factor 0 */
    CC_POLICY_WAITING = 3   /* baseline_policies/waiting_policy.py at randomness_factor 0 */
} cc_policy;

/* actions.py:8-24 */
enum { CC_ACT_RIGHT = 0, CC_ACT_UP = 1, CC_ACT_LEFT = 2, CC_ACT_DOWN = 3, CC_ACT_WAIT = 4 };

/* persistent per-agent state byte, flags[N][A]  (types.py:16-25: active/terminated/truncated) */
enum { CC_F_ACTIVE = 1, CC_F_TERMINATED = 2, CC_F_TRUNCATED = 4 };

/* per-agent output byte of one step, agent_flags[N][A] */
enum {
    CC_O_ACTIVE = 1,       /* post-step Agent.active                                     */
    CC_O_TERMINATED = 2,   /* post-step sticky Agent.terminated                          */
    CC_O_TRUNCATED = 4,    /* post-step sticky Agent.truncated                           */
    CC_O_ALIVE_PREV = 8,   /* agent was neither terminated nor truncated at step start:  *
                            * rewards[id] and truncateds[id] exist (rewards.py:65-66,    *
                            * truncateds.py:57-58)                                        */
    CC_O_TERM_VALUE = 16,  /* terminateds[id] (always present, terminateds.py:37-82)     */
    CC_O_TRUNC_VALUE = 32, /* truncateds[id]; meaningful only with CC_O_ALIVE_PREV       */
    CC_O_OBS_PRESENT = 64  /* observations[id] / infos[id] exist (collectivecrossing.py:243) */
};

/* per-agent info byte, agent_info[N][A]  (collectivecrossing.py:248-254) */
enum { CC_I_IN_TRAM_AREA = 1, CC_I_AT_DOOR = 2, CC_I_ACTIVE = 4, CC_I_AT_DESTINATION = 8 };

/* per-env output byte, env_flags[N]  (collectivecrossing.py:256-259) */
enum { CC_E_TERMINATED_ALL = 1, CC_E_TRUNCATED_ALL = 2, CC_E_WAS_RESET = 4 };

/*
 * Lowered environment description.  Replaces CollectiveCrossingConfig
 * (configs.py:15-77) + TramBoundaries (utils/geometry.py:10-47) + the reward /
 * terminated / truncated config objects.  All geometry is ABSOLUTE.
 */
typedef struct cc_config {
    int32_t width, height, division_y;
    int32_t tram_left, tram_right, door_left, door_right;
    int32_t boarding_dest_y, exiting_dest_y;
    int32_t num_boarding, num_exiting;
    int32_t max_steps;        /* truncated_configs.py:32-37 */
    int32_t reward_kind;      /* cc_reward_kind */
    int32_t terminated_kind;  /* cc_terminated_kind */
    /* reward parameters, float64 like the reference's Python floats:
     *  DEFAULT           {boarding_destination_reward, tram_door_reward, tram_area_reward,
     *                     distance_penalty_factor}            (reward_configs.py:25-58)
     *  SIMPLE_DISTANCE   {distance_penalty_factor}            (reward_configs.py:61-75)
     *  BINARY            {goal_reward, no_goal_reward}        (reward_configs.py:78-97)
     *  CONSTANT_NEGATIVE {step_penalty}                       (reward_configs.py:100-115) */
    double reward_params[4];
} cc_config;

/* Buffers of one step.  N = envs of the handle, A = num_boarding + num_exiting. */
typedef struct cc_step_io {
    const int8_t *actions;   /* [N,A] in {0..4}; required iff policy == CC_POLICY_EXTERNAL     */
    const int8_t *order;     /* [N,A] nullable: order[n][k] = index of the agent moved k-th     *
                              * (the caller's action_dict order, collectivecrossing.py:197);    *
                              * a negative entry ends the list; NULL = agent order 0..A-1       */
    int8_t *actions_out;     /* [N,A] nullable: the actions that were applied                  */
    void *obs;               /* [N,A,6+4A] of obs_dtype ([N,A,4] int8 for CC_OBS_TABLE), nullable iff CC_OBS_NONE */
    void *reward;            /* [N,A] of reward_dtype (0 where !CC_O_ALIVE_PREV)               */
    uint8_t *agent_flags;    /* [N,A] CC_O_* bits                                               */
    uint8_t *agent_info;     /* [N,A] CC_I_* bits, nullable                                     */
    uint8_t *env_flags;      /* [N]   CC_E_* bits                                               */
    int32_t obs_dtype;       /* cc_obs_dtype */
    int32_t reward_dtype;    /* cc_reward_dtype */
    int32_t policy;          /* cc_policy */
    int32_t auto_reset;      /* != 0: envs whose episode ended are re-sampled in the same launch;
                              * obs then shows the NEW episode, reward/flags the finished one  */
} cc_step_io;

/* Episode statistics accumulated on the device since cc_create / cc_stats_reset.
 * Reduced across ranks by the host (one NCCL all-reduce per rollout chunk). */
typedef struct cc_stats {
    int64_t env_steps;        /* env-steps executed                                   */
    int64_t episodes;         /* episodes finished (terminated_all or truncated_all)  */
    int64_t terminated_all;   /* ... of which ended with terminateds["__all__"]       */
    int64_t truncated_all;    /* ... of which ended with truncateds["__all__"]        */
    int64_t arrivals;         /* agents deactivated at their destination              */
    int64_t episode_length_sum; /* sum of step counts of finished episodes            */
    double episode_return_sum;  /* sum over finished episodes of all agents' rewards  */
    double reward_sum;          /* sum of every reward handed out                     */
} cc_stats;

typedef struct cc_handle cc_handle;

/* --- lifetime ------------------------------------------------------------------------- */

/* Replaces CollectiveCrossingEnv.__init__ (collectivecrossing.py:44-89) for n_envs independent
 * envs on CUDA device `device`.  `global_env_offset` is the index of this shard's env 0 in the
 * whole job (counter-based RNG is keyed on the global index, so results do not depend on the
 * sharding).  The handle allocates its own state; all agents start at (0,0), inactive. */
int cc_create(const cc_config *cfg, int64_t n_envs, int device, int64_t global_env_offset,
              uint64_t seed, cc_handle **out);
void cc_destroy(cc_handle *h);

/* Use caller-owned device buffers for the persistent state instead of the handle's own
 * (x,y int8 [N,A]; flags uint8 [N,A]; step int32 [N]; episode_return float32 [N]).
 * The buffers must outlive the handle or the next cc_attach_state call. */
int cc_attach_state(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step,
                    float *episode_return);

/* --- state injection / checkpoint (tests write env._agents[..] directly, SURVEY.md §4) --- */
/* A NULL array is skipped (partial update / partial read-back); cc_set_state* also zeroes the episode returns. */
int cc_set_state(cc_handle *h, const int8_t *x, const int8_t *y, const uint8_t *flags,
                 const int32_t *step, void *stream);
int cc_get_state(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step, void *stream);
/* same with HOST pointers (synchronous) */
int cc_set_state_host(cc_handle *h, const int8_t *x, const int8_t *y, const uint8_t *flags,
                      const int32_t *step);
int cc_get_state_host(cc_handle *h, int8_t *x, int8_t *y, uint8_t *flags, int32_t *step);

/* --- the hot path --------------------------------------------------------------------- */

/* Replaces CollectiveCrossingEnv.step (collectivecrossing.py:161-261) for all envs of the
 * handle in ONE fused kernel launch on `stream` (a cudaStream_t; NULL = legacy default). */
int cc_step(cc_handle *h, const cc_step_io *io, void *stream);

/* Same with every pointer of `io` a HOST pointer.  Pinned buffers are copied to and from directly; ordinary (malloc / numpy)
 * buffers go through pinned mirrors owned by the handle, filled at link speed and moved to / from the caller's memory by the
 * handle's host threads (a direct copy to pageable memory is staged by the driver inside the calling thread: 3x slower for
 * the compact formats) — unless cc_set_host_expand(h, 0) leaves the handle without host threads.
 * This is the call a non-CUDA caller (numpy, the reference's RLlib env-runner) binds.  The envs
 * are processed in chunks on three streams of the handle — chunk c+1's host->device copy of
 * the actions and its kernel overlap chunk c's device->host copies of the outputs — and the call
 * returns when every output is complete in host memory. */
int cc_step_host(cc_handle *h, const cc_step_io *io);

/* cc_rollout_fused with HOST pointers: n_steps env-steps per env, every output time-major
 * [n_steps][N]... in host memory (io->actions [n_steps][N][A] when the policy is EXTERNAL).  Chunks of
 * envs are rolled out one after the other (one fused launch per chunk where the thread-per-env
 * kernel applies) while the previous chunk's slices stream to the host. */
int cc_rollout_host(cc_handle *h, const cc_step_io *io, int32_t n_steps);

/* Envs per chunk of the host pipeline (0 = automatic: about N/8, a multiple of 32). */
int cc_set_host_chunk(cc_handle *h, int64_t chunk_envs);

/* Row delivery of the host path (CC_OBS_INT8 / CC_OBS_FP32 rows requested in host memory).
 *   n_threads == CC_HOST_EXPAND_OFF (0): the kernel writes the rows and they cross PCIe as they are.
 *   n_threads  > 0 or CC_HOST_EXPAND_ALL (-1): the kernel writes the compact table, the table crosses PCIe
 *       (4A bytes per env instead of s_obs*A*(6+4A)) and the rows are rebuilt in the caller's buffer on n_threads
 *       host threads (ALL: every hardware thread the process may run on), chunk by chunk while later chunks are still on the device.
 *   CC_HOST_EXPAND_AUTO (-2, the state of a new handle): as ALL when the process may run on at least 8 hardware threads, the rows
 *       of one call are at least 16 MiB and rebuilding beats the link — CC_OBS_FP32 rows always (one B200's PCIe link
 *       delivers ~54 GB/s; a thread streams ~10 GB/s of float32 rows, sixteen reach the host's DRAM write rate), CC_OBS_INT8
 *       rows for crews of 8 on x86-64 with SSSE3 (a byte-shuffle path, 27 GB/s per thread; other crews: 4 GB/s per thread,
 *       they keep crossing PCIe) —, as OFF otherwise.
 * The bytes that arrive are identical either way (cc_expand_obs_host is the same code, callable on its own). */
enum { CC_HOST_EXPAND_OFF = 0, CC_HOST_EXPAND_ALL = -1, CC_HOST_EXPAND_AUTO = -2 };
int cc_set_host_expand(cc_handle *h, int32_t n_threads);

/* Make the next *_host call wait for everything enqueued on `stream` so far (for work the library cannot see:
 * a caller that owns the state tensors — cc_attach_state — and writes them with its own kernels or copies). */
int cc_order_after(cc_handle *h, void *stream);

/* Host-side expansion of CC_OBS_TABLE output into the reference's observation rows
 * (observations.py:62-94): table int8 [n_envs][A][4] -> obs [n_envs][A][6+4A] of obs_dtype
 * (CC_OBS_INT8 or CC_OBS_FP32), bit-identical to what the kernels write for that dtype.  Pure
 * data movement on `n_threads` host threads (0 = all hardware threads); no CUDA call. */
int cc_expand_obs_host(const cc_config *cfg, int64_t n_envs, const int8_t *table, void *obs,
                       int32_t obs_dtype, int32_t n_threads);

/* T fused steps with an on-device policy and auto-reset (one launch per step, no host
 * round-trip, outputs of the last step only). */
int cc_rollout(cc_handle *h, const cc_step_io *io, int32_t n_steps, void *stream);

/* T steps whose outputs are ALL kept: every output buffer of `io` (obs, reward, agent_flags,
 * agent_info, env_flags, actions_out) is time-major, [n_steps][...] with the per-step shapes of
 * cc_step_io; io->actions, when policy == CC_POLICY_EXTERNAL, is [n_steps][N][A] as well.  This is
 * the loop "policy -> step -> (reset on done)" of the reference's rollouts
 * (scripts/run_greedy_policy_demo.py:60-95) for N envs.  Where the thread-per-env kernel applies
 * (crews of at most 8, float32 rewards) it is ONE launch: an env's state stays in registers for the T
 * steps and is read and written once; otherwise one launch per step.  Results are identical to T
 * calls of cc_step (same RNG counters). */
int cc_rollout_fused(cc_handle *h, const cc_step_io *io, int32_t n_steps, void *stream);

/* Replaces CollectiveCrossingEnv.reset (collectivecrossing.py:91-159): rejection-sampled
 * placement with the handle's counter-based RNG, or with each env's numpy generator under
 * CC_RESET_RNG_NUMPY (cc_set_reset_rng).  mask: [N] uint8 nullable (NULL = all envs).
 * obs nullable; written for the reset envs only when given. */
int cc_reset(cc_handle *h, const uint8_t *mask, void *obs, int32_t obs_dtype, void *stream);

/* Replaces reset(seed=s) bit-exactly: per-env numpy Generator(PCG64(SeedSequence(seed)))
 * (gymnasium's seeding, used at collectivecrossing.py:95,105-106,134-137).
 * seeds: [N] int64 (device) seeds every env's generator afresh, like reset(seed=s).
 * seeds == NULL is reset() without a seed: every env keeps drawing from the generator it was
 * last seeded with (gymnasium keeps env.np_random across resets); an error before any seeding. */
int cc_reset_seeded(cc_handle *h, const int64_t *seeds, void *obs, int32_t obs_dtype,
                    void *stream);

/* Checkpoint of the per-env numpy-compatible generators cc_reset_seeded keeps (what gymnasium holds
 * in env.np_random): uint64 [N][6] = {state hi, state lo, inc hi, inc lo, buffered uint32,
 * has_buffered}.  cc_get_rng_state fails before the first seeded reset; cc_set_rng_state marks the
 * generators as seeded, so a resumed run's reset() continues the stream of the saved run. */
int cc_get_rng_state(cc_handle *h, uint64_t *out, void *stream);
int cc_set_rng_state(cc_handle *h, const uint64_t *in, void *stream);
/* 1 once the generators hold a stream (after cc_reset_seeded(seeds) or cc_set_rng_state) */
int32_t cc_rng_seeded(const cc_handle *h);

/* Where UNSEEDED placements come from: the auto-reset of cc_step, cc_rollout, cc_rollout_fused, cc_step_host and
 * cc_rollout_host, and cc_reset(mask).
 *   CC_RESET_RNG_PHILOX (default): the counter-based generator keyed (seed, global env, t) — new functionality, the
 *       reference has no auto-reset.
 *   CC_RESET_RNG_NUMPY: the reference's reset() without a seed — env n draws from its own numpy generator (the one
 *       cc_reset_seeded keeps, checkpointed by cc_get_rng_state) and advances it, exactly as cc_reset_seeded(NULL)
 *       does for that env.  N envs each reset(seed=s_n) once and then stepped with reset() on "__all__" reproduce the
 *       reference episode after episode.  A call that may place envs (auto_reset != 0, or cc_reset) fails with
 *       CC_ERR_INVALID_ARG before it enqueues anything until the generators are seeded (cc_reset_seeded(seeds) or
 *       cc_set_rng_state).  The step counter t advances as in Philox mode, so random-policy actions are the same.
 * Results of one mode never depend on the kernel mapping (cc_set_kernel_variant) or on the host path's chunking. */
enum { CC_RESET_RNG_PHILOX = 0, CC_RESET_RNG_NUMPY = 1 };
int cc_set_reset_rng(cc_handle *h, int32_t source);
int32_t cc_reset_rng(const cc_handle *h);

/* The baseline policies alone (greedy_policy.py:33-88, waiting_policy.py:33-72) on the
 * current state: actions_out [N,A] int8; agents that are done or inactive get CC_ACT_WAIT. */
int cc_policy_actions(cc_handle *h, int32_t policy, int8_t *actions_out, void *stream);

/* Observations of the current state without stepping (observations.py:43-94). */
int cc_observe(cc_handle *h, void *obs, int32_t obs_dtype, void *stream);

/* --- bookkeeping ---------------------------------------------------------------------- */
int cc_stats_read(cc_handle *h, cc_stats *out, void *stream); /* synchronises `stream` */
int cc_stats_reset(cc_handle *h, void *stream);
/* The same block without a host round trip: 64 bytes (the cc_stats layout) copied to a DEVICE buffer on `stream`, so that the
 * multi-GPU reduction (one NCCL all-reduce per rollout chunk) can be enqueued behind the step kernels with no synchronisation. */
int cc_stats_copy(cc_handle *h, void *out_device, void *stream);
/* sticky device error raised by kernels since the last call (CC_OK if none); clears it. */
int cc_check_error(cc_handle *h, void *stream);
int64_t cc_num_envs(const cc_handle *h);
int32_t cc_num_agents(const cc_handle *h);
int32_t cc_obs_len(const cc_handle *h); /* 6 + 4A, observations.py:113-118 */
uint64_t cc_step_counter(const cc_handle *h);        /* launches so far (RNG counter t) */
int cc_set_step_counter(cc_handle *h, uint64_t t);   /* for checkpoint / resume */
/* number of kernels the library launched through this handle (bench "gpu_launches") */
int64_t cc_launch_count(const cc_handle *h);
/* Which work mapping cc_step uses.  Both produce identical results (tests/test_gpu_parity.py
 * runs every case through both):
 *   CC_KERNEL_LANES    one lane per agent, 4-32 lanes per env (any crew size, dict order, float64 rewards);
 *   CC_KERNEL_THREADS  one thread per env (crews of at most 8, agent order, float32 rewards; int8 rows: 8 agents);
 *   CC_KERNEL_AUTO     THREADS where eligible, else LANES (default).
 * Requesting CC_KERNEL_THREADS makes ineligible steps fail with CC_ERR_UNSUPPORTED. */
enum { CC_KERNEL_AUTO = 0, CC_KERNEL_LANES = 1, CC_KERNEL_THREADS = 2 };
int cc_set_kernel_variant(cc_handle *h, int32_t variant);
int32_t cc_last_kernel_variant(const cc_handle *h); /* mapping of the last cc_step launch (0 = none yet) */
/* instantiation the last step launch ran, e.g. "ccb::cc_step_tpe_kernel<8,4>" (float32 rows), "ccb::cc_step_tpe2_kernel<8,1>"
 * (the small-lattice kernel of the compact modes) or "ccb::cc_kernel<32,2,1,step>"; "" before the first launch */
const char *cc_last_kernel_name(const cc_handle *h);

/* What the last cc_step_host / cc_rollout_host call did: out[0] chunks, out[1] envs per chunk, out[2] host threads that
 * rebuilt observation rows (0: the rows crossed PCIe as the kernel wrote them), out[3] bytes copied host -> device,
 * out[4] bytes copied device -> host (counted from the copies the call enqueued). */
int cc_last_host_call(const cc_handle *h, int64_t out[5]);
/* average device time (ms) of the step kernel launches bracketed by cc_timing_begin/_end,
 * measured with CUDA events on the launching stream */
int cc_timing_begin(cc_handle *h, void *stream);
int cc_timing_end(cc_handle *h, void *stream, float *total_ms);

/* --- output buffers -------------------------------------------------------------------- */
/* `bytes` of zeroed device memory on `device` for step outputs (the zero fill is complete when the call returns).  Where the device supports compressible memory
 * (CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED) and grants it, the memory is compressible (cuMemCreate with
 * CU_MEM_ALLOCATION_COMP_GENERIC): the hardware compresses it between L2 and DRAM, which cuts the DRAM bytes of the
 * very regular float32 observation rows; every value read or written is unchanged.  Otherwise it is cudaMalloc memory.
 * *compressed is 1 for compressible memory, else 0.  Not shareable through CUDA IPC.  Free with cc_device_free. */
int cc_device_alloc(int device, size_t bytes, void **ptr, int32_t *compressed);
/* Waits for the whole device (like cudaFree), then releases memory from cc_device_alloc (NULL: no-op).  It therefore
 * fails while a stream of the device is being captured into a CUDA graph; the memory then stays allocated and the call
 * can be repeated after the capture. */
int cc_device_free(void *ptr);

const char *cc_last_error(void);
int cc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CCB200_H */
