/*
 * d2d_b200.h - C ABI of libd2d_b200.so: the B200 (sm_100a) batched replacement for GymD2D's per-step
 * radio physics.  Plain C types only; no torch, no C++ in the signatures.
 *
 * The reference (davidcotton/gym-d2d) is pure Python and has no FFI of its own, so each entry point
 * cites the reference *interface* it replaces (paths relative to /root/reference/src/gym_d2d/).  The
 * ctypes stub a maintainer would add on the reference side is shown in INTEGRATION.md.
 *
 * Conventions
 *  - every function returns 0 on success or a negative d2d_status; d2d_last_error() gives the message
 *    of the calling thread's last failure.  Nothing here throws or aborts.
 *  - all device buffers are CALLER-OWNED (PyTorch CUDA allocations in the Python shell) and passed as
 *    raw device pointers; the handle owns only its small constant tables and host staging buffers.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *    stream-ordered and asynchronous unless stated; d2d_step performs no allocation and no host
 *    synchronisation, so it can be captured into a CUDA graph.
 *  - a handle is bound to one CUDA device and is not thread-safe.  Multi-GPU = one process (one
 *    handle) per GPU, each owning a contiguous slice of the global environment batch.  Every entry point
 *    selects the handle's device for the duration of the call and restores the caller's current device.
 *
 * Ordering rule (programmatic dependent launch).  Step kernels are launched with programmatic stream
 * serialisation: a launch may begin while the previous kernel in `stream` is still running and orders itself
 * with griddepcontrol.wait.  By DEFAULT a step kernel executes that wait before it reads anything the caller
 * or another kernel may have written - this step's `actions`, the bound positions - so any producer earlier
 * in `stream` (a policy / sampling kernel, a copy, d2d_reset, d2d_set_positions, d2d_episode) is complete
 * and visible, exactly as with an ordinary launch.  Setting D2D_STEP_INPUTS_STABLE in d2d_step_io.flags is
 * the caller's promise that every write to this step's `actions` and to the positions was enqueued on
 * `stream` BEFORE the previous d2d_step / d2d_step_many call on this handle (or had completed by then): the
 * kernel then loads its inputs and computes the whole step while its predecessor drains, and waits only
 * before touching the step counters and the output buffers.  The library honours the flag only when the
 * previous kernel it enqueued for this handle was a step kernel on the same `stream`; after d2d_reset,
 * d2d_set_positions, d2d_episode, or on a different stream, the next step is ordered the default way
 * whatever the flag says.  Pre-generated action buffers (replay, evaluation, benchmarks, CUDA graphs of
 * scripted steps) may set it; a loop whose policy writes the actions between steps must not.
 * Between two consecutive flagged steps the caller may enqueue work that READS the step's outputs, but nothing
 * that WRITES a buffer either step reads or writes (actions, outputs, the bound positions and step counters):
 * consecutive flagged single-launch steps of the same geometry do not wait for each other as whole grids -
 * each warp waits only for the warp that stepped the same environments one launch earlier (a per-warp
 * release / acquire ticket; gym_d2d_b200/csrc/d2d_common.cuh), which is what removes the grid-wide
 * completion-and-release latency from a chain of small steps.  And when the per-link output buffers of a flagged
 * step (obs, obs_dyn, capacity_mbps, rate_bps, rb, tx_pwr_dBm) overlap none of the previous step's - the library
 * compares the pointers itself - the kernel stores them BEFORE it waits: its predecessor cannot touch them, and
 * anything enqueued ahead of the predecessor is complete.  Only the step counters and the per-env scalars (reward,
 * done) are written after the wait.  A caller that rotates two or more output sets gets this without asking; nothing
 * changes for one that reuses a single set.
 * A step with D2D_STEP_AUTORESET is always ordered the default way, whatever D2D_STEP_INPUTS_STABLE says: it reads
 * every input and the step counters after the wait, stores no output ahead of it and takes no per-warp ticket.  It
 * also writes the positions of the envs it resets, so the step after it is ordered the default way too, as after
 * d2d_episode.
 *
 * Index conventions (devices.py:20-25, simulator.py:34-48, envs/d2d_env.py:55-60):
 *   C = num_cues, D = num_due_pairs, N = C + D links, V = 1 + C + 2D devices.
 *   device 0 = 'mbs'; 1..C = 'cue00'..; pair d: tx = 1+C+2d ('due{2d}'), rx = tx+1 ('due{2d+1}').
 *   link j < C : CUE j -> MBS (UPLINK);  link j >= C : DUE pair j-C (SIDELINK).
 */
#ifndef D2D_B200_H
#define D2D_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
#define D2D_API extern "C" __attribute__((visibility("default")))
#else
#define D2D_API __attribute__((visibility("default")))
#endif

#define D2D_ABI_VERSION 5

typedef struct d2d_handle d2d_handle_t;

typedef enum d2d_status {
    D2D_OK = 0,
    D2D_ERR_INVALID_ARG = -1,   /* bad pointer / size / enum: the shell maps this to ValueError / TypeError */
    D2D_ERR_UNSUPPORTED = -2,   /* configuration outside what the kernels implement */
    D2D_ERR_CUDA = -3,          /* a CUDA runtime call failed; message carries cudaGetErrorString */
    D2D_ERR_STATE = -4          /* state buffers not bound / called out of order */
} d2d_status;

/* path_loss_model plugin (envs/env_config.py:21; classes in path_loss.py:42-66, 90-123).  FREE_SPACE is
 * LogDistancePathLoss with ple = 2 (path_loss.py:43,45): it is not a separate class in the reference.
 * COST_HATA (path_loss.py:90-123) is A(h_tx, h_rx) + B(h_tx) log10(d_km): with one transmitter antenna height it is a
 * log-distance law with exponent ple = B / 10 and a per-receiver constant, both folded by the caller: d2d_config.ple and
 * d2d_link.path_loss_const_dB (= A - 3 B for the link's receiver).
 * SHADOWING (path_loss.py:69-81) is the log-distance law plus gauss(0, shadow_chi_dB) beyond shadow_d0_m, drawn anew at EVERY
 * path-loss evaluation (the own link twice per step: once for the SINR, once for the SNR).  The reference draws from
 * Python's global RNG; here the draws are counter-based (Philox4x32-10 keyed by rng_seed; counter = global env, victim link,
 * source link, evaluation kind, step call number), so only distributions match the reference.  General-topology kernel. */
typedef enum d2d_path_loss_model { D2D_PL_LOG_DISTANCE = 0, D2D_PL_FREE_SPACE = 1, D2D_PL_COST_HATA = 2, D2D_PL_SHADOWING = 3 } d2d_path_loss_model;
/* obs_fn plugin (envs/d2d_env.py:27; envs/obs_fn.py:35-61) */
typedef enum d2d_obs_fn { D2D_OBS_LINEAR = 0 } d2d_obs_fn;
/* reward_fn plugin (envs/d2d_env.py:28).  SYSTEM_CAPACITY (envs/reward_fn.py:22-44) is one scalar per env, computed inside
 * the step kernel.  SHANNON (:47-57, parameter min_sinr) and CUE_SINR_SHANNON (:60-78, parameter sinr_threshold_dB) are per
 * agent: a second small kernel derives them from the step's results into d2d_step_io.agent_reward, and `reward` then
 * holds their mean over the acting agents. */
typedef enum d2d_reward_fn { D2D_REWARD_SYSTEM_CAPACITY = 0, D2D_REWARD_SHANNON = 1, D2D_REWARD_CUE_SINR_SHANNON = 2 } d2d_reward_fn;
/* link_type.py:4-7 */
typedef enum d2d_link_type { D2D_LINK_UPLINK = 1, D2D_LINK_DOWNLINK = 2, D2D_LINK_SIDELINK = 3 } d2d_link_type;

/* The hot-path subset of EnvConfig (envs/env_config.py:12-27) plus the plugin enums. */
typedef struct d2d_config {
    int32_t abi_version;        /* must be D2D_ABI_VERSION */
    int32_t cuda_device;        /* ordinal the handle is bound to */
    int64_t num_envs;           /* E: environments resident on this device */
    int32_t num_rbs;            /* envs/env_config.py:12 */
    int32_t num_cues;           /* :13 */
    int32_t num_due_pairs;      /* :14 */
    int32_t n_pwr_cue;          /* envs/d2d_env.py:33  cue_max_tx_power_dBm + 1 */
    int32_t n_pwr_due;          /* envs/d2d_env.py:32  due_max - due_min + 1 */
    int32_t episode_length;     /* envs/d2d_env.py:16  EPISODE_LENGTH = 10 */
    int32_t path_loss_model;    /* d2d_path_loss_model */
    int32_t obs_fn;             /* d2d_obs_fn */
    int32_t reward_fn;          /* d2d_reward_fn */
    int32_t num_downlinks;      /* 0, or num_cues: links C+D .. C+D+C-1 are the DOWNLINK actions 'mbs:cueXX' (envs/d2d_env.py:87-89,
                                   Appendix B.8: never produced by reset(), accepted by step()); the link table then has 2C + D rows
                                   and the step runs on the general-topology kernel */
    int32_t n_pwr_mbs;          /* envs/d2d_env.py:34  mbs_max_tx_power_dBm + 1 */
    int32_t reserved0;
    double carrier_freq_GHz;    /* envs/env_config.py:23 */
    double ple;                 /* path_loss.py:43 path-loss exponent (ignored, = 2, for FREE_SPACE) */
    double cell_radius_m;       /* envs/env_config.py:15 */
    double d2d_radius_m;        /* :16 */
    double min_capacity_mbps;   /* envs/reward_fn.py:23 */
    double reward_param;        /* SHANNON: min_sinr (envs/reward_fn.py:48); CUE_SINR_SHANNON: sinr_threshold_dB (:61) */
    double shadow_d0_m;         /* SHADOWING: close-in reference distance (path_loss.py:72) */
    double shadow_chi_dB;       /* SHADOWING: standard deviation of the per-evaluation Gaussian (path_loss.py:73) */
    uint64_t rng_seed;          /* SHADOWING: Philox key */
    uint64_t first_global_env;  /* SHADOWING: global index of local env 0, so a sharded batch draws the same values whatever the GPU count */
} d2d_config_t;

/* Per-link link-budget constants, folded on the host from the per-device config dicts
 * (device.py:12-41, 51-80, 93-95, 134-140, 158-162; per-device overrides come from the
 * device_config_file, simulator.py:31). */
typedef struct d2d_link {
    double tx_eirp_offset_dB;   /* eirp_dBm(p) - p for the link's transmitter (device.py:60,135,159) */
    double rx_offset_dB;        /* rx_signal_level_dBm(e, pl) - (e - pl) for its receiver (device.py:72,137-140,161-162) */
    double rx_noise_dBm;        /* receiver thermal_noise_dBm (device.py:117-119; used at simulator.py:107,115) */
    double rx_sensitivity_dBm;  /* receiver rx_sensitivity_dBm (device.py:74-80; gate at simulator.py:123,149) */
    double tx_rb_bandwidth_kHz; /* transmitter rb_bandwidth_kHz (device.py:93-95; simulator.py:150) */
    int32_t link_type;          /* d2d_link_type */
    int32_t reserved0;
    double path_loss_const_dB;  /* D2D_PL_COST_HATA only: the path-loss constant toward this link's receiver */
} d2d_link_t;

/* d2d_step_io.flags */
#define D2D_STEP_INPUTS_STABLE 1u   /* see "Ordering rule" above; 0 is always safe */
#define D2D_STEP_ACTIONS_I16 2u     /* d2d_step_host / d2d_step_host_async only: `actions` points to int16_t [E][N] (every Discrete space of
                                       the reference fits: R n_pwr <= 32767; < 0 = agent absent) - half the upload per step; the library widens
                                       them on the device.  A host link shared by several GPUs gives the download what the upload leaves:
                                       profiles/README.md, "host link" */
#define D2D_STEP_AUTORESET 4u       /* d2d_step only (warp-kernel configurations: <= 32 CUEs, <= 32 DUE pairs, <= 64 RBs, no downlinks, no
                                       SHADOWING; D2D_ERR_UNSUPPORTED elsewhere and on every other step entry point): next-step auto-reset.
                                       An env whose step counter is >= episode_length at entry (its previous step returned done = 1) is
                                       reset instead of stepped, as d2d_reset + d2d_sample_actions(step 0) + one uncounted d2d_step would
                                       do it, under the key of d2d_bind_autoreset; its actions in this call are ignored.  Its outputs
                                       are that reset step's with reward = 0 and done = 0, its step counter becomes 0 and its episode
                                       index goes up by 1; the reset step enters no statistic.  Needs d2d_bind_autoreset and a bound
                                       step counter (D2D_ERR_STATE otherwise). */

/* Buffers of one step.  All pointers are device pointers for d2d_step and host pointers for
 * d2d_step_host.  `actions` is required; any output may be NULL to skip it. */
typedef struct d2d_step_io {
    const int32_t *actions;     /* [E][N] raw Discrete actions (envs/d2d_env.py:36-40); < 0 = agent absent this step */
    float *obs;                 /* [E][N][6] compact LinearObsFunction table (envs/obs_fn.py:55-61):
                                   (tx_x, tx_y, rx_x, rx_y, sinr_dB, snr_dB); agent i's reference vector is
                                   rows [i, others...] of this table (envs/obs_fn.py:43-53); the row of an absent agent
                                   keeps its positions and has sinr = snr = 0 */
    float *capacity_mbps;       /* [E][N]  simulator.py:144-154 */
    float *reward;              /* [E]     SystemCapacityRewardFunction scalar (envs/reward_fn.py:27-44) */
    uint8_t *done;              /* [E]     num_steps >= episode_length (envs/d2d_env.py:68) */
    float *rate_bps;            /* [E][N]  simulator.py:118-127 (info['rate_bps'], envs/d2d_env.py:114) */
    int16_t *rb;                /* [E][N]  decoded resource block (envs/d2d_env.py:95) */
    int16_t *tx_pwr_dBm;        /* [E][N]  decoded Tx power (envs/d2d_env.py:96) */
    float *agent_reward;        /* [E][N]  per-agent reward of SHANNON / CUE_SINR_SHANNON (0 for absent agents); with
                                   SYSTEM_CAPACITY the env's scalar broadcast to its acting agents (envs/reward_fn.py:44) */
    float *obs_dyn;             /* [E][N][2] (sinr_dB, snr_dB): the columns of `obs` that change between resets
                                   (envs/obs_fn.py:55-61: the other four are device positions, which only reset() /
                                   set_position move - fetch those once per reset with d2d_get_positions).  A host loop that
                                   asks for obs_dyn instead of obs moves 8N instead of 24N bytes per env-step. */
    int32_t *actions_out;       /* d2d_episode only: [T + 1][E][N] record of the actions taken (NULL to skip) */
    uint32_t flags;             /* D2D_STEP_* */
    uint32_t reserved0;
} d2d_step_io_t;

/* bits of an output mask (d2d_host_slot_buffers) */
enum { D2D_OUT_OBS = 1, D2D_OUT_CAPACITY = 2, D2D_OUT_REWARD = 4, D2D_OUT_DONE = 8, D2D_OUT_RATE = 16, D2D_OUT_RB = 32,
       D2D_OUT_TX_PWR = 64, D2D_OUT_AGENT_REWARD = 128, D2D_OUT_OBS_DYN = 256 };

/* Episode statistics accumulated on the device by d2d_step when a stats buffer is bound;
 * this is the vector the multi-GPU shell all-reduces over NCCL (never inside the step). */
#define D2D_STATS_REPLICAS 1024   /* the stats buffer is [D2D_STATS_REPLICAS][D2D_NUM_STATS]; readers sum over replicas */
enum { D2D_STAT_SUM_REWARD = 0, D2D_STAT_SUM_CAPACITY = 1, D2D_STAT_SUM_REWARD_SQ = 2,
       D2D_STAT_ENV_STEPS = 3, D2D_STAT_PENALTIES = 4, D2D_STAT_RESCUES = 5,
       D2D_STAT_TICKET_TIMEOUTS = 6,   /* diagnostic: per-warp ticket waits that fell back to the grid-wide wait (always 0) */
       D2D_NUM_STATS = 8 };

D2D_API int d2d_abi_version(void);
D2D_API const char *d2d_last_error(void);

/* Replaces Simulator.__init__ + create_devices (simulator.py:18-59) and the plugin construction of
 * D2DEnv.__init__ (envs/d2d_env.py:24-43).  `links` is [N] on the host. */
D2D_API int d2d_create(const d2d_config_t *config, const d2d_link_t *links, d2d_handle_t **out);
D2D_API int d2d_destroy(d2d_handle_t *h);

/* Sizes of the caller-owned state: positions float32 [E][V][2], per-env step counters uint8 [E],
 * stats float64 [D2D_STATS_REPLICAS][D2D_NUM_STATS] (blocks spread their atomics over the replicas). */
D2D_API int d2d_state_bytes(const d2d_handle_t *h, size_t *positions_bytes, size_t *step_count_bytes,
                            size_t *stats_bytes);
/* Binds the device buffers that hold Device.position (device.py:48,82-83) for every env, D2DEnv.num_steps
 * (envs/d2d_env.py:43) and the statistics accumulators (stats may be NULL). */
D2D_API int d2d_bind_state(d2d_handle_t *h, float *positions, uint8_t *step_count, double *stats);

/* Binds what D2D_STEP_AUTORESET needs: episode_index uint32 [E] on the device (caller-owned; NULL unbinds) and the
 * key base.  An env's n-th auto-reset (n = its episode index after the increment) draws its positions and actions under
 * the Philox key splitmix64(base_key + n * 0x9E3779B97F4A7C15) (gym_d2d_b200/csrc/d2d_common.cuh: d2d_autoreset_key),
 * with the global env in the counter: the draws depend on (base_key, global env, n) only, whatever the sharding or
 * chunking, and a replayed CUDA graph draws fresh positions at every replay because episode_index lives on the device.
 * Bases that advance by that same constant (keys seed + k * 0x9E3779B97F4A7C15) would make one base's stream the next one's
 * shifted by an episode: mix them first (VecD2DEnv binds splitmix64 of its reset key).
 * D2D_ERR_UNSUPPORTED on a configuration the warp kernel does not serve. */
D2D_API int d2d_bind_autoreset(d2d_handle_t *h, uint32_t *episode_index, uint64_t base_key);

/* Optional float64 shadow of the positions, float64 [E][V][2] (NULL unbinds).  When bound, d2d_set_positions /
 * d2d_reset also write it, and the step kernels read it in their rare fp64 recomputation path only: links whose
 * results the fp32 rounding of caller-supplied float64 positions could move by more than 1e-4 relative are
 * recomputed from the unrounded positions.  The hot path still reads only the fp32 state. */
D2D_API int d2d_bind_positions_f64(d2d_handle_t *h, double *positions_f64);

/* Replaces Device.set_position over a batch (device.py:82-83; device_config_file positions,
 * simulator.py:65-66).  src is float64 [count][V][2], host memory if src_on_device == 0 (the call then
 * synchronises the stream).  Device 0 (MBS) is pinned to (0,0) as simulator.py:63-64 does. */
D2D_API int d2d_set_positions(d2d_handle_t *h, const double *src, int src_on_device, int64_t first_env,
                              int64_t count, void *stream);

/* Replaces Simulator.reset position sampling (simulator.py:61-75, position.py:18-45) and
 * `num_steps = 0` (envs/d2d_env.py:46) for every env whose env_mask byte is non-zero (NULL = all).
 * Counter-based Philox4x32-10 keyed by (seed, first_global_env + local index, device index), so a
 * sharded batch draws the same scenario for a given global env whatever the number of GPUs. */
D2D_API int d2d_reset(d2d_handle_t *h, uint64_t seed, uint64_t first_global_env, const uint8_t *env_mask,
                      void *stream);

/* Copies the bound float32 positions of envs [first_env, first_env + count) to dst, float32 [count][V][2] (host memory
 * unless dst_on_device; a host copy synchronises the stream).  With d2d_step_io.obs_dyn this is the once-per-reset half
 * of the observation table: row j of obs is (pos[tx_j], pos[rx_j], obs_dyn[j]) with the device indices of the header
 * comment (CUE j: tx = 1 + j, rx = 0; DUE pair d: tx = 1 + C + 2d, rx = tx + 1). */
D2D_API int d2d_get_positions(d2d_handle_t *h, float *dst, int dst_on_device, int64_t first_env, int64_t count, void *stream);

/* Discrete(n).sample() for every agent of every env (envs/d2d_env.py:54-60; gym.spaces.Discrete.sample is uniform over
 * 0 .. n - 1): int32 [E][N] device buffer, counter-based Philox4x32-10 draws keyed by (seed, first_global_env + env, link,
 * step_index), the same values d2d_episode draws internally for that step (step_index 0 = the reset step).  DOWNLINK
 * links, which the reference's reset never samples, are marked absent (-1). */
D2D_API int d2d_sample_actions(d2d_handle_t *h, int32_t *actions, uint64_t seed, uint32_t step_index, void *stream);

/* Replaces D2DEnv.step (envs/d2d_env.py:62-71): _decode_action (:93-101), Simulator.step
 * (simulator.py:77-154), LinearObsFunction (envs/obs_fn.py:43-61), SystemCapacityRewardFunction
 * (envs/reward_fn.py:27-44), the done flag (:68) and the info fields (:106-116), for all E envs. */
D2D_API int d2d_step(d2d_handle_t *h, const d2d_step_io_t *io, void *stream);

/* num_steps consecutive d2d_step calls in ONE kernel launch: the agent loop of the reference's examples
 * (examples/simple_env.py:20-33: `for _ in range(EPISODE_LENGTH): env.step(actions)`) when the actions of every step
 * are known up front (scripted / random policies, replay, evaluation of recorded trajectories).  Every io buffer gains a
 * leading [num_steps] dimension: actions [T][E][N], obs [T][E][N][6], reward [T][E], ...; slice t holds exactly what the
 * t-th d2d_step call would have written.  An env's positions are read once for its T steps. */
D2D_API int d2d_step_many(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, void *stream);

/* One whole episode in ONE launch (SURVEY 8f-1 / 8f-4): D2DEnv.reset (envs/d2d_env.py:45-52: Simulator.reset draws new
 * positions - the values d2d_reset(reset_seed) draws - num_steps = 0, one UNCOUNTED step with sampled actions produces the
 * initial observation) followed by num_steps counted steps, the agent loop of examples/simple_env.py:20-33.  Every io
 * buffer has a leading [num_steps + 1] dimension: slice 0 is the reset step (done = 0; it enters no statistic), slice t
 * the t-th counted step, exactly what d2d_reset + d2d_step x (num_steps + 1) would have produced on the same actions.
 * With D2D_EPISODE_DRAW_ACTIONS the actions are sampled on the device (d2d_sample_actions(action_seed, t) for slice t;
 * io->actions may be NULL, io->actions_out records them); otherwise io->actions is [num_steps + 1][E][N].  The drawn
 * positions are left in the bound state and the step counters at num_steps, so d2d_step can continue the episode.
 * Default-topology configurations run it as one launch of the warp kernel that reads no global memory but its
 * constants; others compose it from d2d_reset, d2d_sample_actions and d2d_step launches. */
#define D2D_EPISODE_DRAW_ACTIONS 1u
D2D_API int d2d_episode(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, uint64_t reset_seed, uint64_t action_seed,
                        uint32_t episode_flags, void *stream);

/* num_steps COUNTED steps from the current state with actions sampled on the device - a random-policy rollout (the loop of
 * examples/simple_env.py:20-33 with Discrete.sample() as the policy) that reads no action buffer: slice t of every io buffer
 * ([num_steps][E]...) is what d2d_sample_actions(action_seed, first_step_index + t) + d2d_step would have produced.
 * io->actions is ignored; io->actions_out records the draws.  One launch on default-topology configurations. */
D2D_API int d2d_rollout(d2d_handle_t *h, const d2d_step_io_t *io, int32_t num_steps, uint64_t action_seed, uint32_t first_step_index,
                        void *stream);

/* Same call with HOST buffers: copies the actions to the device, steps, copies every non-NULL output
 * back and synchronises the stream.  This is the end-to-end path a CPU-side caller (the reference's
 * own env.step loop, INTEGRATION.md) would bind. */
D2D_API int d2d_step_host(d2d_handle_t *h, const d2d_step_io_t *host_io, void *stream);

/* Pipelined form of d2d_step_host for a CPU-side loop that keeps several steps in flight: slot 0 .. D2D_HOST_SLOTS - 1 selects
 * one of the device staging sets; the action upload runs on the library's copy-in stream, the kernel on `stream` (so steps stay
 * ordered), the result download on its copy-out stream.  d2d_step_host_wait(slot) blocks until that slot's results
 * are in the host buffers; a slot may be re-submitted only after it has been waited for.  Host buffers should be
 * pinned.  d2d_step_host(...) == d2d_step_host_async(..., 0, ...) + d2d_step_host_wait(0). */
#define D2D_HOST_SLOTS 4
D2D_API int d2d_step_host_async(d2d_handle_t *h, const d2d_step_io_t *host_io, int slot, void *stream);
D2D_API int d2d_step_host_wait(d2d_handle_t *h, int slot);

/* Library-owned PINNED host buffers of pipeline slot `slot` for the outputs in `outputs` (a D2D_OUT_* mask): fills
 * host_io with pointers into one contiguous pinned allocation (actions first, then the requested outputs, each 256-byte
 * aligned) that has a device twin of the same layout.  Passing this host_io to d2d_step_host_async(slot) brings all
 * outputs back with ONE copy (the caller-owned-buffer form issues one per output); `actions` may be replaced by any
 * other host buffer of the caller's.  The buffers live until the handle
 * is destroyed or the slot is re-laid-out with another mask. */
D2D_API int d2d_host_slot_buffers(d2d_handle_t *h, int slot, uint32_t outputs, d2d_step_io_t *host_io);

/* Materialises the reference's per-agent observation layout (envs/obs_fn.py:43-53) from the compact
 * table: out[e][i] = concat(table[e][i], table[e][k] for k != i), float32 [E][N][6N].  O(N^2) bytes:
 * provided for drop-in use at small E only. */
D2D_API int d2d_per_agent_obs(d2d_handle_t *h, const float *obs_table, float *out, int64_t num_envs,
                              void *stream);

/* Zeroes the bound statistics accumulators. */
D2D_API int d2d_stats_reset(d2d_handle_t *h, void *stream);

/* Introspection for tests and the bench: number of kernel launches issued through this handle, and the
 * launch geometry the step kernel uses for the bound configuration. */
D2D_API int64_t d2d_launch_count(const d2d_handle_t *h);
D2D_API int d2d_step_geometry(const d2d_handle_t *h, int32_t *grid, int32_t *block, int32_t *smem_bytes,
                              int32_t *envs_per_block);

#endif /* D2D_B200_H */
