/* taco_b200.h -- C ABI of the B200-native fused FPV environment step.
 *
 * Drop-in boundary for the hot path of yinzikang/taco: everything below
 * VecTask.step(actions) (IsaacGymEnvs/isaacgymenvs/tasks/base/vec_task_asymmetry.py:290-334)
 * for the fpv_asymmetry tasks (IsaacGymEnvs/isaacgymenvs/tasks/fpv_asymmetry.py:34-1112).
 *
 * The reference's only native boundary is gymtorch.wrap_tensor_impl(data_ptr, device, dtype,
 * shape, ...) (python/isaacgym/_bindings/src/gymtorch/gymtorch.cpp:33-158): the simulator
 * owns device memory and hands raw pointers + shapes to torch.  This library keeps that
 * convention: it owns every state/output buffer, exposes raw device pointers + shapes
 * (taco_env_buffers), takes caller-owned contiguous float32 device actions, and never
 * synchronises the host inside taco_env_step.
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative
 * TACO_E_* code (message via taco_last_error, thread-local); `stream` is a cudaStream_t
 * passed as void* (0 = legacy default stream); one handle per device, not re-entrant per
 * handle; handles of different processes (one per GPU under torchrun) are independent.
 */
#ifndef TACO_B200_H
#define TACO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TACO_ABI_VERSION 1

/* task_mode: isaacgym_task_map keys Fpv_pos / Fpv_rotate / Fpv_flip / Fpv_mix
 * (IsaacGymEnvs/isaacgymenvs/tasks/__init__.py:33-39) */
#define TACO_TASK_POS 0
#define TACO_TASK_ROTATE 1
#define TACO_TASK_FLIP 2
#define TACO_TASK_MIX 3

/* cfg switches, fpv_asymmetry.py:63-112 (names keep the upstream spelling) */
#define TACO_F_RANDOM_COPTER_POS (1u << 0)
#define TACO_F_RANDOM_COPTER_QUAT (1u << 1)
#define TACO_F_RANDOM_COPTER_VEL (1u << 2)
#define TACO_F_RANDOM_TARGET_POS (1u << 3)
#define TACO_F_RANDOM_TARGET_YAW (1u << 4)
#define TACO_F_BATTERY_CONSUMPTION (1u << 5)
#define TACO_F_RANDOM_VOLTAGE (1u << 6)
#define TACO_F_ROTOR_NOISE (1u << 7)
#define TACO_F_ROTOR_RESPONSE (1u << 8)
#define TACO_F_RANDOM_ROTORDYNAMIC_COE (1u << 9)
#define TACO_F_RANDOM_ROTOR_RESPONSE (1u << 10)
#define TACO_F_RANDOM_ROTOR_SPEED (1u << 11)
#define TACO_F_RANDOM_AERODYNAMIC_COE (1u << 12)
#define TACO_F_RAMDOM_DELAY_TIME (1u << 13)
#define TACO_F_RAMDOM_DEPLOY_TIME (1u << 14)
#define TACO_F_RANDOM_COMMAND (1u << 15)
#define TACO_F_OBSERVATION_NOISE (1u << 16)
/* library-only switches */
#define TACO_F_STRICT_FP (1u << 24)   /* kernels compiled with -fmad=false: op-for-op float32 like eager torch */
#define TACO_F_DEBUG_DELAY (1u << 25) /* record the delayed action of every control sub-step (taco_env_debug_delay) */

#define TACO_OK 0
#define TACO_E_INVALID (-1) /* bad argument / unsupported configuration */
#define TACO_E_CUDA (-2)    /* CUDA runtime error, see taco_last_error */
#define TACO_E_NOMEM (-3)

#define TACO_NUM_OBS 26   /* fpv_asymmetry.py:107 */
#define TACO_NUM_ACTS 4   /* fpv_asymmetry.py:102 */
#define TACO_NUM_STATS 8
#define TACO_STATE_WORDS 64 /* floats per env in taco_env_export_state */

typedef struct TacoCfg {
    int32_t abi_version;        /* TACO_ABI_VERSION */
    int32_t num_envs;           /* envs simulated by this handle (cfg["env"]["numEnvs"] of the shard) */
    int64_t env_offset;         /* global id of local env 0 (rank * num_envs under torchrun) */
    int64_t num_envs_global;    /* total envs of the job; mix task groups are thirds of this range (fpv_asymmetry.py:924-926) */
    int32_t task_mode;          /* TACO_TASK_* */
    int32_t len_obs;            /* cfg["env"]["lenObservations"] */
    int32_t len_states;         /* cfg["env"]["lenStates"] */
    int32_t max_episode_length; /* cfg["env"]["maxEpisodeLength"] */
    int32_t control_freq_inv;   /* cfg["env"]["controlFrequencyInv"]; the delay buffer pins it to 10 */
    int32_t substeps;           /* cfg["sim"]["substeps"] */
    int32_t delay_time;         /* cfg["delay_time"], ms, 0..100 */
    uint32_t flags;             /* TACO_F_* */
    float dt;                   /* cfg["sim"]["dt"]; rotor model pins 0.001 */
    float rotor_response_time;  /* cfg["rotor_response_time"] */
    float difficulty;           /* cfg["difficulty"] */
    float clip_actions;         /* cfg["env"]["clipActions"] (inf allowed) */
    uint64_t seed;              /* Philox key */
} TacoCfg;

/* Device pointers of the buffers VecTask exposes (vec_task_asymmetry.py:231-254).  obs is
 * double-buffered (the two alternating addresses are obs_ab).  The state history lives in a strip
 * (taco_env_states_strip): states points at the current window, whose env stride is the strip's row,
 * not len_states * 26.  Both pointers change on every step; call taco_env_buffers again after each
 * taco_env_step.  While a rollout ring is attached, obs and states point into its newest slot. */
typedef struct TacoBuffers {
    float* obs;          /* (num_envs, len_obs, 26) f32, newest frame last */
    float* states;       /* (num_envs, len_states, 26) f32, env stride frames * 26 floats (contiguous in a ring slot) */
    float* rew;          /* (num_envs) f32 */
    int64_t* reset;      /* (num_envs) i64, read at the start of step (lazy reset), written at the end */
    uint8_t* time_outs;  /* (num_envs) bool */
    int32_t* progress;   /* (num_envs) i32 (reference: i64 progress_buf) */
    float* obs_ab[2];
    float* states_ab[2]; /* [0] = base of the state history strip, [1] = NULL */
    int32_t num_envs, len_obs, len_states, num_obs;
} TacoBuffers;

typedef struct TacoEnv TacoEnv;

/* -- lifecycle: FpvBase.__init__ + VecTask.allocate_buffers (fpv_asymmetry.py:54-211, vec_task_asymmetry.py:231-254) */
int taco_env_create(const TacoCfg* cfg, int device, TacoEnv** out);
int taco_env_destroy(TacoEnv* env);
int taco_env_buffers(TacoEnv* env, TacoBuffers* out);

/* -- VecTask.step (vec_task_asymmetry.py:290-334): actions_dev = (num_envs,4) contiguous f32 on the env's
 * device.  Asynchronous on `stream`, no host sync. */
int taco_env_step(TacoEnv* env, const float* actions_dev, void* stream);
/* Same step through HOST buffers; synchronises the stream before returning.  Any output pointer may be NULL.
 * Pinned buffers (cudaHostAlloc / cudaHostRegister; torch pin_memory): ONE launch -- every thread loads its env's action from host
 * memory and posts rew / reset / time_outs into host memory across PCIe itself ("mapped mode").  Pageable buffers, or
 * TACO_HOST_MODE=copy in the environment: a chunked cudaMemcpyAsync pipeline (copy-in / kernel / copy-out of successive env
 * chunks overlap).  Both modes produce the results of taco_env_step and leave them in the device buffers as well. */
int taco_env_step_host(TacoEnv* env, const float* actions_host, float* rew_host, int64_t* reset_host,
                       uint8_t* time_outs_host, void* stream);
/* Opt-in compact result format of the host-buffer step: rew_host (f32, may be NULL) + flags_host, one byte per env with bit 0 =
 * reset_buf != 0 and bit 1 = time_outs: 5 bytes of device->host traffic per env instead of 13.  The reference dtypes (int64
 * reset_buf, vec_task_asymmetry.py:246-247) stay what taco_env_step_host returns.  Pinned (device-mapped) host buffers only. */
int taco_env_step_host_compact(TacoEnv* env, const float* actions_host, float* rew_host, uint8_t* flags_host, void* stream);
/* -- VecTask.reset (vec_task_asymmetry.py:352-361) does not simulate; this additionally marks every env for
 * reset on the next step and zeroes the observation history, i.e. restores the freshly-constructed state. */
int taco_env_reset_all(TacoEnv* env, void* stream);
/* -- CUDA-graph support.  Every launch of the step kernel carries the RL step index (Philox counter word, time slot of the
 * pending-action ring) as a kernel parameter, so a captured launch would replay with a stale index.  Between
 * taco_env_graph_begin and taco_env_graph_end the index of a launch is *counter (one device word, initialised to the current
 * step index) + the number of steps taken since graph_begin: a graph captured over a whole rollout -- rewind, H x (actor, critic,
 * step), taco_env_graph_advance(H) as its last node -- replays correctly any number of times.  taco_env_graph_end reads the counter
 * back (synchronises) and returns to host-side counting.  taco_env_step_counter reports the device word (NULL outside graph mode)
 * for other kernels that need the same index (taco_actor_act_counter) and the host's view of the step index. */
int taco_env_graph_begin(TacoEnv* env, void* stream);
int taco_env_graph_advance(TacoEnv* env, uint32_t steps, void* stream);
int taco_env_graph_end(TacoEnv* env, void* stream);
int taco_env_step_counter(TacoEnv* env, uint32_t** counter_dev, uint32_t* step_index_host);
/* -- zero-copy rollout storage: what PPOReplayBuffer.store copies every step (IsaacGymEnvs/algorithms/buffer_asymmetry.py:49-68:
 * obs_buf (H,N,Lo,26), states_buf (H,N,Ls,26), rew_buf, done_buf) the step kernel writes in place.  obs_ring / states_ring
 * are caller-owned contiguous float32 device buffers of `slots` = horizon + 1 slots of (num_envs, len, 26); with a ring
 * attached, step k of a rollout reads the history in slot k and writes slot k + 1 (slot k is exactly what the agent saw
 * before step k, i.e. obs_buf[k] / states_buf[k]) and, when the row pointers are given, rew_rows[k] / done_rows[k] (float32
 * (horizon, num_envs)) and time_out_rows[k] (u8).  Attaching copies the newest history into slot 0; stepping with the
 * ring full fails with TACO_E_INVALID; taco_env_rewind_rollout moves the newest slot to slot 0 for the next rollout;
 * taco_env_detach_rollout returns to the env's own double buffer.  taco_env_buffers reports the newest slot. */
int taco_env_attach_rollout(TacoEnv* env, float* obs_ring, float* states_ring, int32_t slots, float* rew_rows, float* done_rows,
                            uint8_t* time_out_rows, void* stream);
int taco_env_rewind_rollout(TacoEnv* env, void* stream);
int taco_env_detach_rollout(TacoEnv* env, void* stream);
int taco_env_rollout_cursor(TacoEnv* env);   /* newest slot index, or -1 when no ring is attached */
/* The env-owned state history: `frames` = len_states + period - 1 frames of 26 f32 per env row (num_envs rows).  After a step
 * that ran at step index t the window is the len_states frames from offset (t + 1) % period; a step writes only its newest frame,
 * and the step that wraps the offset to 0 first moves the kept frames to the start of the row.  (Not written while a rollout
 * ring is attached: detaching copies the ring's newest slot back into the window.) */
int taco_env_states_strip(TacoEnv* env, float** base, int32_t* frames, int32_t* period);
/* -- env.difficulty is written by the trainer every epoch (algorithms/ppo_asymmetry.py:173-175) */
int taco_env_set_difficulty(TacoEnv* env, float difficulty);
int taco_env_get_difficulty(TacoEnv* env, float* out);
int taco_env_set_seed(TacoEnv* env, uint64_t seed);

/* -- rollout statistics accumulated on the device since the last call (ppo_asymmetry.py:313-339):
 * [sum_reward, n_done, n_timeout, sum_episode_return, sum_episode_length, n_nonfinite, n_delay_overflow, n_env_steps]
 * written as 8 doubles to out_dev (device) and/or out_host; clears the accumulators.  This is the vector a
 * multi-GPU job all-reduces once per rollout. */
int taco_env_stats(TacoEnv* env, double* out_dev, double* out_host, void* stream);

/* -- synthetic U(-1,1) actions from the Philox action stream (benchmarks, tests): (num_envs,4) f32 */
int taco_env_fill_random_actions(TacoEnv* env, float* actions_dev, uint32_t step_index, void* stream);

/* -- test / checkpoint access: TACO_STATE_WORDS floats per env, layout in DESIGN.md (host pointers) */
int taco_env_export_state(TacoEnv* env, float* out_host);
int taco_env_import_state(TacoEnv* env, const float* in_host);
/* -- env-state checkpoint (the reference never checkpoints the env, SURVEY.md section 5): everything the next step depends on --
 * state and DR planes, pending-action ring, observation / state history, reward / reset / time-out buffers, step index,
 * difficulty, seed -- as one opaque host blob of taco_env_checkpoint_size bytes.  A loaded env continues bit-identically.  The
 * target env must have been created with the same TacoCfg (difficulty and seed are taken from the checkpoint).  Synchronous; not
 * allowed while a rollout ring is attached or in graph mode.  taco_env_import_state keeps the pending-action ring consistent when
 * it changes an env's progress counter (the run end slots are rebased to the new 10 * progress clock). */
int taco_env_checkpoint_size(TacoEnv* env, uint64_t* bytes);
int taco_env_checkpoint_save(TacoEnv* env, void* out_host, uint64_t bytes);
int taco_env_checkpoint_load(TacoEnv* env, const void* in_host, uint64_t bytes);
/* delayed action read at each control sub-step of the last step: (num_envs, control_freq_inv, 4) f32, host */
int taco_env_debug_delay(TacoEnv* env, float* out_host);

/* -- evaluation: per-episode outcome records (DESIGN.md section 6f).  With a log attached, every step (taco_env_step and the
 * host-buffer steps) is followed by one more launch on the step's stream -- capturable in a CUDA graph -- that accumulates per env
 * the quantities below and, for each env whose episode ended in that step (reset_buf != 0), appends one record.  Only whole
 * episodes are recorded: at attach, an env with reset_buf != 0 starts fresh and every other env is mid-episode and is not recorded
 * until after its next end.  taco_env_reset_all, taco_env_import_state and taco_env_checkpoint_load discard the episodes in
 * progress and re-run that initialisation.  The record order is unspecified (records of one step are appended in warp order by
 * atomics); records past the capacity are dropped but counted: dropped = *count - capacity.  Not allowed together with a rollout
 * ring (TACO_E_INVALID either way round).  48 bytes, a multiple of 16. */
typedef struct TacoEpisode {
    int64_t env_id;          /* global env id (env_offset + local index) */
    uint32_t end_step;       /* RL step index (0-based, the Philox step index) of the step that ended the episode */
    int32_t length;          /* progress_buf at the end, the episode length taco_env_stats adds */
    int16_t task;            /* TACO_TASK_POS / _ROTATE / _FLIP; a mix env: the task of its third of the global ids */
    int16_t timed_out;       /* time_outs of the ending step */
    float ret;               /* float32 sum of the rewards in step order: bit-identical to the return taco_env_stats adds */
    float pos_err_mean;      /* |pos - target pos| in m: mean over the episode's steps (after each step) */
    float pos_err_final;     /* ... and its value at the end */
    float tilt_max;          /* largest angle between body z and world z, acos(clamp(1 - 2 (qx^2 + qy^2))), rad */
    float speed_mean;        /* mean |linvel|, m/s */
    float angvel_max;        /* largest |angvel| (world frame), rad/s */
    float roll_travel;       /* flip envs: roll_continuous at the end minus after the first step (flips = roll_travel / 2 pi); else 0 */
} TacoEpisode;
/* allocates the log (capacity records, a counter, two accumulator planes) once, so a captured graph never sees it move; clears the
 * counter and runs the attach initialisation on `stream` */
int taco_env_attach_episode_log(TacoEnv* env, int64_t capacity, void* stream);
int taco_env_detach_episode_log(TacoEnv* env);
/* zero-copy access: records_dev = capacity TacoEpisode, count_dev = one uint64 (records appended since attach / the last clear) */
int taco_env_episode_log_buffers(TacoEnv* env, TacoEpisode** records_dev, uint64_t** count_dev, int64_t* capacity);
/* rewinds the counter on `stream`; the per-env accumulators are kept, so the episodes in progress continue */
int taco_env_episode_log_clear(TacoEnv* env, void* stream);
/* trajectory recorder: the TACO_STATE_WORDS-float taco_env_export_state row of each of the k local env ids in ids_dev (device
 * int32) into out_dev (k, TACO_STATE_WORDS) f32 on the device; an id outside [0, num_envs) gives a row of NaN.  Asynchronous on
 * `stream`, no host sync (capturable). */
int taco_env_record_state(TacoEnv* env, const int32_t* ids_dev, int32_t k, float* out_dev, void* stream);

/* -- training-time episode records and per-task summaries from the rollout ring (DESIGN.md section 6f).  No launch is added to the
 * step: one scan per rollout (taco_env_scan_rollout_episodes, capturable) walks the ring's rew / done / time-out rows written since
 * the last scan or rewind, in step order, one thread per env.  Per env it carries the running return (float32, rew added in step
 * order: bit-identical to TacoEpisode.ret and to the return taco_env_stats adds), the running length and a live flag from one
 * scan to the next, and appends one record per episode that ended in the scanned rows.  Only whole episodes are recorded: at
 * attach, an env with reset_buf != 0 starts fresh and every other env is not recorded until after its next end; taco_env_reset_all,
 * taco_env_import_state, taco_env_attach_rollout (steps taken without a ring are unseen) and a taco_env_rewind_rollout over rows
 * not yet scanned re-run that rule.  The record order is unspecified (one atomic per block); records past the capacity are
 * dropped but counted: dropped = *count - capacity.  The first six fields of TacoEpisode, same order and layout; 24 bytes. */
typedef struct TacoRolloutEpisode {
    int64_t env_id;          /* global env id (env_offset + local index) */
    uint32_t end_step;       /* RL step index (the Philox step index) of the step that ended the episode */
    int32_t length;          /* steps of the episode: the progress_buf value taco_env_stats adds */
    int16_t task;            /* TACO_TASK_POS / _ROTATE / _FLIP; a mix env: the task of its third of the global ids */
    int16_t timed_out;       /* time_outs of the ending step */
    float ret;               /* float32 sum of the rewards in step order */
} TacoRolloutEpisode;
/* summary of one scan, float64: for task t in POS, ROTATE, FLIP, words 5 t .. 5 t + 4 = [episodes, time-outs, sum of lengths,
 * sum of returns, sum of squared returns] over every episode that ended in the scanned rows (dropped records included).  Each env's
 * episodes are summed in step order and the envs in a fixed tree order, so the same rows give a bit-identical summary whatever
 * the launch timing; the vector is SUM-reducible across ranks. */
#define TACO_EPISODE_SUMMARY_WORDS 15
/* allocates records, counter and the per-env planes once (a captured graph never sees them move); clears the counter and runs the
 * start rule on `stream`.  Rows already in an attached ring are treated as scanned. */
int taco_env_attach_rollout_episodes(TacoEnv* env, int64_t capacity, void* stream);
int taco_env_detach_rollout_episodes(TacoEnv* env);
/* zero-copy access: records_dev = capacity records, count_dev = one uint64 (records appended since attach / the last clear) */
int taco_env_rollout_episodes_buffers(TacoEnv* env, TacoRolloutEpisode** records_dev, uint64_t** count_dev, int64_t* capacity);
/* rewinds the counter on `stream`; the per-env planes are kept, so the episodes in progress continue */
int taco_env_rollout_episodes_clear(TacoEnv* env, void* stream);
/* scans the ring rows written since the last scan or rewind and writes the TACO_EPISODE_SUMMARY_WORDS doubles of their episodes to
 * summary_dev (device).  Asynchronous on `stream`, capturable; in graph mode the end steps are read from the device step counter,
 * so capture the scan before the rollout's taco_env_graph_advance, like the steps it scans.  TACO_E_INVALID without attached
 * rollout episodes or without an attached ring with result rows. */
int taco_env_scan_rollout_episodes(TacoEnv* env, double* summary_dev, void* stream);

/* -- actor MLP inference in the rollout loop: MLP.forward + the actor branch of PPO_ActorCritic.act
 * (IsaacGymEnvs/algorithms/nets_asymmetry.py:23-39, :326-346) and PPO.spectral_normalize_actors
 * (IsaacGymEnvs/algorithms/ppo_asymmetry.py:398-404).  Two kernels compute the same function: an FP32 CUDA-core
 * path (parity) and a tcgen05/TMEM bf16 path (throughput; 1..4 hidden layers, widths multiples of 64 up to 256,
 * input width <= 256). */
typedef struct TacoActor TacoActor;
/* sizes = [in, h1, ..., hL, out] (n_sizes entries, out <= 4 = num_acts) */
int taco_actor_create(int device, const int32_t* sizes, int32_t n_sizes, TacoActor** out);
int taco_actor_destroy(TacoActor* actor);
/* weights/biases: float32 arrays in HOST OR DEVICE memory (unified addressing), row-major (out,in) per layer like nn.Linear.  With lipschitz_const > 0 every weight
 * matrix whose largest singular value sigma exceeds it is scaled by lipschitz_const / sigma on the device (power
 * iteration in double precision) -- the reference does this after each optimiser step, so calling it once per update
 * gives rollouts pre-normalised weights; lipschitz_const = 0 only measures the norms (taco_actor_sigmas), a negative value skips
 * the measurement too.  Synchronises the stream (the host buffers are free on return). */
int taco_actor_load(TacoActor* actor, const float* const* weights_host, const float* const* biases_host,
                    float lipschitz_const, void* stream);
/* largest singular value of every layer as measured by the last taco_actor_load (before scaling): n_layers doubles */
int taco_actor_sigmas(TacoActor* actor, double* out_host);
/* the (projected) float32 parameters of one layer, back on the host (either pointer may be NULL) */
int taco_actor_weights(TacoActor* actor, int32_t layer, float* w_host, float* b_host);
/* 1 when the tcgen05 path supports this actor's shape on this device */
int taco_actor_tc_available(TacoActor* actor);
/* PPO.spectral_normalize_actors (ppo_asymmetry.py:398-404) for one (rows, cols) row-major float32 matrix that already lives on the
 * device -- e.g. the storage of an nn.Linear weight between optimiser steps (ppo_asymmetry.py:248-249): sigma = largest singular
 * value (power iteration in double precision) is written to sigma_dev (one double, device); when lipschitz_const > 0 and
 * sigma > lipschitz_const the matrix is scaled in place by lipschitz_const / sigma.  Asynchronous on `stream`, no host sync. */
int taco_spectral_project(int device, float* w_dev, int32_t rows, int32_t cols, float lipschitz_const, double* sigma_dev, void* stream);
/* mean = tanh(MLP(obs)); obs_dev (n, in) f32 contiguous, mean_dev (n, out) f32.  use_tensor_cores = 0 selects the FP32
 * CUDA-core path, 1 the tcgen05 bf16 path (TACO_E_INVALID when unavailable).  Asynchronous on `stream`. */
int taco_actor_forward(TacoActor* actor, const float* obs_dev, float* mean_dev, int32_t n, int32_t use_tensor_cores,
                       void* stream);
/* PPO_ActorCritic.act, actor branch: mean as above; action = mean + exp(log_std)^2 * eps (scale_tril = diag(exp(log_std)^2),
 * nets_asymmetry.py:338), eps ~ N(0,1) from Philox(seed; env_offset + row, step_index, stream 6); clipped =
 * clamp(action, -1, 1) (ppo_asymmetry.py:310); logp = MultivariateNormal.log_prob(action).  log_std_host: `out` floats on
 * the host, or NULL = the values of the last taco_actor_set_log_std / taco_actor_act.  The kernels read std and the log-prob
 * constant from device memory owned by the actor (uploaded when log_std_host differs from the last values; that is refused while
 * `stream` is capturing), so launches captured in a CUDA graph follow taco_actor_set_log_std between replays.
 * clipped_dev / logp_dev may be NULL. */
int taco_actor_set_log_std(TacoActor* actor, const float* log_std_host, void* stream);
int taco_actor_act(TacoActor* actor, const float* obs_dev, int32_t n, const float* log_std_host, int64_t env_offset,
                   uint64_t seed, uint32_t step_index, float* mean_dev, float* action_dev, float* clipped_dev,
                   float* logp_dev, int32_t use_tensor_cores, void* stream);

/* -- critic inference in the rollout loop: the critic branch of PPO_ActorCritic.act (IsaacGymEnvs/algorithms/nets_asymmetry.py:350-352)
 * in the configuration the reference trains with (README.md:60-66: use_critic_encoder, critic_encoder_type=LSTM, lenStates=5):
 * value = MLP(LSTMEncoder(states)), LSTMEncoder = nn.LSTM(in_dim, lstm_hidden, lstm_layers, batch_first=True) with zero initial
 * state, output = top layer's h after the last time step (nets_asymmetry.py:128-136); MLP = [Linear -> ReLU] x L -> Linear(-> 1)
 * (nets_asymmetry.py:23-39, :318).  Two kernels compute the same function: an FP32 CUDA-core path (any shape; parity) and a
 * tcgen05/TMEM bf16 path (1..4 LSTM layers of width multiple of 16 up to 64, even in_dim <= 30, seq_len <= 8, 1..3 MLP hidden layers
 * of widths multiples of 64 up to 256).  A stacked LSTM hands its layers' outputs over through a workspace owned by the handle:
 * one forward at a time per handle.  taco_critic_create allocates it for a fixed chunk of the batch (4 waves of 2-tile pairs of
 * 128 rows, whatever n later calls pass): seq_len x 16 KB per tile, i.e. 97 MB at seq_len = 5 and 155 MB at seq_len = 8 on a
 * 148-SM B200, one buffer for 2 layers and two for 3-4 layers, so that a captured graph never sees it move. */
typedef struct TacoCritic TacoCritic;
/* mlp_sizes = [lstm_hidden, h1, ..., hL, 1] (n_mlp_sizes entries) */
int taco_critic_create(int device, int32_t in_dim, int32_t seq_len, int32_t lstm_hidden, int32_t lstm_layers,
                       const int32_t* mlp_sizes, int32_t n_mlp_sizes, TacoCritic** out);
int taco_critic_destroy(TacoCritic* critic);
/* lstm_host: 4 float32 arrays (host or device memory) per LSTM layer, bottom layer first, in torch's nn.LSTM layout and order: weight_ih (4H, in),
 * weight_hh (4H, H), bias_ih (4H), bias_hh (4H); gate row blocks i, f, g, o.  mlp weights/biases as in taco_actor_load.
 * Synchronises the stream (the host buffers are free on return). */
int taco_critic_load(TacoCritic* critic, const float* const* lstm_host, const float* const* mlp_weights_host,
                     const float* const* mlp_biases_host, void* stream);
/* 1 when the tcgen05 path supports this critic's shape on this device */
int taco_critic_tc_available(TacoCritic* critic);
/* value_dev (n[, 1]) f32 = critic(states_dev (n, seq_len, in_dim) f32 contiguous).  use_tensor_cores as in taco_actor_forward.
 * Asynchronous on `stream`. */
int taco_critic_forward(TacoCritic* critic, const float* states_dev, float* value_dev, int32_t n, int32_t use_tensor_cores,
                        void* stream);

/* taco_actor_act whose Philox step index is step_index + *step_base_dev (step_base_dev: device word, e.g. the env's counter from
 * taco_env_step_counter; NULL = plain taco_actor_act): capturable in a CUDA graph together with the env steps. */
int taco_actor_act_counter(TacoActor* actor, const float* obs_dev, int32_t n, const float* log_std_host, int64_t env_offset,
                           uint64_t seed, uint32_t step_index, const uint32_t* step_base_dev, float* mean_dev, float* action_dev,
                           float* clipped_dev, float* logp_dev, int32_t use_tensor_cores, void* stream);

/* -- native PPO update: PPO.update of the reference (IsaacGymEnvs/algorithms/ppo_asymmetry.py:137-258) for the network
 * configuration it trains with (README.md:60-66; nets_asymmetry.py:270-377): MLP actor (tanh mean, state-independent log_std,
 * std = exp(log_std)^2), critic = MLP(LSTMEncoder(states)) with 1-4 stacked unidirectional LSTM layers of 64 units (taco_ppo_create_layers;
 * the layers run one after another, each over all time steps, and back-propagate top layer first).  Forward / backward are tcgen05 GEMMs fed by TMA tensor maps (bf16
 * operands, fp32 accumulation), master weights / Adam moments / losses in fp32; the KL early stop (:223-226) is decided on the
 * device, so an update is a stream of launches without a host sync.  Per minibatch: taco_ppo_forward_loss -> [data parallel:
 * all-reduce SUM the 8 doubles of taco_ppo_loss_sums] -> taco_ppo_decide -> taco_ppo_backward -> [data parallel: all-reduce SUM
 * the flat gradient of taco_ppo_buffers] -> taco_ppo_apply (clip_grad_norm_ :244, Adam :117 with eps 1e-5, the spectral projection
 * of the actor weights :248-249,:398-404).  sm_100 only; no fallback. */
typedef struct TacoPPO TacoPPO;
typedef struct TacoPPOCfg {
    int32_t batch;               /* minibatch size (samples per optimiser step), multiple of 128 */
    int32_t obs_dim;             /* flattened actor input: num_obs * len_obs */
    int32_t act_dim;             /* <= 4 */
    int32_t state_dim, seq_len;  /* critic input (N, seq_len, state_dim): num_states, len_states */
    int32_t lstm_hidden;         /* 64; the number of stacked LSTM layers is an argument of taco_ppo_create_layers */
    int32_t n_actor_hidden, actor_hidden[4];     /* hidden widths: multiples of 16 in [16, 256] */
    int32_t n_critic_hidden, critic_hidden[4];
} TacoPPOCfg;
typedef struct TacoPPOHyper {
    float lr, clip, target_kl, max_grad, pi_coef, vf_coef, ent_coef;
    float lipschitz;             /* spectral bound c of this epoch (ppo_asymmetry.py:152-162) */
    int32_t use_lipschitz;
    int32_t world;               /* data-parallel ranks whose sums were all-reduced (1 = single process) */
} TacoPPOHyper;
int taco_ppo_create(int device, const TacoPPOCfg* cfg, TacoPPO** out);
/* the same with a stacked LSTM encoder of lstm_layers in [1, 4] unidirectional layers (nn.LSTM(state_dim, 64, lstm_layers));
 * taco_ppo_create is lstm_layers = 1 */
int taco_ppo_create_layers(int device, const TacoPPOCfg* cfg, int32_t lstm_layers, TacoPPO** out);
int taco_ppo_destroy(TacoPPO* ppo);
int taco_ppo_num_params(TacoPPO* ppo, int64_t* n);
/* offsets of the parameter tensors in the flat fp32 vector, in this order: log_std; actor (weight, bias) per layer; per LSTM
 * layer k, bottom first: weight_ih_lk, weight_hh_lk, bias_ih_lk, bias_hh_lk; critic MLP (weight, bias) per layer -- every tensor
 * in torch's layout */
int taco_ppo_param_offsets(TacoPPO* ppo, int64_t* offsets, int32_t count, int32_t* n_out);
/* device addresses of the flat vectors (n_params floats each) and of the int32 optimiser-step counter; any may be NULL */
int taco_ppo_buffers(TacoPPO* ppo, float** params, float** grad, float** adam_m, float** adam_v, int32_t** step);
/* after writing the parameter vector from outside: refresh the bf16 operand copies; the next spectral projection starts its
 * power iteration over (cold start) instead of from the singular vectors of the old weights */
int taco_ppo_params_changed(TacoPPO* ppo, void* stream);
int taco_ppo_begin_update(TacoPPO* ppo, void* stream);
/* rollout tensors as flat device views [N_total][...] (obs (N, obs_dim), states (N, seq_len, state_dim), act (N, act_dim),
 * old_logp / adv / ret (N)); idx_dev = `batch` int64 row indices of the minibatch (buffer_asymmetry.py:34-47) */
int taco_ppo_forward_loss(TacoPPO* ppo, const TacoPPOHyper* hyper, const float* obs, const float* states, const float* act,
                          const float* old_logp, const float* adv, const float* ret, const int64_t* idx_dev, void* stream);
int taco_ppo_loss_sums(TacoPPO* ppo, double** acc_dev);
int taco_ppo_decide(TacoPPO* ppo, const TacoPPOHyper* hyper, void* stream);
int taco_ppo_backward(TacoPPO* ppo, void* stream);
int taco_ppo_apply(TacoPPO* ppo, const TacoPPOHyper* hyper, void* stream);
/* synchronises; log rows of 8 floats per evaluated minibatch: policy-gradient loss, value loss, entropy loss, total loss, approx
 * KL, gradient norm, stopped-here flag, clip coefficient */
int taco_ppo_end_update(TacoPPO* ppo, float* log_host, int32_t max_rows, int32_t* n_rows, int32_t* optim_steps, int32_t* early_stop,
                        void* stream);
int taco_ppo_sigmas(TacoPPO* ppo, double* out_host);
/* test hook: device addresses of the last forward results: action mean (batch, act_dim) and value (batch) */
int taco_ppo_debug_outputs(TacoPPO* ppo, float** mean_dev, float** value_dev);
/* self-test of the GEMM kernel: D (m, n) fp32 = A (m, k) B (n, k)^T for bf16 row-major device matrices, n <= 256, k % 8 == 0 */
int taco_gemm_selftest(int device, const void* a_bf16, const void* b_bf16, float* d_f32, int32_t m, int32_t n, int32_t k, int32_t splits,
                       void* stream);
/* the same product from transposed operands At (k, m), Bt (k, n) (the kernel's MN-major operand mode, used by the weight-gradient
 * GEMMs that read batch-major activations as they are); m % 8 == 0, n % 8 == 0 */
int taco_gemm_selftest_mn(int device, const void* at_bf16, const void* bt_bf16, float* d_f32, int32_t m, int32_t n, int32_t k, int32_t splits,
                          void* stream);

/* -- rollout-buffer post-processing: PPOReplayBuffer.compute_returns_and_advantage
 * (IsaacGymEnvs/algorithms/buffer_asymmetry.py:93-132) and the time-out bootstrap PPO applies to the reward it stores
 * (IsaacGymEnvs/algorithms/ppo_asymmetry.py:313-324).  All buffers are contiguous float32 (horizon, num_envs[, 1]) on
 * `device`, like the reference's rew_buf / done_buf / value_buf / adv_buf / ret_buf; last_value is (num_envs[, 1]).
 * taco_gae_advantages: backward GAE(lambda) scan -> adv (un-normalised), ret = adv + value, and moments_dev[0..2] =
 * [sum adv, sum adv^2, sample count] in float64 (overwritten).  time_outs_dev (horizon, num_envs) bool/u8 may be NULL;
 * when given, rew + gamma * value is used for the steps with time_outs * done != 0.  A multi-GPU job all-reduces (SUM)
 * the three moments, then every rank calls taco_gae_normalize(adv, horizon * num_envs, moments): adv = (adv - mean) /
 * (std + 1e-8) with the unbiased std of ALL samples (buffer_asymmetry.py:132).  Asynchronous on `stream`, no host sync. */
int taco_gae_advantages(int device, int32_t horizon, int32_t num_envs, const float* rew_dev, const float* done_dev,
                        const uint8_t* time_outs_dev, const float* value_dev, const float* last_value_dev, float gamma, float lam,
                        float* adv_dev, float* ret_dev, double* moments_dev, void* stream);
int taco_gae_normalize(int device, float* adv_dev, int64_t count, const double* moments_dev, void* stream);

/* -- self-test: exhaustive comparison (all float bit patterns with |x| in [2^-60, 2^60]) of the kernel's 3-instruction
 * division-by-constant against IEEE division, for every divisor the step kernel uses; writes the mismatch count. */
int taco_selftest_divc(int device, float dt, uint64_t* n_mismatch);
/* atan2_poly of the step kernel (roll angle of refresh_state, fpv_asymmetry.py:334-360 / torch_utils.py:175-196: torch.atan2 in
 * the reference) against double-precision atan2 on n_angles directions x 9 radii, the four axes and the origin:
 * *max_ulp = largest error in units in the last place of the exact result, *n_nonfinite = NaN / Inf results (must be 0). */
int taco_selftest_atan2(int device, uint32_t n_angles, float* max_ulp, uint32_t* n_nonfinite);

/* number of CUDA kernels this library has launched in this process so far (every <<<>>> of libtaco_b200.so; captured launches
 * count once, at capture) */
int taco_launch_count(uint64_t* out);
const char* taco_last_error(void);
int taco_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TACO_B200_H */
