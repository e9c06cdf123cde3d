/*
 * dril_b200.h — C ABI of libdril_b200.so: the B200-native PPO rollout-and-update hot path of
 * DRiL.jl (KristianHolme/DRiL.jl), hand-written CUDA for sm_100a.
 *
 * The reference has no FFI: its "plugin API" is Julia multiple dispatch on the abstract types
 * of src/interfaces/.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference repo).  Julia binds these with `ccall` (see
 * julia/DRiLB200.jl and INTEGRATION.md); the tests in this repo bind them with ctypes.
 *
 * Conventions
 *   - plain C, no C++/torch types; every function returns int32 status: 0 = ok, nonzero =
 *     error (message from dril_last_error(), thread-local).  Nothing throws or aborts.
 *   - all pointers in signatures are HOST pointers unless the name ends in `_dev`; the
 *     library owns all device memory behind opaque handles and keeps no host pointer after
 *     a call returns.  Calls are synchronous at return unless suffixed `_async`.
 *   - sizes are int64, floats are fp32, discrete actions are int64 in env space
 *     (Discrete{Int64}: value = index + start, src/spaces.jl:157-164).
 *   - a ctx is bound to one CUDA device + one stream and is NOT thread-safe: one ctx per
 *     GPU, driven by one host thread (Julia: call from the owning task, no @threadcall).
 *   - there is no CPU fallback: without a CUDA device dril_ctx_create fails.
 */
#ifndef DRIL_B200_H
#define DRIL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRIL_OK 0
#define DRIL_ERR_INVALID 1
#define DRIL_ERR_CUDA 2
#define DRIL_ERR_UNSUPPORTED 3
#define DRIL_ERR_NCCL 4

typedef struct dril_ctx dril_ctx;
typedef struct dril_env dril_env;
typedef struct dril_policy dril_policy;
typedef struct dril_buffer dril_buffer;

/* env kinds (dynamics live in ClassicControlEnvironments.jl for the reference; SYNTHETIC is
 * the rollout-sweep env of SURVEY.md §8d C5).  MOUNTAINCAR and ACROBOT: Discrete(3) actions (Discrete.start = act_start),
 * MOUNTAINCAR_CONTINUOUS: Box(1) force on [-1, 1] */
enum { DRIL_ENV_CARTPOLE = 0, DRIL_ENV_PENDULUM = 1, DRIL_ENV_SYNTHETIC = 2, DRIL_ENV_MOUNTAINCAR = 3,
       DRIL_ENV_MOUNTAINCAR_CONTINUOUS = 4, DRIL_ENV_ACROBOT = 5 };
/* action-space kinds: Discrete / Box (src/spaces.jl:28-44,157-164) */
enum { DRIL_ACT_DISCRETE = 0, DRIL_ACT_CONTINUOUS = 1 };
#define DRIL_MAX_HIDDEN_LAYERS 5
#define DRIL_MAX_ACT_DIM 16
#define DRIL_MAX_OBS_DIM 256

/* NormalizeWrapperEnv kwargs (environment_wrappers/normalizeWrapperEnv.jl:71-80). */
typedef struct {
    int32_t training;    /* default 1 */
    int32_t norm_obs;    /* default 1 */
    int32_t norm_reward; /* default 1 */
    float clip_obs;      /* 10 */
    float clip_reward;   /* 10 */
    float gamma;         /* 0.99 */
    float epsilon;       /* 1e-8 */
} dril_norm_cfg;

/* PPO hyper-parameters (algorithms/ppo.jl:25-40) + the Adam rule of ppo.jl:64-66.
 * Optional fields use a negative value for Julia's `nothing`. */
typedef struct {
    float gamma;
    float gae_lambda;
    float clip_range;
    float clip_range_vf;   /* < 0: nothing */
    float ent_coef;
    float vf_coef;
    float max_grad_norm;   /* < 0: nothing */
    float target_kl;       /* < 0: nothing */
    int32_t normalize_advantage;
    float learning_rate;
    float adam_beta1;      /* 0.9 */
    float adam_beta2;      /* 0.999 */
    float adam_eps;        /* 1e-5 */
} dril_ppo_hyper;

/* Per-iteration training statistics, the fields of learn_stats (algorithms/ppo.jl:301-312)
 * plus the per-rollout monitor aggregates behind log_stats (monitorWrapperEnv.jl:64-70). */
typedef struct {
    float entropy_loss, policy_loss, value_loss, approx_kl_div, clip_fraction, loss;
    float explained_variance, grad_norm, learning_rate, entropy, ratio;
    float rollout_ms, update_ms;      /* device time of the two halves */
    int32_t n_minibatch_steps;        /* Adam steps applied this iteration */
    int32_t kl_stopped;               /* 1 if the target_kl stop fired (ppo.jl:235-238) */
    int64_t episodes;                 /* episodes finished during this rollout */
    double episode_return_sum, episode_length_sum;
    /* the monitor window after this rollout (mean over the last `stats_window` episodes, monitorWrapperEnv.jl:64-70);
     * NaN / 0 when the env has no MonitorWrapperEnv or no episode has finished yet */
    float ep_rew_mean, ep_len_mean;
    int64_t episodes_in_window;
} dril_iter_stats;

/* rollout-buffer fields (buffers/buffer_types.jl:3-15); device layout is time-major
 * [n_steps][n_envs][...]; sample index s = t*n_envs + env. */
enum {
    DRIL_BUF_OBS = 0,        /* float  [T][N][obs_dim]   */
    DRIL_BUF_ACTIONS = 1,    /* int32 [T][N] (discrete, env space) | float [T][N][act_dim] (raw, unclamped) */
    DRIL_BUF_REWARDS = 2,    /* float  [T][N] */
    DRIL_BUF_VALUES = 3,
    DRIL_BUF_LOGPROBS = 4,
    DRIL_BUF_ADVANTAGES = 5,
    DRIL_BUF_RETURNS = 6,
    DRIL_BUF_FLAGS = 7,      /* uint8  [T][N]: bit0 terminated, bit1 truncated */
    DRIL_BUF_BOOT = 8,       /* float  [T][N]: V(terminal_observation) where truncated (trajectory.jl:57-61) */
    DRIL_BUF_LAST_VALUES = 9,/* float  [N]: V(new_obs) after the final step (trajectory.jl:65-70) */
    DRIL_BUF_EPISODE_R = 10, /* float  [T][N]: infos[i]["episode"]["r"] where done (monitorWrapperEnv.jl:54) */
    DRIL_BUF_EPISODE_L = 11  /* int32  [T][N]: infos[i]["episode"]["l"] where done */
};

/* profiled kernel kinds for dril_ctx_get_profile */
enum {
    DRIL_K_ROLLOUT = 0, DRIL_K_GAE = 1, DRIL_K_ADV_STATS = 2, DRIL_K_LOSS_GRAD = 3,
    DRIL_K_GRAD_REDUCE = 4, DRIL_K_ADAM = 5, DRIL_K_EXPLAINED_VAR = 6, DRIL_K_MONITOR = 7,
    DRIL_K_ENV = 8, DRIL_K_POLICY = 9, DRIL_K_ALLREDUCE = 10, DRIL_K_PERMUTE = 11, DRIL_K_COUNT = 12
};

const char* dril_last_error(void);
int32_t dril_version(void);
/* SHA-256 prefix of the sources + compiler flags the library was built from (build.py rebuilds when it differs from the tree) */
const char* dril_source_hash(void);
/* 0 if a CUDA device is usable, else an error (used by hosts to fail loudly, never to fall back) */
int32_t dril_device_count(int32_t* count);
/* process-wide kernel-path switches (all default 1; every combination meets the same parity bounds, tests/
 * test_gpu_parity.py::test_kernel_paths_vs_oracle).  Unknown keys are an error.
 *   "ft"          features-on-lanes tcgen05 loss/grad kernel (fp16 hi/lo split, actor + critic merged) for hidden_dims = [64, 64],
 *                 obs_dim <= 4, Discrete(<= 2): the default for such policies
 *   "ftg"         general-shape features-on-lanes tcgen05 loss/grad kernel (2-3 hidden layers of width 64 / 128, Discrete(<= 4) or
 *                 Box(<= 2) head); 2 = also prefer it where "ft" applies
 *   "tc"          round-1 samples-on-lanes tcgen05 (3xTF32) loss/grad kernel for the "ft" shapes (used when "ft" is 0)
 *   "defer_critic" general rollout kernel: actor-only step loop, values from one batched tcgen05 critic pass afterwards
 *   "persistent"  "ft" kernel with the fused tail: all minibatch steps of an update (epochs x minibatches, tile records of all
 *                 epochs staged up front) run in ONE cooperative launch, a grid barrier between steps; 1 = on a single GPU
 *                 (default), 2 = also data parallel (peer exchange inside the loop: verified on 2 and 4 GPUs only)
 *   "tc_actor"    general rollout kernel with a deferred critic and >= 96 envs per SM: the actor's layers on tcgen05 inside the
 *                 step loop (128-env tiles, rollout_gtc.cuh) instead of mma.sync / FMA tiles
 *   "syn_rollout" thread-per-env rollout kernel for the synthetic env with a small policy (2 = always two envs per thread)
 *   "fused_tail"  partial reduction + (peer-memory allreduce) + clip + KL stop + Adam inside that kernel (cooperative launch)
 *   "tc_rollout"  tensor-core rollout for CartPole with such a policy (actor-only step loop + batched critic pass)
 *   "single_net"  fp32 loss/grad kernel, networks too wide for a 128-sample tile of both nets: one net per pass over the
 *                 minibatch with shared activation rows (applies to policies created afterwards)
 *   "mma"         fp32 loss/grad kernel, sample tiles of a multiple of 16: layers whose padded dims are multiples of 16 run on warp-level
 *                 tensor-core tiles (mma.sync TF32, 3xTF32 split) instead of FMA tiles (policies created afterwards) */
int32_t dril_set_option(const char* key, int32_t value);

/* ---- context ---------------------------------------------------------------------------- */
int32_t dril_ctx_create(int32_t device, uint64_t seed, dril_ctx** out);
int32_t dril_ctx_destroy(dril_ctx* ctx);
int32_t dril_ctx_synchronize(dril_ctx* ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
int32_t dril_ctx_launch_count(dril_ctx* ctx, int64_t* launches);
/* per-kernel CUDA-event timing on the ctx stream (bench.py's live roofline) */
int32_t dril_ctx_set_profiling(dril_ctx* ctx, int32_t on);
int32_t dril_ctx_reset_profile(dril_ctx* ctx);
int32_t dril_ctx_get_profile(dril_ctx* ctx, int32_t kind, double* total_ms, int64_t* launches);
int32_t dril_ctx_sm_count(dril_ctx* ctx, int32_t* sms);
/* CUDA events on the ctx stream (slots 0..15) so hosts can time device work they enqueue */
int32_t dril_ctx_event_record(dril_ctx* ctx, int32_t slot);
int32_t dril_ctx_event_elapsed_ms(dril_ctx* ctx, int32_t slot_start, int32_t slot_stop, float* ms);
/* write a buffer larger than L2 on the ctx stream (benchmark hygiene between timed steps) */
int32_t dril_ctx_flush_l2(dril_ctx* ctx);

/* ---- multi-GPU (new work; the reference is single-process, SURVEY.md §8e) ------------- */
int32_t dril_comm_unique_id(uint8_t id_out[128]);
int32_t dril_comm_init(dril_ctx* ctx, int32_t rank, int32_t nranks, const uint8_t id[128]);
int32_t dril_comm_destroy(dril_ctx* ctx);
/* Optional one-shot NVLink allreduce fused into the reduce/Adam kernels (peer memory through CUDA IPC):
 * every rank exports a region of n_slots floats x 2 buffers, the host exchanges the 64-byte handles (any
 * transport: torch.distributed, MPI.jl, a file) and every rank imports all of them in rank order.
 * Without this the gradient allreduce goes through NCCL. Requires dril_comm_init first. */
int32_t dril_comm_p2p_export(dril_ctx* ctx, int64_t n_slots, uint8_t handle_out[64]);
int32_t dril_comm_p2p_import(dril_ctx* ctx, const uint8_t* handles /* [nranks][64] */);

/* ---- batched env: replaces MultiThreadedParallelEnv (environment_wrappers/
 *      multithreadedParallelEnv.jl:1-92) wrapped in MonitorWrapperEnv (monitorWrapperEnv.jl)
 *      and optionally NormalizeWrapperEnv (normalizeWrapperEnv.jl) ------------------------ */
/* norm == NULL: no NormalizeWrapperEnv. monitor_window <= 0: no MonitorWrapperEnv.
 * gid_offset: global index of env 0 (rank * n_envs) so RNG streams are sharding-invariant.
 * act_start: Discrete.start of the env's action space (ignored for Box). */
int32_t dril_env_create(dril_ctx* ctx, int32_t kind, int64_t n_envs, int32_t max_steps,
                        int32_t obs_dim, int32_t act_start, int64_t gid_offset,
                        const dril_norm_cfg* norm, int32_t monitor_window, dril_env** out);
int32_t dril_env_destroy(dril_env* env);
/* Random.seed!(parallel_env, seed): wrapper_utils.jl:24-44 */
int32_t dril_env_seed(dril_env* env, uint64_t seed);
/* reset!(env): multithreadedParallelEnv.jl:11-16, monitorWrapperEnv.jl:36-42, normalizeWrapperEnv.jl:111-121 */
int32_t dril_env_reset(dril_env* env);
/* observe(env) -> obs[n][obs_dim]; updates obs_rms when training (normalizeWrapperEnv.jl:123-137) */
int32_t dril_env_observe(dril_env* env, float* obs_out);
/* act!(env, actions) -> rewards, terminateds, truncateds, infos (multithreadedParallelEnv.jl:47-74).
 * actions: int64[n] (discrete, env space) or float[n][act_dim] (already through to_env).
 * terminal_obs[n][obs_dim]: rows valid where truncated ("terminal_observation"); episode_r/_l
 * valid where done ("episode"); the three info outputs may be NULL. */
int32_t dril_env_step(dril_env* env, const void* actions, float* rewards, uint8_t* terminated,
                      uint8_t* truncated, float* terminal_obs, float* episode_r, int64_t* episode_l);
int32_t dril_env_num_envs(dril_env* env, int64_t* n);
/* raw internal state, for replay tests: float[state_dim][n] + int32 steps[n]. state_dim: cartpole 4, pendulum 2, synthetic 0,
 * mountaincar 2, mountaincar_continuous 2, acrobot 4 */
int32_t dril_env_get_state(dril_env* env, float* state, int32_t* steps);
int32_t dril_env_set_state(dril_env* env, const float* state, const int32_t* steps);
/* normaliser statistics (save/load/sync_normalization_stats, normalizeWrapperEnv.jl:261-309) */
int32_t dril_env_get_norm_stats(dril_env* env, float* obs_mean, float* obs_var, int64_t* obs_count,
                                float* ret_mean, float* ret_var, int64_t* ret_count);
int32_t dril_env_set_norm_stats(dril_env* env, const float* obs_mean, const float* obs_var, int64_t obs_count,
                                float ret_mean, float ret_var, int64_t ret_count);
int32_t dril_env_set_training(dril_env* env, int32_t training);
/* ScalingWrapperEnv(env) around every env of the batch (environment_wrappers/scalingWrapperEnv.jl:14-49): observations are
 * mapped from the ORIGINAL Box [obs_low, obs_high] to [-1, 1] (observe, :94-99), actions arrive in [-1, 1] and are mapped back
 * to [act_low, act_high] before act! (:112-115).  The wrapper sits below Monitor / Normalize.  Box/Box envs only (pendulum,
 * mountaincar_continuous). */
int32_t dril_env_set_scaling(dril_env* env, int32_t on, const float* obs_low, const float* obs_high,
                             const float* act_low, const float* act_high);
/* original (un-normalised) obs / rewards of the last observe/act (old_obs, old_rewards) */
int32_t dril_env_get_original(dril_env* env, float* obs_out, float* rewards_out);
/* the zeroing of `returns` in sync_normalization_stats! (normalizeWrapperEnv.jl:299-309) */
int32_t dril_env_zero_returns(dril_env* env);
/* log_stats(env): mean return / length over the last `monitor_window` episodes (monitorWrapperEnv.jl:64-70) */
int32_t dril_env_monitor_stats(dril_env* env, float* ep_rew_mean, float* ep_len_mean,
                               int64_t* n_in_window, int64_t* total_episodes);

/* Per-env physical parameters, in this order (names are Gymnasium's attributes; the defaults are the built-in constants):
 *   cartpole                6: gravity 9.8, masscart 1.0, masspole 0.1, length 0.5, force_mag 10.0, tau 0.02
 *   pendulum                4: g 10.0, m 1.0, l 1.0, dt 0.05
 *   mountaincar             2: force 0.001, gravity 0.0025
 *   mountaincar_continuous  2: power 0.0015, gravity 0.0025
 *   acrobot                 6: link_length_1 1, link_mass_1 1, link_mass_2 1, link_com_pos_1 0.5, link_com_pos_2 0.5, link_moi 1
 *   synthetic               0:
 * Env n holds a range [lo[k][n], hi[k][n]] per parameter.  During env n's episode e (the reset counter of the RESET stream) the
 * value of parameter k is lo + (hi - lo) * u, three fp32 roundings, u = u01_f32 of Philox block (gid, e, k / 4, tag 6) word
 * k % 4: a pure function of the seed, the global env id, e and the range, so lo == hi is a fixed value and draws do not depend
 * on sharding.  Every reset draws anew (auto-reset, act!, reset!).
 * dril_env_set_params: lo, hi float[n_params][n_envs], n_params = the kind's count; hi == NULL: hi = lo (fixed values);
 * lo == NULL: back to the built-in constants.  Values must be finite with lo <= hi; masses, lengths, link_moi, tau and dt > 0;
 * gravity, g, force, force_mag and power >= 0 (else DRIL_ERR_INVALID).  The running episode takes the value its own (gid, e)
 * draws from the new ranges.  Thresholds, speed clips, max_torque and the spaces stay fixed.  Envs with parameters do not use
 * the CartPole tensor-core rollout.
 * dril_env_get_params: the current per-env values, float[n_params][n_envs] (the defaults for an env without parameters). */
#define DRIL_ENV_MAX_PARAMS 8
int32_t dril_env_set_params(dril_env* env, int32_t n_params, const float* lo, const float* hi);
int32_t dril_env_get_params(dril_env* env, int32_t n_params, float* values);

/* Parameter-augmented observations.  observe_params = 1: every observation of env n is
 *   [base observation (D components) | p_0 ... p_{P-1}],  obs_dim = D + P,
 * p_k = the value of parameter k in the running episode, in the table order above: exactly what dril_env_get_params returns,
 * raw fp32.  (cartpole 4 + 6, pendulum 3 + 4, mountaincar 2 + 2, mountaincar_continuous 2 + 2, acrobot 6 + 6.)
 *   - ScalingWrapperEnv maps the D base components only; the parameter components pass through raw.
 *   - NormalizeWrapperEnv normalises all D + P columns like any other (running statistics, clip, terminal observations), so
 *     a column that is constant over the batch (lo == hi everywhere) normalises to exactly 0 after the first update.
 *   - The terminal observation of a truncated step (and V(terminal_obs)) carries the values of the episode that ended; the
 *     observation after a reset carries the values just drawn for the new episode.
 *   - An env without ranges observes the defaults (it runs with lo = hi = the defaults); dril_env_set_params(lo = NULL)
 *     returns to that instead of dropping the parameters.  New ranges show as the running episode's own (gid, e) draw.
 * dril_env_set_observe_params is allowed only before the env's first observation (observe, step, rollout, evaluate;
 * reset and set_state do not count), else DRIL_ERR_INVALID: it resizes the obs-sized arrays (normaliser statistics, old and
 * terminal observations).  The synthetic env has no parameters: DRIL_ERR_UNSUPPORTED.  A policy or buffer built for the
 * other width fails the obs_dim check of the rollout.
 * dril_env_obs_dim: the env's current observation width, for hosts that build the policy from the env. */
int32_t dril_env_set_observe_params(dril_env* env, int32_t on);
int32_t dril_env_obs_dim(dril_env* env, int32_t* obs_dim);

/* Observation history (frame stacking) and velocity-free observations.  history_len = k in [1, DRIL_ENV_MAX_HISTORY]: the
 * observation of env n at step t is
 *   [f_{t-k+1} | ... | f_{t-1} | f_t],  oldest first,  obs_dim = F * k,
 * f_j = the frame at step j: the base observation as the wrappers below NormalizeWrapperEnv see it (raw, or mapped to
 * [-1, 1] by ScalingWrapperEnv).  mask_velocities = 1 keeps only the non-velocity components of every frame:
 *   cartpole (x, theta), pendulum (cos theta, sin theta), mountaincar(_continuous) (position),
 *   acrobot (cos th1, sin th1, cos th2, sin th2);
 * F = 4 / 2, 3 / 2, 2 / 1, 2 / 1, 6 / 4 (full / masked).  Scaling maps the kept components with their own bounds.
 *   - Frames from before the episode's first observation are that observation (padding "reset"): after a reset all k frames
 *     are the reset frame.
 *   - On act!, the frame the action was chosen on enters the history, then the env steps.  A truncated step's terminal
 *     observation (and V(terminal_obs)) is the stack ending in the ended episode's final frame; after the auto-reset the
 *     stack is k copies of the reset frame.  observe() never moves the history.
 *   - dril_env_reset, dril_env_set_state, dril_env_set_scaling and dril_evaluate's initial reset restart every env's history
 *     from its current frame.  Chunked collection, compat act! and successive rollouts continue it.
 *   - NormalizeWrapperEnv normalises all F * k columns; Monitor is unaffected; parameter ranges work as without history.
 *   - No RNG is involved: observations do not depend on gid_offset sharding.
 * (k = 1, mask_velocities = 0) is the plain env.  Otherwise the env runs the parametrised kernels (lo = hi = the defaults
 * without ranges; dril_env_set_params(lo = NULL) returns to that), so CartPole leaves the tensor-core rollout.
 * Allowed only before the env's first observation, else DRIL_ERR_INVALID, as is k outside [1, DRIL_ENV_MAX_HISTORY].  The
 * synthetic env, and an env with observe_params (in either call order): DRIL_ERR_UNSUPPORTED.  A policy or buffer built for
 * another width fails the obs_dim check of the rollout.  A policy deployed outside this library expects the stacked
 * observation. */
#define DRIL_ENV_MAX_HISTORY 4
int32_t dril_env_set_obs_history(dril_env* env, int32_t history_len, int32_t mask_velocities);

/* Sensor noise and actuation delay, per env; independent of each other.
 * Observation noise: std = [n_comp][n_envs] standard deviations sigma >= 0 (finite), n_comp = the base observation width
 * (cartpole 4, pendulum 3, mountaincar(_continuous) 2, acrobot 6).  Component j of env n's observation, in its episode e (the
 * index of that episode's reset and parameter draws) after s steps of it, is
 *   o_j + sigma[j][n] * z_j   (fp32: __fadd_rn(o_j, __fmul_rn(sigma, z_j)); sigma == 0 leaves o_j untouched),
 * z_j = Box-Muller in fp64 with one rounding to fp32 (r cos th for even j, r sin th for odd j) of Philox block
 * (gid, e, 2 s + j / 4, DRIL_TAG_OBS_NOISE = 7) word pair (j / 2) % 2 (u1 = u01_f32_open, u2 = u01_f32).
 *   - A sensor: the noise is added to the raw observation, before ScalingWrapperEnv's map, before the velocity mask and
 *     before the frame enters an observation history (the history holds the noisy frames the policy saw).  Dynamics,
 *     rewards, termination and dril_env_get_state use the true state.
 *   - A pure function of (seed, gid, e, s, j): observe() is idempotent, results do not depend on gid_offset sharding, and
 *     chunked collection equals one-shot collection.  A truncated step's terminal observation (and V(terminal_obs)) carries
 *     the noise of (e, max_steps), the observation after the reset that of (e', 0).
 *   - NormalizeWrapperEnv sees the noisy observation, dril_env_get_original returns it; the observation space is unchanged
 *     and a noisy value may leave it.  std may change at any time and takes effect at the next observation.
 * Action delay: delay = [n_envs] d in [0, DRIL_ENV_MAX_ACTION_DELAY].  Env n applies the action chosen d steps earlier in the
 * same episode: every env keeps a FIFO queue of env-space actions, which an action enters as act! receives it (after
 * ClampAdapter; ScalingWrapperEnv's map applies to the action that leaves it).
 *   - The queue restarts at every reset (auto-reset, compat act!, dril_env_reset, dril_evaluate's initial reset), at
 *     dril_env_set_state, at dril_env_set_scaling and whenever delays are set; the first action after a restart fills it, so
 *     for the first d steps the env applies that action.  Chunked collection, successive rollouts and compat act! continue it.
 *   - The rollout buffer keeps the chosen action and its log-prob; forced actions are chosen actions and are delayed too.
 *     Monitor, Normalize and (terminal) observations are unaffected.
 * std / delay = NULL turns the option off.  With either on the env runs the parametrised kernels (lo = hi = the defaults
 * without ranges), so CartPole leaves the tensor-core rollout.  The synthetic env, and an env with observe_params (in either
 * call order): DRIL_ERR_UNSUPPORTED.  A negative or non-finite sigma, n_comp other than the base width, or a delay outside
 * [0, DRIL_ENV_MAX_ACTION_DELAY]: DRIL_ERR_INVALID. */
#define DRIL_ENV_MAX_ACTION_DELAY 4
int32_t dril_env_set_obs_noise(dril_env* env, int32_t n_comp, const float* std);
int32_t dril_env_set_action_delay(dril_env* env, const int32_t* delay);

/* ---- actor-critic layer + optimiser state: replaces Discrete/ContinuousActorCriticLayer
 *      (layers/) and the Lux TrainState held by Agent (agents/agent_types.jl) ------------ */
int32_t dril_policy_create(dril_ctx* ctx, int32_t obs_dim, int32_t n_hidden, const int32_t* hidden_dims,
                           int32_t act_kind, int32_t act_n, int32_t act_start,
                           const float* act_low, const float* act_high, dril_policy** out);
int32_t dril_policy_destroy(dril_policy* p);
int32_t dril_policy_num_params(dril_policy* p, int64_t* n);
/* which loss/grad kernel the update uses for this policy: 1 = tensor cores (tcgen05: hidden_dims = [64, 64], obs_dim <= 4,
 * Discrete(n <= 2), option "tc" on; or 2-3 hidden layers of width 64 / 128, obs_dim <= 15, Discrete(n <= 4) or Box(n <= 2), option
 * "ftg" on), 2 = general-shape kernel with the layers whose padded dims are
 * multiples of 16 on warp-level tensor-core tiles (mma.sync TF32, 3xTF32; option "mma"), 0 = general-shape kernel on
 * fp32 FMA tiles only.  All replace the same reference code (src/algorithms/ppo.jl:188-254 loss functor + Zygote
 * pullback) and meet the same 1e-4 parity bound. */
int32_t dril_policy_update_path(dril_policy* p, int32_t* out);
/* flat fp32 vector in ComponentVector(ps) order: actor_head layers (weight (out,in) column-major,
 * bias), critic_head layers, log_std (layers/layer_lux.jl:4-52) */
int32_t dril_policy_set_params(dril_policy* p, const float* flat, int64_t n);
int32_t dril_policy_get_params(dril_policy* p, float* flat, int64_t n);
/* Adam moments + step (the reference never saves them; exposed for checkpointing) */
int32_t dril_policy_get_opt_state(dril_policy* p, float* m, float* v, int64_t n, int64_t* step);
int32_t dril_policy_set_opt_state(dril_policy* p, const float* m, const float* v, int64_t n, int64_t step);
int32_t dril_policy_seed(dril_policy* p, uint64_t seed, uint64_t step_index);
/* layer(obs, ps, st) -> actions, values, logprobs (layers/layer_forward.jl:3-13,30-39);
 * deterministic=1 gives mode.(ds) (layers/layer_methods.jl:3-26). actions: int64[B] | float[B][act_dim].
 * env_gids may be NULL (sample stream of row i is then env id i). values/logprobs may be NULL. */
int32_t dril_policy_forward(dril_policy* p, const float* obs, int64_t B, int32_t deterministic,
                            const int64_t* env_gids, void* actions, float* values, float* logprobs);
/* evaluate_actions (layers/layer_methods.jl:28-55) */
int32_t dril_policy_evaluate(dril_policy* p, const float* obs, const void* actions, int64_t B,
                             float* values, float* logprobs, float* entropy);
/* predict_values (layers/layer_methods.jl:57-61) */
int32_t dril_policy_predict_values(dril_policy* p, const float* obs, int64_t B, float* values);

/* ---- rollout buffer: replaces RolloutBuffer (buffers/buffer_types.jl:3-15, rollout_buffer.jl:6-44) */
int32_t dril_buffer_create(dril_ctx* ctx, int64_t n_steps, int64_t n_envs, int32_t obs_dim,
                           int32_t act_kind, int32_t act_dim, dril_buffer** out);
int32_t dril_buffer_destroy(dril_buffer* b);
int32_t dril_buffer_download(dril_buffer* b, int32_t field, void* dst, int64_t bytes);
int32_t dril_buffer_upload(dril_buffer* b, int32_t field, const void* src, int64_t bytes);
int32_t dril_buffer_field_bytes(dril_buffer* b, int32_t field, int64_t* bytes);

/* ---- the hot path ----------------------------------------------------------------------- */
/* collect_trajectories (buffers/trajectory.jl:22-78): n_steps fused observe -> forward -> sample ->
 * to_env -> act! -> monitor/normalise steps, written straight into the device buffer.
 * forced_actions (nullable): replay int64[T][N] | float[T][N][act_dim] instead of sampling. */
int32_t dril_rollout_collect(dril_env* env, dril_policy* p, dril_buffer* buf,
                             const void* forced_actions, float* fps_out);
/* Steps [t_begin, t_begin + t_count) of a rollout into the same rows of the buffer: collect_trajectories run in chunks
 * so that on_step callbacks (buffers/trajectory.jl:34-39) see the advancing env and can stop the collection mid-rollout.
 * start != 0 begins a rollout (per-rollout counters zeroed, the observe() of trajectory.jl:32, which precedes the first
 * hook: t_count = 0 requests it alone); Monitor / Normalize state carries across chunks; the bootstrap values of the last
 * chunk are the rollout's.  Follow with dril_gae after the last chunk. */
int32_t dril_rollout_collect_steps(dril_env* env, dril_policy* p, dril_buffer* buf, int64_t t_begin, int64_t t_count,
                                   int32_t start, const void* forced_actions);
/* evaluate_agent (src/evaluation.jl:54-143) with the episode loop on the device: reset!(env), `chunk_steps` fused policy
 * steps per launch (mode of the distribution when deterministic), one device -> host copy of the chunk's episode records
 * per launch; episodes are appended in the reference's order (step, then env index) until n_eval_episodes are
 * collected.  episode_rewards / episode_lengths: host arrays of n_eval_episodes elements. */
int32_t dril_evaluate(dril_env* env, dril_policy* p, int64_t n_eval_episodes, int32_t deterministic, int32_t chunk_steps,
                      float* episode_rewards, int64_t* episode_lengths, int64_t* n_collected, int64_t* env_steps);
/* compute_advantages! + returns = adv + values (trajectory.jl:80-102, rollout_buffer.jl:83-87) */
int32_t dril_gae(dril_buffer* buf, float gamma, float gae_lambda);
/* raw-array parity entry: time-major host arrays [T][N]; boot[T][N], last_values[N] */
int32_t dril_gae_raw(dril_ctx* ctx, const float* rewards, const float* values, const uint8_t* terminated,
                     const uint8_t* truncated, const float* boot, const float* last_values,
                     int64_t T, int64_t N, float gamma, float gae_lambda, float* advantages, float* returns);
/* (alg::PPO)(layer, ps, st, batch) + its Zygote reverse pass (algorithms/ppo.jl:365-407):
 * one minibatch given as host arrays; returns loss, stats[7] = {policy_loss, value_loss,
 * entropy_loss, clip_fraction, approx_kl_div, entropy, ratio} and the flat gradient. */
int32_t dril_ppo_loss_grad(dril_policy* p, const float* obs, const void* actions, const float* advantages,
                           const float* returns, const float* old_logprobs, const float* old_values,
                           int64_t B, const dril_ppo_hyper* hyper, float* loss, float* stats7, float* grads);
/* grad-norm clip + Adam step on a host gradient (ppo.jl:216-239, 64-66); returns pre-clip norm */
int32_t dril_optimizer_step(dril_policy* p, const float* grads, int64_t n, const dril_ppo_hyper* hyper,
                            float* grad_norm);
/* the epoch/minibatch loop of train! (ppo.jl:188-254) over the device buffer */
int32_t dril_ppo_update(dril_policy* p, dril_buffer* buf, const dril_ppo_hyper* hyper, int32_t epochs,
                        int64_t batch_size, uint64_t shuffle_seed, uint64_t epoch_counter,
                        dril_iter_stats* stats_out);
/* Makes every allocation the first iterations would otherwise make lazily (result slots, sample / tile records, moment buffers,
 * deferred-critic scratch).  Optional on one GPU; data-parallel hosts call it on every rank and synchronise the ranks before the
 * first iteration, so that no rank is inside a cudaMalloc while a peer's GPU already spins in a peer-memory exchange. */
int32_t dril_iteration_prepare(dril_env* env, dril_policy* policy, dril_buffer* buf, int32_t epochs, int64_t batch_size);
/* one train! iteration (ppo.jl:154-297): rollout + GAE + update + explained variance.
 * The _async form only enqueues; dril_iteration_result waits for the OLDEST enqueued iteration whose result has not
 * been read yet and returns its statistics (one pinned device->host record per iteration).  Up to 4 iterations may
 * be in flight, so a host loop can enqueue iteration i+1 before it reads iteration i and the device never idles;
 * enqueueing a fifth drops the oldest unread result. */
int32_t dril_ppo_iteration_async(dril_env* env, dril_policy* p, dril_buffer* buf, const dril_ppo_hyper* hyper,
                                 int32_t epochs, int64_t batch_size, uint64_t shuffle_seed,
                                 uint64_t epoch_counter);
int32_t dril_iteration_result(dril_policy* p, dril_iter_stats* stats_out);
int32_t dril_explained_variance(dril_buffer* buf, float* out);

#ifdef __cplusplus
}
#endif
#endif /* DRIL_B200_H */
