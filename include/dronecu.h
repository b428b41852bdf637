/*
 * dronecu.h -- C ABI of libdronecu.so, the B200 (sm_100a) batched quadcopter environment.
 *
 * The reference (henryplas/drone_rl) has no FFI of its own: its boundary is the Python
 * object protocol that Stable-Baselines3 and its scripts call (SURVEY.md section 8b).  Each
 * entry point below names the reference interface it stands in for; the Python classes in
 * drone_rl_b200/ (same names and argument meaning as the reference's) bind to these with
 * ctypes -- see INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; "d_" pointers are CUDA device pointers on the handle's
 *     device, "h_" pointers are host pointers.  `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream).
 *   - every function returns 0 (DRONECU_OK) or a negative dronecu_status; a text for the
 *     last error on the calling thread is available from dronecu_last_error().
 *   - a handle is bound to one device; calls on one handle must be serialised by the caller
 *     (the reference env is single-threaded and not re-entrant either); different handles
 *     are independent.
 *   - there is NO CPU fallback: without a CUDA device dronecu_create fails with
 *     DRONECU_ERR_CUDA.
 */
#ifndef DRONECU_H
#define DRONECU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRONECU_VERSION 100

typedef enum {
  DRONECU_OK = 0,
  DRONECU_ERR_INVALID = -1, /* bad argument */
  DRONECU_ERR_CUDA = -2,    /* CUDA runtime error (text in dronecu_last_error) */
  DRONECU_ERR_ALLOC = -3,
  DRONECU_ERR_UNSUPPORTED = -4
} dronecu_status;

/* dronecu_config.flags */
#define DRONECU_RANDOMIZED 1u /* random start + curriculum target  (DroneEnv.reset, drone.py:48-75)   */
#define DRONECU_AUTORESET 2u  /* SB3 DummyVecEnv semantics: reset a done env inside step (train.py:18-20) */

/* Every literal of the reference lives here so nothing is hard-coded in the kernels.
 * drone.py:14-46 (DroneEnv.__init__) / vectorized_drone.py:13-36 (VectorizedDroneEnv.__init__). */
typedef struct dronecu_config {
  double dt;                /* 0.02   drone.py:14,25                                */
  double mass;              /* 1.0    drone.py:21                                   */
  double gravity;           /* 9.81   drone.py:22                                   */
  double inertia[3];        /* 0.005, 0.005, 0.01   drone.py:24                     */
  double arm_length;        /* 0.5    drone.py:36                                   */
  double k_yaw;             /* 0.01   drone.py:40                                   */
  double reward_scale;      /* 0.01   drone.py:142 / vectorized_drone.py:205        */
  double bonus_radius;      /* 0.05   drone.py:147   | 1.0  vectorized_drone.py:207 */
  double bonus;             /* 1.0    drone.py:148                                  */
  double z_floor;           /* 0.0    drone.py:154                                  */
  double r_max;             /* 50.0   drone.py:154                                  */
  double fixed_target[3];   /* 0,0,10 vectorized_drone.py:30 (when !RANDOMIZED)     */
  double fixed_start[3];    /* .1,.1,.1 vectorized_drone.py:50 (when !RANDOMIZED)   */
  double start_z;           /* 1.0    drone.py:57                                   */
  double target_z;          /* 1.0 + add(=0)   drone.py:30,73                       */
  double curriculum_step;   /* 0.1    drone.py:70                                   */
  int32_t curriculum_period;/* 2000   drone.py:68                                   */
  int32_t max_steps;        /* 200    drone.py:43    | 1000 vectorized_drone.py:33  */
  int32_t obs_dim;          /* 15     drone.py:79    | 12   vectorized_drone.py:61  */
  uint32_t flags;           /* DRONECU_RANDOMIZED | DRONECU_AUTORESET               */
} dronecu_config;

typedef struct dronecu_env dronecu_env;

/* Where the K-step kernel takes its motor forces from. */
typedef enum {
  DRONECU_ACTIONS_STREAMED = 0, /* d_actions[K,n,4] float32, used as given (the env never clips: drone.py:103) */
  DRONECU_ACTIONS_UNIFORM = 1   /* in-kernel Philox U[0, motor_max) -- the "random actions" workload        */
} dronecu_action_mode;

/* Optional outputs of dronecu_rollout; any pointer may be NULL (that output is not written). */
typedef struct dronecu_rollout_out {
  float* d_obs0;        /* [n,D]    observation before the first step                              */
  float* d_next_obs;    /* [K,n,D]  observation returned by step k (post auto-reset, as VecEnv.step) */
  float* d_actions;     /* [K,n,4]  action applied at step k (useful with ACTIONS_UNIFORM)          */
  float* d_reward;      /* [K,n]    float32 reward (SB3's DummyVecEnv stores float32)               */
  uint8_t* d_done;      /* [K,n]    crash | out-of-range | time limit (drone.py:154-157)            */
  uint8_t* d_truncated; /* [K,n]    time limit only (Gymnasium's `truncated`)                       */
} dronecu_rollout_out;

/* Outputs of dronecu_step / dronecu_step_host (device resp. host pointers); d_obs, d_reward and
 * d_done are what VecEnv.step_wait returns, the rest is what SB3 puts into `infos`.  Any pointer
 * may be NULL.  The three "where done" arrays are only written in rows whose done flag is set. */
typedef struct dronecu_step_out {
  float* d_obs;          /* [n,D]  next observation (after the auto-reset, if any)              */
  float* d_reward;       /* [n]    float32                                                      */
  uint8_t* d_done;       /* [n]                                                                 */
  uint8_t* d_truncated;  /* [n]    time limit only                                              */
  float* d_terminal_obs; /* [n,D]  where done: pre-reset observation (info["terminal_observation"]) */
  float* d_episode_r;    /* [n]    where done: VecMonitor episode return (info["episode"]["r"])  */
  int32_t* d_episode_l;  /* [n]    where done: VecMonitor episode length (info["episode"]["l"])  */
} dronecu_step_out;

/* SoA view used by get/set state; any pointer may be NULL.  All device pointers. */
typedef struct dronecu_state_view {
  float* d_pos;     /* [n,3]  DroneEnv.pos    drone.py:57  */
  float* d_vel;     /* [n,3]  DroneEnv.vel    drone.py:58  */
  float* d_euler;   /* [n,3]  DroneEnv.euler  drone.py:59  */
  float* d_omega;   /* [n,3]  DroneEnv.omega  drone.py:60  */
  float* d_target;  /* [n,3]  DroneEnv.target drone.py:73  */
  int32_t* d_step;  /* [n]    DroneEnv.current_step drone.py:66 */
  int32_t* d_ep_num;/* [n]    DroneEnv.ep_num drone.py:61  */
  int32_t* d_ep_len;/* [n]    VecMonitor episode length    */
  float* d_ep_ret;  /* [n]    VecMonitor episode return    */
} dronecu_state_view;

/* Episode statistics accumulated on the device since the last reset of the counters
 * (what SB3's VecMonitor feeds `rollout/ep_rew_mean`, `rollout/ep_len_mean`). */
typedef struct dronecu_stats {
  uint64_t episodes;   /* finished episodes                            */
  uint64_t terminated; /* of which ended by crash / out of range       */
  uint64_t truncated;  /* of which ended by the time limit only        */
  uint64_t length_sum; /* sum of episode lengths                       */
  double return_sum;   /* sum of episode returns (float32 accumulated) */
  uint64_t env_steps;  /* env-steps executed                           */
} dronecu_stats;

int dronecu_version(void);
const char* dronecu_last_error(void);

/* Reference defaults: DroneEnv/DroneGymEnv (drone.py:14-46, :254-264) wrapped the way
 * train.py:18-20 wraps it (auto-reset), and VectorizedDroneEnv (vectorized_drone.py:13-36). */
void dronecu_config_single(dronecu_config* cfg);
void dronecu_config_vector(dronecu_config* cfg);

/* DroneGymEnv() x n_envs / VectorizedDroneGymEnv(batch_size=n_envs): allocates the state on
 * `device` and performs the constructor's reset (drone.py:46, vectorized_drone.py:36), so a
 * fresh env has ep_num == 1.  Env i has global id env_offset + i; all randomness is keyed by
 * (seed, global id), so results do not depend on how envs are sharded over GPUs.
 * 1 <= n_envs <= 2^30 per handle (80 bytes of state each; the kernels index envs with 32 bits). */
int dronecu_create(const dronecu_config* cfg, int device, int64_t n_envs, int64_t env_offset,
                   uint64_t seed, dronecu_env** out);
int dronecu_destroy(dronecu_env* env);

int64_t dronecu_num_envs(const dronecu_env* env);
int dronecu_obs_dim(const dronecu_env* env);
int64_t dronecu_global_step(const dronecu_env* env); /* steps taken since create (Philox index) */
int dronecu_set_global_step(dronecu_env* env, int64_t t); /* checkpoint restore of that index */
double dronecu_motor_max(const dronecu_env* env);    /* 3*m*g/4, drone.py:263 */

/* DroneGymEnv.reset (drone.py:270-271, :48-75) / VectorizedDroneGymEnv.reset
 * (vectorized_drone.py:265-266, :38-57).  d_mask [n] (NULL = every env): rows with a
 * non-zero byte are reset.  d_obs [n,D] (nullable) receives the observation of ALL rows. */
int dronecu_reset(dronecu_env* env, const uint8_t* d_mask, float* d_obs, void* stream);

/* DroneGymEnv.step (drone.py:266-268, :81-159) under DummyVecEnv.step_wait + VecMonitor, or
 * VectorizedDroneGymEnv.step (vectorized_drone.py:262-263, :135-216).  d_actions [n,4] float32,
 * 16-byte aligned, used as given (no clipping, no validation -- like the reference). */
int dronecu_step(dronecu_env* env, const float* d_actions, const dronecu_step_out* out, void* stream);

/* K consecutive steps in ONE launch; the state stays in registers between steps.  Equivalent
 * to K calls of dronecu_step (bit-identical results). */
int dronecu_rollout(dronecu_env* env, int K, int action_mode, const float* d_actions,
                    const dronecu_rollout_out* out, void* stream);

/* Same as dronecu_step but with HOST buffers (numpy arrays): the H2D copy of the actions,
 * the kernel and the D2H copies of obs / reward / done all happen inside the call, through
 * pinned staging buffers owned by the handle.  This is what DroneVecEnv.step_wait uses. */
int dronecu_step_host(dronecu_env* env, const float* h_actions, const dronecu_step_out* host_out);
int dronecu_reset_host(dronecu_env* env, const uint8_t* h_mask, float* h_obs);

/* Attribute access (`env.pos`, `get_attr('pos')`: traj_tb.py:34) and teacher-forced tests. */
int dronecu_get_state(dronecu_env* env, const dronecu_state_view* view, void* stream);
int dronecu_set_state(dronecu_env* env, const dronecu_state_view* view, void* stream);
int dronecu_get_state_host(dronecu_env* env, const dronecu_state_view* host_view);
int dronecu_set_state_host(dronecu_env* env, const dronecu_state_view* host_view);

/* VecMonitor totals.  Synchronises the handle's work first.  reset != 0 zeroes the counters. */
int dronecu_episode_stats(dronecu_env* env, dronecu_stats* h_out, int reset);

/* Number of kernel launches this handle has issued (bench.py's gpu_launches). */
uint64_t dronecu_launch_count(const dronecu_env* env);

/* ------------------------------------------------------------------------------------------------
 * PPO hot path (SB3 `PPO("MlpPolicy", env)` with every default: reference train.py:36-43).  The
 * algorithm lives in stable-baselines3, which is NOT in the reference tree (environment.yaml:16);
 * these entry points restate its published behaviour -- parity unpinned (DESIGN.md).
 *
 * Policy parameters are ONE flat float32 device vector of DRONECU_POLICY_PARAMS values:
 *   pi.W1[64,15] pi.b1[64] pi.W2[64,64] pi.b2[64] pi.W3[4,64] pi.b3[4]
 *   vf.W1[64,15] vf.b1[64] vf.W2[64,64] vf.b2[64] vf.W3[1,64] vf.b3[1]  log_std[4]
 * (torch.nn.Linear [out,in] row-major blocks).
 * ---------------------------------------------------------------------------------------------- */
#define DRONECU_POLICY_PARAMS 10697
#define DRONECU_GRAD_LEN (DRONECU_POLICY_PARAMS + 8) /* gradient sums + 8 statistics sums */

/* Rollout-buffer outputs of dronecu_rollout_policy; any pointer may be NULL. */
typedef struct dronecu_policy_out {
  float* d_obs;        /* [K,n,15] observation each action was computed from (RolloutBuffer.observations) */
  float* d_actions;    /* [K,n,4]  sampled action, unclipped (RolloutBuffer.actions)                      */
  float* d_logp;       /* [K,n]    log-probability of the sampled action                                  */
  float* d_value;      /* [K,n]    value estimate                                                         */
  float* d_reward;     /* [K,n]                                                                           */
  uint8_t* d_done;     /* [K,n]    episode ended at step k (== episode_start of step k+1)                 */
  float* d_last_value; /* [n]      V(observation after the K-th step), the GAE bootstrap                  */
  float* d_last_obs;   /* [n,15]   that observation                                                       */
  int32_t obs_padded;  /* != 0: d_obs rows are 64 bytes -- [K,n,16], the 16th value written as 1.0 (the bias column of the
                          update kernels' X tile); pass the buffer to dronecu_ppo_grad_strided with obs_stride 16          */
  int32_t reserved;
} dronecu_policy_out;

/* SB3 collect_rollouts for K steps in ONE launch: per step a,v,logp = policy(obs); env.step(clip(a));
 * auto-reset; episode statistics.  The env must use obs_dim 15 and DRONECU_AUTORESET.
 * deterministic != 0: a = mean (PPO.predict(deterministic=True), reference test.py:14). */
int dronecu_rollout_policy(dronecu_env* env, int K, const float* d_params, int deterministic,
                           const dronecu_policy_out* out, void* stream);

/* Which float32 kernel dronecu_rollout_policy launches: 0 = automatic (default: one WARP per env -- the hidden units of a layer
 * spread over the lanes -- up to 8192 envs, where a thread-per-env step is a 20 us chain of dependent FMAs; one THREAD per env
 * above), 1 = always thread per env, 2 = always warp per env.  Process-wide; both kernels compute the same float32 arithmetic
 * (identical hidden layers, the head sums are warp reductions in the warp kernel). */
int dronecu_set_rollout_kernel(int mode);

/* Tensor-core variant (tcgen05 + TMEM, tf32 products, fp32 accumulation, tanh.approx): same contract,
 * outputs within ~2e-3 of dronecu_rollout_policy's; the fp32 entry point stays the parity path. */
int dronecu_rollout_policy_tc(dronecu_env* env, int K, const float* d_params, int deterministic,
                              const dronecu_policy_out* out, void* stream);
/* d_dbg1 / d_dbg2 (nullable, [B,128] each): layer-1 / layer-2 pre-activations (pi 0..63 | vf 64..127). */
int dronecu_policy_forward_tc(int device, int64_t B, const float* d_params, const float* d_obs, float* d_mean,
                              float* d_value, float* d_dbg1, float* d_dbg2, void* stream);

/* policy(obs): mean [B,4] and value [B] for arbitrary observation rows d_obs [B,15]
 * (PPO.predict / policy.forward: reference train.py:48-50, test.py:14).  Outputs nullable. */
int dronecu_policy_forward(int device, int64_t B, const float* d_params, const float* d_obs, float* d_mean,
                           float* d_value, void* stream);

/* RolloutBuffer.compute_returns_and_advantage: GAE(gamma, lambda) over [K,n] buffers. */
int dronecu_gae(int device, int K, int64_t n, const float* d_reward, const float* d_value, const uint8_t* d_done,
                const float* d_last_value, float gamma, float lam, float* d_advantage, float* d_returns, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Observation and reward normalisation (SB3 VecNormalize(norm_obs, norm_reward) inside the fused rollout; csrc/obs_norm.cuh,
 * DESIGN.md section 9).  The running statistics are FROZEN for one rollout launch: rollout i normalises with the
 * statistics as they stood after rollout i-1, then its moments are merged in one update (SB3 updates after every step).
 * Per rollout, on one stream (nothing here synchronises; every call can be captured in a CUDA graph):
 *   dronecu_rollout_policy_norm(..., d_affine)   towers see the normalised rows, the buffer receives the raw rows
 *   dronecu_norm_pass                            buffer rows -> normalised in place, rewards -> normalised, moments
 *   dronecu_norm_reduce                          CTA partials -> one moment record (fixed order: bit-reproducible)
 *   [data parallel: sum the DRONECU_NORM_MOMENTS doubles over the ranks, e.g. dronecu_ppo_dp_allreduce_f64]
 *   dronecu_norm_combine                         parallel-variance update of the statistics, next affine record
 * Layouts (device memory):
 *   affine  float32 [31]: mean_f[15] | rstd_f[15] | clip_obs;  x_norm = min(max((x - mean_f) * rstd_f, -clip), clip) with
 *           a round-to-nearest subtract and multiply (no FMA), rstd_f = (float)(1 / sqrt(var + epsilon)); the clip keeps
 *           NaN (np.clip), for the observations and the rewards alike
 *   stats   float64 [34]: obs_mean[15] | obs_var[15] | obs_count | ret_mean | ret_var | ret_count  (SB3 RunningMeanStd;
 *           initial state mean 0, var 1, count 1e-4)
 *   moments float64 [34]: sum(x - c)[15] | sum((x - c)^2)[15] | obs count | sum(ret - c_r) | sum((ret - c_r)^2) | return
 *           count, where c, c_r are the running means the pass read (a shift, so that features far from zero do not cancel)
 * ---------------------------------------------------------------------------------------------- */
#define DRONECU_NORM_AFFINE 31
#define DRONECU_NORM_STATS 34
#define DRONECU_NORM_MOMENTS 34
#define DRONECU_NORM_BLOCK 256 /* envs per CTA of dronecu_norm_pass: ceil(n / 256) partial records */

/* dronecu_rollout_policy (tensor_cores == 0) or dronecu_rollout_policy_tc (!= 0) whose towers see every observation, and
 * the bootstrap observation, normalised with d_norm_affine [DRONECU_NORM_AFFINE].  out->d_obs / d_last_obs still receive
 * the RAW rows.  d_norm_affine == NULL: exactly dronecu_rollout_policy / _tc (same kernels, same results). */
int dronecu_rollout_policy_norm(dronecu_env* env, int K, const float* d_params, int deterministic,
                                const dronecu_policy_out* out, const float* d_norm_affine, int tensor_cores, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Time-limit bootstrap (SB3 handle_timeout_termination: Gymnasium `truncated` / info["TimeLimit.truncated"]; csrc/ppo_timeout.cuh,
 * DESIGN.md section 11).  A step that ends by the time limit alone (timeout && !crashed) gets
 *   reward += f32(f32(gamma) * V(terminal observation))
 * while done stays set (GAE starts a new episode there).  Per rollout, on one stream:
 *   dronecu_rollout_policy_timeouts   the rollout of dronecu_rollout_policy_norm that also records each truncated step's raw
 *                                     pre-reset observation and buffer row in a dronecu_timeout_buf
 *   [dronecu_norm_pass]               rewards normalised first (SB3 adds gamma * V to the VecNormalize reward)
 *   dronecu_bootstrap_timeouts        the float32 value tower on each recorded row (normalised with the rollout's affine
 *                                     record), added to its reward in place
 *   [dronecu_norm_reduce / _combine]  afterwards: the combine overwrites the affine record
 * ---------------------------------------------------------------------------------------------- */
typedef struct dronecu_timeout_buf {
  float* d_obs;          /* [T,n,16] 16-byte aligned: the raw pre-reset observation (info["terminal_observation"]), 16th = 1.0 */
  int32_t* d_row;        /* [T,n]    its rollout-buffer row k * n + i, -1 in an unused slot; env i's j-th truncation of the
                            launch goes to slot j * n + i                                                                    */
  int32_t slots_per_env; /* T >= ceil(K / max_steps): an env truncates at most that often in K steps                        */
} dronecu_timeout_buf;

/* dronecu_rollout_policy_norm (same kernels' choice and results) that also fills *timeouts; every slot is written (row or -1).
 * DRONECU_ERR_INVALID when slots_per_env < ceil(K / max_steps), K * n or slots_per_env * n exceed INT32_MAX, a pointer is
 * NULL or d_obs is misaligned. */
int dronecu_rollout_policy_timeouts(dronecu_env* env, int K, const float* d_params, int deterministic,
                                    const dronecu_policy_out* out, const float* d_norm_affine, int tensor_cores,
                                    const dronecu_timeout_buf* timeouts, void* stream);
/* d_reward[row] = d_reward[row] + f32(gamma * V(norm(d_obs[slot]))) for every slot with row >= 0 of the n envs, V the float32
 * value tower of dronecu_policy_forward (bit-identical to it on the same row); d_norm_affine NULL: rows used raw. */
int dronecu_bootstrap_timeouts(int device, const float* d_params, const dronecu_timeout_buf* timeouts, int64_t n,
                               const float* d_norm_affine, float gamma, float* d_reward, void* stream);

/* One thread per env walks its K steps of the step-major buffers [K,n,...]. */
typedef struct dronecu_norm_pass_args {
  float* d_obs;             /* [K,n,obs_stride] raw rows, rewritten normalised; NULL: observations untouched, no obs moments */
  int32_t obs_stride;       /* 15 or 16 (64-byte rows: the 16th value is kept, 1.0)                                         */
  int32_t K;
  int64_t n;
  const float* d_affine;    /* [31] the record the rollout used (required with d_obs)                                       */
  float* d_reward;          /* [K,n] raw in, out clip(r / sqrt(ret_var + epsilon), +-clip_reward) (float64, then cast); NULL: off */
  const uint8_t* d_done;    /* [K,n] the per-env return restarts after done (in both modes, as SB3's returns[dones] = 0)     */
  double* d_returns;        /* [n] per-env discounted return ret = ret * gamma + r, persistent across rollouts (required with d_reward) */
  const double* d_stats;    /* [34] running statistics (moment shift, reward scale)                                         */
  double gamma, epsilon, clip_reward;
  int32_t update;           /* != 0 (training): returns advance, d_partials written; 0 (evaluation): statistics untouched,
                               returns only zeroed at dones                                                                 */
  int32_t side_env;         /* >= 0 with d_side_obs: copy that env's raw rows to d_side_obs [K,15] before normalising       */
  float* d_side_obs;
  double* d_partials;       /* [ceil(n / DRONECU_NORM_BLOCK), DRONECU_NORM_MOMENTS] scratch, one record per CTA (update != 0) */
} dronecu_norm_pass_args;
int dronecu_norm_pass(int device, const dronecu_norm_pass_args* args, void* stream);
/* d_moments [34] = fixed-order sum of the n_partials records of dronecu_norm_pass (written, not accumulated). */
int dronecu_norm_reduce(int device, const double* d_partials, int64_t n_partials, double* d_moments, void* stream);
/* d_moments != NULL: merge the batch into d_stats (SB3 RunningMeanStd.update_from_moments, float64; a part whose count is 0
 * is skipped).  Then, d_affine != NULL: write the affine record of d_stats (clip = clip_obs). */
int dronecu_norm_combine(int device, double* d_stats, const double* d_moments, double epsilon, float clip_obs, float* d_affine,
                         void* stream);

/* ------------------------------------------------------------------------------------------------
 * Policy evaluation: SB3 evaluate_policy(model, VecMonitor(DummyVecEnv([DroneGymEnv] * N)), n_eval_episodes, deterministic)
 * with the actor alone (csrc/ppo_eval.cuh, DESIGN.md section 10).  Env g (global index among the N = n_global evaluation envs)
 * records target_g = (n_eval_episodes + g) / N episodes; all envs step in lockstep until every env has reached its target,
 * T steps in all.  Step c of an env uses the noise index t0 + c, as dronecu_rollout_policy does.  The caller resets the envs
 * first, then issues probe launches (each env runs until its target or step `limit`; *d_pending counts the envs still
 * below target) until no env is pending, then ONE catch-up launch with limit = T = max(d_steps): every env has then been
 * stepped exactly T times.  The env clock (dronecu_global_step) is not advanced: the caller sets it to t0 + T.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dronecu_eval_args {
  int64_t t0;              /* env clock at the first step of the evaluation                                          */
  int32_t limit;           /* probe: run up to this step (absolute, counted from the reset); catch-up: T              */
  int32_t catch_up;        /* 0 = probe, 1 = catch-up                                                               */
  int32_t deterministic;   /* != 0: action = clip(mean); else clip(mean + std * z), z from the rollout's noise stream */
  int32_t max_eps;         /* row stride of d_ep_return / d_ep_length: >= ceil(n_eval_episodes / n_global)           */
  int64_t env_index0;      /* global index of this handle's env 0 among the n_global evaluation envs                  */
  int64_t n_global;
  int64_t n_eval_episodes; /* >= 1                                                                                   */
  int32_t* d_steps;        /* [n] steps taken since the reset (zero before the first launch), updated                 */
  int32_t* d_count;        /* [n] episodes recorded (zero before the first launch), updated                           */
  float* d_ep_return;      /* [n, max_eps] VecMonitor return of each recorded episode (float32, raw reward)           */
  int32_t* d_ep_length;    /* [n, max_eps] its length                                                               */
  int32_t* d_pending;      /* probe: += number of envs still below their target (zero it first)                       */
} dronecu_eval_args;

/* One launch (probe or catch-up).  d_norm_affine != NULL: the policy sees observations normalised with that record
 * (nothing is updated).  tensor_cores != 0: the tcgen05 kernel (tf32), else the float32 kernel dronecu_set_rollout_kernel
 * selects for dronecu_rollout_policy.  Needs the 15-dim observation and DRONECU_AUTORESET. */
int dronecu_evaluate_policy(dronecu_env* env, const float* d_params, const float* d_norm_affine, int tensor_cores,
                            const dronecu_eval_args* args, void* stream);

typedef struct dronecu_ppo_config {
  float learning_rate; /* 3e-4  */
  float beta1, beta2;  /* 0.9, 0.999 */
  float adam_eps;      /* 1e-5  */
  float clip_range;    /* 0.2   */
  float vf_coef;       /* 0.5   */
  float ent_coef;      /* 0.0   */
  float max_grad_norm; /* 0.5   */
} dronecu_ppo_config;

typedef struct dronecu_ppo dronecu_ppo; /* optimiser handle: Adam moments, step count, scratch */

void dronecu_ppo_config_default(dronecu_ppo_config* cfg); /* the SB3 defaults listed above */
int dronecu_ppo_create(const dronecu_ppo_config* cfg, int device, dronecu_ppo** out);
int dronecu_ppo_destroy(dronecu_ppo* ppo);

/* Minibatch order of one epoch: d_out[0..n) = a pseudo-random permutation of 0..n-1 keyed by (seed, epoch).
 * Replaces SB3's np.random.permutation(buffer_size) (RolloutBuffer.get, called from PPO.train; call site
 * reference train.py:63) with a keyed bijection evaluated per element on the device -- no sort.  The exact
 * function is restated in oracle/philox.py (minibatch_permutation); n < 2^31. */
int dronecu_minibatch_permutation(int device, int64_t n, uint64_t seed, uint64_t epoch, int32_t* d_out, void* stream);

/* The minibatches of one epoch with SORTED rows: the same keyed bijection f read the other way round -- buffer row r belongs
 * to minibatch f(r) / batch (a uniformly random partition into minibatches of exactly `batch` rows; the last one takes the
 * remainder) -- and d_out[b * batch .. (b + 1) * batch) lists minibatch b's rows in ascending order (stable counting sort by
 * minibatch id).  A minibatch gradient is a sum over its rows, so the order inside a minibatch is free; ascending rows make
 * the update kernels' gathers a forward sweep over the rollout buffer instead of random 60-byte reads.  At most 64
 * minibatches per epoch (DRONECU_ERR_UNSUPPORTED beyond: use dronecu_minibatch_permutation).  oracle/philox.py:
 * minibatch_partition. */
int dronecu_minibatch_partition(dronecu_ppo* ppo, int64_t n, int64_t batch, uint64_t seed, uint64_t epoch, int32_t* d_out,
                                void* stream);

/* sum, sum of squares and count of the advantages of a minibatch, ACCUMULATED into d_out[3] (float64;
 * zero it first).  Minibatch = rows d_index[0..m) of the flat buffers, or rows first..first+m when
 * d_index is NULL.  (Data-parallel training all-reduces d_out before forming mean / std.) */
int dronecu_ppo_adv_stats(dronecu_ppo* ppo, const float* d_adv, const int32_t* d_index, int64_t first, int64_t m,
                          double* d_out, void* stream);

/* The same statistics for every minibatch of an epoch in two launches: minibatch b = rows d_index[b * batch ..
 * min((b + 1) * batch, B)) (rows themselves when d_index is NULL); d_out[n_mb][3] is WRITTEN ([sum, sumsq, count] per
 * minibatch; all-reduce the whole array once per epoch for data-parallel training).  At most n_sm * 8 minibatches. */
int dronecu_ppo_adv_stats_epoch(dronecu_ppo* ppo, const float* d_adv, const int32_t* d_index, int64_t B, int64_t batch,
                                double* d_out, void* stream);

/* Forward + backward of one minibatch: d_grad[DRONECU_GRAD_LEN] = SUM over the minibatch of the
 * per-sample loss gradient (clipped surrogate + vf_coef * value MSE + ent_coef * entropy), followed by
 * the sums of: policy loss, squared value error, approx_kl, clip fraction, sample count.  Advantages
 * enter as (adv - adv_mean) * adv_inv_std; when d_adv_stats (the [sum, sumsq, count] written by
 * dronecu_ppo_adv_stats) is not NULL, mean and 1/(unbiased std + 1e-8) are formed from it on the
 * device instead -- no host round trip; with a count of 1 or less the raw advantages are used (SB3
 * normalises only a minibatch of more than one sample; the count is global over data-parallel ranks).
 * Deterministic for a fixed launch configuration. */
int dronecu_ppo_grad(dronecu_ppo* ppo, const float* d_params, const float* d_obs, const float* d_actions,
                     const float* d_old_logp, const float* d_adv, const float* d_returns, const int32_t* d_index,
                     int64_t first, int64_t m, float adv_mean, float adv_inv_std, const double* d_adv_stats,
                     float* d_grad, void* stream);
/* Same contract on the tcgen05 tensor cores: tf32 products with fp32 accumulation, MUFU tanh; the seven
 * matrix products of each tower run as tcgen05.mma with the weight-gradient accumulators resident in
 * TMEM (csrc/ppo_update_tc.cuh).  Agrees with dronecu_ppo_grad to ~1e-3 of each block's largest entry. */
int dronecu_ppo_grad_tc(dronecu_ppo* ppo, const float* d_params, const float* d_obs, const float* d_actions,
                        const float* d_old_logp, const float* d_adv, const float* d_returns, const int32_t* d_index,
                        int64_t first, int64_t m, float adv_mean, float adv_inv_std, const double* d_adv_stats,
                        float* d_grad, void* stream);

/* Same contract, three sample tiles in flight per SM: forward and activation-gradient products as above (tf32, A operand
 * in TMEM), the four weight-gradient products with bf16 operands (kind::f16, fp32 accumulation; dW2 and db2 fused into
 * one N = 72 product), tanh'(layer 1) stashed as bf16 (csrc/ppo_update_tc3.cuh).  Bit-reproducible (the issuer serves
 * the warpgroups in a fixed rotation).  Agrees with dronecu_ppo_grad to a few 1e-3 of each block's largest entry. */
int dronecu_ppo_grad_bf16(dronecu_ppo* ppo, const float* d_params, const float* d_obs, const float* d_actions,
                          const float* d_old_logp, const float* d_adv, const float* d_returns, const int32_t* d_index,
                          int64_t first, int64_t m, float adv_mean, float adv_inv_std, const double* d_adv_stats,
                          float* d_grad, void* stream);

/* The three gradient kernels behind one entry point, with the row stride of d_obs: mode 0 = dronecu_ppo_grad (fp32), 1 =
 * dronecu_ppo_grad_tc, 2 = dronecu_ppo_grad_bf16; obs_stride 15 = packed rows (what the entry points above assume), 16 = the
 * 64-byte rows dronecu_rollout_policy[_tc] writes with obs_padded (16-byte aligned; the bf16 kernel then fetches a row as four
 * 128-bit chunks and stages it with vector stores). */
int dronecu_ppo_grad_strided(dronecu_ppo* ppo, int mode, int obs_stride, const float* d_params, const float* d_obs,
                             const float* d_actions, const float* d_old_logp, const float* d_adv, const float* d_returns,
                             const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                             const double* d_adv_stats, float* d_grad, void* stream);

/* Debugging aid for dronecu_ppo_grad_tc: when d_dbg is not NULL the next calls also dump the raw TMEM image
 * of every warpgroup, float32 [2 * grid.x, 128 lanes, 256 columns] (policy-tower CTAs; grid.x = min(ceil(tiles / 2), SMs / 2)) (grid = min(ceil(tiles / 2), SM count)). */
int dronecu_ppo_debug_buffer(dronecu_ppo* ppo, float* d_dbg);

/* clip_grad_norm_(max_grad_norm) + Adam.step() in place on d_params.  d_grad is the (all-reduced)
 * output of dronecu_ppo_grad, inv_count = 1 / (global minibatch size).  d_info (nullable) receives
 * [policy_loss, value_loss, approx_kl, clip_fraction, count, -, -, -, grad_norm]. */
int dronecu_ppo_apply(dronecu_ppo* ppo, float* d_params, const float* d_grad, double inv_count, float* d_info,
                      void* stream);
/* d_info_sum (nullable, caller-owned, float32 [10]): from now on every dronecu_ppo_apply / dronecu_ppo_apply_dp ADDS
 * its [policy_loss, value_loss, approx_kl, clip_fraction, count, -, -, -, grad_norm] and 1 (number of steps) into it --
 * SB3's PPO.train() logs the mean over all minibatches of all epochs, not the last minibatch's values. */
int dronecu_ppo_set_info_accumulator(dronecu_ppo* ppo, float* d_info_sum);
int64_t dronecu_ppo_num_updates(const dronecu_ppo* ppo);
/* Adam state access for checkpoints: copies [m | v] (2 * DRONECU_POLICY_PARAMS floats) device <-> device. */
int dronecu_ppo_get_state(dronecu_ppo* ppo, float* d_moments, int64_t* h_step, void* stream);
int dronecu_ppo_set_state(dronecu_ppo* ppo, const float* d_moments, int64_t step, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Data-parallel update over NVLink peer memory (csrc/ppo_dp.cuh).  The reference is single-process (train.py:33-43:
 * one env, device="cpu"); this is the exchange north_star's configs[4] adds ("NCCL grad allreduce"), done as ONE
 * kernel per optimiser step: every rank pushes its 42.8 KB sum-form gradient into a mailbox slot in each peer's HBM,
 * publishes a flag (st.release.sys), waits for the flags of all ranks on its own mailbox, sums the slots in fixed rank
 * order (bit-identical on every rank) and runs clip_grad_norm_ + Adam.  Plain launches on the caller's stream:
 * CUDA-graph capturable, no host synchronisation, no NCCL call per step.
 *
 * Set-up, once per optimiser handle: every rank calls dronecu_ppo_dp_alloc, the 64-byte IPC handles are exchanged by
 * the host (torch.distributed all_gather in drone_rl_b200/ppo.py), then dronecu_ppo_dp_connect maps the peers'
 * mailboxes (cudaIpcOpenMemHandle; within one process pass the raw mailbox pointers instead).  A host barrier must
 * separate connect from the first exchange, and the last exchange from dronecu_ppo_destroy.
 * ---------------------------------------------------------------------------------------------- */
#define DRONECU_IPC_HANDLE_BYTES 64
#define DRONECU_DP_MAX_WORLD 16
int dronecu_ppo_dp_alloc(dronecu_ppo* ppo, int rank, int world, void* ipc_handle_out /* [64], nullable */,
                         void** d_mailbox_out /* nullable */);
/* ipc_handles: [world][64] bytes (entry `rank` ignored), or NULL with d_mailboxes[world] = raw device pointers of
 * mailboxes allocated in THIS process (peer access is enabled as needed).  `world` must equal the world passed to
 * dronecu_ppo_dp_alloc (the mailbox is sized for it), and a handle connects once: DRONECU_ERR_INVALID otherwise. */
int dronecu_ppo_dp_connect(dronecu_ppo* ppo, int world, const void* ipc_handles, void* const* d_mailboxes);
/* A rank that waits longer than this for its peers (default 30 s) raises the status flag instead of hanging the GPU. */
int dronecu_ppo_dp_set_timeout(dronecu_ppo* ppo, double seconds);
/* *h_status: 0 = ok, 1 = an exchange timed out (every result after it is invalid); *h_exchanges: exchanges done. */
int dronecu_ppo_dp_status(dronecu_ppo* ppo, int* h_status, int64_t* h_exchanges);
/* In-place sum over the ranks of n <= 5376 float64 values (advantage / episode statistics), rank order fixed. */
int dronecu_ppo_dp_allreduce_f64(dronecu_ppo* ppo, double* d_buf, int n, void* stream);
/* dronecu_ppo_apply for data-parallel training: d_grad (the LOCAL output of dronecu_ppo_grad*, 16-byte aligned) is
 * replaced by its sum over the ranks, the denominator is the summed sample count d_grad[DRONECU_POLICY_PARAMS + 4]
 * (ranks may hold minibatches of different sizes), then clip + Adam as dronecu_ppo_apply.  Every rank must call it
 * the same number of times. */
int dronecu_ppo_apply_dp(dronecu_ppo* ppo, float* d_params, float* d_grad, float* d_info, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRONECU_H */
