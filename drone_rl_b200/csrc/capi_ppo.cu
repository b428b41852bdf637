// C ABI of the PPO half of libdronecu.so (include/dronecu.h): in-kernel policy rollout, GAE,
// minibatch gradient, clip + Adam.  Plain pointers, no torch types, no CPU fallback.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>

#include "../../include/dronecu.h"
#include "capi_common.h"
#include "env_handle.h"
#include "ppo_update.cuh"
#include "ppo_rollout_tc.cuh"
#include "ppo_timeout.cuh"
#include "ppo_eval.cuh"
#include "ppo_update_tc.cuh"
#include "ppo_update_tc3.cuh"
#include "ppo_dp.cuh"
#include "obs_norm.cuh"

using namespace dronecu;

static_assert(kParams == DRONECU_POLICY_PARAMS, "header / kernel parameter count mismatch");
static_assert(kGradLen == DRONECU_GRAD_LEN, "header / kernel gradient length mismatch");

struct dronecu_ppo {
  dronecu_ppo_config cfg;
  int device;
  int n_sm;
  float* partials;   // [2 * n_sm, kGradLen] (the tensor-core kernel writes one vector per warpgroup)
  float* moments;    // [2, kParams]  Adam m | v
  double* adv_partials; // [n_sm * 8, 2]
  uint32_t* part_hist;  // scratch of dronecu_minibatch_partition (grown on demand)
  size_t part_hist_len;
  long long* d_step; // device-resident AdamClock {step count, beta1^step, beta2^step} (ppo_apply*_kernel advance it)
  uint64_t launches;
  float* dbg;        // see dronecu_ppo_debug_buffer
  float* info_sum;   // see dronecu_ppo_set_info_accumulator (caller-owned, nullable)
  // data-parallel exchange over peer memory (ppo_dp.cuh)
  DpArgs dp;         // dp.world == 0: not set up
  float* dp_mail;    // this rank's mailbox (cudaMalloc: exportable with cudaIpcGetMemHandle)
  int dp_alloc_world;  // the world dp_mail was sized for: dronecu_ppo_dp_connect accepts only this one
  bool dp_opened[kDpMaxWorld];   // mail[r] was mapped with cudaIpcOpenMemHandle (to be closed)
};

// 0 = automatic (one warp per env up to kWarpRolloutMaxEnvs envs, one thread per env above), 1 = always one thread per env,
// 2 = always one warp per env: dronecu_set_rollout_kernel (tests pin each kernel against the oracle)
static int g_rollout_kernel_mode = 0;
constexpr int64_t kWarpRolloutMaxEnvs = 8192;   // measured crossover ~12k envs (profiles/r02_rollout_kernel_sweep.txt)

extern "C" int dronecu_set_rollout_kernel(int mode) {
  if (mode < 0 || mode > 2) return fail(DRONECU_ERR_INVALID, "dronecu_set_rollout_kernel: mode must be 0 (auto), 1 (thread per env) or 2 (warp per env)");
  g_rollout_kernel_mode = mode;
  return DRONECU_OK;
}

enum RolloutKernel { kThreadPerEnv, kWarpPerEnv, kTensorCores };

// the kernel flavour of a rollout or an evaluation of env e: tensor cores when asked, else the float32 kernel of
// dronecu_set_rollout_kernel (small batches: one warp per env, ppo_rollout.cuh)
static RolloutKernel choose_kernel(const dronecu_env* e, bool tensor_cores) {
  if (tensor_cores) return kTensorCores;
  return (g_rollout_kernel_mode == 2 || (g_rollout_kernel_mode == 0 && e->n <= kWarpRolloutMaxEnvs)) ? kWarpPerEnv : kThreadPerEnv;
}

// f(std::bool_constant<randomized>, std::bool_constant<norm>): the kernels' RANDOMIZED and NORM template flags
template <class F>
static int with_flags(bool randomized, bool norm, F&& f) {
  if (randomized) return norm ? f(std::true_type{}, std::true_type{}) : f(std::true_type{}, std::false_type{});
  return norm ? f(std::false_type{}, std::true_type{}) : f(std::false_type{}, std::false_type{});
}

template <bool RANDOMIZED, bool NORM, bool TIMEOUT>
static int launch_policy_rollout(RolloutKernel which, int64_t n, const PolicyArgs& a, cudaStream_t st) {
  if (which == kTensorCores) {
    static_assert(tc::kTile == kPolBlock, "tile size");
    CUDA_TRY(cudaFuncSetAttribute(policy_rollout_tc_kernel<RANDOMIZED, NORM, TIMEOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmem));
    policy_rollout_tc_kernel<RANDOMIZED, NORM, TIMEOUT><<<(unsigned)((n + kPolBlock - 1) / kPolBlock), tc::kTile, kTcSmem, st>>>(a);
  } else if (which == kWarpPerEnv) {
    CUDA_TRY(cudaFuncSetAttribute(policy_rollout_warp_kernel<RANDOMIZED, NORM, TIMEOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPolicySmallSmem));
    policy_rollout_warp_kernel<RANDOMIZED, NORM, TIMEOUT><<<(unsigned)((n + kSmallWarps - 1) / kSmallWarps), 32 * kSmallWarps, kPolicySmallSmem, st>>>(a);
  } else {
    CUDA_TRY(cudaFuncSetAttribute(policy_rollout_kernel<RANDOMIZED, NORM, TIMEOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPolicySmem));
    policy_rollout_kernel<RANDOMIZED, NORM, TIMEOUT><<<(unsigned)((n + kPolBlock - 1) / kPolBlock), kPolBlock, kPolicySmem, st>>>(a);
  }
  return DRONECU_OK;
}

// the side buffer of the time-limit bootstrap: slots_per_env slots per env, 16-byte aligned 64-byte rows
static int check_timeout_buf(const dronecu_timeout_buf* tb, const char* what) {
  if (!tb || !tb->d_obs || !tb->d_row) return fail(DRONECU_ERR_INVALID, std::string(what) + ": null timeout buffer");
  if (reinterpret_cast<uintptr_t>(tb->d_obs) & 15) return fail(DRONECU_ERR_INVALID, std::string(what) + ": timeout d_obs must be 16-byte aligned");
  if (tb->slots_per_env <= 0) return fail(DRONECU_ERR_INVALID, std::string(what) + ": slots_per_env must be positive");
  return DRONECU_OK;
}

static int rollout_policy_impl(dronecu_env* e, int K, const float* d_params, int deterministic,
                               const dronecu_policy_out* out, void* stream, bool tensor_cores,
                               const float* d_norm_affine = nullptr, const dronecu_timeout_buf* tb = nullptr) {
  if (!e || !d_params) return fail(DRONECU_ERR_INVALID, "dronecu_rollout_policy: null argument");
  if (K <= 0) return fail(DRONECU_ERR_INVALID, "K must be positive");
  if (e->cfg.obs_dim != 15 || !(e->cfg.flags & DRONECU_AUTORESET))
    return fail(DRONECU_ERR_UNSUPPORTED, "policy rollout needs the 15-dim observation and DRONECU_AUTORESET");
  if (tb) {
    // an env truncates at most 1 + floor((K - 1) / max_steps) = ceil(K / max_steps) times in K steps, whatever its clock
    if ((int64_t)tb->slots_per_env < ((int64_t)K + e->cfg.max_steps - 1) / e->cfg.max_steps)
      return fail(DRONECU_ERR_INVALID, "dronecu_rollout_policy_timeouts: slots_per_env is below ceil(K / max_steps)");
    if ((int64_t)K * e->n > INT32_MAX || (int64_t)tb->slots_per_env * e->n > INT32_MAX)
      return fail(DRONECU_ERR_INVALID, "dronecu_rollout_policy_timeouts: K * n and slots_per_env * n must fit in int32");
  }
  if (out && out->d_actions && (reinterpret_cast<uintptr_t>(out->d_actions) & 15))
    return fail(DRONECU_ERR_INVALID, "out->d_actions must be 16-byte aligned");
  if (out && out->obs_padded && out->d_obs && (reinterpret_cast<uintptr_t>(out->d_obs) & 15))
    return fail(DRONECU_ERR_INVALID, "padded out->d_obs must be 16-byte aligned");
  DeviceGuard guard(e->device);
  PolicyArgs a;
  std::memset(&a, 0, sizeof(a));
  a.state = e->sp; a.P = e->P; a.n = e->n; a.K = K; a.t0 = e->t; a.theta = d_params; a.deterministic = deterministic;
  a.stats = e->stats;
  a.norm = d_norm_affine;
  if (out) {
    a.obs = out->d_obs; a.obs_padded = out->obs_padded ? 1 : 0;
    a.actions = reinterpret_cast<float4*>(out->d_actions); a.logp = out->d_logp;
    a.value = out->d_value; a.reward = out->d_reward; a.done = out->d_done; a.last_value = out->d_last_value;
    a.last_obs = out->d_last_obs;
  }
  if (tb) { a.term_obs = tb->d_obs; a.term_row = tb->d_row; a.term_slots = tb->slots_per_env; }
  const RolloutKernel which = choose_kernel(e, tensor_cores);
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = with_flags((e->cfg.flags & DRONECU_RANDOMIZED) != 0, d_norm_affine != nullptr, [&](auto R, auto N) {
    return tb ? launch_policy_rollout<R, N, true>(which, e->n, a, st) : launch_policy_rollout<R, N, false>(which, e->n, a, st);
  });
  if (rc != DRONECU_OK) return rc;
  e->launches += 1;
  CUDA_TRY(cudaGetLastError());
  e->t += (uint64_t)K;
  e->env_steps += (uint64_t)K * (uint64_t)e->n;
  return DRONECU_OK;
}

extern "C" int dronecu_rollout_policy(dronecu_env* e, int K, const float* d_params, int deterministic,
                                      const dronecu_policy_out* out, void* stream) {
  return rollout_policy_impl(e, K, d_params, deterministic, out, stream, false);
}

extern "C" int dronecu_rollout_policy_tc(dronecu_env* e, int K, const float* d_params, int deterministic,
                                         const dronecu_policy_out* out, void* stream) {
  return rollout_policy_impl(e, K, d_params, deterministic, out, stream, true);
}

extern "C" int dronecu_rollout_policy_norm(dronecu_env* e, int K, const float* d_params, int deterministic,
                                           const dronecu_policy_out* out, const float* d_norm_affine, int tensor_cores,
                                           void* stream) {
  return rollout_policy_impl(e, K, d_params, deterministic, out, stream, tensor_cores != 0, d_norm_affine);
}

extern "C" int dronecu_rollout_policy_timeouts(dronecu_env* e, int K, const float* d_params, int deterministic,
                                               const dronecu_policy_out* out, const float* d_norm_affine, int tensor_cores,
                                               const dronecu_timeout_buf* tb, void* stream) {
  const int rc = check_timeout_buf(tb, "dronecu_rollout_policy_timeouts");
  if (rc != DRONECU_OK) return rc;
  return rollout_policy_impl(e, K, d_params, deterministic, out, stream, tensor_cores != 0, d_norm_affine, tb);
}

extern "C" int dronecu_bootstrap_timeouts(int device, const float* d_params, const dronecu_timeout_buf* tb, int64_t n,
                                          const float* d_norm_affine, float gamma, float* d_reward, void* stream) {
  if (!d_params || !d_reward || n <= 0) return fail(DRONECU_ERR_INVALID, "dronecu_bootstrap_timeouts: bad argument");
  const int rc = check_timeout_buf(tb, "dronecu_bootstrap_timeouts");
  if (rc != DRONECU_OK) return rc;
  DeviceGuard guard(device);
  const int64_t slots = (int64_t)tb->slots_per_env * n;
  const unsigned grid = (unsigned)std::min<int64_t>((slots + kPolBlock - 1) / kPolBlock, 148 * 4);
  const float4* obs = reinterpret_cast<const float4*>(tb->d_obs);
  cudaStream_t st = (cudaStream_t)stream;
  if (d_norm_affine) {
    CUDA_TRY(cudaFuncSetAttribute(timeout_bootstrap_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpSmem)));
    timeout_bootstrap_kernel<true><<<grid, kPolBlock, sizeof(MlpSmem), st>>>(d_params, obs, tb->d_row, slots, d_norm_affine, gamma, d_reward);
  } else {
    CUDA_TRY(cudaFuncSetAttribute(timeout_bootstrap_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpSmem)));
    timeout_bootstrap_kernel<false><<<grid, kPolBlock, sizeof(MlpSmem), st>>>(d_params, obs, tb->d_row, slots, nullptr, gamma, d_reward);
  }
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

// ------------------------------------------------------------------------------------------------
// policy evaluation (csrc/ppo_eval.cuh)
// ------------------------------------------------------------------------------------------------
template <bool RANDOMIZED, bool NORM>
static int launch_policy_eval(RolloutKernel which, int64_t n, const EvalArgs& a, cudaStream_t st) {
  if (which == kTensorCores) {
    CUDA_TRY(cudaFuncSetAttribute(policy_eval_tc_kernel<RANDOMIZED, NORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tc::Smem)));
    policy_eval_tc_kernel<RANDOMIZED, NORM><<<(unsigned)((n + tc::kTile - 1) / tc::kTile), tc::kTile, sizeof(tc::Smem), st>>>(a);
  } else if (which == kWarpPerEnv) {
    CUDA_TRY(cudaFuncSetAttribute(policy_eval_warp_kernel<RANDOMIZED, NORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPolicySmallSmem));
    policy_eval_warp_kernel<RANDOMIZED, NORM><<<(unsigned)((n + kSmallWarps - 1) / kSmallWarps), 32 * kSmallWarps, kPolicySmallSmem, st>>>(a);
  } else {
    CUDA_TRY(cudaFuncSetAttribute(policy_eval_kernel<RANDOMIZED, NORM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpSmem)));
    policy_eval_kernel<RANDOMIZED, NORM><<<(unsigned)((n + kPolBlock - 1) / kPolBlock), kPolBlock, sizeof(MlpSmem), st>>>(a);
  }
  return DRONECU_OK;
}

extern "C" int dronecu_evaluate_policy(dronecu_env* e, const float* d_params, const float* d_norm_affine, int tensor_cores,
                                       const dronecu_eval_args* p, void* stream) {
  if (!e || !d_params || !p) return fail(DRONECU_ERR_INVALID, "dronecu_evaluate_policy: null argument");
  if (e->cfg.obs_dim != 15 || !(e->cfg.flags & DRONECU_AUTORESET))
    return fail(DRONECU_ERR_UNSUPPORTED, "policy evaluation needs the 15-dim observation and DRONECU_AUTORESET");
  if (!p->d_steps || !p->d_count || !p->d_ep_return || !p->d_ep_length || (!p->catch_up && !p->d_pending))
    return fail(DRONECU_ERR_INVALID, "dronecu_evaluate_policy: d_steps, d_count, d_ep_return, d_ep_length and (probe) d_pending are required");
  if (p->t0 < 0 || p->limit < 0 || p->n_eval_episodes < 1 || p->env_index0 < 0 || p->n_global < e->n ||
      p->env_index0 > p->n_global - e->n)
    return fail(DRONECU_ERR_INVALID, "dronecu_evaluate_policy: need t0 >= 0, limit >= 0, n_eval_episodes >= 1 and "
                                     "0 <= env_index0 <= n_global - n");
  if ((int64_t)p->max_eps < (p->n_eval_episodes + p->n_global - 1) / p->n_global)
    return fail(DRONECU_ERR_INVALID, "dronecu_evaluate_policy: max_eps is below ceil(n_eval_episodes / n_global)");
  DeviceGuard guard(e->device);
  EvalArgs a;
  std::memset(&a, 0, sizeof(a));
  a.state = e->sp; a.P = e->P; a.n = e->n; a.t0 = (uint64_t)p->t0; a.limit = p->limit; a.catch_up = p->catch_up ? 1 : 0;
  a.deterministic = p->deterministic; a.max_eps = p->max_eps; a.env_index0 = p->env_index0; a.n_global = p->n_global;
  a.n_eval_episodes = p->n_eval_episodes; a.theta = d_params; a.norm = d_norm_affine;
  a.steps = p->d_steps; a.count = p->d_count; a.ep_return = p->d_ep_return; a.ep_length = p->d_ep_length; a.pending = p->d_pending;
  const RolloutKernel which = choose_kernel(e, tensor_cores != 0);
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = with_flags((e->cfg.flags & DRONECU_RANDOMIZED) != 0, d_norm_affine != nullptr,
                            [&](auto R, auto N) { return launch_policy_eval<R, N>(which, e->n, a, st); });
  if (rc != DRONECU_OK) return rc;
  e->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

// ------------------------------------------------------------------------------------------------
// observation / reward normalisation (csrc/obs_norm.cuh)
// ------------------------------------------------------------------------------------------------
static_assert(kNormAffine == DRONECU_NORM_AFFINE && kNormStats == DRONECU_NORM_STATS && kNormMoments == DRONECU_NORM_MOMENTS &&
              kNormBlock == DRONECU_NORM_BLOCK, "header / kernel normaliser layout mismatch");

extern "C" int dronecu_norm_pass(int device, const dronecu_norm_pass_args* p, void* stream) {
  if (!p || p->K <= 0 || p->n <= 0) return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: bad argument");
  if (p->d_obs && (p->obs_stride != 15 && p->obs_stride != 16))
    return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: obs_stride must be 15 or 16");
  if (p->d_obs && p->obs_stride == 16 && (reinterpret_cast<uintptr_t>(p->d_obs) & 15))
    return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: padded d_obs must be 16-byte aligned");
  if (p->d_obs && !p->d_affine) return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: d_obs needs d_affine");
  if (p->d_reward && (!p->d_done || !p->d_stats || !p->d_returns))
    return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: d_reward needs d_done, d_stats and d_returns");
  if (p->update && (!p->d_stats || !p->d_partials)) return fail(DRONECU_ERR_INVALID, "dronecu_norm_pass: update needs d_stats and d_partials");
  DeviceGuard guard(device);
  NormPassArgs a;
  a.obs = p->d_obs; a.stride = p->obs_stride; a.K = p->K; a.n = p->n; a.affine = p->d_affine;
  a.reward = p->d_reward; a.done = p->d_done; a.returns = p->d_returns; a.stats = p->d_stats;
  a.gamma = p->gamma; a.epsilon = p->epsilon; a.clip_reward = p->clip_reward; a.update = p->update;
  a.side_env = p->side_env; a.side_obs = p->d_side_obs; a.partials = p->d_partials;
  obs_norm_pass_kernel<<<(unsigned)((p->n + kNormBlock - 1) / kNormBlock), kNormBlock, 0, (cudaStream_t)stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_norm_reduce(int device, const double* d_partials, int64_t n_partials, double* d_moments, void* stream) {
  if (!d_partials || !d_moments || n_partials <= 0) return fail(DRONECU_ERR_INVALID, "dronecu_norm_reduce: bad argument");
  DeviceGuard guard(device);
  obs_norm_reduce_kernel<<<1, kNormReduceThreads, 0, (cudaStream_t)stream>>>(d_partials, n_partials, d_moments);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_norm_combine(int device, double* d_stats, const double* d_moments, double epsilon, float clip_obs,
                                    float* d_affine, void* stream) {
  if (!d_stats || !(epsilon >= 0) || !(clip_obs > 0)) return fail(DRONECU_ERR_INVALID, "dronecu_norm_combine: bad argument");
  DeviceGuard guard(device);
  obs_norm_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_stats, d_moments, epsilon, clip_obs, d_affine);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_policy_forward_tc(int device, int64_t B, const float* d_params, const float* d_obs, float* d_mean,
                                         float* d_value, float* d_dbg1, float* d_dbg2, void* stream) {
  if (B <= 0 || !d_params || !d_obs) return fail(DRONECU_ERR_INVALID, "dronecu_policy_forward_tc: bad argument");
  if (d_mean && (reinterpret_cast<uintptr_t>(d_mean) & 15)) return fail(DRONECU_ERR_INVALID, "d_mean must be 16-byte aligned");
  DeviceGuard guard(device);
  CUDA_TRY(cudaFuncSetAttribute(policy_forward_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmem));
  const unsigned grid = (unsigned)std::min<int64_t>((B + tc::kTile - 1) / tc::kTile, 148 * 2);
  policy_forward_tc_kernel<<<grid, tc::kTile, kTcSmem, (cudaStream_t)stream>>>(d_params, d_obs, B, reinterpret_cast<float4*>(d_mean),
                                                                              d_value, d_dbg1, d_dbg2);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_policy_forward(int device, int64_t B, const float* d_params, const float* d_obs, float* d_mean,
                                      float* d_value, void* stream) {
  if (B <= 0 || !d_params || !d_obs) return fail(DRONECU_ERR_INVALID, "dronecu_policy_forward: bad argument");
  if (d_mean && (reinterpret_cast<uintptr_t>(d_mean) & 15)) return fail(DRONECU_ERR_INVALID, "d_mean must be 16-byte aligned");
  DeviceGuard guard(device);
  CUDA_TRY(cudaFuncSetAttribute(policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpSmem)));
  const unsigned grid = (unsigned)std::min<int64_t>((B + kPolBlock - 1) / kPolBlock, 148 * 4);
  policy_forward_kernel<<<grid, kPolBlock, sizeof(MlpSmem), (cudaStream_t)stream>>>(d_params, d_obs, B, reinterpret_cast<float4*>(d_mean), d_value);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_gae(int device, int K, int64_t n, const float* d_reward, const float* d_value,
                           const uint8_t* d_done, const float* d_last_value, float gamma, float lam,
                           float* d_adv, float* d_ret, void* stream) {
  if (K <= 0 || n <= 0 || !d_reward || !d_value || !d_done || !d_last_value || !d_adv || !d_ret)
    return fail(DRONECU_ERR_INVALID, "dronecu_gae: bad argument");
  DeviceGuard guard(device);
  gae_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(K, n, d_reward, d_value, d_done,
                                                                           d_last_value, gamma, lam, d_adv, d_ret);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" void dronecu_ppo_config_default(dronecu_ppo_config* c) {
  c->learning_rate = 3e-4f; c->beta1 = 0.9f; c->beta2 = 0.999f; c->adam_eps = 1e-5f;
  c->clip_range = 0.2f; c->vf_coef = 0.5f; c->ent_coef = 0.0f; c->max_grad_norm = 0.5f;
}

extern "C" int dronecu_ppo_create(const dronecu_ppo_config* cfg, int device, dronecu_ppo** out) {
  if (!cfg || !out) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_create: null argument");
  int ndev = 0;
  cudaError_t err = cudaGetDeviceCount(&ndev);
  if (err != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(DRONECU_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(err));
  }
  if (device < 0 || device >= ndev) return fail(DRONECU_ERR_INVALID, "device index out of range");
  DeviceGuard guard(device);
  dronecu_ppo* p = new (std::nothrow) dronecu_ppo();
  if (!p) return fail(DRONECU_ERR_ALLOC, "host allocation failed");
  std::memset(p, 0, sizeof(*p));
  p->cfg = *cfg; p->device = device;
  CUDA_TRY(cudaDeviceGetAttribute(&p->n_sm, cudaDevAttrMultiProcessorCount, device));
  CUDA_TRY(cudaMalloc(&p->partials, sizeof(float) * 2 * (size_t)p->n_sm * kGradLen));
  CUDA_TRY(cudaMalloc(&p->moments, sizeof(float) * 2 * kParams));
  CUDA_TRY(cudaMalloc(&p->adv_partials, sizeof(double) * 2 * (size_t)p->n_sm * 8));
  CUDA_TRY(cudaMemset(p->moments, 0, sizeof(float) * 2 * kParams));
  CUDA_TRY(cudaMalloc(&p->d_step, sizeof(AdamClock)));
  {
    const AdamClock c0 = {0, 1.0, 1.0};
    CUDA_TRY(cudaMemcpy(p->d_step, &c0, sizeof(c0), cudaMemcpyHostToDevice));
  }
  CUDA_TRY(cudaFuncSetAttribute(ppo_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(UpdSmem)));
  CUDA_TRY(cudaFuncSetAttribute(ppo_grad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcUpdSmem));
  CUDA_TRY(cudaFuncSetAttribute(ppo_grad_bf16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTc3Smem));
  CUDA_TRY(cudaFuncSetAttribute(ppo_grad_bf16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTc3Smem));
  *out = p;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_destroy(dronecu_ppo* p) {
  if (!p) return DRONECU_OK;
  DeviceGuard guard(p->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < kDpMaxWorld; ++r)
    if (p->dp_opened[r]) cudaIpcCloseMemHandle(p->dp.mail[r]);
  cudaFree(p->dp_mail); cudaFree(p->dp.seq); cudaFree(p->dp.status);
  cudaFree(p->partials); cudaFree(p->moments); cudaFree(p->adv_partials); cudaFree(p->d_step); cudaFree(p->part_hist);
  cudaGetLastError();
  delete p;
  return DRONECU_OK;
}

extern "C" int64_t dronecu_ppo_num_updates(const dronecu_ppo* p) {      // synchronises the device (the count lives there)
  if (!p) return 0;
  DeviceGuard guard(p->device);
  long long t = 0;
  if (cudaMemcpy(&t, p->d_step, sizeof(t), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)t;
}

// host copy of Philox4x32-10 (philox.cuh is device code)
static void philox_host(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    c[0] = n0; c[1] = (uint32_t)p1; c[2] = n2; c[3] = (uint32_t)p0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}

static PermKey perm_key_for(int64_t n, uint64_t seed, uint64_t epoch) {
  PermKey K;
  int bits = 1;
  while (((int64_t)1 << bits) < n) ++bits;
  K.mask = (bits >= 32) ? 0xFFFFFFFFu : ((1u << bits) - 1u);
  K.shift = (uint32_t)((bits + 1) / 2);
  for (int r = 0; r < 4; r += 2) {        // two Philox calls: 4 multipliers, 4 addends
    uint32_t c[4] = {(uint32_t)epoch, (uint32_t)(epoch >> 32), (uint32_t)r, 0x5045524Du /* "PERM" */};
    philox_host(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    K.mul[r] = c[0] | 1u; K.mul[r + 1] = c[1] | 1u; K.add[r] = c[2]; K.add[r + 1] = c[3];
  }
  return K;
}

extern "C" int dronecu_minibatch_permutation(int device, int64_t n, uint64_t seed, uint64_t epoch, int32_t* d_out,
                                             void* stream) {
  if (!d_out || n <= 0 || n > ((int64_t)1 << 31) - 1) return fail(DRONECU_ERR_INVALID, "dronecu_minibatch_permutation: bad argument");
  DeviceGuard guard(device);
  const PermKey K = perm_key_for(n, seed, epoch);
  perm_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_out, (uint32_t)n, K);
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_minibatch_partition(dronecu_ppo* p, int64_t n, int64_t batch, uint64_t seed, uint64_t epoch, int32_t* d_out,
                                           void* stream) {
  if (!p || !d_out || n <= 0 || batch <= 0 || n > ((int64_t)1 << 31) - 1) return fail(DRONECU_ERR_INVALID, "dronecu_minibatch_partition: bad argument");
  const int64_t n_bins = (n + batch - 1) / batch;
  if (n_bins > kPartMaxBins) return fail(DRONECU_ERR_UNSUPPORTED, "dronecu_minibatch_partition: more than 64 minibatches per epoch (use dronecu_minibatch_permutation)");
  DeviceGuard guard(p->device);
  const PermKey K = perm_key_for(n, seed, epoch);
  const uint32_t rows_per_warp = 2048;
  const uint32_t n_chunks = (uint32_t)((n + rows_per_warp - 1) / rows_per_warp);
  const size_t len = (size_t)n_chunks * (size_t)n_bins;
  if (len > p->part_hist_len) {            // grown outside any capture: callers warm up before capturing graphs
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    cudaFree(p->part_hist);
    p->part_hist = nullptr; p->part_hist_len = 0;
    CUDA_TRY(cudaMalloc(&p->part_hist, sizeof(uint32_t) * len));
    p->part_hist_len = len;
  }
  const unsigned grid = (n_chunks + kPartWarps - 1) / kPartWarps;
  cudaStream_t st = (cudaStream_t)stream;
  const FastDiv fd = fast_div_make((uint32_t)batch);
  part_hist_kernel<<<grid, 32 * kPartWarps, 0, st>>>((uint32_t)n, fd, (uint32_t)n_bins, rows_per_warp, n_chunks, K, p->part_hist);
  CUDA_TRY(cudaGetLastError());
  part_scan_kernel<<<1, 1024, 0, st>>>(p->part_hist, (uint32_t)len);
  CUDA_TRY(cudaGetLastError());
  part_scatter_kernel<<<grid, 32 * kPartWarps, 0, st>>>((uint32_t)n, fd, (uint32_t)n_bins, rows_per_warp, n_chunks, K, p->part_hist, d_out);
  CUDA_TRY(cudaGetLastError());
  p->launches += 3;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_adv_stats(dronecu_ppo* p, const float* d_adv, const int32_t* d_index, int64_t first,
                                     int64_t m, double* d_out, void* stream) {
  if (!p || !d_adv || !d_out || m <= 0) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_adv_stats: bad argument");
  DeviceGuard guard(p->device);
  const unsigned grid = (unsigned)std::min<int64_t>((m + 255) / 256, (int64_t)p->n_sm * 4);
  adv_stats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_adv, d_index, first, m, p->adv_partials);
  CUDA_TRY(cudaGetLastError());
  adv_stats_finish_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(p->adv_partials, (int)grid, m, d_out);
  p->launches += 2;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_adv_stats_epoch(dronecu_ppo* p, const float* d_adv, const int32_t* d_index, int64_t B,
                                           int64_t batch, double* d_out, void* stream) {
  if (!p || !d_adv || !d_out || B <= 0 || batch <= 0) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_adv_stats_epoch: bad argument");
  DeviceGuard guard(p->device);
  const int64_t n_mb = (B + batch - 1) / batch;
  if (n_mb > 65535) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_adv_stats_epoch: more than 65535 minibatches per epoch");
  // partials share adv_partials ([n_sm * 8, 2] doubles): gx CTAs per minibatch
  const int64_t cap = (int64_t)p->n_sm * 8;
  const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>((batch + 255) / 256, cap / n_mb), (int64_t)p->n_sm * 4));
  if ((int64_t)gx * n_mb > cap) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_adv_stats_epoch: too many minibatches for the scratch buffer");
  adv_stats_epoch_kernel<<<dim3(gx, (unsigned)n_mb), 256, 0, (cudaStream_t)stream>>>(d_adv, d_index, B, batch, p->adv_partials);
  CUDA_TRY(cudaGetLastError());
  adv_stats_epoch_finish_kernel<<<(unsigned)n_mb, 32, 0, (cudaStream_t)stream>>>(p->adv_partials, (int)gx, B, batch, d_out);
  p->launches += 2;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

static int ppo_grad_impl(dronecu_ppo* p, const float* d_params, const float* d_obs, const float* d_actions,
                         const float* d_old_logp, const float* d_adv, const float* d_returns,
                         const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                         const double* d_adv_stats, float* d_grad, void* stream, int mode, int obs_stride = 15) {
  const bool tensor_cores = mode != 0;
  if (obs_stride != 15 && obs_stride != 16) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_grad: obs_stride must be 15 (packed rows) or 16 (64-byte rows)");
  if (obs_stride == 16 && (reinterpret_cast<uintptr_t>(d_obs) & 15)) return fail(DRONECU_ERR_INVALID, "padded d_obs must be 16-byte aligned");
  if (!p || !d_params || !d_obs || !d_actions || !d_old_logp || !d_adv || !d_returns || !d_grad || m <= 0)
    return fail(DRONECU_ERR_INVALID, "dronecu_ppo_grad: bad argument");
  if (reinterpret_cast<uintptr_t>(d_actions) & 15) return fail(DRONECU_ERR_INVALID, "d_actions must be 16-byte aligned");
  if (first < 0 || first + m > ((int64_t)1 << 31) - 1) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_grad: row numbers must fit in 31 bits");
  DeviceGuard guard(p->device);
  UpdArgs a;
  a.theta = d_params; a.obs = d_obs; a.obs_stride = obs_stride; a.actions = reinterpret_cast<const float4*>(d_actions); a.old_logp = d_old_logp;
  a.adv = d_adv; a.ret = d_returns; a.index = d_index; a.first = first; a.m = m;
  a.adv_mean = adv_mean; a.adv_inv_std = adv_inv_std; a.adv_stats = d_adv_stats;
  a.clip = p->cfg.clip_range; a.vf_coef = p->cfg.vf_coef; a.ent_coef = p->cfg.ent_coef;
  a.partials = p->partials; a.direct = nullptr; a.dbg = tensor_cores ? p->dbg : nullptr;
  const int64_t tiles = (m + kUpdBlock - 1) / kUpdBlock;
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == 2) {
    // grid (x, 2): blockIdx.y = tower; one CTA per SM, three 128-sample tiles in flight per CTA, one partial vector per CTA
    const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>((tiles + tcb::kWG3 - 1) / tcb::kWG3, p->n_sm / 2));
    a.direct = (gx == 1) ? d_grad : nullptr;       // one partial vector per tower: the kernel writes the gradient itself
    if (obs_stride == 16) ppo_grad_bf16_kernel<true><<<dim3(gx, 2), tcb::kThreads3, kTc3Smem, st>>>(a);
    else ppo_grad_bf16_kernel<false><<<dim3(gx, 2), tcb::kThreads3, kTc3Smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    if (gx > 1) ppo_reduce_tc_kernel<<<(kGradLen + 255) / 256, 256, 0, st>>>(p->partials, (int)gx, d_grad);
    else p->launches -= 1;
  } else if (tensor_cores) {
    // grid (x, 2): blockIdx.y = tower; one CTA per SM, two 128-sample tiles in flight per CTA
    const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>((tiles + tcu::kWG - 1) / tcu::kWG, p->n_sm / 2));
    ppo_grad_tc_kernel<<<dim3(gx, 2), tcu::kThreads, kTcUpdSmem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    ppo_reduce_tc_kernel<<<(kGradLen + 255) / 256, 256, 0, st>>>(p->partials, (int)gx * tcu::kWG, d_grad);
  } else {
    const unsigned grid = (unsigned)std::min<int64_t>(tiles, p->n_sm);
    ppo_grad_kernel<<<grid, kUpdBlock, sizeof(UpdSmem), st>>>(a);
    CUDA_TRY(cudaGetLastError());
    ppo_reduce_kernel<<<(kGradLen + 255) / 256, 256, 0, st>>>(p->partials, (int)grid, d_grad);
  }
  CUDA_TRY(cudaGetLastError());
  p->launches += 2;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_grad(dronecu_ppo* p, const float* d_params, const float* d_obs, const float* d_actions,
                                const float* d_old_logp, const float* d_adv, const float* d_returns,
                                const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                                const double* d_adv_stats, float* d_grad, void* stream) {
  return ppo_grad_impl(p, d_params, d_obs, d_actions, d_old_logp, d_adv, d_returns, d_index, first, m, adv_mean,
                       adv_inv_std, d_adv_stats, d_grad, stream, 0);
}

extern "C" int dronecu_ppo_grad_tc(dronecu_ppo* p, const float* d_params, const float* d_obs, const float* d_actions,
                                   const float* d_old_logp, const float* d_adv, const float* d_returns,
                                   const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                                   const double* d_adv_stats, float* d_grad, void* stream) {
  return ppo_grad_impl(p, d_params, d_obs, d_actions, d_old_logp, d_adv, d_returns, d_index, first, m, adv_mean,
                       adv_inv_std, d_adv_stats, d_grad, stream, 1);
}

extern "C" int dronecu_ppo_grad_bf16(dronecu_ppo* p, const float* d_params, const float* d_obs, const float* d_actions,
                                     const float* d_old_logp, const float* d_adv, const float* d_returns,
                                     const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                                     const double* d_adv_stats, float* d_grad, void* stream) {
  return ppo_grad_impl(p, d_params, d_obs, d_actions, d_old_logp, d_adv, d_returns, d_index, first, m, adv_mean,
                       adv_inv_std, d_adv_stats, d_grad, stream, 2);
}

extern "C" int dronecu_ppo_grad_strided(dronecu_ppo* p, int mode, int obs_stride, const float* d_params, const float* d_obs,
                                        const float* d_actions, const float* d_old_logp, const float* d_adv, const float* d_returns,
                                        const int32_t* d_index, int64_t first, int64_t m, float adv_mean, float adv_inv_std,
                                        const double* d_adv_stats, float* d_grad, void* stream) {
  if (mode < 0 || mode > 2) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_grad_strided: mode must be 0 (fp32), 1 (tf32) or 2 (bf16 wgrad)");
  return ppo_grad_impl(p, d_params, d_obs, d_actions, d_old_logp, d_adv, d_returns, d_index, first, m, adv_mean,
                       adv_inv_std, d_adv_stats, d_grad, stream, mode, obs_stride);
}

extern "C" int dronecu_ppo_debug_buffer(dronecu_ppo* p, float* d_dbg) {
  if (!p) return fail(DRONECU_ERR_INVALID, "null handle");
  p->dbg = d_dbg;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_apply(dronecu_ppo* p, float* d_params, const float* d_grad, double inv_count,
                                 float* d_info, void* stream) {
  if (!p || !d_params || !d_grad || !(inv_count > 0)) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_apply: bad argument");
  DeviceGuard guard(p->device);
  AdamArgs a;
  a.theta = d_params; a.grad = d_grad; a.m = p->moments; a.v = p->moments + kParams;
  a.inv_count = (float)inv_count;
  a.lr = p->cfg.learning_rate;
  a.step = p->d_step;
  a.beta1 = p->cfg.beta1; a.beta2 = p->cfg.beta2; a.eps = p->cfg.adam_eps; a.max_norm = p->cfg.max_grad_norm;
  a.info = d_info; a.info_sum = p->info_sum;
  ppo_apply_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(a);
  p->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_get_state(dronecu_ppo* p, float* d_moments, int64_t* h_step, void* stream) {
  if (!p) return fail(DRONECU_ERR_INVALID, "null handle");
  DeviceGuard guard(p->device);
  if (d_moments)
    CUDA_TRY(cudaMemcpyAsync(d_moments, p->moments, sizeof(float) * 2 * kParams, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (h_step) {
    long long t = 0;
    CUDA_TRY(cudaMemcpyAsync(&t, p->d_step, sizeof(t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    *h_step = (int64_t)t;
  }
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_set_state(dronecu_ppo* p, const float* d_moments, int64_t step, void* stream) {
  if (!p || step < 0) return fail(DRONECU_ERR_INVALID, "bad argument");
  DeviceGuard guard(p->device);
  if (d_moments)
    CUDA_TRY(cudaMemcpyAsync(p->moments, d_moments, sizeof(float) * 2 * kParams, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  const AdamClock t = {(long long)step, std::pow((double)p->cfg.beta1, (double)step), std::pow((double)p->cfg.beta2, (double)step)};
  CUDA_TRY(cudaMemcpyAsync(p->d_step, &t, sizeof(t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return DRONECU_OK;
}


extern "C" int dronecu_ppo_set_info_accumulator(dronecu_ppo* p, float* d_info_sum) {
  if (!p) return fail(DRONECU_ERR_INVALID, "null handle");
  p->info_sum = d_info_sum;
  return DRONECU_OK;
}

// ------------------------------------------------------------------------------------------------
// data-parallel exchange over NVLink peer memory (csrc/ppo_dp.cuh)
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == DRONECU_IPC_HANDLE_BYTES, "IPC handle size");

extern "C" int dronecu_ppo_dp_alloc(dronecu_ppo* p, int rank, int world, void* ipc_handle_out, void** d_mailbox_out) {
  if (!p || world < 1 || world > kDpMaxWorld || rank < 0 || rank >= world)
    return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_alloc: bad rank / world (at most 16 ranks)");
  if (p->dp_mail) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_alloc: already allocated");
  DeviceGuard guard(p->device);
  const size_t bytes = dp_mailbox_bytes(world);
  CUDA_TRY(cudaMalloc(&p->dp_mail, bytes));
  CUDA_TRY(cudaMemset(p->dp_mail, 0, bytes));
  CUDA_TRY(cudaMalloc(&p->dp.seq, sizeof(unsigned long long)));
  CUDA_TRY(cudaMemset(p->dp.seq, 0, sizeof(unsigned long long)));
  CUDA_TRY(cudaMalloc(&p->dp.status, sizeof(int)));
  CUDA_TRY(cudaMemset(p->dp.status, 0, sizeof(int)));
  CUDA_TRY(cudaDeviceSynchronize());
  p->dp.rank = rank; p->dp.world = 0;          // world is set by dronecu_ppo_dp_connect
  p->dp_alloc_world = world;
  p->dp.timeout_ns = 30ull * 1000000000ull;
  if (ipc_handle_out) {
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, p->dp_mail));
    std::memcpy(ipc_handle_out, &h, sizeof(h));
  }
  if (d_mailbox_out) *d_mailbox_out = p->dp_mail;
  p->dp.mail[rank] = p->dp_mail;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_dp_connect(dronecu_ppo* p, int world, const void* ipc_handles, void* const* d_mailboxes) {
  if (!p || !p->dp_mail) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: call dronecu_ppo_dp_alloc first");
  if (world < 1 || world > kDpMaxWorld || p->dp.rank >= world) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: bad world");
  // the slots and flags are indexed with the connected world: a larger one would write past the end of every mailbox
  if (world != p->dp_alloc_world)
    return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: world differs from the one dronecu_ppo_dp_alloc sized the mailbox for");
  if (p->dp.world > 0) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: already connected");
  if (!ipc_handles && !d_mailboxes && world > 1) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: no peers given");
  DeviceGuard guard(p->device);
  for (int r = 0; r < world; ++r) {
    if (r == p->dp.rank) continue;
    if (d_mailboxes) {                       // same process: raw device pointers (enable peer access when on another GPU)
      void* ptr = d_mailboxes[r];
      cudaPointerAttributes at;
      CUDA_TRY(cudaPointerGetAttributes(&at, ptr));
      if (at.type != cudaMemoryTypeDevice) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_connect: not a device pointer");
      if (at.device != p->device) {
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, p->device, at.device));
        if (!can) return fail(DRONECU_ERR_UNSUPPORTED, "dronecu_ppo_dp_connect: no peer access between the devices");
        cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(e);
        cudaGetLastError();
      }
      p->dp.mail[r] = static_cast<float*>(ptr);
    } else {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, static_cast<const char*>(ipc_handles) + (size_t)r * DRONECU_IPC_HANDLE_BYTES, sizeof(h));
      void* ptr = nullptr;
      CUDA_TRY(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      p->dp.mail[r] = static_cast<float*>(ptr);
      p->dp_opened[r] = true;
    }
  }
  p->dp.world = world;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_dp_set_timeout(dronecu_ppo* p, double seconds) {
  if (!p || !(seconds > 0)) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_set_timeout: bad argument");
  p->dp.timeout_ns = (unsigned long long)(seconds * 1e9);
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_dp_status(dronecu_ppo* p, int* h_status, int64_t* h_exchanges) {   // synchronises the device
  if (!p || !p->dp_mail) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_status: data-parallel exchange not set up");
  DeviceGuard guard(p->device);
  int st = 0; unsigned long long seq = 0;
  CUDA_TRY(cudaMemcpy(&st, p->dp.status, sizeof(st), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(&seq, p->dp.seq, sizeof(seq), cudaMemcpyDeviceToHost));
  if (h_status) *h_status = st;
  if (h_exchanges) *h_exchanges = (int64_t)seq;
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_dp_allreduce_f64(dronecu_ppo* p, double* d_buf, int n, void* stream) {
  if (!p || !d_buf || n <= 0 || n > kDpSlot / 2) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_allreduce_f64: bad argument (at most 5376 values)");
  if (p->dp.world < 1) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_dp_allreduce_f64: call dronecu_ppo_dp_connect first");
  if (reinterpret_cast<uintptr_t>(d_buf) & 15) return fail(DRONECU_ERR_INVALID, "d_buf must be 16-byte aligned");
  DeviceGuard guard(p->device);
  dp_allreduce_f64_kernel<<<1, kDpBlock, 0, (cudaStream_t)stream>>>(p->dp, d_buf, n);
  p->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}

extern "C" int dronecu_ppo_apply_dp(dronecu_ppo* p, float* d_params, float* d_grad, float* d_info, void* stream) {
  if (!p || !d_params || !d_grad) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_apply_dp: bad argument");
  if (p->dp.world < 1) return fail(DRONECU_ERR_INVALID, "dronecu_ppo_apply_dp: call dronecu_ppo_dp_connect first");
  if (reinterpret_cast<uintptr_t>(d_grad) & 15) return fail(DRONECU_ERR_INVALID, "d_grad must be 16-byte aligned");
  DeviceGuard guard(p->device);
  AdamArgs a;
  a.theta = d_params; a.grad = d_grad; a.m = p->moments; a.v = p->moments + kParams;
  a.inv_count = 0.f;                       // unused: the denominator is the summed sample count
  a.lr = p->cfg.learning_rate;
  a.step = p->d_step;
  a.beta1 = p->cfg.beta1; a.beta2 = p->cfg.beta2; a.eps = p->cfg.adam_eps; a.max_norm = p->cfg.max_grad_norm;
  a.info = d_info; a.info_sum = p->info_sum;
  ppo_apply_dp_kernel<<<1, kDpBlock, 0, (cudaStream_t)stream>>>(p->dp, a, d_grad);
  p->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return DRONECU_OK;
}
