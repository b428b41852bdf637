// Policy evaluation (SB3 evaluate_policy over VecMonitor(DummyVecEnv([DroneGymEnv] * N))) with the actor alone: per step
// only the pi tower runs (no value tower, no Box-Muller noise when deterministic) and nothing per step reaches HBM -- the
// only stores are one (return, length) pair per recorded episode and the state at the end of the launch.  DESIGN.md s.10.
//
// Env g of the N evaluation envs (global index) records target_g = (n_eval_episodes + g) / N episodes; all envs step in
// lockstep until every env reached its target (T steps in all), env i's step c uses the Philox noise index t0 + c as the
// rollout does, and an env past its target keeps stepping and auto-resetting without recording.  One launch runs in one
// of two modes, so that no step is computed twice and every env is stepped exactly T times:
//   probe     each env steps from steps[i] until it reached its target or step `limit`; the envs still below target are
//             counted into *pending
//   catch-up  (T known) each env steps from steps[i] to T, recording nothing new
// Same arithmetic as the rollout kernels on the same operands (tower_forward / tower_forward_warp / tc::tower, step_env,
// reset_env, norm_obs_row, noise_normals): each evaluation kernel reproduces its rollout counterpart bit for bit.
#pragma once
#include "ppo_rollout_tc.cuh"

namespace dronecu {

struct EvalArgs {
  StatePlanes state;
  EnvParams P;
  int64_t n;
  uint64_t t0;             // env clock at the evaluation's first step
  int32_t limit;           // probe: chunk end (absolute step); catch-up: T
  int32_t catch_up;
  int32_t deterministic;
  int32_t max_eps;         // row stride of ep_return / ep_length
  int64_t env_index0;      // global index of env 0 among the n_global evaluation envs
  int64_t n_global;
  int64_t n_eval_episodes;
  const float* theta;
  const float* norm;       // [31] affine record, read only by the NORM instantiations
  int32_t* steps;          // [n] steps taken since the evaluation's reset
  int32_t* count;          // [n] episodes recorded
  float* ep_return;        // [n, max_eps]
  int32_t* ep_length;      // [n, max_eps]
  int32_t* pending;        // probe: += envs still below target
};

__device__ __forceinline__ int32_t eval_target(const EvalArgs& A, int64_t i) {
  return (int32_t)((A.n_eval_episodes + A.env_index0 + i) / A.n_global);
}

// does env (c, count) take another step in this launch
__device__ __forceinline__ bool eval_live(const EvalArgs& A, int32_t c, int32_t count, int32_t target) {
  return c < A.limit && (A.catch_up || count < target);
}

// the env step after the policy: action (as the rollout computes it), clip, step, episode record, auto-reset
template <bool RANDOMIZED>
__device__ __forceinline__ void eval_step(const EvalArgs& A, EnvState& s, const float (&mean)[kAct], const float (&std_)[kAct],
                                          uint64_t env_id, int64_t i, int32_t& c, int32_t& count, int32_t target,
                                          bool writer = true) {
  const EnvParams& P = A.P;
  float4 a;
  if (A.deterministic) {
    a = make_float4(mean[0], mean[1], mean[2], mean[3]);
  } else {
    const float4 z = noise_normals(P.keys, env_id, A.t0 + (uint64_t)c);
    a = make_float4(fmaf(std_[0], z.x, mean[0]), fmaf(std_[1], z.y, mean[1]),
                    fmaf(std_[2], z.z, mean[2]), fmaf(std_[3], z.w, mean[3]));
  }
  const float4 f = make_float4(fminf(fmaxf(a.x, 0.f), P.motor_max), fminf(fmaxf(a.y, 0.f), P.motor_max),
                               fminf(fmaxf(a.z, 0.f), P.motor_max), fminf(fmaxf(a.w, 0.f), P.motor_max));
  const StepResult r = step_env(s, P, f);
  if (r.crashed || r.timeout) {
    if (count < target) {                 // VecMonitor's info["episode"]: float32 return, int length
      if (writer) {
        const size_t slot = (size_t)i * (size_t)A.max_eps + (size_t)count;
        A.ep_return[slot] = s.ep_ret;
        A.ep_length[slot] = s.ep_len;
      }
      count += 1;
    }
    reset_env<RANDOMIZED>(s, P, env_id);
  }
  c += 1;
}

__device__ __forceinline__ void eval_std(const float* log_std, float (&std_)[kAct]) {
#pragma unroll
  for (int o = 0; o < kAct; ++o) std_[o] = expf(log_std[o]);
}

// one env per thread; lanes stop independently (the tower reads shared memory only)
template <bool RANDOMIZED, bool NORM>
__global__ void __launch_bounds__(kPolBlock) policy_eval_kernel(const __grid_constant__ EvalArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  load_mlp_smem(S, A.theta);
  if constexpr (NORM) { if (threadIdx.x < kNormAffine) s_norm[threadIdx.x] = A.norm[threadIdx.x]; }
  __syncthreads();

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < A.n;
  const uint64_t env_id = A.P.env_offset + (uint64_t)i;
  bool below = false;
  if (active) {
    EnvState s = load_state(A.state, i);
    float std_[kAct];
    eval_std(S.log_std, std_);
    int32_t c = A.steps[i], count = A.count[i];
    const int32_t target = eval_target(A, i);
    while (eval_live(A, c, count, target)) {
      float x[kObs], mean[kAct];
      write_obs<kObs>(x, s);
      if constexpr (NORM) norm_obs_row(x, s_norm);
      tower_forward<kAct>(S, 0, x, mean);
      eval_step<RANDOMIZED>(A, s, mean, std_, env_id, i, c, count, target);
    }
    store_state(A.state, i, s);
    A.steps[i] = c;
    A.count[i] = count;
    below = count < target;
  }
  const unsigned b = __ballot_sync(0xffffffffu, below);
  if (!A.catch_up && b != 0 && (threadIdx.x & 31) == 0) atomicAdd(A.pending, (int)__popc(b));
}

// one warp per env (small batches): every lane holds the whole state, so the loop condition is warp-uniform
template <bool RANDOMIZED, bool NORM>
__global__ void __launch_bounds__(32 * kSmallWarps) policy_eval_warp_kernel(const __grid_constant__ EvalArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  load_mlp_smem(S, A.theta);
  if constexpr (NORM) { if (threadIdx.x < kNormAffine) s_norm[threadIdx.x] = A.norm[threadIdx.x]; }
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* const hbuf = reinterpret_cast<float*>(smem_raw + sizeof(MlpSmem)) + warp * kHid;
  const int64_t i = (int64_t)blockIdx.x * kSmallWarps + warp;
  if (i >= A.n) return;                                                   // warp-uniform
  const uint64_t env_id = A.P.env_offset + (uint64_t)i;
  EnvState s = load_state(A.state, i);
  float std_[kAct];
  eval_std(S.log_std, std_);
  int32_t c = A.steps[i], count = A.count[i];
  const int32_t target = eval_target(A, i);
  while (eval_live(A, c, count, target)) {
    float x[kObs], mean[kAct];
    write_obs<kObs>(x, s);
    if constexpr (NORM) norm_obs_row(x, s_norm);
    tower_forward_warp<kAct>(S, hbuf, 0, x, mean, lane);
    eval_step<RANDOMIZED>(A, s, mean, std_, env_id, i, c, count, target, lane == 0);   // every lane steps its copy
  }
  if (lane == 0) {
    store_state(A.state, i, s);
    A.steps[i] = c;
    A.count[i] = count;
    if (!A.catch_up && count < target) atomicAdd(A.pending, 1);
  }
}

// tensor cores: 128 envs per CTA through tc::forward_policy; the CTA loops while any of its envs is live, rows of envs that
// are not feed the MMAs but do not advance their env
template <bool RANDOMIZED, bool NORM>
__global__ void __launch_bounds__(tc::kTile) policy_eval_tc_kernel(const __grid_constant__ EvalArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  tc::Smem& S = tc_smem(smem_raw);
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  if constexpr (NORM) { if (threadIdx.x < kNormAffine) s_norm[threadIdx.x] = A.norm[threadIdx.x]; }
  tc::setup(S, A.theta);

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < A.n;
  const uint64_t env_id = A.P.env_offset + (uint64_t)i;
  EnvState s = {};
  int32_t c = 0, count = 0, target = 0;
  if (active) {
    s = load_state(A.state, i);
    c = A.steps[i];
    count = A.count[i];
    target = eval_target(A, i);
  }
  float std_[kAct];
  eval_std(S.log_std, std_);
  uint32_t phase = 0;
  bool live = active && eval_live(A, c, count, target);
  while (__syncthreads_or(live)) {
    float x[kObs], mean[kAct];
    write_obs<kObs>(x, s);
    if constexpr (NORM) norm_obs_row(x, s_norm);
    tc::forward_policy(S, x, phase, mean);
    if (live) {
      eval_step<RANDOMIZED>(A, s, mean, std_, env_id, i, c, count, target);
      live = eval_live(A, c, count, target);
    }
  }
  if (active) {
    store_state(A.state, i, s);
    A.steps[i] = c;
    A.count[i] = count;
  }
  const unsigned b = __ballot_sync(0xffffffffu, active && count < target);
  if (!A.catch_up && b != 0 && (threadIdx.x & 31) == 0) atomicAdd(A.pending, (int)__popc(b));
  tc::teardown(S);
}

}  // namespace dronecu
