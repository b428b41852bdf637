// Tensor-core (tcgen05 / TMEM) versions of policy_forward_kernel and policy_rollout_kernel: same
// contract as ppo_rollout.cuh, the two MLP towers evaluated by tc::forward (tc_mlp.cuh).
#pragma once
#include "ppo_rollout.cuh"
#include "tc_mlp.cuh"

namespace dronecu {

constexpr size_t kTcSmem = sizeof(tc::Smem) + (tc::kTile / 32) * 32 * kObs * sizeof(float);

// no integer round trip: the compiler must keep seeing a shared-memory pointer (LDS, not generic LD)
__device__ __forceinline__ tc::Smem& tc_smem(unsigned char* raw) { return *reinterpret_cast<tc::Smem*>(raw); }

__global__ void __launch_bounds__(tc::kTile) policy_forward_tc_kernel(const float* __restrict__ theta,
                                                                       const float* __restrict__ obs, int64_t B,
                                                                       float4* __restrict__ mean, float* __restrict__ value,
                                                                       float* __restrict__ dbg1, float* __restrict__ dbg2) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  tc::Smem& S = tc_smem(smem_raw);
  tc::setup(S, theta);
  uint32_t phase = 0;
  const int64_t tiles = (B + tc::kTile - 1) / tc::kTile;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t r = tile * tc::kTile + threadIdx.x;
    const bool live = r < B;
    float x[kObs], m[kAct], v;
#pragma unroll
    for (int i = 0; i < kObs; ++i) x[i] = live ? obs[r * kObs + i] : 0.f;
    tc::forward(S, x, phase, m, v, (live && dbg1) ? dbg1 + r * 128 : nullptr, (live && dbg2) ? dbg2 + r * 128 : nullptr);
    if (live) {
      if (mean) mean[r] = make_float4(m[0], m[1], m[2], m[3]);
      if (value) value[r] = v;
    }
  }
  tc::teardown(S);
}

template <bool RANDOMIZED, bool NORM = false, bool TIMEOUT = false>
__global__ void __launch_bounds__(tc::kTile) policy_rollout_tc_kernel(const __grid_constant__ PolicyArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  tc::Smem& S = tc_smem(smem_raw);
  float (*tiles)[32 * kObs] = reinterpret_cast<float (*)[32 * kObs]>(reinterpret_cast<unsigned char*>(&S) + sizeof(tc::Smem));
  __shared__ unsigned long long blk_stats[3];
  __shared__ double blk_ret;
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  cta_stats_init(blk_stats, blk_ret);
  load_norm<NORM>(s_norm, A.norm);
  tc::setup(S, A.theta);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warp_base = (int64_t)blockIdx.x * blockDim.x + warp * 32;
  const int64_t i = warp_base + lane;
  const bool active = i < A.n;
  const int valid = (int)max((int64_t)0, min((int64_t)32, A.n - warp_base));
  float* tile = tiles[warp];
  const EnvParams& P = A.P;
  const uint64_t env_id = P.env_offset + (uint64_t)i;
  const int64_t n = A.n;

  EnvState s = {};
  if (active) s = load_state(A.state, i);
  float std_[kAct];
  const float logstd_sum = policy_std(S.log_std, std_);

  int32_t n_trunc = 0;
  EpisodeTally tally;
  uint32_t phase = 0;
  float4* p_act = A.actions + i;
  float* p_logp = A.logp + i;
  float* p_val = A.value + i;
  float* p_rew = A.reward + i;
  uint8_t* p_done = A.done + i;
  float* p_obs = A.obs + warp_base * kObs;
  const bool fast_obs = emit_fast_ok<kObs>(A.obs, warp_base, n, valid);

  for (int k = 0; k < A.K; ++k) {
    float x[kObs];
    write_obs<kObs>(x, s);
    if (A.obs != nullptr && A.obs_padded) {
      if (active) store_row16(A.obs + ((size_t)k * (size_t)n + (size_t)i) * 16, x);
    } else if (A.obs != nullptr && valid > 0) emit_obs_rows<kObs>(tile, p_obs, s, lane, valid, active, fast_obs);
    if constexpr (NORM) norm_obs_row(x, s_norm);

    float mean[kAct], val;
    tc::forward(S, x, phase, mean, val);

    float logp;
    const float4 a = policy_action(mean, std_, logstd_sum, P.keys, env_id, A.t0 + (uint64_t)k, A.deterministic, logp);
    const StepResult r = step_env(s, P, env_action(a, P.motor_max));
    const bool done = r.crashed || r.timeout;
    if (active) {
      if (A.actions != nullptr) st_quad(p_act, a);
      if (A.logp != nullptr) *p_logp = logp;
      if (A.value != nullptr) *p_val = val;
      if (A.reward != nullptr) *p_rew = r.reward;
      if (A.done != nullptr) *p_done = done ? 1 : 0;
      if (done) {
        tally.add(r.crashed, s);
        if constexpr (TIMEOUT) { if (!r.crashed) record_truncation(A, s, i, k, n_trunc, true); }
        reset_env<RANDOMIZED>(s, P, env_id);
      }
    }
    p_act += n; p_logp += n; p_val += n; p_rew += n; p_done += n; p_obs += n * kObs;
  }

  {
    float x[kObs], val;
    write_obs<kObs>(x, s);
    if (A.last_value != nullptr) {       // uniform across the CTA: every thread takes part in the forward
      if constexpr (NORM) norm_obs_row(x, s_norm);
      val = tc::forward_value(S, x, phase);
      if (active) A.last_value[i] = val;
    }
    if (A.last_obs != nullptr && valid > 0)
      emit_obs_rows<kObs>(tile, A.last_obs + warp_base * kObs, s, lane, valid, active,
                          emit_fast_ok<kObs>(A.last_obs, warp_base, n, valid));
  }
  if (active) store_state(A.state, i, s);
  if constexpr (TIMEOUT) { if (active) close_truncation_slots(A, i, n_trunc); }

  tally.flush_warp(blk_stats, blk_ret, lane);
  tc::teardown(S);        // contains the CTA barrier that orders the atomics above
  if (threadIdx.x == 0) cta_stats_commit(A.stats + (blockIdx.x % kStatSlots), blk_stats, blk_ret);
}

}  // namespace dronecu
