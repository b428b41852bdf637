// Time-limit bootstrap of the policy rollout (SB3 collect_rollouts with Gymnasium time limits; DESIGN.md section 11).  A
// TIMEOUT rollout launch records the raw pre-reset observation of every step that ended by the time limit alone in a side
// buffer [T,n,16] with its buffer row [T,n] (-1: unused slot).  This kernel then adds, for every recorded row,
//   reward[row] = reward[row] + f32(f32(gamma) * V(norm(terminal row)))
// -- SB3's `rewards[idx] += self.gamma * terminal_value` as numpy and torch evaluate it on float32 operands
// (tests/test_timeout_oracle.py pins it).  V is the float32 value tower of policy_forward_kernel (tower_forward<1>), so the
// value is bit-identical to dronecu_policy_forward on the same (normalised) row whatever precision the rollout used.
#pragma once
#include "ppo_rollout.cuh"

namespace dronecu {

template <bool NORM>
__global__ void __launch_bounds__(kPolBlock) timeout_bootstrap_kernel(const float* __restrict__ theta,
                                                                      const float4* __restrict__ term_obs,
                                                                      const int32_t* __restrict__ term_row, int64_t slots,
                                                                      const float* __restrict__ norm, float gamma,
                                                                      float* __restrict__ reward) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  load_mlp_smem(S, theta);
  load_norm<NORM>(s_norm, norm);
  __syncthreads();
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < slots; q += (int64_t)gridDim.x * blockDim.x) {
    const int32_t row = term_row[q];
    if (row < 0) continue;
    const float4* p = term_obs + q * 4;
    const float4 a = p[0], b = p[1], c = p[2], d = p[3];
    float x[kObs] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w, d.x, d.y, d.z};
    if constexpr (NORM) norm_obs_row(x, s_norm);
    float v[1];
    tower_forward<1>(S, 1, x, v);
    reward[row] = __fadd_rn(reward[row], __fmul_rn(gamma, v[0]));
  }
}

}  // namespace dronecu
