// Observation and reward normalisation of the policy rollout (SB3 VecNormalize: RunningMeanStd over the observations and
// over the discounted returns; DESIGN.md section 9).  The statistics are frozen for the length of a rollout launch: the
// rollout kernels normalise every observation with the float32 affine record derived after the previous rollout
// (norm_obs_row below), and afterwards
//   obs_norm_pass_kernel     walks each env's K steps of the rollout buffer: moments of the raw rows (float64, shifted by
//                            the running mean), rows rewritten normalised, per-env discounted returns advanced, rewards
//                            normalised; one partial moment record per CTA (no atomics).  Also the predict-time
//                            normaliser (K = 1, no rewards, no partials).
//   obs_norm_reduce_kernel   fixed-order sum of the CTA partials into one batch record (bit-reproducible)
//   obs_norm_combine_kernel  SB3's parallel-variance update of both running statistics, then the affine record of the next
//                            rollout.  A separate launch so that data-parallel training can all-reduce the batch record
//                            in between and every rank then holds bit-identical statistics.
// Layouts (include/dronecu.h): affine float32 [31] = mean_f[15] | rstd_f[15] | clip_obs; stats float64 [34] = obs_mean[15]
// | obs_var[15] | obs_count | ret_mean | ret_var | ret_count; moments float64 [34] = sum(x - c)[15] | sum((x - c)^2)[15] |
// obs count | sum(ret - c_r) | sum((ret - c_r)^2) | return count, c / c_r = the running means the pass read.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ppo_common.cuh"

namespace dronecu {

constexpr int kNormAffine = 2 * kObs + 1;     // 31 floats
constexpr int kNormStats = 2 * kObs + 4;      // 34 doubles
constexpr int kNormMoments = 2 * kObs + 4;    // 34 doubles
constexpr int kNormBlock = 256;               // envs per CTA of the pass (one partial record each)
constexpr int kNormReduceThreads = 1024;

// THE normalisation of one observation value: every rollout kernel and the pass call this, with explicit round-to-nearest
// subtract and multiply so that no call site can contract them into an FMA and round differently.  The clip is np.clip's:
// NaN stays NaN (max.NaN / min.NaN; fmaxf / fminf would return the other operand, -clip), +-inf goes to +-clip.
__device__ __forceinline__ float norm_obs1(float x, float mean, float rstd, float clip) {
  float y = __fmul_rn(__fsub_rn(x, mean), rstd);
  asm("max.NaN.f32 %0, %0, %1;" : "+f"(y) : "f"(-clip));
  asm("min.NaN.f32 %0, %0, %1;" : "+f"(y) : "f"(clip));
  return y;
}

// a [31]-float affine record staged in shared memory (s) applied to an observation row in registers.  Volatile reads: the
// compiler must not hoist the 31 values out of the step loops into registers (the rollout kernels have none to spare)
__device__ __forceinline__ void norm_obs_row(float (&x)[kObs], const volatile float* s) {
  const float clip = s[2 * kObs];
#pragma unroll
  for (int i = 0; i < kObs; ++i) x[i] = norm_obs1(x[i], s[i], s[kObs + i], clip);
}

// the policy kernels' staging of the record: s = the CTA's __shared__ float[NORM ? kNormAffine : 1]; ordered by the
// kernel's next CTA barrier
template <bool NORM>
__device__ __forceinline__ void load_norm(float* s, const float* affine) {
  if constexpr (NORM) { if (threadIdx.x < kNormAffine) s[threadIdx.x] = affine[threadIdx.x]; }
}

struct NormPassArgs {
  float* obs;              // [K,n,stride], rewritten in place (nullptr: observations untouched, no obs moments)
  int32_t stride;          // 15 or 16 (16th value of padded rows left as it is: 1.0)
  int32_t K;
  int64_t n;
  const float* affine;     // [31]
  float* reward;           // [K,n] raw in, normalised out (nullptr: no reward normalisation)
  const uint8_t* done;     // [K,n]
  double* returns;         // [n] per-env discounted return (persistent)
  const double* stats;     // [34] running statistics: the moment shift and the reward scale
  double gamma, epsilon, clip_reward;
  int32_t update;          // != 0: returns advance and partials are written (training)
  int32_t side_env;        // < 0: no side copy
  float* side_obs;         // [K,15] raw rows of env side_env
  double* partials;        // [gridDim.x][34]
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// 2 CTAs per SM: the 32 float64 accumulators take ~130 registers, and a memory-bound walk wants the warps
__global__ void __launch_bounds__(kNormBlock, 2) obs_norm_pass_kernel(const __grid_constant__ NormPassArgs A) {
  __shared__ float s_aff[kNormAffine];
  __shared__ double s_c[kObs + 1];
  __shared__ double s_part[kNormBlock / 32][kNormMoments];
  const bool do_obs = A.obs != nullptr, do_rew = A.reward != nullptr, upd = A.update != 0;
  if (threadIdx.x < kNormAffine && do_obs) s_aff[threadIdx.x] = A.affine[threadIdx.x];
  if (threadIdx.x < kObs && upd) s_c[threadIdx.x] = A.stats[threadIdx.x];
  if (threadIdx.x == kObs && upd) s_c[kObs] = A.stats[2 * kObs + 1];          // ret_mean
  __syncthreads();

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < A.n;
  double s1[kObs], s2[kObs], r1 = 0.0, r2 = 0.0;
#pragma unroll
  for (int f = 0; f < kObs; ++f) { s1[f] = 0.0; s2[f] = 0.0; }
  if (active) {
    const size_t n = (size_t)A.n;
    const double rden = do_rew ? sqrt(A.stats[2 * kObs + 2] + A.epsilon) : 1.0;
    double ret = do_rew ? A.returns[i] : 0.0;
    for (int k = 0; k < A.K; ++k) {
      const size_t row = (size_t)k * n + (size_t)i;
      if (do_obs) {
        float x[kObs];
        float* p = A.obs + row * (size_t)A.stride;
        if (A.stride == 16) {
          const float4* q = reinterpret_cast<const float4*>(p);
          const float4 a = q[0], b = q[1], c = q[2], d = q[3];
          x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
          x[8] = c.x; x[9] = c.y; x[10] = c.z; x[11] = c.w; x[12] = d.x; x[13] = d.y; x[14] = d.z;
        } else {
#pragma unroll
          for (int f = 0; f < kObs; ++f) x[f] = p[f];
        }
        if (i == A.side_env && A.side_obs != nullptr) {
#pragma unroll
          for (int f = 0; f < kObs; ++f) A.side_obs[(size_t)k * kObs + f] = x[f];
        }
        if (upd) {
#pragma unroll
          for (int f = 0; f < kObs; ++f) { const double d = (double)x[f] - s_c[f]; s1[f] += d; s2[f] = fma(d, d, s2[f]); }
        }
        norm_obs_row(x, s_aff);
        if (A.stride == 16) {
          float4* q = reinterpret_cast<float4*>(p);
          q[0] = make_float4(x[0], x[1], x[2], x[3]); q[1] = make_float4(x[4], x[5], x[6], x[7]);
          q[2] = make_float4(x[8], x[9], x[10], x[11]); q[3] = make_float4(x[12], x[13], x[14], 1.0f);
        } else {
#pragma unroll
          for (int f = 0; f < kObs; ++f) p[f] = x[f];
        }
      }
      if (do_rew) {
        const double r = (double)A.reward[row];
        if (upd) {                                   // SB3 _update_reward: returns = returns * gamma + reward
          ret = __dadd_rn(__dmul_rn(ret, A.gamma), r);
          const double d = ret - s_c[kObs];
          r1 += d; r2 = fma(d, d, r2);
        }
        const double q = r / rden;                   // np.clip: NaN stays NaN (fmax / fmin would return the bound)
        A.reward[row] = (float)(q != q ? q : fmin(fmax(q, -A.clip_reward), A.clip_reward));
        if (A.done[row]) ret = 0.0;                  // SB3 step_wait: returns[dones] = 0, training or not
      }
    }
    if (do_rew) A.returns[i] = ret;
  }
  if (!upd) return;
  // warp shuffle -> CTA (fixed order) -> one partial record per CTA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t cta_first = (int64_t)blockIdx.x * blockDim.x;
  const double envs = (double)max((int64_t)0, min((int64_t)blockDim.x, A.n - cta_first));
#pragma unroll
  for (int f = 0; f < kObs; ++f) {
    const double a = warp_sum_d(s1[f]), b = warp_sum_d(s2[f]);
    if (lane == 0) { s_part[warp][f] = a; s_part[warp][kObs + f] = b; }
  }
  {
    const double a = warp_sum_d(r1), b = warp_sum_d(r2);
    if (lane == 0) { s_part[warp][2 * kObs + 1] = a; s_part[warp][2 * kObs + 2] = b; }
  }
  __syncthreads();
  if (threadIdx.x < kNormMoments) {
    const int j = threadIdx.x;
    double t = 0.0;
    if (j == 2 * kObs) t = do_obs ? envs * (double)A.K : 0.0;
    else if (j == 2 * kObs + 3) t = do_rew ? envs * (double)A.K : 0.0;
    else
      for (int w = 0; w < kNormBlock / 32; ++w) t += s_part[w][j];
    A.partials[(size_t)blockIdx.x * kNormMoments + j] = t;
  }
}

// out[j] = sum over p of partials[p][j], p in a fixed order: thread (g, j) sums p = g, g + G, ... (G = 30 groups of the 34
// columns), then one thread per column adds the G group sums in order.  Bit-reproducible for a given n_partials.
__global__ void __launch_bounds__(kNormReduceThreads) obs_norm_reduce_kernel(const double* __restrict__ partials,
                                                                             int64_t n_partials, double* __restrict__ out) {
  constexpr int G = kNormReduceThreads / kNormMoments;       // 30
  __shared__ double sh[G][kNormMoments];
  const int j = threadIdx.x % kNormMoments, g = threadIdx.x / kNormMoments;
  if (g < G) {
    double t = 0.0;
    for (int64_t p = g; p < n_partials; p += G) t += partials[p * kNormMoments + j];
    sh[g][j] = t;
  }
  __syncthreads();
  if (threadIdx.x < kNormMoments) {
    double t = 0.0;
    for (int q = 0; q < G; ++q) t += sh[q][threadIdx.x];
    out[threadIdx.x] = t;
  }
}

// SB3 RunningMeanStd.update_from_moments for one feature: (mean, var, count) <- combine with a batch given by its shifted
// sums s1 = sum(x - c), s2 = sum((x - c)^2) over cb values, c == mean (the shift the pass read)
__device__ __forceinline__ void rms_combine(double& mean, double& var, const double count, double s1, double s2, double cb) {
  const double delta = s1 / cb;                                    // batch_mean - mean
  const double v = s2 / cb - delta * delta;                        // population variance of the batch, clamped at 0 but
  const double var_b = v < 0.0 ? 0.0 : v;                          // kept NaN (inf - inf) as np.var's NaN (fmax: 0)
  const double tot = count + cb;
  const double m2 = var * count + var_b * cb + delta * delta * count * cb / tot;
  mean = mean + delta * cb / tot;
  var = m2 / tot;
}

// one warp: combine (when moments != nullptr), then the float32 affine record (when affine != nullptr)
__global__ void obs_norm_combine_kernel(double* __restrict__ stats, const double* __restrict__ moments, double epsilon,
                                        float clip_obs, float* __restrict__ affine) {
  const int f = threadIdx.x;
  if (moments != nullptr) {
    if (f < kObs && moments[2 * kObs] > 0.0) {
      double mean = stats[f], var = stats[kObs + f];
      rms_combine(mean, var, stats[2 * kObs], moments[f], moments[kObs + f], moments[2 * kObs]);
      stats[f] = mean; stats[kObs + f] = var;
    }
    if (f == kObs && moments[2 * kObs + 3] > 0.0) {
      double mean = stats[2 * kObs + 1], var = stats[2 * kObs + 2];
      rms_combine(mean, var, stats[2 * kObs + 3], moments[2 * kObs + 1], moments[2 * kObs + 2], moments[2 * kObs + 3]);
      stats[2 * kObs + 1] = mean; stats[2 * kObs + 2] = var; stats[2 * kObs + 3] += moments[2 * kObs + 3];
    }
    __syncwarp();
    if (f == 0 && moments[2 * kObs] > 0.0) stats[2 * kObs] += moments[2 * kObs];   // after every feature read the old count
    __syncwarp();
  }
  if (affine != nullptr && f < kObs) {
    affine[f] = (float)stats[f];
    affine[kObs + f] = (float)(1.0 / sqrt(stats[kObs + f] + epsilon));
    if (f == 0) affine[2 * kObs] = clip_obs;
  }
}

}  // namespace dronecu
