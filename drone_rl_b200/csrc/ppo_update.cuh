// PPO minibatch update, float32 CUDA-core version: clipped-surrogate + value loss, forward and
// backward through both towers, weight gradients, global-norm clip, Adam.  Restates what SB3's
// PPO.train() does per minibatch (SURVEY.md appendix C; call site /root/reference/train.py:63-68) --
// the source is not in /root/reference, parity is against oracle/ppo_oracle.py ("parity unpinned").
//
// Structure: a persistent grid (one CTA of 128 threads per SM) walks tiles of 128 samples.
//   per tile, per tower:  thread-per-sample forward (weights as warp-broadcast LDS.128 from smem),
//   loss gradient, thread-per-sample backward for the activations, and the three weight-gradient
//   products (delta^T . activation, reduction over the 128 samples of the tile) as shared-memory
//   register-tiled GEMMs.  Weight gradients accumulate in shared memory over the tiles of a CTA and
//   leave as one partial vector per CTA; a second kernel sums the partials in a fixed order
//   (deterministic, which the data-parallel equivalence test relies on); a third applies
//   clip_grad_norm_ + Adam.
#pragma once
#include "ppo_rollout.cuh"

namespace dronecu {

constexpr int kUpdBlock = 128;          // threads == samples per tile
constexpr int kRow = 68;                // row stride (floats) of the activation tiles: 16-byte aligned rows
constexpr int kStats = 8;               // policy_loss, value_loss, approx_kl, clip_frac, count, spare...
constexpr int kGradLen = kParams + kStats;

struct UpdSmem {
  MlpSmem fwd;                          // transposed weights for the forward pass
  float W2[2][kHid][kHid];              // natural [out][in] for delta1 = delta2 . W2
  float W3pi[kAct][kHid];               // natural for delta2 = g3 . W3
  float G[kGradLen + 3];                // gradient + statistics accumulators of this CTA
  float bufA[kUpdBlock][kRow];          // h1, later delta1
  float bufB[kUpdBlock][kRow];          // h2, later delta2
  float bufX[kUpdBlock][16];            // observation, x[15] = 1 (bias column)
  float g3[kUpdBlock][kAct];            // head gradient per sample
  float wsum[kUpdBlock / 32][8];        // per-warp partial sums (log_std gradient, statistics)
};

struct UpdArgs {
  const float* theta;        // [kParams]
  const float* obs;          // [B,15] ([B,16] rows of 64 bytes, 16th value 1.0, when obs_stride == 16)
  int obs_stride;            // floats per observation row: 15 or 16
  const float4* actions;     // [B]
  const float* old_logp;     // [B]
  const float* adv;          // [B]
  const float* ret;          // [B]
  const int32_t* index;      // [m] rows of this minibatch (nullptr: rows first .. first+m)
  int64_t first, m;
  float adv_mean, adv_inv_std;   // (adv - mean) * inv_std ; (0, 1) disables normalisation
  const double* adv_stats;       // nullable: [sum, sum of squares, count] -> overrides the two scalars (count <= 1: (0, 1))
  float clip, vf_coef, ent_coef;
  float* partials;           // [gridDim.x, kGradLen]
  float* direct;             // ppo_grad_bf16_kernel with ONE CTA per tower: the gradient vector itself (no reduce launch); else nullptr
  float* dbg;                // nullable (tensor-core kernel only): raw TMEM dump [2 gridDim.x, 128 lanes, 256 columns]
};

// SB3's PPO loss at the head, per sample -- one statement for the three gradient kernels (ppo_grad_kernel, ppo_grad_tc_kernel,
// ppo_grad_bf16_kernel); each accumulates and stores the results its own way.

// the advantage normalisation of the minibatch: adv = (adv_raw - mean) * inv_std
__device__ __forceinline__ void adv_normalizer(const UpdArgs& A, float& mean, float& inv_std) {
  mean = A.adv_mean;
  inv_std = A.adv_inv_std;
  if (A.adv_stats != nullptr && A.adv_stats[2] > 1.0) {   // SB3: (adv - adv.mean()) / (adv.std() + 1e-8), torch.std is unbiased
    const double cnt = A.adv_stats[2], mu = A.adv_stats[0] / cnt;
    const double var = (A.adv_stats[1] - A.adv_stats[0] * mu) / (cnt - 1.0);
    mean = (float)mu;
    inv_std = (float)(1.0 / (sqrt(fmax(var, 0.0)) + 1e-8));
  } else if (A.adv_stats != nullptr) {   // SB3 normalises only `if len(advantages) > 1`: one sample keeps its raw advantage
    mean = 0.f;
    inv_std = 1.f;
  }
}

struct PolicyHead {
  float g_mean[kAct];        // d loss / d mean: clipped surrogate through the Gaussian log-probability
  float g_logstd[kAct];      // d loss / d log_std: the same, plus the entropy term -ent_coef
  float pg_loss;             // -min(s1, s2)
  float kl;                  // (ratio - 1) - log ratio: SB3's approx_kl estimator
  float clipped;             // 1 where |ratio - 1| > clip (clip fraction)
};

// `adv` is the normalised advantage, `mean` the policy head's output including its bias
__device__ __forceinline__ PolicyHead policy_head(const float4 act, const float (&mean)[kAct], const float (&std_inv)[kAct],
                                                  const float logstd_sum, const float old_logp, const float adv,
                                                  const float clip, const float ent_coef) {
  PolicyHead h;
  const float av[4] = {act.x, act.y, act.z, act.w};
  float z[kAct], sq = 0.f;
#pragma unroll
  for (int o = 0; o < kAct; ++o) { z[o] = (av[o] - mean[o]) * std_inv[o]; sq = fmaf(z[o], z[o], sq); }
  const float logp = -0.5f * sq - logstd_sum - kAct * kHalfLog2Pi;
  const float log_ratio = logp - old_logp;
  const float ratio = expf(log_ratio);
  const float lo = 1.0f - clip, hi = 1.0f + clip;
  const float s1 = adv * ratio, s2 = adv * fminf(fmaxf(ratio, lo), hi);
  const bool inside = (ratio >= lo) && (ratio <= hi);
  const float dl_dlogp = (inside || s1 < s2) ? -adv * ratio : 0.f;     // d(-min(s1,s2)) / d logp
#pragma unroll
  for (int o = 0; o < kAct; ++o) {
    h.g_mean[o] = dl_dlogp * z[o] * std_inv[o];
    h.g_logstd[o] = dl_dlogp * (z[o] * z[o] - 1.0f) - ent_coef;
  }
  h.pg_loss = -fminf(s1, s2);
  h.kl = (ratio - 1.0f) - log_ratio;
  h.clipped = (fabsf(ratio - 1.0f) > clip) ? 1.0f : 0.f;
  return h;
}

// value head: returns d(vf_coef * (ret - v)^2) / dv, and the squared error for the value-loss statistic
__device__ __forceinline__ float value_head(const float v, const float ret, const float vf_coef, float& sq_err) {
  const float diff = v - ret;
  sq_err = diff * diff;
  return 2.0f * vf_coef * diff;
}

// forward of one tower keeping what the backward pass needs: h1 -> bufA row, h2 -> bufB row
template <int NOUT>
__device__ __forceinline__ void tower_forward_keep(const MlpSmem& S, const int t, const float (&x)[kObs],
                                                   float* rowA, float* rowB, float (&out)[NOUT]) {
  float h1[kHid];
#pragma unroll
  for (int q = 0; q < kHid / 4; ++q) {
    const float4 b = reinterpret_cast<const float4*>(S.b1[t])[q];
    h1[4 * q] = b.x; h1[4 * q + 1] = b.y; h1[4 * q + 2] = b.z; h1[4 * q + 3] = b.w;
  }
#pragma unroll
  for (int i = 0; i < kObs; ++i) {
    const float xi = x[i];
#pragma unroll
    for (int q = 0; q < kHid / 4; ++q) {
      const float4 w = reinterpret_cast<const float4*>(S.W1T[t][i])[q];
      fma4s(h1 + 4 * q, w, xi);
    }
  }
#pragma unroll
  for (int q = 0; q < kHid / 4; ++q) {
    float4 v;
    v.x = h1[4 * q] = tanh_fast(h1[4 * q]); v.y = h1[4 * q + 1] = tanh_fast(h1[4 * q + 1]);
    v.z = h1[4 * q + 2] = tanh_fast(h1[4 * q + 2]); v.w = h1[4 * q + 3] = tanh_fast(h1[4 * q + 3]);
    reinterpret_cast<float4*>(rowA)[q] = v;
  }
  if constexpr (NOUT == kAct) {
#pragma unroll
    for (int o = 0; o < kAct; ++o) out[o] = S.b3pi[o];
  } else {
    out[0] = S.b3vf;
  }
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    float acc[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 b = reinterpret_cast<const float4*>(S.b2[t] + 16 * c)[q];
      acc[4 * q] = b.x; acc[4 * q + 1] = b.y; acc[4 * q + 2] = b.z; acc[4 * q + 3] = b.w;
    }
#pragma unroll
    for (int i = 0; i < kHid; ++i) {
      const float hi = h1[i];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 w = reinterpret_cast<const float4*>(S.W2T[t][i] + 16 * c)[q];
        fma4s(acc + 4 * q, w, hi);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 v;
      v.x = tanh_fast(acc[4 * q]); v.y = tanh_fast(acc[4 * q + 1]);
      v.z = tanh_fast(acc[4 * q + 2]); v.w = tanh_fast(acc[4 * q + 3]);
      reinterpret_cast<float4*>(rowB + 16 * c)[q] = v;
      const float a4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = 16 * c + 4 * q + e;
        if constexpr (NOUT == kAct) {
          const float4 w = reinterpret_cast<const float4*>(S.W3piT[j])[0];
          fma4s(out, w, a4[e]);
        } else {
          out[0] = fmaf(S.W3vf[j], a4[e], out[0]);
        }
      }
    }
  }
}

// backward of one tower for the thread's own sample.  On entry rowB = h2, rowA = h1, g3 = dL/d(out).
// Leaves delta2 in rowB and returns delta1 (still to be written over rowA by the caller once the
// dW2 product has consumed h1).
template <int NOUT>
__device__ __forceinline__ void tower_backward(const UpdSmem& U, const int t, const float (&g3)[NOUT],
                                               const float* rowA, float* rowB, float (&d1)[kHid]) {
#pragma unroll
  for (int i = 0; i < kHid; ++i) d1[i] = 0.f;
#pragma unroll
  for (int q = 0; q < kHid / 4; ++q) {
    const float4 h = reinterpret_cast<const float4*>(rowB)[q];
    const float h4[4] = {h.x, h.y, h.z, h.w};
    float d4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = 4 * q + e;
      float up;
      if constexpr (NOUT == kAct) {
        up = g3[0] * U.W3pi[0][j] + g3[1] * U.W3pi[1][j] + g3[2] * U.W3pi[2][j] + g3[3] * U.W3pi[3][j];
      } else {
        up = g3[0] * U.fwd.W3vf[j];
      }
      d4[e] = up * (1.0f - h4[e] * h4[e]);                      // tanh'
      const float dj = d4[e];
#pragma unroll
      for (int qq = 0; qq < kHid / 4; ++qq) {
        const float4 w = reinterpret_cast<const float4*>(U.W2[t][j])[qq];
        fma4s(d1 + 4 * qq, w, dj);
      }
    }
    reinterpret_cast<float4*>(rowB)[q] = make_float4(d4[0], d4[1], d4[2], d4[3]);
  }
#pragma unroll
  for (int q = 0; q < kHid / 4; ++q) {
    const float4 h = reinterpret_cast<const float4*>(rowA)[q];
    d1[4 * q] *= 1.0f - h.x * h.x; d1[4 * q + 1] *= 1.0f - h.y * h.y;
    d1[4 * q + 2] *= 1.0f - h.z * h.z; d1[4 * q + 3] *= 1.0f - h.w * h.w;
  }
}

// G[w2off + j*64 + i] += sum_s bufB[s][j] * bufA[s][i]   (64 x 64 outputs, 128 threads x (4 j x 8 i))
// G[b2off + j]        += sum_s bufB[s][j]
__device__ __forceinline__ void wgrad_hidden(UpdSmem& U, int w2off, int b2off, int rows) {
  const int jt = threadIdx.x >> 3, it = threadIdx.x & 7;
  float acc[4][8];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;
  for (int s = 0; s < rows; ++s) {
    const float4 d = reinterpret_cast<const float4*>(U.bufB[s])[jt];
    const float4 h0 = reinterpret_cast<const float4*>(U.bufA[s])[it];
    const float4 h1 = reinterpret_cast<const float4*>(U.bufA[s])[8 + it];
    const float dd[4] = {d.x, d.y, d.z, d.w};
    const float hh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 8; b += 2) fma2(acc[a][b], acc[a][b + 1], hh[b], hh[b + 1], dd[a], dd[a]);
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int j = 4 * jt + a, i = (b < 4) ? (4 * it + b) : (32 + 4 * it + (b - 4));
      U.G[w2off + j * kHid + i] += acc[a][b];
    }
  if (threadIdx.x < kHid) {
    float sum = 0.f;
    for (int s = 0; s < rows; ++s) sum += U.bufB[s][threadIdx.x];
    U.G[b2off + threadIdx.x] += sum;
  }
}

// G[w1off + j*15 + i] += sum_s bufA[s][j] * bufX[s][i] (i < 15);  G[b1off + j] += sum_s bufA[s][j] * 1
__device__ __forceinline__ void wgrad_input(UpdSmem& U, int w1off, int b1off, int rows) {
  const int jt = threadIdx.x >> 2, it = threadIdx.x & 3;     // j = 2 jt + {0,1}, i = 4 it + {0..3}
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  for (int s = 0; s < rows; ++s) {
    const float2 d = reinterpret_cast<const float2*>(U.bufA[s])[jt];
    const float4 x = reinterpret_cast<const float4*>(U.bufX[s])[it];
    fma4s(acc[0], x, d.x);
    fma4s(acc[1], x, d.y);
  }
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int j = 2 * jt + a, i = 4 * it + b;
      if (i < kObs) U.G[w1off + j * kObs + i] += acc[a][b];
      else U.G[b1off + j] += acc[a][b];
    }
}

// head: G[w3off + o*64 + j] += sum_s g3[s][o] * bufB[s][j] ;  G[b3off + o] += sum_s g3[s][o]
template <int NOUT>
__device__ __forceinline__ void wgrad_head(UpdSmem& U, int w3off, int b3off, int rows) {
  for (int idx = threadIdx.x; idx < NOUT * kHid; idx += kUpdBlock) {
    const int o = idx / kHid, j = idx % kHid;
    float sum = 0.f;
    for (int s = 0; s < rows; ++s) sum = fmaf(U.g3[s][o], U.bufB[s][j], sum);
    U.G[w3off + idx] += sum;
  }
  if (threadIdx.x < NOUT) {
    float sum = 0.f;
    for (int s = 0; s < rows; ++s) sum += U.g3[s][threadIdx.x];
    U.G[b3off + threadIdx.x] += sum;
  }
}


__global__ void __launch_bounds__(kUpdBlock, 1) ppo_grad_kernel(const __grid_constant__ UpdArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  UpdSmem& U = *reinterpret_cast<UpdSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31;

  load_mlp_smem(U.fwd, A.theta);
  for (int idx = tid; idx < 2 * kHid * kHid; idx += kUpdBlock) {
    const int t = idx / (kHid * kHid), q = idx % (kHid * kHid);
    U.W2[t][q / kHid][q % kHid] = A.theta[(t ? O_VF_W2 : O_PI_W2) + q];
  }
  for (int idx = tid; idx < kAct * kHid; idx += kUpdBlock) U.W3pi[idx / kHid][idx % kHid] = A.theta[O_PI_W3 + idx];
  for (int idx = tid; idx < kGradLen + 3; idx += kUpdBlock) U.G[idx] = 0.f;
  __syncthreads();

  float std_inv[kAct], logstd_sum = 0.f;
#pragma unroll
  for (int o = 0; o < kAct; ++o) { std_inv[o] = expf(-U.fwd.log_std[o]); logstd_sum += U.fwd.log_std[o]; }
  float adv_mean, adv_inv_std;
  adv_normalizer(A, adv_mean, adv_inv_std);

  const int64_t n_tiles = (A.m + kUpdBlock - 1) / kUpdBlock;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t pos = tile * kUpdBlock + tid;
    const bool live = pos < A.m;
    const int rows = (int)min((int64_t)kUpdBlock, A.m - tile * kUpdBlock);
    const int64_t row = live ? (A.index ? (int64_t)A.index[pos] : A.first + pos) : 0;

    float x[kObs];
#pragma unroll
    for (int i = 0; i < kObs; ++i) x[i] = live ? A.obs[row * A.obs_stride + i] : 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      reinterpret_cast<float4*>(U.bufX[tid])[q] =
          make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], (q == 3) ? 1.0f : x[4 * q + 3]);

    // ---------------- policy tower ----------------
    float mean[kAct];
    tower_forward_keep<kAct>(U.fwd, 0, x, U.bufA[tid], U.bufB[tid], mean);
    PolicyHead h = {};
    if (live)
      h = policy_head(A.actions[row], mean, std_inv, logstd_sum, A.old_logp[row], (A.adv[row] - adv_mean) * adv_inv_std,
                      A.clip, A.ent_coef);
    reinterpret_cast<float4*>(U.g3[tid])[0] = make_float4(h.g_mean[0], h.g_mean[1], h.g_mean[2], h.g_mean[3]);
    // log_std gradient + statistics: warp sums -> smem -> fixed-order sum over the 4 warps (deterministic)
    {
      float v[7] = {h.g_logstd[0], h.g_logstd[1], h.g_logstd[2], h.g_logstd[3], h.pg_loss, h.kl, h.clipped};
#pragma unroll
      for (int q = 0; q < 7; ++q) v[q] = warp_sum(v[q]);
      if (lane == 0) {
#pragma unroll
        for (int q = 0; q < 7; ++q) U.wsum[tid >> 5][q] = v[q];
      }
    }
    __syncthreads();                                   // h2 (bufB), g3, wsum complete for the whole tile
    if (tid < 7) {
      const float sum = ((U.wsum[0][tid] + U.wsum[1][tid]) + U.wsum[2][tid]) + U.wsum[3][tid];
      const int dst = (tid < kAct) ? (O_LOGSTD + tid) : (tid == 4 ? kParams + 0 : (tid == 5 ? kParams + 2 : kParams + 3));
      U.G[dst] += sum;
    }
    wgrad_head<kAct>(U, O_PI_W3, O_PI_B3, rows);
    __syncthreads();                                   // dW3 has consumed h2
    float d1[kHid];
    tower_backward<kAct>(U, 0, h.g_mean, U.bufA[tid], U.bufB[tid], d1);
    __syncthreads();                                   // delta2 rows complete
    wgrad_hidden(U, O_PI_W2, O_PI_B2, rows);
    __syncthreads();                                   // dW2 has consumed h1
#pragma unroll
    for (int q = 0; q < kHid / 4; ++q)
      reinterpret_cast<float4*>(U.bufA[tid])[q] = make_float4(d1[4 * q], d1[4 * q + 1], d1[4 * q + 2], d1[4 * q + 3]);
    __syncthreads();
    wgrad_input(U, O_PI_W1, O_PI_B1, rows);
    __syncthreads();

    // ---------------- value tower ----------------
    float val[1];
    tower_forward_keep<1>(U.fwd, 1, x, U.bufA[tid], U.bufB[tid], val);
    float g_v[1] = {0.f}, st_vl = 0.f;
    if (live) g_v[0] = value_head(val[0], A.ret[row], A.vf_coef, st_vl);
    U.g3[tid][0] = g_v[0];
    {
      const float v0 = warp_sum(st_vl), v1 = warp_sum(live ? 1.0f : 0.f);
      if (lane == 0) { U.wsum[tid >> 5][0] = v0; U.wsum[tid >> 5][1] = v1; }
    }
    __syncthreads();
    if (tid < 2) U.G[kParams + (tid == 0 ? 1 : 4)] += ((U.wsum[0][tid] + U.wsum[1][tid]) + U.wsum[2][tid]) + U.wsum[3][tid];
    wgrad_head<1>(U, O_VF_W3, O_VF_B3, rows);
    __syncthreads();
    tower_backward<1>(U, 1, g_v, U.bufA[tid], U.bufB[tid], d1);
    __syncthreads();
    wgrad_hidden(U, O_VF_W2, O_VF_B2, rows);
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kHid / 4; ++q)
      reinterpret_cast<float4*>(U.bufA[tid])[q] = make_float4(d1[4 * q], d1[4 * q + 1], d1[4 * q + 2], d1[4 * q + 3]);
    __syncthreads();
    wgrad_input(U, O_VF_W1, O_VF_B1, rows);
    __syncthreads();
  }

  float* out = A.partials + (size_t)blockIdx.x * kGradLen;
  for (int idx = tid; idx < kGradLen; idx += kUpdBlock) out[idx] = U.G[idx];
}

// fixed-order sum of the per-CTA partial vectors -> grad[kGradLen] (sum over samples, not yet / M)
__global__ void ppo_reduce_kernel(const float* __restrict__ partials, int n_partials, float* __restrict__ grad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kGradLen) return;
  float sum = 0.f;
  for (int p = 0; p < n_partials; ++p) sum += partials[(size_t)p * kGradLen + idx];
  grad[idx] = sum;
}

// advantage statistics of a minibatch, deterministic: per-CTA partial sums (float64) in a fixed
// grid, then a one-thread fixed-order sum that ACCUMULATES [sum, sum of squares, count] into out[3]
__global__ void adv_stats_kernel(const float* __restrict__ adv, const int32_t* __restrict__ index, int64_t first,
                                 int64_t m, double* __restrict__ partial) {
  __shared__ double sh[2][8];
  double s = 0.0, q = 0.0;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
    const double a = (double)adv[index ? (int64_t)index[p] : first + p];
    s += a; q += a * a;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[threadIdx.x][w];
    partial[2 * blockIdx.x + threadIdx.x] = t;
  }
}

__global__ void adv_stats_finish_kernel(const double* __restrict__ partial, int n_partials, int64_t m,
                                        double* __restrict__ out) {
  // one warp; lane l sums partials l, l+32, ... in order, then a fixed shuffle tree: deterministic
  double s = 0.0, q = 0.0;
  for (int p = threadIdx.x; p < n_partials; p += 32) { s += partial[2 * p]; q += partial[2 * p + 1]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if (threadIdx.x == 0) { out[0] += s; out[1] += q; out[2] += (double)m; }
}

// the same statistics for EVERY minibatch of an epoch in two launches: minibatch b = positions [b * batch, min((b + 1) *
// batch, B)) of the epoch's index array.  grid (gx, n_mb); partial [n_mb][gx][2]; out [n_mb][3] is WRITTEN.
__global__ void adv_stats_epoch_kernel(const float* __restrict__ adv, const int32_t* __restrict__ index, int64_t B,
                                       int64_t batch, double* __restrict__ partial) {
  __shared__ double sh[2][8];
  const int64_t lo = (int64_t)blockIdx.y * batch, hi = min(lo + batch, B);
  double s = 0.0, q = 0.0;
  for (int64_t p = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hi; p += (int64_t)gridDim.x * blockDim.x) {
    const double a = (double)adv[index ? (int64_t)index[p] : p];
    s += a; q += a * a;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[threadIdx.x][w];
    partial[2 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x) + threadIdx.x] = t;
  }
}

__global__ void adv_stats_epoch_finish_kernel(const double* __restrict__ partial, int gx, int64_t B, int64_t batch,
                                              double* __restrict__ out) {
  const double* p0 = partial + 2 * (size_t)blockIdx.x * gx;
  double s = 0.0, q = 0.0;
  for (int p = threadIdx.x; p < gx; p += 32) { s += p0[2 * p]; q += p0[2 * p + 1]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if (threadIdx.x == 0) {
    const int64_t lo = (int64_t)blockIdx.x * batch;
    out[3 * blockIdx.x] = s; out[3 * blockIdx.x + 1] = q; out[3 * blockIdx.x + 2] = (double)(min(lo + batch, B) - lo);
  }
}

struct AdamArgs {
  float* theta; const float* grad; float* m; float* v;
  float inv_count;           // 1 / (global number of samples in the minibatch)
  float lr, beta1, beta2, eps, max_norm;
  long long* step;           // device-resident AdamClock {step, beta1^step, beta2^step} (advanced here: the launch sequence is CUDA-graph capturable)
  float* info;               // [kStats + 1]: mean statistics + pre-clip gradient norm of THIS step (nullable)
  float* info_sum;           // [kStats + 2]: the same values ACCUMULATED over the steps + the number of steps (nullable):
                             // SB3 logs the mean over all minibatches of PPO.train(), not the last one
};

// Adam's bias corrections 1 - beta^t: the powers are kept as running float64 products next to the step count
// ([step][beta1^t][beta2^t], 24 bytes; dronecu_ppo_set_state recomputes them with pow on the host) -- a device-side double
// pow per optimiser step sat on the critical path of this single-CTA kernel.
struct AdamClock { long long step; double b1pow, b2pow; };

// statistics of one optimiser step: threads 0 .. kStats+1 each handle ONE entry (one thread walking ten dependent global
// read-modify-writes was half of this kernel's 19 us)
__device__ __forceinline__ void apply_publish_info(const AdamArgs& A, const float* stats /* [kStats] sums */, const float inv_count,
                                                   const float norm) {
  const int q = threadIdx.x;
  if (q < kStats) {
    const float v = stats[q] * (q == 4 ? 1.0f : inv_count);
    if (A.info) A.info[q] = v;
    if (A.info_sum) A.info_sum[q] += v;
  } else if (q == kStats) {
    if (A.info) A.info[kStats] = norm;
    if (A.info_sum) A.info_sum[kStats] += norm;
  } else if (q == kStats + 1) {
    if (A.info_sum) A.info_sum[kStats + 1] += 1.0f;
  }
}

// torch.nn.utils.clip_grad_norm_(max_norm) + torch.optim.Adam.step() on the flat vector (one CTA of kApplyBlock threads).
// Latency-bound (10,697 parameters: 11 per thread), and on the reference's own shape it runs 320 times per 2048 env steps:
// every thread's gradient entries stay in registers between the norm and the update, and the Adam moments are fetched BEFORE
// the block-wide norm reduction so that their latency hides behind it (18 -> 6 us per launch, serialised ncu figures).
constexpr int kApplyBlock = 1024;
constexpr int kApplyPer = (kParams + kApplyBlock - 1) / kApplyBlock;       // 11

// g[k] = this thread's k-th gradient entry (already the SUM over samples / ranks), scale = 1 / sample count.
// Same arithmetic and the same summation order as the loops this replaces: bit-identical parameters.
__device__ __forceinline__ void clip_adam_apply(const AdamArgs& A, const float (&g_in)[kApplyPer], const float* stats, const float scale,
                                                float* red /* [32] shared */, float* scal /* [3] shared */) {
  const int tid = threadIdx.x;
  if (tid == 0) {      // torch.optim.Adam bias corrections of step t = ++step
    AdamClock* clk = reinterpret_cast<AdamClock*>(A.step);
    const double p1 = clk->b1pow * (double)A.beta1, p2 = clk->b2pow * (double)A.beta2;
    clk->step += 1; clk->b1pow = p1; clk->b2pow = p2;
    scal[1] = (float)((double)A.lr / (1.0 - p1));
    scal[2] = (float)(1.0 / sqrt(1.0 - p2));
  }
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < kApplyPer; ++k) {
    const float g = g_in[k] * scale;             // entries past kParams are 0
    sq = fmaf(g, g, sq);
  }
  float m[kApplyPer], v[kApplyPer];
#pragma unroll
  for (int k = 0; k < kApplyPer; ++k) {
    const int i = tid + k * kApplyBlock;
    m[k] = (i < kParams) ? A.m[i] : 0.f;
    v[k] = (i < kParams) ? A.v[i] : 0.f;
  }
  sq = warp_sum(sq);
  if ((tid & 31) == 0) red[tid >> 5] = sq;
  __syncthreads();
  if (tid < 32) {
    float t = red[tid];
    t = warp_sum(t);
    if (tid == 0) scal[0] = sqrtf(t);            // the pre-clip gradient norm
  }
  __syncthreads();
  const float norm = scal[0];
  apply_publish_info(A, stats, scale, norm);
  // torch.clamp(clip_coef, max=1.0): a non-finite gradient gives a NaN norm and a NaN coefficient that poisons every
  // parameter, as in torch (min.NaN; fminf would return 1 and update every finite entry as if nothing happened)
  float coef = A.max_norm / (norm + 1e-6f);
  asm("min.NaN.f32 %0, %0, %1;" : "+f"(coef) : "f"(1.0f));
  coef *= scale;
  const float lr_over_bc1 = scal[1], inv_sqrt_bc2 = scal[2];
  float th[kApplyPer];
#pragma unroll
  for (int k = 0; k < kApplyPer; ++k) {
    const int i = tid + k * kApplyBlock;
    th[k] = (i < kParams) ? A.theta[i] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < kApplyPer; ++k) {
    const int i = tid + k * kApplyBlock;
    if (i < kParams) {
      const float g = g_in[k] * coef;
      const float mm = A.beta1 * m[k] + (1.0f - A.beta1) * g;
      const float vv = A.beta2 * v[k] + (1.0f - A.beta2) * g * g;
      A.m[i] = mm; A.v[i] = vv;
      A.theta[i] = th[k] - lr_over_bc1 * mm / (sqrtf(vv) * inv_sqrt_bc2 + A.eps);
    }
  }
}

__global__ void __launch_bounds__(kApplyBlock) ppo_apply_kernel(const AdamArgs A) {
  __shared__ float red[32];
  __shared__ float scal[3];
  float g[kApplyPer];
#pragma unroll
  for (int k = 0; k < kApplyPer; ++k) {
    const int i = threadIdx.x + k * kApplyBlock;
    g[k] = (i < kParams) ? A.grad[i] : 0.f;
  }
  clip_adam_apply(A, g, A.grad + kParams, A.inv_count, red, scal);
}

// ---------------------------------------------------------------------------------------------
// Minibatch order: SB3 draws np.random.permutation(B) once per epoch (PPO.train -> RolloutBuffer.get).  Here the
// permutation is a keyed bijection evaluated per element -- no sort, no scratch: on k = ceil(log2 B) bits,
// four rounds of  x = ((x ^ (x >> s)) * odd + add) mod 2^k  (each step is a bijection on k-bit integers), with
// the multipliers / addends taken from Philox4x32-10(key = seed, counter = (epoch, round)), and cycle-walking
// (re-apply until the value is < B; < 2 applications on average).  oracle/philox.py: minibatch_permutation.
// ---------------------------------------------------------------------------------------------
struct PermKey {
  uint32_t mul[4], add[4];
  uint32_t mask, shift;
};

__host__ __device__ inline uint32_t perm_apply(uint32_t x, const PermKey& K, uint32_t n) {
  do {
#ifdef __CUDA_ARCH__
#pragma unroll
#endif
    for (int r = 0; r < 4; ++r) {
      x ^= x >> K.shift;
      x = (x * K.mul[r] + K.add[r]) & K.mask;
    }
  } while (x >= n);
  return x;
}

__global__ void perm_kernel(int32_t* __restrict__ out, uint32_t n, const __grid_constant__ PermKey K) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int32_t)perm_apply(i, K, n);
}

// ---------------------------------------------------------------------------------------------
// Minibatch PARTITION with sorted rows.  The same keyed bijection f, read the other way round: row r of the buffer belongs
// to minibatch f(r) / batch (a uniformly random partition into minibatches of exactly `batch` rows, as the slices of a random
// permutation are), and the index array lists every minibatch's rows in ASCENDING order.  The minibatch gradient is a sum, so
// the order inside a minibatch is free; ascending rows turn the update kernels' observation gathers from 8 M random 60-byte
// reads over a 3 GB buffer (one TLB miss per row: the gather issue alone took 4.8k of 17.6k cycles per tile in the in-kernel
// timeline, profiles/README.md r02) into a forward sweep with ~4-row strides.
// A stable counting sort by minibatch id, one WARP per chunk of `rows_per_warp` consecutive rows:
//   part_hist_kernel     H[key][chunk] = rows of the chunk in minibatch `key`
//   part_scan_kernel     exclusive prefix sum of H in (key, chunk) order, in place (one CTA)
//   part_scatter_kernel  every warp walks its chunk in row order and writes row r to out[H[key][chunk]++]
// ---------------------------------------------------------------------------------------------
constexpr int kPartMaxBins = 64;
constexpr int kPartWarps = 8;

// x / d for an invariant 32-bit divisor (Granlund-Montgomery: q = (t + ((x - t) >> s1)) >> s2 with t = umulhi(M, x)); a hardware-free
// 32-bit division is ~15 instructions, this is 5 -- the partition kernels divide once per buffer row
struct FastDiv { uint32_t M, s1, s2; };
inline FastDiv fast_div_make(uint32_t d) {
  FastDiv f;
  uint32_t l = 0;
  while ((1ull << l) < d) ++l;                                   // l = ceil(log2 d)
  f.M = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
  f.s1 = l < 1 ? l : 1u;
  f.s2 = l < 1 ? 0u : l - 1;
  return f;
}
__host__ __device__ __forceinline__ uint32_t fast_div(uint32_t x, const FastDiv& f) {
#ifdef __CUDA_ARCH__
  const uint32_t t = __umulhi(f.M, x);
#else
  const uint32_t t = (uint32_t)(((uint64_t)f.M * x) >> 32);
#endif
  return (t + ((x - t) >> f.s1)) >> f.s2;
}

__device__ __forceinline__ uint32_t part_key(uint32_t r, const PermKey& K, uint32_t n, const FastDiv& batch) {
  return fast_div(perm_apply(r, K, n), batch);
}

__global__ void __launch_bounds__(32 * kPartWarps) part_hist_kernel(uint32_t n, FastDiv batch, uint32_t n_bins, uint32_t rows_per_warp,
                                                                   uint32_t n_chunks, const __grid_constant__ PermKey K, uint32_t* __restrict__ H) {
  __shared__ uint32_t hist[kPartWarps][kPartMaxBins];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t chunk = blockIdx.x * kPartWarps + warp;
  for (uint32_t b = lane; b < n_bins; b += 32) hist[warp][b] = 0;
  __syncwarp();
  if (chunk < n_chunks) {
    const uint32_t lo = chunk * rows_per_warp, hi = min(n, lo + rows_per_warp);
    for (uint32_t r0 = lo; r0 < hi; r0 += 32) {
      const uint32_t r = r0 + lane;
      const bool on = r < hi;
      const uint32_t key = on ? part_key(r, K, n, batch) : 0xffffffffu;
      const uint32_t same = __match_any_sync(0xffffffffu, key);
      if (on && lane == (uint32_t)(__ffs(same) - 1)) hist[warp][key] += __popc(same);
      __syncwarp();
    }
    for (uint32_t b = lane; b < n_bins; b += 32) H[(size_t)b * n_chunks + chunk] = hist[warp][b];
  }
}

__global__ void __launch_bounds__(1024) part_scan_kernel(uint32_t* __restrict__ H, uint32_t len) {
  // one CTA walks H in tiles of 1024 consecutive elements (coalesced): a shuffle scan per warp + a scan of the 32 warp totals
  // per tile, a running carry across the tiles.  The loads of 16 tiles are issued together (one memory round trip per 16 tiles
  // instead of one per tile: the tile loop is a dependent chain).
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry_s;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  constexpr int kAhead = 16;
  for (uint32_t base0 = 0; base0 < len; base0 += 1024 * kAhead) {
    uint32_t vals[kAhead];
#pragma unroll
    for (int t = 0; t < kAhead; ++t) {
      const uint32_t i = base0 + 1024 * t + threadIdx.x;
      vals[t] = i < len ? H[i] : 0u;
    }
#pragma unroll
    for (int t = 0; t < kAhead; ++t) {
      const uint32_t base = base0 + 1024 * t;
      if (base >= len) break;
      const uint32_t i = base + threadIdx.x;
      const uint32_t v = vals[t];
      uint32_t incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += u; }
      if (lane == 31) wsum[warp] = incl;
      __syncthreads();
      if (warp == 0) {
        uint32_t w = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, w, o); if (lane >= (uint32_t)o) w += u; }
        wsum[lane] = w;                                   // inclusive scan of the warp totals
      }
      __syncthreads();
      const uint32_t carry = carry_s;
      if (i < len) H[i] = carry + (warp ? wsum[warp - 1] : 0u) + incl - v;        // exclusive prefix
      __syncthreads();
      if (threadIdx.x == 0) carry_s = carry + wsum[31];
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(32 * kPartWarps) part_scatter_kernel(uint32_t n, FastDiv batch, uint32_t n_bins, uint32_t rows_per_warp,
                                                                      uint32_t n_chunks, const __grid_constant__ PermKey K,
                                                                      const uint32_t* __restrict__ H, int32_t* __restrict__ out) {
  __shared__ uint32_t base[kPartWarps][kPartMaxBins];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t chunk = blockIdx.x * kPartWarps + warp;
  if (chunk >= n_chunks) return;
  for (uint32_t b = lane; b < n_bins; b += 32) base[warp][b] = H[(size_t)b * n_chunks + chunk];
  __syncwarp();
  const uint32_t lo = chunk * rows_per_warp, hi = min(n, lo + rows_per_warp);
  for (uint32_t r0 = lo; r0 < hi; r0 += 32) {
    const uint32_t r = r0 + lane;
    const bool on = r < hi;
    const uint32_t key = on ? part_key(r, K, n, batch) : 0xffffffffu;
    const uint32_t same = __match_any_sync(0xffffffffu, key);
    if (on) out[base[warp][key] + __popc(same & ((1u << lane) - 1u))] = (int32_t)r;
    __syncwarp();
    if (on && lane == (uint32_t)(__ffs(same) - 1)) base[warp][key] += __popc(same);
    __syncwarp();
  }
}

}  // namespace dronecu
