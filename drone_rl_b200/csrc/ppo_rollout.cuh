// K-step rollout with the PPO policy / value MLP evaluated inside the step loop (float32 CUDA-core
// version: one env per thread, the 10,697 parameters transposed once per CTA into shared memory and
// read back as warp-broadcast 128-bit loads -- every lane multiplies the same weight by its own
// env's activation).  What SB3's collect_rollouts does per step (SURVEY.md appendix C; call site
// /root/reference/train.py:63-68): a, v, logp = policy(obs); env.step(clip(a)); buffer.add(obs, a,
// r, episode_start, v, logp) -- here for K steps without the state or the activations ever leaving
// the SM.
#pragma once
#include "env_kernels.cuh"
#include "ppo_common.cuh"
#include "obs_norm.cuh"

namespace dronecu {

constexpr int kPolBlock = 128;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// shared-memory image of the parameters, transposed to [in][out] so a thread walks the inputs of a
// layer and fetches 4 output weights per LDS.128
struct alignas(16) MlpSmem {
  float W1T[2][kObs][kHid];
  float b1[2][kHid];
  float W2T[2][kHid][kHid];
  float b2[2][kHid];
  float W3piT[kHid][kAct];
  float W3vf[kHid];
  float b3pi[kAct];
  float b3vf, pad[3];
  float log_std[kAct];
};

constexpr size_t kPolicySmem = sizeof(MlpSmem) + (kPolBlock / 32) * 32 * kObs * sizeof(float);

__device__ __forceinline__ void load_mlp_smem(MlpSmem& S, const float* __restrict__ theta) {
  for (int idx = threadIdx.x; idx < kParams; idx += blockDim.x) {
    const float v = theta[idx];
    int o = idx, t = 0;
    if (o >= O_VF_W1 && o < O_LOGSTD) { t = 1; o -= kTowerStride; }
    if (idx >= O_LOGSTD) { S.log_std[idx - O_LOGSTD] = v; continue; }
    if (o < O_PI_B1) { S.W1T[t][o % kObs][o / kObs] = v; }
    else if (o < O_PI_W2) { S.b1[t][o - O_PI_B1] = v; }
    else if (o < O_PI_B2) { const int q = o - O_PI_W2; S.W2T[t][q % kHid][q / kHid] = v; }
    else if (o < O_PI_W3) { S.b2[t][o - O_PI_B2] = v; }
    else if (t == 0) {
      if (o < O_PI_B3) { const int q = o - O_PI_W3; S.W3piT[q % kHid][q / kHid] = v; }
      else S.b3pi[o - O_PI_B3] = v;
    } else {
      // vf head: W3 [1,64] then b3 [1]; offsets relative to the pi block layout
      const int q = idx - O_VF_W3;
      if (q < kHid) S.W3vf[q] = v; else S.b3vf = v;
    }
  }
}

// one tower for one env: x[15] -> NOUT outputs.  h1 stays in registers; layer 2 is produced in four
// chunks of 16 units that are consumed by the head immediately, so h2 is never materialised.
template <int NOUT>
__device__ __forceinline__ void tower_forward(const MlpSmem& S, const int t, const float (&x)[kObs], float (&out)[NOUT]) {
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
  for (int j = 0; j < kHid; ++j) h1[j] = tanh_fast(h1[j]);

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
    for (int jj = 0; jj < 16; ++jj) {
      const float a = tanh_fast(acc[jj]);
      if constexpr (NOUT == kAct) {
        fma4s(out, reinterpret_cast<const float4*>(S.W3piT[16 * c + jj])[0], a);
      } else {
        out[0] = fmaf(S.W3vf[16 * c + jj], a, out[0]);
      }
    }
  }
}

struct PolicyArgs {
  StatePlanes state;
  EnvParams P;
  int64_t n;
  int32_t K;
  uint64_t t0;
  const float* theta;     // [kParams]
  int32_t deterministic;  // != 0: action = mean (SB3 predict(deterministic=True), test.py:14)
  float* obs;             // [K,n,15] observation the action was computed from ([K,n,16] when obs_padded)
  int32_t obs_padded;     // != 0: rows padded to 16 floats (64 bytes, the 16th = 1.0: the bias column of the update kernels' X tile)
  float4* actions;        // [K,n]    sampled action, NOT clipped (what SB3 stores in the buffer)
  float* logp;            // [K,n]
  float* value;           // [K,n]
  float* reward;          // [K,n]
  uint8_t* done;          // [K,n]
  float* last_value;      // [n]      V(observation after the K-th step)
  float* last_obs;        // [n,15]
  StatSlot* stats;
  const float* norm;      // [31] float32 affine record (obs_norm.cuh): read only by the NORM instantiations
  // read only by the TIMEOUT instantiations (DESIGN.md section 11): env i's j-th time-limit truncation of the launch goes to
  // slot j * n + i; term_slots >= ceil(K / max_steps) (checked by the host) always suffices
  float* term_obs;        // [T,n,16] raw pre-reset observation of the truncated step (info["terminal_observation"]), 16th = 1.0
  int32_t* term_row;      // [T,n]    its rollout-buffer row k * n + i; -1 in every slot the launch did not fill
  int32_t term_slots;     // T
};

// ---------------------------------------------------------------------------------------------
// The policy step, stated once for the three rollout kernels and the three evaluation kernels (ppo_eval.cuh): every kernel
// computes the std, the action and its log-prob, the env's clipped action and the episode statistics with these functions,
// so each reproduces the others bit for bit on the same operands.
// ---------------------------------------------------------------------------------------------

// std = exp(log_std) of SB3's state-independent Gaussian; returns sum(log_std), the log-prob's normaliser
__device__ __forceinline__ float policy_std(const float* log_std, float (&std_)[kAct]) {
  float logstd_sum = 0.f;
#pragma unroll
  for (int o = 0; o < kAct; ++o) { std_[o] = expf(log_std[o]); logstd_sum += log_std[o]; }
  return logstd_sum;
}

// the action of env env_id at step t (Philox noise index) and its log-prob: mean (SB3 deterministic) or mean + std * z,
// NOT clipped (what SB3 stores in the buffer)
__device__ __forceinline__ float4 policy_action(const float (&mean)[kAct], const float (&std_)[kAct], float logstd_sum,
                                                const PhiloxKeys& keys, uint64_t env_id, uint64_t t, bool deterministic,
                                                float& logp) {
  float4 a;
  if (deterministic) {
    a = make_float4(mean[0], mean[1], mean[2], mean[3]);
    logp = -logstd_sum - kAct * kHalfLog2Pi;
  } else {
    const float4 z = noise_normals(keys, env_id, t);
    a = make_float4(fmaf(std_[0], z.x, mean[0]), fmaf(std_[1], z.y, mean[1]),
                    fmaf(std_[2], z.z, mean[2]), fmaf(std_[3], z.w, mean[3]));
    // Normal(mean, std).log_prob(a) summed over the 4 dims; (a - mean) / std == z up to rounding
    logp = -0.5f * (z.x * z.x + z.y * z.y + z.z * z.z + z.w * z.w) - logstd_sum - kAct * kHalfLog2Pi;
  }
  return a;
}

// np.clip(a, low, high) for the env only (SB3 collect_rollouts); the buffer keeps `a`
__device__ __forceinline__ float4 env_action(const float4 a, float motor_max) {
  return make_float4(fminf(fmaxf(a.x, 0.f), motor_max), fminf(fmaxf(a.y, 0.f), motor_max),
                     fminf(fmaxf(a.z, 0.f), motor_max), fminf(fmaxf(a.w, 0.f), motor_max));
}

// a 64-byte observation row, the 16th value 1.0 (the bias column of the update kernels' X tile): four 128-bit stores
// straight from the registers
__device__ __forceinline__ void store_row16(float* row, const float (&x)[kObs]) {
  float4* d = reinterpret_cast<float4*>(row);
  st_quad(d, make_float4(x[0], x[1], x[2], x[3]));
  st_quad(d + 1, make_float4(x[4], x[5], x[6], x[7]));
  st_quad(d + 2, make_float4(x[8], x[9], x[10], x[11]));
  st_quad(d + 3, make_float4(x[12], x[13], x[14], 1.0f));
}

// The episodes an env (thread per env) or a warp (warp per env) finished in the launch.  At the end each CTA sums its
// tallies into shared counters, blk[3] (episodes, terminated, length sum) and blk_ret (return sum), zeroed by
// cta_stats_init; after a CTA barrier, thread 0 adds them to the CTA's StatSlot (cta_stats_commit).
struct EpisodeTally {
  // in this order, and declared after the kernels' n_trunc: the rollout kernels keep the register counts (-Xptxas -v)
  // they had with four local counters
  float ret_sum = 0.f;
  uint32_t len_sum = 0, n_term = 0, n_done = 0;

  __device__ __forceinline__ void add(bool crashed, const EnvState& s) {
    n_done += 1;
    n_term += crashed ? 1 : 0;
    len_sum += (uint32_t)s.ep_len;
    ret_sum += s.ep_ret;
  }
  // one env per lane: warp sums, then lane 0's shared atomics (every lane of the warp calls this)
  __device__ __forceinline__ void flush_warp(unsigned long long (&blk)[3], double& blk_ret, int lane) const {
    if (__ballot_sync(0xffffffffu, n_done != 0)) {
      const uint32_t d = __reduce_add_sync(0xffffffffu, n_done);
      const uint32_t t = __reduce_add_sync(0xffffffffu, n_term);
      const uint32_t l = __reduce_add_sync(0xffffffffu, len_sum);
      double rs = (double)ret_sum;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
      if (lane == 0) {
        atomicAdd(&blk[0], (unsigned long long)d);
        atomicAdd(&blk[1], (unsigned long long)t);
        atomicAdd(&blk[2], (unsigned long long)l);
        atomicAdd(&blk_ret, rs);
      }
    }
  }
  // the tally is already the warp's (one env per warp): its writer lane adds it as it stands
  __device__ __forceinline__ void flush_lane(unsigned long long (&blk)[3], double& blk_ret) const {
    if (n_done != 0) {
      atomicAdd(&blk[0], (unsigned long long)n_done);
      atomicAdd(&blk[1], (unsigned long long)n_term);
      atomicAdd(&blk[2], (unsigned long long)len_sum);
      atomicAdd(&blk_ret, (double)ret_sum);
    }
  }
};

__device__ __forceinline__ void cta_stats_init(unsigned long long (&blk)[3], double& blk_ret) {
  if (threadIdx.x < 3) blk[threadIdx.x] = 0;
  if (threadIdx.x == 3) blk_ret = 0.0;
}

// thread 0 after the CTA barrier that follows every flush, slot = stats + blockIdx.x % kStatSlots (the CTA's line)
__device__ __forceinline__ void cta_stats_commit(StatSlot* slot, const unsigned long long (&blk)[3], const double& blk_ret) {
  if (blk[0] != 0) {
    atomicAdd(&slot->episodes, blk[0]);
    atomicAdd(&slot->terminated, blk[1]);
    atomicAdd(&slot->length_sum, blk[2]);
    atomicAdd(&slot->return_sum, blk_ret);
  }
}

// TIMEOUT: a step that ended by the time limit alone (timeout && !crashed: Gymnasium's truncated), recorded after step_env
// and before reset_env -- the observation SB3 keeps as info["terminal_observation"].  j counts this env's truncations.
__device__ __forceinline__ void record_truncation(const PolicyArgs& A, const EnvState& s, const int64_t i, const int k,
                                                  int32_t& j, const bool writer) {
  if (writer && j < A.term_slots) {
    float x[kObs];
    write_obs<kObs>(x, s);
    const size_t slot = (size_t)j * (size_t)A.n + (size_t)i;
    store_row16(A.term_obs + slot * 16, x);
    A.term_row[slot] = (int32_t)((int64_t)k * A.n + i);
  }
  ++j;
}

// TIMEOUT: the slots env i did not fill read -1, so the side buffer is fully defined after every launch
__device__ __forceinline__ void close_truncation_slots(const PolicyArgs& A, const int64_t i, int32_t j) {
  for (; j < A.term_slots; ++j) A.term_row[(size_t)j * (size_t)A.n + (size_t)i] = -1;
}

// NORM: the towers see norm_obs_row(x) (obs_norm.cuh) -- the buffer still receives the raw row, obs_norm_pass_kernel
// normalises it afterwards with the same function and the same record.  TIMEOUT: truncated steps are recorded
// (record_truncation) for timeout_bootstrap_kernel (ppo_timeout.cuh); nothing else changes.
template <bool RANDOMIZED, bool NORM = false, bool TIMEOUT = false>
__global__ void __launch_bounds__(kPolBlock) policy_rollout_kernel(const __grid_constant__ PolicyArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];      // > 48 KB: dynamic shared memory
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  float (*tiles)[32 * kObs] = reinterpret_cast<float (*)[32 * kObs]>(smem_raw + sizeof(MlpSmem));
  __shared__ unsigned long long blk_stats[3];
  __shared__ double blk_ret;
  __shared__ float s_norm[NORM ? kNormAffine : 1];

  load_mlp_smem(S, A.theta);
  load_norm<NORM>(s_norm, A.norm);
  cta_stats_init(blk_stats, blk_ret);
  __syncthreads();

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

    float mean[kAct], val[1];
    tower_forward<kAct>(S, 0, x, mean);
    tower_forward<1>(S, 1, x, val);

    float logp;
    const float4 a = policy_action(mean, std_, logstd_sum, P.keys, env_id, A.t0 + (uint64_t)k, A.deterministic, logp);
    const StepResult r = step_env(s, P, env_action(a, P.motor_max));
    const bool done = r.crashed || r.timeout;
    if (active) {
      if (A.actions != nullptr) st_quad(p_act, a);
      if (A.logp != nullptr) *p_logp = logp;
      if (A.value != nullptr) *p_val = val[0];
      if (A.reward != nullptr) *p_rew = r.reward;
      if (A.done != nullptr) *p_done = done ? 1 : 0;
      if (done) {
        tally.add(r.crashed, s);
        if constexpr (TIMEOUT) { if (!r.crashed) record_truncation(A, s, i, k, n_trunc, true); }
        reset_env<RANDOMIZED>(s, P, env_id);       // the PPO path always auto-resets (DummyVecEnv)
      }
    }
    p_act += n; p_logp += n; p_val += n; p_rew += n; p_done += n; p_obs += n * kObs;
  }

  // bootstrap value of the observation after the last step (SB3: policy.predict_values(new_obs))
  {
    float x[kObs], val[1];
    write_obs<kObs>(x, s);
    if (A.last_value != nullptr) {
      if constexpr (NORM) norm_obs_row(x, s_norm);
      tower_forward<1>(S, 1, x, val);
      if (active) A.last_value[i] = val[0];
    }
    if (A.last_obs != nullptr && valid > 0)
      emit_obs_rows<kObs>(tile, A.last_obs + warp_base * kObs, s, lane, valid, active,
                          emit_fast_ok<kObs>(A.last_obs, warp_base, n, valid));
  }
  if (active) store_state(A.state, i, s);
  if constexpr (TIMEOUT) { if (active) close_truncation_slots(A, i, n_trunc); }

  tally.flush_warp(blk_stats, blk_ret, lane);
  __syncthreads();
  if (threadIdx.x == 0) cta_stats_commit(A.stats + (blockIdx.x % kStatSlots), blk_stats, blk_ret);
}

// ---------------------------------------------------------------------------------------------
// Small batches (the reference's own shape is ONE env: train.py:33-43): one WARP per env.  With one env per thread a step
// is a chain of ~10,000 dependent FMAs in a single thread (20 us per env step whatever the batch size below ~75k envs); here
// the 64 hidden units of a layer are spread over the 32 lanes (units 2 * lane and 2 * lane + 1: one LDS.64 + one packed FMA per input), the env state and the observation
// are replicated in every lane (the env step is computed redundantly: no broadcast, no divergence), the activations of a
// layer go through 256 bytes of shared memory per warp.  Same float32 arithmetic and the same fmaf order per hidden unit as
// policy_rollout_kernel (layers 1 and 2 are bit-identical); the four / one head sums are warp reductions.
// ---------------------------------------------------------------------------------------------
constexpr int kSmallWarps = 4;                  // envs per CTA
constexpr size_t kPolicySmallSmem = sizeof(MlpSmem) + sizeof(float) * kSmallWarps * kHid;

template <int NOUT>
__device__ __forceinline__ void tower_forward_warp(const MlpSmem& S, float* __restrict__ hbuf, const int t, const float (&x)[kObs],
                                                   float (&out)[NOUT], const int lane) {
  // this lane's two hidden units are 2 * lane and 2 * lane + 1: one LDS.64 of weights + one packed FMA per input
  const int u = 2 * lane;
  float2 a = *reinterpret_cast<const float2*>(S.b1[t] + u);
#pragma unroll
  for (int i = 0; i < kObs; ++i) {
    const float2 w = *reinterpret_cast<const float2*>(S.W1T[t][i] + u);
    fma2(a.x, a.y, w.x, w.y, x[i], x[i]);
  }
  a.x = tanh_fast(a.x); a.y = tanh_fast(a.y);
  __syncwarp();                                 // the previous tower's readers of hbuf are done
  *reinterpret_cast<float2*>(hbuf + u) = a;
  __syncwarp();
  float2 c = *reinterpret_cast<const float2*>(S.b2[t] + u);
#pragma unroll
  for (int k4 = 0; k4 < kHid / 4; ++k4) {
    const float4 h = reinterpret_cast<const float4*>(hbuf)[k4];          // warp-broadcast
    const float2 w0 = *reinterpret_cast<const float2*>(S.W2T[t][4 * k4] + u), w1 = *reinterpret_cast<const float2*>(S.W2T[t][4 * k4 + 1] + u);
    const float2 w2 = *reinterpret_cast<const float2*>(S.W2T[t][4 * k4 + 2] + u), w3 = *reinterpret_cast<const float2*>(S.W2T[t][4 * k4 + 3] + u);
    fma2(c.x, c.y, w0.x, w0.y, h.x, h.x);
    fma2(c.x, c.y, w1.x, w1.y, h.y, h.y);
    fma2(c.x, c.y, w2.x, w2.y, h.z, h.z);
    fma2(c.x, c.y, w3.x, w3.y, h.w, h.w);
  }
  const float c0 = tanh_fast(c.x), c1 = tanh_fast(c.y);
  if constexpr (NOUT == kAct) {
    const float4 w0 = reinterpret_cast<const float4*>(S.W3piT[u])[0], w1 = reinterpret_cast<const float4*>(S.W3piT[u + 1])[0];
    out[0] = warp_sum(fmaf(w1.x, c1, w0.x * c0)) + S.b3pi[0];
    out[1] = warp_sum(fmaf(w1.y, c1, w0.y * c0)) + S.b3pi[1];
    out[2] = warp_sum(fmaf(w1.z, c1, w0.z * c0)) + S.b3pi[2];
    out[3] = warp_sum(fmaf(w1.w, c1, w0.w * c0)) + S.b3pi[3];
  } else {
    const float2 w = *reinterpret_cast<const float2*>(S.W3vf + u);
    out[0] = warp_sum(fmaf(w.y, c1, w.x * c0)) + S.b3vf;
  }
}

template <bool RANDOMIZED, bool NORM = false, bool TIMEOUT = false>
__global__ void __launch_bounds__(32 * kSmallWarps) policy_rollout_warp_kernel(const __grid_constant__ PolicyArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  __shared__ unsigned long long blk_stats[3];
  __shared__ double blk_ret;
  __shared__ float s_norm[NORM ? kNormAffine : 1];
  load_mlp_smem(S, A.theta);
  load_norm<NORM>(s_norm, A.norm);
  cta_stats_init(blk_stats, blk_ret);
  __syncthreads();

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* const hbuf = reinterpret_cast<float*>(smem_raw + sizeof(MlpSmem)) + warp * kHid;
  const int64_t i = (int64_t)blockIdx.x * kSmallWarps + warp;          // this warp's env
  const bool active = i < A.n;                                            // warp-uniform
  const EnvParams& P = A.P;
  const uint64_t env_id = P.env_offset + (uint64_t)i;
  const size_t n = (size_t)A.n;
  const bool writer = active && lane == 0;

  EnvState s = {};
  if (active) s = load_state(A.state, i);                                 // every lane holds the whole state
  float std_[kAct];
  const float logstd_sum = policy_std(S.log_std, std_);
  int32_t n_trunc = 0;
  EpisodeTally tally;

  for (int k = 0; k < A.K; ++k) {
    float x[kObs];
    write_obs<kObs>(x, s);
    const size_t row = (size_t)k * n + (size_t)i;
    if (writer && A.obs != nullptr) {
      if (A.obs_padded) {
        float4* d = reinterpret_cast<float4*>(A.obs + row * 16);
        d[0] = make_float4(x[0], x[1], x[2], x[3]); d[1] = make_float4(x[4], x[5], x[6], x[7]);
        d[2] = make_float4(x[8], x[9], x[10], x[11]); d[3] = make_float4(x[12], x[13], x[14], 1.0f);
      } else {
#pragma unroll
        for (int c = 0; c < kObs; ++c) A.obs[row * kObs + c] = x[c];
      }
    }
    if constexpr (NORM) norm_obs_row(x, s_norm);
    float mean[kAct], val[1];
    tower_forward_warp<kAct>(S, hbuf, 0, x, mean, lane);
    tower_forward_warp<1>(S, hbuf, 1, x, val, lane);

    float logp;
    const float4 a = policy_action(mean, std_, logstd_sum, P.keys, env_id, A.t0 + (uint64_t)k, A.deterministic, logp);
    const StepResult r = step_env(s, P, env_action(a, P.motor_max));
    const bool done = r.crashed || r.timeout;
    if (writer) {
      if (A.actions != nullptr) A.actions[row] = a;
      if (A.logp != nullptr) A.logp[row] = logp;
      if (A.value != nullptr) A.value[row] = val[0];
      if (A.reward != nullptr) A.reward[row] = r.reward;
      if (A.done != nullptr) A.done[row] = done ? 1 : 0;
    }
    if (active && done) {                                                 // warp-uniform
      tally.add(r.crashed, s);
      if constexpr (TIMEOUT) { if (!r.crashed) record_truncation(A, s, i, k, n_trunc, lane == 0); }
      reset_env<RANDOMIZED>(s, P, env_id);
    }
  }
  {
    float x[kObs], val[1];
    write_obs<kObs>(x, s);
    if (A.last_value != nullptr) {
      if constexpr (NORM) {                     // x itself is stored raw to last_obs below
        float xn[kObs];
#pragma unroll
        for (int c = 0; c < kObs; ++c) xn[c] = x[c];
        norm_obs_row(xn, s_norm);
        tower_forward_warp<1>(S, hbuf, 1, xn, val, lane);
      } else {
        tower_forward_warp<1>(S, hbuf, 1, x, val, lane);
      }
      if (writer) A.last_value[i] = val[0];
    }
    if (writer && A.last_obs != nullptr) {
#pragma unroll
      for (int c = 0; c < kObs; ++c) A.last_obs[i * kObs + c] = x[c];
    }
  }
  if (writer) {
    store_state(A.state, i, s);
    if constexpr (TIMEOUT) close_truncation_slots(A, i, n_trunc);
    tally.flush_lane(blk_stats, blk_ret);
  }
  __syncthreads();
  if (threadIdx.x == 0) cta_stats_commit(A.stats + (blockIdx.x % kStatSlots), blk_stats, blk_ret);
}

// policy(obs) for arbitrary observation rows: mean [B,4], value [B]  (PPO.predict / policy.forward)
__global__ void __launch_bounds__(kPolBlock) policy_forward_kernel(const float* __restrict__ theta,
                                                                   const float* __restrict__ obs, int64_t B,
                                                                   float4* __restrict__ mean, float* __restrict__ value) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  MlpSmem& S = *reinterpret_cast<MlpSmem*>(smem_raw);
  load_mlp_smem(S, theta);
  __syncthreads();
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < B; r += (int64_t)gridDim.x * blockDim.x) {
    float x[kObs], m[kAct], v[1];
#pragma unroll
    for (int i = 0; i < kObs; ++i) x[i] = obs[r * kObs + i];
    tower_forward<kAct>(S, 0, x, m);
    tower_forward<1>(S, 1, x, v);
    if (mean) mean[r] = make_float4(m[0], m[1], m[2], m[3]);
    if (value) value[r] = v[0];
  }
}

// GAE(gamma, lambda) reverse scan, one env per thread (SB3 RolloutBuffer.compute_returns_and_advantage;
// done[t] == episode_start[t+1]; no bootstrap on time-outs: the reference env sets no TimeLimit key).
__global__ void gae_kernel(int K, int64_t n, const float* __restrict__ reward, const float* __restrict__ value,
                           const uint8_t* __restrict__ done, const float* __restrict__ last_value, float gamma,
                           float lam, float* __restrict__ adv, float* __restrict__ ret) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float next_v = last_value[i], last = 0.f;
  for (int t = K - 1; t >= 0; --t) {
    const int64_t j = (int64_t)t * n + i;
    const float nnt = done[j] ? 0.f : 1.0f;
    const float v = value[j];
    const float delta = reward[j] + gamma * next_v * nnt - v;
    last = delta + gamma * lam * nnt * last;
    adv[j] = last;
    ret[j] = last + v;
    next_v = v;
  }
}

}  // namespace dronecu
