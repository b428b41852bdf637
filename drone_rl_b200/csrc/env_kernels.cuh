// Fused K-step environment kernel and the small state-management kernels.
//
// Thread mapping: one env per thread, 256 envs per CTA, the state of an env lives in the
// registers of its thread for all K steps of a launch (HBM sees the state once in, once out).
// Observations ([n,D] row-major, what the reference's _get_obs returns: drone.py:77-79) are
// transposed through a per-warp shared-memory tile (stride D = 15 or 12 words; 15 is odd, so the
// 32 lanes hit 32 different banks) and leave the SM as 128-bit fully coalesced stores over the
// warp's 32*D contiguous floats instead of D strided 4-byte stores per thread.
#pragma once
#include "env_core.cuh"

namespace dronecu {

constexpr int kBlock = 256;
constexpr int kWarps = kBlock / 32;
constexpr int kStatSlots = 128;   // episode statistics are spread over this many L2 lines

struct StatSlot {   // one 64-byte line per slot
  unsigned long long episodes, terminated, length_sum;
  double return_sum;
  unsigned long long pad[4];
};

struct RolloutArgs {
  StatePlanes state;
  EnvParams P;
  int64_t n;
  int32_t K;
  uint64_t t0;                 // global step index of the first step of this launch (Philox index)
  const float4* actions;       // [K,n] quads (STREAMED)
  float* obs0;                 // [n,D]
  float* next_obs;             // [K,n,D]
  float4* out_actions;         // [K,n]
  float* reward;               // [K,n]
  uint8_t* done;               // [K,n]
  uint8_t* truncated;          // [K,n]
  float* terminal_obs;         // [K,n,D]  written only where done
  float* episode_r;            // [K,n]    written only where done
  int32_t* episode_l;          // [K,n]    written only where done
  StatSlot* stats;             // [kStatSlots]
};

// <= 80 registers/thread, 3 CTAs of 256 threads per SM: no spills and no per-step re-derivation of indices (at 64
// registers ptxas did both); A/B in profiles/README.md
constexpr int kMinBlocks = 3;

// One warp's 32 observations: registers -> per-warp smem tile (stride D words) -> global as
// 128-bit coalesced stores (lane j moves quad j, j+32, ... of the 32*D contiguous floats).
// A cp.async.bulk store of the tile measured no faster (profiles/README.md, round 1): the kernel is
// issue-bound and the async-proxy fence + elect + UBLKCP sequence costs more issue slots per
// warp-step than 4 LDS.128 + 4 STG.128.
template <int OBS_DIM>
__device__ __forceinline__ void emit_obs_rows(float* tile, float* gdst, const EnvState& s, int lane,
                                              int valid, bool active, bool fast) {
  float* const row = tile + lane * OBS_DIM;
  constexpr int kQuads = 32 * OBS_DIM / 4;
  __syncwarp();     // the previous step's read-back of this tile is complete
  if (active) write_obs<OBS_DIM>(row, s);
  if (fast) {       // full warp, 16-byte aligned destination rows: 128-bit read-back + store
    __syncwarp();
    const float4* t4 = reinterpret_cast<const float4*>(tile);
    float4* g4 = reinterpret_cast<float4*>(gdst);
#pragma unroll
    for (int j = lane; j < kQuads; j += 32) st_quad(g4 + j, t4[j]);
    return;
  }
  __syncwarp();
  for (int j = lane; j < valid * OBS_DIM; j += 32) gdst[j] = tile[j];
  __syncwarp();
}

// can every [n,D] row block of this warp take the 128-bit path?  (full warp; base 16-byte aligned;
// consecutive [n,D] slabs keep the alignment when n*D is a multiple of 4 floats)
template <int OBS_DIM>
__device__ __forceinline__ bool emit_fast_ok(const float* base, int64_t warp_base, int64_t n, int valid) {
  return (valid == 32) && ((reinterpret_cast<uintptr_t>(base + warp_base * OBS_DIM) & 15) == 0) &&
         (((n * OBS_DIM) & 3) == 0);
}

// RECORD = true: the "rollout record" output set -- next_obs, reward, done (and the applied action
// when it is generated in-kernel) are all present, nothing else is: no per-step null checks.
// RECORD = false: every output pointer is optional (the VecEnv.step boundary with its info arrays).
//
// Register diet (ncu, round 1: at 64 registers ptxas re-derived thread ids / pointers every step, ~50 of
// 452 warp-instructions per env-step): the thread index is 32-bit (n <= 2^30, checked by the host), the
// per-step output bases are warp-uniform (k * n lives in the uniform datapath) so no per-thread running
// pointers exist, and the episode statistics go straight to shared-memory atomics on the done path.
template <int OBS_DIM, bool RANDOMIZED, bool AUTORESET, int ACT_MODE, bool RECORD>
__global__ void __launch_bounds__(kBlock, kMinBlocks) rollout_kernel(const __grid_constant__ RolloutArgs A) {
  __shared__ __align__(128) float tiles[kWarps][32 * OBS_DIM];
  __shared__ uint32_t blk_stats[3];      // episodes, terminated, length sum of this CTA (<= 256 * K each)
  __shared__ double blk_ret;

  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t warp_base = i - lane;
  const uint32_t n32 = (uint32_t)A.n;
  const bool active = i < n32;
  const int valid = (warp_base >= n32) ? 0 : (int)min(32u, n32 - warp_base);
  float* tile = tiles[warp];
  const EnvParams& P = A.P;

  if (threadIdx.x < 3) blk_stats[threadIdx.x] = 0;
  if (threadIdx.x == 3) blk_ret = 0.0;
  __syncthreads();
  float ret_sum = 0.f;                   // returns of the episodes this thread finished (exact float32 values)

  EnvState s = {};
  if (active) s = load_state(A.state, i);

  if (A.obs0 != nullptr && valid > 0)
    emit_obs_rows<OBS_DIM>(tile, A.obs0 + (size_t)warp_base * OBS_DIM, s, lane, valid, active,
                           emit_fast_ok<OBS_DIM>(A.obs0, warp_base, A.n, valid));

  const bool fast_obs = emit_fast_ok<OBS_DIM>(A.next_obs, warp_base, A.n, valid);
  const bool w_act = RECORD ? (ACT_MODE == 1) : (A.out_actions != nullptr);
  const bool w_rew = RECORD || (A.reward != nullptr);
  const bool w_done = RECORD || (A.done != nullptr);
  const bool w_trunc = !RECORD && (A.truncated != nullptr);
  const bool w_obs = RECORD || (A.next_obs != nullptr);
  const float act_scale = P.motor_max * 5.9604644775390625e-8f;   // exact: a power of two times motor_max
  const size_t n = (size_t)A.n;

  float4 act = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ACT_MODE == 0 && active) act = ld_quad_nc(A.actions + i);
  // in-kernel actions: the Philox block of step k + 1 does not depend on the state, so it is issued one step ahead --
  // its 40-deep dependency chain interleaves with the dynamics of step k instead of preceding them (ILP at 24 warps/SM)
  uint4 wnext = make_uint4(0u, 0u, 0u, 0u);
  if constexpr (ACT_MODE == 1) wnext = env_stream(P.keys, P.env_offset + (uint64_t)i, A.t0, STREAM_ACTION);

  size_t koff = 0;                                   // k * n: uniform, the base of step k in every [K,n,...] output
  for (int k = 0; k < A.K; ++k, koff += n) {
    float4 f = act;
    if constexpr (ACT_MODE == 0) {
      if (active && k + 1 < A.K) act = ld_quad_nc(A.actions + koff + n + i);     // software prefetch of the next quad
    } else {
      const uint4 w = wnext;
      if (k + 1 < A.K) wnext = env_stream(P.keys, P.env_offset + (uint64_t)i, A.t0 + (uint64_t)(k + 1), STREAM_ACTION);
      f = make_float4((float)(w.x >> 8) * act_scale, (float)(w.y >> 8) * act_scale,
                      (float)(w.z >> 8) * act_scale, (float)(w.w >> 8) * act_scale);
    }
    const StepResult r = step_env(s, P, f);
    const bool done = r.crashed || r.timeout;

    if (active) {
      if (w_act) st_quad(A.out_actions + koff + i, f);
      if (w_rew) (A.reward + koff)[i] = r.reward;
      if (w_done) (A.done + koff)[i] = done ? 1 : 0;
      if (w_trunc) (A.truncated + koff)[i] = (r.timeout && !r.crashed) ? 1 : 0;
      if (done) {
        atomicAdd(&blk_stats[0], 1u);
        if (r.crashed) atomicAdd(&blk_stats[1], 1u);
        atomicAdd(&blk_stats[2], (uint32_t)s.ep_len);
        ret_sum += s.ep_ret;
        if constexpr (!RECORD) {
          if (A.terminal_obs != nullptr) write_obs<OBS_DIM>(A.terminal_obs + (koff + i) * OBS_DIM, s);
          if (A.episode_r != nullptr) A.episode_r[koff + i] = s.ep_ret;
          if (A.episode_l != nullptr) A.episode_l[koff + i] = s.ep_len;
        }
        if constexpr (AUTORESET) {
          reset_env<RANDOMIZED>(s, P, P.env_offset + (uint64_t)i);
        } else {
          s.ep_ret = 0.f;   // VecMonitor zeroes its accumulators on done even without a reset
          s.ep_len = 0;
        }
      }
    }
    if (w_obs && valid > 0)
      emit_obs_rows<OBS_DIM>(tile, A.next_obs + (koff + warp_base) * OBS_DIM, s, lane, valid, active, fast_obs);
  }

  if (active) store_state(A.state, i, s);

  // episode statistics: warp shuffle (returns) -> block smem -> one atomic set per CTA into a hashed slot
  if (__ballot_sync(0xffffffffu, ret_sum != 0.f)) {
    double rs = (double)ret_sum;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) rs += __shfl_xor_sync(0xffffffffu, rs, o);
    if (lane == 0) atomicAdd(&blk_ret, rs);
  }
  __syncthreads();
  if (threadIdx.x == 0 && blk_stats[0] != 0) {
    StatSlot* slot = A.stats + (blockIdx.x % kStatSlots);
    atomicAdd(&slot->episodes, (unsigned long long)blk_stats[0]);
    atomicAdd(&slot->terminated, (unsigned long long)blk_stats[1]);
    atomicAdd(&slot->length_sum, (unsigned long long)blk_stats[2]);
    atomicAdd(&slot->return_sum, blk_ret);
  }
}

// ---------------------------------------------------------------------------------------------
// reset (masked) + observation of every row.  drone.py:48-75 / vectorized_drone.py:38-57
// ---------------------------------------------------------------------------------------------
template <int OBS_DIM, bool RANDOMIZED>
__global__ void __launch_bounds__(kBlock) reset_kernel(StatePlanes sp, const __grid_constant__ EnvParams P,
                                                       int64_t n, const uint8_t* mask, float* obs,
                                                       int zero_first) {
  __shared__ __align__(128) float tiles[kWarps][32 * OBS_DIM];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warp_base = (int64_t)blockIdx.x * blockDim.x + warp * 32;
  const int64_t i = warp_base + lane;
  const bool active = i < n;
  const int valid = (int)max((int64_t)0, min((int64_t)32, n - warp_base));
  EnvState s = {};
  if (active) {
    if (!zero_first) s = load_state(sp, i);   // zero_first: the constructor's reset (ep_num 0 -> 1)
    if (zero_first || mask == nullptr || mask[i] != 0) {
      reset_env<RANDOMIZED>(s, P, P.env_offset + (uint64_t)i);
      store_state(sp, i, s);
    }
  }
  if (obs != nullptr && valid > 0)
    emit_obs_rows<OBS_DIM>(tiles[warp], obs + warp_base * OBS_DIM, s, lane, valid, active,
                           emit_fast_ok<OBS_DIM>(obs, warp_base, n, valid));
}

// ---------------------------------------------------------------------------------------------
// SoA views for attribute access / teacher-forced tests (cold path)
// ---------------------------------------------------------------------------------------------
struct StateView {
  float *pos, *vel, *euler, *omega, *target, *ep_ret;
  int32_t *step, *ep_num, *ep_len;
};

static __global__ void get_state_kernel(StatePlanes sp, int64_t n, StateView v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const EnvState s = load_state(sp, i);
  if (v.pos) { v.pos[3 * i] = s.px; v.pos[3 * i + 1] = s.py; v.pos[3 * i + 2] = s.pz; }
  if (v.vel) { v.vel[3 * i] = s.vx; v.vel[3 * i + 1] = s.vy; v.vel[3 * i + 2] = s.vz; }
  if (v.euler) { v.euler[3 * i] = s.roll; v.euler[3 * i + 1] = s.pitch; v.euler[3 * i + 2] = s.yaw; }
  if (v.omega) { v.omega[3 * i] = s.wp; v.omega[3 * i + 1] = s.wq; v.omega[3 * i + 2] = s.wr; }
  if (v.target) { v.target[3 * i] = s.tx; v.target[3 * i + 1] = s.ty; v.target[3 * i + 2] = s.tz; }
  if (v.step) v.step[i] = s.step;
  if (v.ep_num) v.ep_num[i] = s.ep_num;
  if (v.ep_len) v.ep_len[i] = s.ep_len;
  if (v.ep_ret) v.ep_ret[i] = s.ep_ret;
}

static __global__ void set_state_kernel(StatePlanes sp, int64_t n, StateView v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  EnvState s = load_state(sp, i);
  if (v.pos) { s.px = v.pos[3 * i]; s.py = v.pos[3 * i + 1]; s.pz = v.pos[3 * i + 2]; }
  if (v.vel) { s.vx = v.vel[3 * i]; s.vy = v.vel[3 * i + 1]; s.vz = v.vel[3 * i + 2]; }
  if (v.euler) { s.roll = v.euler[3 * i]; s.pitch = v.euler[3 * i + 1]; s.yaw = v.euler[3 * i + 2]; }
  if (v.omega) { s.wp = v.omega[3 * i]; s.wq = v.omega[3 * i + 1]; s.wr = v.omega[3 * i + 2]; }
  if (v.target) { s.tx = v.target[3 * i]; s.ty = v.target[3 * i + 1]; s.tz = v.target[3 * i + 2]; }
  if (v.step) s.step = v.step[i];
  if (v.ep_num) s.ep_num = v.ep_num[i];
  if (v.ep_len) s.ep_len = v.ep_len[i];
  if (v.ep_ret) s.ep_ret = v.ep_ret[i];
  store_state(sp, i, s);
}

}  // namespace dronecu
