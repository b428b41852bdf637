// Policy / value MLP forward on the 5th-generation tensor cores (tcgen05 + TMEM), hand-written PTX.
//
// Tile = 128 envs = the 128 threads of a CTA = the 128 lanes of TMEM: thread i owns env i, TMEM lane i
// and row i of every accumulator.  Per forward, for each tower t in (pi, vf):
//   X  [128 x 16]  (obs | 1.0)     -> tcgen05.st into TMEM columns (A operand, K-major, tf32)
//   D1 [128 x 64]  = X . W1t^T      bias folded in through the ones column       (2 MMAs, K = 8 each)
//   H1 = tanh(D1)                   tcgen05.ld -> MUFU tanh -> tcgen05.st back IN PLACE (A operand of L2)
//   D2 [128 x 64]  = H1 . W2t^T     A from TMEM, B from shared memory              (8 MMAs, K = 8 each)
//   H2 = tanh(D2 + b2), head        tcgen05.ld -> registers; the 4 (or 1) head outputs are 256 (64) FMAs
//                                   per env on the CUDA cores (N = 4 is below the MMA's minimum N of 16)
// Weights (B operands) sit in shared memory in the canonical no-swizzle K-major UMMA layout
// (8-row x 16-byte core matrices; LBO = 128 B between K chunks, SBO = K*32 B between 8-row groups),
// rounded once to tf32.  TMEM budget: 128 columns per CTA (D1/H1 64 | D2 64, X aliases D2), so FOUR
// CTAs share an SM's 512 columns: the MUFU-bound tanh work of one CTA runs under the MMA / mbarrier
// latency of the others (round-1 ncu: the 256-column, both-towers-at-once variant left the SM at 40 %
// issue utilisation with 8 resident warps).
// Precision: tf32 products (10-bit mantissa), fp32 accumulation, tanh.approx.f32 (2^-11): outputs agree
// with the fp32 CUDA-core path to ~2e-3; that path stays the parity reference (tests/test_gpu_ppo.py).  The
// per-element bound is derived in oracle/tc_bound.py.
// Non-finite rows: +-inf, and values that round to inf in tf32, behave as in float32 torch (the first tanh
// saturates).  A row holding NaN gives an unspecified, possibly finite, output: tanh.approx returns the canonical
// NaN 0x7fffffff, which to_tf32_fast wraps to -0, so the NaN does not reach layer 2 (the fp32 path returns NaN).
// The env can emit such rows (body rates that overflow never end the episode: the crash test looks at the position).
#pragma once
#include "ppo_common.cuh"

namespace dronecu {
namespace tc {

constexpr int kTile = 128;          // envs per CTA == threads per CTA == TMEM lanes
constexpr int kTmemCols = 128;
constexpr int kColD1 = 0;           // D1 / H1 : columns [0,64)
constexpr int kColD2 = 64;          // D2      : columns [64,128)
constexpr int kColX = 64;           // X       : columns [64,80), dead before D2 is written
constexpr int kK1 = 16, kN1 = 64, kK2 = 64, kN2 = 64;

struct alignas(128) Smem {
  float W1[2][kN1 * kK1];           // canonical UMMA layout per tower, k = 15 holds the bias
  float W2[2][kN2 * kK2];           // canonical UMMA layout per tower
  float b2[2][kHid];
  float W3piT[kHid][kAct];
  float W3vf[kHid];
  float b3pi[kAct];
  float b3vf, pad0[3];
  float log_std[kAct];
  alignas(8) unsigned long long mbar[2];
  uint32_t tmem_base, pad1[3];
};

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// round-to-nearest tf32 for values that are never inf: the tensor core ignores the low 13 mantissa
// bits, so adding half an ulp of tf32 is all it takes (cvt.rna.tf32 compiles to 3 instructions)
__device__ __forceinline__ float to_tf32_fast(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

__device__ __forceinline__ float tanh_mufu(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// tanh of a 16-wide chunk in place on the MUFU pipe.  Evaluating a share of the activations as a packed odd polynomial on the
// FMA pipe instead measured no faster (profiles/README.md): the MUFU pipe is not what a warp waits for, and the polynomial's
// 7 issue slots per activation (against 1) push the rollout kernel to the issue limit.
__device__ __forceinline__ void tanh_chunk16(float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = tanh_mufu(v[i]);
}

// byte offset of element (n, k) of an [N x K] K-major operand in the canonical no-swizzle layout
__device__ __forceinline__ int umma_off(int n, int k, int K) {
  return (((n >> 3) * (K >> 2) + (k >> 2)) << 5) + ((n & 7) << 2) + (k & 3);   // in floats
}

__device__ __forceinline__ uint64_t make_desc(const void* smem_ptr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr(smem_ptr) >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;          // descriptor version: Blackwell
  return d;                        // layout type 0 = no swizzle, base offset 0
}

__device__ __forceinline__ constexpr uint32_t make_idesc(int M, int N) {
  // c = F32 (1 @4), a = b = TF32 (2 @7, 2 @10), both K-major, N >> 3 @17, M >> 4 @24
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
      :: "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}

__device__ __forceinline__ void mma_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_addr(bar)) : "memory");
}

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  const uint32_t addr = smem_addr(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
  } while (!done);
}

__device__ __forceinline__ uint32_t elect_one() {       // one lane of the (converged) warp; tells ptxas the region is single-threaded
  uint32_t pred = 0;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
  return pred;
}

__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 bit, 16 consecutive columns <-> 16 registers per thread
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  wait_ld();
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
         "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
         "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])),
         "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
         "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])),
         "r"(__float_as_uint(v[15])) : "memory");
}

// One-time CTA setup: weights -> shared memory (canonical layout, tf32-rounded), mbarriers, TMEM.
__device__ __forceinline__ void setup(Smem& S, const float* __restrict__ theta) {
  const int tid = threadIdx.x;
  for (int idx = tid; idx < 2 * kN1 * kK1; idx += blockDim.x) {
    const int t = idx / (kN1 * kK1), q = idx % (kN1 * kK1);
    const int j = q / kK1, k = q % kK1;
    const int wbase = t ? O_VF_W1 : O_PI_W1, bbase = t ? O_VF_B1 : O_PI_B1;
    const float v = (k < kObs) ? theta[wbase + j * kObs + k] : theta[bbase + j];
    S.W1[t][umma_off(j, k, kK1)] = to_tf32(v);
  }
  for (int idx = tid; idx < 2 * kN2 * kK2; idx += blockDim.x) {
    const int t = idx / (kN2 * kK2), q = idx % (kN2 * kK2);
    const int n = q / kK2, k = q % kK2;
    S.W2[t][umma_off(n, k, kK2)] = to_tf32(theta[(t ? O_VF_W2 : O_PI_W2) + q]);
  }
  for (int idx = tid; idx < 2 * kHid; idx += blockDim.x)
    S.b2[idx >> 6][idx & 63] = theta[((idx >> 6) ? O_VF_B2 : O_PI_B2) + (idx & 63)];
  for (int idx = tid; idx < kAct * kHid; idx += blockDim.x) S.W3piT[idx % kHid][idx / kHid] = theta[O_PI_W3 + idx];
  for (int idx = tid; idx < kHid; idx += blockDim.x) S.W3vf[idx] = theta[O_VF_W3 + idx];
  if (tid < kAct) { S.b3pi[tid] = theta[O_PI_B3 + tid]; S.log_std[tid] = theta[O_LOGSTD + tid]; }
  if (tid == 0) {
    S.b3vf = theta[O_VF_B3];
    mbar_init(&S.mbar[0], 1);
    mbar_init(&S.mbar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (tid < 32) {                                      // warp 0 allocates (and later frees) the TMEM columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_addr(&S.tmem_base)), "r"((uint32_t)kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // generic-proxy writes of the weights must be visible to the tensor core's (async proxy) smem reads
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  fence_before();
  __syncthreads();
  fence_after();
}

__device__ __forceinline__ void teardown(Smem& S) {
  fence_before();
  __syncthreads();
  if (threadIdx.x < 32)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(S.tmem_base), "r"((uint32_t)kTmemCols) : "memory");
}

// One tower for the CTA's 128 envs; every thread of the CTA must call it (CTA-wide barriers inside).
// xv: this thread's A row of layer 1 (15 observations, tf32-rounded, and the constant 1).
template <int NOUT>
__device__ __forceinline__ void tower(Smem& S, const int t, const float (&xv)[16], uint32_t& phase, float (&out)[NOUT],
                                      float* dbg1, float* dbg2) {
  const uint32_t lane_base = ((threadIdx.x >> 5) & 3) * 32;
  const uint32_t tbase = S.tmem_base + (lane_base << 16);

  tmem_st16(tbase + kColX, xv);
  wait_st();
  fence_before();
  __syncthreads();
  if (threadIdx.x < 32 && elect_one()) {       // elect.sync: ptxas keeps the descriptors uniform (no per-MMA waterfall loop)
    fence_after();
    constexpr uint32_t idesc1 = make_idesc(kTile, kN1);
#pragma unroll
    for (int s = 0; s < kK1 / 8; ++s) {
      const uint64_t b = make_desc(reinterpret_cast<const char*>(S.W1[t]) + s * 256, 128, kK1 * 32);
      mma_tf32_ts(S.tmem_base + kColD1, S.tmem_base + kColX + 8 * s, b, idesc1, s > 0);
    }
    mma_commit(&S.mbar[0]);
  }
  mbar_wait(&S.mbar[0], phase);
  fence_after();

  // H1 = tanh(D1), in place: becomes the A operand of layer 2
#pragma unroll
  for (int c = 0; c < kN1 / 16; ++c) {
    float v[16];
    tmem_ld16(tbase + kColD1 + 16 * c, v);
    if (dbg1) {
#pragma unroll
      for (int i = 0; i < 16; ++i) dbg1[16 * c + i] = v[i];
    }
    tanh_chunk16(v);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = to_tf32_fast(v[i]);
    tmem_st16(tbase + kColD1 + 16 * c, v);
  }
  wait_st();
  fence_before();
  __syncthreads();
  if (threadIdx.x < 32 && elect_one()) {
    fence_after();
    constexpr uint32_t idesc2 = make_idesc(kTile, kN2);
#pragma unroll
    for (int s = 0; s < kK2 / 8; ++s) {
      const uint64_t b = make_desc(reinterpret_cast<const char*>(S.W2[t]) + s * 256, 128, kK2 * 32);
      mma_tf32_ts(S.tmem_base + kColD2, S.tmem_base + kColD1 + 8 * s, b, idesc2, s > 0);
    }
    mma_commit(&S.mbar[1]);
  }
  mbar_wait(&S.mbar[1], phase);
  fence_after();
  phase ^= 1;

  // H2 = tanh(D2 + b2) and the head on the CUDA cores
  if constexpr (NOUT == kAct) {
#pragma unroll
    for (int o = 0; o < kAct; ++o) out[o] = S.b3pi[o];
  } else {
    out[0] = S.b3vf;
  }
  float odd = 0.f;
#pragma unroll
  for (int c = 0; c < kN2 / 16; ++c) {
    float v[16];
    tmem_ld16(tbase + kColD2 + 16 * c, v);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 b = reinterpret_cast<const float4*>(S.b2[t] + 16 * c)[q];
      add2(v[4 * q], v[4 * q + 1], b.x, b.y);
      add2(v[4 * q + 2], v[4 * q + 3], b.z, b.w);
    }
    if (dbg2) {
#pragma unroll
      for (int i = 0; i < 16; ++i) dbg2[16 * c + i] = v[i];
    }
    tanh_chunk16(v);
    if constexpr (NOUT == kAct) {
#pragma unroll
      for (int i = 0; i < 16; ++i) fma4s(out, reinterpret_cast<const float4*>(S.W3piT[16 * c + i])[0], v[i]);
    } else {                    // one output: even / odd hidden units in the two halves of a packed accumulator
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 w = reinterpret_cast<const float4*>(S.W3vf + 16 * c)[q];
        fma2(out[0], odd, w.x, w.y, v[4 * q], v[4 * q + 1]);
        fma2(out[0], odd, w.z, w.w, v[4 * q + 2], v[4 * q + 3]);
      }
    }
  }
  if constexpr (NOUT != kAct) out[0] += odd;
  // the next tower's X store aliases D2: a thread only ever touches its own lane, and the MMA that
  // wrote D2 has completed (mbarrier), so no further barrier is needed here.
}

// Forward of both towers.  `phase` is the running mbarrier parity (0 before the first call).
// dbg1 / dbg2 (nullable): this thread's 128 pre-activations (pi 0..63 | vf 64..127) of layer 1 / 2.
__device__ __forceinline__ void forward(Smem& S, const float (&x)[kObs], uint32_t& phase, float (&mean)[kAct],
                                        float& value, float* dbg1 = nullptr, float* dbg2 = nullptr) {
  float xv[16];
#pragma unroll
  for (int i = 0; i < kObs; ++i) xv[i] = to_tf32_fast(x[i]);
  xv[15] = 1.0f;
  float v1[1];
  tower<kAct>(S, 0, xv, phase, mean, dbg1, dbg2);
  tower<1>(S, 1, xv, phase, v1, dbg1 ? dbg1 + kHid : nullptr, dbg2 ? dbg2 + kHid : nullptr);
  value = v1[0];
}

// policy tower only (evaluation: ppo_eval.cuh); the same MMAs on the same operands as the pi tower of forward()
__device__ __forceinline__ void forward_policy(Smem& S, const float (&x)[kObs], uint32_t& phase, float (&mean)[kAct]) {
  float xv[16];
#pragma unroll
  for (int i = 0; i < kObs; ++i) xv[i] = to_tf32_fast(x[i]);
  xv[15] = 1.0f;
  tower<kAct>(S, 0, xv, phase, mean, nullptr, nullptr);
}

// value tower only (the GAE bootstrap after the last step)
__device__ __forceinline__ float forward_value(Smem& S, const float (&x)[kObs], uint32_t& phase) {
  float xv[16], v1[1];
#pragma unroll
  for (int i = 0; i < kObs; ++i) xv[i] = to_tf32_fast(x[i]);
  xv[15] = 1.0f;
  tower<1>(S, 1, xv, phase, v1, nullptr, nullptr);
  return v1[0];
}

}  // namespace tc
}  // namespace dronecu
