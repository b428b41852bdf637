// Shared pieces of the PPO kernels: flat parameter layout of the SB3-default MlpPolicy
// (pi: 15-64-64-4, vf: 15-64-64-1, tanh, state-independent log_std; SURVEY.md section 8a row P --
// the reference only *calls* it: /root/reference/train.py:36-43), fast tanh, Box-Muller noise.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "philox.cuh"

namespace dronecu {

constexpr int kObs = 15, kHid = 64, kAct = 4;
// flat float32 vector, torch.nn.Linear [out,in] row-major blocks (oracle/ppo_oracle.py SHAPES)
constexpr int O_PI_W1 = 0, O_PI_B1 = 960, O_PI_W2 = 1024, O_PI_B2 = 5120, O_PI_W3 = 5184, O_PI_B3 = 5440;
constexpr int O_VF_W1 = 5444, O_VF_B1 = 6404, O_VF_W2 = 6468, O_VF_B2 = 10564, O_VF_W3 = 10628, O_VF_B3 = 10692;
constexpr int O_LOGSTD = 10693, kParams = 10697;
constexpr int kTowerStride = O_VF_W1 - O_PI_W1;   // 5444: vf block = pi block shifted (heads differ in size)

constexpr float kHalfLog2Pi = 0.91893853320467274178f;   // 0.5 * ln(2 pi)

// Packed float32 pairs (sm_100: FFMA2 / FMUL2 / FADD2 work on an aligned 64-bit register pair, and one operand may be a
// scalar that is broadcast to both halves).  Each half is the IEEE fmaf / * / + it replaces -- results are bit-identical --
// but a pair costs ONE issue slot: the fp32 towers and the elementwise phases of the tensor-core kernels are bound by
// instruction issue (DESIGN.md section 4), not by the FMA pipe; the scalar forms measured slower.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
// (d0, d1) = (a0, a1) * (b0, b1) + (d0, d1)
__device__ __forceinline__ void fma2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pk2(a0, a1)), "l"(pk2(b0, b1)), "l"(pk2(d0, d1)));
  upk2(d, d0, d1);
}
// acc[0..3] = w * s + acc[0..3]: the inner step of every fp32 tower (four output units per LDS.128 of weights)
__device__ __forceinline__ void fma4s(float* acc, const float4 w, const float s) {
  fma2(acc[0], acc[1], w.x, w.y, s, s);
  fma2(acc[2], acc[3], w.z, w.w, s, s);
}
// (a, b) <- 1 - (a, b)^2
__device__ __forceinline__ void one_minus_sq2(float a, float b, float& ra, float& rb) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(pk2(-a, -b)), "l"(pk2(a, b)), "l"(pk2(1.f, 1.f)));
  upk2(d, ra, rb);
}
__device__ __forceinline__ void mul2(float& a, float& b, float x, float y) {           // (a, b) *= (x, y)
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk2(a, b)), "l"(pk2(x, y)));
  upk2(d, a, b);
}
__device__ __forceinline__ void add2(float& a, float& b, float x, float y) {           // (a, b) += (x, y)
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk2(a, b)), "l"(pk2(x, y)));
  upk2(d, a, b);
}

// tanh(x) = 1 - 2 / (exp(2x) + 1) with the MUFU ex2 / rcp approximations: absolute error of a few
// 1e-7 over the whole range (saturates cleanly to +-1), 2 MUFU + 3 FMA-pipe ops instead of the
// ~25-instruction tanhf.  The PPO parity tolerance (tests/test_gpu_ppo.py) is stated against it.
__device__ __forceinline__ float tanh_fast(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.88539008177792681472f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}

// four standard normals from the NOISE stream (oracle/philox.py noise_normals):
// z0 = r(u0) cos(2 pi u1), z1 = r(u0) sin(2 pi u1), z2 = r(u2) cos(2 pi u3), z3 = r(u2) sin(2 pi u3),
// r(u) = sqrt(-2 ln(u + 2^-24))
__device__ __forceinline__ float4 noise_normals(const PhiloxKeys& keys, uint64_t env_id, uint64_t t) {
  const uint4 w = env_stream(keys, env_id, t, STREAM_NOISE);
  const float r0 = sqrtf(-2.0f * logf(u01(w.x) + 5.9604644775390625e-8f));
  const float r1 = sqrtf(-2.0f * logf(u01(w.z) + 5.9604644775390625e-8f));
  float s0, c0, s1, c1;
  sincospif(2.0f * u01(w.y), &s0, &c0);
  sincospif(2.0f * u01(w.w), &s1, &c1);
  return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}

}  // namespace dronecu
