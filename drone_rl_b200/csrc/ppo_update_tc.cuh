// PPO minibatch gradient on the 5th-generation tensor cores (tcgen05 + TMEM, tf32 operands, fp32
// accumulation): same contract as ppo_grad_kernel (ppo_update.cuh), i.e. what SB3's PPO.train() does
// per minibatch (SURVEY.md appendix C; call site /root/reference/train.py:63-68) -- "parity unpinned".
//
// Grid (x, 2): blockIdx.y selects the tower (0 = policy, 1 = value) -- the towers share nothing but the
// observation.  One CTA per SM: two COMPUTE warpgroups (a warpgroup owns one tile of 128 samples at a time:
// thread i <-> sample i <-> TMEM lane i) and two MMA-ISSUER warps, one per warpgroup (v2; in v1 the
// warpgroup's first thread issued the MMAs itself: ncu showed that thread executing ~1300 descriptor /
// issue instructions per tile on the critical path of its warpgroup, and 640 CUDA-core FMAs per sample for
// the two four-wide head products).  Compute threads hand operands over through a 128-arrival mbarrier
// (`full`), the issuer answers with tcgen05.commit on `done`.  EVERY matrix product is a tcgen05.mma:
//   S1  D1  [128 x 64]  = X . W1^T        A = X in TMEM (K = 16: 15 observations + a ones column carrying b1)
//   S2  D2  [128 x 64]  = H1 . W2^T       A = H1 = tanh(D1), written back to TMEM in place
//   S3  D3  [128 x 16]  = H2 . W3p^T      head outputs (4 policy means or 1 value; N padded to 16)
//   S4  dW3 [ 64 x  8] += H2^T . G        G = (dL/d head output (4) | live | 0 0 0) per sample
//       dH2 [128 x 64]  = G . W3k         A = G in TMEM (K = 8), the gradient entering tanh'(layer 2)
//   S5  dH1 [128 x 64]  = dZ2 . W2        A = dZ2 in TMEM (over H2), B = a transposed copy of W2
//       dW2 [ 64 x 64] += dZ2^T . H1 ,    db2 [64 x 8] += dZ2^T . G   (column 4 = bias gradient)
//   S6  dW1 [ 64 x 16] += dZ1^T . X       (column 15, the ones column, = db1)
// The weight-gradient products reduce over the SAMPLES, so their accumulators (M = 64: 16 TMEM lanes
// per subpartition) stay resident in TMEM for the whole life of the CTA and are read out once at the
// end.  TMEM per warpgroup: P 64 | Q 64 | dW2 64 | dW1 16 | dW3 8 | db2 8 | D3 16 | G 8 = 248 of its 256 columns.
// The CUDA cores keep only the elementwise work: tanh (MUFU), tanh' = 1 - h^2, the loss gradient at the
// head, tf32 rounding, and the staging stores.  Per-sample scalars (log_std gradient, b3 gradient, loss
// statistics) accumulate in registers over the tiles of a thread and are reduced once, in a fixed order.
// The next tile's rows are gathered (random minibatch order) while the current tile computes.
//
// Operand staging for the weight gradients (K = samples).  The "transposed" operands H2^T, dZ2^T, H1,
// dZ1^T are MN-major: a thread writes its sample's 64-float row once, as two 128-byte rows (32 features
// each), and the tensor core reads the buffer as [64 features] x [K = 128 samples].  For tf32 the only
// MN-major shared-memory layout the hardware accepts is SWIZZLE_128B_BASE32B (cute
// Layout_MN_SW128_32B_Atom: atoms of 4 K-rows x 128 bytes, 32-byte chunks XOR-ed with the row index;
// probed on the B200: the 16-byte-base 128B swizzle and the no-swizzle MN-major forms return zeros).
// The narrow operands X (16 wide) and G (8 wide) are scattered transposed into a K-major no-swizzle
// tile whose K-chunk stride is padded to 144 bytes so that the 32 lanes of a warp hit 32 banks.
#pragma once
#include "ppo_update.cuh"
#include "tc_mlp.cuh"

// -DDRONECU_TC_TIMING=1: thread 0 of warpgroup 0 (and its issuer) of CTA (0, 0) log clock64() at every hand-over
// point of their first 16 tiles into the debug buffer (as int64; compute at [0, 16*16), issuer at [1024, ...)).
#ifndef DRONECU_TC_TIMING
#define DRONECU_TC_TIMING 0
#endif
#if DRONECU_TC_TIMING
#define TSTAMP(buf, it, k) do { if ((buf) != nullptr && (it) < 16) (buf)[(it) * 16 + (k)] = clock64(); } while (0)
#else
#define TSTAMP(buf, it, k) do { (void)(buf); } while (0)
#endif

namespace dronecu {
namespace tcu {

using tc::elect_one;
using tc::fence_after;
using tc::fence_before;
using tc::mbar_init;
using tc::mbar_wait;
using tc::mma_commit;
using tc::mma_tf32_ts;
using tc::smem_addr;
using tc::tanh_mufu;
using tc::to_tf32;
using tc::to_tf32_fast;
using tc::umma_off;
using tc::wait_st;

constexpr int kWG = 2;                       // compute warpgroups (= sample tiles in flight) per CTA
constexpr int kComputeThreads = 128 * kWG;
constexpr int kThreads = kComputeThreads + 32 * kWG;   // + one MMA-issuing warp per warpgroup
constexpr int kHalfBytes = 128 * 128;        // one 32-feature half of a [128 samples x 64] fp32 operand buffer
constexpr int kColP = 0, kColQ = 64;         // P: D1 -> H1 (A of S2) -> dH2 -> dH1 ;  Q: X (A of S1) -> D2 -> H2 (A of S3) -> dZ2 (A of S5)
constexpr int kAccW2 = 128, kAccW1 = 192, kAccW3 = 208, kAccB2 = 216, kColD3 = 224, kColGA = 240;
constexpr int kColsPerWG = 256;
constexpr int kTmemCols = kColsPerWG * kWG;  // 512
constexpr int kNS = 12;                      // per-thread scalar accumulators
// K-major no-swizzle tile of the narrow operands: rows 0..15 = X^T (x0..x14, 1), rows 16..23 = G^T
constexpr int kXaLbo = 144;                  // bytes between consecutive 4-sample K chunks (128 + 16 padding)
constexpr int kXaSbo = 32 * kXaLbo;          // bytes between 8-row groups (128 samples = 32 chunks)
constexpr int kXaBytes = 3 * kXaSbo;         // 13,824
// K-major no-swizzle [128 samples x 16] tile of X (A operand of S1): 4 K chunks of 16 B per 8-row group, chunk stride 144 B
constexpr int kXsLbo = 144;
constexpr int kXsSbo = 4 * kXsLbo;           // 576 B between 8-row groups
constexpr int kXsBytes = 16 * kXsSbo;        // 9,216

struct alignas(1024) Smem {
  unsigned char bufA[kWG][2 * kHalfBytes];   // H1, later dZ1         (MN-major, SWIZZLE_128B_BASE32B)
  unsigned char bufB[kWG][2 * kHalfBytes];   // H2, later dZ2
  unsigned char XA[kWG][kXaBytes];
  unsigned char XS[kWG][kXsBytes];           // X as the A operand of S1: K-major [128 samples][16], K-chunk stride padded (bank spread)
  float W1[kHid * 16];                       // this CTA's tower.  canonical no-swizzle K-major [out][k], k = 15 holds b1
  float W2[kHid * kHid];                     // canonical no-swizzle K-major [out][in]   (B of S2)
  float W2T[kHid * kHid];                    // canonical no-swizzle K-major [in][out]   (B of S5: dH1 = dZ2 . W2)
  float W3p[16 * kHid];                      // K-major [N = 16][K = 64]: rows 0..3 (policy) / 0 (value) = W3, rest 0 (B of S3)
  float W3k[kHid * 8];                       // K-major [N = 64][K = 8]: W3k[j][o] = W3[o][j], columns >= 4 (1) zero (B of S4's dH2)
  float b2[kHid];
  float b3[kAct];
  float log_std[kAct];
  float wsum[kWG][4][kNS];                   // per-warp partial sums of the per-thread scalar accumulators
  alignas(8) unsigned long long full[kWG];   // 128 arrivals: the warpgroup's operands of the next MMA step are staged
  alignas(8) unsigned long long done[kWG];   // tcgen05.commit: that MMA step has completed
  uint32_t tmem_base, pad1[3];
};

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start >> 4 @0, LBO >> 4 @16, SBO >> 4 @32,
// version 1 @46, layout type @61 (0 = no swizzle, 1 = 128-byte swizzle with 32-byte base)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
// MN-major [64 features x 8 samples] slice s of an activation buffer: MN atoms (32 features) 16 KB apart, K atoms (4 rows) 512 B apart
__device__ __forceinline__ uint64_t desc_mn(uint32_t buf, int s) { return make_desc(buf + 1024 * s, kHalfBytes, 512, 1); }
// K-major slice s (8 samples) of the narrow tile, starting at row group g (0: X rows 0..15, 2: G rows 16..23)
__device__ __forceinline__ uint64_t desc_xa(uint32_t xa, int g, int s) { return make_desc(xa + g * kXaSbo + 2 * kXaLbo * s, kXaLbo, kXaSbo, 0); }
// canonical no-swizzle K-major weight tile [N x K]: slice s of 8 k
__device__ __forceinline__ uint64_t desc_w(uint32_t w, int K, int s) { return make_desc(w + 256 * s, 128, K * 32, 0); }

// instruction descriptor: D = f32, A = B = tf32, major-ness bits 15 / 16 (1 = MN-major), N >> 3 @17, M >> 4 @24
__host__ __device__ constexpr uint32_t idesc(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t id, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(id), "r"(accumulate) : "memory");
}

__device__ __forceinline__ void wg_barrier(int wg) { asm volatile("bar.sync %0, 128;" :: "r"(wg + 1) : "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_addr(bar)) : "memory");
}

// TMEM <-> registers, 32 lanes x 32 bit.  No "memory" clobber: TMEM is not C++ memory, and the volatile asm
// statements keep their order among themselves (waits, fences, arrives), so ptxas may move shared-memory
// loads / stores of a phase across them.  The loads are asynchronous: ld16_issue starts one, ld_fence waits for
// every outstanding load of the thread and ties the destination registers to the wait (so that the compiler
// cannot move a consumer above it) -- a second load may be in flight while the first chunk is processed.
__device__ __forceinline__ void ld16_issue(uint32_t taddr, float (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]),
        "=f"(v[8]), "=f"(v[9]), "=f"(v[10]), "=f"(v[11]), "=f"(v[12]), "=f"(v[13]), "=f"(v[14]), "=f"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void ld_fence(float (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7]),
                 "+f"(v[8]), "+f"(v[9]), "+f"(v[10]), "+f"(v[11]), "+f"(v[12]), "+f"(v[13]), "+f"(v[14]), "+f"(v[15])
               :);
}
__device__ __forceinline__ void st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      :: "r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]),
         "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]));
}
__device__ __forceinline__ void st8(uint32_t taddr, const float (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]));
}
__device__ __forceinline__ void ld4(uint32_t taddr, float (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];\n\ttcgen05.wait::ld.sync.aligned;"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(taddr));
}

// float4 number c4 (features 4 c4 .. 4 c4 + 3, c4 in 0..15) of sample row r in an MN-major activation buffer
__device__ __forceinline__ float4* mn_quad(unsigned char* buf, int r, int c4) {
  return reinterpret_cast<float4*>(buf + (c4 >> 3) * kHalfBytes + r * 128 + ((((c4 >> 1) & 3) ^ (r & 3)) << 5) + ((c4 & 1) << 4));
}
// element (row n, sample s) of the narrow K-major tile
__device__ __forceinline__ float* xa_elem(unsigned char* xa, int n, int s) {
  return reinterpret_cast<float*>(xa + (n >> 3) * kXaSbo + (s >> 2) * kXaLbo + ((n & 7) << 4) + ((s & 3) << 2));
}

// element (sample m, feature k) of the X tile
__device__ __forceinline__ float* xs_elem(unsigned char* xs, int m, int k) {
  return reinterpret_cast<float*>(xs + (m >> 3) * kXsSbo + (k >> 2) * kXsLbo + ((m & 7) << 4) + ((k & 3) << 2));
}

// a compute thread's staged operands (generic-proxy smem writes, tcgen05.st) are handed to the issuer
__device__ __forceinline__ void hand_over(unsigned long long* full) {
  proxy_fence();
  fence_before();
  mbar_arrive(full);
}

__device__ __forceinline__ void setup(Smem& S, const float* __restrict__ theta, const int tw) {
  const int tid = threadIdx.x;
  const int oW1 = tw ? O_VF_W1 : O_PI_W1, oB1 = tw ? O_VF_B1 : O_PI_B1, oW2 = tw ? O_VF_W2 : O_PI_W2;
  const int nout = tw ? 1 : kAct, oW3 = tw ? O_VF_W3 : O_PI_W3;
  for (int q = tid; q < kHid * 16; q += kThreads) {
    const int j = q / 16, k = q % 16;
    S.W1[umma_off(j, k, 16)] = to_tf32((k < kObs) ? theta[oW1 + j * kObs + k] : theta[oB1 + j]);
  }
  for (int q = tid; q < kHid * kHid; q += kThreads) {
    const int j = q / kHid, i = q % kHid;
    const float v = to_tf32(theta[oW2 + q]);
    S.W2[umma_off(j, i, kHid)] = v;
    S.W2T[umma_off(i, j, kHid)] = v;
  }
  for (int q = tid; q < 16 * kHid; q += kThreads) {
    const int o = q / kHid, j = q % kHid;
    S.W3p[umma_off(o, j, kHid)] = (o < nout) ? to_tf32(theta[oW3 + o * kHid + j]) : 0.f;
  }
  for (int q = tid; q < kHid * 8; q += kThreads) {
    const int j = q / 8, o = q % 8;
    S.W3k[umma_off(j, o, 8)] = (o < nout) ? to_tf32(theta[oW3 + o * kHid + j]) : 0.f;
  }
  for (int q = tid; q < kHid; q += kThreads) S.b2[q] = theta[(tw ? O_VF_B2 : O_PI_B2) + q];
  if (tid < kAct) {
    S.b3[tid] = tw ? (tid == 0 ? theta[O_VF_B3] : 0.f) : theta[O_PI_B3 + tid];
    S.log_std[tid] = theta[O_LOGSTD + tid];
  }
  if (tid == 0) {
    for (int w = 0; w < kWG; ++w) { mbar_init(&S.full[w], 128); mbar_init(&S.done[w], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_addr(&S.tmem_base)), "r"((uint32_t)kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  proxy_fence();
  fence_before();
  __syncthreads();
  fence_after();
}

// ---------------------------------------------------------------------------------------------------------
// MMA issuer warp of one warpgroup: six steps per tile, each answered with a commit on `done`.  The whole warp
// waits on `full`; ONE elected lane issues (inside elect.sync ptxas keeps descriptors in uniform registers
// without a per-instruction waterfall loop -- v2.0 measured ~65 cycles per MMA issued from `if (lane == 0)`).
// Descriptors are built once; a slice s of 8 along K only bumps the 14-bit start-address field.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void issuer(Smem& S, const int wg, const int64_t my_tiles, long long* tlog) {
  unsigned long long* const full = &S.full[wg];
  unsigned long long* const done = &S.done[wg];
  const uint64_t dA = desc_mn(smem_addr(S.bufA[wg]), 0), dB = desc_mn(smem_addr(S.bufB[wg]), 0);
  const uint64_t dXx = desc_xa(smem_addr(S.XA[wg]), 0, 0), dXg = desc_xa(smem_addr(S.XA[wg]), 2, 0);
  const uint64_t dXs = make_desc(smem_addr(S.XS[wg]), kXsLbo, kXsSbo, 0);
  const uint64_t dW1 = desc_w(smem_addr(S.W1), 16, 0), dW2 = desc_w(smem_addr(S.W2), kHid, 0);
  const uint64_t dW2T = desc_w(smem_addr(S.W2T), kHid, 0), dW3p = desc_w(smem_addr(S.W3p), kHid, 0);
  const uint64_t dW3k = desc_w(smem_addr(S.W3k), 8, 0);
  constexpr uint64_t kMn = 1024 >> 4, kXa = (2 * kXaLbo) >> 4, kW = 256 >> 4, kXs = (2 * kXsLbo) >> 4;   // per-slice bumps
  const uint32_t tmem = S.tmem_base + wg * kColsPerWG;
  uint32_t ph = 0;
  for (int64_t it = 0; it < my_tiles; ++it) {
    const uint32_t acc = it > 0;
    // S1: D1 = X . W1^T  (A = X tile in shared memory)
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 0);
    if (elect_one()) {
#pragma unroll
      for (int s = 0; s < 2; ++s) mma_ss(tmem + kColP, dXs + kXs * s, dW1 + kW * s, idesc(128, 64, 0, 0), s > 0);
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 1);
    // S2: D2 = H1 . W2^T
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 2);
    if (elect_one()) {
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_tf32_ts(tmem + kColQ, tmem + kColP + 8 * s, dW2 + kW * s, idesc(128, 64, 0, 0), s > 0);
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 3);
    // S3: D3 = H2 . W3p^T
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 4);
    if (elect_one()) {
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_tf32_ts(tmem + kColD3, tmem + kColQ + 8 * s, dW3p + kW * s, idesc(128, 16, 0, 0), s > 0);
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 5);
    // S4: dH2 = G . W3k ; dW3 += H2^T . G
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 6);
    if (elect_one()) {
      mma_tf32_ts(tmem + kColP, tmem + kColGA, dW3k, idesc(128, 64, 0, 0), 0);
#pragma unroll
      for (int s = 0; s < 16; ++s) mma_ss(tmem + kAccW3, dB + kMn * s, dXg + kXa * s, idesc(64, 8, 1, 0), acc | (s > 0));
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 7);
    // S5: dH1 = dZ2 . W2 ; dW2 += dZ2^T . H1 ; db2 += dZ2^T . G(ones column)
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 8);
    if (elect_one()) {
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_tf32_ts(tmem + kColP, tmem + kColQ + 8 * s, dW2T + kW * s, idesc(128, 64, 0, 0), s > 0);
#pragma unroll
      for (int s = 0; s < 16; ++s) mma_ss(tmem + kAccW2, dB + kMn * s, dA + kMn * s, idesc(64, 64, 1, 1), acc | (s > 0));
#pragma unroll
      for (int s = 0; s < 16; ++s) mma_ss(tmem + kAccB2, dB + kMn * s, dXg + kXa * s, idesc(64, 8, 1, 0), acc | (s > 0));
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 9);
    // S6: dW1 (+ db1 in column 15) += dZ1^T . X
    mbar_wait(full, ph); ph ^= 1; fence_after();
    TSTAMP(tlog, it, 10);
    if (elect_one()) {
#pragma unroll
      for (int s = 0; s < 16; ++s) mma_ss(tmem + kAccW1, dA + kMn * s, dXx + kXa * s, idesc(64, 16, 1, 0), acc | (s > 0));
      mma_commit(done);
    }
    __syncwarp();
    TSTAMP(tlog, it, 11);
  }
}

// inputs of one sample row, gathered through the minibatch index
struct RowIn {
  float xe[16];        // element (lane & 15) of the rows of lanes 2p + (lane >> 4), p = 0..15, of this thread's warp
  float4 act;
  float old_logp, adv_raw, ret;
};

}  // namespace tcu

constexpr size_t kTcUpdSmem = sizeof(tcu::Smem) + 1024;     // + slack to align the dynamic segment to 1024 B

// partials: [2 towers][kWG * gridDim.x][kGradLen]; a CTA writes only its tower's entries (ppo_reduce_tc_kernel)
__global__ void __launch_bounds__(tcu::kThreads, 1) ppo_grad_tc_kernel(const __grid_constant__ UpdArgs A) {
  using namespace tcu;
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  Smem& S = *reinterpret_cast<Smem*>(smem_dyn + ((1024u - (smem_addr(smem_dyn) & 1023u)) & 1023u));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tw = blockIdx.y;

  setup(S, A.theta, tw);

  const int64_t n_tiles = (A.m + 127) / 128;
  const int64_t stride = (int64_t)gridDim.x * kWG;

  if (warp >= 2 * 4) {
    // ---------------- MMA issuer warps ----------------
    const int wg = warp - 8;
    const int64_t first_tile = (int64_t)blockIdx.x * kWG + wg;
    const int64_t my_tiles = first_tile < n_tiles ? (n_tiles - first_tile + stride - 1) / stride : 0;
    long long* tlog = nullptr;
#if DRONECU_TC_TIMING
    if (A.dbg != nullptr && blockIdx.x == 0 && tw == 0 && wg == 0) tlog = reinterpret_cast<long long*>(A.dbg) + 1024;
#endif
    issuer(S, wg, my_tiles, tlog);
  } else {
    // ---------------- compute warpgroups ----------------
    const int wg = tid >> 7, r = tid & 127, wq = r >> 5;
    float std_inv[kAct], logstd_sum = 0.f;
#pragma unroll
    for (int o = 0; o < kAct; ++o) { std_inv[o] = expf(-S.log_std[o]); logstd_sum += S.log_std[o]; }
    float adv_mean, adv_inv_std;
    adv_normalizer(A, adv_mean, adv_inv_std);

    unsigned char* const bufA = S.bufA[wg];
    unsigned char* const bufB = S.bufB[wg];
    unsigned char* const XA = S.XA[wg];
    unsigned long long* const full = &S.full[wg];
    unsigned long long* const done = &S.done[wg];
    const uint32_t tmem = S.tmem_base + wg * kColsPerWG;                   // lane 0, first column of the warpgroup
    const uint32_t tL = tmem + ((uint32_t)(wq * 32) << 16);                // this thread's subpartition
    uint32_t ph = 0;

    // per-thread scalar accumulators over all tiles of this thread (reduced once after the loop)
    // pi: [0..3] d log_std | [4..7] db3 | [8] policy loss | [9] kl | [10] clip fraction ; vf: [0] db3 | [1] value loss | [2] count
    float accs[kNS];
#pragma unroll
    for (int q = 0; q < kNS; ++q) accs[q] = 0.f;

    // row numbers stay 32-bit and untouched until they are used one tile later: any arithmetic on the loaded index
    // (v2.1 sign-extended it) makes the thread wait out the load right where it is issued
    auto row_of = [&](int64_t tile) -> int {
      const int64_t pos = tile * 128 + r;
      if (tile >= n_tiles || pos >= A.m) return -1;
      if (A.index == nullptr) return (int)(A.first + pos);
      int v;
      asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(A.index + pos));
      return v;
    };
    // Observation rows are 60 contiguous bytes at random places: 16 lanes read one row (element = lane & 15, the
    // 16th is the ones column), two rows per warp instruction, instead of every lane walking its own row (v2.0:
    // 15 loads x 32 sectors per warp and tile kept the LSU busy for thousands of cycles).  The row numbers of
    // the warp's 32 samples travel by shuffle.
    auto gather = [&](int row32, RowIn& in) {
      const int col = min(lane & 15, kObs - 1), half = lane >> 4;
      const int64_t row = row32;                      // B < 2^31 rows (checked by the host)
#pragma unroll
      for (int p = 0; p < 16; ++p) {
        // always a valid address: rows past the end of the minibatch read row 0 and are zeroed when staged, so all
        // 16 loads are in flight at once (a select on the loaded value made ptxas serialise them in v2.1)
        const int rr = max(__shfl_sync(0xffffffffu, row32, 2 * p + half), 0);
        asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(in.xe[p]) : "l"(A.obs + (int64_t)rr * A.obs_stride + col));
      }
      in.act = make_float4(0.f, 0.f, 0.f, 0.f);
      in.old_logp = in.adv_raw = in.ret = 0.f;
      if (row >= 0) {
        if (tw == 0) { in.act = A.actions[row]; in.old_logp = A.old_logp[row]; in.adv_raw = A.adv[row]; }
        else in.ret = A.ret[row];
      }
    };
    unsigned char* const XS = S.XS[wg];
    long long* tlog = nullptr;
#if DRONECU_TC_TIMING
    if (A.dbg != nullptr && blockIdx.x == 0 && tw == 0 && wg == 0 && r == 0) tlog = reinterpret_cast<long long*>(A.dbg);
#endif
    (void)tlog;
    int64_t tile = (int64_t)blockIdx.x * kWG + wg;
    int row_cur = row_of(tile), row_nxt = row_of(tile + stride);
    RowIn cur;
    gather(row_cur, cur);
    int it = 0;
    for (; tile < n_tiles; tile += stride, ++it) {
      const bool live = row_cur >= 0;
      TSTAMP(tlog, it, 0);
      // ---------------- X -> shared memory: [samples x 16] (A of S1) and its transpose (B of S6) ----------------
      const float4 act = cur.act;
      const float old_logp = cur.old_logp, adv_raw = cur.adv_raw, ret = cur.ret;
      if (it > 0) { mbar_wait(done, ph); ph ^= 1; fence_after(); }    // S6 of the previous tile has read bufA / XA
      TSTAMP(tlog, it, 1);
      {
        const int col = lane & 15, half = lane >> 4, base = 32 * wq + half;
        const uint32_t live_mask = __ballot_sync(0xffffffffu, live) >> half;      // bit 2p: the row staged in pass p is live
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          float v = (col < kObs) ? to_tf32_fast(cur.xe[p]) : 1.0f;
          if (!((live_mask >> (2 * p)) & 1u)) v = 0.f;
          *xs_elem(XS, base + 2 * p, col) = v;
          *xa_elem(XA, col, base + 2 * p) = v;
        }
      }
      hand_over(full);
      TSTAMP(tlog, it, 2);
      // gather the next tile's rows while this one computes; fetch the row index of the tile after that
      gather(row_nxt, cur);
      row_cur = row_nxt;
      row_nxt = row_of(tile + 2 * stride);
      TSTAMP(tlog, it, 3);

      // ---------------- S1 done: H1 = tanh(D1) -> P in place (A of S2) + bufA ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 4);
      {
        float va[16], vb[16];
        ld16_issue(tL + kColP, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kColP + 16 * (c + 1), w);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = to_tf32_fast(tanh_mufu(v[i]));
          st16(tL + kColP + 16 * c, v);
#pragma unroll
          for (int q = 0; q < 4; ++q) *mn_quad(bufA, r, 4 * c + q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          if (c < 3) ld_fence(w);
        }
      }
      wait_st();
      hand_over(full);
      TSTAMP(tlog, it, 5);

      // ---------------- S2 done: H2 = tanh(D2 + b2) -> Q in place (A of S3) + bufB ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 6);
      {
        float va[16], vb[16];
        ld16_issue(tL + kColQ, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kColQ + 16 * (c + 1), w);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 b = reinterpret_cast<const float4*>(S.b2 + 16 * c)[q];
            add2(v[4 * q], v[4 * q + 1], b.x, b.y);
            add2(v[4 * q + 2], v[4 * q + 3], b.z, b.w);
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = to_tf32_fast(tanh_mufu(v[i]));
          st16(tL + kColQ + 16 * c, v);
#pragma unroll
          for (int q = 0; q < 4; ++q) *mn_quad(bufB, r, 4 * c + q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          if (c < 3) ld_fence(w);
        }
      }
      wait_st();
      hand_over(full);
      TSTAMP(tlog, it, 7);

      // ---------------- S3 done: head outputs -> loss gradient at the head ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 8);
      float out[4];
      ld4(tL + kColD3, out);
      float g3[kAct] = {0.f, 0.f, 0.f, 0.f};
      if (tw == 0) {
        if (live) {
          float mean[kAct];
#pragma unroll
          for (int o = 0; o < kAct; ++o) mean[o] = out[o] + S.b3[o];
          const PolicyHead h = policy_head(act, mean, std_inv, logstd_sum, old_logp, (adv_raw - adv_mean) * adv_inv_std,
                                           A.clip, A.ent_coef);
#pragma unroll
          for (int o = 0; o < kAct; ++o) {
            g3[o] = h.g_mean[o];
            accs[o] += h.g_logstd[o];
            accs[4 + o] += g3[o];
          }
          accs[8] += h.pg_loss;
          accs[9] += h.kl;
          accs[10] += h.clipped;
        }
      } else {
        if (live) {
          float sq_err;
          g3[0] = value_head(out[0] + S.b3[0], ret, A.vf_coef, sq_err);
          accs[0] += g3[0];
          accs[1] += sq_err;
          accs[2] += 1.0f;
        }
      }
      {
        float gv[8] = {to_tf32_fast(g3[0]), to_tf32_fast(g3[1]), to_tf32_fast(g3[2]), to_tf32_fast(g3[3]),
                       live ? 1.0f : 0.f, 0.f, 0.f, 0.f};
        if (!live) { gv[0] = gv[1] = gv[2] = gv[3] = 0.f; }
        st8(tL + kColGA, gv);
#pragma unroll
        for (int o = 0; o < 8; ++o) *xa_elem(XA, 16 + o, r) = gv[o];
      }
      wait_st();
      hand_over(full);
      TSTAMP(tlog, it, 9);

      // ---------------- S4 done: dZ2 = dH2 * (1 - H2^2) -> Q in place (A of S5) + bufB ----------------
      {
        float h[4][16];                          // H2 does not depend on S4: fetch it from TMEM while S4 runs
#pragma unroll
        for (int c = 0; c < 4; ++c) ld16_issue(tL + kColQ + 16 * c, h[c]);
        mbar_wait(done, ph); ph ^= 1; fence_after();
        TSTAMP(tlog, it, 10);
        float da[16], db[16];
        ld16_issue(tL + kColP, da);
#pragma unroll
        for (int c = 0; c < 4; ++c) ld_fence(h[c]);
        ld_fence(da);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&d)[16] = (c & 1) ? db : da;
          float (&w)[16] = (c & 1) ? da : db;
          if (c < 3) ld16_issue(tL + kColP + 16 * (c + 1), w);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            float t0, t1;
            one_minus_sq2(h[c][i], h[c][i + 1], t0, t1);
            mul2(d[i], d[i + 1], t0, t1);
            d[i] = to_tf32_fast(d[i]); d[i + 1] = to_tf32_fast(d[i + 1]);
          }
          st16(tL + kColQ + 16 * c, d);
#pragma unroll
          for (int q = 0; q < 4; ++q) *mn_quad(bufB, r, 4 * c + q) = make_float4(d[4 * q], d[4 * q + 1], d[4 * q + 2], d[4 * q + 3]);
          if (c < 3) ld_fence(w);
        }
      }
      wait_st();
      hand_over(full);
      TSTAMP(tlog, it, 11);

      // ---------------- S5 done: dZ1 = dH1 * (1 - H1^2), over H1 in bufA ----------------
      {
        float4 h1[16];                           // H1 does not depend on S5 either: read it back while S5 runs
#pragma unroll
        for (int q = 0; q < 16; ++q) h1[q] = *mn_quad(bufA, r, q);
        mbar_wait(done, ph); ph ^= 1; fence_after();
        TSTAMP(tlog, it, 12);
        float va[16], vb[16];
        ld16_issue(tL + kColP, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kColP + 16 * (c + 1), w);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 h = h1[4 * c + q];
            float t0, t1, t2, t3;
            one_minus_sq2(h.x, h.y, t0, t1);
            one_minus_sq2(h.z, h.w, t2, t3);
            mul2(v[4 * q], v[4 * q + 1], t0, t1);
            mul2(v[4 * q + 2], v[4 * q + 3], t2, t3);
            *mn_quad(bufA, r, 4 * c + q) =
                make_float4(to_tf32_fast(v[4 * q]), to_tf32_fast(v[4 * q + 1]), to_tf32_fast(v[4 * q + 2]), to_tf32_fast(v[4 * q + 3]));
          }
          if (c < 3) ld_fence(w);
        }
      }
      hand_over(full);                          // S6; its completion is awaited at the top of the next tile / after the loop
      TSTAMP(tlog, it, 13);
    }
    if (it > 0) { mbar_wait(done, ph); ph ^= 1; }
    fence_after();

    if (A.dbg != nullptr && tw == 0 && !DRONECU_TC_TIMING) {       // debugging aid: this thread's TMEM lane, all 256 columns of the warpgroup
      float* d = A.dbg + (((size_t)blockIdx.x * kWG + wg) * 128 + r) * kColsPerWG;
#pragma unroll 1
      for (int c = 0; c < kColsPerWG / 16; ++c) {
        float v[16];
        ld16_issue(tL + 16 * c, v);
        ld_fence(v);
#pragma unroll
        for (int i = 0; i < 16; ++i) d[16 * c + i] = v[i];
      }
    }

    // ---------------- per-thread scalars: warp sums, then a fixed-order sum over the four warps ----------------
#pragma unroll
    for (int q = 0; q < kNS; ++q) accs[q] = warp_sum(accs[q]);
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < kNS; ++q) S.wsum[wg][wq][q] = accs[q];
    }
    wg_barrier(wg);
    auto scalar = [&](int q) { return ((S.wsum[wg][0][q] + S.wsum[wg][1][q]) + S.wsum[wg][2][q]) + S.wsum[wg][3][q]; };

    // ---------------- read the accumulators out: one partial vector per (tower, CTA, warpgroup) ----------------
    float* const outv = A.partials + (((size_t)tw * gridDim.x + blockIdx.x) * kWG + wg) * kGradLen;
    const int oW1 = tw ? O_VF_W1 : O_PI_W1, oB1 = tw ? O_VF_B1 : O_PI_B1, oW2 = tw ? O_VF_W2 : O_PI_W2;
    const int oB2 = tw ? O_VF_B2 : O_PI_B2, oW3 = tw ? O_VF_W3 : O_PI_W3, oB3 = tw ? O_VF_B3 : O_PI_B3;
    const int nB3 = tw ? 1 : kAct;
    if (it == 0) {         // this warpgroup saw no tile: contribute zeros
      for (int idx = r; idx < oB3 + nB3 - oW1; idx += 128) outv[oW1 + idx] = 0.f;
      if (tw == 0 && r < kAct) outv[O_LOGSTD + r] = 0.f;
      if (r < kStats) outv[kParams + r] = 0.f;
    } else {
      const int j = 16 * wq + lane;               // accumulator row held by lanes 0..15 of each subpartition
      const bool own = lane < 16;
      float v[16];
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        ld16_issue(tL + kAccW2 + 16 * c, v);
        ld_fence(v);
        if (own) {
#pragma unroll
          for (int i = 0; i < 16; ++i) outv[oW2 + j * kHid + 16 * c + i] = v[i];
        }
      }
      ld16_issue(tL + kAccW1, v);
      ld_fence(v);
      if (own) {
#pragma unroll
        for (int i = 0; i < kObs; ++i) outv[oW1 + j * kObs + i] = v[i];
        outv[oB1 + j] = v[15];
      }
      ld16_issue(tL + kAccW3, v);                 // columns 208..223: dW3 (8) | db2 (8)
      ld_fence(v);
      if (own) {
        if (tw == 0) {
#pragma unroll
          for (int o = 0; o < kAct; ++o) outv[oW3 + o * kHid + j] = v[o];
        } else {
          outv[oW3 + j] = v[0];
        }
        outv[oB2 + j] = v[8 + 4];
      }
      if (tw == 0) {
        if (r < kAct) { outv[O_LOGSTD + r] = scalar(r); outv[O_PI_B3 + r] = scalar(4 + r); }
        // statistics block: [policy loss, value loss, kl, clip fraction, count, 0, 0, 0]; the policy tower owns 0, 2, 3
        if (r < kStats) outv[kParams + r] = (r == 0) ? scalar(8) : (r == 2) ? scalar(9) : (r == 3) ? scalar(10) : 0.f;
      } else {
        if (r == 0) outv[O_VF_B3] = scalar(0);
        if (r < kStats) outv[kParams + r] = (r == 1) ? scalar(1) : (r == 4) ? scalar(2) : 0.f;
      }
    }
  }

  fence_before();
  __syncthreads();
  if (tid < 32)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(S.tmem_base), "r"((uint32_t)tcu::kTmemCols) : "memory");
}

// fixed-order sum of the partial vectors of ppo_grad_tc_kernel: element idx belongs to one tower (the value tower
// owns its parameter block and the statistics 1 (value loss) and 4 (count)), whose np partials are summed
__global__ void ppo_reduce_tc_kernel(const float* __restrict__ partials, int np, float* __restrict__ grad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kGradLen) return;
  int tw = (idx >= O_VF_W1 && idx < O_LOGSTD) ? 1 : 0;
  if (idx >= kParams) { const int q = idx - kParams; tw = (q == 1 || q == 4) ? 1 : 0; }
  const float* p = partials + (size_t)tw * np * kGradLen + idx;
  float sum = 0.f;
  for (int k = 0; k < np; ++k) sum += p[(size_t)k * kGradLen];
  grad[idx] = sum;
}

}  // namespace dronecu
