// PPO minibatch gradient on tcgen05 / TMEM, three tiles in flight per SM (`update_precision = "bf16"`): same
// contract as ppo_grad_kernel / ppo_grad_tc_kernel (what SB3's PPO.train() does per minibatch; SURVEY.md appendix C;
// call site /root/reference/train.py:63-68 -- "parity unpinned").
//
// ppo_grad_tc_kernel (all-tf32) is bounded by its shared-memory operands: the weight-gradient products reduce over
// the SAMPLES, so both of their operands must come from shared memory as 32-bit words (64 KB per tile in flight;
// 116 KB read by the tensor core in step S5 alone), and 64 KB + 256 TMEM columns per tile allow only two tiles per SM
// (profiles/README.md).  Here the FORWARD and the activation-gradient (dgrad) products keep tf32 operands with the A
// operand in TMEM, exactly as before, but the four WEIGHT-gradient products take bf16 operands (kind::f16, K = 16 per
// instruction, fp32 accumulation) -- the usual mixed-precision recipe, applied to wgrad only:
//   * half the bytes and half the instructions per product; dW2 and db2 become ONE product, dZ2^T . [H1 | G] with
//     N = 72 (MMAs per tile: 91 -> 51);
//   * the bf16 operands use the no-swizzle MN-major ("interleave") layout, which for a thread-per-sample producer
//     is simply [8-feature group][128 samples][16 bytes]: one conflict-free 16-byte store per group (probed on the
//     B200 for A and B operands, N = 8 / 16 / 72: scratch/mma_probe_bf16.cu);
//   * 54 KB of shared memory and 136 TMEM columns per tile: THREE compute warpgroups per CTA; the weight-gradient
//     accumulators (96 columns) are shared by the three and therefore fed by ONE thread (the accumulating issuer: steps
//     S4..S6) in a FIXED order over the CTA's tiles (so that the accumulation order -- hence every bit of the result --
//     does not depend on timing), software-pipelined over consecutive tiles: S4(j) S6(j-1) S5(j), so that the issuer
//     serves another warpgroup while one computes dZ2 / dZ1.  The steps that only touch a warpgroup's private columns
//     (S1..S3) need no order at all: every warpgroup has its OWN private-step issuer warp (512 threads per CTA).  r02:
//     before, one shared private-step issuer warp walked a global order, which made every warpgroup's S1 wait for
//     another warpgroup's tanh phase -- 1.9k idle cycles per tile in the in-kernel timeline; issuing from warp 0 of the
//     warpgroup instead cost 9 %: that warp sits in the MMA issue for ~1k cycles when the tensor queue is full and
//     becomes the straggler of its warpgroup;
//   * the observation rows of the next tile are fetched a tile ahead in four parts spread over the tile; with 64-byte rows
//     in the rollout buffer (template PADDED) a row is four LDG.128 by four lanes and is staged with vector stores; the tf32
//     X tile is staged over the dead bufB (never over memory another warp still reads: the r02 race);
//   * tanh'(layer 1) = 1 - H1^2 is stashed per sample as bf16 (2^-9 relative) next to the operands, because H1 itself
//     survives only as a bf16 operand (1 - h^2 from a rounded h would lose the saturated units); tanh'(layer 2) uses
//     the fp32 H2 still in TMEM.  The stash uses the [8-feature chunk][sample][16 B] layout of the operand buffers
//     (swizzled 128-byte rows per sample measured slower);
//   * the elementwise phases work on the register pairs tcgen05.ld delivers with packed fp32 instructions (FFMA2 / FMUL2 /
//     FADD2, ppo_common.cuh): ~1,180 instructions per thread and tile instead of ~1,400, bit-identical results.
// Steps per tile (S1..S6 as in ppo_update_tc.cuh): S1 D1 = X.W1^T | S2 D2 = H1.W2^T | S3 D3 = H2.W3p^T |
// S4 dH2 = G.W3k, dW3 += H2^T.G | S5 dH1 = dZ2.W2, dW2|db2 += dZ2^T.[H1|G] | S6 dW1|db1 += dZ1^T.[X|1].
// TMEM: per warpgroup P 64 | Q 64 | G 8 (D3 aliases P); shared dW2|db2 72 | dW1 16 | dW3 8 = 504 of 512 columns.
#pragma once
#include "ppo_update_tc.cuh"

namespace dronecu {
namespace tcb {

using namespace tcu;            // descriptors, TMEM ld / st helpers, elect_one, hand_over, RowIn, xs_elem ...

constexpr int kWG3 = 3;
constexpr int kComputeThreads3 = 128 * kWG3;
constexpr int kIssuerWarps3 = kWG3 + 1;                // one private-step issuer warp per warpgroup + the accumulating issuer
constexpr int kThreads3 = kComputeThreads3 + 32 * kIssuerWarps3;   // compute warpgroups + issuer warps (the LAST one is the accumulating issuer: S4..S6)
constexpr int kGrp = 128 * 16;                         // one 8-feature group of a bf16 MN-major operand: [128 samples][16 B]
constexpr int kWgCols = 136;                           // P 64 | Q 64 | G 8
constexpr int kCP = 0, kCQ = 64, kCG = 128;
constexpr int kAcc2 = kWG3 * kWgCols;                  // 408: dW2 (64 columns) | db2 group (8)
constexpr int kAcc1 = kAcc2 + 72;                      // 480: dW1 | db1 (16)
constexpr int kAcc3 = kAcc1 + 16;                      // 496: dW3 (8)
constexpr int kTmem3 = 512;

struct alignas(1024) Smem3 {
  unsigned char bufA[kWG3][9 * kGrp];    // bf16: groups 0..7 = H1, later dZ1; group 8 = G (g3[0..3] | live | 0 0 0)
  unsigned char bufB[kWG3][8 * kGrp];    // bf16: H2, later dZ2
  unsigned char XN[kWG3][2][2 * kGrp];   // bf16: X (x0..x14, 1): B of S6; double-buffered (tile parity) so that the next tile is staged while S6 runs
  unsigned char XG[kWG3][16384];         // bf16(1 - H1^2), 128 B per sample (the tanh' stash; r01 also staged the tf32 X tile here)
  float W1[kHid * 16];
  float W2[kHid * kHid];
  float W2T[kHid * kHid];
  float W3p[16 * kHid];
  float W3k[kHid * 8];
  float b2[kHid];
  float b3[kAct];
  float log_std[kAct];
  float wsum[kWG3][4][kNS];
  alignas(8) unsigned long long full[kWG3];     // operands of S1 / S2 / S3 staged (served by the warpgroup's private-step issuer)
  alignas(8) unsigned long long fullA[kWG3];    // operands of S4 / S5 / S6 staged (served by the accumulating issuer, fixed order)
  alignas(8) unsigned long long done[kWG3];     // S1 / S2 / S3 completed (commit of the private-step issuer)
  alignas(8) unsigned long long doneA[kWG3];    // S4 / S5 / S6 completed (commit of the accumulating issuer)
  uint32_t tmem_base, pad1[3];
};

// MN-major no-swizzle bf16 operand: slice s = 16 samples (two K groups of 8 rows x 16 B); groups along MN are kGrp apart
__device__ __forceinline__ uint64_t desc_il(uint32_t buf, int s) { return make_desc(buf + 256 * s, 128, kGrp, 0); }

// kind::f16 instruction descriptor: D = f32, A = B = bf16
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t id, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(id), "r"(accumulate) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

__device__ __forceinline__ void setup3(Smem3& S, const float* __restrict__ theta, const int tw) {
  const int tid = threadIdx.x;
  const int oW1 = tw ? O_VF_W1 : O_PI_W1, oB1 = tw ? O_VF_B1 : O_PI_B1, oW2 = tw ? O_VF_W2 : O_PI_W2;
  const int nout = tw ? 1 : kAct, oW3 = tw ? O_VF_W3 : O_PI_W3;
  for (int q = tid; q < kHid * 16; q += kThreads3) {
    const int j = q / 16, k = q % 16;
    S.W1[umma_off(j, k, 16)] = to_tf32((k < kObs) ? theta[oW1 + j * kObs + k] : theta[oB1 + j]);
  }
  for (int q = tid; q < kHid * kHid; q += kThreads3) {
    const int j = q / kHid, i = q % kHid;
    const float v = to_tf32(theta[oW2 + q]);
    S.W2[umma_off(j, i, kHid)] = v;
    S.W2T[umma_off(i, j, kHid)] = v;
  }
  for (int q = tid; q < 16 * kHid; q += kThreads3) {
    const int o = q / kHid, j = q % kHid;
    S.W3p[umma_off(o, j, kHid)] = (o < nout) ? to_tf32(theta[oW3 + o * kHid + j]) : 0.f;
  }
  for (int q = tid; q < kHid * 8; q += kThreads3) {
    const int j = q / 8, o = q % 8;
    S.W3k[umma_off(j, o, 8)] = (o < nout) ? to_tf32(theta[oW3 + o * kHid + j]) : 0.f;
  }
  for (int q = tid; q < kHid; q += kThreads3) S.b2[q] = theta[(tw ? O_VF_B2 : O_PI_B2) + q];
  if (tid < kAct) {
    S.b3[tid] = tw ? (tid == 0 ? theta[O_VF_B3] : 0.f) : theta[O_PI_B3 + tid];
    S.log_std[tid] = theta[O_LOGSTD + tid];
  }
  if (tid == 0) {
    for (int w = 0; w < kWG3; ++w) { mbar_init(&S.full[w], 128); mbar_init(&S.fullA[w], 128); mbar_init(&S.done[w], 1); mbar_init(&S.doneA[w], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (tid < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_addr(&S.tmem_base)), "r"((uint32_t)kTmem3) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  proxy_fence();
  fence_before();
  __syncthreads();
  fence_after();
}

// Descriptors are built once per thread that issues; a K slice, and the warpgroup, only bump the 14-bit start-address
// field (16-byte units).
constexpr uint64_t kStrA = (9 * kGrp) >> 4, kStrB = (8 * kGrp) >> 4, kStrXn = (4 * kGrp) >> 4, kParXn = (2 * kGrp) >> 4,
                   kStrXs = 16384 >> 4, kOffG = (8 * kGrp) >> 4;
constexpr uint64_t kBumpW = 256 >> 4, kBumpXs = (2 * kXsLbo) >> 4, kBumpIl = 256 >> 4;      // per-slice bumps of the start-address field

// Private steps S1, S2, S3 of warpgroup w: they write only the warpgroup's private TMEM columns, so there is nothing to
// order against the other warpgroups.  Called by the warpgroup's private-step issuer warp; waits until every thread of the
// warpgroup has arrived on `full`.
// `dA` = descriptor of the step's shared-memory A operand (S1: the X tile) -- unused for S2 / S3 (A in TMEM); `dB` = its weights.
template <int STEP>
__device__ __forceinline__ void issue_private(unsigned long long* full, unsigned long long* done, const uint32_t tmem,
                                              const uint64_t dA, const uint64_t dB, uint32_t& phf) {
  mbar_wait(full, phf);
  phf ^= 1;
  fence_after();
  if (elect_one()) {
    if (STEP == 0) {            // S1: D1 = X . W1^T   (tf32, A = X tile in shared memory)
#pragma unroll
      for (int s = 0; s < 2; ++s) mma_ss(tmem + kCP, dA + kBumpXs * s, dB + kBumpW * s, idesc(128, 64, 0, 0), s > 0);
    } else if (STEP == 1) {     // S2: D2 = H1 . W2^T  (tf32, A = H1 in TMEM)
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_tf32_ts(tmem + kCQ, tmem + kCP + 8 * s, dB + kBumpW * s, idesc(128, 64, 0, 0), s > 0);
    } else {                    // S3: D3 = H2 . W3p^T (tf32, A = H2 in TMEM; D3 over the dead H1 in P)
#pragma unroll
      for (int s = 0; s < 8; ++s) mma_tf32_ts(tmem + kCP, tmem + kCQ + 8 * s, dB + kBumpW * s, idesc(128, 16, 0, 0), s > 0);
    }
    mma_commit(done);
  }
  __syncwarp();
}

// The accumulating issuer: S4, S5, S6 of EVERY tile of the CTA, in one fixed order.  The CTA's tiles in global order are
// j = 3 r + w (round r, warpgroup w); the existing ones are a prefix j = 0 .. n_cta - 1 of that sequence.  Each shared
// accumulator (dW3 by S4, dW2 | db2 by S5, dW1 | db1 by S6) must receive the tiles in order of j; the services are
// software-pipelined over consecutive tiles -- S4(0) S5(0) | S4(j) S6(j-1) S5(j) | ... | S6(n-1) -- so that between the two
// services of one warpgroup that are separated by its dZ2 / dZ1 phases the issuer serves another warpgroup.  The fixed order
// is also what staggers the three warpgroups: the sequential S4(j) S5(j) S6(j) measured 1.625 vs 1.619 ms, and serving
// whichever warpgroup is ready 24 % slower (served eagerly they fall into step and queue on the same phases; profiles/README.md).
__device__ __forceinline__ void issuer_accum(Smem3& S, const int n_cta, long long* tlog) {
  const uint64_t dW2T = desc_w(smem_addr(S.W2T), kHid, 0), dW3k = desc_w(smem_addr(S.W3k), 8, 0);
  const uint64_t dA0 = desc_il(smem_addr(S.bufA[0]), 0), dB0 = desc_il(smem_addr(S.bufB[0]), 0), dXn0 = desc_il(smem_addr(S.XN[0][0]), 0);
  const uint32_t tbase = S.tmem_base;
  uint32_t ph_mask = 0;                                // bit w: parity of warpgroup w's `fullA` barrier
  auto serve = [&](const int j, const int step) __attribute__((always_inline)) {      // step 3, 4, 5 = S4, S5, S6 of tile j
    const int w = j % kWG3, r = j / kWG3;
    mbar_wait(&S.fullA[w], (ph_mask >> w) & 1u);
    ph_mask ^= 1u << w;
    fence_after();
    if (w == 0) TSTAMP(tlog, r, 2 * step);
    if (elect_one()) {
      const uint32_t tmem = tbase + w * kWgCols;
      const uint64_t uw = (uint64_t)w;
      const uint32_t first = j > 0;                    // tile 0 initialises the shared accumulators
      if (step == 3) {            // S4: dH2 = G . W3k (tf32, A = G in TMEM, K = 8) ; dW3 += H2^T . G (bf16)
        mma_tf32_ts(tmem + kCP, tmem + kCG, dW3k, idesc(128, 64, 0, 0), 0);
        const uint64_t dH = dB0 + kStrB * uw, dG = dA0 + kStrA * uw + kOffG;
#pragma unroll
        for (int s = 0; s < 8; ++s) mma_bf16_ss(tbase + kAcc3, dH + kBumpIl * s, dG + kBumpIl * s, idesc_bf16(64, 8, 1, 1), first | (s > 0));
      } else if (step == 4) {     // S5: dH1 = dZ2 . W2 (tf32, A = dZ2 in TMEM) ; dW2 | db2 += dZ2^T . [H1 | G] (bf16, N = 72)
        const uint64_t dZ = dB0 + kStrB * uw, dHG = dA0 + kStrA * uw;
        // The two products are independent: interleave them in the pipe.  Issued one after the other they keep the tensor
        // pipe waiting on shared-memory operands (1.633 vs 1.619 ms); so does committing dH1 on its own so that the dZ1
        // phase starts earlier (+4.5 %, more than the earlier wake-up gains).
#pragma unroll
        for (int s = 0; s < 8; ++s) {
          mma_tf32_ts(tmem + kCP, tmem + kCQ + 8 * s, dW2T + kBumpW * s, idesc(128, 64, 0, 0), s > 0);
          mma_bf16_ss(tbase + kAcc2, dZ + kBumpIl * s, dHG + kBumpIl * s, idesc_bf16(64, 72, 1, 1), first | (s > 0));
        }
      } else {                    // S6: dW1 | db1 += dZ1^T . [X | 1] (bf16, N = 16)
        const uint64_t dZ = dA0 + kStrA * uw, dX = dXn0 + kStrXn * uw + kParXn * (uint64_t)(r & 1);
#pragma unroll
        for (int s = 0; s < 8; ++s) mma_bf16_ss(tbase + kAcc1, dZ + kBumpIl * s, dX + kBumpIl * s, idesc_bf16(64, 16, 1, 1), first | (s > 0));
      }
      mma_commit(&S.doneA[w]);
    }
    __syncwarp();
    if (w == 0) TSTAMP(tlog, r, 2 * step + 1);
  };
#pragma unroll 1
  for (int j = 0; j <= n_cta; ++j) {
    if (j < n_cta) serve(j, 3);
    if (j > 0) serve(j - 1, 5);
    if (j < n_cta) serve(j, 4);
  }
}

}  // namespace tcb

constexpr size_t kTc3Smem = sizeof(tcb::Smem3) + 1024;

// partials: [2 towers][gridDim.x][kGradLen]
// PADDED: the observation rows are 64 bytes (16 floats, the 16th = 1.0: dronecu_policy_out.obs_padded) -- a row is four aligned
// 16-byte chunks, fetched as LDG.128 by four lanes (8 rows per load instruction instead of 2) and staged with one STS.128 (tf32 X
// tile: four consecutive k of a sample are contiguous) + one STS.64 (bf16 X) per chunk instead of eight 4- / 2-byte stores.
template <bool PADDED>
__global__ void __launch_bounds__(tcb::kThreads3, 1) ppo_grad_bf16_kernel(const __grid_constant__ UpdArgs A) {
  using namespace tcb;
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  Smem3& S = *reinterpret_cast<Smem3*>(smem_dyn + ((1024u - (smem_addr(smem_dyn) & 1023u)) & 1023u));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tw = blockIdx.y;

  setup3(S, A.theta, tw);

  const int64_t n_tiles = (A.m + 127) / 128;
  const int64_t stride = (int64_t)gridDim.x * kWG3;

  if (warp >= 4 * kWG3) {
    long long* tlog = nullptr;
    auto tiles_of = [&](int w) -> int {
      const int64_t first = (int64_t)blockIdx.x * kWG3 + w;
      return first < n_tiles ? (int)((n_tiles - first + stride - 1) / stride) : 0;
    };
    const int iw = warp - 4 * kWG3;
    if (iw == kIssuerWarps3 - 1) {
#if DRONECU_TC_TIMING
      if (A.dbg != nullptr && blockIdx.x == 0 && tw == 0) tlog = reinterpret_cast<long long*>(A.dbg) + 1024;
#endif
      issuer_accum(S, tiles_of(0) + tiles_of(1) + tiles_of(2), tlog);
    } else {
      // private-step issuer of warpgroup iw: S1, S2, S3 of each of its tiles, in the warpgroup's own order -- these steps write only
      // the warpgroup's private TMEM columns, so there is nothing to order against the other warpgroups
      const uint32_t tmem_w = S.tmem_base + iw * kWgCols;
      const uint64_t dXs = make_desc(smem_addr(S.bufB[iw]), kXsLbo, kXsSbo, 0), dW1 = desc_w(smem_addr(S.W1), 16, 0);
      const uint64_t dW2 = desc_w(smem_addr(S.W2), kHid, 0), dW3p = desc_w(smem_addr(S.W3p), kHid, 0);
      uint32_t phf = 0;
      const int my_tiles = tiles_of(iw);
#pragma unroll 1
      for (int t = 0; t < my_tiles; ++t) {
        issue_private<0>(&S.full[iw], &S.done[iw], tmem_w, dXs, dW1, phf);
        issue_private<1>(&S.full[iw], &S.done[iw], tmem_w, 0, dW2, phf);
        issue_private<2>(&S.full[iw], &S.done[iw], tmem_w, 0, dW3p, phf);
      }
    }
  } else {
    const int wg = tid >> 7, r = tid & 127, wq = r >> 5;
    float std_inv[kAct], logstd_sum = 0.f;
#pragma unroll
    for (int o = 0; o < kAct; ++o) { std_inv[o] = expf(-S.log_std[o]); logstd_sum += S.log_std[o]; }
    float adv_mean, adv_inv_std;
    adv_normalizer(A, adv_mean, adv_inv_std);

    unsigned char* const rowA = S.bufA[wg] + r * 16;       // + g * kGrp: this sample's 16 bytes of feature group g
    unsigned char* const rowB = S.bufB[wg] + r * 16;
    unsigned char* const XN0 = S.XN[wg][0];
    // tf32 X tile (A operand of S1, 9216 B): staged over the DEAD bufB of the previous tile (dZ2: read only by the tensor core,
    // S5 has completed) -- no thread ever reads that region.  r01 staged it over the tanh' stash, whose rows other warps of the
    // warpgroup still read in their dZ1 phase: that aliasing produced one garbage 8-feature block of dW1 per ~1500 launches at
    // the c5 size (scratch/stress_determinism.py).
    unsigned char* const XS = S.bufB[wg];
    unsigned char* const rowG1 = S.XG[wg] + r * 16;        // chunk c of this sample at c * kGrp (the layout of bufA: conflict-free, immediate offsets)
    unsigned long long* const full = &S.full[wg];
    unsigned long long* const fullA = &S.fullA[wg];
    unsigned long long* const done = &S.done[wg];
    unsigned long long* const doneA = &S.doneA[wg];
    uint32_t phA = 0;
    const uint32_t tmem = S.tmem_base + wg * kWgCols;
    const uint32_t tL = tmem + ((uint32_t)(wq * 32) << 16);
    uint32_t ph = 0;

    float accs[kNS];
#pragma unroll
    for (int q = 0; q < kNS; ++q) accs[q] = 0.f;

    auto row_of = [&](int64_t tile) -> int {
      const int64_t pos = tile * 128 + r;
      if (tile >= n_tiles || pos >= A.m) return -1;
      if (A.index == nullptr) return (int)(A.first + pos);
      int v;
      asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(A.index + pos));
      return v;
    };
    // The next tile's rows are fetched a tile ahead, in FOUR parts spread over the current tile (after the S1 / S2 / S3 / S4
    // hand-overs, where the warp would otherwise only wait for the tensor core): issued in one burst, the ~550 sectors of a
    // tile overflow the SM's outstanding-miss capacity and the load ISSUE stalled for 3-4k of 15k cycles per tile (in-kernel
    // timeline at the c5 size, profiles/r02_grad_timeline_sorted_rows_c5_size.txt).
    auto gather_rows = [&](int row32, RowIn& in, const int p0) {      // observation rows: 4 of the 16 two-row loads
      if constexpr (PADDED) {       // part p0 / 4: samples 8 (p0 / 4) + (lane >> 2) of this warp, chunk lane & 3 of their rows
        const int rr = max(__shfl_sync(0xffffffffu, row32, 2 * p0 + (lane >> 2)), 0);
        asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(in.xe[p0]), "=f"(in.xe[p0 + 1]), "=f"(in.xe[p0 + 2]), "=f"(in.xe[p0 + 3])
                     : "l"(A.obs + (int64_t)rr * 16 + 4 * (lane & 3)));
        return;
      }
      const int col = min(lane & 15, kObs - 1), half = lane >> 4;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int p = p0 + q;
        const int rr = max(__shfl_sync(0xffffffffu, row32, 2 * p + half), 0);
        asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(in.xe[p]) : "l"(A.obs + (int64_t)rr * kObs + col));
      }
    };
    auto gather_scalars = [&](int row32, RowIn& in) {
      const int64_t row = row32;
      in.act = make_float4(0.f, 0.f, 0.f, 0.f);
      in.old_logp = in.adv_raw = in.ret = 0.f;
      // volatile: as plain loads ptxas sank them to the head phase of the next tile, where each cost a full DRAM round trip
      if (row >= 0) {
        if (tw == 0) {
          asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(in.act.x), "=f"(in.act.y), "=f"(in.act.z), "=f"(in.act.w) : "l"(A.actions + row));
          asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(in.old_logp) : "l"(A.old_logp + row));
          asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(in.adv_raw) : "l"(A.adv + row));
        } else {
          asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(in.ret) : "l"(A.ret + row));
        }
      }
    };

    long long* tlog = nullptr;
#if DRONECU_TC_TIMING
    if (A.dbg != nullptr && blockIdx.x == 0 && tw == 0 && wg == 0 && lane == 0) tlog = reinterpret_cast<long long*>(A.dbg) + 256 * wq;
#endif
    int64_t tile = (int64_t)blockIdx.x * kWG3 + wg;
    int row_cur = row_of(tile), row_nxt = row_of(tile + stride);
    RowIn cur;
    for (int p0 = 0; p0 < 16; p0 += 4) gather_rows(row_cur, cur, p0);
    gather_scalars(row_cur, cur);
    int it = 0;
    for (; tile < n_tiles; tile += stride, ++it) {
      const bool live = row_cur >= 0;
      TSTAMP(tlog, it, 0);
      const float4 act = cur.act;
      const float old_logp = cur.old_logp, adv_raw = cur.adv_raw, ret = cur.ret;
      // The next tile is staged and handed over (S1) WITHOUT waiting for S6 of the previous one: X goes to the other XN
      // buffer and to XS (over the dead bufB), neither of which S6 reads.
      __syncwarp();
      TSTAMP(tlog, it, 1);
      // ---------------- X -> shared memory: tf32 [samples x 16] (A of S1) and bf16 MN-major (B of S6) ----------------
      if constexpr (PADDED) {
        const uint32_t live_all = __ballot_sync(0xffffffffu, live);
        const int j = lane & 3;
        unsigned char* const xnb = XN0 + (it & 1) * (2 * kGrp) + (j >> 1) * kGrp + (j & 1) * 8;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int sl = 8 * q + (lane >> 2), m = 32 * wq + sl;               // sample within the warp / within the tile
          const bool on = (live_all >> sl) & 1u;
          float4 v = make_float4(cur.xe[4 * q], cur.xe[4 * q + 1], cur.xe[4 * q + 2], cur.xe[4 * q + 3]);
          if (j == 3) v.w = 1.0f;                                            // the bias column, whatever the buffer holds
          if (!on) v = make_float4(0.f, 0.f, 0.f, 0.f);
          *reinterpret_cast<float4*>(XS + (m >> 3) * kXsSbo + j * kXsLbo + ((m & 7) << 4)) =
              make_float4(to_tf32_fast(v.x), to_tf32_fast(v.y), to_tf32_fast(v.z), to_tf32_fast(v.w));
          *reinterpret_cast<uint2*>(xnb + m * 16) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
        }
      } else
      {
        const int col = lane & 15, half = lane >> 4, base = 32 * wq + half;
        const uint32_t live_mask = __ballot_sync(0xffffffffu, live) >> half;
        unsigned char* const xn = XN0 + (it & 1) * (2 * kGrp) + (col >> 3) * kGrp + (col & 7) * 2;
#pragma unroll
        for (int p = 0; p < 16; ++p) {
          float v = (col < kObs) ? cur.xe[p] : 1.0f;
          if (!((live_mask >> (2 * p)) & 1u)) v = 0.f;
          *xs_elem(XS, base + 2 * p, col) = to_tf32_fast(v);
          *reinterpret_cast<unsigned short*>(xn + (base + 2 * p) * 16) = (unsigned short)(pack_bf16(v, 0.f) & 0xffffu);
        }
      }
      hand_over(full);
      TSTAMP(tlog, it, 2);
      const int row_nn = row_of(tile + 2 * stride);       // the tile after the next: its row numbers are needed a tile from now
      gather_rows(row_nxt, cur, 0);
      TSTAMP(tlog, it, 3);
      if (it > 0) { mbar_wait(doneA, phA); phA ^= 1; fence_after(); }    // S6 of the previous tile has read bufA (H1 goes there next)

      // ---------------- S1 done: H1 = tanh(D1) -> P (tf32, A of S2), bufA (bf16, B of S5), 1 - H1^2 -> stash ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 4);
      {
        float va[16], vb[16];
        ld16_issue(tL + kCP, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kCP + 16 * (c + 1), w);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = tanh_mufu(v[i]);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float* h = v + 8 * j;
            *reinterpret_cast<uint4*>(rowA + (2 * c + j) * kGrp) =
                make_uint4(pack_bf16(h[0], h[1]), pack_bf16(h[2], h[3]), pack_bf16(h[4], h[5]), pack_bf16(h[6], h[7]));
            float t[8];
#pragma unroll
            for (int i = 0; i < 8; i += 2) one_minus_sq2(h[i], h[i + 1], t[i], t[i + 1]);
            *reinterpret_cast<uint4*>(rowG1 + (2 * c + j) * kGrp) =
                make_uint4(pack_bf16(t[0], t[1]), pack_bf16(t[2], t[3]), pack_bf16(t[4], t[5]), pack_bf16(t[6], t[7]));
          }
          // A operands written to TMEM (H1, H2, dZ2) are rounded to nearest tf32 first (one integer add per value) rather
          // than left for the tensor core to truncate: truncation measured 2 % faster, but its error is a coherent bias --
          // the largest block error grew with the minibatch (4.5e-3 at 38k samples, 6.9e-3 at 114k).
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = to_tf32_fast(v[i]);
          st16(tL + kCP + 16 * c, v);
          if (c < 3) ld_fence(w);
        }
      }
      wait_st();
      hand_over(full);
      gather_rows(row_nxt, cur, 4);
      TSTAMP(tlog, it, 5);

      // ---------------- S2 done: H2 = tanh(D2 + b2) -> Q (tf32, A of S3; fp32-accurate copy for tanh'), bufB (bf16) ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 6);
      {
        float va[16], vb[16];
        ld16_issue(tL + kCQ, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kCQ + 16 * (c + 1), w);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 b = reinterpret_cast<const float4*>(S.b2 + 16 * c)[q];
            add2(v[4 * q], v[4 * q + 1], b.x, b.y);
            add2(v[4 * q + 2], v[4 * q + 3], b.z, b.w);
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = tanh_mufu(v[i]);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float* h = v + 8 * j;
            *reinterpret_cast<uint4*>(rowB + (2 * c + j) * kGrp) =
                make_uint4(pack_bf16(h[0], h[1]), pack_bf16(h[2], h[3]), pack_bf16(h[4], h[5]), pack_bf16(h[6], h[7]));
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = to_tf32_fast(v[i]);
          st16(tL + kCQ + 16 * c, v);
          if (c < 3) ld_fence(w);
        }
      }
      wait_st();
      hand_over(full);
      gather_rows(row_nxt, cur, 8);
      TSTAMP(tlog, it, 7);

      // ---------------- S3 done: head outputs -> loss gradient at the head ----------------
      mbar_wait(done, ph); ph ^= 1; fence_after();
      TSTAMP(tlog, it, 8);
      float out[4];
      ld4(tL + kCP, out);
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
        const float one = live ? 1.0f : 0.f;
        float gv[8] = {to_tf32_fast(g3[0]), to_tf32_fast(g3[1]), to_tf32_fast(g3[2]), to_tf32_fast(g3[3]), one, 0.f, 0.f, 0.f};
        if (!live) { gv[0] = gv[1] = gv[2] = gv[3] = 0.f; }
        st8(tL + kCG, gv);
        *reinterpret_cast<uint4*>(rowA + 8 * kGrp) = make_uint4(pack_bf16(g3[0], g3[1]), pack_bf16(g3[2], g3[3]), pack_bf16(one, 0.f), 0u);
      }
      wait_st();
      hand_over(fullA);
      gather_rows(row_nxt, cur, 12);
      gather_scalars(row_nxt, cur);                        // this tile's act / old_logp / adv / ret live in locals since the top
      TSTAMP(tlog, it, 9);

      // ---------------- S4 done: dZ2 = dH2 * (1 - H2^2) -> Q (tf32, A of S5), bufB (bf16, A of S5's wgrad) ----------------
      mbar_wait(doneA, phA); phA ^= 1; fence_after();
      TSTAMP(tlog, it, 10);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float d[16], h[16];
        ld16_issue(tL + kCP + 16 * c, d);
        ld16_issue(tL + kCQ + 16 * c, h);
        ld_fence(d);
        ld_fence(h);
#pragma unroll
        for (int i = 0; i < 16; i += 2) {
          float t0, t1;
          one_minus_sq2(h[i], h[i + 1], t0, t1);
          mul2(d[i], d[i + 1], t0, t1);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const float* z = d + 8 * j;
          *reinterpret_cast<uint4*>(rowB + (2 * c + j) * kGrp) =
              make_uint4(pack_bf16(z[0], z[1]), pack_bf16(z[2], z[3]), pack_bf16(z[4], z[5]), pack_bf16(z[6], z[7]));
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) d[i] = to_tf32_fast(d[i]);
        st16(tL + kCQ + 16 * c, d);
      }
      wait_st();
      hand_over(fullA);
      TSTAMP(tlog, it, 11);

      // ---------------- S5 done: dZ1 = dH1 * (1 - H1^2) -> bufA (bf16, A of S6) ----------------
      {
        uint4 g1[8];                              // the stash does not depend on S5: read it while S5 runs
#pragma unroll
        for (int c = 0; c < 8; ++c) g1[c] = *reinterpret_cast<const uint4*>(rowG1 + c * kGrp);
        mbar_wait(doneA, phA); phA ^= 1; fence_after();
        TSTAMP(tlog, it, 12);
        float va[16], vb[16];
        ld16_issue(tL + kCP, va);
        ld_fence(va);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float (&v)[16] = (c & 1) ? vb : va;
          float (&w)[16] = (c & 1) ? va : vb;
          if (c < 3) ld16_issue(tL + kCP + 16 * (c + 1), w);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 g = g1[2 * c + j];
            float* z = v + 8 * j;
            // fp32 products, one rounding to bf16 (a bf16 product of bf16(dH1) and the stash measured slower and less accurate)
            mul2(z[0], z[1], bf16_lo(g.x), bf16_hi(g.x));
            mul2(z[2], z[3], bf16_lo(g.y), bf16_hi(g.y));
            mul2(z[4], z[5], bf16_lo(g.z), bf16_hi(g.z));
            mul2(z[6], z[7], bf16_lo(g.w), bf16_hi(g.w));
            *reinterpret_cast<uint4*>(rowA + (2 * c + j) * kGrp) =
                make_uint4(pack_bf16(z[0], z[1]), pack_bf16(z[2], z[3]), pack_bf16(z[4], z[5]), pack_bf16(z[6], z[7]));
          }
          if (c < 3) ld_fence(w);
        }
      }
      hand_over(fullA);                          // S6; awaited at the top of the next tile / after the loop
      row_cur = row_nxt;
      row_nxt = row_nn;
      TSTAMP(tlog, it, 13);
    }
    if (it > 0) { mbar_wait(doneA, phA); phA ^= 1; }
    fence_after();

    // ---------------- per-thread scalars: warp sums, then fixed-order sums over warps and warpgroups ----------------
#pragma unroll
    for (int q = 0; q < kNS; ++q) accs[q] = warp_sum(accs[q]);
    if (lane == 0) {
#pragma unroll
      for (int q = 0; q < kNS; ++q) S.wsum[wg][wq][q] = accs[q];
    }
    fence_before();
    asm volatile("bar.sync 1, %0;" :: "n"(kComputeThreads3) : "memory");     // every warpgroup's last S6 has completed
    fence_after();

    if (wg == 0) {          // warpgroup 0 reads the shared accumulators out: one partial vector per (tower, CTA)
      auto scalar = [&](int q) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kWG3; ++w) s += ((S.wsum[w][0][q] + S.wsum[w][1][q]) + S.wsum[w][2][q]) + S.wsum[w][3][q];
        return s;
      };
      // one CTA per tower (minibatches of up to 384 samples -- the reference's batch_size 64): the two towers own disjoint
      // entries of the gradient vector and write it directly, which saves the reduce launch (3 us of a ~23 us optimiser step)
      const bool direct = A.direct != nullptr;
      float* const outv = direct ? A.direct : A.partials + ((size_t)tw * gridDim.x + blockIdx.x) * kGradLen;
      const int oW1 = tw ? O_VF_W1 : O_PI_W1, oB1 = tw ? O_VF_B1 : O_PI_B1, oW2 = tw ? O_VF_W2 : O_PI_W2;
      const int oB2 = tw ? O_VF_B2 : O_PI_B2, oW3 = tw ? O_VF_W3 : O_PI_W3, oB3 = tw ? O_VF_B3 : O_PI_B3;
      const int nB3 = tw ? 1 : kAct;
      const uint32_t tA = S.tmem_base + ((uint32_t)(wq * 32) << 16);
      if (it == 0) {         // no tile in this CTA at all (warpgroup 0 owns the CTA's first tile)
        for (int idx = r; idx < oB3 + nB3 - oW1; idx += 128) outv[oW1 + idx] = 0.f;
        if (tw == 0 && r < kAct) outv[O_LOGSTD + r] = 0.f;
        if (r < kStats && (!direct || ((r == 1 || r == 4) == (tw == 1)))) outv[kParams + r] = 0.f;
      } else {
        const int j = 16 * wq + lane;               // accumulator row held by lanes 0..15 of each subpartition
        const bool own = lane < 16;
        float v[16];
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          ld16_issue(tA + kAcc2 + 16 * c, v);
          ld_fence(v);
          if (own) {
#pragma unroll
            for (int i = 0; i < 16; ++i) outv[oW2 + j * kHid + 16 * c + i] = v[i];
          }
        }
        ld16_issue(tA + kAcc2 + 64, v);             // columns 64..71 = dZ2^T . G: column 68 (the ones column) = db2; then dW1
        ld_fence(v);
        if (own) outv[oB2 + j] = v[4];
        ld16_issue(tA + kAcc1, v);
        ld_fence(v);
        if (own) {
#pragma unroll
          for (int i = 0; i < kObs; ++i) outv[oW1 + j * kObs + i] = v[i];
          outv[oB1 + j] = v[15];
        }
        ld16_issue(tA + kAcc3 - 8, v);              // columns 488..503: tail of dW1 (8) | dW3 (8)
        ld_fence(v);
        if (own) {
          if (tw == 0) {
#pragma unroll
            for (int o = 0; o < kAct; ++o) outv[oW3 + o * kHid + j] = v[8 + o];
          } else {
            outv[oW3 + j] = v[8];
          }
        }
        if (tw == 0) {
          if (r < kAct) { outv[O_LOGSTD + r] = scalar(r); outv[O_PI_B3 + r] = scalar(4 + r); }
          if (r < kStats && !(direct && (r == 1 || r == 4))) outv[kParams + r] = (r == 0) ? scalar(8) : (r == 2) ? scalar(9) : (r == 3) ? scalar(10) : 0.f;
        } else {
          if (r == 0) outv[O_VF_B3] = scalar(0);
          if (r < kStats && (!direct || r == 1 || r == 4)) outv[kParams + r] = (r == 1) ? scalar(1) : (r == 4) ? scalar(2) : 0.f;
        }
      }
    }
  }

  fence_before();
  __syncthreads();
  if (tid < 32)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(S.tmem_base), "r"((uint32_t)tcb::kTmem3) : "memory");
}

}  // namespace dronecu
