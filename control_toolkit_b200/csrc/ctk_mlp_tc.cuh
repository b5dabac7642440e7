// ctk_mlp_tc.cuh -- tcgen05 (UMMA + TMEM) engines of the MLP predictor (6 -> 128 tanh -> 128 tanh -> 5, config C4).
// Replaces PredictorWrapper.predict_core for the neural predictor (reference call sites optimizer_mppi.py:188,
// optimizer_cem_tf.py:57).  Drop-in `Pred`s of the generic rollout kernels (ctk_kernels_mppi.cuh).  Both structures run ONE CTA per
// SM with several 128-rollout tiles in flight (a tile = the M dimension of an MMA), give every CTA an equal contiguous share of the
// population, and run layer 1 on the tensor core (one K = 48 operand row of split inputs per rollout against the resident B1):
//   MlpTcFastPredT (tcgen05_bf16, tcgen05_fast): four tiles, one per warp group, one thread per rollout; layer 2 as ONE bf16
//                                                 product (8 UMMAs per tile-step);
//   MlpTcPred      (tcgen05, fp32-level):        two tiles, an owner and a helper thread per rollout; layer 2 as the six significant
//                                                 products of three-term bf16 splits of h1 and W2, issued by K-quarters (48 UMMAs).
// Layer 3 (128 -> 5) runs on the FP32 pipe from the accumulator rows (tcgen05.ld).  Measurements and the earlier structures: DESIGN §5.2.
#pragma once
#include <cuda_bf16.h>

#include "ctk_args.cuh"
#include "ctk_device.cuh"
#include "ctk_predictor.cuh"

namespace ctk {

constexpr int kTcHidden = 128;
constexpr uint32_t kTcTileBytes = 128 * 128 * 2;  // one bf16 operand tile [128 rows][128 k]
constexpr uint32_t kTcKStride = 2048;             // bytes between core matrices along K  (descriptor LBO)
constexpr uint32_t kTcMnStride = 128;             // bytes between 8-row groups along M/N (descriptor SBO)
// byte offset of element (row, k) inside an operand tile: 8x8 core matrices of 16-byte rows
__host__ __device__ inline uint32_t tc_tile_offset(int row, int k) { return (uint32_t)(k >> 3) * kTcKStride + (uint32_t)row * 16u + (uint32_t)(k & 7) * 2u; }
// device blob: W2 split tiles [3][32768 B] | W1 [6][128] | b1 [128] | b2 [128] | W3T [5][128] | b3 [8]   (floats after the tiles)
constexpr uint32_t kTcBlobFloats = 6 * 128 + 128 + 128 + 5 * 128 + 8;
// ... | B1 [6 k-groups][128 n][8] bf16 (layer 1 on the tensor core): rows of K = 48: W1 term 1 three times (x1, x2, x3), W1 term 2
// twice (x1, x2), W1 term 3 (x1), the three terms of b1 (against 1.0), zeros
constexpr uint32_t kTcB1Bytes = 6 * kTcKStride;
constexpr uint32_t kTcBlobBytes = 3 * kTcTileBytes + kTcBlobFloats * 4 + kTcB1Bytes;
// instruction descriptor of every MMA here: D fp32, A/B bf16, both K-major, N = 128, M = 128
constexpr uint32_t kTcIdescM128N128 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr) {
  // SmemDescriptor (sm_100): start address, leading / stride byte offsets in 16-byte units, version 1, no swizzle
  return (uint64_t)((saddr >> 4) & 0x3fffu) | ((uint64_t)(kTcKStride >> 4) << 16) | ((uint64_t)(kTcMnStride >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the MMAs this thread has issued so far -> one arrival on the mbarrier at shared address `bar` when they complete
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one lane spins until the mbarrier at shared address `bar` has completed the phase of the given parity
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  }
}
// 16 consecutive fp32 columns of this thread's TMEM lane (accumulator row), starting at `taddr`; waits for the load
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// the CTA's TMEM for its lifetime: warp 0 allocates NCOLS columns (base address -> *slot) and gives up the allocation permit
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc_cta(uint32_t* slot) {
  if ((threadIdx.x >> 5) == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(NCOLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
}
// called by every thread of the CTA: after the CTA's last tcgen05 operation, warp 0 frees the columns of tmem_alloc_cta
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc_cta(const uint32_t* slot) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(*slot), "n"(NCOLS) : "memory");
  }
}

// tanh(x) = 1 - 2 / (exp(2x) + 1) for either sign (x -> -inf: e -> 0, t -> -1; x -> +inf: e -> inf, r -> 0, t -> 1):
// FMUL, MUFU.EX2, FADD, MUFU.RCP, FFMA.  Absolute error <= ~3e-7 (the two MUFU approximations), the same bound the
// FP32-pipe engine's tanh_acc has outside its small-|x| series branch.
__device__ __forceinline__ float tanh5(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.8853900817779268f));  // exp(2x) = 2^(2x log2 e)
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
  return fmaf(-2.0f, r, 1.0f);
}
__device__ __forceinline__ float4 lds4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts4(uint32_t addr, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(w0), "r"(w1), "r"(w2), "r"(w3) : "memory");
}
// three bf16 terms of two floats by TRUNCATION (x = t1 + t2 + t3 + O(2^-24 x), every residual exact): the high halves are
// picked by PRMT, the residuals by LOP3 + FADD -- ALU / FMA pipes only, the conversion unit stays free for the MUFU tanh
__device__ __forceinline__ void split3(float a0, float a1, uint32_t& p1, uint32_t& p2, uint32_t& p3) {
  const uint32_t u0 = __float_as_uint(a0), u1 = __float_as_uint(a1);
  p1 = __byte_perm(u0, u1, 0x7632);
  const float r0 = a0 - __uint_as_float(u0 & 0xffff0000u), r1 = a1 - __uint_as_float(u1 & 0xffff0000u);
  const uint32_t v0 = __float_as_uint(r0), v1 = __float_as_uint(r1);
  p2 = __byte_perm(v0, v1, 0x7632);
  const float s0 = r0 - __uint_as_float(v0 & 0xffff0000u), s1 = r1 - __uint_as_float(v1 & 0xffff0000u);
  p3 = __byte_perm(__float_as_uint(s0), __float_as_uint(s1), 0x7632);
}
// layer-1 operand row of one rollout at shared address `arow`: [x1 x2 x3 x1 x2 x1 | 1 1 1 | 0 ...], the three-term bf16 split of the
// six inputs [Q, angleD, cos, sin, position, positionD]; K = 48 = six 16-byte k-groups of the K-major core-matrix layout
__device__ __forceinline__ void store_l1_operand_row(uint32_t arow, float u, const State& z) {
  uint32_t p1[3], p2[3], p3[3];
  split3(u, z.om, p1[0], p2[0], p3[0]);
  split3(z.c, z.s, p1[1], p2[1], p3[1]);
  split3(z.x, z.v, p1[2], p2[2], p3[2]);
  sts4(arow + 0u * kTcKStride, p1[0], p1[1], p1[2], p2[0]);          // k  0.. 7: x1[0..5] x2[0..1]
  sts4(arow + 1u * kTcKStride, p2[1], p2[2], p3[0], p3[1]);          // k  8..15: x2[2..5] x3[0..3]
  sts4(arow + 2u * kTcKStride, p3[2], p1[0], p1[1], p1[2]);          // k 16..23: x3[4..5] x1[0..5]
  sts4(arow + 3u * kTcKStride, p2[0], p2[1], p2[2], p1[0]);          // k 24..31: x2[0..5] x1[0..1]
  sts4(arow + 4u * kTcKStride, p1[1], p1[2], 0x3f803f80u, 0x00003f80u);  // k 32..39: x1[2..5] 1 1 1 0
  sts4(arow + 5u * kTcKStride, 0u, 0u, 0u, 0u);                      // k 40..47
}
// layer 3 over one 16-column chunk of this thread's layer-2 accumulator row (TMEM address `taddr`, hidden units [c0, c0 + 16)):
// bias b2, activation ACT, five FMAs per column into the partial outputs y
template <float (*ACT)(float)>
__device__ __forceinline__ void fold_l3_chunk(uint32_t taddr, int c0, uint32_t ab2, uint32_t aW3, float (&y)[5]) {
  uint32_t v[16];
  tmem_ld16(taddr, v);
#pragma unroll
  for (int q4 = 0; q4 < 4; ++q4) {
    const uint32_t jo = (uint32_t)(c0 + q4 * 4) * 4u;
    const float4 bb = lds4(ab2 + jo);
    const float h0 = ACT(__uint_as_float(v[4 * q4]) + bb.x), h1 = ACT(__uint_as_float(v[4 * q4 + 1]) + bb.y);
    const float h2 = ACT(__uint_as_float(v[4 * q4 + 2]) + bb.z), h3 = ACT(__uint_as_float(v[4 * q4 + 3]) + bb.w);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const float4 w = lds4(aW3 + (uint32_t)k * 512u + jo);
      y[k] = fmaf(h3, w.w, fmaf(h2, w.z, fmaf(h1, w.y, fmaf(h0, w.x, y[k]))));
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Opt-in reduced-precision engines of the same predictor (SURVEY section 7 hard part 4: "ship exact and fast variants, report both"):
// layer 2 as ONE bf16 product (h1 and W2 rounded to bfloat16, round to nearest even; fp32 accumulation in TMEM) -- 8 UMMAs per
// step instead of 48, one 32 KB operand tile per side instead of three.  APPROX = false ("tcgen05_bf16"): tanh as in the exact
// engine; parity is defined against an oracle that applies the same operand rounding (oracle/spec.py MLPPredictor bf16_layer2).
// APPROX = true ("tcgen05_fast"): tanh by the single-instruction MUFU.TANH (tanh.approx.f32, ~2^-11 relative): half the MUFU work;
// reported against the exact engine, not held to a parity bound.
//
// Structure (round 2): ONE CTA per SM with FOUR 128-rollout tiles in flight, one per warp group (4 warps = 128 threads = the M
// dimension of an MMA).  A thread owns its rollout completely -- layer 1 for all 128 hidden units of its row, its row of the A tile,
// its accumulator row out of TMEM, layer 3, the state update and the cost -- so there is no partial-sum exchange, no input broadcast
// and NO block-wide barrier inside a step: a group synchronises only with itself (two named barriers of 128 threads and the
// mbarrier its own MMAs commit to).  The four groups drift apart by construction, so one group's MUFU / FP32 stages run underneath
// another's UMMAs and TMEM loads (the first version of this engine ran the tensor core, the MUFU and the FP32 pipe mostly one after
// another: 27 % of the stall samples on block barriers, profiles/prof_mlp_tc_r01c_summary.txt).  Each CTA takes an equal share of the
// population (kBalanced: 65536 rollouts / 148 SMs = 442.8 -> 14 warps of rows per SM; warps without rows skip the arithmetic), which
// removes the 3.46-waves tail of 512 tiles on 148 SMs.  TMEM: the CTA allocates all 512 columns, 128 per group.
// Layer 1 (6 -> 128) runs on the tensor core too, at fp32-level accuracy: the thread splits its six inputs into three bf16 terms and
// writes ONE 96-byte operand row [x1 x2 x3 x1 x2 x1 | 1 1 1 | 0..] (K = 48); against B1 = [w1 w1 w1 w2 w2 w3 | b1 terms | 0..] three
// K16 UMMAs deliver the six significant products of the split plus the bias -- 900 FP32-pipe instructions per rollout-step less
// (the loaded SM sub-partitions were issue-bound: 4 warps x 2700 instructions per step, profiles/prof_mlp_tc_r02a_pipe_fast_summary.txt).
// ---------------------------------------------------------------------------------------------------------------
template <bool APPROX>
struct MlpTcFastPredT {
  static constexpr bool kCooperative = true;   // every thread of an ACTIVE group must call step() the same number of times
  static constexpr bool kBalanced = true;      // CTA b rolls out the contiguous share [b N / grid, (b + 1) N / grid) of the population
  static constexpr int kMaxThreads = 512;      // 4 warp groups x 128 threads, every thread owns a rollout
  static constexpr int kCemThreads = 512;
  static constexpr int kMinBlocks = 1;
  static constexpr int kRolloutsPerBlock = 512;
  static constexpr size_t kAccSmemBytes = 32 * 1024;  // what the tiles leave of the 227 KB for the MPPI accumulators [n_ind][512]
  uint8_t* sA;        // this group's bf16 tile of h1 [32768]
  uint8_t* sB;        // [32768] W2 rounded to bf16 (resident, shared by the groups)
  const float *W1, *b1, *b2, *W3T, *b3;
  uint64_t* mbar;     // this group's MMA-completion barrier
  uint32_t* tmem_slot;
  uint32_t phase;
  bool row_on;        // this thread's rollout is a real one (warps without any skip the arithmetic of a step)

  uint8_t* sB1;       // [12288] layer-1 operand (W1 / b1 split terms, resident, shared by the groups)

  static size_t smem_floats(const MlpDev&) { return (5 * (size_t)kTcTileBytes + kTcB1Bytes + kTcBlobFloats * 4 + 64 + 1024) / 4; }

  __device__ __forceinline__ MlpTcFastPredT(const DevConsts*, const MlpDev& m, float* sm) {
    uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)sm + 1023) & ~(uintptr_t)1023);
    const int g = threadIdx.x >> 7;
    sA = base + (size_t)g * kTcTileBytes;
    sB = base + 4 * (size_t)kTcTileBytes;
    sB1 = sB + kTcTileBytes;
    {
      const uint4* src1 = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(m.tc_blob) + 3 * kTcTileBytes + kTcBlobFloats * 4);
      uint4* dst1 = reinterpret_cast<uint4*>(sB1);
      for (int i = threadIdx.x; i < (int)(kTcB1Bytes / 16); i += blockDim.x) dst1[i] = src1[i];
    }
    float* f = reinterpret_cast<float*>(sB1 + kTcB1Bytes);
    W1 = f; b1 = W1 + 6 * 128; b2 = b1 + 128; W3T = b2 + 128; b3 = W3T + 5 * 128;
    uint64_t* mb0 = reinterpret_cast<uint64_t*>(f + kTcBlobFloats);  // [4]
    mbar = mb0 + g;
    tmem_slot = reinterpret_cast<uint32_t*>(mb0 + 4);
    phase = 0;
    row_on = true;
    // blob: [3 split tiles of W2][floats]; tile 0 is bf16_rn(W2), the float block follows the three tiles
    const uint4* src = reinterpret_cast<const uint4*>(m.tc_blob);
    uint4* dst = reinterpret_cast<uint4*>(sB);
    for (int i = threadIdx.x; i < (int)(kTcTileBytes / 16); i += blockDim.x) dst[i] = src[i];
    const uint4* srcf = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(m.tc_blob) + 3 * kTcTileBytes);
    uint4* dstf = reinterpret_cast<uint4*>(f);
    for (int i = threadIdx.x; i < (int)(kTcBlobFloats * 4 / 16); i += blockDim.x) dstf[i] = srcf[i];
    if (threadIdx.x < 4) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mb0 + threadIdx.x)) : "memory");
    if (threadIdx.x == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_alloc_cta<512>(tmem_slot);  // the CTA owns the SM: all 512 TMEM columns, 128 per group
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    // caller issues __syncthreads() after construction
  }
  __device__ __forceinline__ ~MlpTcFastPredT() { tmem_dealloc_cta<512>(tmem_slot); }
  __device__ __forceinline__ void substep(State& z, float u, float& omc) { step(z, u, omc); }
  __device__ __forceinline__ bool single_substep() const { return false; }
  __device__ __forceinline__ void use_uniform(const HotUK&) {}
  __device__ __forceinline__ void begin_rollout(bool active = true) { row_on = active; }
  // a group runs a pass of the rollout loop iff its first row is a real rollout (group-uniform: the group's barriers stay matched)
  __device__ __forceinline__ bool group_active(int base, int end) const { return base + (int)(threadIdx.x & ~127u) < end; }

  static __device__ __forceinline__ float act(float x) {
    if (APPROX) {
      float t;
      asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x));
      return t;
    }
    return tanh5(x);
  }
  static __device__ __forceinline__ uint32_t pack2(float lo, float hi) {  // two floats -> bf16x2 (RN-even), first element in the low half
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
  }

  __device__ __forceinline__ void step(State& z, float u, float& omc) {
    const int tid = threadIdx.x, g = tid >> 7, row = tid & 127, wq = (tid >> 5) & 3;
    const uint32_t ab2 = smem_u32(b2), aW3 = smem_u32(W3T);
    const bool warp_on = __any_sync(0xffffffffu, row_on);
    const uint32_t arow = smem_u32(sA) + (uint32_t)row * 16u;
    const uint32_t tmem_g = *tmem_slot + (uint32_t)g * 128u;
    const uint32_t trow = tmem_g + ((uint32_t)(wq * 32) << 16);
    // the group's first thread issues nk K16 UMMAs (A from the group's tile, B from b_base) and commits them to the group's mbarrier;
    // one lane of the group's first warp waits for them, the other three warps sleep in the hardware barrier that follows
    auto mma_round = [&](uint32_t b_base, int nk) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // operand rows -> visible to the tensor core (async proxy)
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // (also orders this thread's TMEM loads before the new MMAs)
      asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");        // the group's operand tile is complete
      if (row == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a0 = smem_u32(sA);
        for (int ks = 0; ks < nk; ++ks)
          umma_bf16(tmem_g, umma_smem_desc(a0 + (uint32_t)ks * 2u * kTcKStride), umma_smem_desc(b_base + (uint32_t)ks * 2u * kTcKStride), kTcIdescM128N128, ks > 0 ? 1u : 0u);
        umma_commit(smem_u32(mbar));
      }
      if (wq == 0) {
        if ((tid & 31) == 0) mbar_wait(smem_u32(mbar), phase);
        __syncwarp();
      }
      phase ^= 1u;
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.sync %0, 128;" ::"r"(5 + g) : "memory");        // the group's accumulator is complete
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // ---- layer 1 on the tensor core: this thread's operand row ----
    if (warp_on) store_l1_operand_row(arow, u, z);
    mma_round(smem_u32(sB1), 3);
    // ---- accumulator row (x W1 + b1) -> activation -> bf16 -> this thread's row of the group's A tile ----
    if (warp_on) {
#pragma unroll 2
      for (int c0 = 0; c0 < 128; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(trow + (uint32_t)c0, v);
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) pk[j] = pack2(act(__uint_as_float(v[2 * j])), act(__uint_as_float(v[2 * j + 1])));
        sts4(arow + (uint32_t)(c0 >> 3) * kTcKStride, pk[0], pk[1], pk[2], pk[3]);
        sts4(arow + (uint32_t)((c0 >> 3) + 1) * kTcKStride, pk[4], pk[5], pk[6], pk[7]);
      }
    }
    // ---- layer 2 on the tensor core: 8 UMMAs (M128 N128 K16) ----
    mma_round(smem_u32(sB), 8);
    if (!warp_on) return;
    // ---- this thread's accumulator row -> bias + activation -> layer 3 -> next state ----
    float y[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
    for (int c0 = 0; c0 < 128; c0 += 16) fold_l3_chunk<act>(trow + (uint32_t)c0, c0, ab2, aW3, y);
    mlp_outputs_to_state(z, y, b3, omc);
  }
};
using MlpTcBf16Pred = MlpTcFastPredT<false>;
using MlpTcFastPred = MlpTcFastPredT<true>;

// ---------------------------------------------------------------------------------------------------------------
// The exact (fp32-level) engine, round-2 structure: the tile-per-warp-group organisation of the single-product engines above with
// six-product bf16 x 3 arithmetic.  TWO 128-rollout tiles in flight per SM (groups), each worked on by 256 threads:
// the 128 OWNER threads (one per rollout: operand row of layer 1, state, cost) and 128 HELPER threads; owner and helper of a row split
// the row's columns in the FP32 / MUFU stages (the row's 512 MUFU operations per step at 8 cycles per warp instruction are the longest
// link of a tile's serial chain: with one thread per row the two tiles ran the tensor core, the MUFU and the FP32 pipe one after
// another -- 2.20 ms per C4 tick, profiles/prof_mlp_tc_r02_exact_v2_summary.txt: tensor 34 %, XU 37 %, issue 34 %, 27 % barrier stalls).
//   layer 1 : on the tensor core (three K16 UMMAs on the K = 48 split operand row, B1 resident) -> L1 accumulator, TMEM columns
//             [0, 128) of the group;
//   layer 2 : K is processed in QUARTERS: owner and helper read 16 columns each of the row's L1 accumulator, apply tanh, split the
//             values into three bf16 terms and write them into one of the group's two quarter buffers (3 terms x 4 k-groups = 24 KB;
//             three full A tiles, 96 KB per tile in flight, would allow only one tile per SM); the group's first
//             thread then issues that quarter's 12 UMMAs (six products x two K16 slices, smallest products first) into the L2
//             accumulator, TMEM columns [128, 256), and commits them to the buffer's mbarrier -- the tensor core works on quarter p
//             while the group's threads produce quarter p + 1 (TMEM load, MUFU, split) and while the OTHER group is in any phase;
//   layer 3 : owner and helper fold 64 columns each of the row's L2 accumulator (bias, tanh, five FMAs per column); the helper hands
//             its five partial sums to the owner through shared memory (aliasing quarter buffer 1, free by then).
// Shared memory: 2 groups x 2 x 24 KB quarter buffers + W2 split tiles 96 KB + B1 12 KB + 6.5 KB of fp32 weights = 211 KB.
// TMEM: 512 columns, 256 per group.  Synchronisation per step and group: six 256-thread named barriers and the mbarrier waits
// (one polling lane per warp; a quarter's MMAs have normally completed by the time its buffer is needed again).
// ---------------------------------------------------------------------------------------------------------------
struct MlpTcPred {
  static constexpr bool kCooperative = true;   // every thread of an ACTIVE group must call step() the same number of times
  static constexpr bool kBalanced = true;      // CTA b rolls out the contiguous share [b N / grid, (b + 1) N / grid) of the population
  static constexpr int kGroups = 2;
  static constexpr int kMaxThreads = 256 * kGroups;  // threads [0, 128 kGroups) own a rollout, the rest are the rows' helpers
  static constexpr int kCemThreads = 256 * kGroups;
  static constexpr int kMinBlocks = 1;
  static constexpr int kRolloutsPerBlock = 128 * kGroups;
  static constexpr size_t kAccSmemBytes = 12 * 1024;  // what the buffers leave of the 227 KB for the MPPI accumulators [n_ind][256]
  static constexpr uint32_t kQBuf = 3u * 4u * kTcKStride;  // one K-quarter (four k-groups) of the three split terms: 24 KB
  uint8_t* sA;        // this group's two quarter buffers [2][kQBuf]; buffer 0 also takes the layer-1 operand rows (six k-groups)
  uint8_t* sB;        // [3][32768] W2 split tiles (resident, shared by the groups)
  uint8_t* sB1;       // [12288] layer-1 operand (W1 / b1 split terms, resident)
  const float *W1, *b1, *b2, *W3T, *b3;
  uint64_t* mbar;     // this group's barriers: [0] layer-1 MMAs, [1] / [2] the MMAs reading quarter buffer 0 / 1
  uint32_t* tmem_slot;
  uint32_t phase;     // parity of the layer-1 barrier (the quarter barriers complete two phases per step: parities 0, 1 every step)
  int grp, half;      // tile of this thread; 0 = owner of row (tid & 127), 1 = its helper
  int tile_rows;      // real rollouts of the pass in flight over the whole CTA (rows >= tile_rows are padding)
  bool row_on;        // this thread's row is a real rollout (warps without any skip the arithmetic of a step)

  static size_t smem_floats(const MlpDev&) { return (kGroups * 2 * (size_t)kQBuf + kTcBlobBytes + 128 + 1024) / 4; }

  __device__ __forceinline__ MlpTcPred(const DevConsts*, const MlpDev& m, float* sm) {
    uint8_t* base = reinterpret_cast<uint8_t*>(((uintptr_t)sm + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x;
    half = tid >= 128 * kGroups ? 1 : 0;
    grp = ((tid - half * 128 * kGroups) >> 7);
    sA = base + (size_t)grp * 2 * kQBuf;
    sB = base + (size_t)kGroups * 2 * kQBuf;
    float* f = reinterpret_cast<float*>(sB + 3 * kTcTileBytes);
    W1 = f; b1 = W1 + 6 * 128; b2 = b1 + 128; W3T = b2 + 128; b3 = W3T + 5 * 128;
    sB1 = reinterpret_cast<uint8_t*>(f + kTcBlobFloats);
    uint64_t* mb0 = reinterpret_cast<uint64_t*>(sB1 + kTcB1Bytes);  // [kGroups][4]
    mbar = mb0 + 4 * grp;
    tmem_slot = reinterpret_cast<uint32_t*>(mb0 + 4 * kGroups);
    phase = 0;
    tile_rows = 128 * kGroups;
    row_on = true;
    // the blob has the resident layout: W2 split tiles | fp32 weights | B1
    const uint4* src = reinterpret_cast<const uint4*>(m.tc_blob);
    uint4* dst = reinterpret_cast<uint4*>(sB);
    for (int i = threadIdx.x; i < (int)(kTcBlobBytes / 16); i += blockDim.x) dst[i] = src[i];
    if (threadIdx.x < 4 * kGroups) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mb0 + threadIdx.x)) : "memory");
    if (threadIdx.x == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tmem_alloc_cta<512>(tmem_slot);  // the CTA owns the SM: all 512 TMEM columns, 256 per group (layer-1 and layer-2 accumulators)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    // caller issues __syncthreads() after construction
  }
  __device__ __forceinline__ ~MlpTcPred() { tmem_dealloc_cta<512>(tmem_slot); }
  __device__ __forceinline__ void substep(State& z, float u, float& omc) { step(z, u, omc); }
  __device__ __forceinline__ bool single_substep() const { return false; }
  __device__ __forceinline__ void use_uniform(const HotUK&) {}
  // (helpers are never `active` in the kernels' sense: their row's state follows from the pass's row count)
  __device__ __forceinline__ void begin_rollout(bool = true) { row_on = grp * 128 + (int)(threadIdx.x & 127u) < tile_rows; }
  // a group runs a pass of the rollout loop iff its first row is a real rollout (group-uniform: the group's barriers stay matched)
  __device__ __forceinline__ bool group_active(int base, int end) { tile_rows = end - base; return grp * 128 < tile_rows; }

  __device__ __forceinline__ void step(State& z, float u, float& omc) {
    const int tid = threadIdx.x, g = grp, row = tid & 127, wq = (tid >> 5) & 3;
    const uint32_t ab2 = smem_u32(b2), aW3 = smem_u32(W3T);
    const bool warp_on = __any_sync(0xffffffffu, row_on);
    const uint32_t a_grp = smem_u32(sA);
    const uint32_t arow = a_grp + (uint32_t)row * 16u;
    const uint32_t tmem_g = *tmem_slot + (uint32_t)g * 256u;
    const uint32_t trow = tmem_g + ((uint32_t)(wq * 32) << 16);
    const uint32_t bar0 = smem_u32(mbar);
    const bool issuer = (row == 0) && (half == 0);
    // operand rows written by this group -> visible to the tensor core; then the group's named barrier
    auto publish = [&]() {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");  // (also orders this thread's TMEM loads before the new MMAs)
      asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
    };
    // one lane per warp polls the mbarrier, the warp's other lanes wait at the warp barrier
    auto wait_mbar = [&](uint32_t bar, uint32_t parity) {
      if ((tid & 31) == 0) mbar_wait(bar, parity);
      __syncwarp();
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // ---- layer 1 on the tensor core: the owner's operand row, at the start of quarter buffer 0, which the previous step's MMAs have
    //      released ----
    if (warp_on && half == 0) store_l1_operand_row(arow, u, z);
    publish();
    if (issuer) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t b1a = smem_u32(sB1);
#pragma unroll
      for (int ks = 0; ks < 3; ++ks)
        umma_bf16(tmem_g, umma_smem_desc(a_grp + (uint32_t)ks * 2u * kTcKStride), umma_smem_desc(b1a + (uint32_t)ks * 2u * kTcKStride), kTcIdescM128N128, ks > 0 ? 1u : 0u);
      umma_commit(bar0);
    }
    wait_mbar(bar0, phase);
    phase ^= 1u;
    // ---- layer 2, one K-quarter at a time: L1 accumulator columns [32 p + 16 half, + 16) -> tanh -> three bf16 terms -> quarter
    //      buffer p & 1 -> 12 UMMAs into the L2 accumulator (TMEM columns [128, 256)) ----
    const uint32_t b2t = smem_u32(sB);
#pragma unroll 1
    for (int p = 0; p < 4; ++p) {
      const uint32_t bsel = (uint32_t)(p & 1);
      if (p >= 2) wait_mbar(bar0 + 8u * (1u + bsel), 0u);  // the MMAs of quarter p - 2 have released this buffer
      const uint32_t brow = arow + bsel * kQBuf;
      if (warp_on) {
        uint32_t v[16];
        tmem_ld16(trow + (uint32_t)(32 * p + 16 * half), v);
        uint32_t q1[8], q2[8], q3[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          split3(tanh5(__uint_as_float(v[2 * j])), tanh5(__uint_as_float(v[2 * j + 1])), q1[j], q2[j], q3[j]);
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          const uint32_t dst = brow + (uint32_t)(2 * half + kk) * kTcKStride;
          sts4(dst, q1[4 * kk], q1[4 * kk + 1], q1[4 * kk + 2], q1[4 * kk + 3]);
          sts4(dst + 4u * kTcKStride, q2[4 * kk], q2[4 * kk + 1], q2[4 * kk + 2], q2[4 * kk + 3]);
          sts4(dst + 8u * kTcKStride, q3[4 * kk], q3[4 * kk + 1], q3[4 * kk + 2], q3[4 * kk + 3]);
        }
      }
      publish();
      if (issuer) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t abuf = a_grp + bsel * kQBuf;
#pragma unroll
        for (int term = 0; term < 6; ++term) {  // smallest products first: (a3 w1) (a2 w2) (a1 w3) (a2 w1) (a1 w2) (a1 w1)
          constexpr int ta[6] = {2, 1, 0, 1, 0, 0}, tb[6] = {0, 1, 2, 0, 1, 0};
#pragma unroll
          for (int ks = 0; ks < 2; ++ks)
            umma_bf16(tmem_g + 128u, umma_smem_desc(abuf + (uint32_t)ta[term] * 4u * kTcKStride + (uint32_t)ks * 2u * kTcKStride),
                      umma_smem_desc(b2t + (uint32_t)tb[term] * kTcTileBytes + (uint32_t)(2 * p + ks) * 2u * kTcKStride), kTcIdescM128N128,
                      (p > 0 || term > 0 || ks > 0) ? 1u : 0u);
        }
        umma_commit(bar0 + 8u * (1u + bsel));
      }
    }
    wait_mbar(bar0 + 8u, 1u);   // quarter 2 (buffer 0 is free for the next step's layer-1 rows)
    wait_mbar(bar0 + 16u, 1u);  // quarter 3: the L2 accumulator is complete (and quarter buffer 1 is free: partial-sum exchange)
    // ---- the row's L2 accumulator, columns [64 half, + 64) -> bias + tanh -> layer 3 partial sums ----
    float y[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    if (warp_on) {
#pragma unroll 2
      for (int c0 = 64 * half; c0 < 64 * half + 64; c0 += 16) fold_l3_chunk<tanh5>(trow + 128u + (uint32_t)c0, c0, ab2, aW3, y);
    }
    // helper -> owner: five partial sums per row through quarter buffer 1 ([128 rows][8 floats])
    float* sy = reinterpret_cast<float*>(sA + kQBuf) + row * 8;
    if (half == 1 && warp_on) {
      reinterpret_cast<float4*>(sy)[0] = make_float4(y[0], y[1], y[2], y[3]);
      sy[4] = y[4];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("bar.sync %0, 256;" ::"r"(1 + g) : "memory");
    if (half == 1 || !warp_on) return;
    {
      const float4 v0 = reinterpret_cast<const float4*>(sy)[0];
      y[0] += v0.x; y[1] += v0.y; y[2] += v0.z; y[3] += v0.w; y[4] += sy[4];
    }
    mlp_outputs_to_state(z, y, b3, omc);
  }
};
#endif  // __CUDACC__


}  // namespace ctk
