// ctk_predictor.cuh -- device predictors: s_{t+1} = f(s_t, Q_t)  (replaces PredictorWrapper.predict_core,
// reference call sites optimizer_mppi.py:188, optimizer_cem_tf.py:57, optimizer_rpgd.py:300).
//   OdePred     : CartPole Euler ODE, one thread per rollout, state in registers.
//   MlpSimtPred : 6 -> hidden tanh -> hidden tanh -> 5 MLP on the FP32 pipe (one thread per rollout, weights in
//                 shared memory).  Numerical anchor for the tcgen05 engines (ctk_mlp_tc.cuh).
#pragma once
#include "ctk_args.cuh"
#include "ctk_device.cuh"

namespace ctk {

struct OdePred {
  static constexpr bool kCooperative = false;
  static constexpr int kRolloutsPerBlock = 0;  // 0: every thread of the block carries a rollout
#ifndef CTK_ODE_MAX_THREADS
#define CTK_ODE_MAX_THREADS 1024
#endif
  static constexpr int kMaxThreads = CTK_ODE_MAX_THREADS;
  static constexpr int kCemThreads = 128;  // block size of the generic CEM rollout kernel
  static constexpr int kMinBlocks = 1;
  FwdK p;  // forward constants, register-resident (ctk_device.cuh load_fwd)
  __device__ __forceinline__ OdePred(const DevConsts* kc, const MlpDev&, float*) : p(load_fwd(kc)) {}
  // take the FMA-multiplier constants from kernel parameters (uniform registers) instead of vector registers
  __device__ __forceinline__ void use_uniform(const HotUK& u) { p.cU = u.cU; p.kTm = u.kTm; p.h = u.h; p.hk = u.hk; p.K1p = u.K1p; }
  // omc = 1 - cos(angle) of the new state (E_pot cost term)
  __device__ __forceinline__ void step(State& z, float u, float& omc) const { ode_step(z, u, p, omc); }
  // intermediate_steps == 1 fast path (no sub-step loop in the rollout's inner loop)
  __device__ __forceinline__ void substep(State& z, float u, float& omc) const { ode_substep(z, u, p, omc); }
  __device__ __forceinline__ bool single_substep() const { return p.isteps == 1; }
  __device__ __forceinline__ void begin_rollout(bool = true) {}  // stateless predictor
  __device__ __forceinline__ bool group_active(int, int) const { return true; }
  static constexpr bool kBalanced = false;
  static size_t smem_floats(const MlpDev&) { return 0; }
};

// tanh with ~1e-7 absolute error on the FP32 pipe + 2 MUFU ops: tanh(x) = 1 - 2/(exp(2x)+1)
__device__ __forceinline__ float tanh_acc(float x) {
  const float ax = fminf(fabsf(x), 15.0f);
  const float e = __expf(2.0f * ax);
  const float r = 1.0f - __fdividef(2.0f, e + 1.0f);
  // small |x|: the formula above cancels; use the odd series (|x| < 0.06: error < 1e-9)
  const float x2 = x * x;
  const float ser = x * fmaf(x2, fmaf(x2, 0.13333334f, -0.33333334f), 1.0f);
  return (ax < 0.06f) ? ser : copysignf(r, x);
}

// network outputs y (before the output bias b3) -> next state [angleD, cos, sin, position, positionD]; angle = atan2(sin, cos)
// (oracle/spec.py MLPPredictor.step).  b3 is a reference to the caller's member: an out-of-line step() re-reads it after each store
// through z (which may alias the functor), so its code is that of the same statements written in place
__device__ __forceinline__ void mlp_outputs_to_state(State& z, const float (&y)[5], const float* const& b3, float& omc) {
  z.om = y[0] + b3[0];
  z.c = y[1] + b3[1];
  z.s = y[2] + b3[2];
  z.x = y[3] + b3[3];
  z.v = y[4] + b3[4];
  z.th = atan2f(z.s, z.c);
  // the network's (cos, sin) outputs are not normalised: cos(atan2(s, c)) = c / hypot(s, c)
  omc = 1.0f - z.c * rsqrtf(fmaf(z.c, z.c, z.s * z.s));
}

struct MlpSimtPred {
  static constexpr bool kCooperative = false;
  static constexpr int kRolloutsPerBlock = 0;
  static constexpr int kMaxThreads = 128;
  static constexpr int kCemThreads = 128;
  static constexpr int kMinBlocks = 1;
  int hid;
  const float *W1, *b1, *W2, *b2, *W3T, *b3;  // shared memory
  __device__ __forceinline__ MlpSimtPred(const DevConsts*, const MlpDev& m, float* sm) {
    // 16-byte align the weight block
    float* base = (float*)(((uintptr_t)sm + 15) & ~(uintptr_t)15);
    hid = m.hidden;
    for (int i = threadIdx.x; i < m.blob_floats; i += blockDim.x) base[i] = m.blob[i];
    W1 = base;
    b1 = W1 + 6 * hid;
    W2 = b1 + hid;
    b2 = W2 + hid * hid;
    W3T = b2 + hid;
    b3 = W3T + 5 * hid;
    // caller issues __syncthreads() after construction
  }
  static size_t smem_floats(const MlpDev& m) { return (size_t)m.blob_floats + 4; }
  __device__ __forceinline__ void substep(State& z, float u, float& omc) const { step(z, u, omc); }
  __device__ __forceinline__ bool single_substep() const { return false; }
  __device__ __forceinline__ void use_uniform(const HotUK&) {}
  __device__ __forceinline__ void begin_rollout(bool = true) {}  // stateless predictor
  __device__ __forceinline__ bool group_active(int, int) const { return true; }
  static constexpr bool kBalanced = false;

  // net input [Q, angleD, cos, sin, position, positionD] -> next [angleD, cos, sin, position, positionD];
  // angle = atan2(sin, cos)  (oracle/spec.py MLPPredictor.step)
  __device__ __noinline__ void step(State& z, float u, float& omc) const {
    constexpr int HMAX = 128;
    float h1[HMAX];
    const float x[6] = {u, z.om, z.c, z.s, z.x, z.v};
#pragma unroll
    for (int j = 0; j < HMAX; ++j) {
      if (j < hid) {
        float acc = 0.0f;  // torch: (x @ W1) + b1 -> accumulate the dot product first, then add the bias
#pragma unroll
        for (int i = 0; i < 6; ++i) acc = fmaf(x[i], W1[i * hid + j], acc);
        h1[j] = tanh_acc(acc + b1[j]);
      }
    }
    float y[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j0 = 0; j0 < hid; j0 += 16) {
      float acc[16];
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) acc[jj] = 0.0f;
#pragma unroll
      for (int i = 0; i < HMAX; ++i) {
        if (i < hid) {
          const float4* wrow = reinterpret_cast<const float4*>(W2 + i * hid + j0);
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const float4 wv = wrow[v];
            acc[4 * v + 0] = fmaf(h1[i], wv.x, acc[4 * v + 0]);
            acc[4 * v + 1] = fmaf(h1[i], wv.y, acc[4 * v + 1]);
            acc[4 * v + 2] = fmaf(h1[i], wv.z, acc[4 * v + 2]);
            acc[4 * v + 3] = fmaf(h1[i], wv.w, acc[4 * v + 3]);
          }
        }
      }
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) {
        const float h2 = tanh_acc(acc[jj] + b2[j0 + jj]);
#pragma unroll
        for (int k = 0; k < 5; ++k) y[k] = fmaf(h2, W3T[k * hid + j0 + jj], y[k]);
      }
    }
    mlp_outputs_to_state(z, y, b3, omc);
  }
};

// ----------------------------------------------------------------------------------------------------------------
// GruSimtPred: stateful recurrent predictor, 6 -> GRU(hid) -> GRU(hid) -> Dense 5 on the FP32 pipe (SURVEY 8f.3; reference hook
// optimizer_mppi.py:195-197 predictor.update).  One thread per rollout; the weights (41 KB at hid = 32) and the per-rollout hidden
// state ([2 hid][threads], conflict-free) live in shared memory.  Every rollout starts from the handle's SAVED hidden state
// (MlpDev::rnn_h), which only gru_update_kernel advances (once per MPPI tick, with the measured state and the control about to be
// applied).  Cell (oracle/spec.py GRUPredictor, gate order [r, z, n]):
//   gi = x Wi + bi, gh = h Wh + bh;  r = sigmoid(gi_r + gh_r), z = sigmoid(gi_z + gh_z), n = tanh(gi_n + r gh_n), h' = (1 - z) n + z h
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

struct GruSimtPred {
  static constexpr bool kCooperative = false;
  static constexpr int kRolloutsPerBlock = 0;
  static constexpr int kMaxThreads = 128;
  static constexpr int kCemThreads = 128;
  static constexpr int kMinBlocks = 1;
  static constexpr int HMAX = 32;
  int hid;
  const float *Wi1, *Wh1, *bi1, *bh1, *Wi2, *Wh2, *bi2, *bh2, *W3T, *b3;  // shared memory
  float* hs;            // shared memory: this thread's hidden state, element j of layer l at hs[(l * HMAX + j) * kMaxThreads]
  const float* h_saved; // global: MlpDev::rnn_h row to start from
  __device__ __forceinline__ GruSimtPred(const DevConsts*, const MlpDev& m, float* sm, int row = 0) {
    float* base = (float*)(((uintptr_t)sm + 15) & ~(uintptr_t)15);
    hid = m.hidden;
    for (int i = threadIdx.x; i < m.blob_floats; i += blockDim.x) base[i] = m.blob[i];
    const int g = 3 * hid;
    Wi1 = base; Wh1 = Wi1 + 6 * g; bi1 = Wh1 + hid * g; bh1 = bi1 + g;
    Wi2 = bh1 + g; Wh2 = Wi2 + hid * g; bi2 = Wh2 + hid * g; bh2 = bi2 + g;
    W3T = bh2 + g; b3 = W3T + 5 * hid;
    hs = base + ((m.blob_floats + 3) & ~3) + (threadIdx.x % kMaxThreads);
    h_saved = m.rnn_h + (size_t)row * 2 * hid;
    // caller issues __syncthreads() after construction
  }
  static size_t smem_floats(const MlpDev& m) { return (size_t)((m.blob_floats + 3) & ~3) + 2 * HMAX * kMaxThreads + 8; }
  __device__ __forceinline__ void substep(State& z, float u, float& omc) { step(z, u, omc); }
  __device__ __forceinline__ bool single_substep() const { return false; }
  __device__ __forceinline__ void use_uniform(const HotUK&) {}
  __device__ __forceinline__ bool group_active(int, int) const { return true; }
  static constexpr bool kBalanced = false;
  // every rollout starts from the saved hidden state (SI_Toolkit's autoregressive RNN predictor restores it before predict_core)
  __device__ __forceinline__ void begin_rollout(bool = true) {
    for (int l = 0; l < 2; ++l)
      for (int j = 0; j < hid; ++j) hs[(l * HMAX + j) * kMaxThreads] = h_saved[l * hid + j];
  }

  // one GRU layer: x [NIN] (registers) and this thread's hidden state hl (shared, stride kMaxThreads) -> new hidden state in hl and out[]
  template <int NIN>
  __device__ __forceinline__ void cell(const float* x, int nin, float* hl, const float* Wi, const float* Wh, const float* bi,
                                       const float* bh, float* out) const {
    const int g3 = 3 * hid;
    float hold[HMAX];
#pragma unroll
    for (int i = 0; i < HMAX; ++i) hold[i] = (i < hid) ? hl[i * kMaxThreads] : 0.0f;
#pragma unroll
    for (int j0 = 0; j0 < HMAX; j0 += 8) {
      if (j0 < hid) {
        float gi[3][8], gh[3][8];
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) { gi[g][jj] = 0.0f; gh[g][jj] = 0.0f; }
#pragma unroll
        for (int i = 0; i < NIN; ++i) {
          if (i < nin) {
#pragma unroll
            for (int g = 0; g < 3; ++g) {
              const float4* w = reinterpret_cast<const float4*>(Wi + i * g3 + g * hid + j0);
              const float4 w0 = w[0], w1 = w[1];
              gi[g][0] = fmaf(x[i], w0.x, gi[g][0]); gi[g][1] = fmaf(x[i], w0.y, gi[g][1]);
              gi[g][2] = fmaf(x[i], w0.z, gi[g][2]); gi[g][3] = fmaf(x[i], w0.w, gi[g][3]);
              gi[g][4] = fmaf(x[i], w1.x, gi[g][4]); gi[g][5] = fmaf(x[i], w1.y, gi[g][5]);
              gi[g][6] = fmaf(x[i], w1.z, gi[g][6]); gi[g][7] = fmaf(x[i], w1.w, gi[g][7]);
            }
          }
        }
#pragma unroll
        for (int i = 0; i < HMAX; ++i) {
          if (i < hid) {
#pragma unroll
            for (int g = 0; g < 3; ++g) {
              const float4* w = reinterpret_cast<const float4*>(Wh + i * g3 + g * hid + j0);
              const float4 w0 = w[0], w1 = w[1];
              gh[g][0] = fmaf(hold[i], w0.x, gh[g][0]); gh[g][1] = fmaf(hold[i], w0.y, gh[g][1]);
              gh[g][2] = fmaf(hold[i], w0.z, gh[g][2]); gh[g][3] = fmaf(hold[i], w0.w, gh[g][3]);
              gh[g][4] = fmaf(hold[i], w1.x, gh[g][4]); gh[g][5] = fmaf(hold[i], w1.y, gh[g][5]);
              gh[g][6] = fmaf(hold[i], w1.z, gh[g][6]); gh[g][7] = fmaf(hold[i], w1.w, gh[g][7]);
            }
          }
        }
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int j = j0 + jj;
          const float r = sigmoid_acc(__fadd_rn(__fadd_rn(gi[0][jj], bi[j]), __fadd_rn(gh[0][jj], bh[j])));
          const float zz = sigmoid_acc(__fadd_rn(__fadd_rn(gi[1][jj], bi[hid + j]), __fadd_rn(gh[1][jj], bh[hid + j])));
          const float n = tanh_acc(__fadd_rn(__fadd_rn(gi[2][jj], bi[2 * hid + j]), __fmul_rn(r, __fadd_rn(gh[2][jj], bh[2 * hid + j]))));
          const float hn = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, zz), n), __fmul_rn(zz, hold[j]));
          out[j] = hn;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < HMAX; ++i)
      if (i < hid) hl[i * kMaxThreads] = out[i];
  }

  // net input [Q, angleD, cos, sin, position, positionD] -> next [angleD, cos, sin, position, positionD]; angle = atan2(sin, cos)
  __device__ __noinline__ void step(State& z, float u, float& omc) {
    const float x[6] = {u, z.om, z.c, z.s, z.x, z.v};
    float a1[HMAX], a2[HMAX];
    cell<6>(x, 6, hs, Wi1, Wh1, bi1, bh1, a1);
    cell<HMAX>(a1, hid, hs + HMAX * kMaxThreads, Wi2, Wh2, bi2, bh2, a2);
    float y[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < HMAX; ++j) {
      if (j < hid) {
#pragma unroll
        for (int k = 0; k < 5; ++k) y[k] = fmaf(a2[j], W3T[k * hid + j], y[k]);
      }
    }
    mlp_outputs_to_state(z, y, b3, omc);  // the same Dense read-out as the MLP
  }
};

}  // namespace ctk
