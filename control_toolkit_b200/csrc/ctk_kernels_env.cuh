// ctk_kernels_env.cuh -- MPPI and CEM ticks for environments registered through the functor registry (SURVEY 8f.3): an environment is
// a struct with NS states, NU control inputs and three device functions (step, stage_cost, terminal_cost) over a flat parameter block.
// The reference's contract is "any predictor + any Control_Toolkit_ASF.Cost_Functions.<env>.<name>" (reference
// Cost_Functions/cost_function_wrapper.py:59-66) with any num_control_inputs (Optimizers/optimizer_mppi.py:173-175,
// optimizer_cem_tf.py:64-65); the CartPole kernels (K1 .. K5) are specialised for ns = 6 / nu = 1, these are the general form:
// one thread per rollout, state and controls in registers, the same counter-based noise blocks (draw index = C order over
// [n_ind or H, nu]), the same top-k (K4) for CEM.  Multi-launch and unsharded: the latency work of the CartPole ticks is not repeated.
#pragma once
#include "ctk_device.cuh"
#include "ctk_env_adjoint.h"
#include "ctk_topk.cuh"

namespace ctk {

// ---- Dubins car: [x, y, yaw], [throttle, steer]; oracle/spec.py dubins_step / DubinsCost; adjoint: ctk_env_adjoint.h -----------
struct DubinsEnv : DubinsAdjoint {
  static constexpr int NS = 3, NU = 2;
  // p: 0 h  1 v_max  2 omega_max  3 dd_weight  4 obstacle_weight  5 cc_weight * R  6 ccrc_weight  7 terminal_weight
  //    8 target_x  9 target_y  10 obstacle_x  11 obstacle_y  12 obstacle_r^2  13 MAX_COST
  static __device__ __forceinline__ void step(float* s, const float* u, const EnvParams& e) {
    const float v = __fmul_rn(e.p[1], u[0]), w = __fmul_rn(e.p[2], u[1]);
    float sn, cs;
    sincosf(s[2], &sn, &cs);
    s[0] = __fadd_rn(s[0], __fmul_rn(__fmul_rn(v, cs), e.p[0]));
    s[1] = __fadd_rn(s[1], __fmul_rn(__fmul_rn(v, sn), e.p[0]));
    const float yaw = __fadd_rn(s[2], __fmul_rn(w, e.p[0]));
    sincosf(yaw, &sn, &cs);
    s[2] = atan2f(sn, cs);  // wrap to (-pi, pi]
  }
  static __device__ __forceinline__ float stage_cost(const float* s, const float* u, const float* up, const EnvParams& e) {
    const float dx = s[0] - e.p[8], dy = s[1] - e.p[9];
    const float dd = __fmul_rn(e.p[3], __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    const float ox = s[0] - e.p[10], oy = s[1] - e.p[11];
    const float obs = (__fadd_rn(__fmul_rn(ox, ox), __fmul_rn(oy, oy)) < e.p[12]) ? e.p[4] : 0.0f;
    const float cc = __fmul_rn(e.p[5], __fadd_rn(__fmul_rn(u[0], u[0]), __fmul_rn(u[1], u[1])));
    const float d0 = u[0] - up[0], d1 = u[1] - up[1];
    const float ccrc = __fmul_rn(e.p[6], __fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)));
    return __fadd_rn(__fadd_rn(__fadd_rn(dd, obs), cc), ccrc) - e.p[13];
  }
  static __device__ __forceinline__ float terminal_cost(const float* s, const EnvParams& e) {
    const float dx = s[0] - e.p[8], dy = s[1] - e.p[9];
    return __fmul_rn(e.p[7], __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
  }
};

template <class Env>
__device__ __forceinline__ void env_log_state(float* log_traj, int n, int t, int H, const float* s) {
#pragma unroll
  for (int i = 0; i < Env::NS; ++i) log_traj[((size_t)n * (H + 1) + t) * Env::NS + i] = s[i];
}

// Compensated (Kahan) sum.  The MPPI correction adds 3 H NU terms into one total that enters the softmin unscaled: at H NU = 1024 a
// plain fp32 running sum is ~4e-4 off (totals ~60), which moves the weights exp(-(S - rho) / LBD) at LBD = 1 and put u_nom 4.6e-5 from
// float64 where the reference's fp32 evaluation is 1e-6 away (tests/test_gpu_env_ticks.py, H = 512).  The _rn intrinsics keep the
// compiler from contracting or reassociating the compensation.
struct KahanSum {
  float s = 0.0f, c = 0.0f;
  __device__ __forceinline__ void add(float x) {
    const float y = __fsub_rn(x, c);
    const float t = __fadd_rn(s, y);
    c = __fsub_rn(__fsub_rn(t, s), y);
    s = t;
  }
};

// ---- MPPI: sample -> rollout -> cost (reference optimizer_mppi.py:170-193 up to the total cost S) ----------------------------
template <class Env, bool LOG>
__global__ void __launch_bounds__(128) env_mppi_rollout_kernel(const EnvMppiArgs a) {
  constexpr int NS = Env::NS, NU = Env::NU;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.N) return;
  const uint32_t ng = (uint32_t)(a.off + n);
  float s[NS], up[NU];
#pragma unroll
  for (int i = 0; i < NS; ++i) s[i] = a.s0.p != nullptr ? a.s0.p[i] : a.s0.v[i];
#pragma unroll
  for (int c = 0; c < NU; ++c) up[c] = a.u_prev[c];
  float jsum = 0.0f;
  KahanSum corr;
  float y0[NU], y1[NU];
  for (int t = 0; t < a.H; ++t) {
    const int seg = t / a.period, j = t - seg * a.period;
    if (j == 0) {  // :173-175 normal * stdev on the inducing points seg, seg + 1 (draw index = point * NU + input)
#pragma unroll
      for (int c = 0; c < NU; ++c) {
        y0[c] = __fmul_rn(noise1(a.noise, ng, seg * NU + c), a.stdev);
        y1[c] = (seg + 1 < a.n_ind) ? __fmul_rn(noise1(a.noise, ng, (seg + 1) * NU + c), a.stdev) : 0.0f;
      }
    }
    float w0, w1;
    interp_weights(seg, j, a.period, a.n_ind, &w0, &w1);  // Interpolator.py:63-74 incl. the last-point quirk
    float u[NU];
#pragma unroll
    for (int c = 0; c < NU; ++c) {
      const float du = fmaf(y1[c], w1, __fmul_rn(y0[c], w0));                                  // Interpolator.py:97-106
      const float un = a.u_nom[(size_t)min(t + 1, a.H - 1) * NU + c];                          // :184 shift on read
      u[c] = fminf(fmaxf(__fadd_rn(un, du), a.lo[c]), a.hi[c]);                                // :186-187
      // :154-155  cc_weight * (0.5 (1 - 1/NU) R du^2 + R u du + 0.5 R u^2)
      corr.add(__fmul_rn(__fmul_rn(du, du), a.k_du2));
      corr.add(__fmul_rn(__fmul_rn(u[c], du), a.k_udu));
      corr.add(__fmul_rn(__fmul_rn(u[c], u[c]), a.k_uu));
      if (LOG) a.log_Q[((size_t)n * a.H + t) * NU + c] = u[c];
    }
    if (LOG) env_log_state<Env>(a.log_traj, n, t, a.H, s);
    jsum += Env::stage_cost(s, u, up, a.env);
    Env::step(s, u, a.env);
#pragma unroll
    for (int c = 0; c < NU; ++c) up[c] = u[c];
  }
  if (LOG) env_log_state<Env>(a.log_traj, n, a.H, a.H, s);
  // Cost_Functions/__init__.py:90-92 (mean over H+1 incl. the terminal cost) + the MPPI correction (optimizer_mppi.py:160)
  a.J[n] = __fadd_rn((jsum + Env::terminal_cost(s, a.env)) / (float)(a.H + 1), corr.s);
}

// ---- MPPI: softmin weights, weighted perturbation average on the inducing points, u_nom update (optimizer_mppi.py:163-168,190-191).
// One block: the population minimum, then every thread accumulates its rollouts' weight and weighted draws (regenerated from the
// counter-based noise), block reduction in a fixed order, interpolation of the n_ind x NU sums (linear: equals the interpolated average).
constexpr int kEnvMaxDraws = 32;  // n_ind * NU
template <int NU>
__global__ void __launch_bounds__(1024) env_mppi_update_kernel(const EnvMppiArgs a) {
  __shared__ float sh_red[32];
  __shared__ float sh_b[kEnvMaxDraws + 1];
  __shared__ float sh_unom[1024];
  const int tid = threadIdx.x, D = a.n_ind * NU;
  float mn = INFINITY;
  for (int n = tid; n < a.N; n += blockDim.x) mn = fminf(mn, a.J[n]);
  const float rho = block_min(mn, sh_red);
  float acc_a = 0.0f, acc_b[kEnvMaxDraws];
#pragma unroll
  for (int d = 0; d < kEnvMaxDraws; ++d) acc_b[d] = 0.0f;
  for (int n = tid; n < a.N; n += blockDim.x) {
    const float S = a.J[n];
    if (!(S < INFINITY)) continue;
    const float w = expf((S - rho) * a.neg_inv_lbd);  // :165
    acc_a += w;
    const uint32_t ng = (uint32_t)(a.off + n);
#pragma unroll
    for (int blk = 0; blk < kEnvMaxDraws / 4; ++blk) {
      if (blk * 4 < D) {
        float zz[4];
        noise4(a.noise, ng, (uint32_t)blk, zz);
#pragma unroll
        for (int q = 0; q < 4; ++q) acc_b[blk * 4 + q] = fmaf(w, zz[q], acc_b[blk * 4 + q]);
      }
    }
  }
  const float tot_a = block_sum(acc_a, sh_red);
#pragma unroll
  for (int d = 0; d < kEnvMaxDraws; ++d) {
    if (d < D) {
      const float t = block_sum(acc_b[d], sh_red);
      if (tid == 0) sh_b[d] = t;
    }
  }
  for (int i = tid; i < a.H * NU; i += blockDim.x) sh_unom[i] = a.u_nom[(size_t)min(i / NU + 1, a.H - 1) * NU + (i % NU)];  // :184
  __syncthreads();
  for (int i = tid; i < a.H * NU; i += blockDim.x) {
    const int t = i / NU, c = i - t * NU;
    const int seg = t / a.period, j = t - seg * a.period;
    float w0, w1;
    interp_weights(seg, j, a.period, a.n_ind, &w0, &w1);
    const float bz0 = sh_b[seg * NU + c];
    const float bz1 = (j > 0) ? sh_b[(seg + 1) * NU + c] : 0.0f;
    const float b = (fmaf(bz1, w1, bz0 * w0) * a.stdev) / tot_a;                      // :167
    const float un = fminf(fmaxf(sh_unom[i] + b, a.lo[c]), a.hi[c]);                   // :190
    a.u_nom[i] = un;
    if (t == 0) {                                                                      // :191 u = u_nom[0, 0, :]
      if (!a.freeze_prev) a.u_prev[c] = un;
      if (a.u_out != nullptr) a.u_out[c] = un;
    }
  }
}

// ---- CEM: sample -> rollout -> cost (reference optimizer_cem_tf.py:54-70); flat column index = t * NU + input -----------------
template <class Env, bool LOG>
__global__ void __launch_bounds__(128) env_cem_rollout_kernel(const EnvCemArgs a) {
  constexpr int NS = Env::NS, NU = Env::NU;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.N) return;
  const uint32_t ng = (uint32_t)(a.off + n);
  float s[NS], up[NU];
#pragma unroll
  for (int i = 0; i < NS; ++i) s[i] = a.s0.p != nullptr ? a.s0.p[i] : a.s0.v[i];
#pragma unroll
  for (int c = 0; c < NU; ++c) up[c] = a.u_prev[c];
  float jsum = 0.0f;
  float zz[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t = 0; t < a.H; ++t) {
    float u[NU];
#pragma unroll
    for (int c = 0; c < NU; ++c) {
      const int d = t * NU + c;
      if ((d & 3) == 0) noise4(a.noise, ng, (uint32_t)(d >> 2), zz);
      const int q = d & 3;
      const float z = q == 0 ? zz[0] : (q == 1 ? zz[1] : (q == 2 ? zz[2] : zz[3]));
      u[c] = fminf(fmaxf(__fadd_rn(a.mu[d], __fmul_rn(z, a.sd[d])), a.lo[c]), a.hi[c]);        // :64-66
      if (LOG) a.log_Q[((size_t)n * a.H + t) * NU + c] = u[c];
    }
    if (LOG) env_log_state<Env>(a.log_traj, n, t, a.H, s);
    jsum += Env::stage_cost(s, u, up, a.env);
    Env::step(s, u, a.env);
#pragma unroll
    for (int c = 0; c < NU; ++c) up[c] = u[c];
  }
  if (LOG) env_log_state<Env>(a.log_traj, n, a.H, a.H, s);
  a.J[n] = (jsum + Env::terminal_cost(s, a.env)) / (float)(a.H + 1);
}

// ---- CEM: merge the candidate keys -> global top-k, regenerate the elite rows, refit mean / population std per column, post-loop
// clip / shift by one time step (= NU columns), u = the best sample's first action (optimizer_cem_tf.py:73-78,99-102) ------------
static __global__ void __launch_bounds__(TOPK_THREADS) env_cem_refit_kernel(const EnvCemRefitArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ uint32_t sh_elite[TOPK_THREADS];
  uint64_t key = KEY_MAX;
  if ((int)threadIdx.x < a.cnt) key = a.cand[threadIdx.x];
  int n_sort = 32;
  while (n_sort < a.cnt) n_sort <<= 1;
  key = block_bitonic_sort(key, sh, n_sort);
  if ((int)threadIdx.x < a.k) {
    sh_elite[threadIdx.x] = (uint32_t)(key & 0xffffffffu);
    if (a.elite_idx_out != nullptr) a.elite_idx_out[threadIdx.x] = (int32_t)(key & 0xffffffffu);
  }
  __syncthreads();
  const int col = threadIdx.x, HC = a.H * a.nu;
  float new_mu = 0.0f, new_sd = 0.0f, first_q = 0.0f;
  if (col < HC) {
    const int c = col % a.nu;
    const float mu = a.mu[col], sd = a.sd[col];
    float acc = 0.0f;
    for (int e = 0; e < a.k; ++e) {
      const float q = fminf(fmaxf(__fadd_rn(mu, __fmul_rn(noise1(a.noise, sh_elite[e], col), sd)), a.lo[c]), a.hi[c]);
      if (e == 0) first_q = q;
      acc += q;
    }
    new_mu = acc / (float)a.k;
    float var = 0.0f;
    for (int e = 0; e < a.k; ++e) {
      const float q = fminf(fmaxf(__fadd_rn(mu, __fmul_rn(noise1(a.noise, sh_elite[e], col), sd)), a.lo[c]), a.hi[c]);
      const float d = q - new_mu;
      var = fmaf(d, d, var);
    }
    new_sd = sqrtf(var / (float)a.k);
  }
  __syncthreads();  // every column has read the old mu / sd
  if (col < HC) {
    const int c = col % a.nu;
    if (!a.last) {
      a.mu[col] = new_mu;
      a.sd[col] = new_sd;
    } else {
      const float sdc = fminf(fmaxf(new_sd, a.sd_min), 1.0e8f);
      if (col >= a.nu) {
        a.mu[col - a.nu] = new_mu;
        a.sd[col - a.nu] = sdc;
      } else {
        if (!a.freeze_prev) a.u_prev[c] = first_q;
        if (a.u_out != nullptr) a.u_out[c] = first_q;
      }
      if (col >= HC - a.nu) {
        a.mu[col] = (a.lo[c] + a.hi[c]) * 0.5f;
        a.sd[col] = a.sd_init;
      }
    }
  }
}

}  // namespace ctk
