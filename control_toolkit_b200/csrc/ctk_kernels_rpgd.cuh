// ctk_kernels_rpgd.cuh -- K6/K7 forward tape + reverse-mode adjoint + Adam for the CartPole; K8 select / shift / resample
// (rpgd_select_body<1>, ctk_kernels_rpgd_select.cuh) fused into the coefficient-form kernel.
// Replaces reference optimizer_rpgd.py:306-338 (grad_step) and :340-380 (get_action) for one tick.  Population arrays are stored
// t-major ([H][N]) on the device so that one-thread-per-trajectory access is coalesced; the C-ABI transposes to the reference's [N,H,nu].
#pragma once
#include "ctk_device.cuh"
#include "ctk_kernels_rpgd_select.cuh"

namespace ctk {

// One thread = one trajectory.  Shared memory per thread: q[H], g[H], tape[H][6].
template <int KIND, bool LOG>
__global__ void __launch_bounds__(32) rpgd_grad_kernel(const RpgdGradArgs a) {
  extern __shared__ float smem[];
  const int B = blockDim.x, tid = threadIdx.x;
  float* sq = smem;                    // [H][B]
  float* sg = sq + (size_t)a.H * B;    // [H][B]
  float* tp = sg + (size_t)a.H * B;    // [H][6][B]
  const int n = blockIdx.x * B + tid;
  pdl_wait();
  pdl_trigger();
  if (n >= a.N) return;
  const float u_prev = a.u_prev[0];
  const float w = a.cost.inv_Hp1;
  State z0;
  z0.th = a.s0.ld(0); z0.om = a.s0.ld(1); z0.c = a.s0.ld(2); z0.s = a.s0.ld(3); z0.x = a.s0.ld(4); z0.v = a.s0.ld(5);
  const float omc0 = 1.0f - cosf(z0.th);

  for (int t = 0; t < a.H; ++t) sq[t * B + tid] = a.Q[(size_t)t * a.N + n];

  for (int it = 0; it < a.iters; ++it) {
    // ---- forward, storing the state tape (optimizer_rpgd.py:310-312 under the tape) ----
    State z = z0;
    for (int t = 0; t < a.H; ++t) {
      float* p = tp + (size_t)t * 6 * B + tid;
      p[0] = z.th; p[B] = z.om; p[2 * B] = z.c; p[3 * B] = z.s; p[4 * B] = z.x; p[5 * B] = z.v;
      float omc_unused;
      ode_step(z, sq[t * B + tid], a.fwd, omc_unused);
    }
    // ---- reverse: lambda_H = d(terminal)/ds = 0 (indicator); dJ/dQ_t (optimizer_rpgd.py:314) ----
    Adj lam = {0.f, 0.f, 0.f, 0.f};
    float nrm2 = 0.0f;
    for (int t = a.H - 1; t >= 0; --t) {
      const float* p = tp + (size_t)t * 6 * B + tid;
      State zt;
      zt.th = p[0]; zt.om = p[B]; zt.c = p[2 * B]; zt.s = p[3 * B]; zt.x = p[4 * B]; zt.v = p[5 * B];
      const float u = sq[t * B + tid];
      float g = ode_step_adjoint(zt, u, a.ode, lam);
      const float up = (t > 0) ? sq[(t - 1) * B + tid] : u_prev;
      const float un = (t < a.H - 1) ? sq[(t + 1) * B + tid] : 0.0f;
      g += stage_cost_adjoint_u(u, up, un, t < a.H - 1, a.cost, w);
      sg[t * B + tid] = g;
      nrm2 = fmaf(g, g, nrm2);
      if (t > 0) stage_cost_adjoint_state<KIND>(zt, zt.c, zt.s, a.cost, w, lam);
    }
    // ---- clip_by_norm over the trajectory (:315), Adam (:317), box clip (:319) ----
    const float l2 = sqrtf(nrm2);
    const float den = fmaxf(l2, a.gradmax_clip);
    const double step = (double)(a.adam_step0 + it + 1);
    const double bc1d = 1.0 - pow(a.beta1, step), bc2d = 1.0 - pow(a.beta2, step);
    const float b1 = (float)a.beta1, b2 = (float)a.beta2;
    const float omb1 = (float)(1.0 - a.beta1), omb2 = (float)(1.0 - a.beta2);
    const float bc1 = (float)bc1d, bc2 = (float)bc2d, eps = (float)a.eps;
    const float alpha = (float)((double)a.lr * sqrt(bc2d) / bc1d);  // Keras step size
    for (int t = 0; t < a.H; ++t) {
      const float g = sg[t * B + tid] * a.gradmax_clip / den;
      const size_t gi = (size_t)t * a.N + n;
      float mm = a.m[gi], vv = a.v[gi];
      float q = sq[t * B + tid];
      if (a.adam_form == 2) {
        // plain gradient descent on the clipped gradient, reference optimizer_cem_naive_grad_tf.py:72-74
        q = __fsub_rn(q, __fmul_rn(a.lr, g));
      } else if (a.adam_form == 1) {
        // torch form, reference optimizer_rpgd.py:56-82
        mm = fmaf(g, omb1, mm * b1);
        vv = fmaf(g * g, omb2, vv * b2);
        q = q - (a.lr * (mm / bc1)) / (sqrtf(vv / bc2) + eps);
      } else {
        // Keras form: m += (g-m)(1-b1); v += (g^2-v)(1-b2); var -= alpha * m / (sqrt(v)+eps)
        mm = fmaf(g - mm, omb1, mm);
        vv = fmaf(g * g - vv, omb2, vv);
        q = q - (alpha * mm) / (sqrtf(vv) + eps);
      }
      q = fminf(fmaxf(q, a.lo), a.hi);
      a.m[gi] = mm;
      a.v[gi] = vv;
      sq[t * B + tid] = q;
    }
  }

  // ---- get_action rollout (:342): cost of the updated population ----
  State z = z0;
  float omc = omc0, u_last = u_prev, jsum = 0.0f;
  for (int t = 0; t < a.H; ++t) {
    const float u = sq[t * B + tid];
    a.Q[(size_t)t * a.N + n] = u;
    if (LOG) {
      float* p = a.log_traj_soa + (size_t)t * 6 * a.N + n;
      p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
    }
    jsum += stage_cost<KIND>(z, omc, u, u_last, a.cost);
    ode_step(z, u, a.fwd, omc);
    u_last = u;
  }
  if (LOG) {
    float* p = a.log_traj_soa + (size_t)a.H * 6 * a.N + n;
    p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
  }
  a.J[n] = (jsum + terminal_cost(z, a.cost)) - a.cost.shift;
}

// The same tick with the adjoint in COEFFICIENT form (ctk_math.cuh adjoint_coefficients / adjoint_apply): the forward pass folds
// everything that depends on the pre-step state into 8 numbers per step, the reverse sweep is a 4-deep FMA chain per step, and
// every constant is register-resident (volatile loads from the device copy) instead of being re-read from the parameter bank
// inside the serial loops.  Block = 32 trajectories x kRpgdWarps warps: warp 0 walks the serial chains (5 x H dependent steps
// per tick -- chain depth IS the run time: the forward pass is the bare state recursion, the reverse sweep the 4-deep FMA
// chain), ALL warps share the phases that are parallel over the horizon (staging Q / Adam moments from global memory, the
// adjoint coefficients from the taped states, the Adam update with its IEEE divisions and square roots, the write-back),
// warp w taking the steps t = w (mod kRpgdWarps).
constexpr int kRpgdWarps = 8;
template <int KIND, bool LOG>
__global__ void __launch_bounds__(32 * kRpgdWarps) rpgd_grad_coef_kernel(const RpgdGradArgs a, const RpgdSelectArgs sel, const int fuse_select) {
  extern __shared__ float smem[];
  constexpr int B = 32, W = kRpgdWarps;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, H = a.H;
  float* sq = smem + lane;                   // [H][B]
  float* sg = sq + (size_t)H * B;            // [H][B]
  float* sm = sg + (size_t)H * B;            // [H][B] Adam first moment  (global loads issued up front by all warps;
  float* sv = sm + (size_t)H * B;            // [H][B] Adam second moment  written back once)
  float* tp = sv + (size_t)H * B;            // [H][8][B]
  __shared__ float sh_den[B];
  const int n_raw = blockIdx.x * B + lane;
  const bool active = n_raw < a.N;
  const int n = active ? n_raw : a.N - 1;    // inactive lanes shadow the last trajectory and never store to global memory
  const FwdK fwd = vload_struct(&a.kc->fwd);  // constants: independent of the previous kernel, loaded while it drains
  const OdeC p = vload_struct(&a.kc->ode);
  const CostC cost = vload_struct(&a.kc->cost);
  pdl_wait();
  pdl_trigger();
  const float u_prev = a.u_prev[0];
  const float w = cost.inv_Hp1;
  const float D2 = p.h * p.inv_mL_kp1L * p.neg_J_fric, KV = p.kp1 * p.neg_M_fric, KU = p.kp1 * p.u_max, hh = p.h;
  const float gu_a = w * 2.0f * (cost.cc_weight * cost.R), gu_b = w * 2.0f * cost.ccrc_weight;
  State z0;
  z0.th = a.s0.ld(0); z0.om = a.s0.ld(1); z0.c = a.s0.ld(2); z0.s = a.s0.ld(3); z0.x = a.s0.ld(4); z0.v = a.s0.ld(5);
  const float omc0 = 1.0f - cosf(z0.th);
  const float lo = a.lo, hi = a.hi, clipc = a.gradmax_clip, lr = a.lr;

  int tslot = 0;
  auto trace = [&]() {  // optional phase timeline (tools/rpgd_trace.py)
    if (a.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0 && tslot < 32) a.trace[tslot] = globaltimer_ns();
    ++tslot;
  };
  trace();
  const bool moments = a.adam_form != 2;
#pragma unroll 4
  for (int t = wid; t < H; t += W) {
    sq[t * B] = a.Q[(size_t)t * a.N + n];
    if (moments) { sm[t * B] = a.m[(size_t)t * a.N + n]; sv[t * B] = a.v[(size_t)t * a.N + n]; }
  }
  __syncthreads();
  trace();

  for (int it = 0; it < a.iters; ++it) {
    if (wid == 0) {
      // ---- forward (warp 0): the bare state chain, pre-step states to the tape ----
      State z = z0;
#pragma unroll 2
      for (int t = 0; t < H; ++t) {
        float* o = tp + (size_t)t * 8 * B;
        o[0] = z.th; o[B] = z.om; o[2 * B] = z.c; o[3 * B] = z.s; o[4 * B] = z.x; o[5 * B] = z.v;
        float omc_unused;
        ode_substep(z, sq[t * B], fwd, omc_unused);
      }
    }
    __syncthreads();
    trace();
    // ---- adjoint coefficients (all warps, step t by warp t mod W): each (step, trajectory) slot of the tape is read and then
    //      overwritten by the same thread, so the 8 coefficients replace the 6 state values in place ----
#pragma unroll 2
    for (int t = wid; t < H; t += W) {
      float* o = tp + (size_t)t * 8 * B;
      State z;
      z.th = o[0]; z.om = o[B]; z.c = o[2 * B]; z.s = o[3 * B]; z.x = o[4 * B]; z.v = o[5 * B];
      const AdjCoef c = adjoint_coefficients<KIND>(z, sq[t * B], p, cost, w);
      o[0] = c.E1; o[B] = c.E2; o[2 * B] = c.C1; o[3 * B] = c.C2; o[4 * B] = c.D1; o[5 * B] = c.cx; o[6 * B] = c.cth; o[7 * B] = c.com;
    }
    __syncthreads();
    trace();
    if (wid == 0) {
      // ---- reverse sweep ----
      Adj lam = {0.f, 0.f, 0.f, 0.f};
      float nrm2 = 0.0f;
#pragma unroll 4
      for (int t = H - 1; t >= 0; --t) {
        const float* o = tp + (size_t)t * 8 * B;
        AdjCoef c;
        c.E1 = o[0]; c.E2 = o[B]; c.C1 = o[2 * B]; c.C2 = o[3 * B]; c.D1 = o[4 * B]; c.cx = o[5 * B]; c.cth = o[6 * B]; c.com = o[7 * B];
        const float u = sq[t * B];
        const float up = (t > 0) ? sq[(t - 1) * B] : u_prev;
        // d(l_t)/d(u_t) + d(l_{t+1})/d(u_t)  (stage_cost_adjoint_u)
        float gu = fmaf(gu_b, u - up, gu_a * u);
        if (t < H - 1) gu = fmaf(-gu_b, sq[(t + 1) * B] - u, gu);
        const float g = adjoint_apply(c, hh, D2, KV, KU, t > 0, lam) + gu;
        sg[t * B] = g;
        nrm2 = fmaf(g, g, nrm2);
      }
      sh_den[lane] = fmaxf(sqrtf(nrm2), clipc);  // clip_by_norm over the trajectory
    }
    __syncthreads();
    trace();
    // ---- optimizer update, box clip: parallel over the horizon ----
    const float den = sh_den[lane];
    const float b1 = (float)a.beta1, b2 = (float)a.beta2;
    const float omb1 = (float)(1.0 - a.beta1), omb2 = (float)(1.0 - a.beta2), eps = (float)a.eps;
    float bc1, bc2, alpha;
    if (it < a.n_host_adam) {  // the double-precision pow / sqrt per thread cost ~1.5 us per gradient step (tools/rpgd_trace.py)
      bc1 = a.bc1_h[it]; bc2 = a.bc2_h[it]; alpha = a.alpha_h[it];
    } else {
      const double step = (double)(a.adam_step0 + it + 1);
      const double bc1d = 1.0 - pow(a.beta1, step), bc2d = 1.0 - pow(a.beta2, step);
      bc1 = (float)bc1d; bc2 = (float)bc2d;
      alpha = (float)((double)a.lr * sqrt(bc2d) / bc1d);
    }
#pragma unroll 2
    for (int t = wid; t < H; t += W) {
      const float g = sg[t * B] * clipc / den;
      float q = sq[t * B];
      if (!moments) {
        q = __fsub_rn(q, __fmul_rn(lr, g));
      } else {
        float mm = sm[t * B], vv = sv[t * B];
        if (a.adam_form == 1) {
          mm = fmaf(g, omb1, mm * b1);
          vv = fmaf(g * g, omb2, vv * b2);
          q = q - (lr * (mm / bc1)) / (sqrtf(vv / bc2) + eps);
        } else {
          mm = fmaf(g - mm, omb1, mm);
          vv = fmaf(g * g - vv, omb2, vv);
          q = q - (alpha * mm) / (sqrtf(vv) + eps);
        }
        sm[t * B] = mm;
        sv[t * B] = vv;
      }
      sq[t * B] = fminf(fmaxf(q, lo), hi);
    }
    __syncthreads();
    trace();
  }
  if (active) {
#pragma unroll 4
    for (int t = wid; t < H; t += W) {
      a.Q[(size_t)t * a.N + n] = sq[t * B];
      if (moments && a.iters > 0) { a.m[(size_t)t * a.N + n] = sm[t * B]; a.v[(size_t)t * a.N + n] = sv[t * B]; }
    }
  }
  trace();
  if (wid == 0 && active) {
    // ---- cost of the updated population ----
    State z = z0;
    float omc = omc0, u_last = u_prev, jsum = 0.0f;
    for (int t = 0; t < H; ++t) {
      const float u = sq[t * B];
      if (LOG) {
        float* o = a.log_traj_soa + (size_t)t * 6 * a.N + n;
        o[0] = z.th; o[a.N] = z.om; o[2 * a.N] = z.c; o[3 * a.N] = z.s; o[4 * (size_t)a.N] = z.x; o[5 * (size_t)a.N] = z.v;
      }
      jsum += stage_cost<KIND>(z, omc, u, u_last, cost);
      ode_substep(z, u, fwd, omc);
      u_last = u;
    }
    if (LOG) {
      float* o = a.log_traj_soa + (size_t)H * 6 * a.N + n;
      o[0] = z.th; o[a.N] = z.om; o[2 * a.N] = z.c; o[3 * a.N] = z.s; o[4 * (size_t)a.N] = z.x; o[5 * (size_t)a.N] = z.v;
    }
    a.J[n] = (jsum + terminal_cost(z, cost)) - cost.shift;
  }
  trace();
  if (fuse_select) {  // the population is this one block: argsort / shift / resample (K8) without a second launch
    __shared__ uint64_t sh_sel[32 * kRpgdWarps];
    __shared__ int sh_best[32 * kRpgdWarps];
    __syncthreads();  // J, Q, m, v of every trajectory are written (same block: visible after the barrier)
    rpgd_select_body<1>(sel, sh_sel, sh_best);
  }
  trace();
}

}  // namespace ctk
