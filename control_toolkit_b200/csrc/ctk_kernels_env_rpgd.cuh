// ctk_kernels_env_rpgd.cuh -- the gradient step of the gradient optimizers (RPGD, gradient-tf, the gradient-assisted CEM variants) on
// environments registered through the functor registry (ctk_kernels_env.cuh).  The CartPole gradient kernels (ctk_kernels_rpgd.cuh)
// are specialised for ns = 6 / nu = 1 and a coefficient-form adjoint; this is the general form: one thread per trajectory, the
// forward pass tapes the pre-step states in shared memory and the reverse sweep runs the environment's adjoint members
// (ctk_env_adjoint.h).  Population arrays are [H][NU][N] (flat column t * NU + c); clip_by_norm(axes=[1,2]) takes ONE norm over the
// horizon and the inputs together.  Select / init / grad-CEM sample and refit are shared with the CartPole
// (ctk_kernels_rpgd_select.cuh).
#pragma once
#include "ctk_kernels_env.cuh"
#include "ctk_kernels_rpgd_select.cuh"

namespace ctk {

// shared-memory floats per trajectory: pre-step states, q, g, m, v
__host__ __device__ constexpr int env_rpgd_tape_floats(int ns, int nu) { return ns + 4 * nu; }

// K6/K7 for an environment: `iters` gradient steps (forward tape, reverse sweep through the Env adjoint, clip_by_norm over the
// whole [H, NU] gradient, Adam / descent, per-input box clip), then the cost of the updated population (_get_action :342).
// fuse_select: the population is this one block, K8 follows in the same launch.
template <class Env, bool LOG>
__global__ void __launch_bounds__(kEnvRpgdBlock) env_rpgd_grad_kernel(const EnvRpgdGradArgs a, const RpgdSelectArgs sel, const int fuse_select) {
  constexpr int NS = Env::NS, NU = Env::NU, B = kEnvRpgdBlock;
  extern __shared__ float smem[];
  const int tid = threadIdx.x, H = a.H, HC = a.H * NU;
  float* ss = smem + tid;               // [H][NS][B] pre-step states
  float* sq = ss + (size_t)H * NS * B;  // [H][NU][B]
  float* sg = sq + (size_t)HC * B;      // [H][NU][B] gradient
  float* sm = sg + (size_t)HC * B;      // [H][NU][B] Adam first moment
  float* sv = sm + (size_t)HC * B;      // [H][NU][B] Adam second moment
  const int n = blockIdx.x * B + tid;
  if (n < a.N) {
    float s0[NS], up0[NU];
#pragma unroll
    for (int i = 0; i < NS; ++i) s0[i] = a.s0.p != nullptr ? a.s0.p[i] : a.s0.v[i];
#pragma unroll
    for (int c = 0; c < NU; ++c) up0[c] = a.u_prev[c];
    const float w = 1.0f / (float)(H + 1);  // Cost_Functions/__init__.py:90-92 mean over H + 1
    const bool moments = a.adam_form != 2;
    for (int i = 0; i < HC; ++i) {
      const size_t gi = (size_t)i * a.N + n;
      sq[i * B] = a.Q[gi];
      if (moments) { sm[i * B] = a.m[gi]; sv[i * B] = a.v[gi]; }
    }
    for (int it = 0; it < a.iters; ++it) {
      // ---- forward, pre-step states to the tape (optimizer_rpgd.py:310-312 under the tape) ----
      float s[NS];
#pragma unroll
      for (int i = 0; i < NS; ++i) s[i] = s0[i];
      for (int t = 0; t < H; ++t) {
        float u[NU];
#pragma unroll
        for (int c = 0; c < NU; ++c) u[c] = sq[(t * NU + c) * B];
#pragma unroll
        for (int i = 0; i < NS; ++i) ss[(t * NS + i) * B] = s[i];
        Env::step(s, u, a.env);
      }
      // ---- reverse sweep: lambda_H = d(w T)/d(s_H); dJ/dQ_t (optimizer_rpgd.py:314) ----
      float lam[NS], carry[NU];
      Env::terminal_cost_grad(s, a.env, w, lam);
#pragma unroll
      for (int c = 0; c < NU; ++c) carry[c] = 0.0f;
      float nrm2 = 0.0f;
      for (int t = H - 1; t >= 0; --t) {
        float st[NS], u[NU], up[NU], gu[NU], gp[NU];
#pragma unroll
        for (int i = 0; i < NS; ++i) st[i] = ss[(t * NS + i) * B];
#pragma unroll
        for (int c = 0; c < NU; ++c) {
          u[c] = sq[(t * NU + c) * B];
          up[c] = t > 0 ? sq[((t - 1) * NU + c) * B] : up0[c];
          gu[c] = carry[c];  // d(w l_{t+1})/d(u_t) through the control-change term
          gp[c] = 0.0f;
        }
        Env::step_adjoint(st, u, a.env, lam, gu);
        Env::stage_cost_grad(st, u, up, a.env, w, lam, gu, gp);
#pragma unroll
        for (int c = 0; c < NU; ++c) {
          sg[(t * NU + c) * B] = gu[c];
          nrm2 = fmaf(gu[c], gu[c], nrm2);
          carry[c] = gp[c];
        }
      }
      // ---- clip_by_norm over the trajectory (:315), Adam (:317), per-input box clip (:319) ----
      const float den = fmaxf(sqrtf(nrm2), a.gradmax_clip);
      const float b1 = (float)a.beta1, b2 = (float)a.beta2;
      const float omb1 = (float)(1.0 - a.beta1), omb2 = (float)(1.0 - a.beta2), eps = (float)a.eps;
      float bc1, bc2, alpha;
      if (it < a.n_host_adam) {
        bc1 = a.bc1_h[it]; bc2 = a.bc2_h[it]; alpha = a.alpha_h[it];
      } else {
        const double step = (double)(a.adam_step0 + it + 1);
        const double bc1d = 1.0 - pow(a.beta1, step), bc2d = 1.0 - pow(a.beta2, step);
        bc1 = (float)bc1d; bc2 = (float)bc2d;
        alpha = (float)((double)a.lr * sqrt(bc2d) / bc1d);
      }
      for (int t = 0; t < H; ++t) {
#pragma unroll
        for (int c = 0; c < NU; ++c) {
          const int i = t * NU + c;
          const float g = sg[i * B] * a.gradmax_clip / den;
          float q = sq[i * B];
          if (!moments) {
            q = __fsub_rn(q, __fmul_rn(a.lr, g));  // optimizer_cem_naive_grad_tf.py:72-74
          } else {
            float mm = sm[i * B], vv = sv[i * B];
            if (a.adam_form == 1) {  // torch form, optimizer_rpgd.py:56-82
              mm = fmaf(g, omb1, mm * b1);
              vv = fmaf(g * g, omb2, vv * b2);
              q = q - (a.lr * (mm / bc1)) / (sqrtf(vv / bc2) + eps);
            } else {  // Keras form
              mm = fmaf(g - mm, omb1, mm);
              vv = fmaf(g * g - vv, omb2, vv);
              q = q - (alpha * mm) / (sqrtf(vv) + eps);
            }
            sm[i * B] = mm;
            sv[i * B] = vv;
          }
          sq[i * B] = fminf(fmaxf(q, a.lo[c]), a.hi[c]);
        }
      }
    }
    for (int i = 0; i < HC; ++i) {
      const size_t gi = (size_t)i * a.N + n;
      a.Q[gi] = sq[i * B];
      if (moments && a.iters > 0) { a.m[gi] = sm[i * B]; a.v[gi] = sv[i * B]; }
    }
    // ---- cost of the updated population (:342) ----
    float s[NS], ul[NU], jsum = 0.0f;
#pragma unroll
    for (int i = 0; i < NS; ++i) s[i] = s0[i];
#pragma unroll
    for (int c = 0; c < NU; ++c) ul[c] = up0[c];
    for (int t = 0; t < H; ++t) {
      float u[NU];
#pragma unroll
      for (int c = 0; c < NU; ++c) {
        u[c] = sq[(t * NU + c) * B];
        if (LOG) a.log_Q[((size_t)n * H + t) * NU + c] = u[c];
      }
      if (LOG) env_log_state<Env>(a.log_traj, n, t, H, s);
      jsum += Env::stage_cost(s, u, ul, a.env);
      Env::step(s, u, a.env);
#pragma unroll
      for (int c = 0; c < NU; ++c) ul[c] = u[c];
    }
    if (LOG) env_log_state<Env>(a.log_traj, n, H, H, s);
    a.J[n] = (jsum + Env::terminal_cost(s, a.env)) / (float)(H + 1);
  }
  if (fuse_select) {  // one block holds the population: argsort / shift / resample without a second launch
    __shared__ uint64_t sh_sel[B];
    __shared__ int sh_best[B];
    __syncthreads();  // J, Q, m, v of every trajectory are written (same block: visible after the barrier)
    rpgd_select_body<NU>(sel, sh_sel, sh_best);
  }
}

}  // namespace ctk
