// ctk_kernels_env_rpgd.cuh -- the gradient optimizers (RPGD, gradient-tf, the gradient-assisted CEM variants) on environments
// registered through the functor registry (ctk_kernels_env.cuh).  The CartPole kernels (ctk_kernels_rpgd.cuh) are specialised for
// ns = 6 / nu = 1 and a coefficient-form adjoint; these are the general form: one thread per trajectory, the forward pass tapes the
// pre-step states in shared memory and the reverse sweep runs the environment's adjoint members (ctk_env_adjoint.h).
// Population arrays are [H][NU][N] (flat column t * NU + c).  Reference semantics for nu > 1 (DESIGN section 2):
//  - sample_actions draws [B, n_ind, nu] in C order: draw index = point * NU + input (as env MPPI);
//  - clip_by_norm(axes=[1,2]) takes ONE norm over the horizon and the inputs together;
//  - the Adam moments shift by one time step (NU columns) with zero fill, whatever shift_previous is;
//  - the gradient-tf tail redraw is [N, 1, nu] uniform in [low_c, high_c];
//  - grad-CEM refits mean and std per (t, c) column and shifts by one time step after the loop.
#pragma once
#include "ctk_kernels_env.cuh"

namespace ctk {

// shared-memory floats per trajectory: pre-step states, q, g, m, v
__host__ __device__ constexpr int env_rpgd_tape_floats(int ns, int nu) { return ns + 4 * nu; }

// v[c] for a run-time c without a local-memory copy of the parameter array
template <int NU>
__device__ __forceinline__ float env_pick(const float* v, int c) {
  float r = v[0];
#pragma unroll
  for (int i = 1; i < NU; ++i) r = c == i ? v[i] : r;
  return r;
}

// sample_actions (optimizer_rpgd.py:275-296) for input c of inducing point p of a new row: clip(z * scale + offset) per input
__device__ __forceinline__ float env_rpgd_sample_point(const EnvRpgdSelectArgs& a, uint32_t row, int d, int c) {
  const float z = noise1(a.noise, row, d);
  const float y = a.dist == 0 ? __fadd_rn(__fmul_rn(z, a.s_std), a.s_mean) : __fadd_rn(__fmul_rn(z, a.s_max[c] - a.s_min[c]), a.s_min[c]);
  return fminf(fmaxf(y, a.lo[c]), a.hi[c]);
}
// column (t, c) of a freshly sampled row: interpolated clipped inducing points (Interpolator.py:97-106)
template <int NU>
__device__ __forceinline__ float env_rpgd_sample_column(const EnvRpgdSelectArgs& a, uint32_t row, int t, int c) {
  const int seg = t / a.period, j = t - seg * a.period;
  float w0, w1;
  interp_weights(seg, j, a.period, a.n_ind, &w0, &w1);
  const float y0 = env_rpgd_sample_point(a, row, seg * NU + c, c);
  const float y1 = (j > 0) ? env_rpgd_sample_point(a, row, (seg + 1) * NU + c, c) : 0.0f;
  return fmaf(y1, w1, __fmul_rn(y0, w0));
}

// K8 for NU columns (rpgd_select_body): argsort, u / u_nom of the best row, shift / resample / moment shift into the next buffers.
// Any block size >= the padded population; every thread of the block takes part.
template <int NU>
__device__ __forceinline__ void env_rpgd_select_body(const EnvRpgdSelectArgs& a, uint64_t* sh, int* sh_best) {
  const int tid = threadIdx.x, HC = a.H * NU;
  uint64_t key = (tid < a.N) ? make_key(a.J[tid], (uint32_t)tid) : KEY_MAX;
  int n_sort = 32;
  while (n_sort < a.N) n_sort <<= 1;
  key = block_bitonic_sort(key, sh, n_sort);  // argsort (:345), stable by index
  if (tid < a.k) {
    sh_best[tid] = (int)(key & 0xffffffffu);
    a.best_idx_out[tid] = sh_best[tid];
  }
  __syncthreads();
  const int best = sh_best[0];
  for (int i = tid; i < HC; i += blockDim.x) {
    const float q = a.Q[(size_t)i * a.N + best];
    a.u_nom_out[i] = q;  // :426
    if (i < NU) {        // :523 u = u_nom[0, 0, :]
      if (!a.freeze_prev) a.u_prev[i] = q;
      if (a.u_out != nullptr) a.u_out[i] = q;
    }
  }
  const int nnew = a.resample ? a.N - a.k : 0;
  for (int idx = tid; idx < a.N * HC; idx += blockDim.x) {
    const int col = idx / a.N, n = idx - col * a.N;
    const int t = col / NU, c = col - t * NU;
    float q, mm, vv;
    if (n < nnew) {  // fresh sample (:451-453)
      q = env_rpgd_sample_column<NU>(a, (uint32_t)n, t, c);
      mm = 0.0f;
      vv = 0.0f;
    } else {
      const int src = a.resample ? sh_best[n - nnew] : n;  // gather in best order (:454) or identity
      const int ts = min(t + a.shift_previous, a.H - 1);   // :376-379 shift, repeat the last
      q = a.Q[(size_t)(ts * NU + c) * a.N + src];
      // optimizer_gradient_tf.py:142-149: the vacated last step gets a fresh uniform control per input
      if (a.tail_resample && t == a.H - 1) q = env_rpgd_sample_point(a, (uint32_t)n, c, c);
      // Adam moments: always shifted by ONE time step with zero fill (:462-513)
      mm = (t + 1 < a.H) ? a.m[(size_t)(col + NU) * a.N + src] : 0.0f;
      vv = (t + 1 < a.H) ? a.v[(size_t)(col + NU) * a.N + src] : 0.0f;
    }
    a.Qn[idx] = q;
    a.mn[idx] = mm;
    a.vn[idx] = vv;
  }
  for (int n = tid; n < a.N; n += blockDim.x) {
    const float age = (n < nnew) ? 0.0f : a.ages[a.resample ? sh_best[n - nnew] : n];
    a.agesn[n] = age + 1.0f;  // :514
  }
}

// K6/K7 for an environment: `iters` gradient steps (forward tape, reverse sweep through the Env adjoint, clip_by_norm over the
// whole [H, NU] gradient, Adam / descent, per-input box clip), then the cost of the updated population (_get_action :342).
// fuse_select: the population is this one block, K8 follows in the same launch.
template <class Env, bool LOG>
__global__ void __launch_bounds__(kEnvRpgdBlock) env_rpgd_grad_kernel(const EnvRpgdGradArgs a, const EnvRpgdSelectArgs sel, const int fuse_select) {
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
    env_rpgd_select_body<NU>(sel, sh_sel, sh_best);
  }
}

template <int NU>
__global__ void __launch_bounds__(TOPK_THREADS) env_rpgd_select_kernel(const EnvRpgdSelectArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ int sh_best[TOPK_THREADS];
  env_rpgd_select_body<NU>(a, sh, sh_best);
}

// initial population (optimizer_reset :540): all N rows sampled; Adam state and ages zeroed
template <int NU>
__global__ void env_rpgd_init_kernel(const EnvRpgdSelectArgs a) {
  const int HC = a.H * NU;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < a.N * HC; idx += gridDim.x * blockDim.x) {
    const int col = idx / a.N, n = idx - col * a.N;
    const int t = col / NU, c = col - t * NU;
    a.Qn[idx] = env_rpgd_sample_column<NU>(a, (uint32_t)n, t, c);
    a.mn[idx] = 0.0f;
    a.vn[idx] = 0.0f;
    if (col == 0) a.agesn[n] = 0.0f;
  }
}

// ---- gradient-assisted CEM (gradcem_sample_kernel / gradcem_refit_kernel over NU columns) -----------------------------------
// Q[col][col0 + r] = clip(mu_col + z_{r,col} sd_col), the draws of row r in C order over [H, NU]
template <int NU>
__global__ void env_gradcem_sample_kernel(const EnvGradCemSampleArgs a) {
  const int HC = a.H * NU;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < a.cnt * HC; idx += gridDim.x * blockDim.x) {
    const int col = idx / a.cnt, r = idx - col * a.cnt, c = col % NU;
    const float z = noise1(a.noise, (uint32_t)r, col);
    a.dst[(size_t)col * a.ld + a.col0 + r] =
        fminf(fmaxf(__fadd_rn(a.mu[col], __fmul_rn(z, a.sd[col])), env_pick<NU>(a.lo, c)), env_pick<NU>(a.hi, c));
  }
}

// argsort of the N <= 1024 costs, elites in rank order, mean / population std per (t, c) column, elites carried into the next
// population buffer; on the last outer iteration the clip / shift by one time step / u of ``step``
template <int NU>
__global__ void __launch_bounds__(TOPK_THREADS) env_gradcem_refit_kernel(const EnvGradCemRefitArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ int sh_best[TOPK_THREADS];
  const int tid = threadIdx.x, HC = a.H * NU;
  uint64_t key = (tid < a.N) ? make_key(a.J[tid], (uint32_t)tid) : KEY_MAX;
  int n_sort = 32;
  while (n_sort < a.N) n_sort <<= 1;
  key = block_bitonic_sort(key, sh, n_sort);
  if (tid < a.k) {
    sh_best[tid] = (int)(key & 0xffffffffu);
    if (a.elite_idx_out != nullptr) a.elite_idx_out[tid] = sh_best[tid];
  }
  __syncthreads();
  for (int col = tid; col < HC; col += blockDim.x) {
    const int c = col % NU;
    const float* row = a.Q + (size_t)col * a.N;
    float acc = 0.0f;
    for (int e = 0; e < a.k; ++e) acc += row[sh_best[e]];
    const float new_mu = acc / (float)a.k;
    float var = 0.0f;
    for (int e = 0; e < a.k; ++e) {
      const float q = row[sh_best[e]];
      const float d = q - new_mu;
      var = fmaf(d, d, var);
      if (a.Q_carry != nullptr) a.Q_carry[(size_t)col * a.N + e] = q;
    }
    const float new_sd = sqrtf(var / (float)a.k);
    if (!a.last) {
      a.mu[col] = new_mu;
      a.sd[col] = new_sd;
    } else {
      const float sdc = fminf(fmaxf(new_sd, a.sd_min), 10.0f);  // naive :103 / bharadhwaj :139
      if (col >= NU) {
        a.mu[col - NU] = new_mu;
        a.sd[col - NU] = sdc;
      } else {
        const float u = a.u_from_mean ? new_mu : row[sh_best[0]];
        if (!a.freeze_prev) a.u_prev[c] = u;
        if (a.u_out != nullptr) a.u_out[c] = u;
      }
    }
  }
  if (a.last) {
    __syncthreads();  // the last time step is written after every shifted store
    if (tid < NU) {
      a.mu[HC - NU + tid] = 0.5f * (a.lo[tid] + a.hi[tid]);
      a.sd[HC - NU + tid] = a.sd_init;
    }
  }
}

}  // namespace ctk
