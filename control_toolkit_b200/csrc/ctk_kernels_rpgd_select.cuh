// ctk_kernels_rpgd_select.cuh -- the population steps of the gradient optimizers, for the CartPole (NU = 1) and the registered
// environments alike: K8 select / shift / resample (reference optimizer_rpgd.py:340-380, :443-516), the initial population
// (:527-548) and the sample / refit halves of the gradient-assisted CEM variants.  Templates only: the header is included by two
// translation units (ctk_rpgd.cu launches every kernel, ctk_env_rpgd.cu fuses rpgd_select_body into its gradient kernel).
// Population arrays are [H][NU][N] (flat column t * NU + c), so one thread per trajectory reads coalesced.  Reference semantics for
// NU > 1 (DESIGN section 2):
//  - sample_actions draws [B, n_ind, nu] in C order: draw index = point * NU + input (as env MPPI);
//  - the Adam moments shift by one time step (NU columns) with zero fill, whatever shift_previous is;
//  - the gradient-tf tail redraw is [N, 1, nu] uniform in [low_c, high_c];
//  - grad-CEM refits mean and std per (t, c) column and shifts by one time step after the loop.
// The host mirror (a.host.p != nullptr, CartPole host-facing ticks only) carries u of input 0 and the best sequence [H * NU].
#pragma once
#include "ctk_device.cuh"
#include "ctk_topk.cuh"

namespace ctk {

// v[c] for a run-time c without a local-memory copy of the parameter array
template <int NU>
__device__ __forceinline__ float env_pick(const float* v, int c) {
  float r = v[0];
#pragma unroll
  for (int i = 1; i < NU; ++i) r = c == i ? v[i] : r;
  return r;
}

// sample_actions (optimizer_rpgd.py:275-296) for input c, noise draw d of a new row: clip(z * scale + offset) per input
__device__ __forceinline__ float rpgd_sample_point(const RpgdSelectArgs& a, uint32_t row, int d, int c) {
  const float z = noise1(a.noise, row, d);
  const float y = a.dist == 0 ? __fadd_rn(__fmul_rn(z, a.s_std), a.s_mean) : __fadd_rn(__fmul_rn(z, a.s_max[c] - a.s_min[c]), a.s_min[c]);
  return fminf(fmaxf(y, a.lo[c]), a.hi[c]);
}
// column (t, c) of a freshly sampled row: interpolated clipped inducing points (Interpolator.py:97-106)
template <int NU>
__device__ __forceinline__ float rpgd_sample_column(const RpgdSelectArgs& a, uint32_t row, int t, int c) {
  const int seg = t / a.period, j = t - seg * a.period;
  float w0, w1;
  interp_weights(seg, j, a.period, a.n_ind, &w0, &w1);
  const float y0 = rpgd_sample_point(a, row, seg * NU + c, c);
  const float y1 = (j > 0) ? rpgd_sample_point(a, row, (seg + 1) * NU + c, c) : 0.0f;
  return fmaf(y1, w1, __fmul_rn(y0, w0));
}

// K8: argsort, u / u_nom of the best row, shift / resample / moment shift into the next buffers.  Any block size >= the padded
// population; every thread of the block takes part (callers: rpgd_select_kernel, and the gradient kernels when the whole population
// is one block -- then the tick is ONE launch)
template <int NU>
__device__ __forceinline__ void rpgd_select_body(const RpgdSelectArgs& a, uint64_t* sh, int* sh_best) {
  const int tid = threadIdx.x, HC = a.H * NU;
  uint64_t key = (tid < a.N) ? make_key(a.J[tid], (uint32_t)tid) : KEY_MAX;
  int n_sort = 32;
  while (n_sort < a.N) n_sort <<= 1;
  key = block_bitonic_sort(key, sh, n_sort);  // argsort (:345), stable by index; C3's 32 costs stay inside one warp's shuffles
  if (tid < a.k) {
    sh_best[tid] = (int)(key & 0xffffffffu);
    a.best_idx_out[tid] = sh_best[tid];
  }
  __syncthreads();
  const int best = sh_best[0];
  for (int i = tid; i < HC; i += blockDim.x) {
    const float q = a.Q[(size_t)i * a.N + best];
    a.u_nom_out[i] = q;  // :426
    if (a.host.p != nullptr) host_put(a.host, 8 + i, q);
  }
  if (tid < NU) {  // :523 u = u_nom[0, 0, :]
    const float u = a.Q[(size_t)tid * a.N + best];
    if (!a.freeze_prev) a.u_prev[tid] = u;
    if (a.u_out != nullptr) a.u_out[tid] = u;
    if (tid == 0 && a.host.p != nullptr) { host_put(a.host, 5, 0.0f); host_put(a.host, 4, u); }
  }
  const int nnew = a.resample ? a.N - a.k : 0;
  // unrolled for the CartPole only: at NU = 2 the unrolled loop moves the register allocation of the environment gradient kernel
#pragma unroll(NU == 1 ? 4 : 1)
  for (int idx = tid; idx < a.N * HC; idx += blockDim.x) {
    const int col = idx / a.N, n = idx - col * a.N;
    const int t = col / NU, c = col - t * NU;
    float q, mm, vv;
    if (n < nnew) {  // fresh sample (:451-453)
      q = rpgd_sample_column<NU>(a, (uint32_t)n, t, c);
      mm = 0.0f;
      vv = 0.0f;
    } else {
      const int src = a.resample ? sh_best[n - nnew] : n;  // gather in best order (:454) or identity
      const int ts = min(t + a.shift_previous, a.H - 1);   // :376-379 shift, repeat the last
      q = a.Q[(size_t)(ts * NU + c) * a.N + src];
      // optimizer_gradient_tf.py:142-149: the vacated last step gets a fresh uniform control per input instead of a repeat
      if (a.tail_resample && t == a.H - 1) q = rpgd_sample_point(a, (uint32_t)n, c, c);
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

template <int NU>
__global__ void __launch_bounds__(TOPK_THREADS) rpgd_select_kernel(const RpgdSelectArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ int sh_best[TOPK_THREADS];
  pdl_wait();
  pdl_trigger();
  rpgd_select_body<NU>(a, sh, sh_best);
}

// initial population (optimizer_reset :540): all N rows sampled; Adam state and ages zeroed
template <int NU>
__global__ void rpgd_init_kernel(const RpgdSelectArgs a) {
  pdl_wait();
  pdl_trigger();
  const int HC = a.H * NU;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < a.N * HC; idx += gridDim.x * blockDim.x) {
    const int col = idx / a.N, n = idx - col * a.N;
    const int t = col / NU, c = col - t * NU;
    a.Qn[idx] = rpgd_sample_column<NU>(a, (uint32_t)n, t, c);
    a.mn[idx] = 0.0f;
    a.vn[idx] = 0.0f;
    if (col == 0) a.agesn[n] = 0.0f;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Gradient-assisted CEM (reference optimizer_cem_naive_grad_tf.py:58-87, optimizer_cem_grad_bharadhwaj_tf.py:93-132)
// ---------------------------------------------------------------------------------------------------------------
// Q[col][col0 + r] = clip(mu_col + z_{r,col} sd_col), the draws of row r in C order over [H, NU]  (multiply and add separately
// rounded, as the reference's tf ops)
template <int NU>
__global__ void gradcem_sample_kernel(const GradCemSampleArgs a) {
  pdl_wait();
  pdl_trigger();
  const int HC = a.H * NU;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < a.cnt * HC; idx += gridDim.x * blockDim.x) {
    const int col = idx / a.cnt, r = idx - col * a.cnt, c = col % NU;
    const float z = noise1(a.noise, (uint32_t)r, col);
    a.dst[(size_t)col * a.ld + a.col0 + r] =
        fminf(fmaxf(__fadd_rn(a.mu[col], __fmul_rn(z, a.sd[col])), env_pick<NU>(a.lo, c)), env_pick<NU>(a.hi, c));
  }
}

// argsort of the N <= 1024 costs (ties to the lower index), elite gather in rank order, mean / population std per (t, c) column,
// elites carried into the next population buffer; on the last outer iteration the clip / shift by one time step / u of ``step``
template <int NU>
__global__ void __launch_bounds__(TOPK_THREADS) gradcem_refit_kernel(const GradCemRefitArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ int sh_best[TOPK_THREADS];
  const int tid = threadIdx.x, HC = a.H * NU;
  pdl_wait();
  pdl_trigger();
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
        if (c == 0 && a.host.p != nullptr) { host_put(a.host, 5, 0.0f); host_put(a.host, 4, u); }
      }
    }
  }
  if (a.last) {
    __syncthreads();  // the last time step is written by the threads of time step H (none) -> fill after every shifted store
    if (tid < NU) {
      a.mu[HC - NU + tid] = 0.5f * (a.lo[tid] + a.hi[tid]);  // mid-range per input
      a.sd[HC - NU + tid] = a.sd_init;
    }
  }
}

}  // namespace ctk
