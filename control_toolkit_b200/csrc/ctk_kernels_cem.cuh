// ctk_kernels_cem.cuh -- K3 fused sample -> rollout -> cost for CEM, K5 elite merge + refit (+ post-loop shift).
// Replaces reference optimizer_cem_tf.py:54-80 (update_distribution) and :99-102 (post-loop) for one tick.
#pragma once
#include "ctk_device.cuh"
#include "ctk_predictor.cuh"
#include "ctk_topk.cuh"
#include "ctk_ode_scaled.cuh"

namespace ctk {

// Q[n,t] = clip(mu_t + z * sd_t): optimizer_cem_tf.py:64-66 (tf.multiply then add, separately rounded)
__device__ __forceinline__ float cem_sample(float mu, float sd, float z, float lo, float hi) {
  return fminf(fmaxf(__fadd_rn(mu, __fmul_rn(z, sd)), lo), hi);
}

// Block geometry comes from the predictor: one thread per rollout (ODE, FP32-pipe networks: 128 threads), or the tile engines of
// ctk_mlp_tc.cuh (MlpTcPred: 128 rollouts + helper threads per block; MlpTcFastPredT: 512 rollouts per block, every block an equal
// contiguous share of the population) -- the same mapping as mppi_rollout_kernel.
template <class Pred, int KIND, bool LOG>
__global__ void __launch_bounds__(Pred::kCemThreads) cem_rollout_kernel(const CemArgs a) {
  extern __shared__ float smem[];
  float* sh_mu = smem;         // [H]
  float* sh_sd = smem + a.H;   // [H]
  Pred pred(a.kc, a.mlp, smem + 2 * a.H);  // constants: independent of the previous kernel, loaded while it drains
  const CostC cost = load_cost(a.kc);
  pdl_wait();
  pdl_trigger();
  for (int t = threadIdx.x; t < a.H; t += blockDim.x) {
    sh_mu[t] = a.mu[t];
    sh_sd[t] = a.sd[t];
  }
  __syncthreads();

  const int tid = threadIdx.x;
  const int rpb = Pred::kRolloutsPerBlock > 0 ? Pred::kRolloutsPerBlock : (int)blockDim.x;
  const bool owner = tid < rpb;
  const int r_first = Pred::kBalanced ? (int)((long long)blockIdx.x * a.N / gridDim.x) : (int)blockIdx.x * rpb;
  const int r_end = Pred::kBalanced ? (int)(((long long)blockIdx.x + 1) * a.N / gridDim.x) : min(a.N, r_first + rpb);
  const State z0 = {a.s0.ld(0), a.s0.ld(1), a.s0.ld(2), a.s0.ld(3), a.s0.ld(4), a.s0.ld(5)};
  const float omc0 = 1.0f - cosf(z0.th);
  const float u_prev0 = a.u_prev[0];
  for (int base = r_first; base < r_end; base += rpb) {
    const int n = base + tid;
    const bool active = owner && n < r_end;
    const bool grp = Pred::kCooperative && pred.group_active(base, r_end);  // (every thread: the tile engines note the tile's row count)
    if (!(active || grp)) continue;
    const uint32_t ng = (uint32_t)(a.off + (active ? n : 0));
    State z = z0;
    float omc = omc0;
    float u_last = u_prev0;
    float jsum = 0.0f;
    pred.begin_rollout(active);  // recurrent predictors: restore the saved hidden state; tile engines: is this row a real rollout
    for (int t0 = 0; t0 < a.H; t0 += 4) {
      float zz[4];
      noise4(a.noise, ng, (uint32_t)(t0 >> 2), zz);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int t = t0 + q;
        if (t < a.H) {
          const float u = cem_sample(sh_mu[t], sh_sd[t], zz[q], a.lo, a.hi);
          if (LOG && active) {
            float* p = a.log_traj_soa + (size_t)t * 6 * a.N + n;
            p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
            a.log_Q_soa[(size_t)t * a.N + n] = u;
          }
          jsum += stage_cost<KIND>(z, omc, u, u_last, cost);
          pred.step(z, u, omc);
          u_last = u;
        }
      }
    }
    if (active) {
      if (LOG) {
        float* p = a.log_traj_soa + (size_t)a.H * 6 * a.N + n;
        p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
      }
      a.J[n] = (jsum + terminal_cost(z, cost)) - cost.shift;
    }
  }
}

// One block of 1024 threads: merge candidates -> global top-k (bitonic), regenerate elite Q, refit mu / sd.
// One CEM rollout in the scaled state variables of K1 (ctk_ode_scaled.cuh): sample -> step -> cost over the horizon, returns the
// trajectory cost.  Full groups of four steps form ONE basic block together with the (independent) Philox block of the next
// four steps, so the scheduler interleaves the draw latency with the state chain.  Shared by K3s and the persistent tick.
// FAST: Philox N(0,1) draws without the run-time noise-mode branches (production CEM ticks).
template <int KIND, bool LOG, bool FAST = false>
__device__ __forceinline__ float cem_rollout_scaled(const NoiseSrc& ns, uint32_t ng, int n, int N, int H, const float* sh_mu,
                                                    const float* sh_sd, const ScaledState& r0, float u_prev, const OdeHot& k,
                                                    float* log_traj_soa, float* log_Q_soa) {
  ScaledState r = r0;
  float ul = u_prev;
  float acc = (k.k_ccrc * u_prev) * u_prev;  // telescoped control-change cost: + k_ccrc u_{-1}^2 here, - k_ccrc u_{H-1}^2 at the end
  float zn[4];
  if (FAST) noise4_normal(ns, ng, 0u, zn); else noise4(ns, ng, 0u, zn);
  auto log_state = [&](int t) {
    float st[6];
    scaled_to_state(r, k, st);
    float* p = log_traj_soa + (size_t)t * 6 * N + n;
    p[0] = st[0]; p[N] = st[1]; p[2 * N] = st[2]; p[3 * N] = st[3]; p[4 * (size_t)N] = st[4]; p[5 * (size_t)N] = st[5];
  };
  auto one_step = [&](int t, float zt) {
    const float u = cem_sample(sh_mu[t], sh_sd[t], zt, k.lo, k.hi);
    if (LOG) {
      log_state(t);
      log_Q_soa[(size_t)t * N + n] = u;
    }
    acc = stage_cost_scaled<KIND>(acc, r, u, ul, 0.0f, k);  // kC == 0 for CEM (no MPPI correction)
    ode_step_scaled(r, u, k);
    ul = u;
  };
  int t0 = 0;
  for (; t0 + 4 <= H; t0 += 4) {
    const float z0 = zn[0], z1 = zn[1], z2 = zn[2], z3 = zn[3];
    if (FAST) noise4_normal(ns, ng, (uint32_t)((t0 >> 2) + 1), zn); else noise4(ns, ng, (uint32_t)((t0 >> 2) + 1), zn);
    one_step(t0, z0);
    one_step(t0 + 1, z1);
    one_step(t0 + 2, z2);
    one_step(t0 + 3, z3);
  }
  for (int q = 0; t0 + q < H; ++q) one_step(t0 + q, zn[q]);
  if (LOG) log_state(H);
  return finish_cost_scaled(acc, r, ul, k);
}

// K3s: the same sample -> rollout -> cost pass for the ODE predictor in the scaled state variables of K1 (12-instruction Euler
// step, cost with the control terms merged into u (kA u + kB u_prev) and the u_prev^2 terms telescoped; constants are kernel
// parameters -> uniform registers); the block can also emit its own top-k candidates (level 0 of K4).
constexpr int kCemOdeTopkThreads = 256;  // block size when the block-level top-k is fused in (CemOdeArgs::cand_out)
template <int KIND, bool LOG>
__global__ void __launch_bounds__(kCemOdeTopkThreads) cem_ode_kernel(const CemOdeArgs a) {
  extern __shared__ float smem[];
  float* sh_mu = smem;         // [H]
  float* sh_sd = smem + a.H;   // [H]
  __shared__ uint64_t sh_keys[kCemOdeTopkThreads];
  const OdeHot& k = a.k;
  pdl_wait();
  pdl_trigger();
  for (int t = threadIdx.x; t < a.H; t += blockDim.x) {
    sh_mu[t] = a.mu[t];
    sh_sd[t] = a.sd[t];
  }
  __syncthreads();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = n < a.N;
  if (!active && a.cand_out == nullptr) return;
  uint64_t key = KEY_MAX;
  if (active) {
    const uint32_t ng = (uint32_t)(a.off + n);
    const float s0v[6] = {a.s0.ld(0), a.s0.ld(1), a.s0.ld(2), a.s0.ld(3), a.s0.ld(4), a.s0.ld(5)};
    ScaledState r0;
    scaled_from_state(s0v, k, r0);
    const float J = cem_rollout_scaled<KIND, LOG>(a.noise, ng, n, a.N, a.H, sh_mu, sh_sd, r0, a.u_prev[0], k, a.log_traj_soa, a.log_Q_soa);
    a.J[n] = J;
    key = make_key(J, ng);
  }
  if (a.cand_out != nullptr) {  // block-level top-k (K4 level 0): blockDim.x == kCemOdeTopkThreads
    key = block_bitonic_sort(key, sh_keys, kCemOdeTopkThreads);
    if ((int)threadIdx.x < a.kk) a.cand_out[(size_t)blockIdx.x * a.kk + threadIdx.x] = key;
  }
}

static __global__ void __launch_bounds__(TOPK_THREADS) cem_refit_kernel(const CemRefitArgs a) {
  __shared__ uint64_t sh[TOPK_THREADS];
  __shared__ uint32_t sh_elite[TOPK_THREADS];
  pdl_wait();
  pdl_trigger();
  uint64_t key = KEY_MAX;
  int cnt = a.cnt;
  if (a.world > 1) {
    // fused candidate exchange: this shard's k keys -> every shard's mailbox; then the world x k keys of the own mailbox
    const int tid = threadIdx.x;
    const size_t base = (size_t)(a.seq & 1u) * CTK_MAX_PEERS * kCemMboxKeys * 2;
    for (int i = tid; i < a.world * a.k; i += blockDim.x) {
      const int r = i / a.k, e = i - r * a.k;
      const uint64_t kv = a.cand[e];
      unsigned long long* dst = a.mbox_peer[r] + base + ((size_t)a.rank * kCemMboxKeys + e) * 2;
      const unsigned long long x0 = ((unsigned long long)a.seq << 32) | (kv >> 32), x1 = ((unsigned long long)a.seq << 32) | (kv & 0xffffffffull);
      asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(x0), "l"(x1) : "memory");
    }
    cnt = a.world * a.k;
    const unsigned long long t0 = globaltimer_ns();
    if (tid < cnt) {
      const int r = tid / a.k, e = tid - r * a.k;
      const unsigned long long* src = a.mbox_local + base + ((size_t)r * kCemMboxKeys + e) * 2;
      unsigned long long v0, v1;
      int spins = 0;
      while (true) {
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(v0), "=l"(v1) : "l"(src) : "memory");
        if ((unsigned int)(v0 >> 32) == a.seq && (unsigned int)(v1 >> 32) == a.seq) break;
        if ((++spins & 1023) == 0 && globaltimer_ns() - t0 > 2000000000ull) { v0 = v1 = 0xffffffffull; break; }  // lost peer: sorts last
      }
      key = ((v0 & 0xffffffffull) << 32) | (v1 & 0xffffffffull);
    }
  } else if (threadIdx.x < a.cnt) {
    key = a.cand[threadIdx.x];
  }
  int n_sort = 32;
  while (n_sort < cnt) n_sort <<= 1;
  key = block_bitonic_sort(key, sh, n_sort);
  if (threadIdx.x < a.k) {
    sh_elite[threadIdx.x] = (uint32_t)(key & 0xffffffffu);
    if (a.elite_idx_out != nullptr) a.elite_idx_out[threadIdx.x] = (int32_t)(key & 0xffffffffu);
  }
  __syncthreads();

  // column t: elite_Q[e, t] for e = 0..k-1 (rank order); mean then population std (tf.math.reduce_std).  The elite rows are
  // regenerated from the counter-based noise: one Philox block (4 consecutive steps of one elite) per thread into shared
  // memory, then every column sums its k entries in rank order (same arithmetic as a per-column loop, 64x fewer Philox calls)
  constexpr int kQCap = 8192;
  __shared__ float sh_q[kQCap];
  float new_mu = 0.0f, new_sd = 0.0f, first_q = 0.0f;
  const int t = threadIdx.x;
  const int H4 = (a.H + 3) >> 2, Hs = H4 * 4;
  if (a.k * Hs <= kQCap) {
    for (int item = threadIdx.x; item < a.k * H4; item += blockDim.x) {
      const int e = item / H4, blk = item - e * H4;
      float zz[4];
      noise4(a.noise, sh_elite[e], (uint32_t)blk, zz);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int tt = blk * 4 + j;
        if (tt < a.H) sh_q[e * Hs + tt] = cem_sample(a.mu[tt], a.sd[tt], zz[j], a.lo, a.hi);
      }
    }
    __syncthreads();
    if (t < a.H) {
      float acc = 0.0f;
      for (int e = 0; e < a.k; ++e) acc += sh_q[e * Hs + t];
      first_q = sh_q[t];
      new_mu = acc / (float)a.k;
      float var = 0.0f;
      for (int e = 0; e < a.k; ++e) {
        const float d = sh_q[e * Hs + t] - new_mu;
        var = fmaf(d, d, var);
      }
      new_sd = sqrtf(var / (float)a.k);
    }
  } else if (t < a.H) {  // k x H too large for the staging buffer: per-column regeneration
    const float mu = a.mu[t], sd = a.sd[t];
    float acc = 0.0f;
    for (int e = 0; e < a.k; ++e) {
      const float q = cem_sample(mu, sd, noise1(a.noise, sh_elite[e], t), a.lo, a.hi);
      if (e == 0) first_q = q;
      acc += q;
    }
    new_mu = acc / (float)a.k;
    float var = 0.0f;
    for (int e = 0; e < a.k; ++e) {
      const float q = cem_sample(mu, sd, noise1(a.noise, sh_elite[e], t), a.lo, a.hi);
      const float d = q - new_mu;
      var = fmaf(d, d, var);
    }
    new_sd = sqrtf(var / (float)a.k);
  }
  __syncthreads();  // every column has read the old mu / sd
  if (t < a.H) {
    if (!a.last) {
      a.mu[t] = new_mu;
      a.sd[t] = new_sd;
    } else {
      // :99-102  stdev = clip(stdev, min, 1e8); shift left, append initial stdev / mid-range mean; u = elite_Q[0,0]
      const float sdc = fminf(fmaxf(new_sd, a.sd_min), 1.0e8f);
      if (t > 0) {
        a.mu[t - 1] = new_mu;
        a.sd[t - 1] = sdc;
      } else {
        if (!a.freeze_prev) a.u_prev[0] = first_q;
        if (a.u_out != nullptr) a.u_out[0] = first_q;
        if (a.host.p != nullptr) { host_put(a.host, 5, 0.0f); host_put(a.host, 4, first_q); }
      }
      if (t == a.H - 1) {
        a.mu[t] = (a.lo + a.hi) * 0.5f;
        a.sd[t] = a.sd_init;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The CEM tick as ONE persistent launch (reference optimizer_cem_tf.py:83-111 incl. the outer loop :93-94).  Block = 512
// threads of which the first 128 own a rollout each (4 warps per SM keep the per-step issue demand below one instruction per
// scheduler and cycle: with 16 rollout warps per SM the same loop measured 224 ns per step instead of ~60); all 512 take part in
// the sorts, merges and the refit.  Per outer iteration: every block rolls out its 128 samples (K3s), sorts its keys and
// publishes its k best as ONE tagged 8-byte slot each (ordered cost | id | 16-bit sequence tag); block 0 polls the grid's
// sorted runs into shared memory, merges them pairwise (elementwise min of one run with the reverse of the other = the lower
// half as a bitonic sequence, then log2 merge stages: a tree of depth log2(runs) instead of a full sort), regenerates the
// elite rows, refits mean / population std (K5) and publishes the new distribution as tagged slots the other blocks poll at the
// top of the next iteration.  No kernel boundary and no host round trip between the outer iterations; the multi-launch path
// (K3s / K4 / K5) remains for sharded ticks and populations beyond one resident grid.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCemTickThreads = 512;
constexpr int kCemTickRollouts = 128;  // rollouts per block
constexpr int kCemTickMaxK = 128;
__device__ __forceinline__ void st_cand(unsigned long long* dst, uint64_t key, unsigned int seq) {
  // key = (ordered cost << 32) | id with id < 65536: one 8-byte store carries cost, id and the tag
  const unsigned long long x = (key & 0xffffffff00000000ull) | ((key & 0xffffull) << 16) | (unsigned long long)(seq & 0xffffu);
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(dst), "l"(x) : "memory");
}
__device__ __forceinline__ unsigned long long ld_slot(const unsigned long long* src) {
  unsigned long long v;
  asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(src) : "memory");
  return v;
}
// Pairwise merge tree over `runs` (power of two) ascending runs of K2 = 32 E keys in shared memory: after the call run 0 holds
// the K2 smallest keys of all runs, ascending.  Warp w merges runs 2 m, 2 m + 1 into run m (m = w, w + warps, ...): elementwise
// min of one run with the reverse of the other is the lower half as a bitonic sequence; log2(K2) compare-exchange stages sort it.
template <int E>
__device__ __forceinline__ void merge_runs_tree(uint64_t* sh_runs, int runs, int tid, int nthreads) {
  constexpr int K2 = 32 * E;
  const int lane = tid & 31, w = tid >> 5, nw = nthreads >> 5;
  for (; runs > 1; runs >>= 1) {
    const int merges = runs >> 1;
    // merge m writes run m, which a LATER pass of this level (merge m' >= m0 + nw reads runs >= 2 m') never reads, and
    // which the merges of this pass have read before the barrier below
    for (int m0 = 0; m0 < merges; m0 += nw) {
      const int m = m0 + w;
      uint64_t x[E];
      if (m < merges) {
        const uint64_t* A = sh_runs + (size_t)(2 * m) * K2;
        const uint64_t* B = A + K2;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int i = lane + 32 * e;
          const uint64_t xa = A[i], xb = B[K2 - 1 - i];
          x[e] = xa < xb ? xa : xb;
        }
#pragma unroll
        for (int stride = K2 >> 1; stride >= 32; stride >>= 1) {  // partners inside the lane: e ^ (stride / 32)
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const int pe = e ^ (stride >> 5);
            if (pe > e) {
              const uint64_t lo = x[e] < x[pe] ? x[e] : x[pe], hi = x[e] < x[pe] ? x[pe] : x[e];
              x[e] = lo;
              x[pe] = hi;
            }
          }
        }
#pragma unroll
        for (int stride = 16; stride > 0; stride >>= 1) {
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const uint64_t other = __shfl_xor_sync(0xffffffffu, x[e], stride);
            const bool lower = (lane & stride) == 0;
            const uint64_t mn = x[e] < other ? x[e] : other, mx = x[e] < other ? other : x[e];
            x[e] = lower ? mn : mx;
          }
        }
      }
      __syncthreads();  // every warp of this pass has read its two input runs
      if (m < merges) {
#pragma unroll
        for (int e = 0; e < E; ++e) sh_runs[(size_t)m * K2 + lane + 32 * e] = x[e];
      }
      __syncthreads();
    }
  }
}

template <int KIND, bool LOG, bool FAST>
__global__ void __launch_bounds__(kCemTickThreads) cem_tick_kernel(const CemTickArgs a) {
  extern __shared__ float smem[];
  float* sh_mu = smem;         // [H]
  float* sh_sd = smem + a.H;   // [H]
  // big buffer: the grid's candidate runs [runs_pad][K2] (uint64) during the merge, then the regenerated elite rows (floats)
  uint64_t* sh_runs = reinterpret_cast<uint64_t*>(smem + ((2 * a.H + 3) & ~3));
  float* sh_q = reinterpret_cast<float*>(sh_runs);
  __shared__ uint64_t sh_sort[kCemTickThreads];
  __shared__ uint32_t sh_elite[kCemTickMaxK];
  const OdeHot& k = a.hot;
  constexpr int T = kCemTickThreads;
  const int RB = a.rb;
  const int tid = threadIdx.x, b = blockIdx.x, H = a.H, G = (int)gridDim.x;
  const int n = b * RB + tid;
  const bool active = tid < RB && n < a.N;
  const uint32_t ng = (uint32_t)(a.off + (active ? n : 0));
  pdl_wait();
  pdl_trigger();
  const unsigned long long t0 = globaltimer_ns();
  const float s0v[6] = {a.s0.ld(0), a.s0.ld(1), a.s0.ld(2), a.s0.ld(3), a.s0.ld(4), a.s0.ld(5)};
  ScaledState r0;
  scaled_from_state(s0v, k, r0);
  const float u_prev = a.u_prev[0];
  int status = 0;
  auto trace = [&](int it, int slot) {  // optional phase timeline of block 0 (tools/cem_trace.py)
    if (a.trace != nullptr && b == 0 && tid == 0 && it < 16) a.trace[it * 8 + slot] = globaltimer_ns();
  };

  for (int it = 0; it < a.iters; ++it) {
    trace(it, 0);
    const unsigned int seq = a.seq0 + (unsigned int)it;
    const bool last = it == a.iters - 1;
    NoiseSrc ns = a.noise;
    ns.stream = a.noise.stream | ((uint32_t)it << 8);
    if (ns.inj != nullptr) ns.inj = a.noise.inj + (size_t)it * a.inj_stride;
    // ---- (A) this iteration's distribution: global state (it == 0), block 0's tagged publication otherwise ----
    if (it == 0) {
      for (int t = tid; t < H; t += T) { sh_mu[t] = a.mu[t]; sh_sd[t] = a.sd[t]; }
    } else if (b != 0) {
      for (int t = tid; t < H; t += T) {
        if (!ld_tagged(a.dist + t, seq, t0, &sh_mu[t])) status = 1;
        if (!ld_tagged(a.dist + H + t, seq, t0, &sh_sd[t])) status = 1;
      }
    }
    __syncthreads();
    trace(it, 1);
    // ---- (B) sample -> rollout -> cost (K3s) ----
    uint64_t key = KEY_MAX;
    if (active) {
      const float J = cem_rollout_scaled<KIND, LOG, FAST>(ns, ng, n, a.N, H, sh_mu, sh_sd, r0, u_prev, k, a.log_traj_soa, a.log_Q_soa);
      if (last) a.J[n] = J;
      key = make_key(J, ng);
    }
    // ---- (C) the block's k best keys, ascending -> tagged candidate slots ----
    trace(it, 2);
    key = block_bitonic_sort(key, sh_sort, RB);
    if (tid < a.k) st_cand(a.cand + (size_t)b * a.k + tid, key, seq);
    trace(it, 3);
    if (b != 0) continue;
    // ---- (D) block 0: poll the grid's sorted runs into shared memory, merge them pairwise ----
    const int K2 = a.k2, runs_pad = a.runs_pad;
    for (int base = 0; base < runs_pad * K2; base += 4 * T) {
      // up to four slots per thread and round, all loads in flight before the first tag is checked
      uint64_t kk[4];
      bool need[4];
      const unsigned long long* src[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = base + j * T + tid;
        const int r = idx / K2, i = idx - r * K2;
        need[j] = idx < runs_pad * K2 && r < G && i < a.k;
        src[j] = a.cand + (size_t)r * a.k + i;
        kk[j] = KEY_MAX;
      }
      int spins = 0;
      while (true) {
        unsigned long long v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = need[j] ? ld_slot(src[j]) : 0ull;
        bool pending = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (!need[j]) continue;
          if ((unsigned int)(v[j] & 0xffffull) == (seq & 0xffffu)) {
            const uint64_t raw = v[j] & 0xffffffff00000000ull;
            // an all-ones cost word is the padding key of a block with fewer than k rollouts
            kk[j] = (raw == 0xffffffff00000000ull && ((v[j] >> 16) & 0xffffull) == 0xffffull) ? KEY_MAX : (raw | ((v[j] >> 16) & 0xffffull));
            need[j] = false;
          } else pending = true;
        }
        if (!pending) break;
        if ((++spins & 1023) == 0 && globaltimer_ns() - t0 > 2000000000ull) { status = 1; break; }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = base + j * T + tid;
        if (idx < runs_pad * K2) sh_runs[idx] = kk[j];
      }
    }
    __syncthreads();
    // merge tree: one WARP per pair of runs, K2 / 32 keys per lane (key e of a lane sits at position lane + 32 e), so the
    // stages with stride >= 32 are register-to-register and the others warp shuffles -- the only block barriers are the ones
    // between the tree's levels
    if (K2 == 32) merge_runs_tree<1>(sh_runs, runs_pad, tid, T);
    else if (K2 == 64) merge_runs_tree<2>(sh_runs, runs_pad, tid, T);
    else merge_runs_tree<4>(sh_runs, runs_pad, tid, T);
    trace(it, 4);
    if (tid < a.k) {
      const uint64_t best = sh_runs[tid];
      sh_elite[tid] = (uint32_t)(best & 0xffffffffu);
      if (a.elite_idx_out != nullptr && it < a.elite_cap) a.elite_idx_out[(size_t)it * a.k + tid] = (int32_t)(best & 0xffffffffu);
    }
    __syncthreads();
    // ---- (E) refit (K5): elite rows regenerated from the counter-based noise, mean then population std in rank order ----
    float new_mu = 0.0f, new_sd = 0.0f, first_q = 0.0f;
    const int H4 = (H + 3) >> 2, Hs = H4 * 4;
    if (a.k * Hs <= a.q_cap) {
      for (int item = tid; item < a.k * H4; item += T) {
        const int e = item / H4, blk = item - e * H4;
        float zz[4];
        noise4(ns, sh_elite[e], (uint32_t)blk, zz);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int tt = blk * 4 + jj;
          if (tt < H) sh_q[e * Hs + tt] = cem_sample(sh_mu[tt], sh_sd[tt], zz[jj], k.lo, k.hi);
        }
      }
      __syncthreads();
      if (tid < H) {
        float accq = 0.0f;
        for (int e = 0; e < a.k; ++e) accq += sh_q[e * Hs + tid];
        first_q = sh_q[tid];
        new_mu = accq / (float)a.k;
        float var = 0.0f;
        for (int e = 0; e < a.k; ++e) {
          const float d = sh_q[e * Hs + tid] - new_mu;
          var = fmaf(d, d, var);
        }
        new_sd = sqrtf(var / (float)a.k);
      }
    } else if (tid < H) {
      const float mu = sh_mu[tid], sd = sh_sd[tid];
      float accq = 0.0f;
      for (int e = 0; e < a.k; ++e) {
        const float q = cem_sample(mu, sd, noise1(ns, sh_elite[e], tid), k.lo, k.hi);
        if (e == 0) first_q = q;
        accq += q;
      }
      new_mu = accq / (float)a.k;
      float var = 0.0f;
      for (int e = 0; e < a.k; ++e) {
        const float d = cem_sample(mu, sd, noise1(ns, sh_elite[e], tid), k.lo, k.hi) - new_mu;
        var = fmaf(d, d, var);
      }
      new_sd = sqrtf(var / (float)a.k);
    }
    status = __syncthreads_or(status);  // also: every column has read the old mu / sd
    trace(it, 5);
    if (tid < H) {
      if (!last) {
        sh_mu[tid] = new_mu;
        sh_sd[tid] = new_sd;
        st_tagged(a.dist + tid, new_mu, seq + 1);
        st_tagged(a.dist + H + tid, new_sd, seq + 1);
      } else {
        // :99-102  stdev = clip(stdev, min, 1e8); shift left, append initial stdev / mid-range mean; u = elite_Q[0,0]
        const float sdc = fminf(fmaxf(new_sd, a.sd_min), 1.0e8f);
        if (tid > 0) {
          a.mu[tid - 1] = new_mu;
          a.sd[tid - 1] = sdc;
        } else {
          const float u = status ? __int_as_float(0x7fc00000) : first_q;
          if (!a.freeze_prev) a.u_prev[0] = u;
          if (a.u_out != nullptr) { a.u_out[0] = u; a.u_out[1] = (float)status; }
          if (a.host.p != nullptr) { host_put(a.host, 5, (float)status); host_put(a.host, 4, u); }
        }
        if (tid == H - 1) {
          a.mu[tid] = (k.lo + k.hi) * 0.5f;
          a.sd[tid] = a.sd_init;
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace ctk
