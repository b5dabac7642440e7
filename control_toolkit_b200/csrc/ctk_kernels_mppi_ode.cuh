// ctk_kernels_mppi_ode.cuh -- K1 for the CartPole ODE predictor: fused sample -> rollout -> cost -> softmin record ->
// (last block) tick finish.  Replaces reference optimizer_mppi.py:170-193 for one tick when the predictor is the Euler
// ODE with intermediate_steps == 1 (the headline configuration); other cases run the generic kernel of
// ctk_kernels_mppi.cuh.
//
// What is different from the generic kernel (all measured with ncu, profiles/):
//  * scaled state variables (OdeHot): T = angle/sqrt(2), W = beta*angleD, V = (cF/g)*positionD remove 6 multiplies per
//    step; every constant multiplier is a kernel parameter that ptxas keeps in a uniform register, so all but five FMAs
//    per step read at most two vector registers (the sm_100 register file feeds 3-source FFMAs at ~2/3 rate);
//  * the control terms of the stage cost and of the MPPI correction collapse to u*(kA u + kB u_prev + kC du); the
//    du^2 term of the correction has a closed form per inducing-point segment and leaves the step loop entirely;
//  * PERIOD is a template parameter: a segment is fully unrolled, the interpolation weight j/PERIOD is an immediate and
//    du = fma(dy, w_j, y0) is one instruction;
//  * ILP rollouts per thread are advanced in lock step (independent dependency chains): the last warps of an SM
//    sub-partition still fill the FMA pipe, which removes the tail the hi-wid-first warp arbiter otherwise produces;
//    with ILP = 2 they are ONE roll of f2 lanes (ctk_ode_scaled.cuh): every add, multiply and fma of the step is one packed
//    FADD2 / FMUL2 / FFMA2 for both rollouts, bit-identical per lane to the float build.  The kernel is issue-bound, and a pair
//    takes one issue slot where two scalar instructions took two (tests/test_k1_packed_sass.py, DESIGN.md 5.1);
//  * the state-independent part of the prologue (the Philox draws of the first rollout group) runs BEFORE griddepcontrol.wait: in a
//    back-to-back chain of ticks (programmatic dependent launch) it overlaps the previous tick's finish / exchange / launch gap;
//    the global reads of the prologue (s0, u_prev, u_nom) follow the wait and were prefetched into L2 before the draws;
//  * work distribution: every block takes an equal contiguous share of the population, cut into UNITS of 32 ILP consecutive rollouts
//    that go round-robin over the block's warps.  The kernel is issue-bound, so its duration is the instruction count of the busiest
//    SM sub-partition (warp w runs on sub-partition w % 4): with 27 warps of four whole iterations each (7 / 7 / 7 / 6 warps: 28 units
//    on three sub-partitions, round 1) the ideal 26.4 units per sub-partition at C5 became 28; with 28 warps and the units dealt out
//    one by one it is 27.
#pragma once
#include <type_traits>

#include "ctk_device.cuh"
#include "ctk_kernels_mppi.cuh"
#include "ctk_ode_scaled.cuh"

namespace ctk {

// The registers of a thread's rollouts: L = float for one rollout per thread, f2 for two advanced in lock step (ctk_ode_scaled.cuh).
template <class L>
struct Roll : ScaledStateT<L> {
  L ul, acc, y0, dy, y1;
#ifdef CTK_K1_DSUM
  double dtot[sizeof(L) / sizeof(float)];
#endif
  L tot, comp;  // running total of the per-segment cost sums (+ its compensation term under CTK_K1_KAHAN; see fold_segment)
};
template <int ILP>
using Lanes = typename std::conditional<ILP == 2, f2, float>::type;

// a thread's draw i of its ILP rollouts: lane q at p[q * T_], p = sh_z + i * ILP * T_ + tid
template <class L>
__device__ L ld_lanes(const float* p, int T_);
template <>
__device__ __forceinline__ float ld_lanes<float>(const float* p, int) { return p[0]; }
template <>
__device__ __forceinline__ f2 ld_lanes<f2>(const float* p, int T_) { return f2(p[0], p[T_]); }

// The total cost S ~ 5e3 enters the softmin as exp(-(S - rho) / lambda) with lambda = 100: one ulp of S (4.9e-4) is 5e-6 relative
// in the weight, and a 100-term sequential fp32 sum wanders by ~3 ulp rms -- more than the reference's torch.mean over [H + 1]
// (vectorised pairwise summation).  The stage costs are therefore summed per inducing-point segment (partial sums an order of
// magnitude below S) and the segment sums enter the total through a compensated (Kahan) addition: 4 FADD per SEGMENT, ~0.5 ulp.
// (-DCTK_K1_PLAIN_SUM adds the segment sums up plainly, ~0.9 ulp rms: the pinned C1 ticks then miss the 1e-5 bound -- measured,
// tests/test_gpu_production_pinning.py c1 / c1_ilp2 -- so the compensation stays.)
template <class L>
__device__ __forceinline__ void fold_segment(Roll<L>& r) {
#if defined(CTK_K1_DSUM)
  for (int q = 0; q < (int)(sizeof(L) / sizeof(float)); ++q)
    r.dtot[q] += (double)lane_of(r.acc, q);  // (experiment) second level in double: exact, one conversion + one DADD per segment
#elif !defined(CTK_K1_PLAIN_SUM)
  const L y = r.acc - r.comp;
  const L t = r.tot + y;
  r.comp = (t - r.tot) - y;
  r.tot = t;
#else
  r.tot = r.tot + r.acc;
#endif
  r.acc = 0.0f;
}

// One step of a thread's rollouts (lane q: rollout n[q]).  wj = j/period (immediate when PERIOD is a template constant).
template <int KIND, bool LOG, class L>
__device__ __forceinline__ void ode_mppi_step(const MppiOdeArgs& a, const OdeHot& k, Roll<L>& r, float unom_t, float wj, bool first,
                                              int t, const int* n, const bool* active) {
  // Interpolator.py:97-106 (two non-zero weights): du = y0 (1 - wj) + y1 wj = y0 + (y1 - y0) wj
  const L du = first ? r.y0 : fmaf(r.dy, wj, r.y0);
  const L u = fminf(fmaxf(unom_t + du, k.lo), k.hi);  // optimizer_mppi.py:186-187
#pragma unroll
  for (int q = 0; q < (int)(sizeof(L) / sizeof(float)); ++q) {
    if (LOG && active[q]) {
      float* p = a.log_traj_soa + (size_t)t * 6 * a.N + n[q];
      p[0] = lane_of(r.T, q) * kSqrt2; p[a.N] = lane_of(r.W, q) * k.inv_beta; p[2 * (size_t)a.N] = lane_of(r.c, q); p[3 * (size_t)a.N] = lane_of(r.s, q);
      p[4 * (size_t)a.N] = lane_of(r.x, q); p[5 * (size_t)a.N] = lane_of(r.V, q) * k.inv_cFg;
      a.log_Q_soa[(size_t)t * a.N + n[q]] = lane_of(u, q);
    }
  }
  // stage cost / (H+1) (spec: DESIGN.md section 3; Cost_Functions/__init__.py:49-64) merged with the MPPI correction
  // (optimizer_mppi.py:154-155), then the Euler step in scaled variables (ctk_ode_scaled.cuh)
  r.acc = stage_cost_scaled<KIND>(r.acc, r, u, r.ul, du, k);
  r.ul = u;
  ode_step_scaled(r, u, k);
}

// INJ: injected-noise mode possible (verification); the production instantiations compile that branch out.
template <int KIND, bool LOG, int PERIOD, int ILP, bool INJ>
__device__ __forceinline__ void mppi_ode_body(const MppiOdeArgs& a) {
  extern __shared__ float smem[];
  const int T_ = blockDim.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = T_ >> 5;
  const int period = PERIOD > 0 ? PERIOD : a.period;
  const int P = a.n_ind + 1;
  float* sh_unom = smem;                                   // [H] shifted nominal (+ pad)
  float2* sh_w = reinterpret_cast<float2*>(smem + ((a.H + 3) & ~3));  // [period] interpolation weights ((period - j)/period, j/period)
  float* sh_red = reinterpret_cast<float*>(sh_w) + 2 * ((period + 3) & ~3);  // [32]
  float* sh_part = sh_red + 32;                            // [12][P + 1]: block record + finish scratch
  float* sh_z = sh_part + 12 * (P + 1);                          // [n_ind][ILP*T] standard draws of the rollouts in flight
  float* sh_acc = sh_z + (size_t)max(a.n_ind * ILP, 2) * T_;  // [n_ind][T] per-thread sum_n e_n z_n,i

  auto trace = [&](int slot) {  // optional per-block timeline (tools/k1_trace.py): globaltimer at the phase boundaries, last 4 launches
    if (a.trace != nullptr && tid == 0) a.trace[((size_t)(a.fuse.seq & 3u) * CTK_MBOX_BLOCKS + blockIdx.x) * 8 + slot] = globaltimer_ns();
  };
  trace(0);
  pdl_trigger();  // the next launch of the stream (the next tick of a chain) may be scheduled as soon as SMs free up
  // ---- prologue.  Prefetch the lines the global reads below will touch (after an L2 flush they come from DRAM), generate the
  //      Philox draws of the first rollout group -- they depend on nothing the previous tick produces -- and only then wait for the
  //      previous launch of the stream to complete (no-op unless launched as a programmatic dependent) ----
  const bool chained = a.fuse.chained != 0;  // the previous launch is the previous tick of this handle's chain (ctk_step_device_n)
  // Not chained: wait for the previous launch of the stream (no-op unless launched as a programmatic dependent) and ISSUE the
  // prologue's global reads now -- after an L2 flush they come from DRAM -- so that they are in flight underneath the Philox draws.
  float s0v = 0.0f, upv_ld = 0.0f, unom_first = 0.0f;
  if (!chained) {
    pdl_wait();
    s0v = (tid < 6) ? a.s0.ld(tid) : 0.0f;
    upv_ld = a.u_prev[0];
    unom_first = (tid < a.H) ? a.u_nom[min(tid + 1, a.H - 1)] : 0.0f;  // optimizer_mppi.py:184 (shift on read)
  }
  const OdeHot& k = a.k;
  const int nblk = (a.n_ind + 3) >> 2;
  // this block's share [r_first, r_end) of the population; unit u of it = rollouts r_first + u * UNIT + [0, UNIT), warp w takes units
  // w, w + nw, w + 2 nw, ...; a thread's ILP rollouts of a unit are 32 apart (coalesced cost / log stores per warp)
  // LOG: the trajectory log is HBM-write bound and wants all SMs inside one contiguous window of rollouts at a time (with contiguous
  // per-block shares the 148 x 7 write streams are scattered over the whole log: 0.62 -> 1.37 ms per C5 tick, measured), so there the
  // units are dealt out over the whole GRID instead: unit (it * gridDim + block) * nw + w.
  constexpr int UNIT = 32 * ILP;
  // Block 0 is the tick's finisher: in a back-to-back chain of ticks it is the block that starts its rollouts last (it was still
  // combining the previous tick's records when the other SMs were already in the new tick's prologue), so its share is smaller
  // (a.fshare16 sixteenths of an ordinary share): shares are cut at N cum(b) / tot with cum(b) = fshare16 + 16 (b - 1), cum(0) = 0.
  // (boundaries by one double multiplication each -- the same expression for a block's end and its successor's start, so the shares
  // tile [0, N) exactly; two 64-bit integer divisions here cost 0.3 us of every tick's prologue)
  const int fs16 = a.fshare16 > 0 ? a.fshare16 : 16;
  const double per16 = a.per16 > 0.0 ? a.per16 : (double)a.N / (double)(fs16 + 16 * ((int)gridDim.x - 1));  // (host-computed)
  const int cum0 = blockIdx.x == 0 ? 0 : fs16 + 16 * ((int)blockIdx.x - 1);
  const int cum1 = fs16 + 16 * (int)blockIdx.x;
  const int r_first = LOG ? 0 : (int)((double)cum0 * per16);
  const int r_end = LOG ? a.N : (blockIdx.x + 1 == gridDim.x ? a.N : (int)((double)cum1 * per16));
  auto gen_noise = [&](int base) {  // K0: draws of the ILP rollouts of a group -> shared-memory stash
#pragma unroll
    for (int q = 0; q < ILP; ++q) {
      const int nq = base + q * 32;
      const uint32_t ng = (uint32_t)(a.off + (nq < r_end ? nq : r_first));
      float* sz = sh_z + q * T_ + tid;
      for (int blk = 0; blk < nblk; ++blk) {
        float zz[4];
        noise4<INJ>(a.noise, ng, (uint32_t)blk, zz);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (blk * 4 + e < a.n_ind) sz[(size_t)(blk * 4 + e) * ILP * T_] = zz[e];
      }
    }
  };
  const int boff = (LOG ? ((int)blockIdx.x * nw + w) * UNIT : r_first + w * UNIT) + lane;  // this thread's first rollout (q = 0)
  const int stride = (LOG ? (int)gridDim.x : 1) * nw * UNIT;
  if (boff - lane < r_end) gen_noise(boff);
  for (int j = tid; j < period; j += T_) interp_weights(j, period, &sh_w[j].x, &sh_w[j].y);  // Interpolator.py:63-74
  for (int i = 0; i < a.n_ind; ++i) sh_acc[(size_t)i * T_ + tid] = 0.0f;
  if (chained) {
    // Chained: the Philox draws above ran underneath the previous tick's finish; its finisher publishes u_prev and u_nom[H] as
    // tagged slots: poll them instead of waiting for that launch to complete (the kernel-completion / dependent-release latency
    // leaves the tick-to-tick critical path).  A chain's states were complete before its first tick was launched.
    s0v = (tid < 6) ? a.s0.ld(tid) : 0.0f;
    const unsigned long long t0p = globaltimer_ns();
    const unsigned int pseq = a.fuse.seq - 1u;
    for (int t = tid; t < a.H; t += T_) ld_tagged(a.fuse.handover + 1 + min(t + 1, a.H - 1), pseq, t0p, &sh_unom[t]);
    if (tid == 31) ld_tagged(a.fuse.handover, pseq, t0p, &sh_red[6]);
  } else {
    if (tid < a.H) sh_unom[tid] = unom_first;
    for (int t = tid + T_; t < a.H; t += T_) sh_unom[t] = a.u_nom[min(t + 1, a.H - 1)];
    if (tid == 31) sh_red[6] = upv_ld;
  }
  if (tid < 6) sh_red[tid] = s0v;
  __syncthreads();
  const float upv = sh_red[6];
  const float th0 = sh_red[0], om0 = sh_red[1], c0 = sh_red[2], sn0 = sh_red[3], x0 = sh_red[4], v0 = sh_red[5];
  const float omc0 = 1.0f - cosf(th0);  // spec: E_pot uses cos(angle) of the measured state
  const float T0 = th0 * kInvSqrt2, W0 = om0 * k.beta, V0 = v0 * k.cFg;
  __syncthreads();  // sh_red is reused below
  trace(1);

  // closed form of sum_j du_j^2 over a full segment: cnt y0^2 + dy (2 W1 y0 + W2 dy)
  const float pf = (float)period;
  const float segW1x2_full = pf - 1.0f;                                             // 2 sum_j j/p
  const float segW2_full = (pf - 1.0f) * (2.0f * pf - 1.0f) / (6.0f * pf);          // sum_j (j/p)^2
  float rho_t = INFINITY, a_t = 0.0f;  // per-thread online softmin (optimizer_mppi.py:163-168, exact combine later)
  float* sa = sh_acc + tid;

  static_assert(ILP == 1 || ILP == 2, "one rollout per thread (float lanes) or two (f2 lanes)");
  using L = Lanes<ILP>;
  const float* sz = sh_z + tid;  // draw i of lane q: sz[(i * ILP + q) * T_]
  for (int base = boff; base - lane < r_end; base += stride) {  // (warp-uniform bound; no block barrier inside the loop)
    Roll<L> r;
    int n[ILP];
    bool active[ILP];
    if (base != boff) gen_noise(base);  // the first group's draws were generated in the prologue
#pragma unroll
    for (int q = 0; q < ILP; ++q) {
      n[q] = base + q * 32;
      active[q] = n[q] < r_end;
    }
    r.T = T0; r.W = W0; r.c = c0; r.s = sn0; r.x = x0; r.V = V0; r.omc = omc0;
    r.ul = upv;
    r.acc = (k.k_ccrc * upv) * upv;  // telescoped ccrc term of u_{-1}
    r.tot = 0.0f; r.comp = 0.0f;
#ifdef CTK_K1_DSUM
    for (int q = 0; q < ILP; ++q) r.dtot[q] = 0.0;
#endif
    r.y0 = 0.0f; r.dy = 0.0f;
    r.y1 = ld_lanes<L>(sz, T_) * k.stdev;  // y0 of segment 0   (:173-175 normal * stdev before interpolation)
    // ---- rollout: segments between inducing points ----
    int t = 0;
    for (int seg = 0; t < a.H; ++seg) {
      const int cnt = min(period, a.H - t);
      const bool full = (cnt == period);
      const float cntf = (float)cnt;
      const float w1x2 = full ? segW1x2_full : cntf * (cntf - 1.0f) / pf;
      const float w2 = full ? segW2_full : (cntf - 1.0f) * cntf * (2.0f * cntf - 1.0f) / (6.0f * pf * pf);
      L y0 = r.y1;
      if (seg == a.n_ind - 1) y0 = y0 * interp_last_point_weight(period);  // reference quirk: last point weighs 1/period (ctk_device.cuh)
      const L y1 = (seg + 1 < a.n_ind) ? ld_lanes<L>(sz + (size_t)(seg + 1) * ILP * T_, T_) * k.stdev : L(0.0f);
      r.y0 = y0;
      r.y1 = y1;
      r.dy = y1 - y0;
      // optimizer_mppi.py:154-155, du^2 term: cc_weight 0.5 (1 - 1/NU) R sum_j du_j^2
      const L sq = fmaf(r.dy, fmaf(w2, r.dy, w1x2 * y0), cntf * (y0 * y0));
      r.acc = fmaf(sq, k.k_du2, r.acc);
      if (PERIOD > 0 && full) {
#pragma unroll
        for (int j = 0; j < (PERIOD > 0 ? PERIOD : 1); ++j) {
          ode_mppi_step<KIND, LOG>(a, k, r, sh_unom[t + j], (float)j / (float)(PERIOD > 0 ? PERIOD : 1), j == 0, t + j, n, active);
        }
      } else {
#pragma unroll 2
        for (int j = 0; j < cnt; ++j) {
          ode_mppi_step<KIND, LOG>(a, k, r, sh_unom[t + j], sh_w[j].y, false, t + j, n, active);
        }
      }
      t += cnt;
      fold_segment(r);
    }

    // ---- per-rollout total + per-thread online softmin ----
#pragma unroll
    for (int q = 0; q < ILP; ++q) {
      const ScaledState rq = lane_of(r, q);
      if (LOG && active[q]) {
        float* p = a.log_traj_soa + (size_t)a.H * 6 * a.N + n[q];
        p[0] = rq.T * kSqrt2; p[a.N] = rq.W * k.inv_beta; p[2 * (size_t)a.N] = rq.c; p[3 * (size_t)a.N] = rq.s;
        p[4 * (size_t)a.N] = rq.x; p[5 * (size_t)a.N] = rq.V * k.inv_cFg;
      }
      // Cost_Functions/__init__.py:90-92 (mean over H+1 incl. the terminal cost); optimizer_mppi.py:160
#ifdef CTK_K1_DSUM
      const float S = finish_cost_scaled((float)r.dtot[q], rq, lane_of(r.ul, q), k);
#else
      const float S = finish_cost_scaled(lane_of(r.tot, q) - lane_of(r.comp, q), rq, lane_of(r.ul, q), k);
#endif
      if (active[q]) {
        a.J[n[q]] = S;
        if (S < INFINITY) {
          const float rho_n = fminf(rho_t, S);
          const float so = (rho_t < INFINITY) ? __expf((rho_t - rho_n) * k.neg_inv_lbd) : 0.0f;  // rescale the old sums
          const float sn = __expf((S - rho_n) * k.neg_inv_lbd);
          a_t = fmaf(a_t, so, sn);
          rho_t = rho_n;
          const float* szq = sz + q * T_;
          for (int i = 0; i < a.n_ind; ++i) {
            const size_t o = (size_t)i * T_;
            sa[o] = fmaf(sa[o], so, sn * szq[(size_t)i * ILP * T_]);
          }
        }
      }
    }
  }

  // ---- one block softmin record [rho_b, a_b, b_z[n_ind]]: column c is summed by warp c straight from shared memory ----
  trace(2);
  const float rho_b = block_min(rho_t, sh_red);
  trace(3);
  float* sh_sc = sh_z;        // the draws stash is free now: [T] rescale factors, [T] rescaled a_t
  float* sh_at = sh_z + T_;
  {
    const float sc = (rho_t < INFINITY) ? expf((rho_t - rho_b) * k.neg_inv_lbd) : 0.0f;
    sh_sc[tid] = sc;
    sh_at[tid] = a_t * sc;
  }
  __syncthreads();
  float* brec = sh_part;  // [P + 1]
  for (int c = w; c < P; c += nw) {
    float acc = 0.0f;
    if (c == 0) {
      for (int t = lane; t < T_; t += 32) acc += sh_at[t];
    } else {
      const float* col = sh_acc + (size_t)(c - 1) * T_;
      for (int t = lane; t < T_; t += 32) acc = fmaf(col[t], sh_sc[t], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) brec[1 + c] = acc;
  }
  if (tid == 0) brec[0] = rho_b;
  trace(4);
  mppi_tick_finish(a.fuse, brec, a.partials, a.n_ind, a.H, period, k.stdev, k.lo, k.hi, k.neg_inv_lbd, sh_unom, sh_w, brec + P + 1, sh_red, sh_z,
                   (int)((size_t)max(a.n_ind * ILP, 2) * T_ + (size_t)a.n_ind * T_));
  trace(5);
}

template <int KIND, bool LOG, int PERIOD, int ILP, int MAXT, bool INJ>
__global__ void __launch_bounds__(MAXT) mppi_ode_kernel(const MppiOdeArgs a) {
  mppi_ode_body<KIND, LOG, PERIOD, ILP, INJ>(a);
}

// ----------------------------------------------------------------------------------------------------------------
// Several clients' ticks in ONE launch (SURVEY 8f.4: the serving edge batches the states of several remote clients; reference
// controller_server/controller_server.py:55-86 serves one ctrl.step per request).  gridDim.y = client slot; every client has its
// own warm-start state (u_nom, u_prev), cost buffer, mailbox and Philox tick counter, laid out with fixed strides behind the
// pointers of client 0; the x-dimension of the grid is one client's ordinary K1 geometry, so a client's tick is bit-identical to
// the tick a handle of its own would run.  The state of client c travels inside the kernel parameters.  Inactive slots return at once.
// ----------------------------------------------------------------------------------------------------------------
template <int KIND, int PERIOD, int MAXT>
__global__ void __launch_bounds__(MAXT) mppi_ode_batch_kernel(const MppiOdeArgs a0, const MppiBatch b) {
  const int c = blockIdx.y;
  if (!b.active[c]) return;
  MppiOdeArgs a = a0;
  a.s0.p = nullptr;
#pragma unroll
  for (int i = 0; i < 6; ++i) a.s0.v[i] = b.s0[c][i];
  a.noise.tick = b.tick[c];
  a.u_nom += (size_t)c * b.stride_unom;
  a.u_prev += c;
  a.J += (size_t)c * b.stride_J;
  a.partials += (size_t)c * b.stride_partials;
  a.trace = nullptr;
  a.fuse.record_out += (size_t)c * b.stride_record;
  a.fuse.mbox_local += (size_t)c * b.stride_mbox;
  a.fuse.mbox_peer[0] = a.fuse.mbox_local;
  a.fuse.handover = nullptr;  // (no chained tick follows a batch launch)
  a.fuse.trace = nullptr;
  a.fuse.chained = 0;
  a.fuse.u_nom += (size_t)c * b.stride_unom;
  a.fuse.u_prev += c;
  a.fuse.u_out += 2 * c;
  a.fuse.host.p = nullptr;
  mppi_ode_body<KIND, false, PERIOD, 1, false>(a);
}

}  // namespace ctk
