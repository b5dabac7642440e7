// ctk_kernels_mppi.cuh -- K1 fused sample -> rollout -> cost -> block softmin partials, K2 combine / u_nom update.
// Replaces reference optimizer_mppi.py:170-193 (_predict_and_cost) for one tick.
#pragma once
#include "ctk_device.cuh"
#include "ctk_predictor.cuh"

namespace ctk {

// One rollout step shared by the segment loops: interpolated perturbation, clip, stage cost, MPPI correction, predictor.
// acc accumulates  mean-scaled stage cost + MPPI correction  (S = J + corr, optimizer_mppi.py:160) in one register.
struct MppiK {  // loop-invariant scalars of K1, register-resident
  float lo, hi, k_du2, k_udu;
};

// One rollout step: interpolated perturbation, clip, stage cost, MPPI correction, predictor.
// acc accumulates  mean-scaled stage cost + MPPI correction  (S = J + corr, optimizer_mppi.py:160) in one register.
template <class Pred, int KIND, bool LOG, bool SINGLE>
__device__ __forceinline__ void mppi_step(const MppiArgs& a, const CostC& cost, const MppiK& k, Pred& pred, State& z, float& omc,
                                          float& u_last, float& acc, float u_nom_t, float y0, float y1, float2 w, int t, int n,
                                          bool active) {
  // Interpolator.py:97-106: delta_u[t] = sum_i y_i W[i,t]  (two non-zero terms)
  const float du = fmaf(y1, w.y, __fmul_rn(y0, w.x));
  const float u = fminf(fmaxf(__fadd_rn(u_nom_t, du), k.lo), k.hi);  // :186-187
  if (LOG && active) {
    float* p = a.log_traj_soa + (size_t)t * 6 * a.N + n;
    p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
    a.log_Q_soa[(size_t)t * a.N + n] = u;
  }
  // cost.k_cc here carries  k_cc(cost) + cc_weight * 0.5 R  (both multiply u^2; merged by the caller)
  stage_cost_acc<KIND>(acc, z, omc, u, u_last, cost);
  // :154-155  cc_weight * (0.5(1-1/NU) R du^2 + R u du [+ 0.5 R u^2 merged above]) = du * (k_udu u + k_du2 du)
  acc = fmaf(du * du, k.k_du2, acc);
  acc = fmaf(u * du, k.k_udu, acc);
  if (SINGLE) pred.substep(z, u, omc); else pred.step(z, u, omc);
  u_last = u;
}

// ----------------------------------------------------------------------------------------------------------------
// Tick finish inside the rollout kernel (MppiFuse): combine softmin records, exchange across GPUs, update u_nom.
// ----------------------------------------------------------------------------------------------------------------
// Poll the nrec records rec_ptr(m) (P tagged slots each, stride even: 16-byte loads) until all their sequence numbers match;
// values -> dst[m * P + c] (dst may be null: wait only).  Thread t owns records t, t + blockDim, ...: all loads of a record are in
// flight before the first tag is checked, and a thread's records are polled in turn, so after the LAST record of the tick has
// landed the poll completes within one or two L2 round trips.  Returns 0, or 1 if a record did not arrive within ~2 s.
template <class RecPtr>
__device__ __forceinline__ int poll_records(RecPtr rec_ptr, int nrec, int P, unsigned int seq, unsigned long long t0, float* dst) {
  constexpr int MAXP2 = 8;  // up to 16 slots (n_ind <= 14) per record take the fast path
  const int tid = threadIdx.x, T = blockDim.x;
  const int P2 = (P + 1) >> 1;
  int lost = 0;
  if (P2 <= MAXP2) {
    unsigned int pending = 0;  // bit j: record tid + j * T still missing
    const int mine = (nrec - tid + T - 1) / T;  // records owned by this thread
    for (int j = 0; j < mine && j < 32; ++j) pending |= 1u << j;
    int spins = 0;
    while (pending) {
      for (int j = 0; j < mine && j < 32; ++j) {
        if (!(pending & (1u << j))) continue;
        const int m = tid + j * T;
        const unsigned long long* p = rec_ptr(m);
        unsigned long long v[2 * MAXP2];
#pragma unroll
        for (int q = 0; q < MAXP2; ++q)
          if (q < P2) asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(v[2 * q]), "=l"(v[2 * q + 1]) : "l"(p + 2 * q) : "memory");
        bool ok = true;
#pragma unroll
        for (int c = 0; c < 2 * MAXP2; ++c)
          if (c < P) ok = ok && ((unsigned int)(v[c] >> 32) == seq);
        if (ok) {
          if (dst != nullptr) {
#pragma unroll
            for (int c = 0; c < 2 * MAXP2; ++c)
              if (c < P) dst[m * P + c] = __uint_as_float((unsigned int)(v[c] & 0xffffffffull));
          }
          pending &= ~(1u << j);
        }
      }
      if (pending && (++spins & 255) == 0 && globaltimer_ns() - t0 > 2000000000ull) { lost = 1; break; }
    }
    if (mine > 32) lost = 1;  // (cannot happen: nrec <= 8 x 320 records over >= 128 threads)
  } else {  // many inducing points: slot by slot
    for (int i = tid; i < nrec * P; i += T) {
      const int m = i / P, c = i - m * P;
      float v;
      if (!ld_tagged(rec_ptr(m) + c, seq, t0, &v)) lost = 1;
      if (dst != nullptr) dst[i] = v;
    }
    // here a record's slots were stored by other threads than its owner (the fast path's thread m stores record m itself), and
    // staged_combine reads every record's rho before its first barrier
    if (dst != nullptr) __syncthreads();
  }
  return lost;
}

// records rec(b, c), b < cnt, c < P: [rho, a, b_z[n_ind]] -> out[P] (shared memory), rescaled exactly to the common minimum.
// Fallback for record sets that do not fit in shared memory (read through L2); every warp derives the common minimum itself.
template <class Rec>
__device__ __forceinline__ void combine_records(Rec rec, int cnt, int P, float neg_inv_lbd, float* out) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  if (w < P - 1) {
    float mn = INFINITY;
    for (int b = lane; b < cnt; b += 32) mn = fminf(mn, rec(b, 0));
    const float rho = warp_min(mn);
    for (int c = w; c < P - 1; c += nw) {
      float acc = 0.0f;
      for (int b = lane; b < cnt; b += 32) {
        const float rb = rec(b, 0);
        const float v = rec(b, 1 + c);
        const float sc = (rb < INFINITY) ? expf((rb - rho) * neg_inv_lbd) : 0.0f;
        acc = fmaf(sc, v, acc);
      }
      acc = warp_sum(acc);
      if (lane == 0) out[1 + c] = acc;
    }
    if (w == 0 && lane == 0) out[0] = rho;
  }
  __syncthreads();
}

// Combine nrec records staged in shared memory (big[m * P + c]) into out[P], rescaled exactly to their common minimum.  The
// summation order depends only on (nrec, P) -- never on the block size -- so every shard computes bit-identical results.
__device__ __forceinline__ void staged_combine(float* big, int nrec, int P, float neg_inv_lbd, int lost, unsigned int* sh_min,
                                               float* out, float* sh_half, int* status) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  // common minimum: the thread's own records (it has just written them) -> warp (redux) -> block (one shared atomic per warp)
  float mn = INFINITY;
  for (int m = tid; m < nrec; m += blockDim.x) mn = fminf(mn, big[m * P]);
  const unsigned int omin = __reduce_min_sync(0xffffffffu, float_to_ordered(mn));
  if (lane == 0) atomicMin(sh_min, omin);
  if (__syncthreads_or(lost)) *status = 1;
  const float rho = ordered_to_float(sh_min[0]);
  // rescale factors exp(-(rho_b - rho) / lambda), one per record, in place of rho_b
  for (int m = tid; m < nrec; m += blockDim.x) {
    const float rb = big[m * P];
    big[m * P] = (rb < INFINITY) ? expf((rb - rho) * neg_inv_lbd) : 0.0f;
  }
  __syncthreads();
  // column sums: (column, half) pairs over the warps; the two halves split the record range at a fixed point
  const int halves = nrec > 256 ? 2 : 1, split = halves == 2 ? (nrec + 1) / 2 : nrec;
  for (int idx = w; idx < (P - 1) * halves; idx += nw) {
    const int c = idx % (P - 1), hf = idx / (P - 1);
    const int b0 = hf == 0 ? 0 : split, b1 = hf == 0 ? split : nrec;
    float acc = 0.0f;
    for (int b = b0 + lane; b < b1; b += 32) acc = fmaf(big[b * P], big[b * P + 1 + c], acc);
    acc = warp_sum(acc);
    if (lane == 0) sh_half[hf * P + 1 + c] = acc;
  }
  __syncthreads();
  if (tid < P - 1) out[1 + tid] = halves == 2 ? sh_half[1 + tid] + sh_half[P + 1 + tid] : sh_half[1 + tid];
  if (tid == 0) out[0] = rho;
  __syncthreads();
}

// Called by ALL threads of EVERY block once the block's record brec[P] = [rho_b, a_b, b_z[n_ind]] is complete in SHARED
// memory (the call starts with a barrier).  mode 0: the record is stored as plain floats to partials[blockIdx.x][P] (a
// separate combine launch follows).  mode >= 1: every value is published as ONE 8-byte (value, sequence number) store -- no
// fence, no atomic, no ticket -- into this shard's mailbox and (mode 2, world > 1) straight into every peer's; block 0, the
// finisher, polls the world x grid records of its own mailbox until their tags match, combines them and updates u_nom.
// scratch: >= 3 * P + 2 floats of shared memory; sh_unom: the shifted nominal (prologue copy); wtab: [period] interpolation weights;
// big / big_floats: larger shared scratch -- when the records fit they are staged there by the polling pass itself.
// The summation order depends only on (world, grid, P) -- never on the block size -- so every shard, whatever its launch geometry,
// computes bit-identical results from the same records.
__device__ __forceinline__ void mppi_tick_finish(const MppiFuse& f, const float* brec, float* partials, int n_ind, int H,
                                                 int period, float stdev, float lo, float hi, float neg_inv_lbd,
                                                 const float* sh_unom, const float2* wtab, float* scratch, float* sh_red,
                                                 float* big = nullptr, int big_floats = 0) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5, P = n_ind + 2, G = (int)gridDim.x;
  unsigned int* sh_min = reinterpret_cast<unsigned int*>(sh_red);
  if (tid == 0) sh_min[0] = 0xffffffffu;
  __syncthreads();
  if (f.mode == 0) {
    for (int c = tid; c < P; c += blockDim.x) partials[(size_t)blockIdx.x * P + c] = brec[c];
    return;
  }
  const int world = (f.mode == 2) ? f.world : 1;
  const int rank = (world > 1) ? f.rank : 0;
  const int RS = mbox_record_stride(n_ind);
  const size_t base = (size_t)(f.seq & 1u) * CTK_MAX_PEERS * CTK_MBOX_BLOCKS * RS;  // parity buffer
  const size_t shard = (size_t)CTK_MBOX_BLOCKS * RS;                                  // slots per source shard
  {
    // hops == 1: the record goes straight to every shard (16-byte stores: two tagged slots per NVLink write); hops == 2: only to
    // this shard's own mailbox, the finisher forwards the shard's combined record
    const size_t mine = base + (size_t)rank * shard + (size_t)blockIdx.x * RS;
    const int dests = (world > 1 && f.hops != 2) ? world : 1;
    const int P2 = (P + 1) >> 1;
    for (int i = tid; i < dests * P2; i += blockDim.x) {
      const int r = i / P2, q = i - r * P2;
      unsigned long long* dst = (dests > 1 ? f.mbox_peer[r] : f.mbox_local) + mine + 2 * q;
      const unsigned long long x0 = ((unsigned long long)f.seq << 32) | (unsigned long long)__float_as_uint(brec[2 * q]);
      const unsigned long long x1 = ((unsigned long long)f.seq << 32) | (unsigned long long)__float_as_uint(2 * q + 1 < P ? brec[2 * q + 1] : 0.0f);
      asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(x0), "l"(x1) : "memory");
    }
  }
  if (blockIdx.x != 0) return;
  float* sh_rec = scratch;          // [P]
  float* sh_half = scratch + P;     // [2][P] partial column sums of the two halves of a large record set
  int status = 0;  // 0 ok, 1 a block record of this grid or of a peer shard did not arrive
  const unsigned long long t0 = globaltimer_ns();
  const int nrec = world * G;
  const unsigned long long* mb = f.mbox_local + base;
  auto rec_ptr = [&](int m) -> const unsigned long long* {  // record m of the world x G records that take part
    const int r = m / G, b = m - r * G;
    return mb + (size_t)r * shard + (size_t)b * RS;
  };
  // hops == 2: first this grid's G block records, then (after forwarding the shard's combined record) the world's shard records;
  // hops == 1 / one shard: all world x G block records at once.  A stage whose records fit into `big` is staged in shared memory by the
  // poll itself; otherwise the poll only waits and the combine reads the low words through L2.
  const int hops2 = (world > 1 && f.hops == 2) ? 1 : 0;
  auto stage = [&](auto rec, int n) {
    if (n * P <= big_floats) {
      const int lost = poll_records(rec, n, P, f.seq, t0, big);
      staged_combine(big, n, P, neg_inv_lbd, lost, sh_min, sh_rec, sh_half, &status);
    } else {
      const int lost = poll_records(rec, n, P, f.seq, t0, nullptr);
      if (__syncthreads_or(lost)) status = 1;
      combine_records([&](int b, int c) { return __ldcg(reinterpret_cast<const float*>(rec(b) + c)); }, n, P, neg_inv_lbd, sh_rec);
    }
  };
  if (hops2) {
    stage([&](int m) -> const unsigned long long* { return mb + (size_t)rank * shard + (size_t)m * RS; }, G);
    if (f.trace != nullptr && tid == 0) f.trace[6] = globaltimer_ns();
    // second hop: this shard's combined record -> every shard's mailbox (slot of block CTK_MBOX_BLOCKS - 1), then the world's
    const size_t mine2 = base + (size_t)rank * shard + (size_t)(CTK_MBOX_BLOCKS - 1) * RS;
    for (int i = tid; i < world * P; i += blockDim.x) {
      const int r = i / P, c = i - r * P;
      st_tagged(f.mbox_peer[r] + mine2 + c, sh_rec[c], f.seq);
    }
    if (tid == 0) sh_min[0] = 0xffffffffu;
    __syncthreads();
    stage([&](int m) -> const unsigned long long* { return mb + (size_t)m * shard + (size_t)(CTK_MBOX_BLOCKS - 1) * RS; }, world);
  } else {
    stage(rec_ptr, nrec);
    if (f.trace != nullptr && tid == 0) f.trace[6] = globaltimer_ns();
  }
  if (f.trace != nullptr && tid == 0) f.trace[7] = globaltimer_ns();
  if (f.record_out != nullptr)
    for (int c = tid; c < P; c += blockDim.x) f.record_out[c] = sh_rec[c];
  if (f.mode < 2) return;
  // optimizer_mppi.py:190-191: u_nom <- clip(shift(u_nom) + interp(sum_n w_n z_n) * stdev / sum_n w_n)
  const float a = sh_rec[1];
  for (int t = tid; t < H; t += blockDim.x) {
    const int seg = t / period, j = t - seg * period;
    const float2 wt = wtab[j];  // ((period - j)/period, j/period), Interpolator.py:63-74
    const float w0 = (seg == n_ind - 1) ? interp_last_point_weight(period) : wt.x;
    const float bz0 = sh_rec[2 + seg];
    const float bz1 = (j > 0) ? sh_rec[2 + seg + 1] : 0.0f;
    const float b = (fmaf(bz1, wt.y, bz0 * w0) * stdev) / a;
    const float un = fminf(fmaxf(sh_unom[t] + b, lo), hi);
    if (f.handover != nullptr && f.publish_handover) {  // first: the next tick of a chain is polling these
      st_tagged(f.handover + 1 + t, un, f.seq);
      if (t == 0) st_tagged(f.handover, f.freeze_prev ? f.u_prev[0] : un, f.seq);
    }
    f.u_nom[t] = un;
    if (f.host.p != nullptr) host_put(f.host, 8 + t, un);
    if (t == 0) {
      if (!f.freeze_prev) f.u_prev[0] = un;
      if (f.u_out != nullptr) { f.u_out[0] = status ? __int_as_float(0x7fc00000) : un; f.u_out[1] = (float)status; }
      if (f.host.p != nullptr) { host_put(f.host, 5, (float)status); host_put(f.host, 4, status ? __int_as_float(0x7fc00000) : un); }
    }
  }
}

// K1.  One CTA per SM slot, grid-stride over rollouts (host sizes grid x block so that every thread runs the same
// number of rollouts: no tail wave).  Each thread keeps an online softmin over its rollouts; the block emits ONE record
// [rho, a, b_z[n_ind]] at the end (a single block-wide reduction per launch).
template <class Pred, int KIND, bool LOG>
__global__ void __launch_bounds__(Pred::kMaxThreads, Pred::kMinBlocks) mppi_rollout_kernel(const MppiArgs a) {
  extern __shared__ float smem[];
  float* sh_unom = smem;                 // [H] shifted nominal
  float2* sh_w = reinterpret_cast<float2*>(smem + ((a.H + 1) & ~1));  // [period] interpolation weights (w0, w1)
  float* sh_red = reinterpret_cast<float*>(sh_w + a.period);          // [32] reduction scratch
  float* sh_part = sh_red + 32;          // [32][n_ind + 1] per-warp partial sums | block record | finish scratch
  float* sh_z = sh_part + 42 * (a.n_ind + 1) + 16;  // [n_ind][rpb] stash of this rollout's standard draws (if a.stash)
  // rollouts per block: blockDim, unless the predictor brings helper threads that own no rollout (MlpTcPred)
  const int rpb = Pred::kRolloutsPerBlock > 0 ? Pred::kRolloutsPerBlock : (int)blockDim.x;
  float* sh_acc = sh_z + (a.stash ? (size_t)a.n_ind * rpb : 0);  // [n_ind][rpb] per-thread sum_n e_n z_n,i
  float* sh_pred = sh_acc + (size_t)a.n_ind * rpb;

  for (int t = threadIdx.x; t < a.H; t += blockDim.x) sh_unom[t] = a.u_nom[min(t + 1, a.H - 1)];
  for (int j = threadIdx.x; j < a.period; j += blockDim.x) interp_weights(j, a.period, &sh_w[j].x, &sh_w[j].y);
  Pred pred(a.kc, a.mlp, sh_pred);
  pred.use_uniform(a.uk);
  CostC cost = load_cost(a.kc);
  // FMA-multiplier weights come from kernel parameters (uniform registers); uk.k_cc already carries
  // k_cc(cost) + cc_weight * 0.5 R: the cost's own R u^2 term and the correction's 0.5 R u^2 share one FMA
  cost.k_dd = a.uk.k_dd; cost.k_bar = a.uk.k_bar; cost.k_ep = a.uk.k_ep; cost.k_cc = a.uk.k_cc; cost.k_ccrc = a.uk.k_ccrc;
  const float* kx = a.kx;  // device copy of {lo, hi}
  const MppiK k = {vld(kx), vld(kx + 1), a.uk.k_du2, a.uk.k_udu};
  const float stdev = a.stdev;
  const bool single = pred.single_substep();
  __syncthreads();

  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  const int P = a.n_ind + 1;
  const int stride = gridDim.x * rpb;
  const bool owner = tid < rpb;  // this thread carries a rollout
  const int nblk = (a.n_ind + 3) >> 2;
  const State z0 = {a.s0.ld(0), a.s0.ld(1), a.s0.ld(2), a.s0.ld(3), a.s0.ld(4), a.s0.ld(5)};
  const float omc0 = 1.0f - cosf(z0.th);  // spec: E_pot uses cos(angle); for t >= 1 the state carries 1 - cos
  const float u_prev0 = a.u_prev[0];
  float* sz = sh_z + min(tid, rpb - 1);
  float* sa = sh_acc + min(tid, rpb - 1);
  if (owner)
    for (int i = 0; i < a.n_ind; ++i) sa[(size_t)i * rpb] = 0.0f;
  // per-thread online softmin over this thread's rollouts: rho_t = running min, a_t = sum e, sa[i] = sum e z_i
  float rho_t = INFINITY, a_t = 0.0f;
  const uint32_t a_unom = smem_u32(sh_unom), a_w = smem_u32(sh_w);

  // rollouts of this block: grid-stride passes of rpb rollouts, or (kBalanced) the block's contiguous, equal share of the population
  const int r_end = Pred::kBalanced ? (int)(((long long)blockIdx.x + 1) * a.N / gridDim.x) : a.N;
  const int r_first = Pred::kBalanced ? (int)((long long)blockIdx.x * a.N / gridDim.x) : (int)blockIdx.x * rpb;
  const int r_stride = Pred::kBalanced ? rpb : stride;
  for (int base = r_first; base < r_end; base += r_stride) {
    const int n = base + tid;
    const bool active = owner && n < r_end;
    const uint32_t ng = (uint32_t)(a.off + (active ? n : 0));
    float S = INFINITY;
    const bool grp = Pred::kCooperative && pred.group_active(base, r_end);  // (every thread: the tile engines note the tile's row count)
    if (active || grp) {
      State z = z0;
      float omc = omc0, u_last = u_prev0, acc = 0.0f;
      pred.begin_rollout(active);  // recurrent predictors: restore the saved hidden state; tile engines: is this row a real rollout
      const int nlog = active ? n : 0;
      // inducing-point draws arrive four at a time (one Philox block); zq is a rotating window, zq[0] = next draw
      float zq[4];
      noise4(a.noise, ng, 0, zq);
      if (a.stash && owner) sz[0] = zq[0];
      float y_prev = __fmul_rn(zq[0], stdev);  // :173-175  normal * stdev (before interpolation)
      zq[0] = zq[1]; zq[1] = zq[2]; zq[2] = zq[3];
      int have = 3, nextblk = 1, i = 1;  // i = next inducing point to load
      uint32_t pu = a_unom;
      int t = 0;
      while (t < a.H) {
        // segment [t, t + cnt): interpolate between inducing points i-1 (y_prev) and i (y_cur)
        float y_cur = 0.0f;  // past the last inducing point only j == 0 (weight 1 on y_prev) is ever evaluated
        if (i < a.n_ind) {
          if (have == 0) {
            noise4(a.noise, ng, (uint32_t)nextblk, zq);
            ++nextblk;
            have = 4;
          }
          if (a.stash && owner) sz[(size_t)i * rpb] = zq[0];
          y_cur = __fmul_rn(zq[0], stdev);
          zq[0] = zq[1]; zq[1] = zq[2]; zq[2] = zq[3];
          --have; ++i;
        } else {
          y_prev = __fmul_rn(y_prev, interp_last_point_weight(a.period));  // segment n_ind - 1: reference quirk (ctk_device.cuh)
        }
        const int cnt = min(a.period, a.H - t);
        uint32_t pw = a_w;
        if (single) {
#pragma unroll 2
          for (int j = 0; j < cnt; ++j, pu += 4, pw += 8)
            mppi_step<Pred, KIND, LOG, true>(a, cost, k, pred, z, omc, u_last, acc, lds_f32(pu), y_prev, y_cur, lds_f32x2(pw),
                                             t + j, nlog, active);
        } else {
#pragma unroll 1
          for (int j = 0; j < cnt; ++j, pu += 4, pw += 8)
            mppi_step<Pred, KIND, LOG, false>(a, cost, k, pred, z, omc, u_last, acc, lds_f32(pu), y_prev, y_cur, lds_f32x2(pw),
                                              t + j, nlog, active);
        }
        t += cnt;
        y_prev = y_cur;
      }

      if (LOG && active) {
        float* p = a.log_traj_soa + (size_t)a.H * 6 * a.N + n;
        p[0] = z.th; p[a.N] = z.om; p[2 * a.N] = z.c; p[3 * a.N] = z.s; p[4 * (size_t)a.N] = z.x; p[5 * (size_t)a.N] = z.v;
      }
      // Cost_Functions/__init__.py:90-92 (mean over H+1 incl. the terminal cost, constants pre-scaled) ; optimizer_mppi.py:160
      S = (acc + terminal_cost(z, cost)) - cost.shift;
      if (active) a.J[n] = S; else S = INFINITY;
    }

    // ---- per-thread online softmin (optimizer_mppi.py:163-168 restated incrementally; exact combine in K2) ----
    if (active && S < INFINITY) {
      const float rho_n = fminf(rho_t, S);
      const float so = (rho_t < INFINITY) ? __expf((rho_t - rho_n) * a.neg_inv_lbd) : 0.0f;  // rescale the old sums
      const float sn = __expf((S - rho_n) * a.neg_inv_lbd);
      a_t = fmaf(a_t, so, sn);
      rho_t = rho_n;
      if (a.stash) {
        for (int i = 0; i < a.n_ind; ++i) {
          const size_t o = (size_t)i * rpb;
          sa[o] = fmaf(sa[o], so, sn * sz[o]);
        }
      } else {
        for (int blk = 0; blk < nblk; ++blk) {
          float zz[4];
          noise4(a.noise, ng, blk, zz);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = blk * 4 + q;
            if (i < a.n_ind) {
              const size_t o = (size_t)i * rpb;
              sa[o] = fmaf(sa[o], so, sn * zz[q]);
            }
          }
        }
      }
    }
  }

  // ---- one block softmin record [rho_b, a_b, b_z[n_ind]] ----
  const float rho_b = block_min(rho_t, sh_red);
  const float sc = (rho_t < INFINITY) ? expf((rho_t - rho_b) * a.neg_inv_lbd) : 0.0f;
  {
    const float ws = warp_sum(a_t * sc);
    if (lane == 0) sh_part[w * P] = ws;
  }
  for (int i = 0; i < a.n_ind; ++i) {
    const float ws = warp_sum((owner ? sa[(size_t)i * rpb] : 0.0f) * sc);
    if (lane == 0) sh_part[w * P + 1 + i] = ws;
  }
  __syncthreads();
  float* brec = sh_part + 32 * P;  // [P + 1] block record, behind the per-warp partial sums
  for (int c = tid; c < P; c += blockDim.x) {
    float s = 0.0f;
    for (int ww = 0; ww < nw; ++ww) s += sh_part[ww * P + c];
    brec[1 + c] = s;
  }
  if (tid == 0) brec[0] = rho_b;
  // fused K2 (+ cross-GPU exchange): block 0 finishes the tick
  mppi_tick_finish(a.fuse, brec, a.partials, a.n_ind, a.H, a.period, a.stdev, a.lo, a.hi, a.neg_inv_lbd, sh_unom, sh_w, brec + P + 1,
                   sh_red, sh_z, (int)((a.stash ? (size_t)a.n_ind * rpb : 0) + (size_t)a.n_ind * rpb));
}

static __global__ void __launch_bounds__(1024) mppi_combine_kernel(const float* __restrict__ in, int cnt, int n_ind,
                                                           float neg_inv_lbd, float* __restrict__ record_out,
                                                           const MppiFinalize fin) {
  extern __shared__ float smem[];
  float* sh_red = smem;            // [32]
  float* sh_rec = smem + 32;       // [2 + n_ind]
  float* sh_u = sh_rec + 2 + n_ind;  // [H] (finalize)
  const int P = n_ind + 2;

  float mn = INFINITY;
  for (int b = threadIdx.x; b < cnt; b += blockDim.x) mn = fminf(mn, in[(size_t)b * P]);
  const float rho = block_min(mn, sh_red);
  for (int c = 0; c < n_ind + 1; ++c) {
    float acc = 0.0f;
    for (int b = threadIdx.x; b < cnt; b += blockDim.x) {
      const float rb = in[(size_t)b * P];
      const float sc = (rb < INFINITY) ? expf((rb - rho) * neg_inv_lbd) : 0.0f;
      acc = fmaf(sc, in[(size_t)b * P + 1 + c], acc);
    }
    const float tot = block_sum(acc, sh_red);
    if (threadIdx.x == 0) sh_rec[1 + c] = tot;
  }
  if (threadIdx.x == 0) sh_rec[0] = rho;
  __syncthreads();
  if (record_out != nullptr)
    for (int c = threadIdx.x; c < P; c += blockDim.x) record_out[c] = sh_rec[c];
  if (!fin.enable) return;

  for (int t = threadIdx.x; t < fin.H; t += blockDim.x) sh_u[t] = fin.u_nom[min(t + 1, fin.H - 1)];
  __syncthreads();
  const float a = sh_rec[1];
  for (int t = threadIdx.x; t < fin.H; t += blockDim.x) {
    const int seg = t / fin.period, j = t - seg * fin.period;
    float w0, w1;
    interp_weights(seg, j, fin.period, fin.n_ind, &w0, &w1);
    const float bz0 = sh_rec[2 + seg];
    const float bz1 = (j > 0) ? sh_rec[2 + seg + 1] : 0.0f;
    const float b = (fmaf(bz1, w1, bz0 * w0) * fin.stdev) / a;
    const float un = fminf(fmaxf(sh_u[t] + b, fin.lo), fin.hi);
    fin.u_nom[t] = un;
    if (t == 0) {
      if (!fin.freeze_prev) fin.u_prev[0] = un;
      if (fin.u_out != nullptr) fin.u_out[0] = un;
    }
  }
}

// [R][C] -> [C][R] tiled transpose (logs are produced SoA/coalesced by the rollout kernels and handed out in the
// reference's [N, H+1, ns] / [N, H, nu] layout)
static __global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int R, int C) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < R && c < C) tile[i][threadIdx.x] = in[(size_t)r * C + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < R && c < C) out[(size_t)c * R + r] = tile[threadIdx.x][i];
  }
}

// Top-M logging (SURVEY 8f.2 "optional top-M-only logging"; consumer: reference Controllers/__init__.py:159-178): rows of the M
// lowest-cost rollouts out of the logs of the last tick.  keys: the M sorted (ordered cost | global id) keys of K4.  src is either
// the SoA log [R][N] the CartPole kernels write (soa != 0) or a log in the reference's layout [N][R]; out is [M][R].
// Block j gathers rollout keys[j]; also J[j] and the global rollout id.
static __global__ void log_gather_kernel(const uint64_t* __restrict__ keys, int off, const float* __restrict__ J, size_t N, const float* __restrict__ src,
                                         int R, int soa, float* __restrict__ out, float* __restrict__ J_out, int32_t* __restrict__ idx_out) {
  const int j = blockIdx.x;
  const uint32_t g = (uint32_t)(keys[j] & 0xffffffffull);
  const size_t n = (size_t)g - (size_t)off;
  if (src != nullptr)
    for (int r = threadIdx.x; r < R; r += blockDim.x) out[(size_t)j * R + r] = soa ? src[(size_t)r * N + n] : src[n * R + r];
  if (threadIdx.x == 0) {
    if (J_out != nullptr) J_out[j] = J[n];
    if (idx_out != nullptr) idx_out[j] = (int32_t)g;
  }
}

}  // namespace ctk
