// ctk_mppi.cu -- translation unit owning the MPPI kernels (K1, K2), the log transpose and the nominal rollout.
#include "ctk_kernels_mppi.cuh"
#include "ctk_kernels_mppi_ode.cuh"
#include "ctk_mlp_tc.cuh"
#include "ctk_launch.h"

namespace ctk {

template <class Pred, int KIND, bool LOG>
static cudaError_t launch_mppi_t(int nblocks, int block, size_t smem, cudaStream_t st, const MppiArgs& a) {
  auto k = mppi_rollout_kernel<Pred, KIND, LOG>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  k<<<nblocks, block, smem, st>>>(a);
  return cudaGetLastError();
}
template <class Pred>
static cudaError_t launch_mppi_p(int kind, bool log, int nblocks, int block, size_t smem, cudaStream_t st, const MppiArgs& a) {
  if (kind == 0) return log ? launch_mppi_t<Pred, 0, true>(nblocks, block, smem, st, a) : launch_mppi_t<Pred, 0, false>(nblocks, block, smem, st, a);
  return log ? launch_mppi_t<Pred, 1, true>(nblocks, block, smem, st, a) : launch_mppi_t<Pred, 1, false>(nblocks, block, smem, st, a);
}
cudaError_t launch_mppi_rollout(PredKind pred, int kind, bool log, int nblocks, int block, size_t smem, cudaStream_t st, const MppiArgs& a) {
  switch (pred) {
    case PredKind::Ode: return launch_mppi_p<OdePred>(kind, log, nblocks, block, smem, st, a);
    case PredKind::MlpSimt: return launch_mppi_p<MlpSimtPred>(kind, log, nblocks, block, smem, st, a);
    case PredKind::MlpTc: return launch_mppi_p<MlpTcPred>(kind, log, nblocks, block, smem, st, a);
    case PredKind::MlpTcBf16: return launch_mppi_p<MlpTcBf16Pred>(kind, log, nblocks, block, smem, st, a);
    case PredKind::MlpTcFast: return launch_mppi_p<MlpTcFastPred>(kind, log, nblocks, block, smem, st, a);
    case PredKind::Gru: return launch_mppi_rollout_gru(kind, log, nblocks, block, smem, st, a);  // ctk_gru.cu
  }
  return cudaErrorInvalidValue;
}

template <class Pred>
static PredInfo pred_info_of(const char* name) {
  PredInfo i{name, Pred::kMaxThreads, Pred::kRolloutsPerBlock, Pred::kBalanced, 0, &Pred::smem_floats};
  if constexpr (Pred::kRolloutsPerBlock > 0) i.acc_smem_bytes = Pred::kAccSmemBytes;
  return i;
}
PredInfo pred_info(PredKind pred) {
  switch (pred) {
    case PredKind::Ode: return pred_info_of<OdePred>("OdePred");
    case PredKind::MlpSimt: return pred_info_of<MlpSimtPred>("MlpSimtPred");
    case PredKind::MlpTc: return pred_info_of<MlpTcPred>("MlpTcPred");
    case PredKind::MlpTcBf16: return pred_info_of<MlpTcBf16Pred>("MlpTcBf16Pred");
    case PredKind::MlpTcFast: return pred_info_of<MlpTcFastPred>("MlpTcFastPred");
    case PredKind::Gru: return pred_info_of<GruSimtPred>("GruSimtPred");
  }
  return {};
}

#ifndef CTK_K1_MAXT2
#define CTK_K1_MAXT2 896
#endif
constexpr int k1_maxt(bool log, int ilp) { return ilp == 2 ? (log ? 768 : CTK_K1_MAXT2) : 1024; }
// K1 for the ODE predictor (ctk_kernels_mppi_ode.cuh).  period_t: 10 -> the segment-unrolled instantiation, else runtime period.
template <int KIND, bool LOG, int PERIOD, int ILP, bool INJ>
static cudaError_t launch_mppi_ode_t(int grid, int block, size_t smem, cudaStream_t st, const MppiOdeArgs& a) {
  // __launch_bounds__ caps the registers at 65536 / MAXT.  Two rollouts per thread need ~70 registers, the logging instantiations more
  // (seven store addresses per rollout): under a bound of 1024 threads ptxas spilled inside the step loop (measured on the same box
  // against the round-1 build: -3 % at C5, -13 % with logging on) -> ILP = 2: blocks of at most 896 threads, logging: 768.
  auto k = mppi_ode_kernel<KIND, LOG, PERIOD, ILP, k1_maxt(LOG, ILP), INJ>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  // A tick of a back-to-back chain (ctk_step_device_n) is launched with programmatic stream serialization: its blocks are scheduled as
  // the previous tick's retire and run their state-independent prologue before the hand-over arrives (ctk_kernels_mppi_ode.cuh).  A
  // single tick gains nothing from the attribute and starts ~1.5 us later with it (measured at C1: event pair 15.3 vs 17.1 us).
  if (a.fuse.chained) return launch_pdl(k, dim3(grid), dim3(block), smem, st, a);
  k<<<grid, block, smem, st>>>(a);
  return cudaGetLastError();
}
// production instantiations: Philox noise only; injected noise (verification) and odd periods with logging run the
// generic-period, one-rollout-per-thread instantiation (any launch geometry is valid for it: grid-stride loop)
template <int KIND>
static cudaError_t launch_mppi_ode_k(bool log, int period_t, int ilp, int grid, int block, size_t smem, cudaStream_t st, const MppiOdeArgs& a,
                                     const char** name) {
  // template arguments after KIND: LOG, PERIOD, ILP, MAXT (k1_maxt), INJ
#define CTK_ODE_CASE(LOG_, P_, I_, INJ_)                                                  \
  do {                                                                                    \
    if (name) *name = (I_ == 2) ? ((LOG_) ? "," #LOG_ "," #P_ "," #I_ ",768," #INJ_ ">" : "," #LOG_ "," #P_ "," #I_ ",896," #INJ_ ">") \
                                : "," #LOG_ "," #P_ "," #I_ ",1024," #INJ_ ">";                       \
    return launch_mppi_ode_t<KIND, LOG_, P_, I_, INJ_>(grid, block, smem, st, a);         \
  } while (0)
  if (a.noise.inj != nullptr) {
    if (log) CTK_ODE_CASE(1, 0, 1, 1);
    CTK_ODE_CASE(0, 0, 1, 1);
  }
  if (log) {  // trajectory logging with in-kernel noise: HBM-write bound, the fast loop keeps the stores fed
    if (period_t == 10) {
      if (ilp == 2) CTK_ODE_CASE(1, 10, 2, 0);
      CTK_ODE_CASE(1, 10, 1, 0);
    }
    CTK_ODE_CASE(1, 0, 1, 1);
  }
  if (period_t == 10) {
    if (ilp == 2) CTK_ODE_CASE(0, 10, 2, 0);
    CTK_ODE_CASE(0, 10, 1, 0);
  }
  if (ilp == 2) CTK_ODE_CASE(0, 0, 2, 0);
  CTK_ODE_CASE(0, 0, 1, 0);
#undef CTK_ODE_CASE
}
// name (optional): the template-argument tail of the instantiation that was launched, e.g. ",0,10,2,896,0>" (after KIND)
cudaError_t launch_mppi_ode(int kind, bool log, int period_t, int ilp, int grid, int block, size_t smem, cudaStream_t st, const MppiOdeArgs& a,
                            const char** name) {
  return kind == 0 ? launch_mppi_ode_k<0>(log, period_t, ilp, grid, block, smem, st, a, name) : launch_mppi_ode_k<1>(log, period_t, ilp, grid, block, smem, st, a, name);
}
int mppi_ode_max_block(int ilp, bool log) { return k1_maxt(log, ilp); }
size_t mppi_ode_smem_bytes(int H, int period, int n_ind, int ilp, int block) {
  return sizeof(float) * ((size_t)((H + 3) & ~3) + 2 * ((period + 3) & ~3) + 32 + 12 * (size_t)(n_ind + 2) + (size_t)(n_ind * ilp > 2 ? n_ind * ilp : 2) * block + (size_t)n_ind * block);
}

cudaError_t launch_mppi_combine(const float* in, int cnt, int n_ind, float neg_inv_lbd, float* record_out,
                                const MppiFinalize& fin, cudaStream_t st) {
  const size_t sm = sizeof(float) * (32 + 2 + n_ind + (fin.enable ? fin.H : 0));
  mppi_combine_kernel<<<1, 1024, sm, st>>>(in, cnt, n_ind, neg_inv_lbd, record_out, fin);
  return cudaGetLastError();
}

// Cross-shard barrier on the device (bench.py: aligns the shards' streams before a timed tick so that skew accumulated OUTSIDE the
// timed region -- the un-synchronised L2 flush -- is not spent waiting inside the tick's exchange): every shard stores a tagged flag
// into every mailbox's barrier area and polls its own.
__global__ void exchange_barrier_kernel(MppiFuse f, size_t bar_off) {
  const int tid = threadIdx.x;
  const size_t o = bar_off + (size_t)(f.seq & 1u) * CTK_MAX_PEERS;
  if (tid < f.world) st_tagged(f.mbox_peer[tid] + o + f.rank, 1.0f, f.seq);
  if (tid < f.world) {
    float v;
    ld_tagged(f.mbox_local + o + tid, f.seq, globaltimer_ns(), &v);
  }
}
cudaError_t launch_exchange_barrier(const MppiFuse& f, size_t bar_off, cudaStream_t st) {
  exchange_barrier_kernel<<<1, 32, 0, st>>>(f, bar_off);
  return cudaGetLastError();
}

cudaError_t launch_transpose(const float* in, float* out, int R, int C, cudaStream_t st) {
  dim3 grid((C + 31) / 32, (R + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, st>>>(in, out, R, C);
  return cudaGetLastError();
}

cudaError_t launch_log_gather(const uint64_t* keys, int m, int off, const float* J, size_t N, const float* src, int R, int soa, float* out,
                              float* J_out, int32_t* idx_out, cudaStream_t st) {
  log_gather_kernel<<<m, 128, 0, st>>>(keys, off, J, N, src, R, soa, out, J_out, idx_out);
  return cudaGetLastError();
}

// nominal single rollout (reference optimizer_mppi.py:199-202 predict_optimal_trajectory, optimizer_rpgd.py:382-386)
template <class Pred>
__global__ void single_rollout_kernel(const float* s0, const float* Q, int H, const DevConsts* kc, MlpDev mlp,
                                      const float* u_prev, float* traj, float* summed) {
  extern __shared__ float smem[];
  Pred pred(kc, mlp, smem);
  const CostC cost = kc->cost;
  __syncthreads();
  if (threadIdx.x != 0) return;
  State z;
  z.th = s0[0]; z.om = s0[1]; z.c = s0[2]; z.s = s0[3]; z.x = s0[4]; z.v = s0[5];
  float omc = 1.0f - cosf(z.th), ul = u_prev[0], sum = 0.0f;
  pred.begin_rollout();
  for (int t = 0; t <= H; ++t) {
    float* p = traj + t * 6;
    p[0] = z.th; p[1] = z.om; p[2] = z.c; p[3] = z.s; p[4] = z.x; p[5] = z.v;
    if (t == H) break;
    const float u = Q[t];
    sum += stage_cost_dyn(cost.kind, z, omc, u, ul, cost);  // get_summed_stage_cost (Cost_Functions/__init__.py:71-72)
    pred.step(z, u, omc);
    ul = u;
  }
  summed[0] = (sum - cost.shift) * (float)(H + 1);  // the device constants carry the 1/(H+1) of the trajectory mean
}

cudaError_t launch_single_rollout(PredKind pred, const float* s0, const float* Q, int H, const DevConsts* kc, const MlpDev& mlp, const float* u_prev, float* traj, float* summed, cudaStream_t st) {
  if (pred == PredKind::Ode) {
    single_rollout_kernel<OdePred><<<1, 32, 0, st>>>(s0, Q, H, kc, mlp, u_prev, traj, summed);
    return cudaGetLastError();
  }
  if (pred == PredKind::Gru) return launch_single_rollout_gru(s0, Q, H, kc, mlp, u_prev, traj, summed, st);  // ctk_gru.cu
  const size_t smem = sizeof(float) * MlpSimtPred::smem_floats(mlp);
  auto k = single_rollout_kernel<MlpSimtPred>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  k<<<1, 128, smem, st>>>(s0, Q, H, kc, mlp, u_prev, traj, summed);
  return cudaGetLastError();
}

}  // namespace ctk
