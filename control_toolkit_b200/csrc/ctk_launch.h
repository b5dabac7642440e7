// ctk_launch.h -- host-callable launch wrappers; each is defined in the translation unit that owns the kernels so the
// library builds as parallel nvcc jobs.  All launches are asynchronous on `st` and return cudaGetLastError().
#pragma once
#include <cuda_runtime.h>

#include "ctk_args.cuh"

#include <cstdlib>
#include <utility>

namespace ctk {

// Launch with programmatic stream serialization (see pdl_wait in ctk_device.cuh).  CTK_NO_PDL=1 falls back to plain launches.
inline bool pdl_enabled() {
  static const bool on = std::getenv("CTK_NO_PDL") == nullptr;
  return on;
}
template <typename... P, typename... A>
inline cudaError_t launch_pdl(void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<A>(args)...);
}

// The predictor functor a rollout kernel is instantiated with (ctk_predictor.cuh, ctk_mlp_tc.cuh)
enum class PredKind {
  Ode,        // OdePred: CartPole ODE
  MlpSimt,    // MlpSimtPred: MLP on the FP32 pipe
  MlpTc,      // MlpTcPred: MLP with layers 1 and 2 on tcgen05, bf16 x 3 split (fp32-level)
  MlpTcBf16,  // MlpTcBf16Pred: one bf16 product
  MlpTcFast,  // MlpTcFastPred: one bf16 product + MUFU.TANH
  Gru         // GruSimtPred: recurrent predictor on the FP32 pipe
};
// What the host needs to know about a predictor functor, read from its type (ctk_mppi.cu)
struct PredInfo {
  const char* name;           // the functor's name, as in the rollout kernel's instantiation
  int max_threads;            // kMaxThreads: block size of the MPPI rollout kernel
  int rollouts_per_pass;      // kRolloutsPerBlock: > 0 for the tile engines (a pass of a block covers that many rollouts), else 0
  bool balanced;              // kBalanced: one CTA per SM, each an equal contiguous share of the population
  size_t acc_smem_bytes;      // tile engines: shared memory left for the MPPI accumulators [n_ind][rollouts_per_pass]
  size_t (*smem_floats)(const MlpDev&);  // dynamic shared memory of the functor
};
PredInfo pred_info(PredKind pred);
// kind: cost class; log: write SoA trajectory logs
cudaError_t launch_mppi_rollout(PredKind pred, int kind, bool log, int nblocks, int block, size_t smem, cudaStream_t st, const MppiArgs& a);
// K1 for the ODE predictor with intermediate_steps == 1 (scaled variables, ILP rollouts per thread)
cudaError_t launch_mppi_ode(int kind, bool log, int period_t, int ilp, int grid, int block, size_t smem, cudaStream_t st, const MppiOdeArgs& a,
                            const char** name = nullptr);
int mppi_ode_max_block(int ilp, bool log);
// several clients' ticks in one launch: grid (grid, nclients); Philox noise, logging off, ILP 1 (ctk_batch.cu)
cudaError_t launch_mppi_ode_batch(int kind, int period_t, int grid, int nclients, int block, size_t smem, cudaStream_t st, const MppiOdeArgs& a,
                                  const MppiBatch& b);
size_t mppi_ode_smem_bytes(int H, int period, int n_ind, int ilp, int block);
cudaError_t launch_mppi_combine(const float* in, int cnt, int n_ind, float neg_inv_lbd, float* record_out,
                                const MppiFinalize& fin, cudaStream_t st);
cudaError_t launch_exchange_barrier(const MppiFuse& f, size_t bar_off, cudaStream_t st);
cudaError_t launch_transpose(const float* in, float* out, int R, int C, cudaStream_t st);
// top-M logging: gather the rows of the rollouts named by m sorted K4 keys out of an SoA [R][N] or reference-layout [N][R] log
cudaError_t launch_log_gather(const uint64_t* keys, int m, int off, const float* J, size_t N, const float* src, int R, int soa, float* out,
                              float* J_out, int32_t* idx_out, cudaStream_t st);
// environments beyond the CartPole (ctk_env.cu): MPPI = rollout + update launches, CEM = rollout, K4 levels, refit
cudaError_t launch_env_mppi(int env, bool log, const EnvMppiArgs& a, cudaStream_t st);
cudaError_t launch_env_cem_rollout(int env, bool log, const EnvCemArgs& a, cudaStream_t st);
cudaError_t launch_env_cem_refit(const EnvCemRefitArgs& a, cudaStream_t st);
void env_dims(int env, int* ns, int* nu);
// gradient kernel on environments (ctk_kernels_env_rpgd.cuh), + fused K8 when fused_select != null (N <= 32); smem: its shared-memory
// tape at horizon H
cudaError_t launch_env_rpgd_grad(int env, bool log, size_t smem, cudaStream_t st, const EnvRpgdGradArgs& a, const RpgdSelectArgs* fused_select);
size_t env_rpgd_smem_bytes(int env, int H);
// recurrent predictor (ctk_gru.cu)
cudaError_t launch_mppi_rollout_gru(int kind, bool log, int nblocks, int block, size_t smem, cudaStream_t st, const MppiArgs& a);
cudaError_t launch_cem_rollout_gru(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemArgs& a);
cudaError_t launch_single_rollout_gru(const float* s0, const float* Q, int H, const DevConsts* kc, const MlpDev& mlp, const float* u_prev,
                                      float* traj, float* summed, cudaStream_t st);
cudaError_t launch_gru_update(const S0& s0, const float* u_nom, const MlpDev& mlp, float* rnn_h, cudaStream_t st);

cudaError_t launch_cem_rollout(PredKind pred, int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemArgs& a);
int cem_rollout_grid(PredKind pred, int N, int num_sms);
cudaError_t launch_cem_ode(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemOdeArgs& a);
cudaError_t launch_cem_tick(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemTickArgs& a);
int cem_tick_rollouts_per_block();
int cem_tick_blocks_per_sm(int kind, bool log, size_t smem);
cudaError_t launch_topk_level(const float* cost, const uint64_t* keys_in, int n, int off, int k, uint64_t* out, cudaStream_t st);
cudaError_t launch_cem_refit(const CemRefitArgs& a, cudaStream_t st);

// coef: coefficient-form adjoint (rpgd_grad_coef_kernel, tape of 12 floats per step) instead of the direct form (8 floats per step)
// fused_select != null (coef only, one block): the select / resample step (K8) runs at the end of the same launch
cudaError_t launch_rpgd_grad(int kind, bool log, bool coef, int nblocks, int block, size_t smem, cudaStream_t st, const RpgdGradArgs& a,
                             const RpgdSelectArgs* fused_select = nullptr);
// population steps of every gradient optimizer over nu control inputs (ctk_kernels_rpgd_select.cuh): K8, initial population,
// gradient-assisted CEM sample / refit; nu outside {1, 2} -> cudaErrorInvalidValue
cudaError_t launch_rpgd_select(int nu, const RpgdSelectArgs& a, cudaStream_t st);
cudaError_t launch_rpgd_init(int nu, const RpgdSelectArgs& a, cudaStream_t st);
cudaError_t launch_gradcem_sample(int nu, const GradCemSampleArgs& a, cudaStream_t st);
cudaError_t launch_gradcem_refit(int nu, const GradCemRefitArgs& a, cudaStream_t st);

// ODE -> OdePred, GRU -> the GRU kernel, every MLP engine -> MlpSimtPred (one rollout: no tile to fill)
cudaError_t launch_single_rollout(PredKind pred, const float* s0, const float* Q, int H, const DevConsts* kc, const MlpDev& mlp, const float* u_prev, float* traj, float* summed, cudaStream_t st);
cudaError_t launch_fma_peak(float* out, int blocks, int threads, int iters, cudaStream_t st);
cudaError_t launch_fp32_micro(int variant, float* out, int blocks, int threads, int iters, const float* seed, cudaStream_t st);
cudaError_t launch_philox_fill(const NoiseSrc& ns, float* out, size_t n, cudaStream_t st);
cudaError_t launch_philox_export(const NoiseSrc& ns, size_t row0, float* out, size_t n, cudaStream_t st);

}  // namespace ctk
