// ctk_cem.cu -- translation unit owning the CEM kernels (K3 rollout, K4 top-k levels, K5 refit).
#include "ctk_kernels_cem.cuh"
#include "ctk_mlp_tc.cuh"
#include "ctk_launch.h"

namespace ctk {

template <class Pred, int KIND, bool LOG>
static cudaError_t launch_cem_t(int nblocks, size_t smem, cudaStream_t st, const CemArgs& a) {
  auto k = cem_rollout_kernel<Pred, KIND, LOG>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  return launch_pdl(k, dim3(nblocks), dim3(Pred::kCemThreads), smem, st, a);
}
template <class Pred>
static cudaError_t launch_cem_p(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemArgs& a) {
  if (kind == 0) return log ? launch_cem_t<Pred, 0, true>(nblocks, smem, st, a) : launch_cem_t<Pred, 0, false>(nblocks, smem, st, a);
  return log ? launch_cem_t<Pred, 1, true>(nblocks, smem, st, a) : launch_cem_t<Pred, 1, false>(nblocks, smem, st, a);
}
cudaError_t launch_cem_rollout(PredKind pred, int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemArgs& a) {
  switch (pred) {
    case PredKind::Ode: return launch_cem_p<OdePred>(kind, log, nblocks, smem, st, a);
    case PredKind::MlpSimt: return launch_cem_p<MlpSimtPred>(kind, log, nblocks, smem, st, a);
    case PredKind::MlpTc: return launch_cem_p<MlpTcPred>(kind, log, nblocks, smem, st, a);
    case PredKind::MlpTcBf16: return launch_cem_p<MlpTcBf16Pred>(kind, log, nblocks, smem, st, a);
    case PredKind::MlpTcFast: return launch_cem_p<MlpTcFastPred>(kind, log, nblocks, smem, st, a);
    case PredKind::Gru: return launch_cem_rollout_gru(kind, log, nblocks, smem, st, a);  // ctk_gru.cu
  }
  return cudaErrorInvalidValue;
}
cudaError_t launch_cem_ode(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemOdeArgs& a) {
  void (*k)(const CemOdeArgs) = nullptr;
  if (kind == 0) k = log ? cem_ode_kernel<0, true> : cem_ode_kernel<0, false>;
  else k = log ? cem_ode_kernel<1, true> : cem_ode_kernel<1, false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  return launch_pdl(k, dim3(nblocks), dim3(a.cand_out != nullptr ? kCemOdeTopkThreads : 128), smem, st, a);
}
// FAST instantiations: Philox normal draws (no injected queue, no uniform mode) -> straight-line noise generation
static void (*cem_tick_fn(int kind, bool log, bool fast))(const CemTickArgs) {
  if (kind == 0) {
    if (log) return fast ? cem_tick_kernel<0, true, true> : cem_tick_kernel<0, true, false>;
    return fast ? cem_tick_kernel<0, false, true> : cem_tick_kernel<0, false, false>;
  }
  if (log) return fast ? cem_tick_kernel<1, true, true> : cem_tick_kernel<1, true, false>;
  return fast ? cem_tick_kernel<1, false, true> : cem_tick_kernel<1, false, false>;
}
cudaError_t launch_cem_tick(int kind, bool log, int nblocks, size_t smem, cudaStream_t st, const CemTickArgs& a) {
  const bool fast = a.noise.inj == nullptr && !a.noise.uniform;
  void (*k)(const CemTickArgs) = cem_tick_fn(kind, log, fast);
  if (smem > 11 * 1024) {  // static shared memory comes on top
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  // The blocks of this kernel wait for each other (tagged-slot grid synchronisation), so the WHOLE grid must be co-resident: a
  // cooperative launch makes the runtime guarantee that -- or fail with cudaErrorCooperativeLaunchTooLarge, in which case the
  // caller takes the multi-launch path -- instead of relying on an occupancy query that assumes an otherwise idle GPU.
  static const bool coop = std::getenv("CTK_CEM_NO_COOP") == nullptr;
  if (!coop) return launch_pdl(k, dim3(nblocks), dim3(kCemTickThreads), smem, st, a);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(nblocks); cfg.blockDim = dim3(kCemTickThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k, a);
}
// grid of the generic CEM rollout kernel: one block per 128 rollouts; the tile engines run one CTA per SM with equal shares (kBalanced)
int cem_rollout_grid(PredKind pred, int N, int num_sms) {
  const int nb = (N + 127) / 128;
  return pred_info(pred).balanced ? (nb < num_sms ? nb : num_sms) : nb;
}
int cem_tick_rollouts_per_block() { return kCemTickRollouts; }
// resident blocks per SM of the persistent tick kernel (its blocks wait for each other: the whole grid must be resident)
int cem_tick_blocks_per_sm(int kind, bool log, size_t smem) {
  void (*k)(const CemTickArgs) = cem_tick_fn(kind, log, false);  // the generic instantiation needs at least as many registers
  if (smem > 11 * 1024 && cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return 0;
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, kCemTickThreads, smem) != cudaSuccess) return 0;
  return nb;
}
// Level 0: keys from costs (global index = off + i).  Each block sorts 1024 keys and emits its k smallest.
// Level >0: same on candidate keys.  out has gridDim.x * k keys.
__global__ void __launch_bounds__(TOPK_THREADS) topk_level_kernel(const float* __restrict__ cost, const uint64_t* __restrict__ keys_in,
                                                                   int n, int off, int k, uint64_t* __restrict__ out) {
  __shared__ uint64_t sh[TOPK_THREADS];
  const int i = blockIdx.x * TOPK_THREADS + threadIdx.x;
  uint64_t key = KEY_MAX;
  pdl_wait();
  pdl_trigger();
  if (i < n) key = (cost != nullptr) ? make_key(cost[i], (uint32_t)(off + i)) : keys_in[i];
  key = block_bitonic_sort(key, sh);
  if (threadIdx.x < k) out[(size_t)blockIdx.x * k + threadIdx.x] = key;
}

cudaError_t launch_topk_level(const float* cost, const uint64_t* keys_in, int n, int off, int k, uint64_t* out, cudaStream_t st) {
  const int nb = (n + TOPK_THREADS - 1) / TOPK_THREADS;
  return launch_pdl(topk_level_kernel, dim3(nb), dim3(TOPK_THREADS), 0, st, cost, keys_in, n, off, k, out);
}
cudaError_t launch_cem_refit(const CemRefitArgs& a, cudaStream_t st) {
  return launch_pdl(cem_refit_kernel, dim3(1), dim3(TOPK_THREADS), 0, st, a);
}

}  // namespace ctk
