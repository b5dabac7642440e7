// ctk_env_rpgd.cu -- translation unit owning the gradient kernel of the general environments (ctk_kernels_env_rpgd.cuh).
// A unit of its own: the shared-memory kernels here would otherwise change the reserved shared memory of ctk_env.cu's kernels.
#include "ctk_kernels_env_rpgd.cuh"
#include "ctk_launch.h"

namespace ctk {

cudaError_t launch_env_rpgd_grad(int env, bool log, size_t smem, cudaStream_t st, const EnvRpgdGradArgs& a, const RpgdSelectArgs* fused_select) {
  if (env != 1) return cudaErrorInvalidValue;
  void (*k)(const EnvRpgdGradArgs, const RpgdSelectArgs, const int) =
      log ? env_rpgd_grad_kernel<DubinsEnv, true> : env_rpgd_grad_kernel<DubinsEnv, false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const RpgdSelectArgs none{};
  k<<<(a.N + kEnvRpgdBlock - 1) / kEnvRpgdBlock, kEnvRpgdBlock, smem, st>>>(a, fused_select ? *fused_select : none, fused_select ? 1 : 0);
  return cudaGetLastError();
}
size_t env_rpgd_smem_bytes(int env, int H) {
  int ns, nu;
  env_dims(env, &ns, &nu);
  return sizeof(float) * (size_t)H * kEnvRpgdBlock * env_rpgd_tape_floats(ns, nu);
}
}  // namespace ctk
