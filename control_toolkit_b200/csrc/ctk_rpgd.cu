// ctk_rpgd.cu -- translation unit owning the CartPole RPGD gradient kernels (K6/K7), the population steps every environment shares
// (K8 select / resample, init, grad-CEM sample / refit) and utilities.
#include "ctk_kernels_rpgd.cuh"
#include "ctk_launch.h"

namespace ctk {

cudaError_t launch_rpgd_grad(int kind, bool log, bool coef, int nblocks, int block, size_t smem, cudaStream_t st, const RpgdGradArgs& a,
                             const RpgdSelectArgs* fused_select) {
  if (coef) {
    void (*k)(const RpgdGradArgs, const RpgdSelectArgs, const int) = nullptr;
    if (kind == 0) k = log ? rpgd_grad_coef_kernel<0, true> : rpgd_grad_coef_kernel<0, false>;
    else k = log ? rpgd_grad_coef_kernel<1, true> : rpgd_grad_coef_kernel<1, false>;
    if (smem > 32 * 1024) {  // 6 KB of static shared memory (fused select) come on top
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
    }
    const RpgdSelectArgs none{};
    return launch_pdl(k, dim3(nblocks), dim3(32 * kRpgdWarps), smem, st, a, fused_select ? *fused_select : none, fused_select ? 1 : 0);
  }
  void (*k)(const RpgdGradArgs) = nullptr;
  if (kind == 0) k = log ? rpgd_grad_kernel<0, true> : rpgd_grad_kernel<0, false>;
  else k = log ? rpgd_grad_kernel<1, true> : rpgd_grad_kernel<1, false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  return launch_pdl(k, dim3(nblocks), dim3(block), smem, st, a);
}

// the population steps are instantiated for nu = 1 (the CartPole) and nu = 2 (the Dubins car)
template <class A>
static cudaError_t launch_nu(int nu, void (*k1)(A), void (*k2)(A), unsigned grid, unsigned block, cudaStream_t st, const A& a) {
  if (nu != 1 && nu != 2) return cudaErrorInvalidValue;
  return launch_pdl(nu == 1 ? k1 : k2, dim3(grid), dim3(block), 0, st, a);
}
cudaError_t launch_rpgd_select(int nu, const RpgdSelectArgs& a, cudaStream_t st) {
  return launch_nu(nu, rpgd_select_kernel<1>, rpgd_select_kernel<2>, 1, TOPK_THREADS, st, a);
}
cudaError_t launch_rpgd_init(int nu, const RpgdSelectArgs& a, cudaStream_t st) {
  return launch_nu(nu, rpgd_init_kernel<1>, rpgd_init_kernel<2>, (a.N * a.H * nu + 255) / 256, 256, st, a);
}
cudaError_t launch_gradcem_sample(int nu, const GradCemSampleArgs& a, cudaStream_t st) {
  return launch_nu(nu, gradcem_sample_kernel<1>, gradcem_sample_kernel<2>, (a.cnt * a.H * nu + 255) / 256, 256, st, a);
}
cudaError_t launch_gradcem_refit(int nu, const GradCemRefitArgs& a, cudaStream_t st) {
  return launch_nu(nu, gradcem_refit_kernel<1>, gradcem_refit_kernel<2>, 1, TOPK_THREADS, st, a);
}

// FP32 FMA-chain microbenchmark: 8 independent chains per thread, 16x unrolled
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}
cudaError_t launch_fma_peak(float* out, int blocks, int threads, int iters, cudaStream_t st) {
  fma_peak_kernel<<<blocks, threads, 0, st>>>(out, iters, 0.999f, 0.001f);
  return cudaGetLastError();
}

// FP32 issue-rate microbenchmarks (DESIGN.md "what the FP32 pipe can actually issue"): 8 independent chains/thread.
//  1: FFMA with three distinct REGISTER sources   2: FMUL reg,reg   3: FADD reg,reg   4: FFMA(3 reg) + FMUL alternating
//  5: FFMA reg,reg,imm-free mix resembling the rollout body (2 FFMA : 1 FMUL : 0.25 FADD), all register operands
template <int V>
__global__ void __launch_bounds__(256) fp32_micro_kernel(float* out, int iters, const float* __restrict__ seed) {
  float x[8], y[8], z[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    x[i] = seed[(threadIdx.x + i) & 63];
    y[i] = seed[(threadIdx.x + 8 + i) & 63] * 1e-3f + 0.999f;
    z[i] = seed[(threadIdx.x + 16 + i) & 63] * 1e-3f;
  }
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (V == 1) x[i] = fmaf(x[i], y[i], z[i]);
        if (V == 2) x[i] = x[i] * y[i];
        if (V == 3) x[i] = x[i] + z[i];
        if (V == 4) { if (u & 1) x[i] = fmaf(x[i], y[i], z[i]); else x[i] = x[i] * y[i]; }
        if (V == 5) { if ((u & 3) == 3) x[i] = x[i] * y[(i + 1) & 7]; else x[i] = fmaf(x[i], y[i], z[(i + u) & 7]); }
      }
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += x[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
cudaError_t launch_fp32_micro(int variant, float* out, int blocks, int threads, int iters, const float* seed, cudaStream_t st) {
  switch (variant) {
    case 1: fp32_micro_kernel<1><<<blocks, threads, 0, st>>>(out, iters, seed); break;
    case 2: fp32_micro_kernel<2><<<blocks, threads, 0, st>>>(out, iters, seed); break;
    case 3: fp32_micro_kernel<3><<<blocks, threads, 0, st>>>(out, iters, seed); break;
    case 4: fp32_micro_kernel<4><<<blocks, threads, 0, st>>>(out, iters, seed); break;
    default: fp32_micro_kernel<5><<<blocks, threads, 0, st>>>(out, iters, seed); break;
  }
  return cudaGetLastError();
}

__global__ void philox_fill_kernel(NoiseSrc ns, float* out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = noise1(ns, (uint32_t)(i / ns.per_rollout), (int)(i % ns.per_rollout));
}
cudaError_t launch_philox_fill(const NoiseSrc& ns, float* out, size_t n, cudaStream_t st) {
  philox_fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ns, out, n);
  return cudaGetLastError();
}
// rows [row0, row0 + n / per_rollout) of a noise block, through the SAME device function the consumers call (noise4)
__global__ void philox_export_kernel(NoiseSrc ns, size_t row0, float* out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = noise1(ns, (uint32_t)(row0 + i / ns.per_rollout), (int)(i % ns.per_rollout));
}
cudaError_t launch_philox_export(const NoiseSrc& ns, size_t row0, float* out, size_t n, cudaStream_t st) {
  philox_export_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ns, row0, out, n);
  return cudaGetLastError();
}

}  // namespace ctk
