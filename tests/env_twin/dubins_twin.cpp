// TEST INFRASTRUCTURE ONLY -- host twin of the Dubins car's adjoint.
// Compiles control_toolkit_b200/csrc/ctk_env_adjoint.h (the SAME source the gradient kernel of ctk_kernels_env_rpgd.cuh runs) for
// the CPU, with the reverse sweep of env_rpgd_grad_kernel, so that dJ/dQ can be checked against torch autograd of the oracle's
// DubinsPredictor + DubinsCost before any GPU time is spent.  tests/test_env_gradient_cpu.py is its only user.
#include <cmath>
#include <vector>

#include "../../control_toolkit_b200/csrc/ctk_env_adjoint.h"

using namespace ctk;

// the forward step of DubinsEnv::step in plain arithmetic
static void dubins_step(float* s, const float* u, const EnvParams& e) {
  const float v = e.p[1] * u[0], w = e.p[2] * u[1];
  const float cs = cosf(s[2]), sn = sinf(s[2]);
  s[0] = s[0] + (v * cs) * e.p[0];
  s[1] = s[1] + (v * sn) * e.p[0];
  const float yaw = s[2] + w * e.p[0];
  s[2] = atan2f(sinf(yaw), cosf(yaw));
}

extern "C" {

// s0 [N][3], Q [N][H][2], u_prev [2], p [np] (DubinsEnv parameter block) -> G [N][H][2] = dJ/dQ of the mean trajectory cost
void twin_dubins_grad(const float* s0, const float* Q, int N, int H, const float* u_prev, const float* p, int np, float* G) {
  EnvParams e{};
  for (int i = 0; i < np && i < 24; ++i) e.p[i] = p[i];
  constexpr int NS = DubinsAdjoint::NS, NU = DubinsAdjoint::NU;
  std::vector<float> tape((size_t)H * NS);
  const float w = 1.0f / (float)(H + 1);
  for (int n = 0; n < N; ++n) {
    const float* q = Q + (size_t)n * H * NU;
    float s[NS] = {s0[n * NS], s0[n * NS + 1], s0[n * NS + 2]};
    for (int t = 0; t < H; ++t) {
      for (int i = 0; i < NS; ++i) tape[(size_t)t * NS + i] = s[i];
      dubins_step(s, q + t * NU, e);
    }
    float lam[NS], carry[NU] = {0.0f, 0.0f};
    DubinsAdjoint::terminal_cost_grad(s, e, w, lam);
    for (int t = H - 1; t >= 0; --t) {
      const float* st = &tape[(size_t)t * NS];
      const float* u = q + t * NU;
      const float* up = t > 0 ? q + (t - 1) * NU : u_prev;
      float gu[NU] = {carry[0], carry[1]}, gp[NU] = {0.0f, 0.0f};
      DubinsAdjoint::step_adjoint(st, u, e, lam, gu);
      DubinsAdjoint::stage_cost_grad(st, u, up, e, w, lam, gu, gp);
      for (int c = 0; c < NU; ++c) {
        G[((size_t)n * H + t) * NU + c] = gu[c];
        carry[c] = gp[c];
      }
    }
  }
}

}  // extern "C"
