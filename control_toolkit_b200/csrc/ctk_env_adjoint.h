// ctk_env_adjoint.h -- reverse-mode members of the environment contract (ctk_kernels_env.cuh), for the gradient optimizers (RPGD,
// gradient-tf, the gradient-assisted CEM variants) on registered environments.  The trajectory cost of the reference
// (Cost_Functions/__init__.py:74-93) is J = w (sum_t l(s_t, u_t, u_{t-1}) + T(s_H)) with w = 1 / (H + 1); every member below is scaled
// by w.  lam[NS] is dJ/ds, gu[NU] is dJ/du; the members ADD to them.  Plain arithmetic in CTK_HD functions: the kernels and the CPU
// twin of the tests (tests/env_twin) compile this same source.  Gradients of indicator terms (the obstacle) are zero, like the
// CartPole's track barrier; the yaw wrap atan2(sin, cos) has unit gradient.
#pragma once
#include <math.h>

#include "ctk_args.cuh"

namespace ctk {

// Dubins car (ctk_kernels_env.cuh DubinsEnv): x' = x + h v cos(yaw), y' = y + h v sin(yaw), yaw' = wrap(yaw + h omega),
// v = v_max u0, omega = omega_max u1; parameter block as DubinsEnv
struct DubinsAdjoint {
  static constexpr int NS = 3, NU = 2;
  // lam: adjoint after the step -> before it; gu += dJ/du through the dynamics (s: the state before the step)
  static CTK_HD void step_adjoint(const float* s, const float* u, const EnvParams& e, float* lam, float* gu) {
    const float h = e.p[0], cs = cosf(s[2]), sn = sinf(s[2]);
    const float hv = h * (e.p[1] * u[0]);
    gu[0] += e.p[1] * h * (lam[0] * cs + lam[1] * sn);
    gu[1] += e.p[2] * h * lam[2];
    lam[2] += hv * (lam[1] * cs - lam[0] * sn);
  }
  // d(w l_t)/d(s_t, u_t, u_{t-1}); up: u_{t-1} (the previous input at t = 0, whose gradient the caller discards)
  static CTK_HD void stage_cost_grad(const float* s, const float* u, const float* up, const EnvParams& e, float w, float* lam, float* gu,
                                     float* gu_prev) {
    const float kd = 2.0f * w * e.p[3];
    lam[0] += kd * (s[0] - e.p[8]);
    lam[1] += kd * (s[1] - e.p[9]);
    const float kc = 2.0f * w * e.p[5], kr = 2.0f * w * e.p[6];
    for (int c = 0; c < NU; ++c) {
      const float r = kr * (u[c] - up[c]);
      gu[c] += kc * u[c] + r;
      gu_prev[c] -= r;
    }
  }
  // lam = d(w T)/d(s_H)
  static CTK_HD void terminal_cost_grad(const float* s, const EnvParams& e, float w, float* lam) {
    const float kt = 2.0f * w * e.p[7];
    lam[0] = kt * (s[0] - e.p[8]);
    lam[1] = kt * (s[1] - e.p[9]);
    lam[2] = 0.0f;
  }
};

}  // namespace ctk
