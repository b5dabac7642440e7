// TEST INFRASTRUCTURE ONLY -- K1's step source (ctk_ode_scaled.cuh) at both lane widths, compiled for the CPU.  Rollouts 2m and 2m+1
// run once as two float rolls and once as one f2 roll, the way K1 runs them with one and with two rollouts per thread;
// tests/test_host_twin_lanes.py compares the results bit for bit.  Never loaded by the product.
#include "../../control_toolkit_b200/csrc/ctk_derive.h"
#include "../../control_toolkit_b200/csrc/ctk_ode_scaled.cuh"

using namespace ctk;

template <int KIND, class L>
static void roll(const ScaledStateT<L>& r0, L ul, const L* u, const L* du, int H, const OdeHot& k, ScaledStateT<L>& r, L& acc) {
  r = r0;
  acc = (k.k_ccrc * ul) * ul;
  for (int t = 0; t < H; ++t) {
    acc = stage_cost_scaled<KIND>(acc, r, u[t], ul, du[t], k);
    acc = fmaf(du[t] * du[t], k.k_du2, acc);
    ul = u[t];
    ode_step_scaled(r, u[t], k);
  }
}

extern "C" {

// S_* [N]: total cost of rollout n (N even); st_* [N][7]: its final scaled state (T, W, c, s, x, V, omc)
void twin_lanes(const float* s0, const float* U, const float* dU, int N, int H, const ctk_ode_params* op, const ctk_cost_params* cp,
                float u_prev, float* S_float, float* S_pair, float* st_float, float* st_pair) {
  OdeHot k;
  MppiCorr mc{1.0, 0.4995, 1.0, 0.5, -0.01, 1.0, -1.0, 1.0};
  derive_ode_hot(*op, *cp, H, mc, k);
  ScaledState r0;
  scaled_from_state(s0, k, r0);
  const ScaledStateT<f2> r0p{r0.T, r0.W, r0.c, r0.s, r0.x, r0.V, r0.omc};
  f2 *up = new f2[H], *dup = new f2[H];
  for (int n = 0; n < N; ++n) {
    ScaledState r;
    float acc;
    if (cp->kind == 0) roll<0>(r0, u_prev, U + (size_t)n * H, dU + (size_t)n * H, H, k, r, acc);
    else roll<1>(r0, u_prev, U + (size_t)n * H, dU + (size_t)n * H, H, k, r, acc);
    S_float[n] = finish_cost_scaled(acc, r, U[(size_t)n * H + H - 1], k);
    const float st[7] = {r.T, r.W, r.c, r.s, r.x, r.V, r.omc};
    for (int i = 0; i < 7; ++i) st_float[n * 7 + i] = st[i];
  }
  for (int n = 0; n + 1 < N; n += 2) {
    for (int t = 0; t < H; ++t) {
      up[t] = f2(U[(size_t)n * H + t], U[(size_t)(n + 1) * H + t]);
      dup[t] = f2(dU[(size_t)n * H + t], dU[(size_t)(n + 1) * H + t]);
    }
    ScaledStateT<f2> r;
    f2 acc;
    if (cp->kind == 0) roll<0>(r0p, f2(u_prev), up, dup, H, k, r, acc);
    else roll<1>(r0p, f2(u_prev), up, dup, H, k, r, acc);
    for (int q = 0; q < 2; ++q) {
      const ScaledState rq = lane_of(r, q);
      S_pair[n + q] = finish_cost_scaled(lane_of(acc, q), rq, U[(size_t)(n + q) * H + H - 1], k);
      const float st[7] = {rq.T, rq.W, rq.c, rq.s, rq.x, rq.V, rq.omc};
      for (int i = 0; i < 7; ++i) st_pair[(n + q) * 7 + i] = st[i];
    }
  }
  delete[] up;
  delete[] dup;
}
}
