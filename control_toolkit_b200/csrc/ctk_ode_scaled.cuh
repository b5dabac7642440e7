// ctk_ode_scaled.cuh -- the per-step arithmetic of K1 (ctk_kernels_mppi_ode.cuh) in the scaled state variables of OdeHot:
// T = angle/sqrt(2), W = beta*angleD, V = (cF/g)*positionD.  __host__ __device__ so that the test-only host twin
// (tests/host_twin) runs the SAME source on the CPU against the oracle spec; the product only instantiates it in kernels.
#pragma once
#include "ctk_args.cuh"
#include "ctk_math.cuh"

namespace ctk {

constexpr float kInvSqrt2 = 0.70710678118654752f;
constexpr float kSqrt2 = 1.41421356237309505f;
// period of T = angle/sqrt(2):  2*pi/sqrt(2) = sqrt(2)*pi, split hi + lo
constexpr float kTPerHi = 4.44288301467895508f;      // fp32(sqrt(2)*pi)
constexpr float kTPerLo = -7.6520588976e-08f;         // sqrt(2)*pi - fp32(sqrt(2)*pi)
constexpr float kInvTPer = 0.22507907903927651f;     // 1/(sqrt(2)*pi)

// Lane types of the step: float (one rollout) or f2 (two rollouts of one thread advanced in lock step).  The step below is written
// once over the lane type L.  On the device every f2 +, -, * and fmaf is ONE packed instruction (FADD2 / FMUL2 / FFMA2): per lane it
// computes exactly what the scalar instruction computes (IEEE single, round to nearest; negation and |.| are operand modifiers), so
// each lane's bits are those of the float build, but it takes one issue slot for two rollouts.  That matters because K1 is
// issue-bound, not FP32-rate-bound (DESIGN.md section 5.1).  Operations without a packed form (FRND, MUFU.RCP, FMNMX) run per lane
// inside the f2 helpers.  The explicit _rn intrinsics are never contracted; the float build contracts nothing in this step either
// (every product that feeds a sum is already an explicit fmaf), so both widths perform the same operations in the same order.
// On the host the helpers are two scalar operations: the host twin (tests/host_twin) compiles the same source.
struct f2 {
#if defined(__CUDACC__)
  float2 v;  // 8-byte aligned: an even register pair
#else
  struct { float x, y; } v;
#endif
  f2() = default;
  CTK_HD f2(float a) : v{a, a} {}  // both lanes (constants, values shared by the two rollouts)
  CTK_HD f2(float a, float b) : v{a, b} {}
};
CTK_HD float lane_of(float a, int) { return a; }
CTK_HD float lane_of(f2 a, int q) { return q == 0 ? a.v.x : a.v.y; }

CTK_HD f2 operator-(f2 a) { return f2(-a.v.x, -a.v.y); }
CTK_HD f2 operator+(f2 a, f2 b) {
#if defined(__CUDA_ARCH__)
  f2 r; r.v = __fadd2_rn(a.v, b.v); return r;
#else
  return f2(a.v.x + b.v.x, a.v.y + b.v.y);
#endif
}
CTK_HD f2 operator-(f2 a, f2 b) { return a + (-b); }  // a - b == a + (-b) exactly
CTK_HD f2 operator*(f2 a, f2 b) {
#if defined(__CUDA_ARCH__)
  f2 r; r.v = __fmul2_rn(a.v, b.v); return r;
#else
  return f2(a.v.x * b.v.x, a.v.y * b.v.y);
#endif
}
// (the using-declarations keep the float overloads visible next to the f2 ones inside namespace ctk)
using ::fmaf; using ::fabsf; using ::fmaxf; using ::fminf; using ::rintf;
CTK_HD f2 fmaf(f2 a, f2 b, f2 c) {
#if defined(__CUDA_ARCH__)
  f2 r; r.v = __ffma2_rn(a.v, b.v, c.v); return r;
#else
  return f2(fmaf(a.v.x, b.v.x, c.v.x), fmaf(a.v.y, b.v.y, c.v.y));
#endif
}
CTK_HD f2 fabsf(f2 a) { return f2(fabsf(a.v.x), fabsf(a.v.y)); }
CTK_HD f2 fmaxf(f2 a, f2 b) { return f2(fmaxf(a.v.x, b.v.x), fmaxf(a.v.y, b.v.y)); }
CTK_HD f2 fminf(f2 a, f2 b) { return f2(fminf(a.v.x, b.v.x), fminf(a.v.y, b.v.y)); }
CTK_HD f2 rintf(f2 a) { return f2(rintf(a.v.x), rintf(a.v.y)); }
CTK_HD f2 fast_rcp(f2 a) { return f2(fast_rcp(a.v.x), fast_rcp(a.v.y)); }
// a > b ? v : 0 per lane
CTK_HD float select_gt(float a, float b, float v) { return a > b ? v : 0.0f; }
CTK_HD f2 select_gt(f2 a, f2 b, float v) { return f2(select_gt(a.v.x, b.v.x, v), select_gt(a.v.y, b.v.y, v)); }

template <class L>
struct ScaledStateT {
  L T, W, c, s, x, V, omc;  // omc = 1 - cos(angle)
};
using ScaledState = ScaledStateT<float>;
CTK_HD const ScaledState& lane_of(const ScaledState& r, int) { return r; }
CTK_HD ScaledState lane_of(const ScaledStateT<f2>& r, int q) {
  return {lane_of(r.T, q), lane_of(r.W, q), lane_of(r.c, q), lane_of(r.s, q), lane_of(r.x, q), lane_of(r.V, q), lane_of(r.omc, q)};
}

CTK_HD void scaled_from_state(const float* s0, const OdeHot& k, ScaledState& r) {
  r.T = s0[0] * kInvSqrt2; r.W = s0[1] * k.beta; r.c = s0[2]; r.s = s0[3]; r.x = s0[4]; r.V = s0[5] * k.cFg;
  r.omc = 1.0f - cosf(s0[0]);  // spec: E_pot uses cos(angle) of the measured state
}
CTK_HD void scaled_to_state(const ScaledState& r, const OdeHot& k, float* out) {
  out[0] = r.T * kSqrt2; out[1] = r.W * k.inv_beta; out[2] = r.c; out[3] = r.s; out[4] = r.x; out[5] = r.V * k.inv_cFg;
}

// stage cost / (H+1) of (state, u, u_prev, du) in the merged form of K1:
//   dd + barrier + E_pot (+ E_kin, border for quadratic_boundary_grad) + u (kA u + kB u_prev + kC du)
// (the u_prev^2 terms of the control-change cost are telescoped into kA; boundary terms are added by the caller)
template <int KIND, class L>
CTK_HD L stage_cost_scaled(L acc, const ScaledStateT<L>& r, L u, L ul, L du, const OdeHot& k) {
  const L d = r.x - k.target;
  const L e = fmaxf(fabsf(r.x) - k.thl_095, 0.0f);  // indicator(|x| > 0.95 THL) * (|x| - 0.95 THL)
  acc = fmaf(d * d, k.k_dd, acc);
  acc = fmaf(e * e, k.k_bar, acc);
  acc = fmaf(r.omc * r.omc, k.k_ep, acc);
  if (KIND == 1) {
    acc = fmaf(r.W * r.W, k.k_ekp2, acc);
    acc = acc + select_gt(fabsf(r.x), k.thl_09, k.k_border);
  }
  L q = u * k.kA;
  q = fmaf(ul, k.kB, q);
  q = fmaf(du, k.kC, q);
  return fmaf(u, q, acc);
}

// One Euler step with the old derivatives (12 FP32 instructions + 1 MUFU), wrap (3), half-angle sincos (14).
template <class L>
CTK_HD void ode_step_scaled(ScaledStateT<L>& r, L u, const OdeHot& k) {
  L nn = fmaf(k.cUg, u, r.V);
  const L ws = r.W * r.s;
  nn = fmaf(-r.W, ws, nn);
  const L t3 = fmaf(k.cTl2, r.W, r.s);
  nn = fmaf(t3, r.c, nn);
  const L Ap = fmaf(-r.c, r.c, k.K1p);
  const L vd = nn * fast_rcp(Ap);
  const L X = fmaf(vd, r.c, fmaf(k.kTm2, r.W, r.s));
  L T = fmaf(r.W, k.h_T, r.T);
  r.W = fmaf(X, k.h_W, r.W);
  r.x = fmaf(r.V, k.h_x, r.x);
  r.V = fmaf(vd, k.h_V, r.V);
  // wrap: angle <- atan2(sin, cos)  ==  T - period * rint(T / period)
  const L kk = rintf(T * kInvTPer);
  T = fmaf(-kk, kTPerHi, T);
  T = fmaf(-kk, kTPerLo, T);
  r.T = T;
  // half-angle sincos (ctk_math.cuh sincos_half with x = T)
  const L tt = T * T;
  L ps = fmaf(tt, kSinHalfLead, -2.4761327949818224e-05f);
  ps = fmaf(tt, ps, 0.002083262661471963f);
  ps = fmaf(tt, ps, -0.08333329111337662f);
  const L sh = fmaf(T * tt, ps, T);
  L pc = fmaf(tt, kCosHalfLead, 2.1885084606765304e-06f);
  pc = fmaf(tt, pc, -0.0002455138601362705f);
  pc = fmaf(tt, pc, 0.01473138015717268f);
  pc = fmaf(tt, pc, -0.3535533845424652f);
  const L ch = fmaf(tt, pc, 1.4142135381698608f);
  r.omc = sh * sh;
  r.c = fmaf(-sh, sh, 1.0f);
  r.s = sh * ch;
}

// terminal cost / (H+1) and the per-rollout boundary terms of the telescoped control-change cost
CTK_HD float finish_cost_scaled(float acc, const ScaledState& r, float u_last, const OdeHot& k) {
  const float th = r.T * kSqrt2;
  const float term = (fabsf(th) > 0.2f || fabsf(r.x - k.target) > k.thl_01) ? k.k_term : 0.0f;
  return (fmaf(-k.k_ccrc * u_last, u_last, acc) + term) - k.shift;
}

}  // namespace ctk
