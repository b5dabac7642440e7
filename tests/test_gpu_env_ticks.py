"""GPU tests of the Dubins-car MPPI and CEM ticks (ctk_kernels_env.cuh: env_mppi_rollout_kernel, env_mppi_update_kernel,
env_cem_rollout_kernel, env_cem_refit_kernel) against float64 and the oracle.

The limits differ per input and no two share a bound or a midpoint (throttle [-0.5, 1], steer [-1, 0.6]), so that a kernel which
mixes up the inputs, or uses input 0's limits for both, fails.  Three kinds of checks:
  * per step, from the logs: every logged transition (s_t, u_t) -> s_{t+1} against float64 dubins_step applied to the device's own
    s_t and u_t; every rollout's cost recomputed in float64 from the device's own states and controls (plus the MPPI correction);
    every logged control recomputed from the draws.  The obstacle term is an indicator: a rollout with a state within a few ulp of
    the circle is exempt from the cost check (counted and bounded).  Yaw is compared as a wrapped angle difference.
  * per tick, against the fp32 and float64 oracles on the same draws (injected, or the in-kernel Philox draws exported with
    ctk_philox_export), the oracles re-synchronised to the device's state before each tick:
    |cuda - fp32 oracle| <= max(2e-5, 8 floor) and |cuda - float64| <= max(1e-5, 4 floor), floor = |fp32 oracle - float64| on that
    tick.  Per-rollout costs as test_gpu_parity._check_J, after setting aside whole obstacle-term flips (counted and bounded).  CEM elite sets identical, except for members that tie with the k-th cost within a few ulp.
  * closed loops and state handling: a free-running device against free-running oracles, reset mid-episode, a frozen previous
    input, get_state / set_state round trips, a degenerate input (low == high).
The per-step bounds and the measured maxima are in DESIGN 8f.3.  Every measured error is appended to the parity report
(test_gpu_parity._report)."""
import numpy as np
import pytest

from helpers import load_golden, make_oracle
from oracle.replay_rng import QueueRNG, ReplayRNG
from test_gpu_parity import _report
from test_gpu_production_pinning import _J_floor, _state_errs

pytestmark = pytest.mark.gpu

LOW, HIGH = np.array([-0.5, -1.0], np.float32), np.array([1.0, 0.6], np.float32)
EPS32 = float(np.finfo(np.float32).eps)
NEAR_ULPS = 8  # a state whose squared distance to the obstacle centre is this many ulp from r^2 may round to either side

# per-step bounds (DESIGN 8f.3): x and y relative to the largest |x|, |y| of the tick; yaw absolute
# (wrapped); J element-wise relative to |J| + 1e-3; the logged MPPI controls absolute (the draws are interpolated in another order)
TOL_XY = 2e-7
TOL_YAW = 2e-6
TOL_J = 1.5e-6
TOL_Q_MPPI = 5e-7


# ---- set-up --------------------------------------------------------------------------------------------------------------
def _meta(optimizer, **over):
    _, meta = load_golden("mppi_dubins_n512" if optimizer == "mppi" else "cem_dubins_n512_k32")
    return dict(meta, cfg=dict(meta["cfg"], **over))


def _controller(meta, logging=False, rng=None, low=LOW, high=HIGH, weights=None, **opt_over):
    """The controller_mpc of the Dubins car with per-input limits; ``weights`` go through config_cost_function (the override path of
    Optimizers/__init__.py: cost_function.weights -> specs.resolve_cost -> dubins_env_params)."""
    from control_toolkit_b200.Controllers.controller_mpc import controller_mpc
    cost_cfg = {"cost_function_name_default": "default"}
    if weights:
        cost_cfg["DubinsCar"] = {"default": dict(weights)}
    ctrl = controller_mpc(
        environment_name="DubinsCar", control_limits=(low, high), initial_environment_attributes={},
        config_controller=dict(optimizer=meta["optimizer"], predictor_specification="ODE", cost_function_specification="default",
                               controller_logging=logging),
        config_optimizers={meta["optimizer"]: dict(meta["cfg"], **opt_over)}, config_cost_function=cost_cfg)
    ctrl.configure(optimizer_name=meta["optimizer"], predictor_specification="ODE")
    if rng is not None:
        ctrl.optimizer.rng = rng
        ctrl.optimizer.optimizer_reset()
    return ctrl


class _Recorder(ReplayRNG):
    """Injected noise that keeps the blocks it hands out, so the oracles can replay exactly the draws of the tick."""

    def __init__(self, seed):
        super().__init__(seed, as_torch=False)
        self.drawn = []

    def standard_draws(self, kind, shape):
        z = super().standard_draws(kind, shape)
        self.drawn.append(z)
        return z

    def take(self):
        out, self.drawn = self.drawn, []
        return out


def _oracles(meta, low=LOW, high=HIGH, cost=None, params=None, **over):
    import torch
    from oracle import spec
    out = []
    for dtype in (torch.float32, torch.float64):
        o = make_oracle(meta, action_low=low, action_high=high, dtype=dtype, **over)
        if params is not None:
            o.predictor = spec.DubinsPredictor(params)
        if cost is not None:
            o.cost = cost
        out.append(o)
    return out


def _states(n, seed):
    from oracle import spec
    return spec.dubins_synthetic_states(n, seed=seed)


def _device_state(opt):
    """The optimizer state the next tick starts from, as the device holds it."""
    from control_toolkit_b200 import _lib as L
    H = opt.mpc_horizon
    st = {"u_prev": opt._get_state(L.STATE_U_PREV, (2,))}
    if opt.optimizer_name == "mppi":
        st["u_nom"] = opt._get_state(L.STATE_U_NOM, (1, H, 2))
    else:
        st["mu"], st["sd"] = opt._get_state(L.STATE_CEM_MU, (1, H, 2)), opt._get_state(L.STATE_CEM_STD, (1, H, 2))
    return st


def _sync(oracles, st, count=None):
    """Re-synchronise the oracles to the device's state: each tick then measures one tick's parity, not the closed loop's drift."""
    import torch
    for o in oracles:
        o.u = np.array(st["u_prev"], np.float32)
        if "u_nom" in st:
            o.u_nom = torch.from_numpy(np.array(st["u_nom"])).to(o.dtype)
        else:
            o.dist_mue, o.stdev = torch.from_numpy(np.array(st["mu"])).to(o.dtype), torch.from_numpy(np.array(st["sd"])).to(o.dtype)
            if count is not None:
                o.count = count


def _mppi_blocks(opt, rec):
    from control_toolkit_b200 import _lib as L
    if rec is not None:
        return rec.take()
    return [opt.export_philox(L.STREAM_MPPI, opt.tick_counter, opt.number_of_interpolation_inducing_points * 2, opt.num_rollouts)]


def _cem_blocks(opt, rec, iters):
    from control_toolkit_b200 import _lib as L
    if rec is not None:
        return rec.take()
    return [opt.export_philox(L.STREAM_CEM, opt.tick_counter, opt.mpc_horizon * 2, opt.num_rollouts, sub=it) for it in range(iters)]


# ---- per-tick parity against the oracles ------------------------------------------------------------------------------------
def _check_J_obstacle(tag, J, J32, J64, H, obstacle_weight):
    """Per-rollout costs against the fp32 oracle (test_gpu_parity._check_J's criterion) after setting aside the rollouts whose two
    costs differ by a whole number of obstacle terms obstacle_weight / (H + 1): a state within rounding of the circle, counted."""
    J, J32 = np.asarray(J, np.float64), np.asarray(J32, np.float64)
    e = np.abs(J - J32) / (np.abs(J32) + 1e-3)
    step = float(np.float32(obstacle_weight)) / (H + 1)
    m = np.rint((J - J32) / step)
    flip = (m != 0) & (np.abs(J - J32 - m * step) <= 1e-4 * (np.abs(J32) + step))
    keep = ~flip
    fl = _J_floor(np.asarray(J32)[keep], np.asarray(J64)[keep]) if keep.any() else {"J": 0.0, "J_q99": 0.0}
    mx = float(e[keep].max()) if keep.any() else 0.0
    q99 = float(np.quantile(e[keep], 0.99)) if keep.sum() >= 1000 else mx
    _report(f"{tag}: J q99 {q99:.2e} max {mx:.2e} (fp32 floor q99 {fl['J_q99']:.2e} max {fl['J']:.2e}); obstacle-term flips {int(flip.sum())} of {J.size}")
    assert int(flip.sum()) <= max(3, J.size // 1000), (tag, int(flip.sum()))
    if keep.sum() >= 1000:
        assert q99 < 1e-4 + 3 * fl["J_q99"], (tag, q99, fl)
        assert mx < 1e-3 + 10 * fl["J"], (tag, mx, fl)
    else:
        assert mx < 1e-2 + 10 * fl["J"], (tag, mx, fl)


def _assert_parity(tag, e32, e64, floor):
    """|cuda - fp32 oracle| bounded, |cuda - float64| <= max(1e-5, 4 x |fp32 oracle - float64|) on this tick."""
    _report(f"{tag}: |cuda-ref32| {e32:.2e} |cuda-f64| {e64:.2e} | floor |ref32-f64| {floor:.2e}")
    assert e32 <= max(2e-5, 8.0 * floor), (tag, e32, floor)
    assert e64 <= max(1e-5, 4.0 * floor), (tag, "distance to the float64 truth", e64, floor)


def _mppi_oracle_tick(tag, opt, oracles, s, blocks, u, chunked=False):
    from control_toolkit_b200 import _lib as L
    o32, o64 = oracles
    run = (lambda o: o.step_chunked(s, QueueRNG(list(blocks)), chunk=16384)) if chunked else (lambda o: o.step(s, QueueRNG(list(blocks))))
    u32 = run(o32)
    run(o64)
    e32, e64, floor = _state_errs(opt.u_nom, o32.u_nom.numpy(), o64.u_nom.numpy())
    _assert_parity(f"{tag} u_nom", e32, e64, floor)
    scale = max(float(np.max(np.abs(o64.u_nom.numpy()))), 1e-2)
    eu = float(np.max(np.abs(np.ravel(u) - np.ravel(u32)))) / scale
    assert np.shape(u) == (2,) and eu <= max(2e-5, 8 * floor), (tag, "u", eu, floor)
    J = opt._get_log(L.LOG_J, (opt.num_rollouts,))
    _check_J_obstacle(tag, J, o32.last["J"], o64.last["J"], opt.mpc_horizon, o32.cost.obstacle_weight)
    return floor


def _cem_oracle_tick(tag, opt, oracles, s, blocks, u, iters):
    """True when the elite sets of every outer iteration equal the oracle's (then the distribution is compared), False after an
    admissible ulp-level tie at the k-th cost (test_gpu_parity.test_cem_edge_geometries_match_oracle)."""
    o32, o64 = oracles
    k, N = opt.cem_best_k, opt.num_rollouts
    u32 = o32.step(s, QueueRNG(list(blocks)))
    o64.step(s, QueueRNG(list(blocks)))
    got, ref = opt.last_elite_indices(iters), np.asarray(o32.last["elite_idx"])
    J = opt.last_costs()
    # the index work is bit-exact on the device's own costs: ties broken by index (tf.argsort semantics)
    np.testing.assert_array_equal(got[-1], np.argsort(J, kind="stable")[:k])
    differ = [it for it in range(iters) if set(got[it].tolist()) != set(ref[it].tolist())]
    if differ:
        it = differ[0]
        Jo = np.asarray(o32.last["J_iters"][it], np.float32)
        Jk = float(Jo[np.argsort(Jo, kind="stable")[k - 1]])
        ulp = float(np.spacing(np.float32(abs(Jk))))
        diff = sorted(set(got[it].tolist()) ^ set(ref[it].tolist()))
        _report(f"{tag}: elite sets differ in iteration {it} at {diff} (J_k {Jk:.6e}, ulp {ulp:.2e})")
        for i in diff:
            assert abs(float(Jo[i]) - Jk) <= 4 * ulp, (tag, it, i, float(Jo[i]), Jk, ulp)
        return False
    floors = []
    for nm, a, b32, b64 in (("mu", opt.dist_mue, o32.dist_mue, o64.dist_mue), ("sd", opt.stdev, o32.stdev, o64.stdev)):
        e32, e64, floor = _state_errs(a, b32.numpy(), b64.numpy())
        _assert_parity(f"{tag} {nm}", e32, e64, floor)
        floors.append(floor)
    eu = float(np.max(np.abs(np.ravel(u) - np.ravel(u32))))
    assert np.shape(u) == (2,) and eu <= max(2e-5, 8 * max(floors)), (tag, "u", eu, floors)
    _check_J_obstacle(tag, J, o32.last["J"], o64.last["J"], opt.mpc_horizon, o32.cost.obstacle_weight)
    return True


# ---- per-step checks of the logs against float64 ---------------------------------------------------------------------------
def _check_logged_steps(tag, opt, s0, st, low, high, cost, params, blocks=None):
    """Every logged transition and every rollout's cost against float64 from the device's own logged states and controls; with
    ``blocks`` (the draws of the tick) also every logged control.  Returns the share of rollouts that enter the obstacle."""
    import torch
    from oracle import spec
    from oracle.mppi import interpolation_matrix
    lv = opt.logging_values
    Q32, tr32 = np.asarray(lv["Q_logged"], np.float32), np.asarray(lv["rollout_trajectories_logged"], np.float32)
    J = np.asarray(lv["J_logged"], np.float64)
    N, H = Q32.shape[:2]
    Q, tr = Q32.astype(np.float64), tr32.astype(np.float64)
    assert Q.shape == (N, H, 2) and tr.shape == (N, H + 1, 3) and J.shape == (N,)
    assert np.array_equal(tr32[:, 0], np.broadcast_to(np.asarray(s0, np.float32), (N, 3))), tag
    for c in range(2):  # every control inside its own input's limits
        assert Q32[..., c].min() >= low[c] and Q32[..., c].max() <= high[c], (tag, c, Q32[..., c].min(), Q32[..., c].max())
    # transitions
    nxt = spec.dubins_step(torch.from_numpy(tr[:, :-1].reshape(-1, 3)), torch.from_numpy(Q.reshape(-1, 2)), params.f32()).numpy().reshape(N, H, 3)
    scale = max(float(np.max(np.abs(nxt[..., :2]))), 1e-2)
    e_xy = float(np.max(np.abs(tr[:, 1:, :2] - nxt[..., :2]))) / scale
    e_yaw = float(np.max(np.abs(np.remainder(tr[:, 1:, 2] - nxt[..., 2] + np.pi, 2 * np.pi) - np.pi)))
    assert np.all(np.abs(tr[:, 1:, 2]) <= np.float32(np.pi)), tag  # wrapped
    # costs, from the device's own states and controls
    u_prev = np.asarray(st["u_prev"], np.float64)
    J64 = spec.trajectory_cost(torch.from_numpy(tr), torch.from_numpy(Q), torch.from_numpy(u_prev), cost).numpy()
    mppi = opt.optimizer_name == "mppi"
    e_Q = 0.0
    if mppi:
        z = np.asarray(blocks[0], np.float32).reshape(N, -1, 2)
        W = interpolation_matrix(H, opt.period_interpolation_inducing_points).astype(np.float64)  # [n_ind, H]
        du = np.einsum("nic,ih->nhc", (z * np.float32(opt.SQRTRHODTINV)).astype(np.float64), W)
        cw, R, NU = float(np.float32(opt.cc_weight)), float(np.float32(opt.R)), float(np.float32(opt.NU))
        J64 = J64 + np.sum(cw * (0.5 * (1 - 1 / NU) * R * du ** 2 + R * Q * du + 0.5 * R * Q ** 2), (1, 2))
        un = np.asarray(st["u_nom"], np.float64)[0]
        shifted = np.concatenate([un[1:], un[-1:]], 0)
        Qx = np.clip(shifted[None] + du, low.astype(np.float64), high.astype(np.float64))
        e_Q = float(np.max(np.abs(Q - Qx)))
    else:  # CEM, one outer iteration: Q = clip(mu + z sd) in fp32, bit for bit
        assert len(blocks) == 1, "the logged controls are those of the last outer iteration: run one"
        z = np.asarray(blocks[-1], np.float32).reshape(N, H, 2)
        mu, sd = np.asarray(st["mu"], np.float32), np.asarray(st["sd"], np.float32)
        Qx = np.minimum(np.maximum(mu + z * sd, low), high)
        e_Q = float(np.max(np.abs(Q32 - Qx)))
        assert np.array_equal(Q32, Qx), (tag, "logged controls", e_Q)
    cf = cost.f32()
    d = (tr[:, :H, 0] - cf["obstacle_x"]) ** 2 + (tr[:, :H, 1] - cf["obstacle_y"]) ** 2
    near = np.any(np.abs(d - cf["obstacle_r2"]) <= NEAR_ULPS * EPS32 * cf["obstacle_r2"], 1)
    inside = float(np.mean(np.any(d < cf["obstacle_r2"], 1)))
    eJ = np.abs(J - J64) / (np.abs(J64) + 1e-3)
    e_J = float(eJ[~near].max()) if (~near).any() else 0.0
    _report(f"env_ticks per-step {tag}: xy {e_xy:.2e} yaw {e_yaw:.2e} J {e_J:.2e} Q {e_Q:.2e} | near-circle rollouts {int(near.sum())} "
            f"of {N}, rollouts entering the obstacle {inside:.1%}")
    assert e_xy <= TOL_XY and e_yaw <= TOL_YAW, (tag, e_xy, e_yaw)
    assert e_J <= TOL_J, (tag, "J", e_J, int(np.argmax(np.where(near, 0, eJ))))
    assert e_Q <= TOL_Q_MPPI, (tag, "logged controls", e_Q)
    assert int(near.sum()) <= max(2, N // 100), (tag, "near-circle rollouts", int(near.sum()))
    return inside


def _logged_ticks(tag, meta, states, ticks_oracle=True, low=LOW, high=HIGH, weights=None, cost=None, params=None, seed=7):
    """Logging on, injected noise: per tick the per-step check and (``ticks_oracle``) the oracle tick.  Returns the obstacle shares."""
    from oracle import spec
    cost = cost or spec.DubinsCost()
    params = params or spec.DubinsParams(dt=meta["cfg"]["mpc_timestep"])
    rec = _Recorder(seed)
    ctrl = _controller(meta, logging=True, rng=rec, low=low, high=high, weights=weights)
    opt = ctrl.optimizer
    oracles = _oracles(meta, low, high, cost=cost, params=params)
    mppi = meta["optimizer"] == "mppi"
    shares = []
    for t, s in enumerate(states):
        st = _device_state(opt)
        count = None if mppi else opt.count
        u = ctrl.step(s)
        assert opt.last_kernel == ("env_mppi_rollout_kernel" if mppi else "env_cem_rollout_kernel") + "<DubinsEnv,1> [injected noise]", opt.last_kernel
        blocks = rec.take()
        shares.append(_check_logged_steps(f"{tag} tick {t}", opt, s, st, low, high, cost, params, blocks))
        if ticks_oracle:
            _sync(oracles, st, count)
            if mppi:
                _mppi_oracle_tick(f"env_ticks oracle {tag} tick {t}", opt, oracles, s, blocks, u)
            else:
                _cem_oracle_tick(f"env_ticks oracle {tag} tick {t}", opt, oracles, s, blocks, u, meta["cfg"]["cem_outer_it"])
    return shares


# ---- 1. per-step checks of the logs ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("optimizer,over", [("mppi", dict(num_rollouts=1000)), ("cem-tf", dict(num_rollouts=1000, cem_outer_it=1, cem_best_k=50))],
                         ids=["mppi", "cem"])
def test_logged_transitions_costs_and_controls_match_float64(optimizer, over):
    _logged_ticks(optimizer, _meta(optimizer, **over), _states(3, seed=61))


# ---- 2. MPPI edge geometries ------------------------------------------------------------------------------------------------
MPPI_EDGES = [(1, 1, 10), (1, 7, 3), (33, 2, 10), (129, 11, 50), (257, 101, 10), (1000, 30, 7), (64, 21, 10), (200, 16, 1), (64, 512, 35)]


@pytest.mark.parametrize("N,H,period", MPPI_EDGES)
def test_mppi_edge_geometries_match_oracle(N, H, period):
    """A single rollout, one step, a period longer than the horizon, N not a multiple of the 128-thread block, H - 1 a multiple of the
    period (the last inducing point), n_ind * nu = 32 (every register of the update kernel's accumulator) and H * nu = 1024."""
    meta = _meta("mppi", num_rollouts=N, mpc_horizon=H, period_interpolation_inducing_points=period)
    rec = _Recorder(5)
    ctrl = _controller(meta, rng=rec)
    opt = ctrl.optimizer
    n_ind = opt.number_of_interpolation_inducing_points
    assert n_ind * 2 <= 32 and H * 2 <= 1024
    oracles = _oracles(meta)
    for t, s in enumerate(_states(3, seed=21)):
        st = _device_state(opt)
        _sync(oracles, st)
        u = ctrl.step(s)
        assert opt.last_kernel == "env_mppi_rollout_kernel<DubinsEnv,0> [injected noise]", opt.last_kernel
        assert opt.u_nom.shape == (1, H, 2)
        _mppi_oracle_tick(f"env_ticks mppi edge N={N} H={H} p={period} n_ind*nu={n_ind * 2} tick {t}", opt, oracles, s, rec.take(), u)


# ---- 3. CEM edge geometries -------------------------------------------------------------------------------------------------
CEM_EDGES = [(1, 5, 1, 2), (33, 1, 4, 3), (130, 7, 130, 1), (1025, 20, 64, 2), (5000, 12, 512, 2), (257, 50, 1, 4), (64, 512, 8, 2)]


def _cem_run(tag, meta, states, rec=None, iters_first=None, **ctrl_over):
    ctrl = _controller(meta, rng=rec, **ctrl_over)
    opt = ctrl.optimizer
    oracles = _oracles(meta)
    same_ticks = 0
    for t, s in enumerate(states):
        st = _device_state(opt)
        _sync(oracles, st, opt.count)
        iters = iters_first if (iters_first is not None and t == 0) else meta["cfg"]["cem_outer_it"]
        u = ctrl.step(s)
        assert opt.last_kernel == "env_cem_rollout_kernel<DubinsEnv,0> " + ("[injected noise]" if rec is not None else "[philox]"), opt.last_kernel
        same_ticks += _cem_oracle_tick(f"{tag} tick {t}", opt, oracles, s, _cem_blocks(opt, rec, iters), u, iters)
    return same_ticks


@pytest.mark.parametrize("N,H,k,iters", CEM_EDGES)
def test_cem_edge_geometries_match_oracle(N, H, k, iters):
    """One rollout, one step, k == N, k == 1, the 512-elite maximum, N > 1024 (several top-k levels before the refit's sort), and
    H * nu = 1024 (one refit thread per column, every thread of the block)."""
    meta = _meta("cem-tf", num_rollouts=N, mpc_horizon=H, cem_best_k=k, cem_outer_it=iters)
    same = _cem_run(f"env_ticks cem edge N={N} H={H} k={k} it={iters}", meta, _states(3, seed=22), rec=_Recorder(6))
    assert same >= 1


def test_cem_warmup_tick_matches_oracle():
    meta = _meta("cem-tf", num_rollouts=300, mpc_horizon=20, cem_best_k=16, cem_outer_it=2, warmup=True, warmup_iterations=6)
    same = _cem_run("env_ticks cem warm-up", meta, _states(3, seed=23), rec=_Recorder(8), iters_first=6)
    assert same >= 1


# ---- 4. the production path: in-kernel Philox -------------------------------------------------------------------------------
@pytest.mark.parametrize("N,H,period", [(65536, 40, 10), (30011, 23, 5)])
def test_mppi_philox_matches_oracle(N, H, period):
    meta = _meta("mppi", num_rollouts=N, mpc_horizon=H, period_interpolation_inducing_points=period)
    ctrl = _controller(meta)
    opt = ctrl.optimizer
    assert opt.rng is None
    oracles = _oracles(meta)
    for t, s in enumerate(_states(3, seed=24)):
        st = _device_state(opt)
        _sync(oracles, st)
        u = ctrl.step(s)
        assert opt.last_kernel == "env_mppi_rollout_kernel<DubinsEnv,0> [philox]", opt.last_kernel
        _mppi_oracle_tick(f"env_ticks mppi philox N={N} H={H} p={period} tick {t}", opt, oracles, s, _mppi_blocks(opt, None), u, chunked=True)


@pytest.mark.parametrize("N,H,k,iters", [(16384, 40, 64, 3), (9001, 37, 100, 2)])
def test_cem_philox_matches_oracle(N, H, k, iters):
    meta = _meta("cem-tf", num_rollouts=N, mpc_horizon=H, cem_best_k=k, cem_outer_it=iters)
    assert _cem_run(f"env_ticks cem philox N={N} H={H} k={k} it={iters}", meta, _states(3, seed=25)) >= 2


# ---- 5. closed loops and state handling ------------------------------------------------------------------------------------
@pytest.mark.parametrize("optimizer,over", [("mppi", dict(num_rollouts=2000)), ("cem-tf", dict(num_rollouts=2000, cem_best_k=40))], ids=["mppi", "cem"])
def test_closed_loop_free_running_with_reset(optimizer, over):
    """20 ticks.  The device runs free; one oracle pair is re-synchronised to it before every tick (one tick's parity), a second pair
    runs free as well (the closed loop's drift, bounded by the float64 distance scaled by that pair's own fp32 floor).  The
    controller is reset before tick 12: MPPI keeps its previous input, CEM zeroes it (optimizer_mppi.py:227-231, optimizer_cem_tf.py:113-117)."""
    meta = _meta(optimizer, **over)
    rec = _Recorder(9)
    ctrl = _controller(meta, rng=rec)
    opt = ctrl.optimizer
    synced, free = _oracles(meta), _oracles(meta)
    mppi = optimizer == "mppi"
    iters = meta["cfg"].get("cem_outer_it", 1)
    for t, s in enumerate(_states(20, seed=26)):
        if t == 12:
            ctrl.controller_reset()
            for o in free:
                o.reset()
            st = _device_state(opt)
            assert np.array_equal(np.asarray(st["u_nom" if mppi else "mu"])[0], np.broadcast_to((LOW + HIGH) / 2, (opt.mpc_horizon, 2)))
            if not mppi:
                assert np.array_equal(st["u_prev"], np.zeros(2, np.float32))
        st = _device_state(opt)
        _sync(synced, st, None if mppi else opt.count)
        u = ctrl.step(s)
        blocks = rec.take()
        tag = f"env_ticks closed loop {optimizer} tick {t}"
        if mppi:
            _mppi_oracle_tick(tag, opt, synced, s, blocks, u)
        elif not _cem_oracle_tick(tag, opt, synced, s, blocks, u, iters):
            break  # an ulp-level elite tie: the free-running oracles legitimately part from here on
        f32, f64 = free
        f32.step(s, QueueRNG(list(blocks)))
        f64.step(s, QueueRNG(list(blocks)))
        a, b32, b64 = (opt.u_nom, f32.u_nom.numpy(), f64.u_nom.numpy()) if mppi else (opt.dist_mue, f32.dist_mue.numpy(), f64.dist_mue.numpy())
        e32, e64, floor = _state_errs(a, b32, b64)
        _report(f"{tag}: free-running |cuda-ref32| {e32:.2e} |cuda-f64| {e64:.2e} floor {floor:.2e}")
        assert e32 < 1e-4 and e64 <= max(1e-5, 4 * floor), (tag, e32, e64, floor)
    assert t >= 12


@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
def test_freeze_previous_input(optimizer):
    """freeze_previous_input: the cost's previous input stays at its reset value 0 on every tick (oracle with u = 0 before each tick)."""
    meta = _meta(optimizer, num_rollouts=512)
    rec = _Recorder(10)
    ctrl = _controller(meta, rng=rec, freeze_previous_input=True)
    opt = ctrl.optimizer
    oracles = _oracles(meta)
    moved = False
    for t, s in enumerate(_states(4, seed=27)):
        st = _device_state(opt)
        assert np.array_equal(st["u_prev"], np.zeros(2, np.float32)), (t, st["u_prev"])
        _sync(oracles, st, None if optimizer == "mppi" else opt.count)
        u = ctrl.step(s)
        moved |= bool(np.any(np.asarray(u) != 0))
        tag = f"env_ticks frozen previous input {optimizer} tick {t}"
        if optimizer == "mppi":
            _mppi_oracle_tick(tag, opt, oracles, s, rec.take(), u)
        else:
            _cem_oracle_tick(tag, opt, oracles, s, rec.take(), u, meta["cfg"]["cem_outer_it"])
    assert moved and np.array_equal(_device_state(opt)["u_prev"], np.zeros(2, np.float32))


@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
def test_state_round_trip_continues_bit_identical(optimizer):
    """get_state of one handle into set_state of another (u_nom, or mu and sd, of shape [1, H, 2] and u of shape (2,)): with the
    same Philox tick counter both continue bit for bit."""
    from control_toolkit_b200 import _lib as L
    meta = _meta(optimizer, num_rollouts=300)
    a, b = _controller(meta), _controller(meta)
    states = _states(6, seed=28)
    for s in states[:3]:
        a.step(s)
    st = a.optimizer.get_state()
    H = meta["cfg"]["mpc_horizon"]
    for key in ("u_nom",) if optimizer == "mppi" else ("dist_mue", "stdev"):
        assert st[key].shape == (1, H, 2), (key, st[key].shape)
    assert np.shape(st["u"]) == (2,) and np.array_equal(st["u"], np.ravel(a.optimizer.u))
    b.optimizer.set_state(st)
    b.optimizer._set_counter(L.COUNTER_TICK, a.optimizer._get_counter(L.COUNTER_TICK))
    st_b = b.optimizer.get_state()
    for key in st:
        assert np.array_equal(np.asarray(st[key]), np.asarray(st_b[key])), key
    for s in states[3:]:
        np.testing.assert_array_equal(a.step(s), b.step(s))
        for key, v in a.optimizer.get_state().items():
            assert np.array_equal(np.asarray(v), np.asarray(b.optimizer.get_state()[key])), key


@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
def test_degenerate_input_stays_constant(optimizer):
    """Steer limits low == high == 0.3: the steer is 0.3 in every logged control, in u and in the optimizer state; the throttle is
    still optimised, and the tick matches the oracle."""
    low, high = np.array([-0.5, 0.3], np.float32), np.array([1.0, 0.3], np.float32)
    meta = _meta(optimizer, num_rollouts=500, **({} if optimizer == "mppi" else dict(cem_outer_it=1, cem_best_k=25)))
    shares = _logged_ticks(f"degenerate steer {optimizer}", meta, _states(3, seed=29), low=low, high=high, seed=11)
    assert len(shares) == 3
    ctrl = _controller(meta, logging=True, rng=_Recorder(11), low=low, high=high)
    opt = ctrl.optimizer
    for s in _states(3, seed=29):
        u = ctrl.step(s)
        Q = opt.logging_values["Q_logged"]
        assert np.all(Q[..., 1] == np.float32(0.3)) and np.ravel(u)[1] == np.float32(0.3)
        assert np.ptp(Q[..., 0]) > 0.5  # the throttle is sampled
        state = opt.u_nom if optimizer == "mppi" else opt.dist_mue
        if optimizer == "mppi":  # u_nom is clipped to [0.3, 0.3]
            assert np.all(state[0, :, 1] == np.float32(0.3))
        else:  # the mean is not clipped: an fp32 mean of k copies of 0.3 is 0.3 to a few ulp; the reset tail is exact
            assert np.max(np.abs(state[0, :, 1].astype(np.float64) - np.float64(np.float32(0.3)))) <= 1e-6
            assert state[0, -1, 1] == np.float32(0.3)
        assert np.ptp(state[0, :, 0]) > 0  # and optimised: it leaves the uniform mid-range start


# ---- 6. non-default environment parameters ---------------------------------------------------------------------------------
# every overridable field of the cost distinct (MAX_COST is not overridable: specs.resolve_cost), the obstacle across the start region
WEIGHTS = dict(dd_weight=3.5, obstacle_weight=250.0, cc_weight=0.7, ccrc_weight=2.5, R=0.3, terminal_weight=40.0, target_x=-0.6,
               target_y=0.45, obstacle_x=0.12, obstacle_y=-0.05, obstacle_r=0.17)
OBSTACLE_STATES = np.array([[-0.3, 0.0, 0.3], [0.12, -0.4, 1.5], [0.45, -0.1, 3.0]], np.float32)  # outside the circle, facing it


@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
def test_non_default_cost_and_ode_parameters(optimizer):
    from control_toolkit_b200 import specs
    from oracle import spec
    meta = _meta(optimizer, num_rollouts=1000, **({} if optimizer == "mppi" else dict(cem_outer_it=1, cem_best_k=50)))
    saved = specs.ODE_REGISTRY["DubinsCar"]
    try:
        specs.ODE_REGISTRY["DubinsCar"] = specs.DubinsCarODE(v_max=1.7, omega_max=1.3)
        shares = _logged_ticks(f"non-default parameters {optimizer}", meta, OBSTACLE_STATES, weights=WEIGHTS,
                               cost=spec.DubinsCost(**WEIGHTS), params=spec.DubinsParams(v_max=1.7, omega_max=1.3, dt=meta["cfg"]["mpc_timestep"]))
    finally:
        specs.ODE_REGISTRY["DubinsCar"] = saved
    _report(f"env_ticks non-default parameters {optimizer}: share of rollouts entering the obstacle per tick {[f'{x:.1%}' for x in shares]}")
    assert all(0.02 <= x <= 0.98 for x in shares), shares


# ---- 7. edge states ----------------------------------------------------------------------------------------------------------
EDGE_STATES = [("yaw_pi", [0.1, -0.1, np.pi]), ("yaw_minus_pi", [0.1, -0.1, -np.pi]), ("yaw_below_pi", [-0.05, 0.1, np.pi - 1e-6]),
               ("yaw_above_minus_pi", [-0.05, 0.1, -(np.pi - 1e-6)]), ("yaw_unwrapped", [0.0, 0.0, 3 * np.pi + 0.1]),
               ("far_away", [-150.0, 250.0, 0.7])]


@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
@pytest.mark.parametrize("name,s", EDGE_STATES, ids=[e[0] for e in EDGE_STATES])
def test_edge_states(optimizer, name, s):
    over = dict(cem_outer_it=1, cem_best_k=16) if optimizer == "cem-tf" else {}
    if name == "far_away" and optimizer == "mppi":
        # costs ~1e6 with an fp32 rounding of ~0.1: a temperature on the scale of the cost keeps the softmin well conditioned
        over["LBD"] = 1e4
    meta = _meta(optimizer, num_rollouts=256, **over)
    _logged_ticks(f"edge state {name} {optimizer}", meta, [np.asarray(s, np.float32)], seed=12)
