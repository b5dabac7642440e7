"""-m gpu: the network predictors step by step against float64, on weight sets that exercise every bias, every hidden width,
saturated activations and the tile engines' edge populations (weight sets: tests/test_predictor_weight_sets.py).

One-step residual.  The closed-loop checks (u_nom after the softmin average, per-rollout J under a q99 criterion) average a predictor
error confined to a few rows away.  Here every logged transition is checked on its own: the float64 network applied to the device's
own (s[n, t], Q[n, t]) against the device's s[n, t + 1], max over rollouts, steps and the six outputs of |dev - ref| / (1 + |ref|),
the angle modulo 2 pi.  One step is not amplified by the pendulum's chaos, so the bound is per row and tight:
  * simt, tcgen05 (exact): an fp32-level bound;
  * tcgen05_bf16: against the oracle with the same bf16 rounding of h1 and W2 (layer 1 is a three-term split on the tensor core,
    fp32-level); an fp32 ulp of h1 can flip one bf16 rounding, which the float64 oracle does not reproduce;
  * tcgen05_fast (MUFU tanh, ~2^-11 relative per activation, bf16 layer 2): a loose bound, no parity claim.
The GRU is checked teacher-forced: the float64 cell walks each logged rollout on the device's states and controls, carrying its own
hidden state from the one the tick's rollouts started from.  Measured maxima go to the parity report of test_gpu_parity._report.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from gpu_helpers import make_controller, max_rel
from helpers import load_golden, make_oracle
from test_gpu_parity import _check_J, _report
from test_gpu_production_pinning import _J_floor, _assert_state, _state_errs
from test_predictor_weight_sets import (GRU_ONE_STEP_BOUND, ONE_STEP_MEDIAN_BOUND, gru_spec, gru_weights, mlp_spec, mlp_weights,
                                        one_step_bound, one_step_residual, predictor_name)

pytestmark = pytest.mark.gpu

TILE_ROLLOUTS_PER_PASS = {"tcgen05": 256, "tcgen05_bf16": 512, "tcgen05_fast": 512}  # rollouts per CTA pass (tiles in flight x 128)
CEM_CFG = dict(seed=42, mpc_horizon=30, mpc_timestep=0.02, cem_outer_it=2, cem_initial_action_stdev=0.5, num_rollouts=1000,
               cem_stdev_min=0.01, cem_best_k=16, warmup=False, warmup_iterations=250)


def _meta(set_name, optimizer="mppi", **cfg_over):
    _, meta = load_golden("mppi_mlp_c4_n256")
    cfg = dict(meta["cfg"]) if optimizer == "mppi" else dict(CEM_CFG)
    cfg.update(cfg_over)
    return dict(meta, optimizer=optimizer, predictor=predictor_name(set_name), cfg=cfg)


def _gru_meta(hidden, optimizer, **cfg_over):
    _, meta = load_golden("mppi_gru_n256" if optimizer == "mppi" else "cem_gru_n256_k16")
    return dict(meta, predictor=predictor_name(f"gru{hidden}"), cfg=dict(meta["cfg"], **cfg_over))


def _mlp_oracles(meta, set_name, **over):
    o32, o64 = make_oracle(meta, **over), make_oracle(meta, dtype=torch.float64, **over)
    o32.predictor = spec_mlp(set_name, torch.float32)
    o64.predictor = spec_mlp(set_name, torch.float64)
    return o32, o64


def spec_mlp(set_name, dtype, bf16=False, device="cpu"):
    from oracle import spec
    p = spec.MLPPredictor(mlp_weights(set_name), dtype=dtype, bf16_layer2=bf16)
    p.t = {k: v.to(device) for k, v in p.t.items()}
    return p


def _logs(opt):
    lv = opt.logging_values
    return np.asarray(lv["rollout_trajectories_logged"]), np.asarray(lv["Q_logged"])


def _mlp_one_step(set_name, traj, Q, bf16=False, chunk=1 << 20):
    """[N, H] one-step residuals of the logged rollouts against the float64 network (evaluated on the GPU in float64)."""
    p = spec_mlp(set_name, torch.float64, bf16=bf16, device="cuda")
    N, H = Q.shape[0], Q.shape[1]
    s, q, nxt = traj[:, :-1].reshape(-1, 6), Q.reshape(-1, 1), traj[:, 1:].reshape(-1, 6)
    out = np.empty(N * H)
    for c in range(0, N * H, chunk):
        y = p.step(torch.from_numpy(np.ascontiguousarray(s[c:c + chunk])).cuda().double(),
                   torch.from_numpy(np.ascontiguousarray(q[c:c + chunk])).cuda().double())
        out[c:c + chunk] = one_step_residual(nxt[c:c + chunk], y.cpu().numpy())
    return out.reshape(N, H)


def _where(e, engine):
    """The worst (rollout, step) and, on the tile engines, where that row sits in its CTA's share of the population."""
    n, t = (int(i) for i in np.unravel_index(int(np.argmax(e)), e.shape))
    loc = f"rollout {n} step {t}"
    if engine in TILE_ROLLOUTS_PER_PASS:
        N = e.shape[0]
        S = torch.cuda.get_device_properties(0).multi_processor_count
        G = max(1, min(S, (N + 127) // 128))
        b = max(i for i in range(G) if i * N // G <= n)
        r, share, rpp = n - b * N // G, (b + 1) * N // G - b * N // G, TILE_ROLLOUTS_PER_PASS[engine]
        loc += f" = CTA {b}/{G}, row {r} of its {share}-row share (pass {r // rpp}, tile {r % rpp // 128}, tile row {r % 128})"
    return loc


def _check_one_step(tag, e, engine, bound, median_bound=None):
    med = float(np.median(e))
    _report(f"{tag}: one-step max {e.max():.2e} median {med:.2e} at {_where(e, engine)} | bound {bound:.1e}"
            + (f", median bound {median_bound:.0e}" if median_bound else ""))
    assert e.max() < bound, (tag, float(e.max()), _where(e, engine))
    if median_bound is not None:
        assert med < median_bound, (tag, "median", med)


# ---------------------------------------------------------------------------------------------------------------------------------
# a. one-step residual of every MLP engine
# ---------------------------------------------------------------------------------------------------------------------------------
MLP_CASES = ([("mppi", e, s) for e in ("simt", "tcgen05", "tcgen05_bf16", "tcgen05_fast") for s in ("biased", "saturating")]
             + [("mppi", "simt", s) for s in ("w16", "w48", "w112")]
             + [("cem-tf", e, s) for e in ("simt", "tcgen05") for s in ("biased", "saturating")]
             + [("cem-tf", "simt", s) for s in ("w16", "w48", "w112")])


@pytest.mark.parametrize("optimizer,engine,set_name", MLP_CASES)
def test_mlp_one_step_matches_float64(optimizer, engine, set_name):
    """Every logged transition of an MPPI / CEM tick (in-kernel noise, a population that leaves a partial last tile) against the
    float64 network on the device's own state and control."""
    N = 3001 if optimizer == "mppi" else 1000
    meta = _meta(set_name, optimizer, num_rollouts=N, mpc_horizon=30)
    ctrl = make_controller(meta, rng=None, logging=True, weights=mlp_spec(set_name), mlp_engine=engine)
    opt = ctrl.optimizer
    from oracle import spec
    for t, s in enumerate(spec.synthetic_states(2, seed=31)):
        ctrl.step(s)
        traj, Q = _logs(opt)
        assert np.isfinite(traj).all()
        e = _mlp_one_step(set_name, traj, Q, bf16=engine in ("tcgen05_bf16", "tcgen05_fast"))
        _check_one_step(f"one-step {optimizer} [{opt.last_kernel}] {set_name} N={N} tick {t}", e, engine, one_step_bound(engine, set_name),
                        ONE_STEP_MEDIAN_BOUND.get(engine))


# ---------------------------------------------------------------------------------------------------------------------------------
# b. GRU, teacher-forced, every width
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("optimizer", ["mppi", "cem-tf"])
@pytest.mark.parametrize("hidden", [8, 16, 24, 32])
def test_gru_teacher_forced_matches_float64(optimizer, hidden):
    """The float64 GRU walks each logged rollout on the device's states and controls from the hidden state the tick's rollouts started
    from (read before the tick: MPPI advances it after its rollouts, CEM never does); the per-step residual is asserted, and for
    MPPI the saved state after the tick against the oracle's predictor.update(s, u_nom[0])."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    meta = _gru_meta(hidden, optimizer, num_rollouts=500)
    ctrl = make_controller(meta, rng=None, logging=True, weights=gru_spec(hidden))
    opt = ctrl.optimizer
    p64 = spec.GRUPredictor(gru_weights(hidden), dtype=torch.float64)
    p64.t = {k: v.cuda() for k, v in p64.t.items()}
    upd = spec.GRUPredictor(gru_weights(hidden), dtype=torch.float64)
    for tick, s in enumerate(spec.synthetic_states(3, seed=32)):
        h0 = opt._get_state(L.STATE_RNN_H, (2, hidden)).astype(np.float64)
        if tick == 0:
            assert not h0.any()
        ctrl.step(s)
        traj, Q = _logs(opt)
        N, H = Q.shape[0], Q.shape[1]
        h1 = torch.from_numpy(h0[0]).cuda().repeat(N, 1)
        h2 = torch.from_numpy(h0[1]).cuda().repeat(N, 1)
        e = np.empty((N, H))
        for t in range(H):
            y, h1, h2 = p64._net(torch.from_numpy(traj[:, t]).cuda().double(), torch.from_numpy(Q[:, t]).cuda().double(), h1, h2)
            e[:, t] = one_step_residual(traj[:, t + 1], y.cpu().numpy())
        _check_one_step(f"gru teacher-forced {optimizer} hidden={hidden} N={N} tick {tick}", e, "simt", GRU_ONE_STEP_BOUND)
        if optimizer == "mppi":
            upd.h1, upd.h2 = torch.from_numpy(h0[:1].copy()), torch.from_numpy(h0[1:].copy())
            upd.update(s=np.asarray(s, np.float32)[None], Q0=np.float32(opt.u_nom[0, 0, 0]))
            ref = torch.cat([upd.h1, upd.h2]).numpy()
            e_h = max_rel(opt._get_state(L.STATE_RNN_H, (2, hidden)), ref)
            _report(f"gru {optimizer} hidden={hidden} tick {tick}: saved hidden state after the update {e_h:.2e}")
            assert e_h < 1e-5, (hidden, tick, e_h)
        else:
            assert not opt._get_state(L.STATE_RNN_H, (2, hidden)).any()  # CEM has no predictor.update


# ---------------------------------------------------------------------------------------------------------------------------------
# c. closed-loop parity on the new weight sets
# ---------------------------------------------------------------------------------------------------------------------------------
# Not on the saturating set: its closed loop is not reproducible in fp32 at all -- the fp32 oracle's u_nom is 1.9 (relative) away from
# the float64 oracle's on the first tick (B200 run, 1000 rollouts, H = 50): saturated units and the track barrier make the softmin
# weights jump on rounding.  One step of that network is well conditioned and is checked above, per row.
@pytest.mark.parametrize("engine,set_name", [("simt", "biased"), ("tcgen05", "biased"), ("simt", "w16"), ("simt", "w48"), ("simt", "w112")])
def test_mppi_mlp_weight_sets_match_oracle(engine, set_name):
    """MPPI on injected noise, every tick from the fp32 oracle's state: u_nom under the symmetric fp32 / float64 criterion of
    test_gpu_production_pinning.py, per-rollout J under test_gpu_parity.py's."""
    from oracle import spec
    from oracle.replay_rng import ReplayRNG
    meta = _meta(set_name, num_rollouts=1000, mpc_horizon=50)
    ctrl = make_controller(meta, rng=None, logging=True, weights=mlp_spec(set_name), mlp_engine=engine)
    opt = ctrl.optimizer
    opt.rng = ReplayRNG(61, as_torch=False)
    opt.optimizer_reset()
    o32, o64 = _mlp_oracles(meta, set_name)
    r32, r64 = ReplayRNG(61), ReplayRNG(61)
    for t, s in enumerate(spec.synthetic_states(3, seed=33)):
        if t > 0:
            opt.set_state({"u_nom": o32.u_nom.numpy().astype(np.float32), "u": float(o32.u)})
            o64.u_nom, o64.u = o32.u_nom.double().clone(), np.float64(o32.u)
        u = ctrl.step(s)
        o32.step(s, r32)
        o64.step(s, r64)
        e32, e64, floor = _state_errs(opt.u_nom, o32.u_nom.numpy(), o64.u_nom.numpy())
        _assert_state(f"mppi mlp {set_name} [{opt.last_kernel}] tick {t} u_nom", e32, e64, floor, False)
        assert abs(float(u) - float(o32.u)) < 1e-4
        _check_J(opt.logging_values["J_logged"], o32.last["J"], _J_floor(o32.last["J"], o64.last["J"]), (f"mppi mlp {set_name} {engine}", t))


@pytest.mark.parametrize("engine,set_name", [("simt", "biased"), ("tcgen05", "biased"), ("simt", "w48")])
def test_cem_mlp_weight_sets_match_oracle(engine, set_name):
    """CEM on injected noise, every tick from the fp32 oracle's distribution: elite index sets of every outer iteration identical,
    (mu, sigma) under the symmetric criterion, J under test_gpu_parity.py's."""
    from oracle import spec
    from oracle.replay_rng import ReplayRNG
    meta = _meta(set_name, "cem-tf")
    ctrl = make_controller(meta, rng=None, logging=True, weights=mlp_spec(set_name), mlp_engine=engine)
    opt = ctrl.optimizer
    opt.rng = ReplayRNG(62, as_torch=False)
    opt.optimizer_reset()
    o32, o64 = _mlp_oracles(meta, set_name)
    r32, r64 = ReplayRNG(62), ReplayRNG(62)
    for t, s in enumerate(spec.synthetic_states(3, seed=34)):
        if t > 0:
            opt.set_state({"dist_mue": o32.dist_mue.numpy(), "stdev": o32.stdev.numpy(), "count": o32.count, "u": float(o32.u)})
            o64.dist_mue, o64.stdev, o64.u = o32.dist_mue.double().clone(), o32.stdev.double().clone(), np.float64(o32.u)
        u = ctrl.step(s)
        o32.step(s, r32)
        o64.step(s, r64)
        got, ref = opt.elite_indices, np.asarray(o32.last["elite_idx"])
        for it in range(ref.shape[0]):
            assert set(got[it].tolist()) == set(ref[it].tolist()), (set_name, engine, t, it, sorted(set(got[it].tolist()) ^ set(ref[it].tolist())))
        for nm, a, b32, b64 in (("mu", opt.dist_mue, o32.dist_mue, o64.dist_mue), ("sd", opt.stdev, o32.stdev, o64.stdev)):
            e32, e64, floor = _state_errs(a, b32.numpy(), b64.numpy())
            _assert_state(f"cem mlp {set_name} [{opt.last_kernel}] tick {t} {nm}", e32, e64, floor, False)
        assert abs(float(u) - float(o32.u)) < 1e-4
        _check_J(opt.logging_values["J_logged"], o32.last["J"], _J_floor(o32.last["J"], o64.last["J"]), (f"cem mlp {set_name} {engine}", t))


# ---------------------------------------------------------------------------------------------------------------------------------
# d. tile-engine edge populations
# ---------------------------------------------------------------------------------------------------------------------------------
EDGE_N = {  # S = SM count.  Tile engines: grid min(S, ceil(N / 128)) CTAs, CTA b rolls out rows [b N / grid, (b + 1) N / grid)
    "1": lambda S: 1,                     # a single real row in one tile
    "129": lambda S: 129,                 # two CTAs of 64 / 65 rows: half tiles
    "128S+1": lambda S: 128 * S + 1,      # one CTA with a 129-row share
    "257S": lambda S: 257 * S,            # every CTA one row past two tiles: a one-row second pass on the exact engine
    "512S+1": lambda S: 512 * S + 1,      # one CTA with a one-row second pass on the four-tile engines
}


@pytest.mark.parametrize("engine", ["tcgen05", "tcgen05_bf16", "tcgen05_fast"])
@pytest.mark.parametrize("pop", list(EDGE_N))
def test_tile_engine_edge_populations(engine, pop):
    """Populations at which group_active / begin_rollout / tile_rows / row_on decide which warps compute: the one-step residual over
    every row, and u_nom on the exact engine against the oracle on the exported Philox draws (H = 50, period 10)."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    from oracle.replay_rng import QueueRNG
    S = torch.cuda.get_device_properties(0).multi_processor_count
    N = EDGE_N[pop](S)
    meta = _meta("biased", num_rollouts=N, mpc_horizon=50)
    ctrl = make_controller(meta, rng=None, logging=True, weights=mlp_spec("biased"), mlp_engine=engine)
    opt = ctrl.optimizer
    s = spec.synthetic_states(1, seed=35)[0]
    u = ctrl.step(s)
    traj, Q = _logs(opt)
    assert traj.shape[0] == N and np.isfinite(traj).all()
    e = _mlp_one_step("biased", traj, Q, bf16=engine != "tcgen05")
    _check_one_step(f"edge population N={pop}={N} [{opt.last_kernel}]", e, engine, one_step_bound(engine, "biased"),
                    ONE_STEP_MEDIAN_BOUND.get(engine))
    if engine == "tcgen05" and N <= 128 * S + 1:
        z = opt.export_philox(L.STREAM_MPPI, opt.tick_counter, opt.number_of_interpolation_inducing_points, N)
        o32, o64 = _mlp_oracles(meta, "biased")
        u32 = o32.step_chunked(s, QueueRNG([z]), chunk=8192)
        o64.step_chunked(s, QueueRNG([z]), chunk=8192)
        e32, e64, floor = _state_errs(opt.u_nom, o32.u_nom.numpy(), o64.u_nom.numpy())
        _assert_state(f"edge population N={pop}={N} [{opt.last_kernel}] u_nom", e32, e64, floor, False)
        assert abs(float(u) - float(np.ravel(u32)[0])) < 1e-4


# ---------------------------------------------------------------------------------------------------------------------------------
# e. weight replacement on a live handle
# ---------------------------------------------------------------------------------------------------------------------------------
def _set_weights(opt, w):
    from control_toolkit_b200 import _lib as L
    lib = L.load()
    c = w.to_c()  # (w keeps the arrays alive)
    rc = (lib.ctk_set_gru_weights if hasattr(w, "_KEYS") else lib.ctk_set_mlp_weights)(opt._h, C.byref(c))
    return rc, (lib.ctk_last_error() or b"").decode()


def _same_next_tick(a, b, s):
    """b takes a's optimizer state and Philox tick counter; both tick on s and must agree bit for bit."""
    from control_toolkit_b200 import _lib as L
    b.optimizer.set_state(a.optimizer.get_state())
    b.optimizer._set_counter(L.COUNTER_TICK, a.optimizer.tick_counter)
    ua, ub = a.step(s), b.step(s)
    assert float(ua) == float(ub)
    np.testing.assert_array_equal(a.optimizer.u_nom, b.optimizer.u_nom)


@pytest.mark.parametrize("engine,first,second", [("simt", "biased", "w48"), ("tcgen05", "biased", "saturating")])
def test_mlp_weight_replacement_equals_a_fresh_handle(engine, first, second):
    """ctk_set_mlp_weights on a handle that has ticked (the simt engine changes the width 128 -> 48; tcgen05 rebuilds its tile blob):
    the next tick equals that of a fresh handle holding the new weights, on the same optimizer state and noise."""
    from oracle import spec
    s = spec.synthetic_states(2, seed=36)
    meta = _meta(first, num_rollouts=2000, mpc_horizon=30)
    a = make_controller(meta, rng=None, logging=False, weights=mlp_spec(first), mlp_engine=engine)
    a.step(s[0])
    rc, msg = _set_weights(a.optimizer, mlp_spec(second))
    assert rc == 0, msg
    b = make_controller(_meta(second, num_rollouts=2000, mpc_horizon=30), rng=None, logging=False, weights=mlp_spec(second), mlp_engine=engine)
    _same_next_tick(a, b, s[1])


def test_gru_weight_replacement_zeroes_the_saved_state():
    """include/ctk_b200.h: replacing the GRU weights zeroes the saved hidden state; the next tick equals a fresh handle's."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    s = spec.synthetic_states(3, seed=37)
    a = make_controller(_gru_meta(32, "mppi"), rng=None, logging=False, weights=gru_spec(32))
    a.step(s[0])
    a.step(s[1])
    assert np.abs(a.optimizer._get_state(L.STATE_RNN_H, (2, 32))).max() > 0
    rc, msg = _set_weights(a.optimizer, gru_spec(16))
    assert rc == 0, msg
    assert not a.optimizer._get_state(L.STATE_RNN_H, (2, 16)).any()
    b = make_controller(_gru_meta(16, "mppi"), rng=None, logging=False, weights=gru_spec(16))
    _same_next_tick(a, b, s[2])
    np.testing.assert_array_equal(a.optimizer._get_state(L.STATE_RNN_H, (2, 16)), b.optimizer._get_state(L.STATE_RNN_H, (2, 16)))


def test_rejected_mlp_weights_leave_the_handle_as_it_was():
    """A width the tcgen05 engine cannot run is refused with CTK_EINVAL and its message, and the handle keeps its weights: the next
    tick equals that of a twin that never saw the call."""
    import control_toolkit_b200 as ctk
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    s = spec.synthetic_states(2, seed=38)
    meta = _meta("biased", num_rollouts=2000, mpc_horizon=30)
    a = make_controller(meta, rng=None, logging=False, weights=mlp_spec("biased"), mlp_engine="tcgen05")
    twin = make_controller(meta, rng=None, logging=False, weights=mlp_spec("biased"), mlp_engine="tcgen05")
    a.step(s[0])
    twin.step(s[0])
    rc, msg = _set_weights(a.optimizer, ctk.MLPSpec.random_init(5, hidden=64))
    assert rc == L.CTK_EINVAL
    assert "the tcgen05 MLP engines are built for hidden == 128" in msg
    _same_next_tick(twin, a, s[1])


# ---------------------------------------------------------------------------------------------------------------------------------
# f. nominal rollout (calculate_optimal_trajectory)
# ---------------------------------------------------------------------------------------------------------------------------------
NOMINAL_CASES = [("mppi_ode", None), ("mppi_mlp", "simt"), ("mppi_mlp", "tcgen05"), ("mppi_mlp", "tcgen05_bf16"), ("mppi_mlp", "tcgen05_fast"),
                 ("mppi_gru", None), ("rpgd_ode", None)]


@pytest.mark.parametrize("case,engine", NOMINAL_CASES)
def test_nominal_rollout_matches_oracle(case, engine):
    """optimal_trajectory (ctk_rollout_single: single_rollout_kernel<OdePred | MlpSimtPred> -- every MLP engine rolls the nominal
    sequence out on the FP32 pipe -- and single_rollout_gru_kernel, which starts from the hidden state before the tick's update)
    against the oracle's predict_core(s, u_nom) under the symmetric fp32 / float64 criterion, and the summed stage cost against
    sum_t (stage_cost - MAX_COST) with the previous input the handle holds after the tick: the control just returned."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    over = {}
    if case == "mppi_ode":
        _, meta = load_golden("mppi_c1_n64")
        net = lambda dt: spec.ODEPredictor(spec.CartPoleParams(dt=meta["cfg"]["mpc_timestep"]))  # noqa: E731
    elif case == "rpgd_ode":
        _, meta = load_golden("rpgd_c3")
        over["adam_form"] = "torch"
        net = lambda dt: spec.ODEPredictor(spec.CartPoleParams(dt=meta["cfg"]["mpc_timestep"]))  # noqa: E731
    elif case == "mppi_mlp":
        meta = _meta("biased", num_rollouts=1000, mpc_horizon=50)
        over.update(weights=mlp_spec("biased"), mlp_engine=engine)
        net = lambda dt: spec_mlp("biased", dt)  # noqa: E731
    else:
        meta = _gru_meta(24, "mppi")
        over["weights"] = gru_spec(24)
        net = lambda dt: spec.GRUPredictor(gru_weights(24), dtype=dt)  # noqa: E731
    ctrl = make_controller(meta, rng=None, logging=False, optimal_trajectory=True, **over)
    opt = ctrl.optimizer
    cp = spec.CostParams(name=meta["cost"])
    H = opt.mpc_horizon
    for t, s in enumerate(spec.synthetic_states(3, seed=39)):
        h0 = opt._get_state(L.STATE_RNN_H, (2, 24)).astype(np.float64) if case == "mppi_gru" else None
        u = ctrl.step(s)
        traj = np.asarray(opt.optimal_trajectory, np.float64)
        assert traj.shape == (1, H + 1, 6)
        u_prev = float(opt._get_state(L.STATE_U_PREV, (1,))[0])
        assert u_prev == float(np.ravel(u)[0])  # the previous input the nominal rollout's cost sees
        summed = opt.summed_stage_cost if case == "rpgd_ode" else opt.rollout_single(s, opt.u_nom)[1]
        ref, cost = {}, {}
        for dt in (torch.float32, torch.float64):
            p = net(dt)
            if h0 is not None:
                p.h1, p.h2 = torch.from_numpy(h0[:1]).to(dt), torch.from_numpy(h0[1:]).to(dt)
            s_t = torch.from_numpy(np.asarray(s, np.float32)[None]).to(dt)
            Q = torch.from_numpy(np.asarray(opt.u_nom, np.float32)).to(dt)
            r = p.predict_core(s_t, Q)
            ref[dt] = r.numpy()
            sc = spec.stage_cost(r[:, :-1], Q, torch.tensor(u_prev, dtype=dt), cp) - cp.f32()["MAX_COST"]
            cost[dt] = float(torch.sum(sc))
        e32, e64, floor = _state_errs(traj, ref[torch.float32], ref[torch.float64])
        _assert_state(f"nominal rollout {case} {engine or ''} tick {t}", e32, e64, floor, False)
        c64 = cost[torch.float64]
        ec = abs(float(np.ravel(summed)[0]) - c64) / (abs(c64) + 1e-3)
        fc = abs(cost[torch.float32] - c64) / (abs(c64) + 1e-3)
        _report(f"nominal rollout {case} {engine or ''} tick {t}: summed stage cost {float(np.ravel(summed)[0]):.6g} vs float64 {c64:.6g} "
                f"rel {ec:.2e} (fp32 oracle {fc:.2e})")
        assert ec <= max(1e-4, 4 * fc), (case, t, ec, fc)


def test_nominal_rollout_is_cartpole_only():
    from control_toolkit_b200 import _lib as L
    _, meta = load_golden("mppi_dubins_n512")
    ctrl = make_controller(meta, rng=None, logging=False)
    lib = L.load()
    s, q = np.zeros(3, np.float32), np.zeros(ctrl.optimizer.mpc_horizon * 2, np.float32)
    traj, summed = np.zeros((ctrl.optimizer.mpc_horizon + 1) * 6, np.float32), np.zeros(1, np.float32)
    rc = lib.ctk_rollout_single(ctrl.optimizer._h, L.fptr(s), L.fptr(q), L.fptr(traj), L.fptr(summed))
    assert rc == L.CTK_EINVAL
    assert "implemented for the CartPole environment" in (lib.ctk_last_error() or b"").decode()
