"""GPU tests of the gradient optimizers on the Dubins car (env_rpgd_grad_kernel + K8 over nu = 2 columns, ctk_kernels_env_rpgd.cuh):
the gradient of one step against float64 autograd, closed loops of RPGD and its three siblings against the oracles on injected noise,
the production path on in-kernel Philox (one launch per tick at C3 geometry), edge geometries, logging, state round trips and the
device-resident tick.  Limits differ per input (throttle [-0.5, 1], steer [-1, 1]) so that mixed-up inputs show.

Tolerances: |cuda - fp32 oracle| <= 2e-4 on controls in [-1, 1] while the cost ranking is identical (as the CartPole sibling tests of
test_gpu_parity.py); the oracle's own fp32-vs-float64 floor is reported beside every number."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

LOW, HIGH = np.array([-0.5, -1.0], np.float32), np.array([1.0, 1.0], np.float32)
DT = 0.02
BASE = {
    "rpgd": dict(mpc_horizon=50, num_rollouts=32, outer_its=2, sample_stdev=0.5, sample_mean=0.0, sample_whole_control_space=True,
                 uniform_dist_min=-1.0, uniform_dist_max=1.0, resamp_per=3, period_interpolation_inducing_points=10,
                 SAMPLING_DISTRIBUTION="uniform", shift_previous=1, warmup=False, warmup_iterations=250, learning_rate=0.05,
                 opt_keep_k_ratio=0.25, gradmax_clip=5, adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1e-8, adam_form="keras"),
    "gradient-tf": dict(mpc_horizon=35, num_rollouts=40, gradient_steps=5, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999,
                        adam_epsilon=1e-7, gradmax_clip=5, warmup=False, warmup_iterations=250),
    "cem-naive-grad-tf": dict(mpc_horizon=35, num_rollouts=200, cem_outer_it=1, cem_stdev_min=0.1, cem_initial_action_stdev=0.5,
                              cem_best_k=40, learning_rate=0.1, gradmax_clip=10),
    "cem-grad-bharadhwaj-tf": dict(mpc_horizon=50, num_rollouts=32, cem_best_k=8, cem_outer_it=2, cem_initial_action_stdev=2,
                                   cem_stdev_min=1e-6, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1e-8,
                                   gradmax_clip=5, warmup=False, warmup_iterations=250),
}


def _report(msg):
    print(msg)  # pytest -s shows the measured errors and floors


def _meta(optimizer, **over):
    cfg = dict(BASE[optimizer], mpc_timestep=DT, seed=42)
    cfg.update(over)
    return dict(optimizer=optimizer, predictor="ODE", cost="default", environment="DubinsCar", noise_seed=1, cfg=cfg)


def _controller(meta, logging=False, seed=None, low=LOW, high=HIGH, optimal_trajectory=False):
    from control_toolkit_b200.Controllers.controller_mpc import controller_mpc
    from oracle.replay_rng import ReplayRNG
    ctrl = controller_mpc(
        environment_name="DubinsCar", control_limits=(low, high), initial_environment_attributes={},
        config_controller=dict(optimizer=meta["optimizer"], predictor_specification="ODE", cost_function_specification="default",
                               controller_logging=logging, calculate_optimal_trajectory=optimal_trajectory),
        config_optimizers={meta["optimizer"]: dict(meta["cfg"])}, config_cost_function={"cost_function_name_default": "default"})
    ctrl.configure(optimizer_name=meta["optimizer"], predictor_specification="ODE")
    if seed is not None:
        ctrl.optimizer.rng = ReplayRNG(seed, as_torch=False)
        ctrl.optimizer.optimizer_reset()
    return ctrl


def _oracles(meta, low=LOW, high=HIGH):
    """fp32 and float64 oracles of the optimizer (tests/env_gradient_oracles.py: the oracle/ restatements for nu inputs)."""
    import torch
    from env_gradient_oracles import ORACLES
    from oracle import spec

    def make(dtype):
        return ORACLES[meta["optimizer"]](spec.DubinsPredictor(spec.DubinsParams(dt=DT)), spec.DubinsCost(name=meta["cost"]),
                                          action_low=low, action_high=high, dtype=dtype, **meta["cfg"])
    return make(torch.float32), make(torch.float64)


def _states(n, seed=31):
    from oracle import spec
    return spec.dubins_synthetic_states(n, seed=seed)


def _rel(a, b, floor=1e-2):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), floor))


# ---- 1. the gradient of one step -----------------------------------------------------------------------------------------
def test_gradient_of_one_step_matches_float64_autograd():
    """m = v = 0, count 1 (no resampling with resamp_per 1000), one Keras step, clip out of reach: after the tick
    m[:, t-1, :] = (1 - b1) dJ/dQ[:, t, :] (the moments shift by one step).  Compared with float64 autograd from the device's Q."""
    import torch
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    N, H = 64, 50
    meta = _meta("rpgd", num_rollouts=N, mpc_horizon=H, outer_its=1, resamp_per=1000, gradmax_clip=1e9)
    ctrl = _controller(meta, seed=5)
    opt = ctrl.optimizer
    rng = np.random.default_rng(3)
    Q = np.stack([rng.uniform(-0.5, 1.0, (N, H)), rng.uniform(-1, 1, (N, H))], 2).astype(np.float32)
    up = np.array([0.3, -0.2], np.float32)
    opt._set_state(L.STATE_RPGD_Q, Q)
    opt._set_state(L.STATE_RPGD_M, np.zeros_like(Q))
    opt._set_state(L.STATE_RPGD_V, np.zeros_like(Q))
    opt._set_state(L.STATE_U_PREV, up)
    opt._set_counter(L.COUNTER_COUNT, 1)
    opt.count = 1
    Qd = opt.Q_tf
    assert np.array_equal(Qd, Q)
    s = np.array([0.1, -0.1, 2.9], np.float32)
    ctrl.step(s)
    m = opt.adam_weights()[1]

    def grad(dtype):
        q = torch.tensor(Qd, dtype=dtype, requires_grad=True)
        traj = spec.DubinsPredictor(spec.DubinsParams(dt=DT)).predict_core(torch.tensor(np.tile(s, (N, 1)), dtype=dtype), q)
        J = spec.trajectory_cost(traj, q, torch.tensor(up, dtype=dtype), spec.DubinsCost())
        return torch.autograd.grad(J.sum(), q)[0].numpy().astype(np.float64)

    g64, g32 = grad(torch.float64), grad(torch.float32)
    g_dev = m[:, :-1, :].astype(np.float64) / (1.0 - 0.9)
    row = np.abs(g64[:, 1:, :]).reshape(N, -1).max(1)[:, None, None]
    err = np.abs(g_dev - g64[:, 1:, :])
    bound = np.maximum(1e-4 * row, 4 * np.abs(g32[:, 1:, :] - g64[:, 1:, :]))
    _report(f"env gradient one step [{opt.last_kernel}]: max err/row {float((err / row).max()):.2e}, max err/bound {float((err / bound).max()):.3f}, "
            f"fp32 autograd floor {float((np.abs(g32 - g64)[:, 1:, :] / row).max()):.2e}")
    assert float((err / bound).max()) <= 1.0
    assert "env_rpgd_grad_kernel<DubinsEnv,0>" in opt.last_kernel


# ---- 2. closed loops against the oracles ----------------------------------------------------------------------------------
LOOPS = [
    ("rpgd_keras_uniform", "rpgd", {}),
    ("rpgd_torch_normal_shift2", "rpgd", dict(adam_form="torch", SAMPLING_DISTRIBUTION="normal", shift_previous=2, resamp_per=2,
                                              num_rollouts=64, mpc_horizon=30, period_interpolation_inducing_points=5)),
    ("rpgd_keras_normal_resample_every_tick", "rpgd", dict(SAMPLING_DISTRIBUTION="normal", resamp_per=1, num_rollouts=48)),
    ("rpgd_not_whole_space", "rpgd", dict(sample_whole_control_space=False, uniform_dist_min=-0.3, uniform_dist_max=0.6)),
    ("gradient_tf", "gradient-tf", {}),
    ("cem_naive_grad", "cem-naive-grad-tf", {}),
    ("cem_bharadhwaj", "cem-grad-bharadhwaj-tf", {}),
]


def _same_ranking(opt, o, optimizer):
    if optimizer == "rpgd":
        return np.array_equal(opt.best_indices(), o.last["best_idx"])
    if optimizer == "gradient-tf":
        return opt.best_index() == o.last["best_idx"]
    got, ref = opt.elite_indices(), o.last["elite_idx"]
    return got.shape == ref.shape and all(set(a.tolist()) == set(b.tolist()) for a, b in zip(got, ref))


def _opt_state(opt, o, optimizer):
    """(device, fp32 oracle, float64 oracle) arrays of the optimizer state this tick leaves."""
    if optimizer in ("rpgd", "gradient-tf"):
        return [("Q", opt.Q_tf, o[0].Q.numpy(), o[1].Q.numpy()), ("m", opt.adam_weights()[1], o[0].m.numpy(), o[1].m.numpy()),
                ("v", opt.adam_weights()[2], o[0].v.numpy(), o[1].v.numpy())]
    out = [("dist_mue", opt.dist_mue, o[0].dist_mue.numpy(), o[1].dist_mue.numpy()), ("stdev", opt.stdev, o[0].stdev.numpy(), o[1].stdev.numpy())]
    if optimizer == "cem-grad-bharadhwaj-tf":
        out.append(("m", opt.adam_weights()[1], o[0].m.numpy(), o[1].m.numpy()))
    return out


@pytest.mark.parametrize("name,optimizer,over", LOOPS, ids=[x[0] for x in LOOPS])
def test_closed_loop_matches_oracle_on_injected_noise(name, optimizer, over):
    from oracle.replay_rng import ReplayRNG
    meta = _meta(optimizer, **over)
    ctrl = _controller(meta, seed=11)
    opt = ctrl.optimizer
    o32, o64 = _oracles(meta)
    r32, r64 = ReplayRNG(11), ReplayRNG(11)
    if optimizer in ("rpgd", "gradient-tf"):
        o32.reset(r32)
        o64.reset(r64)
    ticks = 0
    for t, s in enumerate(_states(12)):
        u = ctrl.step(s)
        u32, u64 = o32.step(s, r32), o64.step(s, r64)
        assert np.shape(u) == (2,)
        same = _same_ranking(opt, o32, optimizer)
        e_u, f_u = float(np.max(np.abs(np.ravel(u) - np.ravel(u32)))), float(np.max(np.abs(np.ravel(u32) - np.ravel(u64))))
        msg = [f"{name} [{opt.last_kernel}] tick {t}: u {e_u:.2e} (floor {f_u:.2e})"]
        errs = []
        for key, dev, a32, a64 in _opt_state(opt, (o32, o64), optimizer):
            scale = 1e-2 if key in ("Q", "dist_mue", "stdev") else 1e-30
            e, f = _rel(dev, a32, scale), _rel(a32, a64, scale)
            msg.append(f"{key} {e:.2e} (floor {f:.2e})")
            errs.append((key, e))
        if optimizer == "rpgd":
            e_ages = float(np.max(np.abs(opt.trajectory_ages - o32.ages.numpy())))
            msg.append(f"ages {e_ages:.0f}")
        J = opt.last_costs()
        eJ = float(np.max(np.abs(J - o32.last["J"]) / (np.abs(o32.last["J"]) + 1e-3)))
        msg.append(f"J {eJ:.2e} same_ranking {same}")
        _report(" ".join(msg))
        if not same:
            break  # a rounding-level swap in the cost ranking changes the population from here on
        ticks += 1
        assert e_u < 2e-4 and eJ < 1e-4, msg
        for key, e in errs:
            # the Adam moments are compared relative to their largest element; the Adam quirk (a control moved by O(lr) where
            # |g| ~ 1e-6) makes the population states diverge faster than u, as on the CartPole
            assert e < (2e-4 if t == 0 else 5e-3), (key, msg)
        if optimizer == "rpgd":
            assert e_ages == 0
    assert ticks >= 2, "the first ticks ranked differently from the oracle"


# ---- 3. production path: in-kernel Philox, one launch per tick ----------------------------------------------------------------
def test_production_philox_rpgd_c3_geometry_one_launch_per_tick():
    from control_toolkit_b200 import _lib as L
    from oracle.replay_rng import QueueRNG
    N, H = 32, 50
    meta = _meta("rpgd", num_rollouts=N, mpc_horizon=H, resamp_per=3)
    ctrl = _controller(meta)  # rng None: in-kernel Philox
    opt = ctrl.optimizer
    nu, n_ind, k = 2, opt.number_of_interpolation_inducing_points, opt.opt_keep_k
    o32, o64 = _oracles(meta)
    z0 = opt.export_philox(L.STREAM_RPGD_INIT, opt.tick_counter, n_ind * nu, N, uniform=True)
    o32.reset(QueueRNG([z0]))
    o64.reset(QueueRNG([z0]))
    assert np.array_equal(opt.Q_tf, o32.Q.numpy())
    lib = L.load()
    for t, s in enumerate(_states(12, seed=41)):
        before = C_int64(lib, opt)
        u = ctrl.step(s)
        assert C_int64(lib, opt) - before == 1, "RPGD at N = 32, logging off: one launch per tick"
        assert opt.last_kernel == "env_rpgd_grad_kernel<DubinsEnv,0> [fused select]"
        blocks = [opt.export_philox(L.STREAM_RPGD_RESAMPLE, opt.tick_counter, n_ind * nu, N - k, uniform=True)] if t % 3 == 0 else []
        u32 = o32.step(s, QueueRNG(blocks))
        o64.step(s, QueueRNG(list(blocks)))
        same = np.array_equal(opt.best_indices(), o32.last["best_idx"])
        e_Q, f_Q = _rel(opt.Q_tf, o32.Q.numpy()), _rel(o32.Q.numpy(), o64.Q.numpy())
        e_u = float(np.max(np.abs(np.ravel(u) - np.ravel(u32))))
        _report(f"production rpgd philox tick {t}: u {e_u:.2e} Q {e_Q:.2e} (floor {f_Q:.2e}) same_ranking {same}")
        if not same:
            break
        assert e_u < 2e-4 and e_Q < (2e-4 if t == 0 else 5e-3)
    assert t >= 2


def C_int64(lib, opt):
    import ctypes as C
    v = C.c_int64()
    assert lib.ctk_get_launch_count(opt._h, C.byref(v)) == 0
    return v.value


# ---- 4. edges ---------------------------------------------------------------------------------------------------------------
EDGES = [
    ("N1_H1", "rpgd", dict(num_rollouts=1, mpc_horizon=1)),
    ("N33_H2_two_launches", "rpgd", dict(num_rollouts=33, mpc_horizon=2, resamp_per=1)),
    ("N1024_H2", "rpgd", dict(num_rollouts=1024, mpc_horizon=2, period_interpolation_inducing_points=1)),
    ("H164_largest", "rpgd", dict(num_rollouts=40, mpc_horizon=164, outer_its=1)),
    ("period1", "rpgd", dict(period_interpolation_inducing_points=1, mpc_horizon=20)),
    ("last_inducing_point_quirk", "rpgd", dict(mpc_horizon=41, period_interpolation_inducing_points=10)),
    ("keep_k_all", "rpgd", dict(opt_keep_k_ratio=1.0, resamp_per=1)),
    ("gradient_tf_N1_H1", "gradient-tf", dict(num_rollouts=1, mpc_horizon=1)),
    ("gradient_tf_N1024", "gradient-tf", dict(num_rollouts=1024, mpc_horizon=8, gradient_steps=1)),
    ("bharadhwaj_k_all", "cem-grad-bharadhwaj-tf", dict(num_rollouts=65, cem_best_k=65, mpc_horizon=3)),
    ("naive_N1000", "cem-naive-grad-tf", dict(num_rollouts=1000, cem_best_k=7, mpc_horizon=24)),
]


@pytest.mark.parametrize("name,optimizer,over", EDGES, ids=[x[0] for x in EDGES])
def test_edge_geometries_match_oracle(name, optimizer, over):
    from oracle.replay_rng import ReplayRNG
    meta = _meta(optimizer, **over)
    ctrl = _controller(meta, seed=13)
    opt = ctrl.optimizer
    o32, _ = _oracles(meta)
    rng = ReplayRNG(13)
    if optimizer in ("rpgd", "gradient-tf"):
        o32.reset(rng)
    for t, s in enumerate(_states(4, seed=43)):
        u = ctrl.step(s)
        uo = o32.step(s, rng)
        same = _same_ranking(opt, o32, optimizer)
        e_u = float(np.max(np.abs(np.ravel(u) - np.ravel(uo))))
        _report(f"edge {name} [{opt.last_kernel}] tick {t}: u {e_u:.2e} same_ranking {same}")
        if not same:
            break
        assert e_u < 2e-4
    assert t >= 1


def test_logging_reference_layouts():
    from control_toolkit_b200 import _lib as L
    from oracle.replay_rng import ReplayRNG
    N, H = 33, 20
    meta = _meta("rpgd", num_rollouts=N, mpc_horizon=H, period_interpolation_inducing_points=5)
    ctrl = _controller(meta, logging=True, seed=17)
    opt = ctrl.optimizer
    o32, _ = _oracles(meta)
    rng = ReplayRNG(17)
    o32.reset(rng)
    for t, s in enumerate(_states(3, seed=47)):
        ctrl.step(s)
        o32.step(s, rng)
        lv = opt.logging_values
        assert lv["Q_logged"].shape == (N, H, 2) and lv["rollout_trajectories_logged"].shape == (N, H + 1, 3)
        assert lv["J_logged"].shape == (N,) and lv["trajectory_ages_logged"].shape == (N,)
        e_Q = _rel(lv["Q_logged"], o32.last["Q"])
        e_tr = _rel(lv["rollout_trajectories_logged"], o32.last["rollouts"])
        assert np.array_equal(lv["trajectory_ages_logged"], o32.last["ages"])
        _report(f"logging tick {t} [{opt.last_kernel}]: Q_logged {e_Q:.2e} rollouts {e_tr:.2e}")
        assert e_Q < 2e-4 and e_tr < 2e-4
        assert "[fused select]" not in opt.last_kernel and "env_rpgd_grad_kernel<DubinsEnv,1>" in opt.last_kernel


@pytest.mark.parametrize("optimizer", ["rpgd", "gradient-tf", "cem-grad-bharadhwaj-tf"])
def test_state_round_trip_continues_bit_identical(optimizer):
    meta = _meta(optimizer)
    a, b = _controller(meta), _controller(meta)  # in-kernel Philox: the same seed gives the same draws
    states = _states(6, seed=53)
    for s in states[:3]:
        a.step(s)
    from control_toolkit_b200 import _lib as L
    if optimizer == "rpgd":  # the plugin's own get_state / set_state (u of shape (nu,))
        st = a.optimizer.get_state()
        assert st["Q"].shape[2] == 2 and np.shape(st["u"]) == (2,)
        b.optimizer.set_state(st)
        b.optimizer._set_counter(L.COUNTER_TICK, a.optimizer._get_counter(L.COUNTER_TICK))
    else:  # the C-ABI state arrays in the reference layouts
        opt, H = a.optimizer, a.optimizer.mpc_horizon
        arrays = [(L.STATE_RPGD_Q, (opt.num_rollouts, H, 2)), (L.STATE_RPGD_M, (opt.num_rollouts, H, 2)),
                  (L.STATE_RPGD_V, (opt.num_rollouts, H, 2)), (L.STATE_U_PREV, (2,))]
        if optimizer == "cem-grad-bharadhwaj-tf":
            arrays += [(L.STATE_CEM_MU, (1, H, 2)), (L.STATE_CEM_STD, (1, H, 2))]
        for which, shape in arrays:
            b.optimizer._set_state(which, a.optimizer._get_state(which, shape))
        for c in (L.COUNTER_COUNT, L.COUNTER_ADAM_STEP, L.COUNTER_TICK):
            b.optimizer._set_counter(c, a.optimizer._get_counter(c))
        b.optimizer.count = a.optimizer.count
    for s in states[3:]:
        assert np.array_equal(a.step(s), b.step(s))
        assert np.array_equal(a.optimizer.last_costs(), b.optimizer.last_costs())


@pytest.mark.parametrize("optimizer,over", [("rpgd", {}), ("rpgd", dict(num_rollouts=100)), ("gradient-tf", {}), ("cem-naive-grad-tf", {})])
def test_device_tick_equals_host_tick(optimizer, over):
    import torch
    from control_toolkit_b200 import _lib as L
    meta = _meta(optimizer, **over)
    a, b = _controller(meta), _controller(meta)
    s = _states(2, seed=59)
    a.step(s[0])
    b.step(s[0])
    u_host = a.step(s[1])
    ob = b.optimizer
    s_dev = torch.tensor(s[1], device="cuda")
    u_dev = torch.zeros(4, device="cuda")
    torch.cuda.synchronize()
    assert L.load().ctk_step_device(ob._h, s_dev.data_ptr(), u_dev.data_ptr()) == 0
    torch.cuda.synchronize()
    assert np.array_equal(u_dev.cpu().numpy()[:2], np.ravel(u_host))
    assert np.array_equal(a.optimizer.last_costs(), ob.last_costs())
    which = L.STATE_CEM_MU if optimizer == "cem-naive-grad-tf" else L.STATE_RPGD_Q
    n = ob.mpc_horizon * 2 * (1 if optimizer == "cem-naive-grad-tf" else ob.num_rollouts)
    assert np.array_equal(a.optimizer._get_state(which, (n,)), ob._get_state(which, (n,)))


def test_optimal_trajectory_is_refused_on_the_dubins_car():
    with pytest.raises(ValueError, match="CartPole"):
        _controller(_meta("rpgd"), optimal_trajectory=True)
