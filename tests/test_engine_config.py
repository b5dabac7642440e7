"""ctk_create refuses a configuration that cannot run with CTK_EINVAL and its message before it touches the device, so the
same answer comes back on a machine without a GPU (where a valid configuration fails at the device query)."""
import ctypes as C

import pytest

from control_toolkit_b200 import _lib as L

PERIOD = "period_interpolation_inducing_points must be >= 1"
CEM = "CEM needs 1 <= cem_best_k <= min(512, num_rollouts), mpc_horizon <= 1024, cem_outer_it >= 1"
RPGD = ("RPGD needs num_rollouts <= 1024 (replicas only, no sharding), the ODE predictor with intermediate_steps == 1 and "
        "1 <= keep_k <= num_rollouts")
GRADCEM = "gradient-assisted CEM needs 1 <= cem_best_k <= num_rollouts, cem_outer_it >= 1 and inducing-point period 1"
ENV_MPPI = "environment MPPI: n_ind * nu <= 32 and H * nu <= 1024"
ENV_CEM = "environment CEM needs 1 <= cem_best_k <= min(512, num_rollouts), H * nu <= 1024, cem_outer_it >= 1"


def _create(optimizer, ode_over=None, **over):
    cfg, ode, cost = L.ctk_config(), L.ctk_ode_params(), L.ctk_cost_params()
    cfg.abi_version, cfg.optimizer, cfg.predictor, cfg.device = L.CTK_ABI_VERSION, optimizer, L.PRED_ODE, 0
    cfg.num_rollouts = cfg.num_rollouts_global = 64
    cfg.mpc_horizon, cfg.num_states, cfg.num_control_inputs = 20, 6, 1
    cfg.action_low, cfg.action_high = -1.0, 1.0
    cfg.period_interpolation_inducing_points = 1
    cfg.cem_outer_it, cfg.cem_best_k, cfg.cem_initial_action_stdev = 1, 8, 0.5
    cfg.rpgd_outer_its, cfg.rpgd_resamp_per, cfg.rpgd_keep_k = 1, 1, 4
    cfg.environment = L.ENV_CARTPOLE
    for k, v in over.items():
        setattr(cfg, k, v)
    ode.intermediate_steps = 1
    for k, v in (ode_over or {}).items():
        setattr(ode, k, v)
    cost.kind = L.COST_DEFAULT
    h = C.c_void_p()
    rc = L.load().ctk_create(C.byref(cfg), C.byref(ode), C.byref(cost), C.byref(h))
    if rc == L.CTK_OK:  # a machine with a GPU accepted it
        L.load().ctk_destroy(h)
    return rc, (L.load().ctk_last_error() or b"").decode()


DUBINS = dict(environment=L.ENV_DUBINS_CAR, num_states=3, num_control_inputs=2)

CASES = [
    ("mppi_period_0", L.OPT_MPPI, None, dict(period_interpolation_inducing_points=0), PERIOD),
    ("rpgd_period_0", L.OPT_RPGD, None, dict(period_interpolation_inducing_points=0), PERIOD),
    ("cem_best_k_0", L.OPT_CEM, None, dict(cem_best_k=0), CEM),
    ("cem_best_k_over_512", L.OPT_CEM, None, dict(num_rollouts=1024, num_rollouts_global=1024, cem_best_k=513), CEM),
    ("cem_best_k_over_population", L.OPT_CEM, None, dict(cem_best_k=65), CEM),
    ("cem_horizon_over_1024", L.OPT_CEM, None, dict(mpc_horizon=1025), CEM),
    ("cem_outer_it_0", L.OPT_CEM, None, dict(cem_outer_it=0), CEM),
    ("rpgd_over_1024_rollouts", L.OPT_RPGD, None, dict(num_rollouts=5000, num_rollouts_global=5000), RPGD),
    ("rpgd_keep_k_0", L.OPT_RPGD, None, dict(rpgd_keep_k=0), RPGD),
    ("rpgd_keep_k_over_population", L.OPT_RPGD, None, dict(rpgd_keep_k=65), RPGD),
    ("rpgd_sharded", L.OPT_RPGD, None, dict(num_rollouts=32, num_rollouts_global=64), RPGD),
    ("rpgd_mlp_predictor", L.OPT_RPGD, None, dict(predictor=L.PRED_MLP), RPGD),
    ("rpgd_intermediate_steps_2", L.OPT_RPGD, dict(intermediate_steps=2), {}, RPGD),
    ("rpgd_negative_shift", L.OPT_RPGD, None, dict(rpgd_shift_previous=-1), RPGD),
    ("gradcem_mode_4", L.OPT_RPGD, None, dict(rpgd_gradient_mode=4), GRADCEM),
    ("gradcem_best_k_0", L.OPT_RPGD, None, dict(rpgd_gradient_mode=2, cem_best_k=0), GRADCEM),
    ("gradcem_best_k_over_population", L.OPT_RPGD, None, dict(rpgd_gradient_mode=3, cem_best_k=65), GRADCEM),
    ("gradcem_outer_it_0", L.OPT_RPGD, None, dict(rpgd_gradient_mode=2, cem_outer_it=0), GRADCEM),
    ("gradcem_period_2", L.OPT_RPGD, None, dict(rpgd_gradient_mode=3, period_interpolation_inducing_points=2), GRADCEM),
    ("dubins_mppi_inducing_points", L.OPT_MPPI, None, dict(DUBINS, mpc_horizon=20), ENV_MPPI),  # n_ind 20 x nu 2 > 32
    ("dubins_mppi_horizon", L.OPT_MPPI, None, dict(DUBINS, mpc_horizon=600, period_interpolation_inducing_points=100), ENV_MPPI),
    ("dubins_cem_best_k_0", L.OPT_CEM, None, dict(DUBINS, cem_best_k=0), ENV_CEM),
    ("dubins_cem_best_k_over_population", L.OPT_CEM, None, dict(DUBINS, cem_best_k=65), ENV_CEM),
    ("dubins_cem_horizon", L.OPT_CEM, None, dict(DUBINS, mpc_horizon=513), ENV_CEM),
    ("dubins_cem_outer_it_0", L.OPT_CEM, None, dict(DUBINS, cem_outer_it=0), ENV_CEM),
]


@pytest.mark.parametrize("optimizer,ode_over,over,message", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_create_rejects_before_the_device(optimizer, ode_over, over, message):
    rc, err = _create(optimizer, ode_over, **over)
    assert rc == L.CTK_EINVAL, err
    assert message in err
