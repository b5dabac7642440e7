"""CPU tests of the host-side logic of the plugin layer: registry / naming / config plumbing, parameter derivation
(independently written in control_toolkit_b200/specs.py and oracle/spec.py), shard geometry."""
import math
import os

import numpy as np
import pytest

from oracle import spec as ospec
from oracle.refharness.workspace import REFERENCE, reference_has

TEMPLATE_YAML = os.path.join("Control_Toolkit_ASF_Template", "config_optimizers.yml")


def test_ode_and_cost_constants_agree_with_oracle_spec():
    from control_toolkit_b200 import specs
    c = specs.CartPoleODE().to_c(0.02)
    o = ospec.CartPoleParams(dt=0.02).f32()
    for k, v in o.items():
        assert float(getattr(c, k)) == v, k
    for name in ("default", "quadratic_boundary_grad"):
        cc = specs.resolve_cost("CartPole", name).to_c(0.05, 1.0)
        oc = ospec.CostParams(name=name, target_position=0.05).f32()
        for k, v in oc.items():
            assert float(getattr(cc, k)) == v, (name, k)


def test_registry_fails_loudly_for_unregistered_names():
    from control_toolkit_b200 import specs
    with pytest.raises(ValueError, match="no registered CUDA functor"):
        specs.resolve_cost("CartPole", "quadratic_boundary_nonconvex")
    with pytest.raises(ValueError):
        specs.resolve_cost("Pendulum", "default")
    with pytest.raises(ValueError):
        specs.resolve_predictor("CartPole", "LSTM-6IN-32H1-32H2-5OUT-0")
    assert specs.resolve_cost("CartPole", "quadratic-boundary-grad").kind == 1  # '-' <-> '_' like the reference


def test_optimizer_discovery_by_name():
    """reference others/globals_and_utils.py:103-133: 'cem-tf' -> file optimizer_cem_tf.py, class optimizer_cem_tf."""
    import control_toolkit_b200 as ctk
    for key, cls in (("mppi", "optimizer_mppi"), ("cem-tf", "optimizer_cem_tf"), ("rpgd", "optimizer_rpgd"),
                     ("random-action-tf", "optimizer_random_action_tf"), ("gradient-tf", "optimizer_gradient_tf"),
                     ("cem-naive-grad-tf", "optimizer_cem_naive_grad_tf"), ("cem-grad-bharadhwaj-tf", "optimizer_cem_grad_bharadhwaj_tf")):
        C = ctk.import_optimizer_by_name(key)
        assert C.__name__ == cls
        assert "template_optimizer" in [b.__name__ for b in C.__mro__[1:]]
    with pytest.raises(ValueError, match="not found"):
        ctk.import_optimizer_by_name("rpgd-tf")  # the stale template key (SURVEY.md section 2 row 11)


def test_optimizer_constructor_contract():
    """Same ctor kwargs as the reference (mpc_timestep arrives through **kwargs), optimizer_name property, u init."""
    import control_toolkit_b200 as ctk
    lim = (np.array([-1.0]), np.array([1.0]))
    M = ctk.import_optimizer_by_name("mppi")
    o = M(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, computation_library=None,
          seed=None, cc_weight=1.0, R=1.0, LBD=100.0, mpc_horizon=35, num_rollouts=3500, NU=1000.0, SQRTRHOINV=0.03,
          period_interpolation_inducing_points=10, optimizer_logging=False, calculate_optimal_trajectory=False, mpc_timestep=0.02)
    assert o.optimizer_name == "mppi" and o.u == 0.0 and o.num_rollouts == 3500 and o.mpc_horizon == 35
    assert isinstance(o.seed, int)  # seed None -> datetime seed (reference globals_and_utils.py:87-91)
    with pytest.raises(RuntimeError, match="configure"):
        o.step(np.zeros(6))
    R = ctk.import_optimizer_by_name("rpgd")
    with pytest.raises(ValueError, match="sampling type"):
        R(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, SAMPLING_DISTRIBUTION="cauchy")
    r = R(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, num_rollouts=32,
          opt_keep_k_ratio=0.25, warmup=True, warmup_iterations=7, outer_its=2)
    assert r.opt_keep_k == 8 and r.first_iter_count == 7 and r.optimizer_name == "rpgd"
    with pytest.raises(ValueError, match="dt and predictor_specification"):
        r.configure(num_states=6, num_control_inputs=1)
    # the sibling optimizers: the reference's ctor kwargs (template blocks of config_optimizers.yml:23-61) and warm-up rules
    G = ctk.import_optimizer_by_name("gradient-tf")
    g = G(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, computation_library=None, seed=1,
          mpc_horizon=35, gradient_steps=5, num_rollouts=40, initial_action_stdev=0.5, learning_rate=0.05, adam_beta_1=0.9,
          adam_beta_2=0.999, adam_epsilon=1.0e-07, gradmax_clip=5, rtol=1.0e-3, warmup=True, warmup_iterations=250,
          optimizer_logging=False, calculate_optimal_trajectory=False, mpc_timestep=0.02)
    assert g.first_iter_count == 250 and g.optimizer_name == "gradient-tf"  # optimizer_gradient_tf.py:66-68
    B = ctk.import_optimizer_by_name("cem-grad-bharadhwaj-tf")
    b = B(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, computation_library=None, seed=1,
          mpc_horizon=50, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1.0e-08, num_rollouts=32, cem_best_k=8,
          cem_outer_it=2, cem_initial_action_stdev=2, cem_stdev_min=1.e-6, gradmax_clip=5, warmup=True, warmup_iterations=9,
          optimizer_logging=False, calculate_optimal_trajectory=False, mpc_timestep=0.02)
    assert b._iterations() == 9 and b.optimizer_name == "cem-grad-bharadhwaj-tf"  # optimizer_cem_grad_bharadhwaj_tf.py:162
    assert [blk[1][0] for blk in b._noise_blocks(2)] == [8, 24, 24]  # :159 k "elites", then N - k fresh samples per iteration (:95)
    Nv = ctk.import_optimizer_by_name("cem-naive-grad-tf")
    nv = Nv(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=lim, computation_library=None, seed=1,
            mpc_horizon=35, cem_outer_it=1, num_rollouts=200, cem_stdev_min=0.1, cem_initial_action_stdev=0.5, cem_best_k=40,
            learning_rate=0.1, gradmax_clip=10, optimizer_logging=False, calculate_optimal_trajectory=False, mpc_timestep=0.02)
    assert nv._iterations() == 1 and nv.optimizer_name == "cem-naive-grad-tf"
    for o2 in (g, b, nv):
        with pytest.raises(RuntimeError, match="configure"):
            o2.step(np.zeros(6))


def test_mppi_host_constants_follow_reference_evaluation_order():
    """optimizer_mppi.py:130,154-155,165: fp32 coefficients as the reference's fp32 tensor ops produce them."""
    import torch
    import control_toolkit_b200 as ctk
    from control_toolkit_b200 import _lib as L
    M = ctk.import_optimizer_by_name("mppi")
    o = M(predictor=ctk.PredictorWrapper(), cost_function=ctk.CostFunctionWrapper(), control_limits=(np.array([-1.0]), np.array([1.0])),
          NU=1000.0, R=1.3, LBD=37.0, SQRTRHOINV=0.03, cc_weight=0.7)
    o.SQRTRHODTINV = np.float32(np.array(0.03) * (1 / np.sqrt(0.02)))
    cfg = L.ctk_config()
    o._fill_config(cfg)
    NU, R = torch.tensor(1000.0), torch.tensor(1.3)
    assert cfg.mppi_coef_du2 == float(0.5 * (1 - 1.0 / NU) * R)
    assert cfg.mppi_half_R == float(0.5 * R)
    assert cfg.mppi_neg_inv_LBD == float(torch.tensor(-1.0 / 37.0, dtype=torch.float32))
    assert cfg.mppi_stdev == float(torch.tensor(np.array(0.03) * (1 / np.sqrt(0.02)), dtype=torch.float32))


def test_shard_geometry_partitions_the_population():
    from control_toolkit_b200.distributed import shard_geometry
    for n in (1, 7, 2000, 4096, 1_000_000, 1_000_003):
        for w in (1, 2, 3, 4, 8):
            parts = [shard_geometry(n, r, w) for r in range(w)]
            assert parts[0][0] == 0
            assert sum(c for _, c in parts) == n
            for (o0, c0), (o1, _) in zip(parts, parts[1:]):
                assert o0 + c0 == o1
            assert max(c for _, c in parts) - min(c for _, c in parts) <= 1


def test_interpolation_inducing_point_count():
    """reference others/Interpolator.py:79-84"""
    for H, p, n in ((50, 10, 6), (100, 10, 11), (43, 10, 6), (20, 1, 20), (35, 10, 5), (41, 10, 5), (1, 10, 1)):
        assert int(math.ceil((H - 1) / p) + 1) == n


def test_environment_registry_second_environment_and_recurrent_predictor():
    """SURVEY 8f.3: the functor registry knows a second environment (Dubins car: 3 states, 2 control inputs) and a recurrent predictor;
    the product-side specs (control_toolkit_b200.specs) and the oracle's (oracle/spec.py) are written independently and must agree;
    anything unregistered raises instead of falling back."""
    import pytest
    from control_toolkit_b200 import specs
    from oracle import spec as ospec
    info = specs.environment_info("DubinsCar")
    assert (info.num_states, info.num_control_inputs) == (ospec.DUBINS_NUM_STATES, ospec.DUBINS_NUM_CONTROLS) == (3, 2)
    with pytest.raises(ValueError):
        specs.environment_info("Acrobot")
    with pytest.raises(ValueError):
        specs.resolve_cost("DubinsCar", "quadratic_boundary_grad")  # registered for the CartPole only
    kind, ode = specs.resolve_predictor("DubinsCar", "ODE")
    cost = specs.resolve_cost("DubinsCar", "default", {"dd_weight": 12.0, "unknown_key": 1.0})
    assert cost.dd_weight == 12.0
    p = specs.dubins_env_params(ode, specs.resolve_cost("DubinsCar", "default"), 0.02)
    oc, od = ospec.DubinsCost().f32(), ospec.DubinsParams(dt=0.02).f32()
    expect = [od["h"], od["v_max"], od["omega_max"], oc["dd_weight"], oc["obstacle_weight"], np.float32(oc["cc_weight"]) * np.float32(oc["R"]),
              oc["ccrc_weight"], oc["terminal_weight"], oc["target_x"], oc["target_y"], oc["obstacle_x"], oc["obstacle_y"], oc["obstacle_r2"], oc["MAX_COST"]]
    np.testing.assert_array_equal(p, np.array(expect, np.float32))
    # recurrent predictor: same draws, same order, same scaling on both sides
    a, b = specs.GRUSpec.random_init(3), ospec.GRUWeights.random_init(3)
    for k in ("Wi1", "Wh1", "bi1", "bh1", "Wi2", "Wh2", "bi2", "bh2", "W3", "b3"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
    specs.register_gru("GRU-6IN-32H1-32H2-5OUT-0", a)
    from control_toolkit_b200 import _lib as L
    assert specs.resolve_predictor("CartPole", "GRU-6IN-32H1-32H2-5OUT-0")[0] == L.PRED_GRU
    with pytest.raises(ValueError):
        specs.GRUSpec(**{**{k: getattr(a, k) for k in a._KEYS}, "W3": np.zeros((32, 4), np.float32)})


@pytest.mark.skipif(not reference_has(TEMPLATE_YAML), reason="needs a Control_Toolkit checkout: set CTK_REFERENCE to its path")
@pytest.mark.parametrize("key", ["mppi", "cem-tf", "random-action-tf", "gradient-tf", "cem-naive-grad-tf", "cem-grad-bharadhwaj-tf"])
def test_reference_template_yaml_blocks_feed_the_plugins_unchanged(key):
    """The reference's OWN template blocks (Control_Toolkit_ASF_Template/config_optimizers.yml) go into the plugin constructors exactly as
    controller_mpc passes them (**config_optimizer, Controllers/controller_mpc.py:56-65) -- every key accepted, values arrive -- and
    configure() gets as far as ctk_create (no GPU here: BackendUnavailable, the first thing that can fail).  Only mpc_timestep is added:
    the reference reads config_optimizer["mpc_timestep"] (:68,85) but its template blocks do not carry the key (an application adds it).
    ('rpgd' has no usable template block: 'rpgd-tf' is a stale key without the constructor's sample_mean / uniform_dist_* arguments.)"""
    import yaml
    import control_toolkit_b200 as ctk
    from control_toolkit_b200._lib import BackendUnavailable
    from control_toolkit_b200.Controllers.controller_mpc import controller_mpc
    with open(os.path.join(REFERENCE, TEMPLATE_YAML)) as f:
        block = dict(yaml.safe_load(f)[key])
    block["mpc_timestep"] = 0.02
    predictor = "ODE"
    ctrl = controller_mpc(
        environment_name="CartPole", control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)),
        initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0},
        config_controller=dict(optimizer=key, predictor_specification=predictor, cost_function_specification="default",
                               controller_logging=False, calculate_optimal_trajectory=False),
        config_optimizers={key: block}, config_cost_function={"cost_function_name_default": "default"})
    try:
        ctrl.configure(optimizer_name=key, predictor_specification=predictor)
    except BackendUnavailable:
        pass  # no CUDA device: everything above ctk_create has run
    opt = ctrl.optimizer
    assert type(opt).__name__ == "optimizer_" + key.replace("-", "_") and opt.optimizer_name == key
    assert (opt.num_rollouts, opt.mpc_horizon) == (int(block["num_rollouts"]), int(block["mpc_horizon"]))
    for k, v in block.items():  # constructor arguments the plugin keeps under the reference's attribute names
        if hasattr(opt, k) and isinstance(v, (int, float)) and not isinstance(v, bool) and k != "seed":
            assert float(getattr(opt, k)) == pytest.approx(float(v)), k
