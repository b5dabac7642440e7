"""Helpers for the -m gpu parity tests: build the CUDA optimizer through the reference-facing API
(control_toolkit_b200.Controllers.controller_mpc -> optimizer plugin -> C ABI) from a golden fixture's config."""
import numpy as np

from helpers import replay


def has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def make_controller(meta, logging=True, rng="replay", shard=None, weights=None, optimal_trajectory=False, **optimizer_over):
    """weights: an MLPSpec / GRUSpec registered under meta["predictor"] (default: the fixture's random_init network)."""
    import control_toolkit_b200 as ctk
    from control_toolkit_b200.Controllers.controller_mpc import controller_mpc

    if isinstance(weights, ctk.MLPSpec):
        ctk.register_mlp(meta["predictor"], weights)
    elif isinstance(weights, ctk.GRUSpec):
        ctk.register_gru(meta["predictor"], weights)
    elif meta["predictor"].startswith("Dense"):
        ctk.register_mlp(meta["predictor"], ctk.MLPSpec.random_init(meta["mlp_seed"]))
    elif meta["predictor"].startswith("GRU"):
        ctk.register_gru(meta["predictor"], ctk.GRUSpec.random_init(meta["gru_seed"]))
    cfg = dict(meta["cfg"])
    cfg.update(optimizer_over)
    if shard is not None:
        cfg["shard"] = shard
    env = meta.get("environment", "CartPole")
    nu = 2 if env == "DubinsCar" else 1
    ctrl = controller_mpc(
        environment_name=env,
        control_limits=(np.full(nu, -1.0, np.float32), np.full(nu, 1.0, np.float32)),
        initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0},
        config_controller=dict(optimizer=meta["optimizer"], predictor_specification=meta["predictor"],
                               cost_function_specification=meta["cost"], controller_logging=logging,
                               calculate_optimal_trajectory=optimal_trajectory),
        config_optimizers={meta["optimizer"]: cfg},
        config_cost_function={"cost_function_name_default": "default"},
    )
    ctrl.configure(optimizer_name=meta["optimizer"], predictor_specification=meta["predictor"])
    if rng == "replay":
        ctrl.optimizer.rng = replay(meta)
        ctrl.optimizer.rng.as_torch = False
        ctrl.optimizer.optimizer_reset()
    return ctrl


def max_rel(a, b, floor=1e-6):
    """max |a-b| / max(|b|_inf, floor): error relative to the array's scale (state vectors, controls)."""
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), floor))


def max_elem_rel(a, b, floor=1e-3):
    """max over elements of |a-b| / (|b| + floor): element-wise relative error (per-rollout costs span 1e0..1e14)."""
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))
