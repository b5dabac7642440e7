"""optimizer_cem_tf -- B200 backend behind the reference's CEM plugin interface
(reference Optimizers/optimizer_cem_tf.py:13-117; the class keeps the reference's name so that the
``cem-tf`` key of config_optimizers.yml resolves to it, although no TensorFlow is involved).

Per outer iteration: fused sample -> rollout -> cost kernel, bitonic top-k of (cost, index) keys (ties -> lower
index, tf.argsort semantics), elite refit with the elite rows REGENERATED from the counter-based noise (never stored).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .. import _lib as L
from . import template_optimizer


class optimizer_cem_tf(template_optimizer):
    _OPT = L.OPT_CEM

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        mpc_horizon: int = 40,
        cem_outer_it: int = 3,
        cem_initial_action_stdev: float = 0.5,
        num_rollouts: int = 200,
        cem_stdev_min: float = 0.01,
        cem_best_k: int = 40,
        warmup: bool = False,
        warmup_iterations: int = 250,
        optimizer_logging: bool = False,
        calculate_optimal_trajectory: bool = False,
        **kwargs,
    ):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         optimizer_logging=optimizer_logging, seed=seed, num_rollouts=num_rollouts,
                         mpc_horizon=mpc_horizon, computation_library=computation_library, **kwargs)
        self.cem_outer_it = int(cem_outer_it)
        self.cem_initial_action_stdev = cem_initial_action_stdev
        self.cem_stdev_min = cem_stdev_min
        self.cem_best_k = int(cem_best_k)
        self.warmup = bool(warmup)
        self.warmup_iterations = int(warmup_iterations)
        self.count = 0
        self.elite_indices = None

    def configure(self, num_states: int, num_control_inputs: int, default_configure: bool = True, **kwargs):
        # the reference's CEM relies on template_optimizer.configure (Optimizers/__init__.py:52-63); dt and
        # predictor_specification arrive through **kwargs (controller_mpc.py:84-89)
        self.num_states, self.num_control_inputs = num_states, num_control_inputs
        dt = kwargs.get("dt", None)
        predictor_specification = kwargs.get("predictor_specification", None)
        self._create_backend(dt, predictor_specification)
        if default_configure:
            self.optimizer_reset()

    def _fill_config(self, cfg: L.ctk_config) -> None:
        cfg.cem_outer_it = self.cem_outer_it
        cfg.cem_best_k = self.cem_best_k
        cfg.cem_warmup = int(self.warmup)
        cfg.cem_warmup_iterations = self.warmup_iterations
        cfg.cem_initial_action_stdev = float(np.float32(self.cem_initial_action_stdev))
        cfg.cem_stdev_min = float(np.float32(self.cem_stdev_min))

    def step(self, s: np.ndarray, time=None):
        lib = self._require_backend()
        if self.optimizer_logging:
            self.logging_values = {"s_logged": np.asarray(s).copy()}
        self._refresh_live_cost(lib)
        iterations = self.warmup_iterations if self.warmup and self.count == 0 else self.cem_outer_it  # :92
        self._feed_noise(lib, [("normal", (self.num_rollouts, self.mpc_horizon, self.num_control_inputs))] * iterations)
        u = self._tick(lib, s)
        self.u = np.squeeze(u)  # :101
        H, nu, N = self.mpc_horizon, self.num_control_inputs, self._n_local
        if self.optimizer_logging:
            self._collect_rollout_logs(N)
            self.logging_values["u_logged"] = self.u
            self.elite_indices = self._get_log(L.LOG_ELITE_IDX, (iterations, self.cem_best_k), np.int32)
        self.count += 1  # :110
        return self.u

    def optimizer_reset(self):
        lib = self._require_backend()
        L.check(lib.ctk_reset(self._h))
        self.count = 0
        self.u = 0.0

    # reference attributes dist_mue / stdev [1,H,nu] (:113-117), read from the device on demand
    @property
    def dist_mue(self) -> np.ndarray:
        return self._get_state(L.STATE_CEM_MU, (1, self.mpc_horizon, int(self.num_control_inputs)))

    @property
    def stdev(self) -> np.ndarray:
        return self._get_state(L.STATE_CEM_STD, (1, self.mpc_horizon, int(self.num_control_inputs)))

    def last_costs(self) -> np.ndarray:
        return self._get_log(L.LOG_J, (self._n_local,))

    def last_elite_indices(self, iterations: int) -> np.ndarray:
        return self._get_log(L.LOG_ELITE_IDX, (iterations, self.cem_best_k), np.int32)

    # dist_mue / stdev [1, H, nu]; u: a float for nu == 1, (nu,) otherwise (the shape step() returns)
    def get_state(self) -> dict:
        nu = int(self.num_control_inputs)
        u = self._get_state(L.STATE_U_PREV, (nu,))
        return {"dist_mue": self.dist_mue, "stdev": self.stdev, "count": self.count, "u": float(u[0]) if nu == 1 else u}

    def set_state(self, state: dict) -> None:
        self._set_state(L.STATE_CEM_MU, state["dist_mue"])
        self._set_state(L.STATE_CEM_STD, state["stdev"])
        self._set_state(L.STATE_U_PREV, np.reshape(state["u"], (int(self.num_control_inputs),)))
        self.count = int(state["count"])
        self._set_counter(L.COUNTER_COUNT, self.count)
