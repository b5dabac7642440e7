"""optimizer_gradient_tf -- B200 backend behind the reference's population gradient-descent plugin
(reference Optimizers/optimizer_gradient_tf.py:12-185; the class keeps the reference's name so that the ``gradient-tf`` key of
config_optimizers.yml resolves to it, although no TensorFlow is involved).

Every tick: ``gradient_steps`` (first tick: ``warmup_iterations`` if ``warmup``) Adam steps on the whole population through
the rollout (per-trajectory ``clip_by_norm``, Keras Adam, box clip), one more rollout for the costs, u = first control of the
cheapest sequence; then every sequence and both Adam moments shift by one step, the vacated last control is redrawn from
U[action_low, action_high) and the moments are zero-filled.  On the device this is the RPGD machinery
(``rpgd_grad_kernel`` or ``env_rpgd_grad_kernel`` + ``rpgd_select_kernel<nu>``) with inducing-point period 1, no ranking-based
resampling and the tail redraw (ctk_config.rpgd_gradient_mode).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .. import _lib as L
from . import template_optimizer


class optimizer_gradient_tf(template_optimizer):
    _OPT = L.OPT_RPGD

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        mpc_horizon: int = 35,
        gradient_steps: int = 5,
        num_rollouts: int = 40,
        initial_action_stdev: float = 0.5,
        learning_rate: float = 0.05,
        adam_beta_1: float = 0.9,
        adam_beta_2: float = 0.999,
        adam_epsilon: float = 1.0e-07,
        gradmax_clip: float = 5,
        rtol: float = 1.0e-3,
        warmup: bool = False,
        warmup_iterations: int = 250,
        optimizer_logging: bool = False,
        calculate_optimal_trajectory: bool = False,
        **kwargs,
    ):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         optimizer_logging=optimizer_logging, seed=seed, num_rollouts=num_rollouts,
                         mpc_horizon=mpc_horizon, computation_library=computation_library, **kwargs)
        self.gradient_steps = int(gradient_steps)
        self.initial_action_stdev = initial_action_stdev  # stored, never used by the reference either (:52)
        self.learning_rate, self.adam_beta_1, self.adam_beta_2, self.adam_epsilon = learning_rate, adam_beta_1, adam_beta_2, adam_epsilon
        self.gradmax_clip = np.float32(gradmax_clip)
        self.rtol = rtol
        self.warmup = bool(warmup)
        self.warmup_iterations = int(warmup_iterations)
        self.first_iter_count = self.warmup_iterations if self.warmup else self.gradient_steps  # :66-68
        self.count = 0

    def configure(self, num_states: int, num_control_inputs: int, default_configure: bool = True, **kwargs):
        # template_optimizer.configure (reference Optimizers/__init__.py:52-63); dt and predictor_specification arrive
        # through **kwargs (controller_mpc.py:84-89)
        self.num_states, self.num_control_inputs = num_states, num_control_inputs
        self._create_backend(kwargs.get("dt", None), kwargs.get("predictor_specification", None))
        if default_configure:
            self.optimizer_reset()

    def _fill_config(self, cfg: L.ctk_config) -> None:
        cfg.period_interpolation_inducing_points = 1  # every control is its own inducing point (:171-177 samples [N,H,nu])
        cfg.rpgd_gradient_mode = 1
        cfg.rpgd_outer_its = self.gradient_steps
        cfg.rpgd_first_iter_count = self.first_iter_count
        cfg.rpgd_resamp_per = 1
        cfg.rpgd_shift_previous = 1
        cfg.rpgd_keep_k = self.num_rollouts
        cfg.rpgd_distribution = L.DIST_UNIFORM
        cfg.rpgd_adam_form = L.ADAM_KERAS  # tf.keras.optimizers.Adam (:55-60)
        cfg.rpgd_sample_mean, cfg.rpgd_sample_stdev = 0.0, 1.0
        cfg.rpgd_sample_min, cfg.rpgd_sample_max = float(self.action_low[0]), float(self.action_high[0])
        cfg.rpgd_learning_rate = float(np.float32(self.learning_rate))
        cfg.rpgd_gradmax_clip = float(self.gradmax_clip)
        cfg.rpgd_beta_1, cfg.rpgd_beta_2, cfg.rpgd_epsilon = float(self.adam_beta_1), float(self.adam_beta_2), float(self.adam_epsilon)

    def step(self, s: np.ndarray, time=None):
        lib = self._require_backend()
        if self.optimizer_logging:
            self.logging_values = {"s_logged": np.asarray(s).copy()}
        self._refresh_live_cost(lib)
        N, H, nu = self.num_rollouts, self.mpc_horizon, self.num_control_inputs
        self._feed_noise(lib, [("uniform", (N, 1, nu))])  # the tail redraw of this tick (:142-147)
        u = self._tick(lib, s)
        self.u = np.squeeze(u)  # :132
        if self.optimizer_logging:
            self.logging_values["Q_logged"] = self._get_log(L.LOG_Q, (N, H, nu))
            self.logging_values["J_logged"] = self._get_log(L.LOG_J, (N,))
            self.logging_values["rollout_trajectories_logged"] = self._get_log(L.LOG_ROLLOUTS, (N, H + 1, int(self.num_states)))
            self.logging_values["u_logged"] = self.u
        self.count += 1  # :141
        return self.u

    def optimizer_reset(self):
        lib = self._require_backend()
        self._feed_noise(lib, [("uniform", (self.num_rollouts, self.mpc_horizon, self.num_control_inputs))])  # :171-176
        L.check(lib.ctk_reset(self._h))
        self.count = 0
        # self.u (the cost's previous_input) survives optimizer_reset() in the reference: only optimizer_cem_tf.py:117 resets it

    # reference attributes, read from the device on demand
    @property
    def Q_tf(self) -> np.ndarray:
        return self._get_state(L.STATE_RPGD_Q, (self.num_rollouts, self.mpc_horizon, self.num_control_inputs))

    def adam_weights(self):
        """[iterations, m, v] like ``self.optim.get_weights()`` (:151)."""
        shape = (self.num_rollouts, self.mpc_horizon, self.num_control_inputs)
        return [self._get_counter(L.COUNTER_ADAM_STEP), self._get_state(L.STATE_RPGD_M, shape), self._get_state(L.STATE_RPGD_V, shape)]

    def best_index(self) -> int:
        return int(self._get_log(L.LOG_ELITE_IDX, (self.num_rollouts,), np.int32)[0])

    def last_costs(self) -> np.ndarray:
        return self._get_log(L.LOG_J, (self.num_rollouts,))
