"""optimizer_cem_naive_grad_tf -- B200 backend behind the reference's CEM + naive gradient plugin
(reference Optimizers/optimizer_cem_naive_grad_tf.py:15-119; the class keeps the reference's name so that the
``cem-naive-grad-tf`` key of config_optimizers.yml resolves to it, although no TensorFlow is involved).

Every outer iteration: Q ~ clip(N(dist_mue, stdev)) for the whole population, ONE plain gradient-descent step on every sample
(``Q - learning_rate * clip_by_norm(dJ/dQ)``, box clip), rollout + cost of the updated samples, top-k refit of mean / population
std.  After the loop the stdev is clipped to [cem_stdev_min, 10] and both arrays shift by one step; u is the first element of the
refit MEAN (:105).  On the device: ``gradcem_sample_kernel<nu>`` -> ``rpgd_grad_kernel`` or ``env_rpgd_grad_kernel`` (forward tape +
hand-derived adjoint, plain GD form) -> ``gradcem_refit_kernel<nu>`` (bitonic argsort with ties to the lower index, elite gather,
refit, shift).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .. import _lib as L
from . import template_optimizer


class optimizer_cem_naive_grad_tf(template_optimizer):
    _OPT = L.OPT_RPGD
    _MODE = 2

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        mpc_horizon: int = 35,
        cem_outer_it: int = 1,
        num_rollouts: int = 200,
        cem_initial_action_stdev: float = 0.5,
        cem_stdev_min: float = 0.1,
        cem_best_k: int = 40,
        learning_rate: float = 0.1,
        gradmax_clip: float = 10,
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
        self.learning_rate = np.float32(learning_rate)
        self.gradmax_clip = np.float32(gradmax_clip)
        self.warmup, self.warmup_iterations = False, 1
        self.adam_beta_1, self.adam_beta_2, self.adam_epsilon = 0.9, 0.999, 1.0e-8  # unused by the plain gradient step
        self.count = 0

    def configure(self, num_states: int, num_control_inputs: int, default_configure: bool = True, **kwargs):
        # template_optimizer.configure (reference Optimizers/__init__.py:52-63); dt and predictor_specification arrive
        # through **kwargs (controller_mpc.py:84-89)
        self.num_states, self.num_control_inputs = num_states, num_control_inputs
        self._create_backend(kwargs.get("dt", None), kwargs.get("predictor_specification", None))
        self.optimizer_reset()

    def _fill_config(self, cfg: L.ctk_config) -> None:
        cfg.period_interpolation_inducing_points = 1
        cfg.rpgd_gradient_mode = self._MODE
        cfg.rpgd_keep_k = self.num_rollouts
        cfg.rpgd_outer_its = 1
        cfg.rpgd_first_iter_count = 1
        cfg.rpgd_resamp_per = 1
        cfg.rpgd_shift_previous = 1
        cfg.rpgd_distribution = L.DIST_NORMAL
        cfg.rpgd_adam_form = L.ADAM_KERAS
        cfg.rpgd_sample_mean, cfg.rpgd_sample_stdev = 0.0, 1.0
        cfg.rpgd_sample_min, cfg.rpgd_sample_max = float(self.action_low[0]), float(self.action_high[0])
        cfg.rpgd_learning_rate = float(np.float32(self.learning_rate))
        cfg.rpgd_gradmax_clip = float(self.gradmax_clip)
        cfg.rpgd_beta_1, cfg.rpgd_beta_2, cfg.rpgd_epsilon = float(self.adam_beta_1), float(self.adam_beta_2), float(self.adam_epsilon)
        cfg.cem_outer_it = self.cem_outer_it
        cfg.cem_best_k = self.cem_best_k
        cfg.cem_initial_action_stdev = float(np.float32(self.cem_initial_action_stdev))
        cfg.cem_stdev_min = float(np.float32(self.cem_stdev_min))
        cfg.cem_warmup = int(self.warmup)
        cfg.cem_warmup_iterations = self.warmup_iterations

    def _iterations(self) -> int:
        return self.cem_outer_it

    def _noise_blocks(self, iterations):
        N, H, nu = self.num_rollouts, self.mpc_horizon, self.num_control_inputs
        return [("normal", (N, H, nu))] * iterations  # :61-62, one population per outer iteration

    def step(self, s: np.ndarray, time=None):
        lib = self._require_backend()
        if self.optimizer_logging:
            self.logging_values = {"s_logged": np.asarray(s).copy()}
        self._refresh_live_cost(lib)
        iterations = self._iterations()
        self._feed_noise(lib, self._noise_blocks(iterations))
        u = self._tick(lib, s)
        self.u = np.squeeze(u)  # :105 / bharadhwaj :168
        N, H, nu = self.num_rollouts, self.mpc_horizon, self.num_control_inputs
        if self.optimizer_logging:
            self.logging_values["Q_logged"] = self._get_log(L.LOG_Q, (N, H, nu))
            self.logging_values["J_logged"] = self._get_log(L.LOG_J, (N,))
            self.logging_values["rollout_trajectories_logged"] = self._get_log(L.LOG_ROLLOUTS, (N, H + 1, int(self.num_states)))
            self.logging_values["u_logged"] = self.u
        self._last_iterations = iterations
        self.count += 1
        return self.u

    def optimizer_reset(self):
        lib = self._require_backend()
        L.check(lib.ctk_reset(self._h))
        self.count = 0
        # self.u (the cost's previous_input) survives optimizer_reset() in the reference: only optimizer_cem_tf.py:117 resets it

    # reference attributes, read from the device on demand
    @property
    def dist_mue(self) -> np.ndarray:
        return self._get_state(L.STATE_CEM_MU, (1, self.mpc_horizon, self.num_control_inputs))

    @property
    def stdev(self) -> np.ndarray:
        return self._get_state(L.STATE_CEM_STD, (1, self.mpc_horizon, self.num_control_inputs))

    def elite_indices(self) -> np.ndarray:
        """[outer iterations of the last tick, cem_best_k] population indices, best first."""
        return self._get_log(L.LOG_ELITE_IDX, (self._last_iterations, self.cem_best_k), np.int32)

    def last_costs(self) -> np.ndarray:
        return self._get_log(L.LOG_J, (self.num_rollouts,))
