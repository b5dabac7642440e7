"""optimizer_cem_grad_bharadhwaj_tf -- B200 backend behind the reference's CEM + Adam plugin after Bharadhwaj et al. 2020
(reference Optimizers/optimizer_cem_grad_bharadhwaj_tf.py:17-184; the class keeps the reference's name so that the
``cem-grad-bharadhwaj-tf`` key of config_optimizers.yml resolves to it, although no TensorFlow is involved).

Every tick starts from ``cem_best_k`` samples of the current distribution as "elites" (:159).  Every outer iteration: the elites are
kept, ``num_rollouts - cem_best_k`` fresh samples are appended, the whole population takes ONE Keras-Adam step on the
norm-clipped gradient (the Adam moments belong to the population ROWS and persist across iterations, ticks and
``optimizer_reset``), box clip, rollout + cost, top-k -> new elites and refit of mean / population std.  u is the first control
of the best sample (:168).  Device path: see optimizer_cem_naive_grad_tf (same kernels, Keras-Adam form, elites carried in the
double-buffered population).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .. import _lib as L
from .optimizer_cem_naive_grad_tf import optimizer_cem_naive_grad_tf


class optimizer_cem_grad_bharadhwaj_tf(optimizer_cem_naive_grad_tf):
    _MODE = 3

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        mpc_horizon: int = 50,
        cem_outer_it: int = 2,
        num_rollouts: int = 32,
        cem_initial_action_stdev: float = 2,
        cem_stdev_min: float = 1.0e-6,
        cem_best_k: int = 8,
        learning_rate: float = 0.05,
        adam_beta_1: float = 0.9,
        adam_beta_2: float = 0.999,
        adam_epsilon: float = 1.0e-8,
        gradmax_clip: float = 5,
        warmup: bool = False,
        warmup_iterations: int = 250,
        optimizer_logging: bool = False,
        calculate_optimal_trajectory: bool = False,
        **kwargs,
    ):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         computation_library=computation_library, seed=seed, mpc_horizon=mpc_horizon, cem_outer_it=cem_outer_it,
                         num_rollouts=num_rollouts, cem_initial_action_stdev=cem_initial_action_stdev, cem_stdev_min=cem_stdev_min,
                         cem_best_k=cem_best_k, learning_rate=learning_rate, gradmax_clip=gradmax_clip,
                         optimizer_logging=optimizer_logging, calculate_optimal_trajectory=calculate_optimal_trajectory, **kwargs)
        self.adam_beta_1, self.adam_beta_2, self.adam_epsilon = adam_beta_1, adam_beta_2, adam_epsilon
        self.warmup = bool(warmup)
        self.warmup_iterations = int(warmup_iterations)

    def _iterations(self) -> int:
        return self.warmup_iterations if self.warmup and self.count == 0 else self.cem_outer_it  # :162

    def _noise_blocks(self, iterations):
        N, H, nu, k = self.num_rollouts, self.mpc_horizon, self.num_control_inputs, self.cem_best_k
        blocks = [("normal", (k, H, nu))]  # :159 the tick's first "elites"
        if N - k > 0:
            blocks += [("normal", (N - k, H, nu))] * iterations  # :95 fresh samples per outer iteration
        return blocks

    def adam_weights(self):
        """[iterations, m, v] like ``self.optim.get_weights()``; m, v are attached to the population rows."""
        shape = (self.num_rollouts, self.mpc_horizon, self.num_control_inputs)
        return [self._get_counter(L.COUNTER_ADAM_STEP), self._get_state(L.STATE_RPGD_M, shape), self._get_state(L.STATE_RPGD_V, shape)]
