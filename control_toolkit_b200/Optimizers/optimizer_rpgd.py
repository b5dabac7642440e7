"""optimizer_rpgd -- B200 backend behind the reference's RPGD plugin interface
(reference Optimizers/optimizer_rpgd.py:144-548).

The reference differentiates the rollout with a GradientTape / autograd; here a forward kernel stores the state tape in
shared memory and a hand-derived reverse-mode (adjoint) sweep produces dJ/dQ, followed by the per-trajectory norm clip,
Adam, box clip, and -- in a second kernel -- the argsort / shift / resample / Adam-moment bookkeeping of ``step``.

``adam_form``: "keras" (default; the TF reference uses tf.keras.optimizers.Adam, :34-43) or "torch" (the reference's
manual torch update, :56-82).  They differ in the epsilon placement and are NOT interchangeable at 1e-5
(tests/test_oracle_golden.py::test_rpgd_keras_vs_torch_adam_form).
"""
from __future__ import annotations

import math
from typing import Tuple

import numpy as np

from .. import _lib as L
from . import template_optimizer


class optimizer_rpgd(template_optimizer):
    _OPT = L.OPT_RPGD

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        mpc_horizon: int = 40,
        num_rollouts: int = 32,
        outer_its: int = 2,
        sample_stdev: float = 0.5,
        sample_mean: float = 0.0,
        sample_whole_control_space: bool = True,
        uniform_dist_min: float = -1.0,
        uniform_dist_max: float = 1.0,
        resamp_per: int = 10,
        period_interpolation_inducing_points: int = 10,
        SAMPLING_DISTRIBUTION: str = "uniform",
        shift_previous: int = 1,
        warmup: bool = False,
        warmup_iterations: int = 250,
        learning_rate: float = 0.05,
        opt_keep_k_ratio: float = 0.25,
        gradmax_clip: float = 5,
        rtol: float = 1.0e-3,
        adam_beta_1: float = 0.9,
        adam_beta_2: float = 0.999,
        adam_epsilon: float = 1.0e-8,
        optimizer_logging: bool = False,
        calculate_optimal_trajectory: bool = False,
        adam_form: str = "keras",
        **kwargs,
    ):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         optimizer_logging=optimizer_logging, seed=seed, num_rollouts=num_rollouts,
                         mpc_horizon=mpc_horizon, computation_library=computation_library, **kwargs)
        self.predictor_single_trajectory = self.predictor.copy() if hasattr(self.predictor, "copy") else None
        self.outer_its = int(outer_its)
        self.sample_stdev = np.float32(sample_stdev)
        self.sample_mean = np.float32(sample_mean)
        self.sample_whole_control_space = bool(sample_whole_control_space)
        if self.sample_whole_control_space:  # :199-205, per input
            self.sample_min, self.sample_max = np.asarray(self.action_low, np.float32), np.asarray(self.action_high, np.float32)
        else:
            self.sample_min, self.sample_max = np.float32(uniform_dist_min), np.float32(uniform_dist_max)
        self.resamp_per = int(resamp_per)
        self.period_interpolation_inducing_points = int(period_interpolation_inducing_points)
        self.shift_previous = int(shift_previous)
        self.do_warmup = bool(warmup)
        self.warmup_iterations = int(warmup_iterations)
        self.opt_keep_k = int(max(int(num_rollouts * opt_keep_k_ratio), 1))  # :213
        self.gradmax_clip = np.float32(gradmax_clip)
        self.rtol = rtol
        self.SAMPLING_DISTRIBUTION = SAMPLING_DISTRIBUTION
        if SAMPLING_DISTRIBUTION not in ("normal", "uniform"):  # :291
            raise ValueError(f"RPGD cannot interpret sampling type {SAMPLING_DISTRIBUTION}")
        self.first_iter_count = self.warmup_iterations if self.do_warmup else self.outer_its  # :219-221
        self.learning_rate, self.adam_beta_1, self.adam_beta_2, self.adam_epsilon = learning_rate, adam_beta_1, adam_beta_2, adam_epsilon
        if adam_form not in ("keras", "torch"):
            raise ValueError(f"adam_form must be 'keras' or 'torch', got {adam_form}")
        self.adam_form = adam_form
        self.calculate_optimal_trajectory = bool(calculate_optimal_trajectory)
        self.optimal_trajectory = None
        self.summed_stage_cost = None
        self.optimal_control_sequence = None
        self.rollout_trajectories = None
        self.u_nom = None
        self.count = 0

    # reference optimizer_rpgd.py:245-273
    def configure(self, num_states: int, num_control_inputs: int, **kwargs):
        dt = kwargs.get("dt", None)
        predictor_specification = kwargs.get("predictor_specification", None)
        super().configure(num_states=num_states, num_control_inputs=num_control_inputs, default_configure=False)
        if dt is None or predictor_specification is None:
            raise ValueError("RPGD requires dt and predictor_specification to be passed.")
        self.number_of_interpolation_inducing_points = int(
            math.ceil((self.mpc_horizon - 1) / self.period_interpolation_inducing_points) + 1)
        self._create_backend(dt, predictor_specification)
        if self.calculate_optimal_trajectory and self._env_info.env_id != L.ENV_CARTPOLE:
            raise ValueError("calculate_optimal_trajectory: the nominal rollout (ctk_rollout_single) is implemented for the CartPole "
                             f"environment only, not {self._environment()!r}")
        self.optimizer_reset()

    def _fill_config(self, cfg: L.ctk_config) -> None:
        cfg.period_interpolation_inducing_points = self.period_interpolation_inducing_points
        cfg.rpgd_outer_its = self.outer_its
        cfg.rpgd_first_iter_count = self.first_iter_count
        cfg.rpgd_resamp_per = self.resamp_per
        cfg.rpgd_shift_previous = self.shift_previous
        cfg.rpgd_keep_k = self.opt_keep_k
        cfg.rpgd_distribution = L.DIST_NORMAL if self.SAMPLING_DISTRIBUTION == "normal" else L.DIST_UNIFORM
        cfg.rpgd_adam_form = L.ADAM_KERAS if self.adam_form == "keras" else L.ADAM_TORCH
        cfg.rpgd_sample_mean, cfg.rpgd_sample_stdev = float(self.sample_mean), float(self.sample_stdev)
        # the CartPole reads the scalar range; other environments sample each input over its own limits when the whole space is sampled
        cfg.rpgd_sample_min, cfg.rpgd_sample_max = float(np.ravel(self.sample_min)[0]), float(np.ravel(self.sample_max)[0])
        cfg.rpgd_sample_whole_space = int(self.sample_whole_control_space)
        cfg.rpgd_learning_rate = float(np.float32(self.learning_rate))
        cfg.rpgd_gradmax_clip = float(self.gradmax_clip)
        cfg.rpgd_beta_1, cfg.rpgd_beta_2, cfg.rpgd_epsilon = float(self.adam_beta_1), float(self.adam_beta_2), float(self.adam_epsilon)

    def _draw_kind(self) -> str:
        return "normal" if self.SAMPLING_DISTRIBUTION == "normal" else "uniform"

    def step(self, s: np.ndarray, time=None):
        lib = self._require_backend()
        if self.optimizer_logging:
            self.logging_values = {"s_logged": np.asarray(s).copy()}
        self._refresh_live_cost(lib)
        u_before = self.u
        if self.count % self.resamp_per == 0 and self.num_rollouts - self.opt_keep_k > 0:  # :449-453
            self._feed_noise(lib, [(self._draw_kind(), (self.num_rollouts - self.opt_keep_k,
                                                        self.number_of_interpolation_inducing_points,
                                                        self.num_control_inputs))])
        H, nu, N = self.mpc_horizon, self.num_control_inputs, self.num_rollouts
        u = self._tick(lib, s, L.STATE_U_NOM, H * nu)  # u and Q[best] (:426) come back through the same host mirror
        self.u_nom = (self._state_buf.reshape(1, H, nu).copy() if self._state_buf is not None
                      else self._get_log(L.LOG_U_NOM, (1, H, nu)))
        if self.optimizer_logging:
            self.rollout_trajectories = self._collect_rollout_logs(N)
            self.logging_values["trajectory_ages_logged"] = self._get_log(L.LOG_AGES, (N,))
            self.logging_values["u_logged"] = u_before  # :416 logs the PREVIOUS u
        self.optimal_control_sequence = self.u_nom.copy()
        self.count += 1  # :516
        if self.calculate_optimal_trajectory:  # :518-521
            self.optimal_trajectory, self.summed_stage_cost = self.rollout_single(s, self.u_nom)
        self.u = u.reshape(nu).copy()  # :523 shape (nu,)
        return self.u

    def optimizer_reset(self):
        lib = self._require_backend()
        self._feed_noise(lib, [(self._draw_kind(), (self.num_rollouts, self.number_of_interpolation_inducing_points,
                                                    self.num_control_inputs))])  # :540
        L.check(lib.ctk_reset(self._h))
        self.count = 0
        # self.u (the cost's previous_input) survives optimizer_reset() in the reference: only optimizer_cem_tf.py:117 resets it

    # reference attributes, read from the device on demand
    @property
    def Q_tf(self) -> np.ndarray:
        return self._get_state(L.STATE_RPGD_Q, (self.num_rollouts, self.mpc_horizon, self.num_control_inputs))

    @property
    def trajectory_ages(self) -> np.ndarray:
        return self._get_state(L.STATE_RPGD_AGES, (self.num_rollouts,))

    def adam_weights(self):
        """[step, m, v] like ADAM.get_weights() (reference :84-99)."""
        shape = (self.num_rollouts, self.mpc_horizon, self.num_control_inputs)
        return [self._get_counter(L.COUNTER_ADAM_STEP), self._get_state(L.STATE_RPGD_M, shape), self._get_state(L.STATE_RPGD_V, shape)]

    def best_indices(self) -> np.ndarray:
        return self._get_log(L.LOG_ELITE_IDX, (self.opt_keep_k,), np.int32)

    def last_costs(self) -> np.ndarray:
        return self._get_log(L.LOG_J, (self.num_rollouts,))

    def get_state(self) -> dict:
        step, m, v = self.adam_weights()
        return {"Q": self.Q_tf, "adam_step": step, "adam_m": m, "adam_v": v, "ages": self.trajectory_ages,
                "count": self.count, "u": self._get_state(L.STATE_U_PREV, (self.num_control_inputs,))}

    def set_state(self, state: dict) -> None:
        self._set_state(L.STATE_RPGD_Q, state["Q"])
        self._set_state(L.STATE_RPGD_M, state["adam_m"])
        self._set_state(L.STATE_RPGD_V, state["adam_v"])
        self._set_state(L.STATE_RPGD_AGES, state["ages"])
        self._set_state(L.STATE_U_PREV, np.reshape(state["u"], (self.num_control_inputs,)))
        self._set_counter(L.COUNTER_ADAM_STEP, int(state["adam_step"]))
        self.count = int(state["count"])
        self._set_counter(L.COUNTER_COUNT, self.count)
