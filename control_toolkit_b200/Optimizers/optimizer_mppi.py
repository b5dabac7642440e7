"""optimizer_mppi -- B200 backend behind the reference's MPPI plugin interface.

Same constructor kwargs, ``configure(num_states, num_control_inputs, dt, predictor_specification)``,
``step(s, time) -> u`` (0-d numpy for nu=1), ``optimizer_reset()``, ``logging_values`` keys and public attributes
(``u_nom``, ``rollout_trajectories``, ``optimal_control_sequence``, ``optimal_trajectory``) as reference
Optimizers/optimizer_mppi.py:13-231.  One tick = one C call: fused sample -> rollout -> cost -> softmin kernels.
"""
from __future__ import annotations

import math
from typing import Tuple

import numpy as np

from .. import _lib as L
from . import template_optimizer


class optimizer_mppi(template_optimizer):
    _OPT = L.OPT_MPPI

    def __init__(
        self,
        predictor,
        cost_function,
        control_limits: "Tuple[np.ndarray, np.ndarray]",
        computation_library=None,
        seed: int = None,
        cc_weight: float = 1.0,
        R: float = 1.0,
        LBD: float = 100.0,
        mpc_horizon: int = 35,
        num_rollouts: int = 3500,
        NU: float = 1000.0,
        SQRTRHOINV: float = 0.03,
        period_interpolation_inducing_points: int = 10,
        optimizer_logging: bool = False,
        calculate_optimal_trajectory: bool = False,
        **kwargs,
    ):
        super().__init__(predictor=predictor, cost_function=cost_function, control_limits=control_limits,
                         optimizer_logging=optimizer_logging, seed=seed, num_rollouts=num_rollouts,
                         mpc_horizon=mpc_horizon, computation_library=computation_library, **kwargs)
        self.predictor_single_trajectory = self.predictor.copy() if hasattr(self.predictor, "copy") else None
        self.cc_weight = cc_weight
        self.R = R
        self.LBD = LBD
        self.NU = NU
        self._SQRTRHOINV = SQRTRHOINV
        self.period_interpolation_inducing_points = int(period_interpolation_inducing_points)
        self.calculate_optimal_trajectory = bool(calculate_optimal_trajectory)
        self.optimal_trajectory = None
        self.optimal_control_sequence = None
        self.rollout_trajectories = None
        self.u_nom = None

    # reference optimizer_mppi.py:114-139
    def configure(self, num_states: int, num_control_inputs: int, dt: float, predictor_specification: str, **kwargs):
        super().configure(num_states=num_states, num_control_inputs=num_control_inputs, default_configure=False)
        # :130  SQRTRHODTINV = fp32(SQRTRHOINV * (1/sqrt(dt)))  (float64 product, one rounding)
        self.SQRTRHODTINV = np.float32(np.array(self._SQRTRHOINV) * (1 / np.sqrt(dt)))
        self.number_of_interpolation_inducing_points = int(
            math.ceil((self.mpc_horizon - 1) / self.period_interpolation_inducing_points) + 1)  # Interpolator.py:79-84
        self._create_backend(dt, predictor_specification)
        self.optimizer_reset()

    def _fill_config(self, cfg: L.ctk_config) -> None:
        f = np.float32
        cfg.period_interpolation_inducing_points = self.period_interpolation_inducing_points
        # :154-155, evaluated in the reference's order in fp32: (0.5 * (1 - 1/NU)) * R ; R ; 0.5 * R
        cfg.mppi_coef_du2 = float(f(f(0.5) * (f(1) - f(1.0) / f(self.NU))) * f(self.R))
        cfg.mppi_R = float(f(self.R))
        cfg.mppi_half_R = float(f(0.5) * f(self.R))
        cfg.mppi_cc_weight = float(f(self.cc_weight))
        cfg.mppi_neg_inv_LBD = float(f(-1.0 / self.LBD))  # :165 python double folded to an fp32 constant
        cfg.mppi_stdev = float(self.SQRTRHODTINV)

    def step(self, s: np.ndarray, time=None):
        lib = self._require_backend()
        if self.optimizer_logging:
            self.logging_values = {"s_logged": np.asarray(s).copy()}
        self._refresh_live_cost(lib)
        self._feed_noise(lib, [("normal", (self.num_rollouts, self.number_of_interpolation_inducing_points,
                                           self.num_control_inputs))])
        H, nu, ns, N = self.mpc_horizon, self.num_control_inputs, int(self.num_states), self._n_local
        u = self._tick(lib, s, L.STATE_U_NOM, H * nu)
        self.u = np.squeeze(u)  # :212 0-d for nu == 1, (nu,) otherwise
        if self._state_buf is not None:
            self.u_nom = self._state_buf.reshape(1, H, nu).copy()
        else:
            self.u_nom = self._get_state(L.STATE_U_NOM, (1, H, nu))
        if self.optimizer_logging:
            self.rollout_trajectories = self._collect_rollout_logs(N)
            self.logging_values["u_logged"] = self.u
        self.optimal_control_sequence = self.u_nom.copy()
        if self.calculate_optimal_trajectory:
            self.optimal_trajectory, _ = self.rollout_single(s, self.u_nom)
        return self.u

    def step_batch(self, states: np.ndarray, active=None) -> np.ndarray:
        """Ticks of several clients in ONE kernel launch (``num_clients`` > 1; SURVEY 8f.4 -- what the reference's server does with one
        ``ctrl.step`` per request, controller_server/controller_server.py:55-86): ``states`` [num_clients, num_states], ``active``
        [num_clients] bools (None: all).  Returns u [num_clients] (NaN for inactive slots).  Every client keeps its own warm-start
        sequence, previous input and Philox tick counter, so its controls equal those of a controller of its own."""
        import ctypes as C
        lib = self._require_backend()
        self._refresh_live_cost(lib)
        B = self.num_clients
        s32 = np.ascontiguousarray(np.asarray(states, dtype=np.float32).reshape(B, -1))
        if s32.shape[1] != 6:
            raise ValueError(f"states must be [{B}, 6], got {s32.shape}")
        act = np.ones(B, np.int32) if active is None else np.ascontiguousarray(np.asarray(active).astype(np.int32).reshape(B))
        u = np.full(B, np.nan, np.float32)
        L.check(lib.ctk_step_batch(self._h, L.fptr(s32), act.ctypes.data_as(C.POINTER(C.c_int32)), L.fptr(u)))
        return u

    def reset_client(self, client: int) -> None:
        """A new client takes over slot ``client``: fresh warm-start sequence, previous input and tick counter."""
        lib = self._require_backend()
        L.check(lib.ctk_reset_client(self._h, int(client)))

    def optimizer_reset(self):
        lib = self._require_backend()
        L.check(lib.ctk_reset(self._h))
        # self.u (the cost's previous_input) survives optimizer_reset() in the reference: only optimizer_cem_tf.py:117 resets it
        self.u_nom = self._get_state(L.STATE_U_NOM, (self.num_clients, self.mpc_horizon, self.num_control_inputs))

    # state access (part of the parity contract: "optimizer state within 1e-5")
    # u_nom [1, H, nu]; u: a float for nu == 1, (nu,) otherwise (the shape step() returns)
    def get_state(self) -> dict:
        nu = int(self.num_control_inputs)
        u = self._get_state(L.STATE_U_PREV, (nu,))
        return {"u_nom": self._get_state(L.STATE_U_NOM, (1, self.mpc_horizon, nu)), "u": float(u[0]) if nu == 1 else u}

    def set_state(self, state: dict) -> None:
        nu = int(self.num_control_inputs)
        self._set_state(L.STATE_U_NOM, state["u_nom"])
        self._set_state(L.STATE_U_PREV, np.reshape(state["u"], (nu,)))
        self.u_nom = np.asarray(state["u_nom"], np.float32).reshape(1, self.mpc_horizon, nu)
