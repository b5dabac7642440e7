"""TEST INFRASTRUCTURE ONLY: the gradient optimizers' oracles (oracle/rpgd.py, oracle/gradient.py, oracle/cem_grad.py) for any
number of control inputs nu, read from the predictor, with per-input limits.  The files under oracle/ are pinned to the fixtures of
the unmodified reference at nu = 1 and stay as they are; these subclasses replace only the methods that hard-code a trailing control
dimension of 1.  At nu = 1 they compute the same numbers as their base classes (tests/test_env_gradient_cpu.py checks it).

Semantics for nu > 1, read from the reference source (DESIGN section 2; not pinned to fixtures of the unmodified reference):
sample_actions draws [B, n_ind, nu]; clip_by_norm(axes=[1,2]) takes one norm per trajectory; the Adam moments shift by one time step;
the gradient-tf tail redraw is [N, 1, nu] uniform over each input's limits; grad-CEM refits mean and std per (t, input) column."""
from __future__ import annotations

import numpy as np
import torch

from oracle.cem_grad import CEMBharadhwajOracle, CEMNaiveGradOracle
from oracle.gradient import GradientOracle
from oracle.rpgd import RPGDOracle


def _per_input(v, nu):
    return np.broadcast_to(np.asarray(v, np.float32), (nu,)).copy()


class RPGDOracleNu(RPGDOracle):
    def __init__(self, predictor, cost, *, action_low=-1.0, action_high=1.0, sample_whole_control_space=True, **kw):
        super().__init__(predictor, cost, sample_whole_control_space=sample_whole_control_space, **kw)
        self.nu = int(getattr(predictor, "num_control_inputs", 1))
        self.low = torch.tensor(_per_input(action_low, self.nu).astype(np.float64), dtype=self.dtype)
        self.high = torch.tensor(_per_input(action_high, self.nu).astype(np.float64), dtype=self.dtype)
        if sample_whole_control_space:  # :200-205, per input
            self.sample_min, self.sample_max = self.low.clone(), self.high.clone()

    def sample_actions(self, rng, batch):  # :275-296 with [batch, n_ind, nu] draws
        if self.dist == "normal":
            Qn = rng.normal([batch, self.n_ind, self.nu], mean=self.sample_mean.float(), stddev=self.sample_stdev.float(), dtype=torch.float32).to(self.dtype)
        elif self.dist == "uniform":
            Qn = rng.uniform([batch, self.n_ind, self.nu], minval=self.sample_min.float(), maxval=self.sample_max.float(), dtype=torch.float32).to(self.dtype)
        else:
            raise ValueError(f"RPGD cannot interpret sampling type {self.dist}")
        Qn = torch.minimum(torch.maximum(Qn, self.low), self.high)
        return torch.matmul(Qn.permute(2, 0, 1), self.W[None]).permute(1, 2, 0)

    def step(self, s: np.ndarray, rng) -> np.ndarray:  # RPGDOracle.step with the zero fills over nu columns
        s = torch.as_tensor(np.tile(np.asarray(s, np.float32), (self.N, 1))).to(self.dtype)
        iters = self.first_iter_count if self.count == 0 else self.outer_its
        for _ in range(iters):
            self.Q, _ = self.grad_step(s, self.Q)
        with torch.no_grad():
            J, rollout = self._cost(s, self.Q)
            best_idx = torch.argsort(J, dim=0, stable=True)[: self.k]
            sp = self.shift_previous
            Qn = torch.cat([self.Q[:, sp:, :], self.Q[:, -1:, :].repeat(1, sp, 1)], dim=1)
            u_nom = self.Q[best_idx[0]][None].clone()
            Q_logged, ages_logged = self.Q.clone(), self.ages.clone()
            m_t, v_t = self.m, self.v
            if self.count % self.resamp_per == 0:
                Qres = self.sample_actions(rng, self.N - self.k)
                Qn = torch.cat([Qres, torch.index_select(Qn, 0, best_idx)], 0)
                self.ages = torch.cat([torch.zeros((self.N - self.k,), dtype=self.dtype), torch.index_select(self.ages, 0, best_idx)], 0)
                zk = torch.zeros([self.k, 1, self.nu], dtype=self.dtype)
                wk1 = torch.cat([torch.index_select(m_t, 0, best_idx)[:, 1:, :], zk], 1)
                wk2 = torch.cat([torch.index_select(v_t, 0, best_idx)[:, 1:, :], zk], 1)
                z = torch.zeros([self.N - self.k, self.H, self.nu], dtype=self.dtype)
                self.m, self.v = torch.cat([z, wk1], 0), torch.cat([z, wk2], 0)
            else:
                zn = torch.zeros([self.N, 1, self.nu], dtype=self.dtype)
                self.m = torch.cat([m_t[:, 1:, :], zn], 1)
                self.v = torch.cat([v_t[:, 1:, :], zn], 1)
            self.ages = self.ages + 1
            self.Q = Qn.clone()
            self.count += 1
        self.u = u_nom[0, 0, :].numpy().copy()
        self.last = dict(J=J.numpy(), Q=Q_logged.numpy(), rollouts=rollout.numpy(), ages=ages_logged.numpy(),
                         u_nom=u_nom.numpy(), best_idx=best_idx.numpy())
        return self.u


class GradientOracleNu(GradientOracle):
    def __init__(self, predictor, cost, *, action_low=-1.0, action_high=1.0, **kw):
        super().__init__(predictor, cost, **kw)
        self.nu = int(getattr(predictor, "num_control_inputs", 1))
        self.low, self.high = torch.from_numpy(_per_input(action_low, self.nu)), torch.from_numpy(_per_input(action_high, self.nu))

    def _clip(self, Q):
        return torch.minimum(torch.maximum(Q, self.low.to(self.dtype)), self.high.to(self.dtype))

    def reset(self, rng):  # :169-185 with [N, H, nu] draws over each input's limits
        self.Q = self._clip(rng.uniform([self.N, self.H, self.nu], self.low, self.high, dtype=torch.float32).to(self.dtype))
        self.count = 0
        self.adam_step, self.m, self.v = 0, None, None

    def _grad_step(self, s):  # GradientOracle._grad_step with the per-input box clip
        Q = self.Q.detach().clone().requires_grad_(True)
        J, _ = self._cost(s, Q)
        (g,) = torch.autograd.grad(J.sum(), Q)
        n = torch.sqrt(torch.sum(g * g, dim=(1, 2), keepdim=True))
        c = torch.tensor(self.gradmax_clip, dtype=self.dtype)
        g = g * c / torch.maximum(n, c)
        if self.m is None:
            self.m, self.v = torch.zeros_like(g), torch.zeros_like(g)
        t = self.adam_step + 1
        f32 = np.float32
        if self.dtype == torch.float32:
            lr_t = float(f32(f32(self.lr) * np.sqrt(f32(1) - np.power(f32(self.b2), f32(t))) / (f32(1) - np.power(f32(self.b1), f32(t)))))
            one_b1, one_b2, eps = float(f32(1 - self.b1)), float(f32(1 - self.b2)), float(f32(self.eps))
        else:
            lr_t = self.lr * np.sqrt(1 - self.b2 ** t) / (1 - self.b1 ** t)
            one_b1, one_b2, eps = 1 - self.b1, 1 - self.b2, self.eps
        self.m = self.m + (g - self.m) * one_b1
        self.v = self.v + (g * g - self.v) * one_b2
        Qn = Q.detach() - lr_t * self.m / (torch.sqrt(self.v) + eps)
        self.adam_step = t
        self.Q = self._clip(Qn)

    def step(self, s: np.ndarray, rng) -> np.ndarray:  # GradientOracle.step with the [N, 1, nu] tail redraw and zero fill
        s = torch.as_tensor(np.tile(np.asarray(s, np.float32), (self.N, 1))).to(self.dtype)
        iters = self.first_iter_count if self.count == 0 else self.gradient_steps
        for _ in range(iters):
            self._grad_step(s)
        Q = self.Q
        traj_cost, rollout = self._cost(s, Q)
        best_idx = int(torch.argsort(traj_cost.detach(), stable=True)[0])
        self.u = Q[best_idx, 0, :].squeeze().detach().numpy().astype(np.float32)
        self.last = dict(J=traj_cost.detach().numpy(), Q=Q.detach().numpy().copy(), rollouts=rollout.detach().numpy(), best_idx=best_idx)
        self.count += 1
        Q_s = rng.uniform(shape=[self.N, 1, self.nu], minval=self.low, maxval=self.high, dtype=torch.float32).to(self.dtype)
        self.Q = torch.cat([self.Q[:, 1:, :], Q_s], dim=1)
        if self.m is not None:
            z = torch.zeros((self.N, 1, self.nu), dtype=self.dtype)
            self.m = torch.cat([self.m[:, 1:, :], z], dim=1)
            self.v = torch.cat([self.v[:, 1:, :], z], dim=1)
        return self.u


class _CEMGradNu:
    """Per-input limits and mid-range fill; mean and std per (t, input) column (the base classes' reductions run over dim 0)."""

    def _setup(self, predictor, action_low, action_high, dtype):
        self.nu = int(getattr(predictor, "num_control_inputs", 1))
        lo, hi = _per_input(action_low, self.nu).astype(np.float64), _per_input(action_high, self.nu).astype(np.float64)
        self._lim = (torch.tensor(lo, dtype=dtype), torch.tensor(hi, dtype=dtype))
        self.mid = torch.tensor((lo + hi) * 0.5, dtype=dtype)

    def reset(self, rng=None):
        self.dist_mue = self.mid * torch.ones([1, self.H, self.nu], dtype=self.dtype)
        self.stdev = self.init_std * torch.ones([1, self.H, self.nu], dtype=self.dtype)
        self.count = 0

    def _time_shift(self):
        self.stdev = torch.clamp(self.stdev, self.std_min, 10.0)
        self.stdev = torch.cat([self.stdev[:, 1:, :], self.init_std * torch.ones((1, 1, self.nu), dtype=self.dtype)], dim=1)
        self.dist_mue = torch.cat([self.dist_mue[:, 1:, :], self.mid * torch.ones((1, 1, self.nu), dtype=self.dtype)], dim=1)


class CEMNaiveGradOracleNu(_CEMGradNu, CEMNaiveGradOracle):
    def __init__(self, predictor, cost, *, action_low=-1.0, action_high=1.0, dtype=torch.float32, **kw):
        self._setup(predictor, action_low, action_high, dtype)
        super().__init__(predictor, cost, dtype=dtype, **kw)
        self.low, self.high = self._lim

    def step(self, s: np.ndarray, rng) -> np.ndarray:  # CEMNaiveGradOracle.step with [N, H, nu] draws
        s = torch.as_tensor(np.tile(np.asarray(s, np.float32), (self.N, 1))).to(self.dtype)
        elite_log = []
        for _ in range(self.outer_it):
            Q = self.dist_mue.repeat(self.N, 1, 1) + rng.normal([self.N, self.H, self.nu], dtype=torch.float32).to(self.dtype) * self.stdev
            Q = torch.clamp(Q, self.low, self.high)
            g = self._clipped_gradient(s, Q)
            Qn = torch.clamp(Q - self.lr * g, self.low, self.high)
            traj_cost, rollout = self._cost(s, Qn)
            best_idx, _ = self._refit(Qn, traj_cost)
            elite_log.append(best_idx.numpy().copy())
        self.stdev = torch.clamp(self.stdev, self.std_min, 10.0)
        self.stdev = torch.cat([self.stdev[:, 1:, :], self.init_std * torch.ones((1, 1, self.nu), dtype=self.dtype)], dim=1)
        self.u = self.dist_mue[0, 0, :].squeeze().numpy().astype(np.float32).copy()  # the refit MEAN
        self.dist_mue = torch.cat([self.dist_mue[:, 1:, :], self.mid * torch.ones((1, 1, self.nu), dtype=self.dtype)], dim=1)
        self.last = dict(J=traj_cost.detach().numpy(), Q=Qn.detach().numpy(), rollouts=rollout.detach().numpy(), elite_idx=np.stack(elite_log))
        self.count += 1
        return self.u


class CEMBharadhwajOracleNu(_CEMGradNu, CEMBharadhwajOracle):
    def __init__(self, predictor, cost, *, action_low=-1.0, action_high=1.0, dtype=torch.float32, **kw):
        self._setup(predictor, action_low, action_high, dtype)
        super().__init__(predictor, cost, dtype=dtype, **kw)
        self.low, self.high = self._lim

    def _sample(self, rng, n):  # :125-132 with [n, H, nu] draws
        return self.dist_mue.repeat(n, 1, 1) + self.stdev * rng.normal([n, self.H, self.nu], dtype=torch.float32).to(self.dtype)


ORACLES = {"rpgd": RPGDOracleNu, "gradient-tf": GradientOracleNu, "cem-naive-grad-tf": CEMNaiveGradOracleNu,
           "cem-grad-bharadhwaj-tf": CEMBharadhwajOracleNu}
