"""Shared helpers for the parity tests: fixture loading and oracle construction."""
import json
import os

import numpy as np

from oracle import spec
from oracle.cem import CEMOracle
from oracle.cem_grad import CEMBharadhwajOracle, CEMNaiveGradOracle
from oracle.gradient import GradientOracle
from oracle.mppi import MPPIOracle
from oracle.random_action import RandomActionOracle
from oracle.replay_rng import ReplayRNG
from oracle.rpgd import RPGDOracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names(prefix=""):
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and f.startswith(prefix))


def load_interpolation_weights():
    """{(horizon, period): W [n_ind, horizon] float32}: the reference Interpolator's weights over the sweep of
    tests/dropin/drive_reference_interpolator.py, stored in tests/golden/interpolator/weights_sweep.npz."""
    z = np.load(os.path.join(GOLDEN, "interpolator", "weights_sweep.npz"))
    out, off = {}, 0
    for H, period, n_ind in z["geometry"].tolist():
        out[(H, period)] = z["weights"][off:off + n_ind * H].reshape(n_ind, H)
        off += n_ind * H
    assert off == z["weights"].size
    return out


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = json.loads(str(z["config"]))
    return z, meta


def make_predictor(meta):
    if meta.get("environment", "CartPole") == "DubinsCar":
        return spec.DubinsPredictor(spec.DubinsParams(dt=meta["cfg"]["mpc_timestep"]))
    if meta["predictor"].startswith("ODE"):
        return spec.ODEPredictor(spec.CartPoleParams(dt=meta["cfg"]["mpc_timestep"]))
    if meta["predictor"].startswith("GRU"):
        return spec.GRUPredictor(spec.GRUWeights.random_init(meta["gru_seed"]))
    return spec.MLPPredictor(spec.MLPWeights.random_init(meta["mlp_seed"]))


def make_oracle(meta, **over):
    pred = make_predictor(meta)
    cost = spec.CostParams(name=meta["cost"])
    cfg = dict(meta["cfg"])
    cfg.update(over)
    if meta.get("environment", "CartPole") == "DubinsCar":
        cost = spec.DubinsCost(name=meta["cost"])
        nu = spec.DUBINS_NUM_CONTROLS
        cfg.setdefault("action_low", np.full(nu, -1.0, np.float32))
        cfg.setdefault("action_high", np.full(nu, 1.0, np.float32))
    cls = {"mppi": MPPIOracle, "cem-tf": CEMOracle, "rpgd": RPGDOracle, "random-action-tf": RandomActionOracle,
           "gradient-tf": GradientOracle, "cem-naive-grad-tf": CEMNaiveGradOracle, "cem-grad-bharadhwaj-tf": CEMBharadhwajOracle}[meta["optimizer"]]
    return cls(pred, cost, **cfg)


def replay(meta):
    return ReplayRNG(meta["noise_seed"])


def maybe_reset_oracle(o, meta, t, rng):
    """controller_reset() before tick t of the reset-mid-episode fixtures (oracle side)."""
    if t == meta.get("reset_before_tick", -1):
        if meta["optimizer"] in ("mppi", "cem-tf"):
            o.reset()
        else:
            o.reset(rng)


def rel_err(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def elem_rel(a, b, floor=1e-3):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor)))


def oracle_state(o, meta):
    """The optimizer state array the parity contract names (u_nom / dist_mue / Q)."""
    if meta["optimizer"] == "random-action-tf":
        return np.atleast_1d(np.asarray(o.u, np.float32))
    return {"mppi": lambda: o.u_nom, "cem-tf": lambda: o.dist_mue, "rpgd": lambda: o.Q, "gradient-tf": lambda: o.Q,
            "cem-naive-grad-tf": lambda: o.dist_mue, "cem-grad-bharadhwaj-tf": lambda: o.dist_mue}[meta["optimizer"]]().numpy()


_FLOOR_CACHE = {}


def fp32_noise_floor(name, ticks=None, **over):
    """Per tick: how far the reference algorithm evaluated in fp32 (the oracle, == the unmodified reference files, see
    test_oracle_golden.py) is from the SAME algorithm evaluated in float64 on the same injected noise.  This is the
    rounding noise floor of the path: the rollouts integrate an unstable pendulum for 50-100 steps, so 1-ulp differences
    (e.g. another libm's sin/cos) are amplified by 1e2..1e3.  No independent fp32 implementation can agree with the
    reference more closely than the reference agrees with exact arithmetic, so the GPU tolerances are
    1e-5 + 2 x this floor (north-star tolerance plus the reference's own rounding noise).  Measured values are written to gpurun_out/parity_errors.txt and quoted in DESIGN.md."""
    import torch
    key = (name, ticks, tuple(sorted(over.items())))
    if key in _FLOOR_CACHE:
        return _FLOOR_CACHE[key]
    z, meta = load_golden(name)
    ticks = ticks or meta["ticks"]
    o32, o64 = make_oracle(meta, **over), make_oracle(meta, dtype=torch.float64, **over)
    if meta["predictor"].startswith("Dense"):
        o64.predictor = spec.MLPPredictor(spec.MLPWeights.random_init(meta["mlp_seed"]), dtype=torch.float64)
    if meta["predictor"].startswith("GRU"):
        o64.predictor = spec.GRUPredictor(spec.GRUWeights.random_init(meta["gru_seed"]), dtype=torch.float64)
    r32, r64 = replay(meta), replay(meta)
    if meta["optimizer"] in ("rpgd", "random-action-tf", "gradient-tf"):
        o32.reset(r32)
        o64.reset(r64)
    out = []
    for t in range(ticks):
        maybe_reset_oracle(o32, meta, t, r32)
        maybe_reset_oracle(o64, meta, t, r64)
        u32, u64 = o32.step(z["states"][t], r32), o64.step(z["states"][t], r64)
        s32, s64 = oracle_state(o32, meta), oracle_state(o64, meta)
        scale = max(float(np.max(np.abs(s64))), 1e-2)
        eJ = np.abs(o32.last["J"].astype(np.float64) - o64.last["J"]) / (np.abs(o64.last["J"]) + 1e-3)
        out.append(dict(state=rel_err(s32, s64), J=float(eJ.max()), J_q99=float(np.quantile(eJ, 0.99)),
                        u=float(np.max(np.abs(np.ravel(u32) - np.ravel(u64)))) / scale,
                        state64=np.array(s64, np.float64), state32=np.array(s32, np.float64)))  # the float64 truth / fp32 reference of this tick
    _FLOOR_CACHE[key] = out
    return out
