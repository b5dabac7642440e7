"""oracle.gen_golden -- TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz.

Runs the reference's UNMODIFIED ``controller_mpc`` + ``optimizer_mppi`` / ``optimizer_rpgd`` /
``optimizer_cem_tf`` / ``optimizer_random_action_tf`` files (imported from the checkout CTK_REFERENCE names, through the shims in oracle/refharness) on
torch-CPU fp32 with the build's pinned predictor / cost spec and INJECTED noise, and stores inputs +
outputs as small fixtures.  Needs a checkout of the original Control_Toolkit:

    CTK_REFERENCE=<checkout> python -m oracle.gen_golden            # writes tests/golden/*.npz
    python -m oracle.gen_golden --out DIR mppi_c1_n64 rpgd_c3   # some cases, into another directory

Each fixture holds: the case config (json), the per-tick states, the noise seed (noise is regenerated from
``numpy.random.default_rng(seed)`` by oracle.replay_rng.ReplayRNG; a checksum of the draws is stored), and
the reference's outputs per tick.
"""
from __future__ import annotations

import copy
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
GOLDEN = os.path.join(REPO, "tests", "golden")

# ------------------------------------------------------------------------------------------------
# case table.  C1..C4 = BASELINE.json configs (reduced N where a fixture would be too large).
# ------------------------------------------------------------------------------------------------
MPPI_BASE = dict(seed=42, mpc_horizon=50, mpc_timestep=0.02, num_rollouts=2000, cc_weight=1.0, R=1.0, LBD=100.0,
                 NU=1000.0, SQRTRHOINV=0.03, period_interpolation_inducing_points=10)
CEM_BASE = dict(seed=42, mpc_horizon=50, mpc_timestep=0.02, cem_outer_it=3, cem_initial_action_stdev=0.5,
                num_rollouts=4096, cem_stdev_min=0.01, cem_best_k=64, warmup=False, warmup_iterations=250)
RPGD_BASE = dict(seed=42, mpc_horizon=50, mpc_timestep=0.02, SAMPLING_DISTRIBUTION="uniform",
                 period_interpolation_inducing_points=10, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999,
                 adam_epsilon=1.0e-8, gradmax_clip=5, rtol=1.0e-3, num_rollouts=32, opt_keep_k_ratio=0.25,
                 outer_its=2, resamp_per=10, sample_stdev=0.5, sample_mean=0.0, sample_whole_control_space=True,
                 uniform_dist_min=-1.0, uniform_dist_max=1.0, shift_previous=1, warmup=False, warmup_iterations=250)


def _c(base, **kw):
    d = copy.deepcopy(base)
    d.update(kw)
    return d


CASES = {
    # name: (optimizer, predictor_spec, cost, optimizer-config, ticks, keep_rollouts)
    "mppi_c1_n64": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=64), 4, True),
    "mppi_c1_n2000": ("mppi", "ODE", "default", _c(MPPI_BASE), 3, False),
    "mppi_h100_n256": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=256, mpc_horizon=100), 3, False),
    "mppi_h43_p10_n64": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=64, mpc_horizon=43), 2, True),
    "mppi_h20_p1_n96": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=96, mpc_horizon=20,
                                                      period_interpolation_inducing_points=1), 2, False),
    "mppi_lbd1_n512": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=512, LBD=1.0, SQRTRHOINV=0.1), 3, False),
    "cem_c2_n256_k16": ("cem-tf", "ODE", "default", _c(CEM_BASE, num_rollouts=256, cem_best_k=16), 3, True),
    "cem_c2_n4096_k64": ("cem-tf", "ODE", "default", _c(CEM_BASE), 2, False),
    "cem_warmup_n128": ("cem-tf", "ODE", "default", _c(CEM_BASE, num_rollouts=128, cem_best_k=8, warmup=True,
                                                       warmup_iterations=5, mpc_horizon=30), 2, False),
    "rpgd_c3": ("rpgd", "ODE", "quadratic_boundary_grad", _c(RPGD_BASE), 12, True),
    "rpgd_normal_shift2": ("rpgd", "ODE", "quadratic_boundary_grad",
                           _c(RPGD_BASE, SAMPLING_DISTRIBUTION="normal", shift_previous=2, resamp_per=3,
                              num_rollouts=48, mpc_horizon=35, outer_its=3), 7, False),
    "rpgd_warmup_n64": ("rpgd", "ODE", "quadratic_boundary_grad",
                        _c(RPGD_BASE, num_rollouts=64, warmup=True, warmup_iterations=6, resamp_per=2,
                           period_interpolation_inducing_points=5), 4, False),
    # reference Optimizers/optimizer_random_action_tf.py (SURVEY 8f.1: sibling optimizer on the same kernels)
    "random_action_n512": ("random-action-tf", "ODE", "default",
                           dict(seed=42, mpc_horizon=50, mpc_timestep=0.02, num_rollouts=512), 3, True),
    "random_action_n4096_h30": ("random-action-tf", "ODE", "default",
                                dict(seed=42, mpc_horizon=30, mpc_timestep=0.02, num_rollouts=4096), 2, False),
    # reference Optimizers/optimizer_gradient_tf.py (template block config_optimizers.yml:48-61): Adam on the whole population
    "gradient_n40": ("gradient-tf", "ODE", "quadratic_boundary_grad",
                     dict(seed=42, mpc_horizon=35, mpc_timestep=0.02, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999,
                          adam_epsilon=1.0e-07, rtol=1.0e-3, gradient_steps=5, num_rollouts=40, initial_action_stdev=0.5,
                          gradmax_clip=5, warmup=False, warmup_iterations=250), 6, True),
    "gradient_warmup_n33": ("gradient-tf", "ODE", "quadratic_boundary_grad",
                            dict(seed=42, mpc_horizon=20, mpc_timestep=0.02, learning_rate=0.1, adam_beta_1=0.9, adam_beta_2=0.999,
                                 adam_epsilon=1.0e-07, rtol=1.0e-3, gradient_steps=2, num_rollouts=33, initial_action_stdev=0.5,
                                 gradmax_clip=2, warmup=True, warmup_iterations=7), 4, False),
    # reference Optimizers/optimizer_cem_naive_grad_tf.py (template block config_optimizers.yml:23-32): CEM whose samples take one
    # clipped gradient-descent step before they are ranked
    "gradcem_naive_n200": ("cem-naive-grad-tf", "ODE", "quadratic_boundary_grad",
                            dict(seed=42, mpc_horizon=35, mpc_timestep=0.02, cem_outer_it=1, num_rollouts=200, cem_stdev_min=0.1,
                                 cem_initial_action_stdev=0.5, cem_best_k=40, learning_rate=0.1, gradmax_clip=10), 5, True),
    "gradcem_naive_it3_n96": ("cem-naive-grad-tf", "ODE", "quadratic_boundary_grad",
                               dict(seed=42, mpc_horizon=20, mpc_timestep=0.02, cem_outer_it=3, num_rollouts=96, cem_stdev_min=0.05,
                                    cem_initial_action_stdev=0.7, cem_best_k=12, learning_rate=0.2, gradmax_clip=2), 4, False),
    # reference Optimizers/optimizer_cem_grad_bharadhwaj_tf.py (template block config_optimizers.yml:33-47): elites carried between the
    # outer iterations, one Adam step (persistent moments) on the whole population before ranking
    "gradcem_bharadhwaj_n32": ("cem-grad-bharadhwaj-tf", "ODE", "quadratic_boundary_grad",
                           dict(seed=42, mpc_horizon=50, mpc_timestep=0.02, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999,
                                adam_epsilon=1.0e-08, num_rollouts=32, cem_best_k=8, cem_outer_it=2, cem_initial_action_stdev=2,
                                cem_stdev_min=1.e-6, gradmax_clip=5, warmup=False, warmup_iterations=250), 6, True),
    "gradcem_bharadhwaj_warmup_n64": ("cem-grad-bharadhwaj-tf", "ODE", "quadratic_boundary_grad",
                                  dict(seed=42, mpc_horizon=30, mpc_timestep=0.02, learning_rate=0.1, adam_beta_1=0.9, adam_beta_2=0.999,
                                       adam_epsilon=1.0e-08, num_rollouts=64, cem_best_k=16, cem_outer_it=3, cem_initial_action_stdev=0.8,
                                       cem_stdev_min=1.e-3, gradmax_clip=3, warmup=True, warmup_iterations=5), 3, False),
    # controller_reset() in the middle of an episode: only optimizer_cem_tf.optimizer_reset zeroes self.u (optimizer_cem_tf.py:117);
    # MPPI (:227-231) and RPGD (:527-548) keep the last applied control as the cost's previous_input
    "mppi_reset_mid_n64": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=64), 4, False),
    "rpgd_reset_mid_n32": ("rpgd", "ODE", "quadratic_boundary_grad", _c(RPGD_BASE, resamp_per=2), 5, False),
    "cem_reset_mid_n128": ("cem-tf", "ODE", "default", _c(CEM_BASE, num_rollouts=128, cem_best_k=8, mpc_horizon=30), 4, False),
    "mppi_mlp_c4_n256": ("mppi", "Dense-6IN-128H1-128H2-5OUT-0", "default",
                         _c(MPPI_BASE, num_rollouts=256, mpc_horizon=100), 2, False),
    "mppi_mlp_h50_n64": ("mppi", "Dense-6IN-128H1-128H2-5OUT-0", "default",
                         _c(MPPI_BASE, num_rollouts=64, mpc_horizon=50), 2, True),
    # SURVEY 8f.3: recurrent predictor (two GRU layers + read-out) with the predictor.update state hook the reference calls every
    # MPPI tick (optimizer_mppi.py:192,195-197); CEM never calls the hook (optimizer_cem_tf.py), its rollouts start from the zero state
    "mppi_gru_n256": ("mppi", "GRU-6IN-32H1-32H2-5OUT-0", "default", _c(MPPI_BASE, num_rollouts=256), 4, True),
    "cem_gru_n256_k16": ("cem-tf", "GRU-6IN-32H1-32H2-5OUT-0", "default", _c(CEM_BASE, num_rollouts=256, cem_best_k=16, mpc_horizon=30), 2, False),
    # SURVEY 8f.3: a second environment through the functor registry -- Dubins car, 3 states, TWO control inputs
    # (optimizer_mppi.py:173-175 / optimizer_cem_tf.py:64-65 sample [N, ., num_control_inputs])
    "mppi_dubins_n512": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=512, mpc_horizon=40, LBD=1.0, SQRTRHOINV=0.1, R=0.1), 4, True),
    "mppi_dubins_h23_p5_n96": ("mppi", "ODE", "default", _c(MPPI_BASE, num_rollouts=96, mpc_horizon=23, LBD=0.5, SQRTRHOINV=0.08, R=0.1,
                                                               period_interpolation_inducing_points=5), 3, False),
    "cem_dubins_n512_k32": ("cem-tf", "ODE", "default", _c(CEM_BASE, num_rollouts=512, cem_best_k=32, mpc_horizon=40), 3, True),
}
ENV_OF_CASE = {"mppi_dubins_n512": "DubinsCar", "mppi_dubins_h23_p5_n96": "DubinsCar", "cem_dubins_n512_k32": "DubinsCar"}
RESET_BEFORE_TICK = {"mppi_reset_mid_n64": 2, "rpgd_reset_mid_n32": 3, "cem_reset_mid_n128": 2}  # controller_reset() before that tick
NOISE_SEED = 1
STATE_SEED = 0
MLP_SEED = 2
GRU_SEED = 3


def run_reference_case(name: str) -> dict:
    """Execute one case through the unmodified reference.  Requires enter_workspace() to have been called."""
    import torch
    torch.set_num_threads(1)  # deterministic reduction order for the fixtures
    from oracle import spec
    from oracle.replay_rng import ReplayRNG
    from SI_Toolkit.Predictors import predictor_wrapper as pw
    import yaml

    opt_name, pred_spec, cost_name, cfg, ticks, keep_rollouts = CASES[name]
    env = ENV_OF_CASE.get(name, "CartPole")
    pw.ENVIRONMENT["name"] = env
    nu = spec.DUBINS_NUM_CONTROLS if env == "DubinsCar" else 1

    # controller config is read at controller construction time (reference Controllers/__init__.py:39)
    cc = dict(mpc=dict(optimizer=opt_name, predictor_specification=pred_spec, cost_function_specification=cost_name,
                       computation_library="tensorflow" if opt_name.endswith("-tf") else "pytorch", device="cpu",
                       controller_logging=True, calculate_optimal_trajectory=False))
    with open(os.path.join("Control_Toolkit_ASF", "config_controllers.yml"), "w") as f:
        yaml.safe_dump(cc, f)

    if pred_spec.startswith("Dense"):
        pw.MLP_REGISTRY[pred_spec] = spec.MLPWeights.random_init(MLP_SEED)
    if pred_spec.startswith("GRU"):
        pw.GRU_REGISTRY[pred_spec] = spec.GRUWeights.random_init(GRU_SEED)

    from Control_Toolkit.Controllers import controller_mpc as cm  # noqa: the reference module
    cm.config_optimizers[opt_name] = copy.deepcopy(cfg)  # optimizer kwargs (module-global dict loaded at import)

    ctrl = cm.controller_mpc(
        environment_name=env,
        control_limits=(np.full(nu, -1.0, np.float32), np.full(nu, 1.0, np.float32)),
        initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0},
    )
    ctrl.configure(optimizer_name=opt_name, predictor_specification=pred_spec)
    opt = ctrl.optimizer
    rng = ReplayRNG(NOISE_SEED)
    opt.rng = rng
    opt.optimizer_reset()  # RPGD draws its initial population here; re-done so it comes from the replay rng
    if opt_name == "rpgd":
        # reference quirk: optimizer_rpgd.py:416 logs the PREVIOUS u, which is the python float 0.0 on the first
        # tick (Optimizers/__init__.py:35) and has no .copy() (Controllers/__init__.py:177) -> give it a numpy 0.
        opt.u = np.float32(0.0)

    if opt_name.endswith("-tf"):
        import tensorflow as tfshim
        argsort_log = []
        _orig = tfshim.argsort

        def _logging_argsort(x, axis=-1):
            r = _orig(x, axis)
            argsort_log.append(r.numpy().copy())
            return r

        tfshim.argsort = _logging_argsort

    states = spec.dubins_synthetic_states(ticks, STATE_SEED) if env == "DubinsCar" else spec.synthetic_states(ticks, STATE_SEED)
    out = {"config": np.array(json.dumps(dict(case=name, optimizer=opt_name, predictor=pred_spec, cost=cost_name, environment=env,
                                              cfg=cfg, ticks=ticks, noise_seed=NOISE_SEED, state_seed=STATE_SEED,
                                              mlp_seed=MLP_SEED, gru_seed=GRU_SEED, reset_before_tick=RESET_BEFORE_TICK.get(name, -1)))),
           "states": states}
    if opt_name in ("rpgd", "gradient-tf"):
        out["Q_init"] = opt.Q_tf.numpy().copy()

    for t in range(ticks):
        if t == RESET_BEFORE_TICK.get(name, -1):
            ctrl.controller_reset()  # reference Controllers/controller_mpc.py:108-109
        u = ctrl.step(states[t], time=0.02 * t)
        out[f"u_{t}"] = np.asarray(u, np.float32).reshape(-1)
        lv = opt.logging_values
        if opt_name == "mppi":
            out[f"u_nom_{t}"] = opt.u_nom.numpy().copy()
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()
            if pred_spec.startswith("GRU"):  # the saved hidden state after this tick's predictor.update
                g = opt.predictor.predictor
                out[f"rnn_h_{t}"] = np.concatenate([g.h1.numpy().ravel(), g.h2.numpy().ravel()]).astype(np.float32)
        elif opt_name == "cem-tf":
            out[f"dist_mue_{t}"] = opt.dist_mue.numpy().copy()
            out[f"stdev_{t}"] = opt.stdev.numpy().copy()
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()  # costs of the LAST outer iteration
            k = cfg["cem_best_k"]
            out[f"elite_idx_{t}"] = np.stack([a[:k] for a in argsort_log]).astype(np.int64)  # [iters, k]
            out[f"sorted_gap_{t}"] = np.array([float(np.sort(np.asarray(lv["J_logged"]))[k] -
                                                      np.sort(np.asarray(lv["J_logged"]))[k - 1])], np.float32)
            argsort_log.clear()
        elif opt_name in ("cem-naive-grad-tf", "cem-grad-bharadhwaj-tf"):
            out[f"dist_mue_{t}"] = opt.dist_mue.numpy().copy()
            out[f"stdev_{t}"] = opt.stdev.numpy().copy()
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()  # costs of the LAST outer iteration (after the gradient step)
            k = cfg["cem_best_k"]
            out[f"elite_idx_{t}"] = np.stack([a[:k] for a in argsort_log]).astype(np.int64)  # [iters, k]
            out[f"Qn_{t}"] = np.asarray(lv["Q_logged"]).copy()  # the population after the gradient step, last outer iteration
            if opt_name == "cem-grad-bharadhwaj-tf":
                step, m, v = opt.optim.get_weights()
                out[f"adam_m_{t}"] = np.asarray(m).copy()
                out[f"adam_v_{t}"] = np.asarray(v).copy()
                out[f"adam_step_{t}"] = np.array([int(step)], np.int64)
            argsort_log.clear()
        elif opt_name == "random-action-tf":
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()
            out[f"best_idx_{t}"] = np.array([int(argsort_log[-1][0])], np.int64)  # tf.argsort(traj_cost)[0]  (:66-67)
            argsort_log.clear()
        elif opt_name == "gradient-tf":
            step, m, v = opt.optim.get_weights()
            out[f"Q_{t}"] = opt.Q_tf.numpy().copy()  # AFTER the warm-start shift (:136-144)
            out[f"adam_m_{t}"] = np.asarray(m).copy()
            out[f"adam_v_{t}"] = np.asarray(v).copy()
            out[f"adam_step_{t}"] = np.array([int(step)], np.int64)
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()
            out[f"best_idx_{t}"] = np.array([int(argsort_log[-1][0])], np.int64)
            argsort_log.clear()
        elif opt_name == "rpgd":
            step, m, v = opt.opt.get_weights()
            out[f"Q_{t}"] = opt.Q_tf.numpy().copy()
            out[f"adam_m_{t}"] = np.asarray(m).copy()
            out[f"adam_v_{t}"] = np.asarray(v).copy()
            out[f"adam_step_{t}"] = np.array([int(step)], np.int64)
            out[f"ages_{t}"] = opt.trajectory_ages.numpy().copy()
            out[f"J_{t}"] = np.asarray(lv["J_logged"]).copy()
            out[f"u_nom_{t}"] = np.asarray(opt.optimal_control_sequence).copy()
        if keep_rollouts and t == 0:
            out["Q_logged_0"] = np.asarray(lv["Q_logged"]).copy()
            out["rollouts_0"] = np.asarray(lv["rollout_trajectories_logged"]).copy()

    out["noise_blocks"] = np.array(json.dumps(rng.blocks))
    # checksum of the full noise stream, to detect a numpy Generator stream change on another box
    chk = ReplayRNG(NOISE_SEED, as_torch=False)
    acc = 0.0
    for kind, shape in rng.blocks:
        acc += float(np.sum(chk.standard_draws(kind, shape).astype(np.float64)))
    out["noise_checksum"] = np.array([acc], np.float64)

    if opt_name.endswith("-tf"):
        tfshim.argsort = _orig
    return out


def main(argv=None):
    from oracle.refharness.workspace import enter_workspace
    args = list(argv if argv is not None else sys.argv[1:])
    out_dir = GOLDEN
    if "--out" in args:  # write somewhere else (tests/test_oracle_golden.py regenerates fixtures and compares them bit for bit)
        i = args.index("--out")
        out_dir = os.path.abspath(args[i + 1])
        del args[i:i + 2]
    names = args or list(CASES)
    enter_workspace()
    import logging
    logging.disable(logging.INFO)
    os.makedirs(out_dir, exist_ok=True)
    for name in names:
        out = run_reference_case(name)
        path = os.path.join(out_dir, f"{name}.npz")
        np.savez_compressed(path, **out)
        print(f"{name}: wrote {path} ({os.path.getsize(path) / 1024:.1f} KiB)  u0={out['u_0']}")


if __name__ == "__main__":
    main()
