"""CPU tests of the gradient optimizers on registered environments (ctk_kernels_env_rpgd.cuh), no GPU needed:
- the Dubins car's adjoint (ctk_env_adjoint.h, compiled for the host by tests/env_twin) against float64 torch autograd of the oracle's
  DubinsPredictor + DubinsCost;
- the configurations ctk_create refuses before it touches the device;
- the oracles for nu inputs (tests/env_gradient_oracles.py): at nu = 1 the same numbers as oracle/, at nu = 2 their invariants (shapes,
  one gradient norm per trajectory, the moment shift by one time step);
- the shipped gradient kernel's machine code: no spill, no local-memory traffic but the trigonometric slow path."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from control_toolkit_b200 import _lib as L
from control_toolkit_b200 import specs
from oracle import spec
from env_gradient_oracles import CEMBharadhwajOracleNu, CEMNaiveGradOracleNu, GradientOracleNu, RPGDOracleNu
from helpers import load_golden, make_oracle, make_predictor
from oracle.replay_rng import ReplayRNG

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
DT = 0.02


@pytest.fixture(scope="module")
def twin(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("env_twin") / "libdubins_twin.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", os.path.join(HERE, "env_twin", "dubins_twin.cpp"), "-o", out], check=True)
    return C.CDLL(out)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _params():
    _, ode = specs.resolve_predictor("DubinsCar", "ODE")
    return specs.dubins_env_params(ode, specs.resolve_cost("DubinsCar", "default"), DT)


def _autograd(s0, Q, u_prev, dtype):
    pred, cost = spec.DubinsPredictor(spec.DubinsParams(dt=DT)), spec.DubinsCost()
    q = torch.tensor(Q, dtype=dtype, requires_grad=True)
    J = spec.trajectory_cost(pred.predict_core(torch.tensor(s0, dtype=dtype), q), q, torch.tensor(u_prev, dtype=dtype), cost)
    (g,) = torch.autograd.grad(J.sum(), q)
    return g.numpy().astype(np.float64)


def _cases():
    rng = np.random.default_rng(7)
    N, H = 48, 50
    c = spec.DubinsCost()
    out = {}
    s0 = np.stack([rng.uniform(-0.3, 1.2, N), rng.uniform(-0.3, 0.8, N), rng.uniform(-math.pi, math.pi, N)], 1)
    out["random"] = (s0, rng.uniform(-1, 1, (N, H, 2)), rng.uniform(-1, 1, 2))
    # yaw near +-pi: the wrap atan2(sin, cos) is crossed inside the horizon (steer pushes the yaw through pi)
    s0 = np.stack([rng.uniform(-0.2, 0.2, N), rng.uniform(-0.2, 0.2, N), np.where(np.arange(N) % 2 == 0, math.pi - 1e-3, -math.pi + 1e-3)], 1)
    Q = rng.uniform(-1, 1, (N, H, 2))
    Q[:, :, 1] = np.where(np.arange(N)[:, None] % 2 == 0, 0.8, -0.8) + 0.1 * rng.uniform(-1, 1, (N, H))
    out["yaw_wrap"] = (s0, Q, np.zeros(2))
    # straight through the obstacle: the indicator switches on and off along the trajectory
    s0 = np.stack([np.full(N, c.obstacle_x - 0.4), np.full(N, c.obstacle_y) + rng.uniform(-0.1, 0.1, N), np.zeros(N)], 1)
    Q = np.stack([rng.uniform(0.7, 1.0, (N, H)), 0.05 * rng.uniform(-1, 1, (N, H))], 2)
    out["obstacle"] = (s0, Q, rng.uniform(-1, 1, 2))
    return {k: (a.astype(np.float32), b.astype(np.float32), u.astype(np.float32)) for k, (a, b, u) in out.items()}


CASES = _cases()


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("prev", ["zero", "given"])
def test_dubins_adjoint_matches_float64_autograd(twin, case, prev):
    """dJ/dQ of the mean trajectory cost through the hand-written adjoint, both previous-input cases (zero: the state after a
    reset; given: the last applied control).  Bound per element: max(1e-4 x the row's largest |g|, 4 x |fp32 - float64 autograd|).
    Measured (x86-64, g++ -O2): worst error / bound 0.004-0.010, worst |err| / row max 1.0e-6."""
    s0, Q, up = CASES[case]
    if prev == "zero":
        up = np.zeros(2, np.float32)
    N, H = Q.shape[:2]
    p = _params()
    G = np.zeros_like(Q)
    twin.twin_dubins_grad(_fp(np.ascontiguousarray(s0)), _fp(np.ascontiguousarray(Q)), N, H, _fp(up), _fp(p), p.size, _fp(G))
    g64, g32 = _autograd(s0, Q, up, torch.float64), _autograd(s0, Q, up, torch.float32)
    if case == "obstacle":  # the case does reach the obstacle: the stage cost carries the indicator on some steps
        traj = spec.DubinsPredictor(spec.DubinsParams(dt=DT)).predict_core(torch.tensor(s0, dtype=torch.float64), torch.tensor(Q, dtype=torch.float64))
        c = spec.DubinsCost()
        inside = (traj[:, :, 0] - c.obstacle_x) ** 2 + (traj[:, :, 1] - c.obstacle_y) ** 2 < c.obstacle_r ** 2
        assert inside.any(dim=1).float().mean() > 0.5
    row = np.abs(g64).reshape(N, -1).max(1)[:, None, None]
    err = np.abs(G.astype(np.float64) - g64)
    bound = np.maximum(1e-4 * row, 4 * np.abs(g32 - g64))
    worst = float((err / bound).max())
    print(f"{case}/{prev}: max err/bound {worst:.3f}, max err/row max {float((err / row).max()):.2e}")
    assert worst <= 1.0, (case, prev, worst)


# ---- configurations refused before the device ----------------------------------------------------------------------------
ENV = ("environments other than the CartPole: MPPI, CEM and the gradient optimizers with the environment's ODE, unsharded, one client "
       "(the network predictors are CartPole functors)")
RPGD = ("RPGD needs num_rollouts <= 1024 (replicas only, no sharding), the ODE predictor with intermediate_steps == 1 and "
        "1 <= keep_k <= num_rollouts")
TAPE = "environment gradient optimizers: mpc_horizon too large for the shared-memory tape of H * (ns + 4 nu) floats per trajectory (max 164)"
GRADCEM = "gradient-assisted CEM needs 1 <= cem_best_k <= num_rollouts, cem_outer_it >= 1 and inducing-point period 1"


def _create(**over):
    cfg, ode, cost = L.ctk_config(), L.ctk_ode_params(), L.ctk_cost_params()
    cfg.abi_version, cfg.optimizer, cfg.predictor, cfg.device = L.CTK_ABI_VERSION, L.OPT_RPGD, L.PRED_ODE, 0
    cfg.environment, cfg.num_states, cfg.num_control_inputs = L.ENV_DUBINS_CAR, 3, 2
    cfg.num_rollouts = cfg.num_rollouts_global = 32
    cfg.mpc_horizon, cfg.period_interpolation_inducing_points = 50, 10
    cfg.action_low, cfg.action_high = -1.0, 1.0
    cfg.rpgd_outer_its, cfg.rpgd_resamp_per, cfg.rpgd_keep_k = 2, 10, 8
    cfg.cem_outer_it, cfg.cem_best_k = 1, 8
    for k, v in over.items():
        setattr(cfg, k, v)
    ode.intermediate_steps = 1
    cost.kind = L.COST_DEFAULT
    h = C.c_void_p()
    rc = L.load().ctk_create(C.byref(cfg), C.byref(ode), C.byref(cost), C.byref(h))
    if rc == L.CTK_OK:
        L.load().ctk_destroy(h)
    return rc, (L.load().ctk_last_error() or b"").decode()


REJECT = [
    ("horizon_over_tape", dict(mpc_horizon=165), TAPE),
    ("gradient_tf_horizon_over_tape", dict(mpc_horizon=400, period_interpolation_inducing_points=1, rpgd_gradient_mode=1), TAPE),
    ("over_1024_rollouts", dict(num_rollouts=1025, num_rollouts_global=1025, rpgd_keep_k=8), RPGD),
    ("sharded", dict(num_rollouts=16, num_rollouts_global=32), ENV),
    ("multi_client", dict(num_clients=2), ENV),
    ("mlp_predictor", dict(predictor=L.PRED_MLP), ENV),
    ("gru_predictor", dict(predictor=L.PRED_GRU), ENV),
    ("gradcem_period_10", dict(rpgd_gradient_mode=2), GRADCEM),
]


@pytest.mark.parametrize("over,message", [r[1:] for r in REJECT], ids=[r[0] for r in REJECT])
def test_dubins_gradient_config_rejected_before_the_device(over, message):
    rc, err = _create(**over)
    assert rc == L.CTK_EINVAL, err
    assert message in err


@pytest.mark.parametrize("over", [dict(mpc_horizon=164), dict(rpgd_gradient_mode=1, period_interpolation_inducing_points=1),
                                  dict(rpgd_gradient_mode=3, period_interpolation_inducing_points=1)], ids=["largest_horizon", "gradient_tf", "bharadhwaj"])
def test_dubins_gradient_config_passes_the_checks(over):
    """Accepted configurations get past check_config: on a machine without a GPU the first failure is the device query."""
    rc, err = _create(**over)
    assert rc == L.CTK_OK or (rc != L.CTK_EINVAL), err


# ---- the oracles at nu = 2 ---------------------------------------------------------------------------------------------
def _dubins():
    return spec.DubinsPredictor(spec.DubinsParams(dt=DT)), spec.DubinsCost()


LO, HI = np.array([-0.5, -1.0], np.float32), np.array([1.0, 1.0], np.float32)


@pytest.mark.parametrize("fixture", ["rpgd_c3", "rpgd_normal_shift2", "gradient_n40", "gradcem_naive_n200", "gradcem_bharadhwaj_n32"])
def test_nu_oracles_reproduce_the_pinned_oracles_at_one_input(fixture):
    """At nu = 1 the oracles for nu inputs compute exactly what oracle/ computes, which test_oracle_golden.py pins to the fixtures of
    the unmodified reference: same draws, same u, same optimizer state, same costs, tick by tick."""
    from env_gradient_oracles import ORACLES
    z, meta = load_golden(fixture)
    ref = make_oracle(meta)
    new = ORACLES[meta["optimizer"]](make_predictor(meta), spec.CostParams(name=meta["cost"]), **meta["cfg"])
    r_ref, r_new = ReplayRNG(meta["noise_seed"]), ReplayRNG(meta["noise_seed"])
    if meta["optimizer"] in ("rpgd", "gradient-tf"):
        ref.reset(r_ref)
        new.reset(r_new)
    state = {"rpgd": "Q", "gradient-tf": "Q"}.get(meta["optimizer"], "dist_mue")
    for t in range(3):
        u_ref, u_new = ref.step(z["states"][t], r_ref), new.step(z["states"][t], r_new)
        assert np.array_equal(np.ravel(u_ref), np.ravel(u_new)), (fixture, t)
        assert torch.equal(getattr(ref, state), getattr(new, state)), (fixture, t)
        assert np.array_equal(ref.last["J"], new.last["J"]), (fixture, t)
    assert r_ref.blocks == r_new.blocks


def test_rpgd_oracle_nu2_shapes_single_norm_and_moment_shift():
    pred, cost = _dubins()
    o = RPGDOracleNu(pred, cost, mpc_horizon=21, num_rollouts=16, outer_its=2, sample_stdev=0.5, sample_mean=0.0, sample_whole_control_space=True,
                   uniform_dist_min=-1.0, uniform_dist_max=1.0, resamp_per=3, period_interpolation_inducing_points=5, SAMPLING_DISTRIBUTION="uniform",
                   shift_previous=2, warmup=False, warmup_iterations=0, learning_rate=0.05, opt_keep_k_ratio=0.25, gradmax_clip=0.05,
                   adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1e-8, action_low=LO, action_high=HI, adam_form="keras")
    rng = ReplayRNG(3)
    o.reset(rng)
    assert tuple(o.Q.shape) == (16, 21, 2) and rng.blocks[-1] == ("uniform", (16, 5, 2))
    assert (o.Q[:, :, 0] >= -0.5).all() and (o.Q[:, :, 0] <= 1.0).all()  # per-input limits
    s = np.array([0.0, 0.0, 0.3], np.float32)
    # one gradient step with a tiny clip: every trajectory's clipped gradient has norm exactly gradmax_clip over [H, nu] together
    ss = torch.as_tensor(np.tile(s, (16, 1)))
    Q = o.Q.clone().detach().requires_grad_(True)
    J, _ = o._cost(ss, Q)
    (g,) = torch.autograd.grad(J.sum(), Q)
    n = torch.sqrt((g * g).sum(dim=(1, 2)))
    assert (n > 0.05).all()
    Qn, _ = o.grad_step(ss, o.Q)
    m_first = o.m.clone()  # (1 - b1) g_clipped
    assert torch.allclose(torch.sqrt((m_first * m_first).sum(dim=(1, 2))) / 0.1, torch.full((16,), 0.05), rtol=1e-4)
    o.adam_step, o.m, o.v = 0, None, None
    u = o.step(s, rng)
    assert np.shape(u) == (2,) and o.last["Q"].shape == (16, 21, 2) and o.last["u_nom"].shape == (1, 21, 2)
    # tick 0 resamples (count 0 % 3 == 0): rows 12.. are the elites in best order, their moments shifted by ONE time step
    assert o.m.shape == (16, 21, 2) and (o.m[:12] == 0).all() and (o.m[12:, -1, :] == 0).all()
    m_before = m_first  # unused past this point
    del m_before
    u = o.step(s, rng)  # tick 1: no resampling, every row's moments shift by one step with zero fill
    assert (o.m[:, -1, :] == 0).all()


def test_gradient_oracle_nu2_tail_redraw_per_input():
    pred, cost = _dubins()
    o = GradientOracleNu(pred, cost, mpc_horizon=12, num_rollouts=8, gradient_steps=2, learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999,
                       adam_epsilon=1e-7, gradmax_clip=5, warmup=False, warmup_iterations=0, action_low=LO, action_high=HI)
    rng = ReplayRNG(5)
    o.reset(rng)
    assert tuple(o.Q.shape) == (8, 12, 2)
    u = o.step(np.array([0.1, 0.0, -0.2], np.float32), rng)
    assert np.shape(u) == (2,) and rng.blocks[-1] == ("uniform", (8, 1, 2))
    Q_before = torch.as_tensor(o.last["Q"])
    assert torch.equal(o.Q[:, :-1, :], Q_before[:, 1:, :])  # shift by one time step
    assert (o.Q[:, -1, 0] >= -0.5).all() and (o.Q[:, -1, 0] <= 1.0).all()
    assert o.m.shape == (8, 12, 2) and (o.m[:, -1, :] == 0).all()


@pytest.mark.parametrize("cls", [CEMNaiveGradOracleNu, CEMBharadhwajOracleNu])
def test_gradcem_oracles_nu2_refit_per_column(cls):
    pred, cost = _dubins()
    kw = dict(mpc_horizon=10, num_rollouts=24, cem_outer_it=2, cem_initial_action_stdev=0.5, cem_stdev_min=0.01, cem_best_k=6,
              learning_rate=0.05, gradmax_clip=5, action_low=LO, action_high=HI)
    if cls is CEMBharadhwajOracleNu:
        kw.update(adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1e-8)
    o = cls(pred, cost, **kw)
    assert tuple(o.dist_mue.shape) == (1, 10, 2) and torch.allclose(o.dist_mue[0, 0], torch.tensor([0.25, 0.0]))
    u = o.step(np.array([0.0, 0.1, 0.0], np.float32), ReplayRNG(9))
    assert np.shape(u) == (2,) and o.last["Q"].shape == (24, 10, 2)
    assert tuple(o.stdev.shape) == (1, 10, 2) and torch.allclose(o.dist_mue[0, -1], torch.tensor([0.25, 0.0]))  # per-input mid fill


# ---- machine code of the shipped gradient kernel ---------------------------------------------------------------------------
LIB = os.path.join(REPO, "control_toolkit_b200", "libctk_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
KERNEL = "_ZN3ctk20env_rpgd_grad_kernelINS_9DubinsEnvELb0EEEvNS_15EnvRpgdGradArgsENS_14RpgdSelectArgsEi"


@pytest.mark.skipif(not (os.path.exists(LIB) and os.path.exists(CUOBJDUMP)), reason="needs the built library and cuobjdump")
def test_env_gradient_kernel_spills_nothing_and_uses_local_memory_only_in_the_trig_slow_path():
    """Nothing spills.  The only local memory of the kernel is the argument-reduction buffer of the slow path of sincosf / cosf / sinf
    (|yaw| > 105615, never taken: the yaw is wrapped to (-pi, pi]) -- the same 32-byte frame the env MPPI / CEM rollout kernels
    have from the same DubinsEnv::step.  Every LDL / STL must therefore belong to such a reduction: it follows a load of the 2/pi
    table (constant bank 4) within a few instructions, five per reduction.  The reductions sit inside the address range of the
    forward loop (the compiler inlines them behind a branch), so "not inside a loop" is not the criterion; "nothing else" is."""
    res = subprocess.run([CUOBJDUMP, "--dump-resource-usage", LIB], capture_output=True, text=True, check=True).stdout
    block = res[res.index(KERNEL):].splitlines()[1]
    reg, stack = (int(x) for x in re.search(r"REG:(\d+) STACK:(\d+)", block).groups())
    assert reg <= 255 and stack <= 32, block
    sass = subprocess.run([CUOBJDUMP, "-sass", "-fun", KERNEL, LIB], capture_output=True, text=True).stdout
    lines = [ln for ln in sass.splitlines() if re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln)]
    assert len(lines) > 500
    addr = lambda ln: int(re.match(r"\s+/\*([0-9a-f]{4,})\*/", ln).group(1), 16)  # noqa: E731
    local = [addr(ln) for ln in lines if re.search(r"\b(LDL|STL)\b", ln)]
    table = [addr(ln) for ln in lines if re.search(r"\bLDCU?\.64\b.*c\[0x4\]", ln)]
    assert table and len(local) == 5 * len(table), (len(local), len(table))
    for x in local:
        assert any(0 < x - t <= 0x200 for t in table), hex(x)
