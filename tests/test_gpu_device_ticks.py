"""-m gpu: the device-resident tick (ctk_step_device) and back-to-back chains of ticks (ctk_step_device_n) -- the two paths bench.py
times -- against the host tick (ctrl.step -> ctk_step / ctk_step_state), the golden fixtures and the float64 oracle.

The host tick passes the state inside the kernel parameters (S0::v) and returns u through the mapped host mirror; the device tick
reads the state through S0::p and writes [u, status] to device memory.  A chain additionally runs code no other path runs: ticks
1.. of an MPPI/ODE chain skip griddepcontrol.wait and poll u_prev and the shifted u_nom from the previous finisher's tagged
hand-over slots, every tick but the last publishes them, and consecutive ticks are launched as programmatic dependents.

The reference for most checks is a TWIN handle: same config, same seed, same reset -- hence the same Philox tick counter -- running
the same states one tick at a time through the host path.  Both paths launch the same kernel instantiation (asserted) with a fixed
summation order, so the bar is bit-identical: u, status, the whole optimizer state read from the handle, the counters, the
per-rollout costs and (logging on) the logged controls and trajectories.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from gpu_helpers import make_controller, max_rel
from helpers import fp32_noise_floor, golden_names, load_golden, replay
from test_gpu_parity import _check_J, _report, _tols, _u_err
from test_gpu_production_pinning import TOL, _J_floor, _assert_state, _oracles, _state_errs

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U_STRIDE = 4  # floats per tick in the u_out buffers: [u (nu), status] + padding that must stay untouched


def _L():
    from control_toolkit_b200 import _lib as L
    return L, L.load()


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _with_cfg(meta, cfg):
    return dict(meta, cfg=dict(meta["cfg"], **cfg)) if cfg else meta


def _nu(meta):
    return 2 if meta.get("environment", "CartPole") == "DubinsCar" else 1


def _states(meta, z, n, seed):
    """n states: the fixture's own for the Dubins car (3 states), synthetic CartPole states otherwise."""
    from oracle import spec
    if meta.get("environment", "CartPole") == "DubinsCar":
        assert z["states"].shape[0] >= n
        return np.ascontiguousarray(z["states"][:n], np.float32)
    return np.ascontiguousarray(spec.synthetic_states(n, seed=seed), np.float32)


def _snapshot(opt, logging):
    """Everything a tick leaves in the handle, read straight from the C handle (the plugin's Python attributes only follow
    ctrl.step): every state array the optimizer has (a state it does not have is kept as the refusal message, which must be the
    same on both handles), the counters, the per-rollout costs and, with logging on, the logs of the last tick."""
    L, _ = _L()
    N, H, nu, ns = opt._n_local, opt.mpc_horizon, int(opt.num_control_inputs), int(opt.num_states)
    hidden = getattr(getattr(opt, "_mlp_keepalive", None), "hidden", 0)
    sizes = {L.STATE_U_NOM: H * nu, L.STATE_CEM_MU: H * nu, L.STATE_CEM_STD: H * nu, L.STATE_U_PREV: nu, L.STATE_RNN_H: 2 * hidden}
    if opt._OPT == L.OPT_RPGD:  # (the population arrays; gradient-assisted CEM runs on the RPGD handle too)
        sizes.update({L.STATE_RPGD_Q: N * H, L.STATE_RPGD_M: N * H, L.STATE_RPGD_V: N * H, L.STATE_RPGD_AGES: N})
    out = {}
    for which, n in sizes.items():
        try:
            out[f"state {which}"] = opt._get_state(which, (max(n, 1),))
        except ValueError as e:
            out[f"state {which}"] = str(e)
    for c in (L.COUNTER_COUNT, L.COUNTER_ADAM_STEP, L.COUNTER_TICK):
        out[f"counter {c}"] = opt._get_counter(c)
    out["J"] = np.array(opt._get_log(L.LOG_J, (N,)))
    if logging:
        out["Q_logged"] = np.array(opt._get_log(L.LOG_Q, (N, H, nu)))
        out["trajectories"] = np.array(opt._get_log(L.LOG_ROLLOUTS, (N, H + 1, ns)))
    return out


def _assert_same(a, b, tag):
    assert a.keys() == b.keys()
    for k in a:
        if isinstance(a[k], str) or isinstance(b[k], str):
            assert a[k] == b[k], (tag, k, a[k], b[k])
        else:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"{tag}: {k}")


def _main_state(opt):
    """The state array every handle of the optimizer has: MPPI u_nom, CEM dist_mue, RPGD Q (so that a snapshot never compares
    two refusals only)."""
    L, _ = _L()
    return {L.OPT_MPPI: L.STATE_U_NOM, L.OPT_CEM: L.STATE_CEM_MU, L.OPT_RPGD: L.STATE_RPGD_Q}[opt._OPT]


def _writes_status(meta, kernel):
    """Ticks that store a status word after u (include/ctk_b200.h ctk_step_device): the CartPole MPPI tick (its finisher) and the
    one-launch CEM tick; every other tick writes u only."""
    cartpole = meta.get("environment", "CartPole") == "CartPole"
    return cartpole and (meta["optimizer"] == "mppi" or kernel.startswith("cem_tick_kernel"))


def _check_u_rows(meta, kernel, rows, u_host, tag):
    """rows [K, U_STRIDE] from the device path (prefilled with NaN) against the twin's host-path controls."""
    nu = _nu(meta)
    for i, (row, u) in enumerate(zip(rows, u_host)):
        np.testing.assert_array_equal(row[:nu], np.ravel(u).astype(np.float32), err_msg=f"{tag}: u of tick {i}")
        if _writes_status(meta, kernel):
            assert row[nu] == 0.0, (tag, i, row)
            assert np.isnan(row[nu + 1:]).all(), (tag, i, row)
        else:
            assert np.isnan(row[nu:]).all(), (tag, i, row)


# ---------------------------------------------------------------------------------------------------------------------
# 1. one device tick == one host tick
# ---------------------------------------------------------------------------------------------------------------------
TICK_CASES = [
    # id, fixture for the config, config overrides, make_controller options, environment
    ("mppi_ode_c1", "mppi_c1_n2000", {}, {}, {}),
    ("mppi_ode_1m", "mppi_h100_n256", {"num_rollouts": 1_000_000, "mpc_horizon": 100}, {}, {}),
    ("mppi_ode_1m_log_reduced", "mppi_h100_n256", {"num_rollouts": 20_000, "mpc_horizon": 100}, {"logging": True}, {}),
    ("cem_ode_c2", "cem_c2_n4096_k64", {}, {}, {}),
    ("cem_ode_c2_multi_launch", "cem_c2_n4096_k64", {}, {}, {"CTK_CEM_MULTI_LAUNCH": "1"}),
    ("cem_ode_large", "cem_c2_n4096_k64", {"num_rollouts": 1_000_000}, {}, {}),
    ("rpgd_ode_c3", "rpgd_c3", {}, {}, {}),
    ("rpgd_n64_multi_launch", "rpgd_c3", {"num_rollouts": 64}, {}, {}),
    ("mppi_mlp_c4_tcgen05", "mppi_mlp_c4_n256", {"num_rollouts": 65536, "mpc_horizon": 100}, {"mlp_engine": "tcgen05"}, {}),
    ("mppi_mlp_c4_simt", "mppi_mlp_c4_n256", {"num_rollouts": 65536, "mpc_horizon": 100}, {"mlp_engine": "simt"}, {}),
    ("gradient_tf", "gradient_n40", {}, {}, {}),
    ("cem_naive_grad_tf", "gradcem_naive_n200", {}, {}, {}),
    ("cem_grad_bharadhwaj_tf", "gradcem_bharadhwaj_n32", {}, {}, {}),
    ("random_action_tf", "random_action_n512", {}, {}, {}),
    ("mppi_gru", "mppi_gru_n256", {}, {}, {}),
    ("cem_gru", "cem_gru_n256_k16", {}, {}, {}),
    ("mppi_dubins", "mppi_dubins_n512", {}, {}, {}),
    ("cem_dubins", "cem_dubins_n512_k32", {}, {}, {}),
]
ONE_LAUNCH_TICKS = {"mppi_ode_c1", "mppi_ode_1m", "cem_ode_c2", "rpgd_ode_c3"}


@pytest.mark.parametrize("cid,fixture,cfg,kw,env", TICK_CASES, ids=[c[0] for c in TICK_CASES])
def test_device_tick_equals_host_tick(monkeypatch, cid, fixture, cfg, kw, env):
    """ctk_step_device (state read through S0::p, [u, status] to device memory) against ctrl.step on a twin handle, tick by tick,
    bit for bit.  The state of each tick is written on the handle's stream right before the call, into a buffer that held NaN."""
    import torch
    L, lib = _L()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    z, meta = load_golden(fixture)
    meta = _with_cfg(meta, cfg)
    kw = dict(kw)
    logging = kw.pop("logging", False)
    dev = make_controller(meta, rng=None, logging=logging, **kw)
    twin = make_controller(meta, rng=None, logging=logging, **kw)
    opt = dev.optimizer
    states = _states(meta, z, 3, seed=51)
    stream = torch.cuda.Stream(device=0)
    L.check(lib.ctk_set_stream(opt._h, C.c_void_p(stream.cuda_stream)))
    src = torch.from_numpy(states).cuda()
    s_dev = torch.full((states.shape[1],), float("nan"), device="cuda")
    u_dev = torch.full((U_STRIDE,), float("nan"), device="cuda")
    torch.cuda.synchronize()
    for t in range(3):
        l0, m0 = opt.gpu_launches, twin.optimizer.gpu_launches
        with torch.cuda.stream(stream):
            s_dev.copy_(src[t])  # the tick must see this write: it precedes the launch on the same stream
            u_dev.fill_(float("nan"))
            L.check(lib.ctk_step_device(opt._h, _ptr(s_dev), _ptr(u_dev)))
            if logging:
                opt._collect_rollout_logs(opt._n_local)  # the log reads the host tick's step() makes (layout transposes)
        stream.synchronize()
        launches = opt.gpu_launches - l0
        u_t = twin.step(states[t])
        assert opt.last_kernel == twin.optimizer.last_kernel, (opt.last_kernel, twin.optimizer.last_kernel)
        assert launches == twin.optimizer.gpu_launches - m0, (cid, t, launches, twin.optimizer.gpu_launches - m0)
        if cid in ONE_LAUNCH_TICKS:
            assert launches == 1, (cid, t, launches, opt.last_kernel)
        _check_u_rows(meta, opt.last_kernel, u_dev.cpu().numpy()[None], [u_t], f"{cid} tick {t}")
        a, b = _snapshot(opt, logging), _snapshot(twin.optimizer, logging)
        assert not isinstance(a[f"state {_main_state(opt)}"], str)
        _assert_same(a, b, f"{cid} tick {t} [{opt.last_kernel}]")
    _report(f"device tick {cid} [{opt.last_kernel}]: 3 ticks bit-identical to the host tick, {launches} launch(es) per tick")


# ---------------------------------------------------------------------------------------------------------------------
# 2. a chain == one tick at a time
# ---------------------------------------------------------------------------------------------------------------------
def _chain(opt, states, on_stream=False, u_stride=U_STRIDE):
    """ctk_step_device_n over states [K, ns] -> (u rows [K, u_stride], launches of the chain).  on_stream: the states are written on
    the handle's stream right before the call (into a buffer that held NaN), and nothing synchronises in between."""
    import torch
    L, lib = _L()
    K, ns = states.shape
    u_dev = torch.full((K, u_stride), float("nan"), device="cuda")
    l0 = opt.gpu_launches
    if on_stream:
        stream = torch.cuda.Stream(device=0)
        L.check(lib.ctk_set_stream(opt._h, C.c_void_p(stream.cuda_stream)))
        src = torch.from_numpy(states).cuda()
        s_dev = torch.full((K, ns), float("nan"), device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            s_dev.copy_(src)
            L.check(lib.ctk_step_device_n(opt._h, _ptr(s_dev), ns, _ptr(u_dev), u_stride, K))
        stream.synchronize()
    else:
        s_dev = torch.from_numpy(states).cuda()
        torch.cuda.synchronize()
        L.check(lib.ctk_step_device_n(opt._h, _ptr(s_dev), ns, _ptr(u_dev), u_stride, K))
        torch.cuda.synchronize()
    return u_dev.cpu().numpy(), opt.gpu_launches - l0


def _twin_ticks(twin, states):
    """The same states through the host path, one tick at a time -> (controls, launches of the ticks)."""
    m0 = twin.optimizer.gpu_launches
    u = [twin.step(s) for s in states]
    return u, twin.optimizer.gpu_launches - m0


def _chain_vs_twin(meta, states, tag, on_stream=False, logging=False, one_launch=False, **kw):
    dev = make_controller(meta, rng=None, logging=logging, **kw)
    twin = make_controller(meta, rng=None, logging=logging, **kw)
    rows, launches = _chain(dev.optimizer, states, on_stream=on_stream)
    kernel = dev.optimizer.last_kernel
    u, twin_launches = _twin_ticks(twin, states)
    assert kernel == twin.optimizer.last_kernel, (tag, kernel, twin.optimizer.last_kernel)
    _check_u_rows(meta, kernel, rows, u, tag)
    if not logging:  # (with logging on, the twin's step() also reads the logs back through layout-transpose launches)
        assert launches == twin_launches, (tag, launches, twin_launches)
    if one_launch:
        assert launches == len(states), (tag, launches, kernel)
    _assert_same(_snapshot(dev.optimizer, logging), _snapshot(twin.optimizer, logging), f"{tag} [{kernel}] after the chain")
    return dev, twin, rows


CHAIN_CASES = [
    # id, fixture, config overrides, options, environment, K, expected kernel (regular expression)
    ("c1", "mppi_c1_n2000", {}, {}, {}, 8, r"mppi_ode_kernel<0,0,10,1,1024,0>"),
    ("c1_ilp2", "mppi_c1_n2000", {}, {}, {"CTK_K1_ILP": "2"}, 8, r"mppi_ode_kernel<0,0,10,2,896,0>"),
    ("c1_period7", "mppi_c1_n2000", {"period_interpolation_inducing_points": 7}, {}, {}, 6, r"mppi_ode_kernel<0,0,0,1,1024,0>"),
    ("ragged_n30011_h97", "mppi_h100_n256", {"num_rollouts": 30011, "mpc_horizon": 97}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,\d,\d+,0>"),
    ("full_grid_n125000", "mppi_h100_n256", {"num_rollouts": 125_000, "mpc_horizon": 100}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,\d,\d+,0>"),
    ("c5_n1m", "mppi_h100_n256", {"num_rollouts": 1_000_000, "mpc_horizon": 100}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,2,896,0>"),
    ("h300_over_the_block", "mppi_c1_n64", {"num_rollouts": 256, "mpc_horizon": 300}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,1,1024,0>"),
    ("n1_h1", "mppi_c1_n64", {"num_rollouts": 1, "mpc_horizon": 1}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,1,1024,0>"),
    ("n33_h2", "mppi_c1_n64", {"num_rollouts": 33, "mpc_horizon": 2}, {}, {}, 4, r"mppi_ode_kernel<0,0,10,1,1024,0>"),
    ("quadratic_boundary_grad", "mppi_c1_n2000", {}, {"cost": "quadratic_boundary_grad"}, {}, 6, r"mppi_ode_kernel<1,0,10,1,1024,0>"),
    ("freeze_previous_input", "mppi_c1_n2000", {}, {"freeze_previous_input": True}, {}, 6, r"mppi_ode_kernel<0,0,10,1,1024,0>"),
    ("logging_n4000", "mppi_c1_n2000", {"num_rollouts": 4000, "mpc_horizon": 50}, {"logging": True}, {}, 4, r"mppi_ode_kernel<0,1,10,1,1024,0>"),
]


@pytest.mark.parametrize("cid,fixture,cfg,kw,env,K,kernel", CHAIN_CASES, ids=[c[0] for c in CHAIN_CASES])
def test_mppi_ode_chain_equals_single_ticks(monkeypatch, cid, fixture, cfg, kw, env, K, kernel):
    """Every row of the chain's u_out (u and status), then the whole state, the counters, the costs and the last tick's logs, against
    K host ticks of a twin.  Ticks 1.. of the chain take u_prev and the shifted u_nom from the hand-over of the tick before: the
    cases reach the unrolled and runtime periods, ragged shares, the full grid with the finisher's reduced share, a horizon longer
    than the block (the poll loop makes several passes), min(t + 1, H - 1) at H = 1 and 2, the boundary-gradient cost, the frozen
    previous input and the logging instantiation."""
    from oracle import spec
    L, lib = _L()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    z, meta = load_golden(fixture)
    meta = _with_cfg(meta, cfg)
    kw = dict(kw)
    if "cost" in kw:
        meta = dict(meta, cost=kw.pop("cost"))
    logging = kw.pop("logging", False)
    states = np.ascontiguousarray(spec.synthetic_states(K, seed=52), np.float32)
    dev, twin, rows = _chain_vs_twin(meta, states, f"chain {cid}", on_stream=cid.startswith("c1"), logging=logging, one_launch=True, **kw)
    assert re.fullmatch(kernel, dev.optimizer.last_kernel), dev.optimizer.last_kernel
    if cid == "h300_over_the_block":  # K1 geometry (ctk_engine.cu mppi_ode_geometry): 2 blocks of 128 threads for 300 hand-over slots
        grid = C.c_int()
        L.check(lib.ctk_debug_trace(dev.optimizer._h, 0, None, 0, C.byref(grid)))
        assert grid.value == 2, grid.value
    if cid == "freeze_previous_input":  # u_prev stays 0, so the hand-over slot 0 must be u_prev, not the new u_nom[0]
        assert float(dev.optimizer._get_state(L.STATE_U_PREV, (1,))[0]) == 0.0 and np.abs(rows[:, 0]).max() > 0.0
    _report(f"chain {cid} K={K} [{dev.optimizer.last_kernel}]: bit-identical to {K} single ticks")


OTHER_CHAIN_CASES = [
    # id, fixture, config overrides, options, environment
    ("mlp_tcgen05", "mppi_mlp_c4_n256", {"num_rollouts": 16384, "mpc_horizon": 100}, {"mlp_engine": "tcgen05"}, {}),
    ("mlp_simt", "mppi_mlp_c4_n256", {"num_rollouts": 4096, "mpc_horizon": 100}, {"mlp_engine": "simt"}, {}),
    ("mppi_gru", "mppi_gru_n256", {}, {}, {}),
    ("cem_persistent", "cem_c2_n4096_k64", {}, {}, {}),
    ("cem_multi_launch", "cem_c2_n4096_k64", {}, {}, {"CTK_CEM_MULTI_LAUNCH": "1"}),
    ("rpgd_one_launch", "rpgd_c3", {}, {}, {}),
    ("rpgd_multi_launch", "rpgd_c3", {"num_rollouts": 64}, {}, {}),
    ("mppi_dubins", "mppi_dubins_n512", {}, {}, {}),
    ("cem_dubins", "cem_dubins_n512_k32", {}, {}, {}),
]


@pytest.mark.parametrize("cid,fixture,cfg,kw,env", OTHER_CHAIN_CASES, ids=[c[0] for c in OTHER_CHAIN_CASES])
def test_other_chains_equal_single_ticks(monkeypatch, cid, fixture, cfg, kw, env):
    """Chains of the handles without a hand-over (network predictors -- the GRU's update launch sits between the ticks --, CEM, RPGD,
    the Dubins car): consecutive ticks are programmatic dependents on one stream and must still equal single host ticks."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    z, meta = load_golden(fixture)
    meta = _with_cfg(meta, cfg)
    K = 3 if meta.get("environment") == "DubinsCar" else 5
    states = _states(meta, z, K, seed=53)
    dev, _, _ = _chain_vs_twin(meta, states, f"chain {cid}", one_launch=cid in ("cem_persistent", "rpgd_one_launch"), **kw)
    _report(f"chain {cid} K={K} [{dev.optimizer.last_kernel}]: bit-identical to {K} single ticks")


def _c1_meta():
    return load_golden("mppi_c1_n2000")[1]


def test_chain_of_zero_one_and_invalid_ticks():
    """n = 0 is a no-op, n = 1 is one tick, n < 0 and a null state pointer are refused and count no tick."""
    import torch
    from oracle import spec
    L, lib = _L()
    meta = _c1_meta()
    dev = make_controller(meta, rng=None, logging=False)
    twin = make_controller(meta, rng=None, logging=False)
    opt = dev.optimizer
    s_dev = torch.from_numpy(np.ascontiguousarray(spec.synthetic_states(2, seed=54), np.float32)).cuda()
    u_dev = torch.full((2, U_STRIDE), float("nan"), device="cuda")
    torch.cuda.synchronize()
    t0, l0 = opt.tick_counter, opt.gpu_launches
    assert lib.ctk_step_device_n(opt._h, _ptr(s_dev), 6, _ptr(u_dev), U_STRIDE, 0) == L.CTK_OK
    assert lib.ctk_step_device_n(opt._h, _ptr(s_dev), 6, _ptr(u_dev), U_STRIDE, -1) == L.CTK_EINVAL
    assert lib.ctk_step_device_n(opt._h, None, 6, _ptr(u_dev), U_STRIDE, 1) == L.CTK_EINVAL
    assert (opt.tick_counter, opt.gpu_launches) == (t0, l0)
    assert np.isnan(u_dev.cpu().numpy()).all()
    states = s_dev.cpu().numpy()
    rows, launches = _chain(opt, states[:1])
    u, _ = _twin_ticks(twin, states[:1])
    assert launches == 1 and opt.tick_counter == t0 + 1
    _check_u_rows(meta, opt.last_kernel, rows, u, "chain n=1")
    _assert_same(_snapshot(opt, False), _snapshot(twin.optimizer, False), "chain n=1")


def test_chain_strides_and_no_u_out():
    """States 8 floats apart (the gaps hold NaN), results 4 floats apart, then a chain with u_out_dev = NULL (results only in the
    state)."""
    import torch
    from oracle import spec
    L, lib = _L()
    meta = _c1_meta()
    dev = make_controller(meta, rng=None, logging=False)
    twin = make_controller(meta, rng=None, logging=False)
    opt = dev.optimizer
    K = 5
    states = np.ascontiguousarray(spec.synthetic_states(2 * K, seed=55), np.float32)
    padded = np.full((2 * K, 8), np.nan, np.float32)
    padded[:, :6] = states
    s_dev = torch.from_numpy(padded).cuda()
    u_dev = torch.full((K, 4), float("nan"), device="cuda")
    torch.cuda.synchronize()
    L.check(lib.ctk_step_device_n(opt._h, _ptr(s_dev), 8, _ptr(u_dev), 4, K))
    torch.cuda.synchronize()
    u, _ = _twin_ticks(twin, states[:K])
    _check_u_rows(meta, opt.last_kernel, u_dev.cpu().numpy(), u, "chain s_stride 8 u_stride 4")
    L.check(lib.ctk_step_device_n(opt._h, C.c_void_p(s_dev[K:].data_ptr()), 8, None, 4, K))
    torch.cuda.synchronize()
    _twin_ticks(twin, states[K:])
    _assert_same(_snapshot(opt, False), _snapshot(twin.optimizer, False), "chain with u_out_dev = NULL")


def test_two_chains_back_to_back_without_synchronisation():
    """Two chains enqueued one after the other with nothing in between: the second chain's first tick is not a polling tick and
    must wait for the first chain's last tick through the stream."""
    import torch
    from oracle import spec
    L, lib = _L()
    meta = _c1_meta()
    dev = make_controller(meta, rng=None, logging=False)
    twin = make_controller(meta, rng=None, logging=False)
    opt = dev.optimizer
    states = np.ascontiguousarray(spec.synthetic_states(9, seed=56), np.float32)
    s_dev = torch.from_numpy(states).cuda()
    u_dev = torch.full((9, U_STRIDE), float("nan"), device="cuda")
    torch.cuda.synchronize()
    L.check(lib.ctk_step_device_n(opt._h, _ptr(s_dev), 6, _ptr(u_dev), U_STRIDE, 4))
    L.check(lib.ctk_step_device_n(opt._h, C.c_void_p(s_dev[4:].data_ptr()), 6, C.c_void_p(u_dev[4:].data_ptr()), U_STRIDE, 5))
    torch.cuda.synchronize()
    u, _ = _twin_ticks(twin, states)
    _check_u_rows(meta, opt.last_kernel, u_dev.cpu().numpy(), u, "two chains back to back")
    _assert_same(_snapshot(opt, False), _snapshot(twin.optimizer, False), "two chains back to back")


@pytest.mark.parametrize("between", ["set_state", "host_step"])
def test_chain_state_change_chain(between):
    """A chain, then set_state(u_nom, u) or a host ctrl.step on the same handle, then a chain: the second chain's first tick must
    read the new u_nom / u_prev from the state, not the stale hand-over of the first chain's last tick."""
    from oracle import spec
    meta = _c1_meta()
    dev = make_controller(meta, rng=None, logging=False)
    twin = make_controller(meta, rng=None, logging=False)
    opt = dev.optimizer
    states = np.ascontiguousarray(spec.synthetic_states(9, seed=57), np.float32)
    rows1, _ = _chain(opt, states[:4])
    u1, _ = _twin_ticks(twin, states[:4])
    if between == "set_state":
        new = {"u_nom": np.linspace(-0.7, 0.6, opt.mpc_horizon, dtype=np.float32).reshape(1, -1, 1), "u": -0.25}
        opt.set_state(new)
        twin.optimizer.set_state(new)
    else:
        np.testing.assert_array_equal(np.ravel(dev.step(states[4])), np.ravel(twin.step(states[4])))
    rows2, _ = _chain(opt, states[5:])
    u2, _ = _twin_ticks(twin, states[5:])
    _check_u_rows(meta, opt.last_kernel, np.concatenate([rows1, rows2]), u1 + u2, f"chain, {between}, chain")
    _assert_same(_snapshot(opt, False), _snapshot(twin.optimizer, False), f"chain, {between}, chain")


# ---------------------------------------------------------------------------------------------------------------------
# 3. chains against the reference fixtures (injected noise) and the float64 oracle (in-kernel noise)
# ---------------------------------------------------------------------------------------------------------------------
_ODE_FIXTURE_KERNEL = r"mppi_ode_kernel<\d,0,0,1,1024,1>"  # injected-noise instantiation: runtime period, one rollout per thread


@pytest.mark.parametrize("name", golden_names("mppi_"))
def test_chain_matches_reference_golden(name):
    """The draws of every tick are queued up front (the (kind, shape) blocks optimizer_mppi.step feeds), then the fixture's states
    run as ONE ctk_step_device_n call (two around controller_reset for the reset fixture).  Each tick's u and the final u_nom against
    the fixture with the tolerances of test_mppi_matches_reference_golden, the last tick's costs with _check_J, and the whole run
    bit-identical to the per-tick replay on the host path."""
    import torch
    L, lib = _L()
    z, meta = load_golden(name)
    T, reset_at = meta["ticks"], meta.get("reset_before_tick", -1)
    dev = make_controller(meta, rng=None, logging=False)
    twin = make_controller(meta, logging=False)  # replay rng: the host path, one tick at a time
    opt = dev.optimizer
    nu, ns = _nu(meta), int(opt.num_states)
    rng = replay(meta)
    for _ in range(T):
        d = np.ascontiguousarray(rng.standard_draws("normal", (opt.num_rollouts, opt.number_of_interpolation_inducing_points, nu)),
                                 np.float32).ravel()
        L.check(lib.ctk_push_injected_noise(opt._h, L.fptr(d), d.size))
    states = np.ascontiguousarray(z["states"][:T], np.float32)
    s_dev = torch.from_numpy(states).cuda()
    u_dev = torch.full((T, U_STRIDE), float("nan"), device="cuda")
    torch.cuda.synchronize()
    cuts = [0, reset_at, T] if reset_at > 0 else [0, T]
    for a, b in zip(cuts[:-1], cuts[1:]):
        if a == reset_at:
            dev.controller_reset()
        L.check(lib.ctk_step_device_n(opt._h, C.c_void_p(s_dev[a:].data_ptr()), ns, C.c_void_p(u_dev[a:].data_ptr()), U_STRIDE, b - a))
        torch.cuda.synchronize()
    rows = u_dev.cpu().numpy()
    if meta["predictor"] == "ODE" and meta.get("environment", "CartPole") == "CartPole":
        assert re.fullmatch(_ODE_FIXTURE_KERNEL, opt.last_kernel), opt.last_kernel
    floors = fp32_noise_floor(name)
    u_twin = []
    for t in range(T):
        if t == reset_at:
            twin.controller_reset()
        u_twin.append(twin.step(z["states"][t], time=0.02 * t))
        tol_s, tol_u, _ = _tols(floors[t], name)
        e_u = _u_err(rows[t, :nu], z[f"u_{t}"], z[f"u_nom_{t}"])
        _report(f"test_chain_matches_reference_golden[{name}] tick {t}: u {e_u:.2e} | fp32 floor: state {floors[t]['state']:.2e}")
        assert e_u < tol_u, (name, t, e_u, floors[t])
    assert opt.last_kernel == twin.optimizer.last_kernel
    _check_u_rows(meta, opt.last_kernel, rows, u_twin, f"golden chain {name}")
    snap = _snapshot(opt, False)
    _assert_same(snap, _snapshot(twin.optimizer, False), f"golden chain {name}")
    tol_s, _, _ = _tols(floors[T - 1], name)
    e_nom = max_rel(snap[f"state {L.STATE_U_NOM}"], z[f"u_nom_{T - 1}"])
    _report(f"test_chain_matches_reference_golden[{name}] final u_nom {e_nom:.2e} [{opt.last_kernel}]")
    assert e_nom < tol_s, (name, e_nom, floors[T - 1])
    _check_J(snap["J"], z[f"J_{T - 1}"], floors[T - 1], (f"test_chain_matches_reference_golden[{name}]", T - 1))


def test_chain_matches_float64_oracle_in_kernel_noise(monkeypatch):
    """C1 (N = 2000, H = 50, period 10) on the production ILP-2 kernel with in-kernel Philox noise: a K = 3 chain against the fp32 and
    float64 oracles stepped through the same states on the exported draws without resynchronising (as the free-running twin of
    test_mppi_production_kernel_matches_oracle).  Catches a bug the chain and the single tick would share."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    from oracle.replay_rng import QueueRNG
    monkeypatch.setenv("CTK_K1_ILP", "2")
    meta = _c1_meta()
    kernel = "mppi_ode_kernel<0,0,10,2,896,0>"
    dev = make_controller(meta, rng=None, logging=False)
    first = make_controller(meta, rng=None, logging=False)  # the chain's tick 0 on its own: its state after that tick
    opt = dev.optimizer
    N, n_ind, K = opt.num_rollouts, opt.number_of_interpolation_inducing_points, 3
    o32, o64 = _oracles(meta)
    states = np.ascontiguousarray(spec.synthetic_states(K, seed=31), np.float32)  # tick 0: the state the production pinning test holds to 1e-5
    t0 = opt.tick_counter
    rows, launches = _chain(opt, states)
    rows0, _ = _chain(first.optimizer, states[:1])
    assert opt.last_kernel == kernel and first.optimizer.last_kernel == kernel, (opt.last_kernel, first.optimizer.last_kernel)
    assert launches == K and rows[0, 0] == rows0[0, 0]
    tag = "test_chain_matches_float64_oracle_in_kernel_noise"
    for i in range(K):
        zi = opt.export_philox(L.STREAM_MPPI, t0 + 1 + i, n_ind, N)  # tick i of the chain ran with counter t0 + 1 + i
        u32 = o32.step_chunked(states[i], QueueRNG([zi]))
        o64.step_chunked(states[i], QueueRNG([zi]))
        scale = max(float(np.abs(o32.u_nom.numpy()).max()), 1e-2)
        e_u = abs(float(rows[i, 0]) - float(np.ravel(u32)[0])) / scale
        _report(f"{tag} tick {i}: u {e_u:.2e}")
        assert rows[i, 1] == 0.0
        if i == 0:
            got = first.optimizer._get_state(L.STATE_U_NOM, (opt.mpc_horizon,))
            e32, e64, floor = _state_errs(got, o32.u_nom.numpy(), o64.u_nom.numpy())
            _assert_state(f"{tag} tick 0 u_nom", e32, e64, floor, True)
            assert e_u < TOL, e_u
            _check_J(first.optimizer._get_log(L.LOG_J, (N,)), o32.last["J"], _J_floor(o32.last["J"], o64.last["J"]), (tag, 0))
        else:
            assert e_u < 1e-4, (i, e_u)
    e32, e64, floor = _state_errs(opt._get_state(L.STATE_U_NOM, (opt.mpc_horizon,)), o32.u_nom.numpy(), o64.u_nom.numpy())
    _report(f"{tag} tick {K - 1} (free-running) u_nom: |cuda-ref32| {e32:.2e} |cuda-f64| {e64:.2e} | floor |ref32-f64| {floor:.2e}")
    assert e32 < 1e-4, e32


# ---------------------------------------------------------------------------------------------------------------------
# 4. hand-over and PDL switched off (read once per process: child processes)
# ---------------------------------------------------------------------------------------------------------------------
def _baseline_chains():
    """The C1 chain and the frozen-previous-input chain: their u rows, and the state after them."""
    from control_toolkit_b200 import _lib as L
    from oracle import spec
    out = {}
    for tag, kw in (("c1", {}), ("freeze", {"freeze_previous_input": True})):
        ctrl = make_controller(_c1_meta(), rng=None, logging=False, **kw)
        rows, _ = _chain(ctrl.optimizer, np.ascontiguousarray(spec.synthetic_states(8, seed=59), np.float32))
        out[f"{tag}_u"] = rows
        out[f"{tag}_u_nom"] = ctrl.optimizer._get_state(L.STATE_U_NOM, (ctrl.optimizer.mpc_horizon,))
        out[f"{tag}_u_prev"] = ctrl.optimizer._get_state(L.STATE_U_PREV, (1,))
        out[f"{tag}_J"] = np.array(ctrl.optimizer._get_log(L.LOG_J, (ctrl.optimizer.num_rollouts,)))
    return out


_CHILD = """
import os, sys
import numpy as np
repo, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [repo, os.path.join(repo, "tests")]
from test_gpu_device_ticks import _baseline_chains
for k, v in _baseline_chains().items():
    np.save(os.path.join(out, k + ".npy"), v)
"""


@pytest.mark.parametrize("switch", ["CTK_NO_HANDOVER", "CTK_NO_PDL"])
def test_chain_without_handover_or_pdl_is_bit_identical(tmp_path, switch):
    """The same chains in a child process with the hand-over (ticks wait for the previous launch through griddepcontrol.wait) or the
    programmatic dependent launches switched off: bit-identical to this process's default run."""
    for k in ("CTK_NO_HANDOVER", "CTK_NO_PDL"):
        assert k not in os.environ, k  # the default run below must have both on
    env = dict(os.environ, **{switch: "1"})
    r = subprocess.run([sys.executable, "-c", _CHILD, REPO, str(tmp_path)], env=env, cwd=REPO, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    here = _baseline_chains()
    for k, v in here.items():
        np.testing.assert_array_equal(np.load(tmp_path / (k + ".npy")), v, err_msg=f"{switch}: {k}")
    _report(f"test_chain_without_handover_or_pdl_is_bit_identical[{switch}]: C1 and freeze chains bit-identical to the default")


# ---------------------------------------------------------------------------------------------------------------------
# 5. two GPUs: chained shards through the fused exchange
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("over", [{}, {"num_rollouts": 40_000, "mpc_horizon": 11}], ids=["c1", "n40000_h11_unstaged"])
def test_fused_exchange_two_shards_chained(over):
    """The fused cross-GPU exchange of test_fused_exchange_two_shards_one_launch_each, driven by ctk_step_device_n (K = 4, one call
    per shard) on GPU 0 and GPU 1.  Never on one GPU: chained shards spin-wait on each other's records and hand-over."""
    import torch
    from oracle import spec
    from test_gpu_parity import _FixedShard
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L, lib = _L()
    meta = _with_cfg(_c1_meta(), over)
    K = 4
    H = meta["cfg"]["mpc_horizon"]
    states = np.ascontiguousarray(spec.synthetic_states(K, seed=60), np.float32)
    full = make_controller(meta, rng=None, logging=False)
    rows_full, _ = _chain(full.optimizer, states)
    devs = [0, 1]
    shards = [make_controller(meta, rng=None, logging=False, shard=_FixedShard(r, 2), device_index=devs[r]).optimizer for r in range(2)]
    streams = [torch.cuda.Stream(device=d) for d in devs]
    boxes = (C.c_void_p * 2)()
    for r, o in enumerate(shards):
        L.check(lib.ctk_set_stream(o._h, C.c_void_p(streams[r].cuda_stream)))
        p = C.c_void_p()
        L.check(lib.ctk_exchange_mailbox(o._h, C.byref(p)))
        boxes[r] = p.value
    dv = (C.c_int * 2)(*devs)
    for r, o in enumerate(shards):
        L.check(lib.ctk_exchange_connect_ptrs(o._h, r, 2, boxes, dv))
    s_dev = [torch.from_numpy(states).to(f"cuda:{d}") for d in devs]
    u_dev = [torch.full((K, U_STRIDE), float("nan"), device=f"cuda:{d}") for d in devs]
    for d in devs:
        torch.cuda.synchronize(d)
    for r, o in enumerate(shards):
        L.check(lib.ctk_step_device_n(o._h, _ptr(s_dev[r]), 6, _ptr(u_dev[r]), U_STRIDE, K))
    for d in devs:
        torch.cuda.synchronize(d)
    us = [u.cpu().numpy() for u in u_dev]
    np.testing.assert_array_equal(us[0][:, 0], us[1][:, 0])
    assert (us[0][:, 1] == 0.0).all() and (us[1][:, 1] == 0.0).all(), us
    a, b = shards[0]._get_state(L.STATE_U_NOM, (H,)), shards[1]._get_state(L.STATE_U_NOM, (H,))
    np.testing.assert_array_equal(a, b)
    e = float(np.abs(us[0][:, 0] - rows_full[:, 0]).max())
    _report(f"test_fused_exchange_two_shards_chained {over}: K={K} shards vs unsharded chain: u {e:.2e}")
    assert e < 2e-6, (us[0][:, 0], rows_full[:, 0])
    assert np.abs(a - full.optimizer._get_state(L.STATE_U_NOM, (H,))).max() < 2e-6
