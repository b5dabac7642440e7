#!/usr/bin/env python
"""bench.py -- rollout-steps/s of the batched MPC rollout hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload mppi_ode_1m|...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Own arm ("ours"): one step = one MPPI tick (sample -> rollout -> cost -> softmin update) over the configured rollout
population.  Default workload = BASELINE.json configs[4]: MPPI, 1,000,000 rollouts x horizon 100, ODE CartPole,
in-kernel Philox noise, sharded by sample over the N GPUs ("strong" scaling: the population is fixed at 1M).
  value    : N_global*H / device time per tick, states already resident in HBM, CUDA events on the launching stream,
             max over ranks.
  e2e      : the same metric through the public plugin API (controller_mpc.step with a HOST state, H2D + D2H inside).
  roofline : the fused rollout kernel (K1) against the measured FP32 FMA-chain peak (the kernel is FP32-pipe bound:
             < 1 byte of HBM traffic per rollout-step), algorithmic 80 FLOP per rollout-step (DESIGN.md).
  cpu_baseline : the oracle port of the reference's MPPI (torch-CPU fp32, all host threads) on a bounded sample.
Reference arm (--impl reference): the reference's UNMODIFIED optimizer file through controller_mpc and the oracle/refharness shims
where CTK_REFERENCE names a checkout of the original Control_Toolkit, the oracle port where it does not (cpu_baseline.kind says which),
timed on the host cores, K steps of a bounded sample each; under torchrun rank 0 alone runs it.
--dump-outputs DIR (own arm): after the K timed ticks, rank 0 writes what the last of them computed to DIR/<name>.npy (see
timed_path_outputs).  Inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every worker; the CPU baseline / reference arm (rank 0 only) must be allowed to
# use all host cores, and the variable is read when numpy / torch are imported -- so fix it up before those imports.
if os.environ.get("RANK", "0") == "0" and os.environ.get("OMP_NUM_THREADS", "") in ("", "1"):
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
# Keep stdout clean for the ONE JSON line: libraries (e.g. the NCCL version banner) write to fd 1.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)

import numpy as np  # noqa: E402

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

FLOP_PER_ROLLOUT_STEP = {"mppi_ode": 80.0, "cem_ode": 65.0, "rpgd_grad": 200.0, "rpgd_fwd": 66.0}  # SURVEY.md 8d convention (DESIGN.md)
MPPI_CFG = dict(seed=42, mpc_timestep=0.02, cc_weight=1.0, R=1.0, LBD=100.0, NU=1000.0, SQRTRHOINV=0.03,
                period_interpolation_inducing_points=10)
CEM_CFG = dict(seed=42, mpc_timestep=0.02, cem_outer_it=3, cem_initial_action_stdev=0.5, cem_stdev_min=0.01, cem_best_k=64,
               warmup=False, warmup_iterations=250)
RPGD_CFG = dict(seed=42, mpc_timestep=0.02, SAMPLING_DISTRIBUTION="uniform", period_interpolation_inducing_points=10,
                learning_rate=0.05, adam_beta_1=0.9, adam_beta_2=0.999, adam_epsilon=1e-08, gradmax_clip=5, rtol=0.001,
                opt_keep_k_ratio=0.25, outer_its=2, resamp_per=10, sample_stdev=0.5, sample_mean=0.0,
                sample_whole_control_space=True, uniform_dist_min=-1.0, uniform_dist_max=1.0, shift_previous=1, warmup=False,
                warmup_iterations=250)
WORKLOADS = {
    # name: (optimizer, predictor, cost, N_global, H)
    "mppi_ode_1m": ("mppi", "ODE", "default", 1_000_000, 100),   # BASELINE configs[4] (the metric's config)
    "mppi_ode_1m_log": ("mppi", "ODE", "default", 1_000_000, 100),  # the same tick with optimizer_logging on: HBM-write bound (SURVEY 8d)
    "mppi_ode_c1": ("mppi", "ODE", "default", 2000, 50),         # configs[0]
    "cem_ode_c2": ("cem-tf", "ODE", "default", 4096, 50),        # configs[1]
    "cem_ode_large": ("cem-tf", "ODE", "default", 1_000_000, 50),  # sharded CEM (SURVEY 8e): candidate keys exchanged through the NVLink mailboxes
    "rpgd_ode_c3": ("rpgd", "ODE", "quadratic_boundary_grad", 32, 50),  # configs[2]
    "mppi_mlp_c4": ("mppi", "Dense-6IN-128H1-128H2-5OUT-0", "default", 65536, 100),  # configs[3]
}
OPT_CFG = {"mppi": MPPI_CFG, "cem-tf": CEM_CFG, "rpgd": RPGD_CFG}


def passes_per_tick(opt_name):
    """rollout passes one optimizer.step() makes over the population (SURVEY 8d: CEM cem_outer_it; RPGD fwd+bwd per Adam step + 1)."""
    return {"mppi": 1, "cem-tf": CEM_CFG["cem_outer_it"], "rpgd": 2 * RPGD_CFG["outer_its"] + 1}[opt_name]


def _emit(line: dict) -> None:
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def synthetic_states(n, seed=0):
    rng = np.random.default_rng(seed)
    angle = rng.uniform(-np.pi, np.pi, n)
    s = np.stack([angle, rng.uniform(-5, 5, n), np.cos(angle), np.sin(angle), rng.uniform(-0.15, 0.15, n),
                  rng.uniform(-0.5, 0.5, n)], 1)
    return s.astype(np.float32)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  The timed region of this bench
    is only a few milliseconds, so NVML is polled from a thread (~1 kHz) instead of `nvidia-smi -lms`."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        self.device, self.samples, self.bits, self._stop, self.t, self.err = device, [], 0, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception as e:  # noqa
                self.err = repr(e)
                break
            time.sleep(0.0005)

    def start(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {self.err}"]}
        self._stop = True
        self.t.join(timeout=2)
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.samples), "reasons": reasons}


def build_controller(workload, shard=None, device=0, logging=False, n_override=None, mlp_engine="simt"):
    import control_toolkit_b200 as ctk
    from control_toolkit_b200.Controllers.controller_mpc import controller_mpc
    opt_name, pred, cost, N, H = WORKLOADS[workload]
    N = n_override or N
    if pred.startswith("Dense"):
        ctk.register_mlp(pred, ctk.MLPSpec.random_init(2))
    cfg = dict(OPT_CFG[opt_name], mpc_horizon=H, num_rollouts=N, shard=shard, device_index=device)
    if pred.startswith("Dense"):
        cfg["mlp_engine"] = mlp_engine
    ctrl = controller_mpc("CartPole", (np.array([-1.0], np.float32), np.array([1.0], np.float32)),
                          {"target_position": 0.0, "target_equilibrium": 1.0},
                          config_controller=dict(optimizer=opt_name, predictor_specification=pred, cost_function_specification=cost,
                                                 controller_logging=logging, calculate_optimal_trajectory=False),
                          config_optimizers={opt_name: cfg}, config_cost_function={"cost_function_name_default": cost})
    ctrl.configure(optimizer_name=opt_name, predictor_specification=pred)
    return ctrl, N, H


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's MPPI on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_mppi_rate(workload, n_sample, ticks, warm=1):
    """rollout-steps/s of the oracle port of the reference optimizer (oracle/{mppi,cem,rpgd}.py, torch-CPU fp32)."""
    import torch
    from oracle import spec
    from oracle.cem import CEMOracle
    from oracle.mppi import MPPIOracle
    from oracle.rpgd import RPGDOracle
    torch.set_num_threads(os.cpu_count() or 1)
    opt_name, pred, cost, _, H = WORKLOADS[workload]
    predictor = spec.ODEPredictor() if pred == "ODE" else spec.MLPPredictor(spec.MLPWeights.random_init(2))
    cls = {"mppi": MPPIOracle, "cem-tf": CEMOracle, "rpgd": RPGDOracle}[opt_name]
    o = cls(predictor, spec.CostParams(name=cost), mpc_horizon=H, num_rollouts=n_sample,
            **{k: v for k, v in OPT_CFG[opt_name].items() if k != "seed"})
    g = torch.Generator().manual_seed(42)

    class _Rng:  # the reference's torch rng duck type (others/globals_and_utils.py:61-82)
        @staticmethod
        def normal(shape, dtype=torch.float32, mean=0.0, stddev=1.0):
            return torch.normal(mean=mean, std=stddev, size=tuple(shape), generator=g, dtype=dtype)

        @staticmethod
        def uniform(shape, dtype=torch.float32, minval=0.0, maxval=1.0):
            return torch.rand(tuple(shape), generator=g, dtype=dtype) * (maxval - minval) + minval

    if opt_name == "rpgd":
        o.reset(_Rng)
    states = synthetic_states(ticks + warm, 0)
    times = []
    for t in range(ticks + warm):
        t0 = time.perf_counter()
        o.step(states[t], _Rng)
        if t >= warm:
            times.append(time.perf_counter() - t0)
    return n_sample * H * passes_per_tick(opt_name) / statistics.mean(times), statistics.mean(times), torch.get_num_threads()


def cpu_reference_rate(workload, n_sample, ticks, warm=1):
    """rollout-steps/s of the reference's UNMODIFIED optimizer file (imported from that checkout through the test-only shims of
    oracle/refharness: SI_Toolkit stand-in with the pinned spec predictor / cost, torch-CPU fp32).  Only where CTK_REFERENCE names a
    checkout of the original Control_Toolkit; without one the reference arm times the oracle port instead."""
    import copy
    import logging
    import torch
    import yaml
    from oracle.refharness.workspace import enter_workspace
    torch.set_num_threads(os.cpu_count() or 1)
    opt_name, pred, cost, _, H = WORKLOADS[workload]
    cwd = os.getcwd()
    enter_workspace()
    try:
        logging.disable(logging.INFO)
        from oracle import spec
        from SI_Toolkit.Predictors import predictor_wrapper as pw
        cc = dict(mpc=dict(optimizer=opt_name, predictor_specification=pred, cost_function_specification=cost,
                           computation_library="tensorflow" if opt_name.endswith("-tf") else "pytorch", device="cpu",
                           controller_logging=False, calculate_optimal_trajectory=False))
        with open(os.path.join("Control_Toolkit_ASF", "config_controllers.yml"), "w") as f:
            yaml.safe_dump(cc, f)
        if pred.startswith("Dense"):
            pw.MLP_REGISTRY[pred] = spec.MLPWeights.random_init(2)
        from Control_Toolkit.Controllers import controller_mpc as cm  # the reference module, unmodified
        cm.config_optimizers[opt_name] = dict(copy.deepcopy(OPT_CFG[opt_name]), mpc_horizon=H, num_rollouts=n_sample)
        ctrl = cm.controller_mpc(environment_name="CartPole", control_limits=(np.array([-1.0], np.float32), np.array([1.0], np.float32)),
                                 initial_environment_attributes={"target_position": 0.0, "target_equilibrium": 1.0})
        ctrl.configure(optimizer_name=opt_name, predictor_specification=pred)
        if opt_name == "rpgd":
            ctrl.optimizer.u = np.float32(0.0)
        states = synthetic_states(ticks + warm, 0)
        times = []
        for t in range(ticks + warm):
            t0 = time.perf_counter()
            ctrl.step(states[t], time=0.02 * t)
            if t >= warm:
                times.append(time.perf_counter() - t0)
    finally:
        os.chdir(cwd)
    return n_sample * H * passes_per_tick(opt_name) / statistics.mean(times), statistics.mean(times), torch.get_num_threads()


def reference_checkout_available():
    try:
        from oracle.refharness.workspace import reference_available
        return reference_available()
    except Exception:
        return False


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    opt_name, _, _, N, H = WORKLOADS[args.workload]
    n_sample = min(N, args.cpu_sample)
    kind = "reference" if reference_checkout_available() else "port"
    if kind == "reference":
        rate, sec, threads = cpu_reference_rate(args.workload, n_sample, args.steps, args.warmup)
        what = f"the reference's UNMODIFIED optimizer_{opt_name.replace('-', '_')}.py through controller_mpc (oracle/refharness shims), torch-CPU fp32"
    else:
        rate, sec, threads = cpu_mppi_rate(args.workload, n_sample, args.steps, args.warmup)
        what = (f"oracle PORT of the reference's optimizer_{opt_name.replace('-', '_')}.py (torch-CPU fp32, eager); the reference checkout is not on this box -- "
                "profiles/reference_vs_port_r02.json shows the port and the unmodified file within a few percent of each other on the same host")
    sample = f"{args.steps} ticks of {n_sample} rollouts x H={H} (of {N}) per step, {what}"
    line = {"impl": "reference", "metric": "rollout-steps/s", "value": rate, "unit": "rollout-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "optimizer": opt_name, "num_rollouts": N, "mpc_horizon": H, "predictor": WORKLOADS[args.workload][1]},
            "cpu_baseline": {"value": rate, "unit": "rollout-steps/s", "cores": threads, "kind": kind, "sample": sample,
                             "same_config": n_sample == N},
            "e2e": {"value": rate, "unit": "rollout-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


# ------------------------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20
DUMP_LOG_ROWS = 4096  # rollouts of the logged controls / trajectories written with logging on (the whole log is GBs at 10^6 rollouts)


def timed_path_outputs(opt, u_dev, logging_on) -> dict:
    """What the last timed tick computed, as a caller of the tick receives it: the control u, the optimizer state the next tick
    starts from (get_state(): MPPI u_nom, CEM mean and stdev, RPGD the population and its Adam moments) and, with logging on, the
    cost of every rollout plus the logged controls and trajectories of a fixed, seeded sample of DUMP_LOG_ROWS rollouts.  u and the
    state are the same on every shard; the logs are this rank's shard of the population (rank 0's when several GPUs run).  The logs
    come to the host whole, as optimizer.step hands them over, once, after the timed passes."""
    nu = int(opt.num_control_inputs)
    out = {"u": u_dev[:nu].cpu().numpy()}
    for k, v in opt.get_state().items():
        v = np.asarray(v)
        out[f"state_{k}"] = v if v.dtype == np.float32 else v.astype(np.float64)
    if logging_on:
        n = opt._n_local
        opt._collect_rollout_logs(n)
        rows = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_LOG_ROWS), replace=False))
        out["J_logged"] = np.array(opt.logging_values["J_logged"], np.float32)
        out["log_rows"] = rows.astype(np.float64)
        for k in ("Q_logged", "rollout_trajectories_logged"):
            out[f"{k}_rows"] = np.array(opt.logging_values[k][rows], np.float32)
    return out


def write_outputs(directory, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"outputs to dump take {total} bytes, more than the {DUMP_LIMIT_BYTES} allowed")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from control_toolkit_b200 import _lib as L
    from control_toolkit_b200.distributed import ShardPlan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    lib = L.load()
    plan = ShardPlan(rank, world)
    logging_on = args.workload.endswith("_log")
    ctrl, N, H = build_controller(args.workload, shard=plan if world > 1 else None, device=local_rank, n_override=args.rollouts,
                                  mlp_engine=args.mlp_engine, logging=logging_on)
    opt = ctrl.optimizer
    plan.attach(opt, lib)  # handle runs on torch's current stream (events + NCCL ordering)
    K, W = args.steps, max(args.warmup, 3)  # timing rule: at least three untimed warm-up ticks (the line reports the W used)
    states = torch.from_numpy(synthetic_states(K + W, 0)).to(dev)
    u_dev = torch.zeros(4, dtype=torch.float32, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def tick(i):
        plan.run_tick_device(opt, lib, states[i].data_ptr(), u_dev.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    fused = getattr(opt, "_exchange", "none") in ("p2p", "none")  # the tick is ctk_step_device (one C call, no NCCL in between)

    n_align = [0]  # alignment-barrier launches (outside the timed event pairs; not part of a tick)

    def align():
        """Device-side barrier across the shards (mailbox flags, one tiny kernel) enqueued BEFORE a timed tick: the shards' L2
        flushes run un-synchronised, and without it their skew would be spent waiting inside the timed tick's exchange."""
        if world > 1 and getattr(opt, "_exchange", "") == "p2p":
            L.check(lib.ctk_exchange_barrier(opt._h))
            n_align[0] += 1

    for i in range(W):
        tick(i)
    barrier()
    # ---- device-resident timing: one CUDA-event pair per tick, L2 flushed between ticks ----
    launches0 = opt.gpu_launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    wall0 = time.perf_counter()
    for i in range(K):
        flush.zero_()
        align()
        ev[i][0].record()
        tick(W + i)
        ev[i][1].record()
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, timed_path_outputs(opt, u_dev, logging_on))
    per_tick_ms = [a.elapsed_time(b) for a, b in ev]
    launches = opt.gpu_launches - launches0 - n_align[0]  # kernels of the K timed ticks
    # ---- second pass, same ticks: CUDA events around the rollout kernel only (roofline.achieved); kept out of the pass
    #      above so that the extra event records do not sit inside the timed ticks ----
    single_launch_tick = launches == K
    if world > 1 and (single_launch_tick or fused):
        # sharded MPPI: the tick IS one launch, already bracketed by an event pair in the pass above.  A second pass with extra
        # event records inside the handle skews the ranks against each other and the skew is then spent waiting inside the fused
        # exchange (measured: 0.18 ms "kernel" at 8 GPUs for a 0.042 ms tick), so the kernel time is this rank's tick time of
        # the timed pass (an upper bound: it includes the ~6 us event-pair overhead)
        ms_sum, n_k = C.c_double(sum(per_tick_ms)), C.c_int64(K if single_launch_tick else 0)
        tick2_ms = sum(per_tick_ms) / K
        kernel_ms_source = "event pair around the one-launch tick in the timed pass (rank 0)"
    else:
        L.check(lib.ctk_enable_kernel_timing(opt._h, 1))
        ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for i in range(K):
            flush.zero_()
            ev2[i][0].record()
            tick(W + i)
            ev2[i][1].record()
        barrier()
        tick2_ms = sum(a.elapsed_time(b) for a, b in ev2) / K  # this rank's tick in the SAME pass the kernel events were taken in
        ms_sum, n_k = C.c_double(), C.c_int64()
        L.check(lib.ctk_get_kernel_timing(opt._h, C.byref(ms_sum), C.byref(n_k)))
        L.check(lib.ctk_enable_kernel_timing(opt._h, 0))
        kernel_ms_source = "CUDA events around the kernel launch on the handle's stream, second pass over the same ticks"
    # ---- third figure, clearly separate: the same K ticks BACK TO BACK inside ONE event pair (no per-tick flush, no per-tick
    #      events): consecutive ticks overlap through programmatic dependent launch, which a per-tick event pair forbids.  The
    #      difference to ms_per_step is the event-pair / launch gap and the cold prologue, not work. ----
    pipelined_ms = None
    if fused:
        st_rep = states[W:W + K].contiguous()
        u_rep = torch.zeros(K, 2, dtype=torch.float32, device=dev)
        L.check(lib.ctk_step_device_n(opt._h, C.c_void_p(st_rep.data_ptr()), 6, C.c_void_p(u_rep.data_ptr()), 2, min(K, 10)))  # warm
        barrier()
        align()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        L.check(lib.ctk_step_device_n(opt._h, C.c_void_p(st_rep.data_ptr()), 6, C.c_void_p(u_rep.data_ptr()), 2, K))
        p1.record()
        barrier()
        pm = torch.tensor([p0.elapsed_time(p1) / K], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(pm, op=dist.ReduceOp.MAX)
        pipelined_ms = float(pm.item())
        if not bool(torch.isfinite(u_rep).all()) or float(u_rep[:, 1].abs().max()) != 0.0:
            raise RuntimeError("pipelined ticks reported an exchange failure")
    total_ms = torch.tensor([sum(per_tick_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / K
    opt_name = WORKLOADS[args.workload][0]
    passes = passes_per_tick(opt_name)
    value = N * H * passes / (ms_per_step * 1e-3)

    # ---- e2e through the public plugin API: host state in, host control out, every step ----
    host_states = synthetic_states(K + W, 1)
    # logging workload: the plugin boundary itself (optimizer.step -> u + logging_values as host arrays); the reference
    # controller's own history copy of those arrays (Controllers/__init__.py:159-178) is the caller's business, not the path's
    api_step = opt.step if logging_on else ctrl.step
    api_name = ("optimizer.step(s_host) -> u_host, logging_values (pinned host views of Q / J / trajectories)" if logging_on
                else "controller_mpc.step(s_host) -> u_host")
    for i in range(min(W, 3) if not logging_on else 2):
        api_step(host_states[i])
    barrier()
    lat = []
    Ke = min(K, 5) if logging_on else K  # with logging every step hands 2.8 GB of trajectories to the host
    t0 = time.perf_counter()
    for i in range(Ke):
        t1 = time.perf_counter()
        api_step(host_states[W + i])
        lat.append(time.perf_counter() - t1)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = N * H * passes * Ke / float(e2e_s.item())

    if rank == 0:
        # ---- roofline of the dominant kernel (K1 fused rollout), measured live above ----
        k1_ms = ms_sum.value / max(n_k.value, 1)
        n_local = opt._n_local
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(REPO, "MEASURED_PEAKS.json")) else {}
        is_mlp = WORKLOADS[args.workload][1].startswith("Dense")
        if is_mlp:
            # dense contraction: 2*(6*128 + 128*128 + 128*5) FLOP per rollout-step (SURVEY 8d); the 128x128 layer (92 %) runs on the
            # tensor cores as six bf16 products (3-term split operands) when mlp_engine == tcgen05
            fl_step = 35584.0
            flop = fl_step * n_local * H
            achieved = flop / (k1_ms * 1e-3) / 1e12
            tpeak = float(peaks.get("bf16_tflops", 1648.0))
            pred_name = {"tcgen05": "MlpTcPred", "tcgen05_bf16": "MlpTcBf16Pred", "tcgen05_fast": "MlpTcFastPred"}.get(args.mlp_engine, "MlpSimtPred")
            products = {"tcgen05": 6.0, "tcgen05_bf16": 1.0, "tcgen05_fast": 1.0}.get(args.mlp_engine, 0.0)
            roofline = {"bound": "tensor", "kernel": f"mppi_rollout_kernel<{pred_name}>",
                        "achieved": achieved, "peak": tpeak, "unit": "TFLOP/s", "frac": achieved / tpeak, "traffic": None,
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst, cuBLAS 8192^3)" if peaks else "fallback 1648",
                        "flop_per_rollout_step": fl_step, "kernel_ms": k1_ms, "kernel_share_of_tick": k1_ms / tick2_ms,
                        "tensor_flop_issued_per_algorithmic": products * 32768.0 / fl_step,
                        "precision": {"tcgen05": "fp32-level (six products of three-term bf16 splits)", "tcgen05_bf16": "one bf16 product (operands rounded to bfloat16): opt-in, parity vs an oracle with the same rounding",
                                      "tcgen05_fast": "one bf16 product + MUFU.TANH: opt-in, no parity bound"}.get(args.mlp_engine, "fp32")}
        elif logging_on:
            # optimizer_logging on: rollout_trajectories_logged [N,H+1,6] + Q_logged [N,H,1] + J [N] are written by the rollout kernel
            byt = 4.0 * n_local * ((H + 1) * 6 + H + 1)
            hpk = float(peaks.get("hbm_gbs", 6650.0))
            ach = byt / (k1_ms * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": "mppi_ode_kernel<LOG> (fused tick + coalesced SoA trajectory log)", "achieved": ach, "peak": hpk,
                        "unit": "GB/s", "frac": ach / hpk, "traffic": None, "algorithmic_bytes_per_launch": byt,
                        "bytes_per_rollout_step": 28.0, "peak_source": "MEASURED_PEAKS.json hbm_gbs (copy bandwidth)" if peaks else "fallback 6650",
                        "kernel_ms": k1_ms, "kernel_share_of_tick": k1_ms / tick2_ms}
        elif opt_name == "cem-tf":
            fl_step = FLOP_PER_ROLLOUT_STEP["cem_ode"]
            peak, clk = C.c_double(), C.c_double()
            L.check(lib.ctk_fp32_peak(local_rank, C.byref(peak), C.byref(clk)))
            one_launch = launches == K  # persistent tick: all outer iterations (rollouts, top-k, refit) in ONE launch
            per_launch = passes if one_launch else 1
            if not n_k.value:  # sharded run: no kernel-event pass (it would skew the shards): the tick's own event pair, an upper bound
                k1_ms = tick2_ms / (1 if one_launch else passes)
            achieved = fl_step * n_local * H * per_launch / (k1_ms * 1e-3) / 1e12
            roofline = {"bound": "fp32", "kernel": ("cem_tick_kernel (persistent: the whole tick -- rollouts, top-k and refit of all outer iterations)" if one_launch
                                                    else "cem_ode_kernel (one launch per outer iteration)"), "achieved": achieved,
                        "peak": peak.value, "unit": "TFLOP/s", "frac": achieved / peak.value, "traffic": None,
                        "peak_source": "measured live: FP32 FMA-chain microbenchmark (ctk_fp32_peak)", "flop_per_rollout_step": fl_step,
                        "kernel_ms": k1_ms, "kernel_share_of_tick": k1_ms * (1 if one_launch else passes) / tick2_ms,
                        "note": "4096 rollouts = 32 blocks of 4 rollout warps: the tick is a chain of dependent phases (rollouts, block sort, grid merge, refit per outer iteration), latency-bound by construction"}
        elif opt_name == "rpgd":
            its = RPGD_CFG["outer_its"]
            fl_launch = (FLOP_PER_ROLLOUT_STEP["rpgd_grad"] * its + FLOP_PER_ROLLOUT_STEP["rpgd_fwd"]) * n_local * H
            peak, clk = C.c_double(), C.c_double()
            L.check(lib.ctk_fp32_peak(local_rank, C.byref(peak), C.byref(clk)))
            achieved = fl_launch / (k1_ms * 1e-3) / 1e12
            roofline = {"bound": "fp32", "kernel": "rpgd_grad_coef_kernel (all Adam iterations + the final rollout of a tick in one launch)",
                        "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s", "frac": achieved / peak.value, "traffic": None,
                        "peak_source": "measured live: FP32 FMA-chain microbenchmark (ctk_fp32_peak)",
                        "flop_per_launch": fl_launch, "kernel_ms": k1_ms, "kernel_share_of_tick": k1_ms / tick2_ms,
                        "note": "32 trajectories = one warp: a serial dependency chain of 5 x 50 steps, latency-bound by construction"}
        else:
            flop = FLOP_PER_ROLLOUT_STEP["mppi_ode"] * n_local * H
            peak, clk = C.c_double(), C.c_double()
            L.check(lib.ctk_fp32_peak(local_rank, C.byref(peak), C.byref(clk)))
            achieved = flop / (k1_ms * 1e-3) / 1e12
            roofline = {"bound": "fp32", "kernel": "mppi_ode_kernel (fused sample+rollout+cost+softmin+exchange+update, the whole tick)",
                        "achieved": achieved, "peak": peak.value,
                        "unit": "TFLOP/s", "frac": achieved / peak.value if peak.value else None, "traffic": None,
                        "peak_source": "measured live: FP32 FMA-chain microbenchmark (ctk_fp32_peak), implied FFMA clock %.0f MHz; "
                                       "theoretical 148 SM x 128 lanes x 2 x 1.965 GHz = 74.5" % clk.value,
                        "flop_per_rollout_step": FLOP_PER_ROLLOUT_STEP["mppi_ode"], "kernel_ms": k1_ms,
                        "kernel_share_of_tick": k1_ms / tick2_ms,
                        "hbm": {"algorithmic_bytes_per_launch": 4.0 * n_local, "achieved_gbs": 4.0 * n_local / (k1_ms * 1e-3) / 1e9,
                                "peak_gbs": peaks.get("hbm_gbs", 6650.0)}}
        # measured DRAM traffic of that kernel (ncu --set full capture, per launch), when a capture of this workload is on file
        tpath = os.path.join(REPO, "profiles", "ncu_traffic_r02.json")
        if not os.path.exists(tpath):
            tpath = os.path.join(REPO, "profiles", "ncu_traffic_r01.json")
        ttab = json.load(open(tpath)) if os.path.exists(tpath) else {}
        tkey = args.workload if args.rollouts is None else ""
        tr = ttab.get(f"{tkey}:{args.mlp_engine}" if is_mlp and args.mlp_engine != "tcgen05" else tkey, None)
        if tr and world == 1:
            roofline["traffic"] = tr["bytes"]
            roofline["traffic_source"] = tr["source"]
        roofline["tick_ms_same_pass"] = tick2_ms
        roofline["kernel_ms_source"] = kernel_ms_source
        # ---- CPU baseline: oracle port on a bounded sample of the same workload ----
        if world == 1:  # the CPU baseline is timed at N = 1 only (the multi-GPU lines would just repeat it)
            n_sample = min(N, args.cpu_sample)
            rate, sec, threads = cpu_mppi_rate(args.workload, n_sample, 2, 1)
            cpu = {"value": rate, "unit": "rollout-steps/s", "cores": threads, "kind": "port", "same_config": n_sample == N,
                   "sample": f"2 ticks of {n_sample} rollouts x H={H} (of {N}); oracle PORT (torch-CPU fp32, eager) of reference optimizer_{opt_name.replace('-', '_')}.py; "
                             f"{sec:.2f} s/tick"}
            if n_sample < N:  # throughput is flat in N once the population is large: a second, smaller sample next to it
                rate2, sec2, _ = cpu_mppi_rate(args.workload, max(n_sample // 4, 1), 2, 1)
                cpu["flat_in_N"] = {"rollouts": max(n_sample // 4, 1), "value": rate2, "s_per_tick": sec2}
        else:
            cpu = None
        line = {"metric": "rollout-steps/s", "value": value, "unit": "rollout-steps/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": args.workload, "optimizer": opt_name, "rollout_passes_per_tick": passes, "num_rollouts": N, "mpc_horizon": H,
                           "predictor": WORKLOADS[args.workload][1], "cost": WORKLOADS[args.workload][2], "noise": "in-kernel Philox4x32-10",
                           **({"mlp_engine": args.mlp_engine} if WORKLOADS[args.workload][1].startswith("Dense") else {}),
                           "parallelism": f"rollouts sharded over {world} GPU(s); exchange per tick: {getattr(opt, '_exchange', 'none')} "
                                          f"({'in-kernel NVLink mailbox stores, ' if getattr(opt, '_exchange', '') == 'p2p' else ''}"
                                          + (f"{H // 10 + 3} floats per shard)" if opt_name == "mppi" else f"{CEM_CFG['cem_best_k']} (cost, id) keys per shard and outer iteration)" if opt_name == "cem-tf" else "none)"),
                           "l2": "flushed between timed ticks (256 MiB memset" + ("; shards aligned by a device-side mailbox barrier before each timed tick" if world > 1 else "") + "); inputs are 24 B per tick", "logging": logging_on},
                "e2e": {"value": e2e_value, "unit": "rollout-steps/s", "h2d_bytes_per_step": 24, "d2h_bytes_per_step": (4 * N * ((H + 1) * 6 + H + 1) + 8 + 4 * H) if logging_on else ((8 + 4 * H) if opt_name == "mppi" else 8),
                        "p50_step_latency_ms": statistics.median(lat) * 1e3, "api": api_name},
                "pipelined": (None if pipelined_ms is None else
                              {"value": N * H * passes / (pipelined_ms * 1e-3), "unit": "rollout-steps/s", "ms_per_step": pipelined_ms,
                               "ticks": K, "how": "ticks back to back inside ONE CUDA-event pair (ctk_step_device_n), no per-tick L2 flush, "
                                                           "max over ranks; consecutive ticks overlap through programmatic dependent launch"}),
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
                "wall_s_timed_region": wall}
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mppi_ode_1m", choices=sorted(WORKLOADS))
    ap.add_argument("--rollouts", type=int, default=None, help="override the global rollout count")
    ap.add_argument("--mlp-engine", default="tcgen05", choices=["simt", "tcgen05", "tcgen05_bf16", "tcgen05_fast"], help="MLP predictor engine (mppi_mlp_c4 workload)")
    ap.add_argument("--cpu-sample", type=int, default=250_000, help="rollouts per CPU-baseline tick (bounded sample; C1-C4 run at their full size)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed tick computed to DIR/<name>.npy (own arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
