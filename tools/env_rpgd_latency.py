"""p50 controller.step() latency and gradient-kernel time (CUDA events) of RPGD on the Dubins car at C3 geometry (N = 32, H = 50,
outer_its 2, in-kernel Philox, logging off), timed in the same process, alternating tick by tick, with the CartPole C3 RPGD tick.
Records the device name and power limit next to the numbers (read-only nvidia-smi query).
Usage on a GPU machine:  python tools/env_rpgd_latency.py [ticks] [out.json]   -> prints one JSON line (and writes it to out.json)"""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
from gpu_helpers import make_controller  # noqa: E402
from helpers import load_golden  # noqa: E402
from oracle import spec  # noqa: E402  (synthetic states only)
from test_gpu_env_gradient import _controller, _meta  # noqa: E402


def _gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    from control_toolkit_b200 import _lib as L
    ticks = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
    lib = L.load()
    _, meta = load_golden("rpgd_c3")
    runs = {
        "dubins_rpgd_c3": (_controller(_meta("rpgd", num_rollouts=32, mpc_horizon=50, outer_its=2)), spec.dubins_synthetic_states(ticks + 50, 7)),
        "cartpole_rpgd_c3": (make_controller(meta, rng=None, logging=False), spec.synthetic_states(ticks + 50, 7)),
    }
    lat = {k: [] for k in runs}
    for k, (ctrl, states) in runs.items():  # warm-up: module load, first launches
        for i in range(50):
            ctrl.step(states[i])
        L.check(lib.ctk_enable_kernel_timing(ctrl.optimizer._h, 1))
    launches0 = {k: ctrl.optimizer.gpu_launches for k, (ctrl, _) in runs.items()}
    for i in range(ticks):
        for k, (ctrl, states) in runs.items():
            t0 = time.perf_counter()
            ctrl.step(states[50 + i])  # returns after the device has delivered u (host mirror / synchronised copy)
            lat[k].append((time.perf_counter() - t0) * 1e6)
            if (i + 1) % 200 == 0:  # drain the event pairs before the handle's pool of 256 runs out
                ms, n = C.c_double(), C.c_int64()
                L.check(lib.ctk_get_kernel_timing(ctrl.optimizer._h, C.byref(ms), C.byref(n)))
                lat.setdefault(k + "_kernel", []).append(ms.value * 1e3 / max(n.value, 1))
    out = {"device": _gpu_info(), "ticks": ticks}
    for k, (ctrl, _) in runs.items():
        s = sorted(lat[k])
        out[k] = dict(p50_us=statistics.median(s), p90_us=s[int(0.9 * len(s))], kernel_us_mean=statistics.mean(lat.get(k + "_kernel", [float("nan")])),
                      launches_per_tick=(ctrl.optimizer.gpu_launches - launches0[k]) / ticks, last_kernel=ctrl.optimizer.last_kernel)
    print(json.dumps(out))
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
