"""torch.profiler capture of K1 on the bench's mppi_ode_1m tick (10^6 rollouts x H = 100, in-kernel noise, host state).

    python tools/k1_profile.py OUT_DIR [--ticks 50] [--workload mppi_ode_1m]

Writes OUT_DIR/k1_profile.txt (per-kernel CUDA time table) and OUT_DIR/k1_profile.pt.trace.json (chrome trace).  Run it on its own:
the profiler slows the host, so the end-to-end numbers come from bench.py with the profiler off."""
import argparse
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--ticks", type=int, default=50)
    ap.add_argument("--workload", default="mppi_ode_1m")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    os.makedirs(args.out, exist_ok=True)
    ctrl, N, H = bench.build_controller(args.workload, logging=args.workload.endswith("_log"))
    states = bench.synthetic_states(args.ticks + 5, seed=3)
    for s in states[:5]:
        ctrl.step(s)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for s in states[5:]:
            ctrl.step(s)
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
    head = (f"{args.workload}: {N} rollouts x H={H}, {args.ticks} ticks through controller_mpc.step(s_host); "
            f"kernel {ctrl.optimizer.last_kernel}; device {torch.cuda.get_device_name(0)}\n")
    with open(os.path.join(args.out, "k1_profile.txt"), "w") as f:
        f.write(head + table + "\n")
    prof.export_chrome_trace(os.path.join(args.out, "k1_profile.pt.trace.json"))
    print(head + table)


if __name__ == "__main__":
    main()
