#!/usr/bin/env python
"""Rollout time of distance networks of other shapes than the shipped 256 x 4, in both scoring modes.

    python tools/net_shape_bench.py [--steps K] [--warmup W] [--out FILE]

Workloads (bench.py's definitions): planar-7 at 1000 samples x 30 steps with M = 4 obstacles (whole-horizon kernel)
and the Franka shelf at 4096 x 50 with M = 294 spheres (tensor-core prefilter + per-step scoring).  Networks: seeded
random-init 256 x 4, 128 x 3, 128 x 2 and 64 x 4 (random weights for all four, so that only the shape differs: the
prefilter's candidate count depends on the weights).  Modes: `ffma` (strict IEEE fp32 on the CUDA cores, which runs
the network's own width and depth) and `tc_split` (tensor cores, which run the 256 x 4 embedding of every network).

One MPPI.propagate() per timed step, timed with CUDA events; a 256 MB buffer is overwritten between timed steps so
that no step finds the previous one's weights or activations in the 126 MB L2.  Prints the card's name and power
limit with the numbers (they are part of them), then one line per (workload, network, mode): median and min ms per
propagate over the timed steps.
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions, seeded policy)

WORKLOADS = ("planar7", "franka_shelf_294")
SHAPES = (("256x4", [256] * 4), ("128x3", [128] * 3), ("128x2", [128] * 2), ("64x4", [64] * 4))
MODES = ("ffma", "tc_split")


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name()} (nvidia-smi unavailable)"


def make(p, layers, mode, dev):
    from optimalmodulationds_b200 import MPPI, LinDS
    from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
    torch.manual_seed(0)
    net = RobotSdfCollisionNet(in_channels=p["dof"] + 3, out_channels=p["out"], layers=layers, skips=[])
    t = lambda x: x.to(dev)  # noqa: E731
    DS = [LinDS(t(p["qf"])), LinDS(t(p["q0"]))]
    m = MPPI(t(p["q0"]), t(p["qf"]), t(p["dh"]), t(p["obs"]), p["dt"], p["H"], p["N"], DS, t(p["dh_a"]), net, p["K"])
    m.set_pass1_mode("auto")
    m.set_score_mode(mode)
    m.dst_thr, m.ker_thr, m.ignored_links = p["dst_thr"], p["ker_thr"], list(p["ignored"])
    m.Cost.q_min, m.Cost.q_max = t(p["qlim"][0]), t(p["qlim"][1])
    bench.load_policy(m, p, bench.seeded_policy(p, p["N"], 0), dev)
    return m


def time_propagate(m, steps, warmup, flush):
    for _ in range(warmup):
        m.propagate()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.zero_()
        a.record()
        m.propagate()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("net_shape_bench.py measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lines = [f"card: {card()}",
             f"steps {args.steps} (warm-up {args.warmup}), L2 overwritten (256 MB) before every timed step; "
             "ms per MPPI.propagate(), CUDA events"]
    print("\n".join(lines), flush=True)
    for wl in WORKLOADS:
        p = bench.problem(wl)
        for mode in MODES:
            base = None
            for name, layers in SHAPES:
                m = make(p, layers, mode, dev)
                ts = time_propagate(m, args.steps, args.warmup, flush)
                med = statistics.median(ts)
                base = base or med
                line = (f"{wl:18s} N={p['N']:5d} H={p['H']:3d} M={p['obs'].shape[0]:4d}  {name:6s} {mode:8s}  "
                        f"median {med:8.3f} ms  min {min(ts):8.3f} ms  vs 256x4 {base / med:5.2f}x")
                print(line, flush=True)
                lines.append(line)
                del m
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
