#!/usr/bin/env python
"""Rollout time with constant-velocity obstacles (MPPI.obs_vel) against static obstacles.

    python tools/moving_obstacles_bench.py [--steps K] [--rounds R] [--out FILE]

Workloads (bench.py's definitions, shipped networks, default pass-1 and scoring modes): the Franka shelf with 2064 and
with 294 spheres at 4096 samples x 50 steps (tensor-core prefilter + per-step scoring), and planar-7 at 1000 x 30 with
M = 4 (whole-horizon kernel).  Variants, on one object and alternated round by round: no velocities (obs_vel = None),
zero velocities, and random nonzero velocities that move a sphere by about 0.2 units over the horizon.  Without
velocities the library launches exactly what it launched before it had them; with velocities every step of the
per-step paths costs one more launch, which writes that step's positions (and the prefilter's per-obstacle table),
and the whole-horizon kernels compute the positions inside.

One MPPI.propagate() per timed step, timed with CUDA events; a 256 MB buffer is overwritten between timed steps so
that no step finds the previous one's weights or activations in the 126 MB L2.  Prints the card's name and power
limit with the numbers (they are part of them), then one line per (workload, variant): median and min ms per
propagate over all rounds, launches per propagate, and the median relative to no velocities.
"""
import argparse
import os
import statistics
import subprocess
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (workload definitions, seeded policy)

WORKLOADS = ("franka_shelf_2064", "franka_shelf_294", "planar7")
VARIANTS = ("none", "zero", "moving")


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name()} (nvidia-smi unavailable)"


def velocities(p, dev):
    M, H, dt = p["obs"].shape[0], p["H"], p["dt"]
    g = torch.Generator().manual_seed(1)
    v = {"none": None, "zero": torch.zeros(M, 3), "moving": torch.randn(M, 3, generator=g) * (0.2 / (H * dt))}
    return {k: None if x is None else x.to(dev) for k, x in v.items()}


def time_block(m, steps, flush):
    m.propagate()                           # untimed: uploads the variant's velocities
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    l0 = m.launch_count()
    for a, b in ev:
        flush.zero_()
        a.record()
        m.propagate()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev], (m.launch_count() - l0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="timed propagates per variant and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("moving_obstacles_bench.py measures on a CUDA device; none found")
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lines = [f"card: {card()}",
             f"{args.rounds} rounds x {args.steps} steps per variant (warm-up {args.warmup}), variants alternated; L2 "
             "overwritten (256 MB) before every timed step; ms per MPPI.propagate(), CUDA events"]
    print("\n".join(lines), flush=True)
    opts = SimpleNamespace(pass1="auto", score="auto", per_step=False)
    for wl in WORKLOADS:
        p = bench.problem(wl)
        m, _, _ = bench.build_mppi(p, p["N"], p["H"], dev, opts, 0, 1)
        vel = velocities(p, dev)
        for _ in range(args.warmup):
            for v in VARIANTS:
                m.obs_vel = vel[v]
                m.propagate()
        times = {v: [] for v in VARIANTS}
        launches = {}
        for _ in range(args.rounds):
            for v in VARIANTS:
                m.obs_vel = vel[v]
                ts, launches[v] = time_block(m, args.steps, flush)
                times[v] += ts
        base = statistics.median(times["none"])
        for v in VARIANTS:
            med = statistics.median(times[v])
            line = (f"{wl:18s} N={p['N']:5d} H={p['H']:3d} M={p['obs'].shape[0]:5d}  {v:7s}  median {med:8.3f} ms  "
                    f"min {min(times[v]):8.3f} ms  launches {launches[v]:7.1f}  vs none {med / base:6.3f}x")
            print(line, flush=True)
            lines.append(line)
        del m
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
