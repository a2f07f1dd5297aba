#!/usr/bin/env python
"""Writes the input file of `tc_microbench phase`: the shipped Franka net and the obstacles of a bench workload.

    python tools/tc_phase_inputs.py OUT [--workload franka_shelf_2064]

Layout: int32 M, then float32 W0, b0, ..., W4, b4 (torch orientation), then the (M, 4) obstacles.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("out")
ap.add_argument("--workload", default="franka_shelf_2064")
args = ap.parse_args()

p = bench.problem(args.workload)
W, b, src = bench.load_net_arrays("franka")
obs = p["obs"].float().numpy()
with open(args.out, "wb") as f:
    f.write(np.int32(obs.shape[0]).tobytes())
    for w, x in zip(W, b):
        f.write(w.float().numpy().astype(np.float32).tobytes())
        f.write(x.float().numpy().astype(np.float32).tobytes())
    f.write(np.ascontiguousarray(obs, dtype=np.float32).tobytes())
print(f"{args.out}: {src} franka net, {obs.shape[0]} obstacles of {args.workload}")
