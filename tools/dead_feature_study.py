#!/usr/bin/env python
"""Dead hidden features of the prefilter's network on the bench shelf (CPU, fp64).

    python tools/dead_feature_study.py [--net franka] [--census 128] [--heldout 96]

1. census: features of hidden layers 2..4 never active over `census` random q in [-pi, pi]^d x every shelf sphere;
2. held-out: how often those features fire on other random q and on the q0 -> qf line (expected: never);
3. what skipping their K-steps saves: tcgen05 K-steps per tile (K = 16) with the dead features permuted last;
4. why the skip is certified per row by computing the dead columns: a shared "envelope" column per group of dead
   features (sum_k max_f W[f, k] h_k + max_f b_f >= every member's pre-activation, since h >= 0) certifies nothing.
"""
import argparse
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--net", default="franka")
ap.add_argument("--census", type=int, default=128)
ap.add_argument("--heldout", type=int, default=96)
args = ap.parse_args()
torch.set_num_threads(os.cpu_count() or 1)

p = bench.problem("franka_shelf_2064")
W, b, src = bench.load_net_arrays(args.net)
Wd = [w.double() for w in W]
bd = [x.double() for x in b]
obs = p["obs"].double()
M, d = obs.shape[0], p["dof"]
# enc([q, p]) = [q, p, sin q, sin p, cos q, cos p]: layer 1 splits into a per-sample and a per-obstacle table
n_in = d + 3
qcols = [o * n_in + k for o in range(3) for k in range(d)]
pcols = [o * n_in + d + k for o in range(3) for k in range(3)]
P3 = obs[:, :3]
B = torch.cat((P3, P3.sin(), P3.cos()), 1) @ Wd[0][:, pcols].T


def rand_q(seed, n):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, d, generator=g, dtype=torch.float64) * 2 - 1) * math.pi


def hidden(Q):
    """post-ReLU activations of hidden layers 1..4 for every (q, sphere) pair, (n*M, 256) each"""
    A = torch.cat((Q, Q.sin(), Q.cos()), 1) @ Wd[0][:, qcols].T + bd[0]
    hs = [[], [], [], []]
    for s0 in range(0, Q.shape[0], 16):
        h = torch.relu(A[s0:s0 + 16, None, :] + B[None]).reshape(-1, 256)
        hs[0].append(h)
        for i, l in enumerate((1, 2, 3)):
            h = torch.relu(h @ Wd[l].T + bd[l])
            hs[i + 1].append(h)
    return [torch.cat(x) for x in hs]


hs = hidden(rand_q(1, args.census))
dead = [(h > 0).sum(0) == 0 for h in hs]
print(f"network: {args.net} ({src}); census: {args.census} random q x {M} spheres")
print("  features never active, hidden layers 1..4:", [int(x.sum()) for x in dead])
del hs

line = p["q0"].double() + (p["qf"] - p["q0"]).double() * torch.linspace(0, 1, 32, dtype=torch.float64)[:, None]
ht = hidden(torch.cat((rand_q(7, args.heldout), line)))
fired = [float((ht[i][:, dead[i]] > 0).any(1).double().mean()) if dead[i].any() else 0.0 for i in range(4)]
print(f"  held-out ({args.heldout} random q + 32 states on q0 -> qf, x {M} spheres): share of pairs where a census-dead "
      "feature fires, layers 1..4:", fired)

# K-steps of the GEMM that READS layer l's features: layer l+1's hidden GEMM, or the output layer after layer 4
drop = [int(x.sum()) // 16 for x in dead]
hid_full, hid_new = 3 * 16, sum(16 - s for s in drop[:3])
print(f"  droppable K-steps: layer 2 GEMM {drop[0]}, layer 3 {drop[1]}, layer 4 {drop[2]}, output {drop[3]}")
print(f"  hidden-layer MMA K-steps per tile {hid_full} -> {hid_new} ({hid_new / hid_full:.3f}); "
      f"output layer 16 -> {16 - drop[3]}")

for g in (1, 2, 4, 8):
    res = []
    for i, l in enumerate((1, 2, 3)):
        D = torch.nonzero(dead[i + 1]).flatten()
        D = D[bd[l][D].argsort()]
        x = ht[i] * (~dead[i])                          # earlier dead features dropped (exact while certified)
        ok = torch.ones(x.shape[0], dtype=torch.bool)
        cols = 0
        for s in range(0, len(D), g):
            G = D[s:s + g]
            cols += 1
            ok &= (x @ Wd[l][G].max(0)[0] + bd[l][G].max()) <= 0
        res.append((cols, round(float(ok.double().mean()), 4)))
    print(f"  certificate columns per group of {g} dead features: (columns, share of pairs certified), "
          f"layers 2..4: {res}")
