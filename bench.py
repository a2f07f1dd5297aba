#!/usr/bin/env python
"""bench.py -- MPPI rollout state-steps/s (samples x horizon per MPPI iteration) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A "step" is one MPPI iteration of the hot path (propagate + get_cost + shift_policy_means; sampling the
policy noise is excluded, SURVEY.md 8(d)) over one batch of synthetic input.  Default workload =
BASELINE.json configs[2] / the metric's named config: Franka Panda 7-DoF, shelf point cloud of 2064 spheres
("~2k points"), 4096 samples x 50 steps per GPU (weak scaling; configs[4] is the same sharded), K = 5,
10 policy kernels, shipped Franka checkpoint (tests/golden/weights/franka.npz).

Prints ONE JSON line (rank 0).  `value` = whole-job state-steps/s with inputs resident in HBM, CUDA-event
timed, max over ranks; `e2e` = the same through the C ABI host-buffer entry point with pinned host tensors
(H2D + D2H inside the timed region); `roofline` = tensor-core prefilter kernel vs the measured bf16 peak;
`cpu_baseline` = the reference's own classes (oracle/_ref, staged by oracle/make_ref.sh; torch CPU, all host
threads) on a bounded sample -- the oracle port only when that tree is absent.
`--impl reference` times that CPU arm alone with the same --steps / --warmup.
`--dump-outputs DIR` writes what the last timed step returned (trajectories, distances, kernel values, dot products,
activations, qdot, cost, the updated policy means, n_updated) as DIR/<name>.npy, at most 64 MB (a fixed, seeded
subset of samples beyond that); the inputs are seeded, so two builds run with the same arguments compare array for
array.  On N > 1 GPUs only rank 0's shard of the samples is written (the policy means are the same on every rank).
`--steps K` is the number of timed iterations of `value` and of `e2e`; on the latency workload `integrator` a step is
one control tick (30 untimed warm-up ticks; a few hundred timed ticks give a stable rate).
On N > 1 GPUs the run first proves the NCCL path (`multi_gpu_check`: ranks bit-identical, sharded == single-rank
update; exit 3 otherwise) and adds `c5`, the BASELINE configs[4] shard shape (125 000 samples x 50 steps per GPU).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (net, shelf n_pts or None, N per GPU, H, K, nk, dt, dst_thr, ker_thr, alpha_s, sigma, ignored)
    "franka_shelf_2064": dict(net="franka", n_pts=32, N=4096, H=50, K=5, nk=10, dt=0.5, dst_thr=0.01, ker_thr=0.1,
                              alpha_s=3.0, sigma=1.0, ignored=[0, 1, 2]),
    "franka_shelf_294": dict(net="franka", n_pts=12, N=4096, H=50, K=5, nk=10, dt=0.5, dst_thr=0.01, ker_thr=0.1,
                             alpha_s=3.0, sigma=1.0, ignored=[0, 1, 2]),
    "planar7": dict(net="planar7", n_pts=None, N=1000, H=30, K=1, nk=10, dt=0.3, dst_thr=0.25, ker_thr=1e-3,
                    alpha_s=0.75, sigma=0.5, ignored=[]),
    # BASELINE.json configs[0]: planar 2-DoF, script defaults (standalonePlanar2d.py:76-77,109-129)
    "planar2": dict(net="planar2", n_pts=None, N=100, H=10, K=2, nk=10, dt=0.3, dst_thr=0.25, ker_thr=1e-3,
                    alpha_s=2.0, sigma=0.5, ignored=[]),
    # BASELINE.json configs[3]: dense velocity-field evaluation over a 1000 x 1000 joint-space grid (policy-plot
    # path, standalonePlanar2d_policyPlots.py:160,257-259): H = 1, per-sample start states
    "field_1m": dict(net="planar2", n_pts=None, N=1_000_000, H=1, K=1, nk=10, dt=0.05, dst_thr=0.25, ker_thr=1e-3,
                     alpha_s=2.0, sigma=0.5, ignored=[], grid=1000),
    # SURVEY 8(f).3: the integrator process's control tick (frankaIntegrator.py:101-121): ONE sample, TWO steps, 28
    # spheres, CPU caller tensors -- a latency workload: `value` = 2 x tick rate, `ms_per_step` = wall clock per tick
    "integrator": dict(net="franka", n_pts=12, N=1, H=2, K=5, nk=5, dt=0.01, dst_thr=0.03, ker_thr=0.1,
                       alpha_s=0.0, sigma=1.0, ignored=[0, 1, 2], n_obs=28),
}


def shelf(n_pts):
    """Shelf point cloud of the reference's obstacle streamer (obstacleStreamer.py:87-108), restated."""
    r = 0.03
    length = max(1, 2 * n_pts - 2) * r * 1.5
    posA = torch.tensor([0.45, 0.0, 0.15 + length, r])
    posB = posA + torch.tensor([length / 3, 0.0, 0.0, 0.0])
    line = posA + torch.linspace(0, 1, n_pts // 2).reshape(-1, 1) * (posB - posA)
    out = line
    span = torch.linspace(0, 1, n_pts).reshape(-1, 1)
    for s in line:
        down = s + span * (torch.tensor([0, 0, -length, 0]))
        left = s + torch.tensor([0, -length / 2, -length / 2, 0])
        right = s + torch.tensor([0, length / 2, -length / 2, 0])
        lr = left + span * (right - left)
        out = torch.vstack((out, down, lr, lr + torch.tensor([0, 0, length / 2, 0]),
                            lr + torch.tensor([0, 0, -length / 2, 0])))
    return out


def problem(name):
    w = WORKLOADS[name]
    pi = math.pi
    if w["net"] == "franka":
        dh_a = torch.tensor([0, 0, 0, 0.0825, -0.0825, 0, 0.088, 0])
        dh_d = torch.tensor([0.333, 0, 0.316, 0, 0.384, 0, 0, 0.107])
        dh_alpha = torch.tensor([0, -pi / 2, pi / 2, pi / 2, -pi / 2, pi / 2, pi / 2, 0])
        dh = torch.vstack((dh_d, dh_a * 0, dh_a, dh_alpha)).T.contiguous()
        q0 = torch.tensor([-0.88, 0.38, 0.5, -1, 0.45, 1.9, 0.31])
        qf = torch.tensor([-1.24, 1.53, 1.22, -1.21, -0.21, 1.55, 0.08])
        obs = shelf(w["n_pts"])
        if w.get("n_obs"):
            obs = obs[:w["n_obs"]].clone()
        qlim = (torch.tensor([-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973]),
                torch.tensor([2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973]))
        dof, out = 7, 9
    elif w["net"] == "planar2":
        dof, out = 2, 2
        dh_a = torch.zeros(dof + 1); dh_a[1:] = 3
        dh = torch.vstack((dh_a * 0, dh_a * 0, dh_a, dh_a * 0)).T.contiguous()
        q0 = torch.tensor([-3.14, 0.0])
        qf = torch.tensor([3.14, 0.0])
        obs = torch.tensor([[6, 0, 0, .5], [0., 4.5, 0, .5]])
        qlim = (-0.99 * 3.14 * torch.ones(dof), 0.99 * 3.14 * torch.ones(dof))
    else:
        dof, out = 7, 7
        dh_a = torch.zeros(dof + 1); dh_a[1:] = 1
        dh = torch.vstack((dh_a * 0, dh_a * 0, dh_a, dh_a * 0)).T.contiguous()
        q0 = torch.zeros(dof); q0[0] = pi / 2
        qf = torch.zeros(dof); qf[0] = -pi / 2
        obs = torch.tensor([[6, 2, 0, .5], [4., -1, 0, .5], [5, 0, 0, .5], [6, 6, 6, .1]])
        qlim = (-3.2 * torch.ones(dof), 3.2 * torch.ones(dof))
    return dict(w, dof=dof, out=out, dh=dh, dh_a=dh_a, q0=q0, qf=qf, obs=obs, qlim=qlim)


def flops_per_state_step(p):
    d, O, M, K = p["dof"], p["out"], p["obs"].shape[0], p["K"]
    f_fwd = 2 * (3 * (d + 3) * 256 + 3 * 256 * 256 + 256 * O)
    f_bwd = 2 * (3 * 256 * 256 + 3 * (d + 3) * 256)
    return f_fwd, f_bwd, M * f_fwd + K * (f_fwd + f_bwd)


def load_net_arrays(name):
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "weights", name + ".npz")
    if os.path.exists(path):
        z = np.load(path)
        return [torch.from_numpy(z[f"W{i}"]) for i in range(5)], [torch.from_numpy(z[f"b{i}"]) for i in range(5)], "shipped"
    torch.manual_seed(0)
    d, O = {"franka": (7, 9), "planar7": (7, 7), "planar2": (2, 2)}[name]
    dims = [3 * (d + 3), 256, 256, 256, 256, O]
    lin = [torch.nn.Linear(dims[i], dims[i + 1]) for i in range(5)]
    return [l.weight.detach() for l in lin], [l.bias.detach() for l in lin], "random-init"


def seeded_policy(p, N, seed, mean_seed=100):
    """nk kernels pre-placed along q0 + 0.1 k (SURVEY 8(d)) and one Gaussian draw of the weights.  The policy MEANS
    come from `mean_seed` (every rank of a sharded job holds the same means, SURVEY 8(e)); the per-sample noise from
    `seed` (each rank draws its own samples; seed == mean_seed continues the same stream)."""
    g = torch.Generator().manual_seed(mean_seed)
    nk, d = p["nk"], p["dof"]
    mu_c = torch.zeros(50, d); sigma_c = torch.zeros(50); alpha_c = torch.zeros(50, d)
    for k in range(nk):
        mu_c[k] = p["q0"] + 0.1 * k
    sigma_c[:nk] = p["sigma"]
    alpha_c[:nk] = 0.5 * torch.randn(nk, d, generator=g)
    if seed != mean_seed:
        g = torch.Generator().manual_seed(seed)
    mu_tmp = torch.zeros(N, 50, d); sigma_tmp = torch.zeros(N, 50); alpha_tmp = torch.zeros(N, 50, d)
    mu_tmp[:, :nk] = mu_c[:nk]
    sigma_tmp[:, :nk] = sigma_c[:nk]
    alpha_tmp[:, :nk] = alpha_c[:nk] + p["alpha_s"] * torch.randn(N, nk, d, generator=g)
    alpha_tmp[0, :nk] = alpha_c[:nk]
    return mu_c, sigma_c, alpha_c, mu_tmp, sigma_tmp, alpha_tmp


# ---------------------------------------------------------------------------------------- CPU arm
def _sample_text(p, N, H, what, cores):
    return (f"{N} samples x {H} steps of the same workload (M={p['obs'].shape[0]}, K={p['K']}, nk={p['nk']}), "
            f"propagate+get_cost+shift_policy_means, {what}, torch CPU {cores} threads")


def cpu_reference_rate(p, target_seconds, steps=1, warmup=0):
    """state-steps/s of the REFERENCE'S OWN classes (oracle/_ref staged by oracle/make_ref.sh, imported through
    oracle/ref_harness.py with its two import shims) on the host cores, on a bounded sample of the workload: the full
    horizon, as many samples as fit `target_seconds` per step.  Falls back to the oracle port (kind "port") when the
    staged reference is absent."""
    from oracle import ref_harness as rh
    if not rh.available():
        return cpu_port_rate(p, target_seconds, steps, warmup)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    H = p["H"]
    q_grid = None
    if p.get("grid"):
        g = torch.linspace(-math.pi, math.pi, p["grid"])
        q_grid = torch.stack(torch.meshgrid(g, g, indexing="ij"), -1).reshape(-1, p["dof"])

    def build(N, Hh):
        it = rh.ReferenceIteration(p, N, Hh, seed=0, policy=seeded_policy(p, N, 100))
        if q_grid is not None:
            it.set_q_cur(q_grid[torch.linspace(0, q_grid.shape[0] - 1, N).long()].contiguous())
        return it

    def timed(it):
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):        # shift_policy_means prints (MPPI.py:343)
            t0 = time.perf_counter()
            it.step()
            return time.perf_counter() - t0

    probe = build(8, min(H, 2))            # the constructor runs the reference's five warm-up rollouts itself
    timed(probe)
    rate = 8 * min(H, 2) / timed(probe)
    N = int(max(2, min(p["N"], rate * target_seconds / H)))
    it = build(N, H)
    for _ in range(warmup):
        timed(it)
    times = [timed(it) for _ in range(steps)]
    t = sum(times) / len(times)
    return dict(value=N * H / t, ms_per_step=t * 1e3, cores=cores, N=N, H=H, kind="reference",
                sample=_sample_text(p, N, H, "UNMODIFIED reference classes from oracle/_ref (MPPI.py, cost.py, "
                                             "policy.py, robot_sdf.py)", cores))


def cpu_port_rate(p, target_seconds, steps=1, warmup=0):
    """The same measurement on the oracle port (oracle/mppi_oracle.py) -- only when the reference is not staged."""
    from oracle import mppi_oracle as orc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    W, b, _ = load_net_arrays(p["net"])
    net = orc.Net(W, b)
    prm = lambda H: orc.RolloutParams(dt=p["dt"], dt_H=H, n_closest_obs=p["K"], dst_thr=p["dst_thr"],  # noqa: E731
                                      ignored_links=p["ignored"], p=2.0, with_basis=False)

    def one(N, H, seed):
        mu_c, sigma_c, alpha_c, mu, sg, al = seeded_policy(p, N, seed)
        t0 = time.perf_counter()
        o = orc.rollout(net, p["q0"], p["qf"], p["obs"], mu, sg, al, p["nk"], prm(H), N)
        cost = orc.evaluate_costs(o.all_traj, o.closest_dist_all, p["qf"], p["dh"], p["qlim"][0], p["qlim"][1])
        orc.policy_update(cost, o.kernel_val_all, o.kernel_activations, mu, sg, al, mu_c, sigma_c, alpha_c, p["nk"],
                          p["ker_thr"])
        return time.perf_counter() - t0

    one(4, 1, 0)                                   # thread-pool / allocator warm-up
    t = one(8, 2, 1)
    rate = 16 / t
    H = p["H"]
    N = int(max(2, min(p["N"], rate * target_seconds / H)))
    for _ in range(warmup):
        one(N, H, 2)
    times = [one(N, H, 3 + i) for i in range(steps)]
    t = sum(times) / len(times)
    return dict(value=N * H / t, ms_per_step=t * 1e3, cores=cores, N=N, H=H, kind="port",
                sample=_sample_text(p, N, H, "oracle port (reference not staged)", cores))


# ---------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    NAMES = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.NAMES.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons),
                    samples=len(s))


# ---------------------------------------------------------------------------------------- GPU arm
C5_SAMPLES_PER_GPU = 125_000       # BASELINE.json configs[4]: 10^6 samples x 50 steps sharded over 8 GPUs


def build_mppi(p, N, H, dev, args, seed, world):
    """The drop-in MPPI object on `dev` with the workload's parameters and a seeded sampled policy."""
    from optimalmodulationds_b200 import MPPI, LinDS
    from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
    W, b, wsrc = load_net_arrays(p["net"])
    net = RobotSdfCollisionNet(in_channels=p["dof"] + 3, out_channels=p["out"], layers=[256] * 4, skips=[])
    net.load_arrays(W, b)
    t = lambda x: x.to(dev)  # noqa: E731
    DS = [LinDS(t(p["qf"])), LinDS(t(p["q0"]))]
    mppi = MPPI(t(p["q0"]), t(p["qf"]), t(p["dh"]), t(p["obs"]), p["dt"], H, N, DS, t(p["dh_a"]), net, p["K"])
    mppi.set_pass1_mode(args.pass1)
    mppi.set_score_mode(args.score)
    if args.per_step:
        mppi.set_whole_horizon(False)
    mppi.dst_thr, mppi.ker_thr, mppi.ignored_links = p["dst_thr"], p["ker_thr"], list(p["ignored"])
    mppi.Cost.q_min, mppi.Cost.q_max = t(p["qlim"][0]), t(p["qlim"][1])
    if world > 1:
        mppi.enable_sample_sharding()
    pol = seeded_policy(p, N, seed)
    load_policy(mppi, p, pol, dev)
    return mppi, pol, wsrc


def load_policy(mppi, p, pol, dev):
    mu_c, sigma_c, alpha_c, mu_tmp, sigma_tmp, alpha_tmp = pol
    P = mppi.Policy
    P.n_kernels = p["nk"]
    for dst, src in ((P.mu_c, mu_c), (P.sigma_c, sigma_c), (P.alpha_c, alpha_c), (P.mu_tmp, mu_tmp),
                     (P.sigma_tmp, sigma_tmp), (P.alpha_tmp, alpha_tmp)):
        dst.copy_(src.to(dev))


def policy_vector(mppi):
    P = mppi.Policy
    return torch.cat((P.mu_c.flatten(), P.sigma_c.flatten(), P.alpha_c.flatten())).float()


DUMP_BYTES = 63_000_000     # array data of one --dump-outputs directory; the .npy headers stay well inside 64 MB


def dump_outputs(out_dir, per_sample, other, seed=0):
    """Writes every array as <out_dir>/<name>.npy: float32 stays float32, anything else becomes float64.
    `per_sample` arrays have the sample axis first; when all arrays together would pass DUMP_BYTES, the same fixed,
    seeded subset of samples is kept of each of them and its indices are written as sample_index.npy."""
    import numpy as np

    def host(t):
        t = torch.as_tensor(t).detach().cpu()
        return (t if t.dtype == torch.float32 else t.double()).numpy()

    per_sample = {k: host(v) for k, v in per_sample.items()}
    other = {k: host(v) for k, v in other.items()}
    n = next(iter(per_sample.values())).shape[0]
    row_bytes = sum(a.nbytes for a in per_sample.values()) // n
    budget = DUMP_BYTES - sum(a.nbytes for a in other.values())
    if row_bytes * n > budget:
        keep = np.sort(np.random.default_rng(seed).choice(n, budget // (row_bytes + 8), replace=False))
        per_sample = {k: a[keep] for k, a in per_sample.items()}
        other["sample_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in {**per_sample, **other}.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure_control_tick(dev_index, ticks=400, n_obs=28):
    """The integrator process's loop (frankaIntegrator.py:101-121): ONE sample, TWO steps per control tick, CPU tensors
    in and out as that script uses them -- update_obstacles, sample_policy, propagate, q += qdot * dt, clamp.  Wall
    clock per tick, everything included (this is a latency figure, the reference logs ~500 Hz for it).  The drop-in
    replays one CUDA graph per propagate() at this size (MPPI._propagate_tick).  Returns the timing and what the last
    tick computed."""
    from optimalmodulationds_b200 import MPPI, LinDS
    from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
    torch.manual_seed(0)                                   # sample_policy draws from the global generator
    p = problem("franka_shelf_294")
    obs = p["obs"][:n_obs].clone()
    W, b, _ = load_net_arrays("franka")
    net = RobotSdfCollisionNet(in_channels=10, out_channels=9, layers=[256] * 4, skips=[])
    net.load_arrays(W, b)
    os.environ.setdefault("DSMPPI_DEVICE", str(dev_index))
    m = MPPI(p["q0"].clone(), p["qf"].clone(), p["dh"], obs, 0.01, 2, 1, [LinDS(p["qf"].clone()), LinDS(p["q0"].clone())],
             p["dh_a"], net, p["K"])
    m.dst_thr = 0.03
    P = m.Policy
    P.alpha_s, P.sigma_c_nominal = 0.0, 1.0
    for k in range(5):                                     # the planner has published a few kernels
        P.add_kernel(p["q0"] + 0.1 * k, 0.1, torch.eye(7))
    P.alpha_c[:5] = 0.3

    def tick():
        m.update_obstacles(obs)
        P.sample_policy()
        out = m.propagate()
        m.q_cur = torch.clamp(m.q_cur + m.qdot[0, :] * 0.01, m.Cost.q_min, m.Cost.q_max)
        return out

    for _ in range(30):
        tick()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(ticks):
        out = tick()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / ticks
    traj, dist_all, kval, dots, acts = out
    outputs = dict(all_traj=traj, closest_dist_all=dist_all, kernel_val_all=kval, dot_products=dots,
                   kernel_activations=acts, qdot=m.qdot), dict(q_cur=m.q_cur)
    return dict(hz=1.0 / dt, ms_per_tick=dt * 1e3, ticks=ticks, graphed="_tick" in m.__dict__,
                config=f"Franka net, {n_obs} spheres, N=1, H=2, K={p['K']}, 5 kernels, CPU caller tensors, "
                       "loop of frankaIntegrator.py:101-121 (update_obstacles, sample_policy, propagate, q += qdot dt)",
                timing="wall clock per tick incl. host wrapper, H2D, launch, D2H"), outputs


def check_sharding(p, dev, args, rank, world, mppi_main):
    """Evidence that the NCCL path computes the unsharded update (exit != 0 otherwise):
      1. after the timed iterations every rank holds bit-identical policy means;
      2. a small job (256 samples per rank, 8 steps, the workload's obstacles) run sample-sharded over the ranks gives
         the policy of ONE rank running all world x 256 samples, and the same trajectories for its slice."""
    import torch.distributed as dist
    mine = policy_vector(mppi_main)
    every = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(every, mine)
    identical = all(torch.equal(every[0], e) for e in every)
    n_small, h_small = 256, 8
    pol_all = seeded_policy(p, world * n_small, 4242, mean_seed=4242)  # the same global draw on every rank
    lo, hi = rank * n_small, (rank + 1) * n_small
    sl = (pol_all[0], pol_all[1], pol_all[2], pol_all[3][lo:hi].clone(), pol_all[4][lo:hi].clone(),
          pol_all[5][lo:hi].clone())
    sharded, _, _ = build_mppi(p, n_small, h_small, dev, args, 0, world)
    load_policy(sharded, p, sl, dev)
    traj_s = sharded.propagate()[0].clone()
    cost_s = sharded.get_cost().clone()
    n_upd_s = int(sharded.shift_policy_means()[1])
    whole, _, _ = build_mppi(p, world * n_small, h_small, dev, args, 0, 1)
    load_policy(whole, p, pol_all, dev)
    traj_w = whole.propagate()[0]
    cost_w = whole.get_cost()
    n_upd_w = int(whole.shift_policy_means()[1])
    a, b = policy_vector(sharded), policy_vector(whole)
    pol_err = float(((a - b).abs() / (b.abs() + 1e-6)).max())
    traj_err = float((traj_s - traj_w[lo:hi]).abs().max())
    cost_err = float(((cost_s - cost_w[lo:hi]).abs() / (cost_w[lo:hi].abs() + 1e-6)).max())
    res = torch.tensor([pol_err, traj_err, cost_err, float(n_upd_s != n_upd_w), float(not identical)], device=dev)
    dist.all_reduce(res, op=dist.ReduceOp.MAX)
    out = dict(ranks_hold_identical_policy=bool(res[4] == 0), sharded_vs_single_rank_policy_max_rel=float(res[0]),
               sharded_vs_single_rank_traj_max_abs=float(res[1]), sharded_vs_single_rank_cost_max_rel=float(res[2]),
               n_updated_equal=bool(res[3] == 0), small_job=f"{world} x {n_small} samples x {h_small} steps",
               tolerance="policy 1e-4 rel, trajectories 1e-5 abs, cost 1e-4 rel")
    out["ok"] = bool(out["ranks_hold_identical_policy"] and out["n_updated_equal"] and res[0] <= 1e-4 and
                     res[1] <= 1e-5 and res[2] <= 1e-4)
    del sharded, whole
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="franka_shelf_2064", choices=sorted(WORKLOADS))
    ap.add_argument("--samples", type=int, default=0, help="samples per GPU (default: the workload's)")
    ap.add_argument("--pass1", default="auto", choices=["auto", "exact", "tc_f16", "tc_bf16"])
    ap.add_argument("--score", default="auto", choices=["auto", "ffma", "tc_split"],
                    help="arithmetic of the scoring rows: split-fp16 tcgen05 (default) or strict IEEE FFMA")
    ap.add_argument("--per-step", action="store_true", help="disable the whole-horizon single-launch path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the configs[4]-shaped record of multi-GPU runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0's samples)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    p = problem(args.workload)
    if args.samples:
        p["N"] = args.samples
    N, H = p["N"], p["H"]
    M = p["obs"].shape[0]
    f_fwd, f_bwd, f_step = flops_per_state_step(p)
    robot = {"franka": "franka_panda_7dof", "planar7": "planar_7dof", "planar2": "planar_2dof"}[p["net"]]
    warm = max(args.warmup, 3)
    # `config` is the same dictionary in both arms (the driver compares them); run-time diagnostics go to "diagnostics"
    config = dict(workload=args.workload, robot=robot,
                  n_obstacles=M, samples_per_gpu=N, horizon=H, n_closest_obs=p["K"], n_kernels=p["nk"],
                  weights="shipped checkpoint (tests/golden/weights == mlp_learn/models/*.pt)",
                  sharding=f"samples x{world}",
                  l2="flushed between timed steps (256 MiB write, outside the per-step event pairs)")
    if world > 1 and args.workload.startswith("franka_shelf") and not args.no_c5:
        config["c5"] = dict(workload="BASELINE.json configs[4] shard shape", samples_per_gpu=C5_SAMPLES_PER_GPU,
                            horizon=H, n_obstacles=M, timed_iterations=2)

    if args.impl == "reference":
        if rank != 0:
            return
        K = max(1, args.steps)
        r = cpu_reference_rate(p, target_seconds=max(1.0, 75.0 / (K + warm)), steps=K, warmup=warm)
        line = dict(metric="mppi_rollout_state_steps_per_sec", value=r["value"], unit="state-steps/s", n_gpus=0,
                    steps=K, warmup=warm, ms_per_step=r["ms_per_step"], higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", config=config, impl="reference",
                    cpu_baseline=dict(value=r["value"], unit="state-steps/s", cores=r["cores"], kind=r["kind"],
                                      sample=r["sample"]),
                    e2e=dict(value=r["value"], unit="state-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0)
        print(json.dumps(line))
        return

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if args.workload == "integrator":
        # a latency workload: no batch to shard, every rank would run the same tick -- rank 0 reports it
        if rank != 0:
            return
        sampler = ClockSampler(local_rank)
        sampler.start()
        tick, outputs = measure_control_tick(local_rank, ticks=args.steps)
        sampler.stop_flag = True
        sampler.join()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *outputs)
        line = dict(metric="mppi_rollout_state_steps_per_sec", value=2 * tick["hz"], unit="state-steps/s", n_gpus=1,
                    steps=tick["ticks"], warmup=30, ms_per_step=tick["ms_per_tick"], higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="f32 (scoring: split-fp16 tcgen05, fp32-accurate)",
                    data="synthetic", config=config, clocks=sampler.summary(), control_tick=tick,
                    e2e=dict(value=2 * tick["hz"], unit="state-steps/s", h2d_bytes_per_step=4 * (7 + 28 * 4 + 50 * 15),
                             d2h_bytes_per_step=4 * (2 * 7 * 2 + 2 * 3 + 2 * 50 + 7), ms_per_step=tick["ms_per_tick"],
                             api="MPPI.propagate on CPU tensors -> dsmppi_tick (C ABI, one replayed CUDA graph)"),
                    gpu_launches=2 * tick["ticks"], roofline=None,
                    note="latency workload: the tick IS the end-to-end call (host tensors in and out); reference logs "
                         "~500 Hz for this loop (experiment_logs/my_*.txt)")
        print(json.dumps(line))
        return
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t = lambda x: x.to(dev)  # noqa: E731
    mppi, pol, wsrc = build_mppi(p, N, H, dev, args, 100 + rank, world)
    mu_c, sigma_c, alpha_c, mu_tmp, sigma_tmp, alpha_tmp = pol
    q_start = p["q0"]
    if p.get("grid"):            # dense field: every sample starts at its own grid point (MPPI.py:99 broadcast)
        g = torch.linspace(-math.pi, math.pi, p["grid"])
        q_start = torch.stack(torch.meshgrid(g, g, indexing="ij"), -1).reshape(-1, p["dof"])[:N].contiguous()
        mppi.q_cur = t(q_start)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)

    def step(m=mppi):
        out = m.propagate()
        cost = m.get_cost()
        _, n_updated = m.shift_policy_means()
        return out, cost, n_updated

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed_steps(m, n_steps, with_kernel_timing):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
        kt_ms, kt_n, name = 0.0, 0, "exact_mlp_kernel"
        sync_all()
        last = None
        for a, bq in evs:
            flush.fill_(1.0)
            a.record()
            last = step(m)
            bq.record()
            bq.synchronize()
            if with_kernel_timing:
                kt = m.kernel_timing_ex()
                name = kt["kernel"]
                kt_ms += kt["ms"] * kt["launches"]
                kt_n += kt["launches"]
        sync_all()
        ms = torch.tensor([sum(a.elapsed_time(bq) for a, bq in evs) / n_steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), kt_ms, kt_n, name, last

    for _ in range(warm):
        step()
    sync_all()
    mppi.enable_kernel_timing(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = mppi.launch_count()
    ms_per_step, kt_ms, kt_n, kern_name, last = timed_steps(mppi, args.steps, True)
    launches = mppi.launch_count() - launches0
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs and rank == 0:
        (traj, dist_all, kval, dots, acts), cost, n_updated = last
        P = mppi.Policy
        dump_outputs(args.dump_outputs,
                     dict(all_traj=traj, closest_dist_all=dist_all, kernel_val_all=kval, dot_products=dots,
                          kernel_activations=acts, qdot=mppi.qdot, cost=cost),
                     dict(mu_c=P.mu_c, sigma_c=P.sigma_c, alpha_c=P.alpha_c, n_updated=n_updated))
    value = world * N * H / (ms_per_step * 1e-3)
    stats = mppi.pass1_stats()
    xstats = mppi.exactness_stats()
    mppi.enable_kernel_timing(False)

    # ---- multi-GPU: prove the NCCL path before reporting it
    mg_check = None
    if world > 1:
        mg_check = check_sharding(p, dev, args, rank, world, mppi)
        if not mg_check["ok"]:
            if rank == 0:
                print(json.dumps(dict(error="sample-sharded update disagrees with the single-rank update",
                                      multi_gpu_check=mg_check)), file=sys.stderr)
            dist.destroy_process_group()
            sys.exit(3)

    # ---- e2e: the same iteration through the C ABI with pinned HOST buffers (H2D + D2H inside the timed region);
    #      on several GPUs it stays sample-sharded: the library calls back for the two all-reduces (NCCL)
    pin = lambda x: x.contiguous().pin_memory()  # noqa: E731
    d = p["dof"]
    host = dict(q_cur=pin(q_start), mu_tmp=pin(mu_tmp), sigma_tmp=pin(sigma_tmp), alpha_tmp=pin(alpha_tmp),
                mu_c=pin(mu_c), sigma_c=pin(sigma_c), alpha_c=pin(alpha_c),
                all_traj=pin(torch.empty(N, H, d)), closest_dist_all=pin(torch.empty(N, H)),
                kernel_val_all=pin(torch.zeros(N, H, 50)), dot_products=pin(torch.empty(N, H)),
                kernel_activations=pin(torch.empty(N, H)), qdot=pin(torch.empty(N, d)), cost=pin(torch.empty(N)),
                n_updated=pin(torch.zeros(1, dtype=torch.int32)))
    for _ in range(2):
        h2d, d2h = mppi.iteration_host(host)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        h2d, d2h = mppi.iteration_host(host)
    torch.cuda.synchronize(dev)
    e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.steps], device=dev)
    if world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
        hp = torch.cat((host["mu_c"].flatten(), host["sigma_c"], host["alpha_c"].flatten())).to(dev)
        every = [torch.empty_like(hp) for _ in range(world)]
        dist.all_gather(every, hp)
        mg_check["e2e_ranks_hold_identical_policy"] = all(torch.equal(every[0], e) for e in every)
        if not mg_check["e2e_ranks_hold_identical_policy"]:
            if rank == 0:
                print(json.dumps(dict(error="ranks disagree after the sharded host-buffer iteration")), file=sys.stderr)
            dist.destroy_process_group()
            sys.exit(3)
    e2e_value = world * N * H / (float(e_ms) * 1e-3)

    # ---- configs[4]: 10^6 samples x 50 steps over 8 GPUs = 125 000 samples per GPU, sample-sharded
    c5 = None
    if "c5" in config:
        del mppi, host
        torch.cuda.empty_cache()
        m5, _, _ = build_mppi(p, C5_SAMPLES_PER_GPU, H, dev, args, 500 + rank, world)
        step(m5)
        ms5, _, _, _, _ = timed_steps(m5, 2, False)
        c5 = dict(samples_per_gpu=C5_SAMPLES_PER_GPU, samples_total=world * C5_SAMPLES_PER_GPU, horizon=H,
                  n_obstacles=M, ms_per_iteration=ms5, timed_iterations=2, warmup=1,
                  value=world * C5_SAMPLES_PER_GPU * H / (ms5 * 1e-3), unit="state-steps/s",
                  timing="CUDA events per iteration, max over ranks", exactness=m5.exactness_stats())
        mppi = m5

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (measured)" if peaks else "fallback 1.4 PFLOP/s sustained"
    mode = {0: "exact_fp32", 1: "tc_f16", 2: "tc_bf16"}.get(stats["mode"], str(stats["mode"]))
    sstats = mppi.score_stats()
    tensor_kernel = kern_name.startswith("tc_")
    if not tensor_kernel:
        peak_tf, peak_src = 74.0, "FFMA nominal 74 TFLOP/s (IEEE fp32 scoring kernel; no tensor cores in this mode)"
    kern_ms = kt_ms / max(kt_n, 1)
    traffic, traffic_src = None, None
    try:      # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu capture
        prof = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        ent = prof.get(f"{args.workload}:{kern_name}")
        if ent and ent.get("samples") == N:
            traffic = ent["dram_bytes_per_launch"]
            traffic_src = ent.get("source")
    except Exception:  # noqa: BLE001
        pass
    # algorithmic FLOPs of the dominant kernel: the all-pairs forward (tensor-core prefilter, or the scoring kernel's
    # forward when M > 16), or forward + input gradient on every pair when few obstacles make one launch cheaper; the
    # whole-horizon kernels do that for all H steps in one launch
    whole = kern_name in ("rollout_fused_kernel", "tc_exact_kernel<whole horizon>")
    if whole:
        launches_per_iter = max(1, round(kt_n / args.steps))         # > 1 when a huge batch is rolled out in blocks
        flops_per_launch = N * M * (f_fwd + f_bwd) * H / launches_per_iter
    else:
        f_pair = f_fwd if (stats["mode"] or M > 16) else f_fwd + f_bwd
        launches_per_step = max(1, round(kt_n / (args.steps * H)))
        flops_per_launch = N * M * f_pair / launches_per_step
    achieved = flops_per_launch / (kern_ms * 1e-3) / 1e12 if kern_ms > 0 else 0.0
    hacc = mode == "tc_f16" and os.environ.get("DSMPPI_PASS1_ACC", "f16") != "f32"
    pipe = {"tc_pass1_kernel": ("tcgen05 f16 operands, f16 accumulators in the hidden layers, f32 in the output layer "
                                "(obstacle-ranking prefilter)" if hacc else
                                "tcgen05 f16 operands, f32 accumulators (obstacle-ranking prefilter)"),
            "tc_exact_kernel": "tcgen05 f16, split operands: 3 MMAs per algorithmic product sum",
            "tc_exact_kernel<whole horizon>": "tcgen05 f16, split operands: 3 MMAs per algorithmic product sum"}.get(
                kern_name, "fp32 FFMA (compute-bound; no tensor cores)")
    roofline = dict(bound="tensor", pipe=pipe, kernel=kern_name,
                    achieved=achieved, peak=peak_tf, unit="TFLOP/s", frac=achieved / peak_tf, traffic=traffic,
                    traffic_source=traffic_src,
                    peak_source=peak_src, flops_per_launch=flops_per_launch, ms_per_launch=kern_ms, launches_timed=kt_n,
                    share_of_step=kt_ms / args.steps / ms_per_step)
    if kern_name == "tc_pass1_kernel" and hacc:
        # the denominator is a power-capped cuBLAS bf16 GEMM with fp32 accumulators; an MMA with fp16 accumulators
        # draws less power, so on this power-bound kernel the fraction may pass 1 (tools/tc_microbench.cu `power`:
        # the bare MMA loop sustains 1.63 PFLOP/s with fp32 and 1.68 PFLOP/s with fp16 accumulators on this part)
        roofline["peak_note"] = ("peak = power-capped bf16 GEMM with fp32 accumulators; this kernel's hidden layers "
                                 "accumulate in fp16 (less energy per MMA), bare-MMA-loop ceiling 1677 TFLOP/s")
        roofline["frac_of_mma_loop_ceiling"] = achieved / 1677.0
    if kern_name.startswith("tc_exact"):
        # fp32-accurate scoring issues three fp16 MMAs per algorithmic multiply-add: its ceiling is a third of the peak
        roofline["mma_flops_per_algorithmic_flop"] = 3
        roofline["frac_of_split_ceiling"] = 3 * achieved / peak_tf
    line = dict(metric="mppi_rollout_state_steps_per_sec", value=value, unit="state-steps/s", n_gpus=world,
                steps=args.steps, warmup=warm, ms_per_step=ms_per_step, higher_is_better=True,
                scaling="weak", vs_baseline=None,
                dtype=("f32 (scoring: split-fp16 tcgen05, fp32 accumulate, fp32-accurate; obstacle-ranking prefilter: "
                       "f16 tcgen05, re-scored in fp32 inside its calibrated guard band)" if sstats["mode"] == "tc_split" else
                       "f32 (IEEE FFMA scoring; obstacle-ranking prefilter: f16 tcgen05, f32 accumulate)"),
                data="synthetic", config=config,
                diagnostics=dict(pass1=mode, score=sstats["mode"], weights_source=wsrc,
                                 range_fixup_rows=sstats["range_fixup_rows"],
                                 rescored_pairs_per_state_step=stats["rescored_pairs"] / (N * H),
                                 crowded_bands=stats["band_overflows"], guard_band_m=xstats["guard_band"],
                                 prefilter_calibration_error_m=xstats["calibration_error"],
                                 capacity_retries=xstats["capacity_retries"], exact_fallbacks=xstats["exact_fallbacks"],
                                 flops_per_state_step=f_step),
                clocks=sampler.summary(),
                e2e=dict(value=e2e_value, unit="state-steps/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                         ms_per_step=float(e_ms),
                         api="dsmppi_iteration_host (C ABI, pinned host buffers" +
                             (", sample-sharded: two NCCL all-reduces per iteration through the exchange hook)"
                              if world > 1 else ")")),
                gpu_launches=launches, roofline=roofline,
                ms_per_mppi_iteration=ms_per_step)
    if mg_check is not None:
        line["multi_gpu_check"] = mg_check
    if c5 is not None:
        line["c5"] = c5
    if world == 1:
        del mppi
        torch.cuda.empty_cache()
        line["control_tick"] = measure_control_tick(local_rank)[0]
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_rate(p, target_seconds=15.0)
        line["cpu_baseline"] = dict(value=r["value"], unit="state-steps/s", cores=r["cores"], kind=r["kind"],
                                    sample=r["sample"])
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
