#!/usr/bin/env python
"""Planner + stepper loop for the planar 7-DoF arm, written the way the reference's single-process demos use
the MPPI object (ds_mppi/scripts/standalonePlanar7d.py:95-185): the modules are imported under the REFERENCE'S
names (`from MPPI import *`, `from LinDS import *`, `from sdf.robot_sdf import RobotSdfCollisionNet`) through
optimalmodulationds_b200/dropin, CPU tensors go in and come out, attributes are poked after construction, and a
second 1-sample x 1-step MPPI object moves the robot.  Headless (the drop-in `plots` module draws nothing).

    python examples/planar7_loop.py [--iters 200] [--checkpoint path/to/7dof_sdf_256x5_mesh.pt] [--layers 128x3]

--layers WxL builds a seeded random-init network of L hidden layers of width W instead of the shipped 256 x 4 weights
(any 1 <= L <= 4, W <= 256 runs; a checkpoint of that shape can be loaded with --checkpoint as well).
"""
import argparse
import copy
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "optimalmodulationds_b200", "dropin"))   # what PYTHONPATH would do

from MPPI import *  # noqa: E402,F401,F403  (torch, time, np, plt, numeric_fk_model, MPPI, ...)
from LinDS import *  # noqa: E402,F401,F403
from sdf.robot_sdf import RobotSdfCollisionNet  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--layers", default=None, help="WxL: L hidden layers of width W (default: the shipped 256x4)")
    args = ap.parse_args()
    params = {'device': 'cpu', 'dtype': torch.float32}                       # noqa: F405
    DOF, L = 7, 1
    width, depth = (int(x) for x in (args.layers or "256x4").split("x"))
    torch.manual_seed(0)                                                     # noqa: F405
    nn_model = RobotSdfCollisionNet(in_channels=DOF + 3, out_channels=DOF, layers=[width] * depth, skips=[])
    if args.checkpoint:
        nn_model.load_weights(args.checkpoint, params)
    elif args.layers:
        print(f"seeded random-init {width}x{depth} distance network")
    else:
        z = np.load(os.path.join(ROOT, "tests", "golden", "weights", "planar7.npz"))   # noqa: F405
        nn_model.load_arrays([z[f"W{i}"] for i in range(5)], [z[f"b{i}"] for i in range(5)])
    nn_model.model.to(**params)
    nn_model.update_aot_lambda()

    q_0 = torch.zeros(DOF).to(**params)                                      # noqa: F405
    q_f = torch.zeros(DOF).to(**params)                                      # noqa: F405
    q_0[0], q_f[0] = torch.pi / 2, -torch.pi / 2                             # noqa: F405
    dh_a = torch.zeros(DOF + 1).to(**params)                                 # noqa: F405
    dh_a[1:] = L
    dh_params = torch.vstack((dh_a * 0, dh_a * 0, dh_a, dh_a * 0)).T         # noqa: F405
    obs = torch.tensor([[6, 2, 0, .5], [4., -1, 0, .5], [5, 0, 0, .5], [6, 6, 6, .1]]).to(**params)   # noqa: F405
    r_h = init_robot_plot(dh_params, -10, 10, -10, 10)                       # noqa: F405
    c_h = init_kernel_means(100)                                             # noqa: F405
    plot_obs_init(obs)                                                       # noqa: F405
    DS_ARRAY = [LinDS(q_f), LinDS(q_0)]                                      # noqa: F405
    N_traj, dt_H, dt, dt_sim = 20, 10, 0.3, 0.02
    dst_thr, thr_rbf_add, thr_dot_add = 0.5, 0.2, -0.9

    mppi = MPPI(q_0, q_f, dh_params, obs, dt, dt_H, N_traj, DS_ARRAY, dh_a, nn_model, 1)   # noqa: F405
    mppi.Policy.sigma_c_nominal = 0.5
    mppi.Policy.alpha_s = 0.75
    mppi.Policy.policy_upd_rate = 0.5
    mppi.dst_thr = dst_thr / 2
    mppi.ker_thr = 1e-3
    mppi.ignored_links = []
    mppi_step = MPPI(q_0, q_f, dh_params, obs, dt_sim, 1, 1, DS_ARRAY, dh_a, nn_model, 1)   # noqa: F405
    mppi_step.Policy.alpha_s *= 0
    mppi_step.ignored_links = []
    mppi_step.dst_thr = 1

    torch.manual_seed(0)                                                     # noqa: F405
    d0 = float(torch.norm(mppi.q_cur - q_f))                                 # noqa: F405
    n_iter, t0 = 0, time.time()                                              # noqa: F405
    while torch.norm(mppi.q_cur - q_f) > 0.1 and n_iter < args.iters:        # noqa: F405
        mppi.Policy.sample_policy()
        with record_function("TAG: general propagation"):                    # noqa: F405
            all_traj, closest_dist_all, kernel_val_all, dot_all, _ = mppi.propagate()
        with record_function("TAG: cost calculation"):                       # noqa: F405
            cost = mppi.get_cost()
            best_idx = torch.argmin(cost)                                    # noqa: F405,F841
            mppi.shift_policy_means()
        cand = mppi.Policy.check_traj_for_kernels(all_traj, closest_dist_all, dot_all, dst_thr - mppi.dst_thr,
                                                  thr_rbf_add, thr_dot_add)
        if len(cand) > 0:
            pick = torch.randint(cand.shape[0], (1,))[0]                     # noqa: F405
            near_norm, near_idx = torch.norm(cand - mppi.q_cur, 2, -1).min(dim=0)   # noqa: F405
            if near_norm < 1e-1:
                pick = near_idx
            idx_i, idx_h = torch.where((all_traj == cand[pick]).all(dim=-1))  # noqa: F405
            mppi.Policy.add_kernel(cand[pick], closest_dist_all[idx_i[0], idx_h[0]],
                                   mppi.norm_basis[idx_i[0], idx_h[0]].squeeze())
            kernel_fk, _ = numeric_fk_model(cand[pick], dh_params, 2)        # noqa: F405
            upd_r_h(kernel_fk.to('cpu'), c_h[(mppi.Policy.n_kernels - 1) % len(c_h)])   # noqa: F405
        mppi_step.Policy.mu_c = mppi.Policy.mu_c
        mppi_step.Policy.sigma_c = mppi.Policy.sigma_c
        mppi_step.Policy.alpha_c = mppi.Policy.alpha_c
        mppi_step.Policy.n_kernels = mppi.Policy.n_kernels
        mppi_step.Policy.sample_policy()
        mppi_step.q_cur = copy.copy(mppi.q_cur)
        mppi_step.propagate()
        mppi.q_cur = mppi.q_cur + mppi_step.qdot[0, :] * dt_sim
        cur_fk, _ = numeric_fk_model(mppi.q_cur, dh_params, 10)              # noqa: F405
        upd_r_h(cur_fk.to('cpu'), r_h)                                       # noqa: F405
        plt.pause(0.0001)                                                    # noqa: F405
        n_iter += 1
    td = time.time() - t0                                                    # noqa: F405
    d1 = float(torch.norm(mppi.q_cur - q_f))                                 # noqa: F405
    print(f"RESULT iterations={n_iter} start_dist={d0:.4f} final_dist={d1:.4f} kernels={mppi.Policy.n_kernels} "
          f"hz={n_iter / td:.1f} min_clearance={float(closest_dist_all.min()):.4f}")


if __name__ == '__main__':
    main()
