import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.golden_util import load_npz
from tests import mppi_factory as F
for tag in ("planar7", "planar7_near", "planar2_near", "franka_shelf"):
    c = load_npz(f"case_{tag}")
    H = int(c["H"])
    for mode, dbg in (("ffma", "0"), ("tc_split", "0"), ("tc_split", "4")):
        os.environ["DSMPPI_TCX_DEBUG"] = dbg
        F.DEFAULT_SCORE = mode
        m = F.make_mppi(c, device="cpu", H=1)
        errs = []
        for t in range(H):
            m.q_cur = c["all_traj"][:, t, :]
            traj, dist, kv, dots, acts = m.propagate()
            errs.append((dist[:, 0] - c["closest_dist_all"][:, t]).double())
        e = torch.stack(errs)
        print(f"{tag:14s} {mode:8s} dbg={dbg}: dist err vs reference: rms {e.pow(2).mean().sqrt():.2e} max {e.abs().max():.2e} mean {e.mean():+.2e}   |dist| rms {c['closest_dist_all'].pow(2).mean().sqrt():.3f}", m.score_stats())
