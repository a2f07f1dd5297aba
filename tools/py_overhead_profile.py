import cProfile, os, pstats, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.golden_util import load_npz
from tests.mppi_factory import make_mppi
for dev in ("cuda", "cpu"):
    m = make_mppi(load_npz("case_planar2"), device=dev, pass1="auto")
    def it():
        m.propagate(); m.get_cost(); m.shift_policy_means()
    for _ in range(20): it()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(300): it()
    torch.cuda.synchronize()
    print(dev, "ms per iteration", (time.perf_counter() - t0) / 300 * 1e3)
    pr = cProfile.Profile(); pr.enable()
    for _ in range(300): it()
    torch.cuda.synchronize(); pr.disable()
    pstats.Stats(pr).sort_stats("cumulative").print_stats(22)
