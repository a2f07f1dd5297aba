"""GPU tests of the prefilter's tile schedule (run with -m gpu on a B200).

The row warps release the output layer's accumulator before they consume the next tile's table loads.  Batches
whose tile count is odd, smaller than two tiles per CTA pair, or a single tile run the schedule's first and last
iterations with an empty second slot; with fp32 accumulators the other kernel instantiation runs.  The rollout must
stay bit for bit the all-pairs fp32 rollout."""
import pytest
import torch

import bench
from tests.golden_util import load_npz

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def factory():
    from tests import mppi_factory
    return mppi_factory


def _rollout(factory, c, N, H, mode, obs):
    torch.manual_seed(5)
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    m = factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1=mode, copy_policy=False)
    m.Policy.alpha_s = 3.0
    m.update_obstacles(obs.cuda())
    torch.manual_seed(11)
    m.Policy.sample_policy()
    out = m.propagate()
    return m, [x.clone() for x in (*out, m.get_cost())]


# 2064 spheres: N = 1 -> 9 tiles on 5 CTA pairs, N = 7 -> 57 tiles on 29 pairs, N = 75 -> 605 tiles (odd, several
# iterations per pair and a ragged last one), N = 256 -> 2064 tiles
@pytest.mark.parametrize("N", [1, 7, 75, 256])
@pytest.mark.parametrize("acc", ["f16", "f32"])
def test_prefilter_schedule_is_exact_at_any_tile_count(factory, monkeypatch, N, acc):
    monkeypatch.setenv("DSMPPI_PASS1_ACC", acc)           # read when the context is created
    c = load_npz("case_franka_shelf")
    obs = bench.problem("franka_shelf_2064")["obs"]
    _, ref = _rollout(factory, c, N, 3, "exact", obs)
    m, got = _rollout(factory, c, N, 3, "tc_f16", obs)
    assert m.pass1_stats()["mode"] == 1
    assert m.exactness_stats()["exact_fallbacks"] == 0
    for x, y in zip(ref, got):
        assert torch.equal(x, y)
