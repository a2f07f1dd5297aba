"""GPU tests of the prefilter's dead-feature skip (run with -m gpu on a B200).

The guard-band calibration takes a census of the hidden features of layers 2..4 that never fire, moves them last and
leaves whole K-steps of them out of the tensor-core GEMMs; every prefiltered row proves its skip, and a call in which
a skipped feature fired is repeated without it.  Whatever the skip does, the rollout must stay bit for bit the
all-pairs fp32 rollout."""
import pytest
import torch

import bench
from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
from tests.golden_util import load_npz

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def factory():
    from tests import mppi_factory
    return mppi_factory


def _rollout(factory, c, N, H, mode, obs=None, m=None):
    if m is None:
        torch.manual_seed(5)
        q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
        m = factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1=mode, copy_policy=False)
        m.Policy.alpha_s = 3.0
    if obs is not None:
        m.update_obstacles(obs.cuda())
    torch.manual_seed(11)
    m.Policy.sample_policy()
    traj, dist, kv, dots, acts = m.propagate()
    return m, [x.clone() for x in (traj, dist, kv, dots, acts, m.get_cost())]


def _equal(a, b):
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_shipped_franka_on_the_bench_shelf_skips_the_census_k_steps(factory):
    """tools/dead_feature_study.py finds 41, 90 and 118 never-active features in hidden layers 2..4 of the shipped
    net on this shelf: 2, 5 and 7 whole K-steps of the layer 3, layer 4 and output GEMMs."""
    c = load_npz("case_franka_shelf")
    obs = bench.problem("franka_shelf_2064")["obs"]
    outs = {}
    for mode in ("exact", "tc_f16"):
        m, outs[mode] = _rollout(factory, c, 1024, 6, mode, obs)
        if mode == "tc_f16":
            assert m.pass1_stats()["mode"] == 1
            assert m.prefilter_skip_stats() == dict(skipped_ksteps=(2, 5, 7), repeated_calls=0)
            assert m.exactness_stats()["exact_fallbacks"] == 0
    _equal(outs["exact"], outs["tc_f16"])


def _sleeping_net():
    """Franka-shaped random net whose layer-4 feature 255 only fires for obstacles at x > 0.05: layer-1 feature 0 is
    relu(10 x), carried unchanged through features 0 of layers 2 and 3; layer-4 feature 255 = relu(h3_0 - 0.5).
    Layer-4 features 128..254 never fire (zero weights, bias -1); every other feature gets a bias of +1, so that no
    other whole K-step is dead (a rarely firing random feature would make the first call repeat as well)."""
    torch.manual_seed(7)
    net = RobotSdfCollisionNet(in_channels=10, out_channels=9, skips=[], layers=[256] * 4)
    lin = [m for m in net.model.modules() if isinstance(m, torch.nn.Linear)]
    W, b = [m.weight.detach().clone() for m in lin], [m.bias.detach().clone() for m in lin]
    for l in range(4):
        b[l] += 1.0
    W[0][0].zero_(); W[0][0, 7] = 10.0; b[0][0] = 0.0          # input column 7: the obstacle's x
    for l in (1, 2):
        W[l][0].zero_(); W[l][0, 0] = 1.0; b[l][0] = 0.0
    W[3][128:].zero_(); b[3][128:] = -1.0
    W[3][255, 0] = 1.0; b[3][255] = -0.5
    W[4][:, 255] = 0.5
    net.load_arrays(W, b)
    return net


def test_a_feature_that_wakes_up_is_caught_and_the_call_repeated(factory, monkeypatch):
    net = _sleeping_net()
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    c = load_npz("case_franka_shelf")
    obs = c["obs"].clone().float()
    left = obs.clone()
    left[:, 0] = -obs[:, 0].abs() - 0.3
    right = left.clone()
    right[:, 0] = -left[:, 0]
    # (the constructor's first rollout takes the census: the scene must start on the dead side)
    c_left = dict(c, obs=left)
    N, H = 777, 4
    m, _ = _rollout(factory, c_left, N, H, "tc_f16")
    s = m.prefilter_skip_stats()
    assert s == dict(skipped_ksteps=(0, 0, 8), repeated_calls=0), s
    # the same obstacle count, moved across the plane: no new census, the skipped feature fires
    _, got = _rollout(factory, c_left, N, H, "tc_f16", right, m=m)
    assert m.prefilter_skip_stats()["repeated_calls"] == 1
    _, ref = _rollout(factory, c_left, N, H, "exact", right)
    _equal(ref, got)
    assert m.exactness_stats()["exact_fallbacks"] == 0
    # the next call takes the census again on the current scene (the feature now counts as active: the skip stays
    # on, one fewer dead feature) and needs no repeat
    _, again = _rollout(factory, c_left, N, H, "tc_f16", m=m)
    s = m.prefilter_skip_stats()
    assert s["repeated_calls"] == 1 and s["skipped_ksteps"][2] >= 7, s
    _equal(ref, again)


def test_a_random_init_network_drops_nothing(factory, monkeypatch):
    torch.manual_seed(1)
    net = RobotSdfCollisionNet(in_channels=10, out_channels=9, skips=[], layers=[256] * 4)
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    c = load_npz("case_franka_shelf")
    outs, launches = {}, []
    for mode in ("exact", "tc_f16"):
        m, outs[mode] = _rollout(factory, c, 512, 4, mode)
        if mode == "tc_f16":
            assert m.prefilter_skip_stats() == dict(skipped_ksteps=(0, 0, 0), repeated_calls=0)
            for _ in range(2):
                n0 = m.launch_count()
                _, again = _rollout(factory, c, 512, 4, mode, m=m)
                launches.append(m.launch_count() - n0)
                _equal(outs[mode], again)
    _equal(outs["exact"], outs["tc_f16"])
    # after the calibration's one-off census, the rollout launches the same kernels every call
    assert launches[0] == launches[1]
