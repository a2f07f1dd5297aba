"""GPU tests of distance networks other than the shipped 256 x 4 (run with -m gpu on a B200): seeded random-init
networks of 1..4 hidden layers of width 64..256, through the drop-in MPPI object and the C ABI.

- the strict FFMA mode runs the network's own width and depth, and must give the same bits as the same network
  embedded by hand in 256 x 4 (zero padding, identity layers);
- both scoring modes agree with the CPU oracle (which runs any depth and width) to the tolerances of
  test_gpu_parity.py, and stay as close to an fp64 evaluation as the oracle's own fp32 numbers are;
- the tensor-core prefilter still only prunes, and the whole-horizon kernels and the graphed control tick still equal
  the per-step launch path bit for bit."""
import pytest
import torch

from oracle import mppi_oracle as orc
from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
from tests.golden_util import frac_within, load_npz

pytestmark = pytest.mark.gpu

SHAPES = {"128x2": [128] * 2, "128x3": [128] * 3, "64x4": [64] * 4, "200x3": [200] * 3, "256x1": [256] * 1}
# (d, P, O) of the shipped nets the random ones stand in for, and the golden case that provides the scene
ROBOTS = {"planar7": (7, 3, 7, "case_planar7"), "planar2": (2, 3, 2, "case_planar2"),
          "franka": (7, 3, 9, "case_franka_shelf"), "toy": (2, 2, 1, "toycase_toy2")}
DIST_ATOL = 2e-6
DOT_ATOL = 1e-5


def check(a, b, rtol, atol, name, min_frac=0.99, loose=20, kink_samples=0):
    """>= min_frac of the elements within rtol/atol and none beyond `loose` x that.  Quantities that follow the
    DIRECTION of the distance gradient (dot product, basis, modulated velocity) may name `kink_samples`: that many
    samples (leading index) may be off altogether -- a hidden unit whose pre-activation is within rounding distance
    of zero flips its ReLU under ANY change of summation order, which moves the gradient by a finite amount while the
    distance stays within 1e-6.  (The same semantics as test_gpu_parity.py.)"""
    a, b = a.detach().cpu(), b.detach().cpu()
    assert a.shape == b.shape, f"{name}: shape {tuple(a.shape)} vs {tuple(b.shape)}"
    if kink_samples and a.shape[0] > 1:
        viol = ((a.double() - b.double()).abs() / (atol + rtol * b.double().abs())).reshape(a.shape[0], -1)
        worst = viol.max(dim=1)[0]
        drop = torch.argsort(worst, descending=True)[:kink_samples]
        keep = torch.ones(a.shape[0], dtype=torch.bool)
        keep[drop[worst[drop] > 1.0]] = False
        a, b = a[keep], b[keep]
    f = frac_within(a, b, rtol, atol)
    min_frac = min(min_frac, 1.0 - 1.0 / max(a.numel(), 1)) if min_frac < 1.0 else 1.0   # always allow one outlier
    assert f >= min_frac, f"{name}: only {f:.4f} within rtol={rtol} (max abs diff {(a - b).abs().max():.3e})"
    assert frac_within(a, b, loose * rtol, loose * atol) == 1.0, \
        f"{name}: outliers beyond {loose}x tolerance (max abs diff {(a - b).abs().max():.3e})"


def random_net(robot, layers, seed=0):
    d, P, O, _ = ROBOTS[robot]
    torch.manual_seed(seed)
    return RobotSdfCollisionNet(in_channels=d + P, out_channels=O, skips=[], layers=layers)


def arrays(net):
    lin = [m for m in net.model.modules() if isinstance(m, torch.nn.Linear)]
    return [m.weight.detach().clone() for m in lin], [m.bias.detach().clone() for m in lin]


def embed_256x4(net):
    """The same network as a 256 x 4 one: zero rows / columns for the missing features, identity layers appended."""
    W, b = arrays(net)
    L, width, O, nenc = len(W) - 1, W[0].shape[0], W[-1].shape[0], W[0].shape[1]
    W4 = [torch.zeros(256, nenc)] + [torch.zeros(256, 256) for _ in range(3)] + [torch.zeros(O, 256)]
    b4 = [torch.zeros(256) for _ in range(4)] + [b[L].clone()]
    for l in range(4):
        if l < L:
            W4[l][:width, :W[l].shape[1]] = W[l]
            b4[l][:width] = b[l]
        else:
            W4[l][:width, :width] = torch.eye(width)
    W4[4][:, :width] = W[L]
    big = RobotSdfCollisionNet(in_channels=net.in_channels, out_channels=O, skips=[], layers=[256] * 4)
    big.load_arrays(W4, b4)
    return big


@pytest.fixture(scope="module")
def factory():
    from tests import mppi_factory
    return mppi_factory


def make(factory, monkeypatch, robot, net, score, **kw):
    """factory.make_mppi / make_toy_mppi with `net` in place of the shipped weights."""
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    monkeypatch.setattr(factory, "make_toy_net", lambda: net)
    monkeypatch.setattr(factory, "DEFAULT_SCORE", score)
    c = load_npz(ROBOTS[robot][3])
    if robot == "toy":
        kw.pop("copy_policy", None)
        kw.pop("q_cur", None)
        return factory.make_toy_mppi(c, **kw), c
    return factory.make_mppi(c, **kw), c


def _iteration(m, seed):
    torch.manual_seed(seed)
    m.Policy.sample_policy()
    out = [x.clone() for x in m.propagate()] + [m.qdot.clone()]
    out.append(m.get_cost().clone())
    res = m.shift_policy_means()             # the toy variant returns 0, like the reference's MPPI_toy.py
    P = m.Policy
    out += [P.mu_c.clone(), P.sigma_c.clone(), P.alpha_c.clone()]
    return out + ([torch.as_tensor(int(res[1]))] if isinstance(res, tuple) else [])


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("robot", list(ROBOTS))
def test_ffma_native_width_and_depth_equal_the_256x4_embedding_bitwise(shape, robot, factory, monkeypatch):
    """The FFMA kernels run W features (rounded up to 64 / 128 / 256) and L layers; zero features and identity layers
    change no bit, so the narrow network must reproduce the hand-embedded 256 x 4 one exactly: propagate, get_cost,
    shift_policy_means."""
    net = random_net(robot, SHAPES[shape], seed=3)
    outs = []
    for n in (net, embed_256x4(net)):
        m, _ = make(factory, monkeypatch, robot, n, "ffma", device="cuda", N=333, H=4)
        m.Policy.alpha_s = 1.5
        outs.append(_iteration(m, 17))
    bits = lambda x: x.detach().cpu().contiguous().view(torch.int32) if x.is_floating_point() else x.cpu()  # noqa: E731
    for i, (a, b) in enumerate(zip(*outs)):
        assert torch.equal(bits(a), bits(b)), f"output {i} differs"


@pytest.mark.parametrize("score", ["tc_split", "ffma"])
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("robot,N,H,M,K", [("franka", 300, 3, 37, 5), ("planar7", 257, 4, 5, 2),
                                           ("planar2", 129, 5, 3, 3), ("toy", 77, 4, 5, 3)])
def test_rollout_vs_oracle_random_inputs(robot, N, H, M, K, shape, score, factory, monkeypatch):
    """Fresh seeded inputs (ragged N) against the CPU oracle running the same network, step by step on the GPU's own
    states (the pattern of test_gpu_parity.test_rollout_vs_oracle_random_inputs)."""
    dist_atol = DIST_ATOL if score == "ffma" else 5e-6
    dot_atol = DOT_ATOL if score == "ffma" else 3e-5
    torch.manual_seed(1234)
    d, P_dim, _, _ = ROBOTS[robot]
    net = random_net(robot, SHAPES[shape], seed=7)
    W, b = arrays(net)
    onet = orc.Net(W, b)
    base = load_npz(ROBOTS[robot][3])
    scale = 0.6 if robot == "franka" else 4.0
    obs = torch.cat(((torch.rand(M, P_dim) - 0.5) * 2 * scale, 0.03 + 0.2 * torch.rand(M, 1)), 1)
    q_cur = base["q0"] + 0.3 * torch.randn(N, d)
    nk = 6
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    monkeypatch.setattr(factory, "make_toy_net", lambda: net)
    monkeypatch.setattr(factory, "DEFAULT_SCORE", score)
    c = dict(base, obs=obs, K=K, N=N, H=H, nk=nk)
    if robot == "toy":
        m = factory.make_toy_mppi(dict(base, obs=obs, K=K), device="cpu", N=N, H=H)   # fresh policy samples below
        m.q_cur = q_cur
        ign = []
        prm = orc.toy_params(float(base["dt"]), 1, K, base["A"], dst_thr=float(base["dst_thr"]), p=2.0,
                             with_basis=False)
    else:
        m = factory.make_mppi(c, device="cpu", N=N, H=H, q_cur=q_cur, copy_policy=False)
        ign = base["ignored_links"].tolist()
        prm = orc.RolloutParams(dt=float(base["dt"]), dt_H=1, n_closest_obs=K, dst_thr=float(base["dst_thr"]),
                                ignored_links=ign, p=2.0, with_basis=False)
    P = m.Policy
    P.n_kernels = nk
    P.mu_c[:nk] = base["q0"] + 0.3 * torch.randn(nk, d)
    P.sigma_c[:nk] = 0.7
    P.alpha_c[:nk] = torch.randn(nk, d)
    P.alpha_s = 1.5
    P.p = 2.0
    P.sample_policy()
    traj, dist, kv, dots = m.propagate()[:4]            # (the toy variant returns no activations)
    acts = m.kernel_activations
    kink = max(1, N // 200)
    for t in range(H):
        o = orc.rollout(onet, traj[:, t, :], base["qf"], obs, P.mu_tmp, P.sigma_tmp, P.alpha_tmp, nk, prm, N)
        check(dist[:, t], o.closest_dist_all[:, 0], 1e-5, dist_atol, f"dist[{t}]")
        check(dots[:, t], o.dot_products[:, 0], 1e-5, dot_atol, f"dot[{t}]", min_frac=0.9, kink_samples=kink)
        check(acts[:, t], o.kernel_activations[:, 0], 1e-4, 1e-5, f"act[{t}]", kink_samples=kink)
        # (the toy folds the activation, a function of the gradient's direction, into its kernel values)
        check(kv[:, t, :], o.kernel_val_all[:, 0, :nk], 1e-4, 1e-6, f"kval[{t}]", kink_samples=kink if robot == "toy" else 0)
        if t + 1 < H:
            check(traj[:, t + 1, :], traj[:, t, :] + float(base["dt"]) * o.qdot, 1e-5, 1e-5, f"traj[{t + 1}]",
                  kink_samples=kink)
    if robot == "toy":
        return            # the toy's cost and update are covered by the embedding test and tests/test_gpu_toy.py
    cost = m.get_cost()
    ocost = orc.evaluate_costs(traj, dist, base["qf"], base["dh_params"], base["q_min"], base["q_max"])
    check(cost, ocost, 1e-5, 1e-4, "cost")
    mu0, sg0, al0 = P.mu_c.clone(), P.sigma_c.clone(), P.alpha_c.clone()
    _, n_upd = m.shift_policy_means()
    mu1, sg1, al1, on, _ = orc.policy_update(cost, m.kernel_val_all, acts, P.mu_tmp, P.sigma_tmp, P.alpha_tmp, mu0,
                                             sg0, al0, nk, float(base["ker_thr"]))
    assert int(n_upd) == on
    check(P.mu_c, mu1, 1e-4, 1e-6, "mu_c")
    check(P.alpha_c, al1, 1e-4, 1e-6, "alpha_c")


@pytest.mark.parametrize("score", ["tc_split", "ffma"])
@pytest.mark.parametrize("shape", ["128x2", "128x3", "64x4", "200x3"])
@pytest.mark.parametrize("robot", ["planar7", "franka"])
def test_gradient_error_vs_fp64(robot, shape, score, factory, monkeypatch):
    """Distance and gradient are as close to an fp64 evaluation of the same network as the oracle's fp32 CPU numbers
    are.  In tc_split mode this holds only with the truncation compensation computed from the network's real width
    (a narrow network's hidden GEMMs have fewer non-zero MMA steps than 256 x 4's)."""
    net = random_net(robot, SHAPES[shape], seed=11)
    d, P_dim, _, _ = ROBOTS[robot]
    g = torch.Generator().manual_seed(21)
    base = load_npz(ROBOTS[robot][3])
    M, K = 24, 3
    scale = 0.6 if robot == "franka" else 4.0
    obs = torch.cat(((torch.rand(M, P_dim, generator=g) - 0.5) * 2 * scale, 0.03 + 0.2 * torch.rand(M, 1, generator=g)), 1)
    q = base["q0"] + 0.5 * torch.randn(1000, d, generator=g)
    ign = base["ignored_links"].tolist()
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    monkeypatch.setattr(factory, "DEFAULT_SCORE", score)
    m = factory.make_mppi(dict(base, obs=obs, K=K, ignored_links=base["ignored_links"]), device="cpu", H=1)
    dist, grad = m.distance_repulsion_nn(q)
    W, b = arrays(net)
    d32, g32 = orc.distance_repulsion(orc.Net(W, b), q, obs, K, ign)
    d64, g64 = orc.distance_repulsion(orc.Net([w.double() for w in W], [x.double() for x in b]), q.double(),
                                      obs.double(), K, ign)
    ref_err_d = (d32.double() - d64).abs().max().item()
    gpu_err_d = (dist.double() - d64).abs().max().item()
    ref_err_g = (g32.double() - g64).abs().max().item()
    gpu_err_g = (grad.double() - g64).abs().max().item()
    print(f"{robot} {shape} {score}: distance err vs fp64  oracle fp32 {ref_err_d:.2e} gpu {gpu_err_d:.2e};  "
          f"grad err oracle fp32 {ref_err_g:.2e} gpu {gpu_err_g:.2e}")
    assert gpu_err_d <= 4 * ref_err_d + 1e-6
    assert gpu_err_g <= 4 * ref_err_g + 1e-6 * g64.abs().max().item()


@pytest.mark.parametrize("score", ["tc_split", "ffma"])
@pytest.mark.parametrize("shape", ["128x3", "64x4"])
def test_prefilter_only_prunes_for_a_narrow_network(shape, score, factory, monkeypatch):
    """294 spheres: the fp16 tensor-core prefilter (run on the 256 x 4 embedding, guard band calibrated for this
    network) must leave the rollout bit for bit equal to scoring every pair in fp32, with no fall-back."""
    net = random_net("franka", SHAPES[shape], seed=5)
    N, H = 777, 4
    torch.manual_seed(5)
    c = load_npz("case_franka_shelf")
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    monkeypatch.setattr(factory, "DEFAULT_SCORE", score)
    outs = {}
    for mode in ("exact", "tc_f16"):
        m = factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1=mode, copy_policy=False)
        m.Policy.alpha_s = 3.0
        torch.manual_seed(11)
        m.Policy.sample_policy()
        traj, dist, kv, dots, acts = m.propagate()
        outs[mode] = (traj.clone(), dist.clone(), dots.clone(), acts.clone(), m.get_cost().clone())
        if mode == "tc_f16":
            st, xs = m.pass1_stats(), m.exactness_stats()
            assert st["mode"] == 1 and xs["exact_fallbacks"] == 0, (st, xs)
    for a, b in zip(outs["exact"], outs["tc_f16"]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("score", ["tc_split", "ffma"])
@pytest.mark.parametrize("shape", ["128x2", "64x4"])
@pytest.mark.parametrize("robot", ["planar7", "planar2"])
def test_whole_horizon_kernel_equals_per_step_launches(robot, shape, score, factory, monkeypatch):
    net = random_net(robot, SHAPES[shape], seed=9)
    outs = []
    for whole in (True, False):
        m, c = make(factory, monkeypatch, robot, net, score, device="cuda")
        m.set_whole_horizon(whole)
        n0 = m.launch_count()
        res = [x.clone() for x in m.propagate()]
        outs.append((res + [m.qdot.clone(), m.norm_basis.clone()], m.launch_count() - n0))
    (a, la), (b, lb) = outs
    assert la <= 4 and lb >= 3 * int(c["H"]), (la, lb)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("score", ["tc_split", "ffma"])
def test_graphed_control_tick_equals_the_plain_path(score, factory, monkeypatch):
    """N = 1, H = 2 with CPU tensors (the integrator's tick) runs as one replayed CUDA graph; a narrow network must give
    the plain path's bits."""
    net = random_net("franka", [128] * 3, seed=13)
    c = load_npz("case_franka_shelf")
    obs = c["obs"][:28].clone()
    monkeypatch.setattr(factory, "make_net", lambda name: net)
    monkeypatch.setattr(factory, "DEFAULT_SCORE", score)
    torch.manual_seed(5)
    q_start = c["q0"] + 0.05 * torch.randn(7)
    outs = {}
    for mode in ("graph", "plain"):
        monkeypatch.setenv("DSMPPI_GRAPH_TICK", "1" if mode == "graph" else "0")
        m = factory.make_mppi(dict(c, obs=obs.clone()), device="cpu", N=1, H=2, pass1="auto", copy_policy=False)
        m.Policy.alpha_s = 1.0
        outs[mode] = []
        for tick in range(3):
            torch.manual_seed(100 + tick)
            m.Policy.sample_policy()
            m.q_cur = q_start + 0.01 * tick
            traj, dist, kv, dots, acts = m.propagate()
            outs[mode].append([t.clone() for t in (traj, dist, kv, dots, acts, m.qdot, m.nn_grad)])
        if mode == "graph":
            assert "_tick" in m.__dict__, "the tick did not take the graphed path"
    for a, b in zip(outs["graph"], outs["plain"]):
        for x, y in zip(a, b):
            assert torch.equal(x, y)
