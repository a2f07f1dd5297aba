"""GPU tests of the API edges the first round left uncovered (run with -m gpu):
  * MPPI.get_qdot, both modes (MPPI.py:319-329), against the reference's own values;
  * MPPI.update_kernel_normal_bases (MPPI.py:284-304) against the reference's kernel_obstacle_bases;
  * the constructor leaves torch's generator where the reference's constructor leaves it (untouched: its five
    warm-up draws act on empty views), so a seeded script sees the same noise afterwards;
  * the obstacle count may change on a live object across the prefilter threshold (dynamic obstacles through
    update_obstacles): the workspace follows the resolved pass-1 mode;
  * the prefilter is exact by construction: adversarial obstacle sets (many spheres at the same distance, a crowded
    band for every sample) and a random-init network give bit-for-bit the all-pairs-fp32 rollout;
  * torch.profiler sees the reference's stage tags around the fused call."""
import pytest
import torch

from oracle import mppi_oracle as orc
from tests.golden_util import frac_within, load_npz, load_weights

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def factory():
    from tests import mppi_factory
    return mppi_factory


@pytest.fixture(autouse=True, params=["tc_split", "ffma"])
def score_mode(request, factory):
    factory.DEFAULT_SCORE = request.param
    yield request.param
    factory.DEFAULT_SCORE = None


def _close(a, b, rtol, atol, name):
    a, b = a.detach().cpu(), b.detach().cpu()
    assert a.shape == b.shape, f"{name}: {tuple(a.shape)} vs {tuple(b.shape)}"
    assert frac_within(a, b, rtol, atol) == 1.0, f"{name}: max abs diff {(a - b).abs().max():.3e}"


@pytest.mark.parametrize("device", ["cpu", "cuda"])
def test_get_qdot_both_modes_vs_reference(device, factory):
    """bench_c3_franka2064 holds the reference's qdot of all 64 samples, its cost and both get_qdot results."""
    g = load_npz("bench_c3_franka2064")
    c = dict(g, N=64, H=50)
    m = factory.make_mppi(c, device=device, pass1="auto")
    # (a) on the reference's own velocities and costs: the method's arithmetic alone
    m.qdot, m.cur_cost = g["qdot"].to(device), g["cost"].to(device)
    _close(m.get_qdot('best'), g["qdot_best"], 0, 0, "get_qdot('best') on reference inputs")
    _close(m.get_qdot('weighted'), g["qdot_weighted"], 1e-5, 1e-6, "get_qdot('weighted') on reference inputs")
    assert m.get_qdot('best').device.type == device
    # (b) end to end: our rollout + cost, then get_qdot; step-1 velocities are not chaotic yet
    m.propagate()
    cost = m.get_cost()
    qd_b, qd_w = m.get_qdot('best'), m.get_qdot('weighted')
    assert qd_b.shape == (7,) and qd_w.shape == (7,)
    _close(qd_b, m.qdot[torch.argmin(cost)], 0, 0, "best == qdot[argmin cost]")
    beta = cost.mean() / 50
    w = torch.exp(-cost / beta)
    _close(qd_w, ((w / w.sum()).unsqueeze(1) * m.qdot).sum(0), 1e-5, 1e-6, "weighted")
    assert m.get_qdot('other') == 0                                      # MPPI.py:320: unknown mode returns 0


@pytest.mark.parametrize("tag,case", [("planar2", "case_c1_planar2"), ("planar7", "bench_c2_planar7"),
                                      ("franka2064", "bench_c3_franka2064")])
def test_update_kernel_normal_bases_vs_reference(tag, case, factory, score_mode):
    e = load_npz(f"edges_{tag}_bases")
    g = load_npz(case)
    nk = e["mu_c"].shape[0]
    c = dict(g, N=8, H=2)
    m = factory.make_mppi(c, device="cpu", N=8, H=2, pass1="auto", copy_policy=False)
    m.Policy.n_kernels = nk
    m.Policy.mu_c[:nk] = e["mu_c"]
    before = m.Policy.kernel_obstacle_bases.clone()
    assert m.update_kernel_normal_bases() == 0
    E = m.Policy.kernel_obstacle_bases[:nk]
    atol = 1e-5 if score_mode == "ffma" else 5e-5
    # the Householder basis follows the gradient direction: allow one ReLU-kink centre (SURVEY 8(c))
    err = (E - e["bases"]).abs().reshape(nk, -1).max(1)[0]
    assert int((err > atol + 1e-4).sum()) <= 1, f"bases differ: {err}"
    d = E.shape[-1]
    eye = torch.eye(d).expand(nk, d, d)
    assert (E.transpose(1, 2) @ E - eye).abs().max() < 1e-5              # orthonormal
    assert torch.equal(m.Policy.kernel_obstacle_bases[nk:], before[nk:])  # untouched beyond n_kernels
    m.Policy.n_kernels = 0
    assert m.update_kernel_normal_bases() == 0                            # MPPI.py:301-302: no kernels, no-op


def test_constructor_leaves_the_torch_generator_untouched(factory):
    """Reference: MPPI.__init__ runs five sample_policy + propagate warm-ups (MPPI.py:69-73); with n_kernels = 0
    their normal_() calls draw nothing (checked on the reference itself in the build container: the generator state
    is identical before and after), so RNG lock-step == the constructor consumes no random numbers."""
    import optimalmodulationds_b200 as pkg
    c = load_npz("case_planar7")
    net = factory.make_net("planar7")               # nn.Linear initialisation draws from the generator: before seeding,
    DS = [pkg.LinDS(c["qf"]), pkg.LinDS(c["q0"])]   # as in the scripts (the network is built before the MPPI object)
    torch.manual_seed(2024)
    s0 = torch.get_rng_state().clone()
    m = pkg.MPPI(c["q0"], c["qf"], c["dh_params"], c["obs"], float(c["dt"]), int(c["H"]), int(c["N"]), DS, c["dh_a"],
                 net, int(c["K"]))
    assert torch.equal(torch.get_rng_state(), s0)
    # and from there a seeded script draws exactly the reference's noise: mu, sigma, alpha in this order
    m.Policy.n_kernels = 3
    m.Policy.alpha_s = 0.75
    m.Policy.sample_policy()
    torch.manual_seed(2024)
    # the reference's statements (policy.py:65-74), on views of (N, 50, ..) buffers like its own (a strided view
    # takes torch's serial normal_ path, a contiguous tensor would take the vectorised one: different streams)
    N = int(c["N"])
    mu_b, sg_b, al_b = torch.zeros(N, 50, 7), torch.zeros(N, 50), torch.zeros(N, 50, 7)
    ref_mu = mu_b[:, :3].normal_(mean=0, std=0.0) + m.Policy.mu_c[:3]
    ref_sg = sg_b[:, :3].normal_(mean=0, std=0.0) + m.Policy.sigma_c[:3]
    ref_al = al_b[:, :3].normal_(mean=0, std=0.75) + m.Policy.alpha_c[:3]
    ref_al[0] = m.Policy.alpha_c[:3]
    assert torch.equal(m.Policy.alpha_tmp[:, :3], ref_al)
    assert torch.equal(m.Policy.mu_tmp[:, :3], ref_mu)
    assert torch.equal(m.Policy.sigma_tmp[:, :3], ref_sg)


def _rollout_outputs(m):
    traj, dist, kv, dots, acts = m.propagate()
    return [t.clone() for t in (traj, dist, kv, dots, acts, m.qdot)]


def test_obstacle_count_may_cross_the_prefilter_threshold_on_a_live_object(factory):
    """ADVICE r1 (high): AUTO resolves to the tensor-core prefilter from 64 obstacles on and to dense fp32 scoring
    below; a workspace sized for one mode was reused for the other.  M = 100 -> 40 -> 20 -> 300 on ONE object, each
    compared with a fresh object at that obstacle count."""
    c = load_npz("case_franka_shelf")
    torch.manual_seed(3)
    N, H = 192, 3
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    live = factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1="auto", copy_policy=False)
    torch.manual_seed(4)
    live.Policy.alpha_s = 2.0
    live.Policy.sample_policy()
    pol = [t.clone() for t in (live.Policy.mu_tmp, live.Policy.sigma_tmp, live.Policy.alpha_tmp)]
    for M in (100, 40, 20, 300, 17):
        g = torch.Generator().manual_seed(M)
        obs = torch.cat(((torch.rand(M, 3, generator=g) - 0.5) * 1.2 + torch.tensor([0.4, 0.0, 0.5]),
                         0.03 + 0.05 * torch.rand(M, 1, generator=g)), 1).cuda()
        live.update_obstacles(obs)
        got = _rollout_outputs(live)
        assert live.pass1_stats()["mode"] == (1 if M >= 64 else 0)
        fresh = factory.make_mppi(dict(c, obs=obs.cpu()), device="cuda", N=N, H=H, q_cur=q_cur, pass1="auto",
                                  copy_policy=False)
        for dst, src in zip((fresh.Policy.mu_tmp, fresh.Policy.sigma_tmp, fresh.Policy.alpha_tmp), pol):
            dst.copy_(src)
        want = _rollout_outputs(fresh)
        for a, b, name in zip(got, want, ("traj", "dist", "kval", "dots", "acts", "qdot")):
            assert torch.equal(a, b), f"M={M}: {name} differs between the live and a fresh object"
    torch.cuda.synchronize()


def _adversarial_obstacles(kind, M):
    g = torch.Generator().manual_seed(7)
    if kind == "ring":        # M spheres on a circle around the arm's base axis: near-equal distances to a link
        ang = torch.linspace(0, 2 * torch.pi, M + 1)[:-1]
        return torch.stack((0.45 * torch.cos(ang), 0.45 * torch.sin(ang), torch.full((M,), 0.5),
                            torch.full((M,), 0.03)), 1)
    if kind == "stack":       # M copies of ONE sphere: exactly equal distances, ties broken by index
        return torch.tensor([[0.45, 0.05, 0.6, 0.03]]).repeat(M, 1)
    if kind == "cluster":     # M spheres within a few millimetres of each other
        return torch.cat((torch.tensor([0.45, 0.0, 0.55]) + 2e-3 * torch.randn(M, 3, generator=g),
                          torch.full((M, 1), 0.03)), 1)
    raise ValueError(kind)


@pytest.mark.parametrize("kind,M", [("ring", 96), ("stack", 128), ("cluster", 200)])
def test_crowded_guard_band_is_rescored_not_truncated(kind, M, factory):
    """More than 16 obstacles inside the guard band of every sample (what round 1 truncated to the 16 smallest
    approximate values): the prefiltered rollout must still equal the all-pairs fp32 rollout BIT FOR BIT, with the
    candidate list grown by a counted retry."""
    c = load_npz("case_franka_shelf")
    obs = _adversarial_obstacles(kind, M)
    torch.manual_seed(9)
    N, H = 300, 4
    q_cur = c["q0"] + 0.1 * torch.randn(N, 7)
    outs, stats = {}, {}
    for mode in ("exact", "tc_f16"):
        m = factory.make_mppi(dict(c, obs=obs), device="cuda", N=N, H=H, q_cur=q_cur, pass1=mode, copy_policy=False)
        m.Policy.alpha_s = 3.0
        torch.manual_seed(11)
        m.Policy.sample_policy()
        outs[mode] = _rollout_outputs(m) + [m.get_cost().clone()]
        stats[mode] = (m.pass1_stats(), m.exactness_stats())
    p1, xs = stats["tc_f16"]
    print(f"{kind} M={M}: {p1}, {xs}")
    assert p1["mode"] == 1
    if kind != "ring":        # (the ring only produces near-ties; the other two put every sphere inside the band)
        assert p1["band_overflows"] > 0, "the adversarial set was meant to crowd the band"
        assert p1["rescored_pairs"] / (N * H) > 16
        assert xs["capacity_retries"] >= 1, "a list budgeted at 16 rows per sample cannot have held them"
    for a, b, name in zip(outs["exact"], outs["tc_f16"], ("traj", "dist", "kval", "dots", "acts", "qdot", "cost")):
        assert torch.equal(a, b), f"{kind}: {name} differs from the all-pairs fp32 rollout"
    # distance_repulsion_nn goes through the same protocol
    m = factory.make_mppi(dict(c, obs=obs), device="cuda", N=N, H=1, pass1="tc_f16", copy_policy=False)
    m2 = factory.make_mppi(dict(c, obs=obs), device="cuda", N=N, H=1, pass1="exact", copy_policy=False)
    d1, g1 = m.distance_repulsion_nn(q_cur.cuda())
    d2, g2 = m2.distance_repulsion_nn(q_cur.cuda())
    assert torch.equal(d1, d2) and torch.equal(g1, g2)


def test_guard_band_is_calibrated_per_network(factory):
    """A random-init network (much larger prefilter error than the shipped checkpoints) gets its own measured guard
    band, and with it the prefiltered rollout is still bitwise the all-pairs fp32 one."""
    import optimalmodulationds_b200 as pkg
    from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
    c = load_npz("case_franka_shelf")
    torch.manual_seed(21)
    net = RobotSdfCollisionNet(in_channels=10, out_channels=9, layers=[256] * 4, skips=[])
    for mod in net.model.modules():
        if isinstance(mod, torch.nn.Linear):
            torch.nn.init.normal_(mod.weight, std=2.0 / mod.in_features ** 0.5)
            torch.nn.init.normal_(mod.bias, std=0.5)
    with torch.no_grad():      # centimetre-scale outputs like the shipped Franka net
        last = [mod for mod in net.model.modules() if isinstance(mod, torch.nn.Linear)][-1]
        last.weight.mul_(20.0)
        last.bias.add_(40.0)
    t = lambda x: x.cuda()  # noqa: E731
    N, H = 256, 3
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    res, bands = {}, {}
    for mode in ("exact", "tc_f16"):
        DS = [pkg.LinDS(t(c["qf"])), pkg.LinDS(t(c["q0"]))]
        m = pkg.MPPI(t(c["q0"]), t(c["qf"]), t(c["dh_params"]), t(c["obs"]), float(c["dt"]), H, N, DS, t(c["dh_a"]),
                     net, 5)
        m.set_pass1_mode(mode)
        m.dst_thr, m.ignored_links = 0.01, [0, 1, 2]
        m.q_cur = t(q_cur)
        res[mode] = _rollout_outputs(m)
        bands[mode] = m.exactness_stats()
    shipped = factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1="tc_f16", copy_policy=False)
    shipped.propagate()
    b_ship, b_rand = shipped.exactness_stats(), bands["tc_f16"]
    print(f"guard band: shipped net {b_ship}, random-init net {b_rand}")
    # (the shipped Franka net: ~2 mm with fp32 accumulators in the prefilter, ~4 mm with the default fp16 ones)
    assert 0 < b_ship["calibration_error"] < 1e-2 and b_ship["guard_band"] >= 3 * b_ship["calibration_error"] * 0.999
    assert b_rand["guard_band"] > 0 and b_rand["guard_band"] != b_ship["guard_band"]
    for a, b, name in zip(res["exact"], res["tc_f16"], ("traj", "dist", "kval", "dots", "acts", "qdot")):
        assert torch.equal(a, b), f"random-init net: {name} differs from the all-pairs fp32 rollout"


@pytest.mark.parametrize("variant", ["f16_fp32acc", "bf16", "f16_few_obstacles", "bf16_few_obstacles", "f16_40_obstacles",
                                     "f16_single_sample", "f16_three_samples"])
def test_prefilter_variants_are_bitwise_the_all_pairs_rollout(factory, variant, monkeypatch):
    """The prefilter kernel has six instantiations (fp16 operands with fp16 or fp32 accumulators, bf16 operands; the
    per-sample table staged through shared memory from 32 obstacles on, read per lane below).  The default one is
    covered by every tensor-core test; here the others: each gets its own calibrated band and must reproduce the
    all-pairs fp32 rollout bit for bit."""
    c = load_npz("case_franka_shelf")
    if variant == "f16_fp32acc":
        monkeypatch.setenv("DSMPPI_PASS1_ACC", "f32")           # read when the context is created
    mode = "tc_bf16" if variant.startswith("bf16") else "tc_f16"
    obs = c["obs"][:24] if variant.endswith("few_obstacles") else c["obs"][:40] if "40" in variant else c["obs"]
    torch.manual_seed(17)
    # (one / three samples: the last tile is mostly pair-rows past the end of the batch, and a warp's second table row
    # is the clamped one)
    N, H = (1, 4) if variant.endswith("single_sample") else (3, 4) if variant.endswith("three_samples") else (160, 4)
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    outs, bands = {}, {}
    for m_ in ("exact", mode):
        m = factory.make_mppi(dict(c, obs=obs), device="cuda", N=N, H=H, q_cur=q_cur, pass1=m_, copy_policy=False)
        torch.manual_seed(11)
        m.Policy.sample_policy()
        outs[m_] = _rollout_outputs(m) + [m.get_cost().clone()]
        bands[m_] = (m.pass1_stats(), m.exactness_stats())
    p1, xs = bands[mode]
    print(f"{variant}: {p1}, {xs}")
    assert p1["mode"] == (2 if mode == "tc_bf16" else 1) and xs["exact_fallbacks"] == 0
    assert xs["guard_band"] > 0
    for a, b in zip(outs["exact"], outs[mode]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("n_obs", [294, 24], ids=["shelf", "shelf_first24"])
def test_prefilter_overflow_falls_back_to_all_pairs_fp32(factory, n_obs):
    """A network whose hidden activations leave the fp16 range (layer 3 scaled by 1e5, layer 4 by 1e-5: the fp32
    function is an ordinary one) makes the prefilter's fp16 accumulators overflow.  The kernel reports the inf / NaN
    outputs, the call is repeated with every pair scored in fp32, and the result is bitwise the all-pairs one -- for
    the rollout and for distance_repulsion_nn.  With 24 obstacles the fp32 repeat is the whole-horizon kernel.  The
    caller's mode outlives the fallback: it is still the one reported, and the next call falls back again."""
    import optimalmodulationds_b200 as pkg
    from optimalmodulationds_b200.sdf.robot_sdf import RobotSdfCollisionNet
    c = load_npz("case_franka_shelf")
    torch.manual_seed(33)
    net = RobotSdfCollisionNet(in_channels=10, out_channels=9, layers=[256] * 4, skips=[])
    lin = [mod for mod in net.model.modules() if isinstance(mod, torch.nn.Linear)]
    with torch.no_grad():
        for mod in lin:
            torch.nn.init.normal_(mod.weight, std=1.5 / mod.in_features ** 0.5)
            torch.nn.init.normal_(mod.bias, std=0.3)
        lin[2].weight.mul_(1e5); lin[2].bias.mul_(1e5)
        lin[3].weight.mul_(1e-5)
        lin[-1].weight.mul_(20.0); lin[-1].bias.add_(40.0)
    t = lambda x: x.cuda()  # noqa: E731
    N, H = 64, 2
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    res, xs, nn = {}, {}, {}
    for mode in ("exact", "tc_f16"):
        DS = [pkg.LinDS(t(c["qf"])), pkg.LinDS(t(c["q0"]))]
        m = pkg.MPPI(t(c["q0"]), t(c["qf"]), t(c["dh_params"]), t(c["obs"][:n_obs]), float(c["dt"]), H, N, DS,
                     t(c["dh_a"]), net, 5)
        m.set_pass1_mode(mode)
        m.dst_thr, m.ignored_links = 0.01, [0, 1, 2]
        m.q_cur = t(q_cur)
        fallbacks = [m.exactness_stats()["exact_fallbacks"]]
        res[mode] = _rollout_outputs(m)
        fallbacks.append(m.exactness_stats()["exact_fallbacks"])
        assert m.pass1_stats()["mode"] == (1 if mode == "tc_f16" else 0)
        again = _rollout_outputs(m)
        fallbacks.append(m.exactness_stats()["exact_fallbacks"])
        for a, b, name in zip(res[mode], again, ("traj", "dist", "kval", "dots", "acts", "qdot")):
            assert torch.equal(a, b), f"{mode}: {name} differs between two calls"
        nn[mode] = [x.clone() for x in m.distance_repulsion_nn(t(q_cur))]
        fallbacks.append(m.exactness_stats()["exact_fallbacks"])
        xs[mode] = [b - a for a, b in zip(fallbacks, fallbacks[1:])]
    print(f"exact fallbacks per call (rollout, rollout, distance_repulsion_nn): {xs}")
    assert all(x >= 1 for x in xs["tc_f16"]) and xs["exact"] == [0, 0, 0]
    for a, b, name in zip(res["exact"], res["tc_f16"], ("traj", "dist", "kval", "dots", "acts", "qdot")):
        assert torch.isfinite(a).all(), name
        assert torch.equal(a, b), f"overflowing net: {name} differs from the all-pairs fp32 rollout"
    for a, b, name in zip(nn["exact"], nn["tc_f16"], ("distance", "gradient")):
        assert torch.isfinite(a).all(), name
        assert torch.equal(a, b), f"overflowing net: distance_repulsion_nn {name} differs from the all-pairs fp32 one"


def test_debug_pass1_refuses_a_mode_without_a_kernel(factory):
    """dsmppi_debug_pass1 runs the fp32 scoring or one of the two prefilters; AUTO (3) and unknown values return 2
    and leave the object as it was: its next rollout equals a fresh object's bit for bit."""
    c = load_npz("case_franka_shelf")
    torch.manual_seed(13)
    N, H = 64, 2
    q_cur = c["q0"] + 0.2 * torch.randn(N, 7)
    objs = [factory.make_mppi(c, device="cuda", N=N, H=H, q_cur=q_cur, pass1="auto", copy_policy=False)
            for _ in range(2)]
    for m in objs:
        torch.manual_seed(11)
        m.Policy.sample_policy()
    m, fresh = objs
    with torch.cuda.device(m._dev):
        m._upload_obstacles()
        q = q_cur.cuda()
        out = torch.empty(N, c["obs"].shape[0], device="cuda")
        for mode in (3, 7):
            rc = m._lib.dsmppi_debug_pass1(m._ctx, q.data_ptr(), N, m._ignore_mask(), mode, out.data_ptr(), m._stream())
            assert rc == 2 and b"bad pass-1 mode" in m._lib.dsmppi_last_error(), mode
    got, want = _rollout_outputs(m), _rollout_outputs(fresh)
    for a, b, name in zip(got, want, ("traj", "dist", "kval", "dots", "acts", "qdot")):
        assert torch.equal(a, b), f"{name} differs from a fresh object's after refused debug_pass1 calls"


def test_profiler_sees_the_reference_stage_tags(factory, score_mode):
    if score_mode != "tc_split":
        pytest.skip("independent of the scoring arithmetic")
    from torch.profiler import ProfilerActivity, profile
    c = load_npz("case_planar7")
    m = factory.make_mppi(c, device="cpu")
    with profile(activities=[ProfilerActivity.CPU]) as prof:
        m.propagate()
    names = {e.key for e in prof.key_averages()}
    for tag in ("TAG: Nominal vector field", "TAG: evaluate NN", "TAG: QR decomposition", "TAG: Modulation-propagation",
                "TAG: Apply policies", "TAG: Apply policy", "TAG: Propagate", "TAG: evaluate NN_2 (forward pass)",
                "TAG: evaluate NN_4 (forward+backward pass)"):
        assert tag in names, f"{tag} missing from the profiler trace"
    m.propagate()        # and without a profiler attached nothing is opened (no per-call overhead)


def test_graphed_control_tick_equals_the_plain_path(factory, monkeypatch):
    """The integrator's shape (N = 1, H = 2, CPU tensors: frankaIntegrator.py:101-121) and the planner's (40 x 10) run
    as ONE replayed CUDA graph per propagate(); outputs must equal the plain launch path bit for bit, follow obstacle
    and state changes from tick to tick, and re-capture when a script pokes a parameter that is baked into the graph."""
    c = load_npz("case_franka_shelf")
    obs = c["obs"][:28].clone()
    for N, H in ((1, 2), (40, 10)):
        torch.manual_seed(5)
        q_start = c["q0"] + 0.05 * torch.randn(7)
        objs = {}
        for mode in ("graph", "plain"):
            monkeypatch.setenv("DSMPPI_GRAPH_TICK", "1" if mode == "graph" else "0")
            m = factory.make_mppi(dict(c, obs=obs.clone()), device="cpu", N=N, H=H, pass1="auto", copy_policy=False)
            m.Policy.alpha_s = 1.0
            objs[mode] = m
        outs = {k: [] for k in objs}
        for tick in range(6):
            for mode, m in objs.items():
                monkeypatch.setenv("DSMPPI_GRAPH_TICK", "1" if mode == "graph" else "0")
                if tick == 2:
                    m.dst_thr = 0.03                          # parameter poke -> re-capture
                if tick == 3:
                    m.update_obstacles(m.obs + torch.tensor([0.01, 0.0, -0.01, 0.0]))   # streamed obstacles, same count
                if tick == 4:
                    m.Policy.n_kernels = 3                    # fewer live kernels -> new staging shapes
                torch.manual_seed(100 + tick)
                m.Policy.sample_policy()
                m.q_cur = q_start + 0.01 * tick
                traj, dist, kv, dots, acts = m.propagate()
                outs[mode].append([t.clone() for t in (traj, dist, kv, dots, acts, m.qdot, m.nn_grad,
                                                       m.norm_basis, m.kernel_val_all)])
        assert "_tick" in objs["graph"].__dict__ and "_tick" not in objs["plain"].__dict__
        for tick, (a, b) in enumerate(zip(outs["graph"], outs["plain"])):
            for x, y, name in zip(a, b, ("traj", "dist", "kval", "dots", "acts", "qdot", "nn_grad", "norm_basis",
                                         "kernel_val_all")):
                assert x.device.type == "cpu" and x.shape == y.shape, (N, tick, name)
                assert torch.equal(x, y), f"N={N} tick {tick}: {name} differs between the graphed and the plain path"
        # cost / update keep working on the graphed outputs
        g = objs["graph"]
        cost = g.get_cost()
        assert cost.shape == (N,) and torch.isfinite(cost).all()
        g.shift_policy_means()


def test_half_tiles_equal_full_tiles_bitwise(factory, monkeypatch):
    """tc_exact_kernel<2, true> (M = 128 over the CTA pair, 64 rows per CTA) against the full-tile kernel on the
    whole-horizon workloads it serves: planar-7 / planar-2 planner batches and a Franka control tick."""
    cases = [("case_planar7", {}), ("case_c1_planar2", {}), ("case_franka_shelf", dict(obs_n=28, N=3, H=4))]
    for tag, opt in cases:
        c = load_npz(tag)
        if "obs_n" in opt:
            c = dict(c, obs=c["obs"][:opt["obs_n"]].clone())
        outs = {}
        for half in ("1", "0"):
            monkeypatch.setenv("DSMPPI_HALF_TILES", half)
            m = factory.make_mppi(c, device="cuda", N=opt.get("N"), H=opt.get("H"), pass1="auto",
                                  copy_policy="N" not in opt)
            if "N" in opt:
                m.Policy.alpha_s = 1.0
                torch.manual_seed(3)
                m.Policy.sample_policy()
            outs[half] = _rollout_outputs(m) + [m.get_cost().clone()]
        for a, b, name in zip(outs["1"], outs["0"], ("traj", "dist", "kval", "dots", "acts", "qdot", "cost")):
            assert torch.equal(a, b), f"{tag}: {name} differs between half and full tiles"


def test_tick_entry_point_refuses_what_it_cannot_capture(factory):
    """dsmppi_tick covers the dense fp32 scoring path only: with 64+ obstacles (prefilter + host-side verdict) the
    drop-in falls back to the plain path by itself, and the C entry point reports an error instead of capturing."""
    from optimalmodulationds_b200 import _capi
    c = load_npz("case_franka_shelf")                       # 294 spheres
    m = factory.make_mppi(c, device="cpu", N=2, H=2, pass1="auto", copy_policy=False)
    m.propagate()
    assert "_tick" not in m.__dict__                        # not eligible: took the plain path
    ta = _capi.TickArgs()
    dummy = torch.empty(1, device="cuda")
    out = {k: dummy for k in ("all_traj", "closest", "kval", "dots", "acts", "qdot", "grads")}
    ta.rollout = m._rollout_args(2, 2, 0, dummy, dummy, dummy, dummy, out)
    ta.n_obs = 294
    host = torch.zeros(4096)
    for f in ("q_cur_host", "obs_host", "all_traj_host", "closest_dist_all_host", "kernel_val_all_host",
              "dot_products_host", "kernel_activations_host", "qdot_host", "nn_grad_all_host"):
        setattr(ta, f, host.data_ptr())
    rc = m._lib.dsmppi_tick(m._ctx, _capi.C.byref(ta), m._stream())
    assert rc != 0 and b"dense fp32 scoring path" in m._lib.dsmppi_last_error()
