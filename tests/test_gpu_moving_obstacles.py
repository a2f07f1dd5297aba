"""GPU tests of constant-velocity obstacles (MPPI.obs_vel / update_obstacles(obs, obs_vel),
dsmppi_set_obstacle_velocities; run with -m gpu).  The contract: rollout step t = 1..H scores all_traj[:, t-1] against
obs[:, :P] + obs_vel * tau_t with tau_t = (float)(t - 1) * dt in fp32, so
  * zero velocities give the static rollout bit for bit, on every scoring path;
  * each step equals distance_repulsion_nn of an object whose obstacles were moved in torch, bit for bit;
  * teacher-forced steps agree with the CPU oracle run on the moved obstacles;
  * the prefilter stays exact and the whole-horizon kernels equal the per-step launches."""
import pytest
import torch

from oracle import mppi_oracle as orc
from tests.golden_util import load_npz, load_weights
from tests.test_gpu_parity import DIST_ATOL, DOT_ATOL, _host_buffers, check

pytestmark = pytest.mark.gpu

CASES = {"franka": "case_franka_shelf", "planar7": "case_planar7", "planar2": "case_planar2"}
NAMES = ("traj", "dist", "kval", "dots", "acts", "qdot", "grads")


@pytest.fixture(scope="module")
def factory():
    from tests import mppi_factory
    return mppi_factory


def _tau(t, dt):
    """tau of 0-based step t, rounded like the library: (float)t * (float)dt."""
    return torch.tensor(float(t), dtype=torch.float32) * torch.tensor(dt, dtype=torch.float32)


def _moved(obs, vel, tau):
    out = obs.clone()
    out[:, :vel.shape[1]] = obs[:, :vel.shape[1]] + vel * tau
    return out


def _velocities(M, P, H, dt, span, seed):
    """random velocities that move an obstacle by about `span` over the horizon"""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(M, P, generator=g) * (span / (H * dt))


def _make(factory, name, N, H, M=None, obs=None, K=None, pass1="exact", score="ffma", seed=0, device="cuda"):
    """a random-input rollout object like test_rollout_vs_oracle_random_inputs's (fresh policy samples, 6 kernels)"""
    g = torch.Generator().manual_seed(seed)
    base = load_npz(CASES[name])
    d = base["q0"].shape[0]
    if obs is None:
        scale = 0.6 if name == "franka" else 4.0
        obs = torch.cat(((torch.rand(M, 3, generator=g) - 0.5) * 2 * scale, 0.03 + 0.2 * torch.rand(M, 1, generator=g)), 1)
    q_cur = base["q0"] + 0.3 * torch.randn(N, d, generator=g)
    nk = 6
    c = dict(base, obs=obs, N=N, H=H, nk=nk, K=int(base["K"]) if K is None else K)
    m = factory.make_mppi(c, device=device, N=N, H=H, q_cur=q_cur, pass1=pass1, copy_policy=False)
    m.set_score_mode(score)
    P = m.Policy
    P.n_kernels = nk
    P.mu_c[:nk] = (base["q0"] + 0.3 * torch.randn(nk, d, generator=g)).to(P.mu_c.device)
    P.sigma_c[:nk] = 0.7
    P.alpha_c[:nk] = torch.randn(nk, d, generator=g).to(P.alpha_c.device)
    torch.manual_seed(seed)
    P.sample_policy()
    return m, obs, base


def _rollout(m):
    traj, dist, kv, dots, acts = m.propagate()
    grads = m._dev_last["grads"]
    if grads is None:                                        # the graphed tick hands the gradients over on the host
        grads = m._dev_last["grads_host"]
    return [x.detach().cpu().clone() for x in (traj, dist, kv, dots, acts, m.qdot, grads)]


def _assert_equal(a, b, tag):
    for x, y, name in zip(a, b, NAMES):
        assert torch.equal(x, y), f"{tag}: {name} differs"


def _shelf():
    return load_npz("case_franka_shelf")["obs"]


# (id, robot, N, H, M, K, pass1, score, whole horizon)
ZERO_CASES = [
    ("planar7_whole_ffma", "planar7", 300, 8, 4, 2, "exact", "ffma", True),
    ("planar7_whole_tc", "planar7", 300, 8, 4, 2, "exact", "tc_split", True),
    ("planar7_steps_ffma", "planar7", 300, 8, 4, 2, "exact", "ffma", False),
    ("planar7_steps_tc", "planar7", 300, 8, 4, 2, "exact", "tc_split", False),
    ("franka40_two_launch_ffma", "franka", 512, 5, 40, 5, "exact", "ffma", True),
    ("franka40_two_launch_tc", "franka", 512, 5, 40, 5, "exact", "tc_split", True),
    ("shelf294_prefilter_ffma", "franka", 256, 4, 294, 5, "tc_f16", "ffma", True),
    ("shelf294_prefilter_tc", "franka", 256, 4, 294, 5, "tc_f16", "tc_split", True),
]


@pytest.mark.parametrize("tag,name,N,H,M,K,pass1,score,whole", ZERO_CASES, ids=[c[0] for c in ZERO_CASES])
def test_zero_velocities_equal_static_obstacles(factory, tag, name, N, H, M, K, pass1, score, whole):
    obs = _shelf() if M == 294 else None
    m, obs, base = _make(factory, name, N, H, M=M, obs=obs, K=K, pass1=pass1, score=score)
    m.set_whole_horizon(whole)
    static = _rollout(m)
    m.obs_vel = torch.zeros(M, 3, device="cuda")
    _assert_equal(static, _rollout(m), f"{tag}, zero velocities")
    m.obs_vel = _velocities(M, 3, H, float(base["dt"]), 0.3, 1).cuda()
    moving = _rollout(m)
    assert torch.equal(moving[1][:, 0], static[1][:, 0]), "step 1 scores the current positions"
    assert not torch.equal(moving[1], static[1]), "the velocities had no effect"


def test_zero_velocities_equal_static_obstacles_fk_provider(factory):
    m, obs, base = _make(factory, "planar7", 200, 6, M=4)
    m.distance_provider = "fk"
    static = _rollout(m)
    m.obs_vel = torch.zeros(4, 3, device="cuda")
    _assert_equal(static, _rollout(m), "fk provider, zero velocities")
    m.obs_vel = _velocities(4, 3, 6, float(base["dt"]), 0.5, 2).cuda()
    moving = _rollout(m)
    assert torch.equal(moving[1][:, 0], static[1][:, 0]) and not torch.equal(moving[1], static[1])


@pytest.mark.parametrize("whole", [True, False], ids=["whole_horizon", "per_step"])
@pytest.mark.parametrize("score", ["ffma", "tc_split"])
def test_each_step_scores_the_obstacles_moved_in_torch(factory, whole, score):
    """closest_dist[:, t-1] + its stored gradient == distance_repulsion_nn(all_traj[:, t-1]) of an object whose
    obstacles torch moved to tau_t, bit for bit (the distance minus dst_thr in fp32)"""
    N, H, M = 200, 6, 4
    m, obs, base = _make(factory, "planar7", N, H, M=M, K=2, score=score)
    m.set_whole_horizon(whole)
    dt = float(base["dt"])
    vel = _velocities(M, 3, H, dt, 1.0, 3)
    m.update_obstacles(obs, vel.cuda())
    traj, dist, _, _, _, _, grads = _rollout(m)
    ref, _, _ = _make(factory, "planar7", N, 1, M=M, K=2, score=score)
    for t in range(H):
        ref.update_obstacles(_moved(obs, vel, _tau(t, dt)).cuda())
        d2, g2 = ref.distance_repulsion_nn(traj[:, t].cuda())
        assert torch.equal((d2 - m.dst_thr).cpu(), dist[:, t]), f"distance of step {t + 1}"
        assert torch.equal(g2.cpu(), grads[:, t]), f"gradient of step {t + 1}"


@pytest.mark.parametrize("name", ["franka", "planar7", "planar2"])
def test_moving_rollout_vs_oracle(factory, name):
    """teacher-forced against the oracle on the obstacles moved to each step's tau (a CPU-tensor caller)"""
    N, H, M, K = 203, 5, 6, 3
    m, obs, base = _make(factory, name, N, H, M=M, K=K, device="cpu", seed=7)
    dt = float(base["dt"])
    vel = _velocities(M, 3, H, dt, 0.4 if name == "franka" else 2.0, 8)
    m.obs_vel = vel
    P = m.Policy
    traj, dist, kv, dots, acts = m.propagate()
    W, b = load_weights(name)
    net, nk = orc.Net(W, b), int(P.n_kernels)
    prm = orc.RolloutParams(dt=dt, dt_H=1, n_closest_obs=K, dst_thr=float(base["dst_thr"]),
                            ignored_links=base["ignored_links"].tolist(), p=float(P.p), with_basis=False)
    kink = max(1, N // 200)
    for t in range(H):
        o = orc.rollout(net, traj[:, t, :], base["qf"], _moved(obs, vel, _tau(t, dt)), P.mu_tmp, P.sigma_tmp,
                        P.alpha_tmp, nk, prm, N)
        check(dist[:, t], o.closest_dist_all[:, 0], 1e-5, DIST_ATOL, f"dist[{t}]")
        check(dots[:, t], o.dot_products[:, 0], 1e-5, DOT_ATOL, f"dot[{t}]", min_frac=0.9, kink_samples=kink)
        check(acts[:, t], o.kernel_activations[:, 0], 1e-4, 1e-5, f"act[{t}]", kink_samples=kink)
        check(kv[:, t, :], o.kernel_val_all[:, 0, :nk], 1e-4, 1e-6, f"kval[{t}]")
        if t + 1 < H:
            check(traj[:, t + 1, :], traj[:, t, :] + dt * o.qdot, 1e-5, 1e-5, f"traj[{t + 1}]", kink_samples=kink)


def test_moving_toy_vs_oracle(factory):
    """the planar toy network (P = 2): (M, 2) velocities, z stays 0"""
    c = load_npz("toycase_toy2")
    g = torch.Generator().manual_seed(5)
    M, N, H, nk, K = 12, 37, 5, 3, 2
    ang = torch.rand(M, generator=g) * 6.283
    rad = 2 + 2 * torch.rand(M, generator=g)
    obs = torch.stack((rad * torch.cos(ang), rad * torch.sin(ang), 0.2 + 0.3 * torch.rand(M, generator=g)), 1)
    c = dict(c, obs=obs, nk=nk, K=K)
    c["q_cur"] = c["q0"] = torch.tensor([-0.3, 0.2])
    dt = float(c["dt"])
    vel = _velocities(M, 2, H, dt, 1.5, 9)
    m = factory.make_toy_mppi(c, device="cuda", N=N, H=H)
    torch.manual_seed(11)
    m.Policy.sample_policy()
    with pytest.raises(ValueError):
        m.obs_vel = torch.zeros(M, 3).cuda()         # the toy network takes two coordinates
        m.propagate()
    m.obs_vel = vel.cuda()
    mu, sg, al = m.Policy.mu_tmp.cpu(), m.Policy.sigma_tmp.cpu(), m.Policy.alpha_tmp.cpu()
    traj, dist, kv, dots = [x.cpu() for x in m.propagate()]       # MPPI_toy.propagate returns four
    W, b = load_weights("toy2")
    prm = orc.toy_params(dt, 1, K, c["A"], dst_thr=float(c["dst_thr"]), p=float(c["p"]), with_basis=False)
    for t in range(H):
        o = orc.rollout(orc.Net(W, b), traj[:, t], c["qf"], _moved(obs, vel, _tau(t, dt)), mu, sg, al, nk, prm, N)
        check(dist[:, t], o.closest_dist_all[:, 0], 1e-5, 2e-6, f"dist[{t}]")
        check(kv[:, t], o.kernel_val_all[:, 0, :nk], 1e-4, 1e-6, f"kval[{t}]")
        if t + 1 < H:
            check(traj[:, t + 1], traj[:, t] + dt * o.qdot, 1e-5, 1e-5, f"traj[{t + 1}]", kink_samples=1)


def test_prefilter_stays_exact_with_obstacles_crossing_the_arm(factory):
    """the 294-sphere shelf swept through its own centre over the horizon: the fp16 prefilter path equals the
    all-pairs fp32 path bit for bit, without falling back"""
    obs = _shelf()
    base = load_npz("case_franka_shelf")
    N, H = 256, 6
    dt = float(base["dt"])
    centre = obs[:, :3].mean(0)
    vel = (centre - obs[:, :3]) * (2.0 / ((H - 1) * dt))       # every sphere ends mirrored through the centre
    res = {}
    for mode in ("exact", "tc_f16"):
        m, _, _ = _make(factory, "franka", N, H, obs=obs, K=5, pass1=mode, score="tc_split", seed=4)
        m.obs_vel = vel.cuda()
        res[mode] = _rollout(m)
        st, ex = m.pass1_stats(), m.exactness_stats()
        if mode == "tc_f16":
            assert st["mode"] == 1 and st["rescored_pairs"] > 0
            assert ex["exact_fallbacks"] == 0 and ex["guard_band"] > 0
    _assert_equal(res["exact"], res["tc_f16"], "moving shelf, tc_f16 vs exact")


@pytest.mark.parametrize("name,M,score", [("planar7", 4, "ffma"), ("planar7", 4, "tc_split"), ("franka", 24, "ffma"),
                                          ("franka", 24, "tc_split")])
def test_whole_horizon_equals_per_step_launches_with_motion(factory, name, M, score):
    N, H = 96, 6
    out = {}
    for whole in (True, False):
        m, obs, base = _make(factory, name, N, H, M=M, K=3, score=score, seed=6)
        m.set_whole_horizon(whole)
        m.obs_vel = _velocities(M, 3, H, float(base["dt"]), 0.4, 10).cuda()
        out[whole] = _rollout(m)
    _assert_equal(out[True], out[False], f"{name} M={M} {score}: whole horizon vs per step")


def test_update_obstacles_without_velocities_is_static_again(factory):
    m, obs, base = _make(factory, "franka", 128, 4, M=40, K=5)
    static = _rollout(m)
    m.update_obstacles(obs, _velocities(40, 3, 4, float(base["dt"]), 0.3, 11))
    assert not torch.equal(_rollout(m)[1], static[1])
    m.update_obstacles(obs)                                  # the same tensor: only the velocities change
    _assert_equal(static, _rollout(m), "after update_obstacles(obs)")


def test_wrong_velocity_shape_raises(factory):
    m, obs, _ = _make(factory, "planar7", 64, 3, M=4)
    for bad in (torch.zeros(5, 3), torch.zeros(4, 2), torch.zeros(4, 3, 1)):
        m.obs_vel = bad
        with pytest.raises(ValueError):
            m.propagate()


def test_tick_refuses_while_velocities_are_set(factory):
    from optimalmodulationds_b200 import _capi
    m, obs, base = _make(factory, "planar7", 2, 2, M=4, device="cpu")
    static = _rollout(m)
    assert "_tick" in m.__dict__                             # a small CPU-tensor caller takes the graphed tick
    m.obs_vel = _velocities(4, 3, 2, float(base["dt"]), 0.5, 12)
    moving = _rollout(m)
    ta = _capi.TickArgs()
    dummy = torch.empty(1, device="cuda")
    ta.rollout = m._rollout_args(2, 2, 0, dummy, dummy, dummy, dummy, {k: dummy for k in ("all_traj", "closest", "kval",
                                                                                          "dots", "acts", "qdot", "grads")})
    ta.n_obs = 4
    host = torch.zeros(4096)
    for f in ("q_cur_host", "obs_host", "all_traj_host", "closest_dist_all_host", "kernel_val_all_host",
              "dot_products_host", "kernel_activations_host", "qdot_host", "nn_grad_all_host"):
        setattr(ta, f, host.data_ptr())
    rc = m._lib.dsmppi_tick(m._ctx, _capi.C.byref(ta), m._stream())
    assert rc == 2 and b"static obstacles" in m._lib.dsmppi_last_error()
    assert not torch.equal(moving[1], static[1])
    m.obs_vel = None                                         # back to the tick, with the velocities cleared
    again = m.propagate()
    assert torch.equal(again[1], static[1]) and torch.equal(again[0], static[0])


def test_cpu_caller_equals_cuda_caller(factory):
    c = load_npz("case_planar7")
    vel = _velocities(4, 3, int(c["H"]), float(c["dt"]), 1.0, 13)
    out = {}
    for dev in ("cpu", "cuda"):
        m = factory.make_mppi(c, device=dev, pass1="exact")
        m.obs_vel = vel.to(dev)
        out[dev] = [x.detach().cpu().clone() for x in m.propagate()]
    for a, b, name in zip(out["cpu"], out["cuda"], NAMES):
        assert torch.equal(a, b), f"{name}: CPU caller differs from CUDA caller"


def test_iteration_host_equals_device_path_with_motion(factory):
    N, H, M = 300, 4, 40
    m, obs, base = _make(factory, "franka", N, H, M=M, K=5, seed=14)
    vel = _velocities(M, 3, H, float(base["dt"]), 0.3, 15)
    q_cur = m.q_cur.cpu()
    host0 = _host_buffers(m, q_cur)
    m2, _, _ = _make(factory, "franka", N, H, M=M, K=5, seed=14)
    m.obs_vel, m2.obs_vel = vel.cuda(), vel
    traj, dist, kv, dots, acts = m.propagate()
    cost = m.get_cost()
    m.shift_policy_means()
    want = dict(all_traj=traj, closest_dist_all=dist, dot_products=dots, kernel_activations=acts, qdot=m.qdot, cost=cost,
                mu_c=m.Policy.mu_c, sigma_c=m.Policy.sigma_c, alpha_c=m.Policy.alpha_c)
    host = {k: v.clone().pin_memory() for k, v in host0.items()}
    m2.iteration_host(host)
    torch.cuda.synchronize()
    for k, v in want.items():
        assert torch.equal(host[k], v.detach().cpu()), f"{k} differs from the device path"
