"""Drop-in `MPPI` object: the reference's Python API over the sm_100a CUDA library.

Mirror of the reference's ds_mppi/functions/MPPI.py:21-353 -- same constructor arguments, the same
`propagate` / `get_cost` / `shift_policy_means` / `get_qdot` / `update_obstacles` / `switch_DS_idx` /
`reset_DS` / `reset_tensors` / `update_kernel_normal_bases` / `distance_repulsion_nn` / `build_nn_input`
call shapes, the same mutable attributes read at call time, torch tensors in and out on `q0.device`.
Every numerical stage runs in libdsmppi_b200.so (include/dsmppi_b200.h); torch is used for device
memory, streams and (optionally) torch.distributed.  There is NO CPU fallback: without the shared library
or without a CUDA device the constructor raises.

`from MPPI import *` in the reference's scripts also pulls torch, time, np, plt, pi, profile,
record_function, ProfilerActivity, the fk helpers, the plot helpers, TensorPolicyMPPI, eval_rbf and Cost
into the caller's namespace (MPPI.py:1-8); the same names are re-exported here.
"""
import contextlib
import os
import time  # noqa: F401  (re-exported)
from math import pi  # noqa: F401  (re-exported)

import numpy as np  # noqa: F401  (re-exported)
import torch
from torch.profiler import ProfilerActivity, profile, record_function  # noqa: F401  (re-exported)

from . import _capi
from .cost import Cost
from .fk_num import *  # noqa: F401,F403  (numeric_fk_model, numeric_fk_model_vec, dh_fk, plots, plt, np)
from .policy import *  # noqa: F401,F403  (TensorPolicyMPPI, eval_rbf, ...)
from .policy import TensorPolicyMPPI


def generalized_sigmoid(x, y_min, y_max, x0, x1, k):
    return y_min + (y_max - y_min) / (1 + torch.exp(k * (-x + (x0 + x1) / 2)))


# The reference brackets the stages of a rollout step with torch-profiler tags (MPPI.py:102,111,120,134,164,187,218 and
# 229-268); here those stages are ONE fused launch sequence inside the library, so the same names are opened around it
# (nested, outermost first) and existing traces keep their stage names.  Entering a record_function costs ~10 us even
# with no profiler attached, so the tags are only opened while one is.
_ROLLOUT_TAGS = ("TAG: Nominal vector field", "TAG: evaluate NN", "TAG: evaluate NN_2 (forward pass)",
                 "TAG: evaluate NN_3 (get closest obstacle)", "TAG: evaluate NN_4 (forward+backward pass)",
                 "TAG: evaluate NN_5 (process outputs)", "TAG: QR decomposition", "TAG: Modulation-propagation",
                 "TAG: Apply policies", "TAG: Apply policy", "TAG: Propagate")
_DISTANCE_TAGS = ("TAG: evaluate NN_1 (build input)",) + _ROLLOUT_TAGS[2:6]


@contextlib.contextmanager
def _stage_tags(names):
    if not torch.autograd._profiler_enabled():
        yield
        return
    with contextlib.ExitStack() as stack:
        for n in names:
            stack.enter_context(record_function(n))
        yield


_NET_FAMILY = ("the supported distance networks are 3(d+P) -> W -> ... -> W -> O MLPs without skips: 1 to 4 hidden "
               "layers of one width W <= 256, O <= 16 outputs")


def _network_arrays(nn_model):
    """The (out, in) weight matrices and biases of nn_model.model as contiguous fp32 CPU tensors: L hidden layers, then
    the output layer.  Raises NotImplementedError for a network outside the family the library runs."""
    if len(getattr(nn_model.model, 'skips', ()) or ()) > 0:
        raise NotImplementedError(f"skip connections are not supported; {_NET_FAMILY}")
    lin = [m for m in nn_model.model.modules() if isinstance(m, torch.nn.Linear)]
    W = [m.weight.detach().to('cpu', torch.float32).contiguous() for m in lin]
    b = [m.bias.detach().to('cpu', torch.float32).contiguous() for m in lin]
    L = len(W) - 1
    if not 1 <= L <= _capi.MAX_HIDDEN_LAYERS:
        raise NotImplementedError(f"found {max(L, 0)} hidden layers; {_NET_FAMILY}")
    width = W[0].shape[0]
    shapes = [(width, 3 * nn_model.in_channels)] + [(width, width)] * (L - 1) + [(nn_model.out_channels, width)]
    if [tuple(w.shape) for w in W] != shapes or not 1 <= width <= _capi.MAX_HIDDEN \
            or not 1 <= nn_model.out_channels <= _capi.MAX_LINKS:
        raise NotImplementedError(f"layer shapes {[tuple(w.shape) for w in W]}; {_NET_FAMILY}")
    return W, b


class MPPI:
    # which of the two constant sets the reference compiles into its sources (MPPI.py vs MPPI_toy.py); the toy
    # subclass (optimalmodulationds_b200/MPPI_toy.py) overrides these
    _TOY = False
    _COST_TERMS = _capi.COST_ALL
    _UPDATE_VARIANT = 0
    _DEFAULT_DST_THR = 0.5
    _COST_CLASS = Cost

    def __init__(self, q0: torch.Tensor, qf: torch.Tensor, dh_params: torch.Tensor, obs: torch.Tensor, dt: float,
                 dt_H: int, N_traj: int, DS_ARRAY, dh_a, nn_model, n_closest_obs):
        self.tensor_args = {'device': q0.device, 'dtype': q0.dtype}
        if q0.dtype != torch.float32:
            raise NotImplementedError("the CUDA path computes in fp32 (as every reference script does)")
        if not torch.cuda.is_available():
            raise RuntimeError("optimalmodulationds_b200.MPPI needs a CUDA device (B200); there is no CPU fallback")
        self._lib = _capi.load()
        if q0.is_cuda:
            self._dev = q0.device
        else:
            self._dev = torch.device('cuda', int(os.environ.get('DSMPPI_DEVICE', os.environ.get('LOCAL_RANK', 0))))
        self.n_dof = q0.shape[0]
        self.Policy = TensorPolicyMPPI(N_traj, self.n_dof, self.tensor_args)
        self.Policy._backend = self
        self.q0 = q0
        self.DS_idx = 0
        self.DS_ARRAY = DS_ARRAY
        self.DS = DS_ARRAY[self.DS_idx]
        self.qf = self.DS.q_goal.squeeze()
        self.dh_params = dh_params
        self.obs = obs
        self.n_obs = obs.shape[0]
        self.dt = dt
        self.dt_H = dt_H
        self.N_traj = N_traj
        self.dh_a = dh_a
        self.nn_model = nn_model
        self.q_cur = q0
        self.policy_upd_rate = 0.1
        self.dst_thr = self._DEFAULT_DST_THR
        self.ker_thr = 1e-3
        self.ignored_links = [0, 1, 2] if self.n_dof >= 7 else []
        self.n_closest_obs = n_closest_obs
        # 'nn': learned distance network (MPPI.py:113, the live path); 'fk': forward kinematics + sphere distances
        # (the alternative the reference keeps one comment away, MPPI.py:115,306-313)
        self.distance_provider = 'nn'
        self.fk_n_pts = 10
        self.traj_range = torch.arange(self.N_traj, device=q0.device)
        self.kernel_obstacle_bases_tmp = torch.zeros((self.Policy.N_KERNEL_MAX, self.n_dof, self.n_dof),
                                                     **self.tensor_args)
        self._shard = None            # set by enable_sample_sharding
        self._mirror = {}             # device copies of the last outputs, keyed by id() of what we returned
        self._norm_basis = None
        self._ctx = None
        self._make_context()
        self.Cost = self._COST_CLASS(self.qf, self.dh_params, backend=self)
        self.reset_tensors()
        self.qdot = torch.zeros((self.N_traj, self.n_dof), **self.tensor_args)
        self.nn_grad = torch.zeros(N_traj, self.n_dof, **self.tensor_args)
        self.ker_w = torch.zeros((N_traj, 0, 1), **self.tensor_args)
        self.cur_cost = torch.zeros(N_traj, **self.tensor_args)
        # The reference runs five sample_policy + propagate warm-ups here (MPPI.py:69-73).  With no kernels yet their
        # normal_() calls act on empty views and draw nothing from torch's generator (checked against the reference:
        # tests/test_gpu_api_edges.py), so the RNG stream a seeded script sees afterwards is the same with any number
        # of them; the five policy draws are kept, and ONE rollout is enough to size the library's workspace.
        for _ in range(5):
            self.Policy.sample_policy()
        self.propagate()

    # ------------------------------------------------------------------ backend plumbing
    def _make_context(self):
        W, b = _network_arrays(self.nn_model)
        # network input = [q, obstacle coordinates]: 3 coordinates for the robot nets, 2 for the planar toy net
        self._point_dim = int(self.nn_model.in_channels) - self.n_dof
        if self._point_dim not in (2, 3):
            raise ValueError(f"network takes {self.nn_model.in_channels} inputs, q0 has {self.n_dof} joints: "
                             "expected n_dof + 3 (or n_dof + 2 for the planar toy net)")
        net = _capi.Net()
        net.n_dof, net.n_out, net.n_point_dim = self.n_dof, self.nn_model.out_channels, self._point_dim
        net.n_hidden, net.hidden_width = len(W) - 1, W[0].shape[0]
        for i in range(len(W)):
            net.W_host[i] = W[i].data_ptr()
            net.b_host[i] = b[i].data_ptr()
        dh = self.dh_params.detach().to('cpu', torch.float32).contiguous()
        if dh.dim() != 2 or dh.shape[1] != 4 or dh.shape[0] < self.n_dof + 1:
            raise ValueError("dh_params must be (n_dof + 1, 4) = [d, theta, a, alpha]")
        dh = dh[:self.n_dof + 1].contiguous()      # standaloneToy2d.py:55 passes a (4, 4) dummy for 2 joints
        handle = _capi.C.c_void_p()
        with torch.cuda.device(self._dev):
            _capi.check(self._lib.dsmppi_ctx_create(_capi.C.byref(handle), _capi.C.byref(net), dh.data_ptr(),
                                                    int(self.N_traj), int(self._dev.index or 0)))
        self._ctx = handle

    def __del__(self):
        ctx, self._ctx = getattr(self, '_ctx', None), None
        if ctx:
            try:
                self._lib.dsmppi_ctx_destroy(ctx)
            except Exception:  # noqa: BLE001 - interpreter shutdown
                pass

    def _stream(self):
        return _capi.C.c_void_p(torch.cuda.current_stream(self._dev).cuda_stream)

    def _host_vec(self, t):
        """Small parameter vectors (goal, joint limits) as Python floats.  A CUDA tensor is copied to the host once per
        (tensor, in-place version): a `.to('cpu')` on every call would synchronise with the device and keep the CPU
        from running ahead of the rollout it has just launched."""
        if isinstance(t, torch.Tensor):
            cache = self.__dict__.setdefault('_hostvec_cache', {})
            hit = cache.get(id(t))
            if hit is not None and hit[0] is t and hit[1] == t._version:
                return hit[2]
            vals = t.detach().reshape(-1).to('cpu', torch.float32).tolist()
            if len(cache) > 64:
                cache.clear()
            cache[id(t)] = (t, t._version, vals)
            return vals
        return torch.as_tensor(t).detach().reshape(-1).to('cpu', torch.float32).tolist()

    def _d(self, t):
        """Tensor on the compute device, fp32, contiguous (no copy when it already is)."""
        return torch.as_tensor(t).detach().to(self._dev, torch.float32).contiguous()

    def _u(self, t):
        """Tensor on the caller's device."""
        return t if t.device == self.tensor_args['device'] else t.to(self.tensor_args['device'])

    def _dev_of(self, user_tensor):
        """Device copy of a tensor we handed out earlier (identity match), else a fresh upload."""
        hit = self._mirror.get(id(user_tensor))
        if hit is not None and hit[0] is user_tensor and hit[1] == user_tensor._version:
            return hit[2]
        return self._d(user_tensor)

    def _remember(self, user_tensor, dev_tensor):
        # the version counter catches in-place edits the caller made after we uploaded the tensor
        self._mirror[id(user_tensor)] = (user_tensor, user_tensor._version, dev_tensor)

    def set_pass1_mode(self, mode='auto', guard_band=0.0):
        """How obstacles are ranked: 'exact' (fp32 on every pair), 'tc_f16' / 'tc_bf16' (tcgen05 prefilter +
        fp32 re-score of everything within `guard_band` metres of the K-th), or 'auto'."""
        code = {'exact': _capi.PASS1_EXACT_FP32, 'tc_f16': _capi.PASS1_TC_F16, 'tc_bf16': _capi.PASS1_TC_BF16,
                'auto': _capi.PASS1_AUTO}[mode]
        _capi.check(self._lib.dsmppi_set_pass1_mode(self._ctx, code, float(guard_band)))
        self._pass1_forced = mode
        self.__dict__.pop('_tick', None)

    def set_score_mode(self, mode='auto'):
        """Arithmetic of the rows that produce outputs: 'ffma' (IEEE fp32 on the CUDA cores, the strict mode),
        'tc_split' (tcgen05 with split-fp16 operands, fp32-accurate) or 'auto' (tc_split when the network fits)."""
        code = {'ffma': _capi.SCORE_FFMA, 'tc_split': _capi.SCORE_TC_SPLIT, 'auto': _capi.SCORE_AUTO}[mode]
        _capi.check(self._lib.dsmppi_set_score_mode(self._ctx, code))
        self.__dict__.pop('_tick', None)

    def score_stats(self):
        """Scoring arithmetic in effect and the rows the tensor-core path handed to the FFMA kernel (fp16 range)."""
        mode, fix, drop = _capi.C.c_int32(), _capi.C.c_int64(), _capi.C.c_int64()
        _capi.check(self._lib.dsmppi_score_stats(self._ctx, _capi.C.byref(mode), _capi.C.byref(fix),
                                                 _capi.C.byref(drop), self._stream()))
        return dict(mode={_capi.SCORE_FFMA: 'ffma', _capi.SCORE_TC_SPLIT: 'tc_split'}[mode.value],
                    range_fixup_rows=fix.value, dropped_rows=drop.value)

    def set_whole_horizon(self, on=True):
        """Small obstacle sets are rolled out by one launch over the whole horizon; False forces per-step launches."""
        _capi.check(self._lib.dsmppi_set_whole_horizon(self._ctx, 1 if on else 0))
        self.__dict__.pop('_tick', None)

    def _upload_obstacles(self):
        # scripts hand the same tensor back every iteration (frankaPlanner.py:129-130 re-assigns the last message):
        # upload and re-encode only when the object or its in-place version changed
        src = self.obs
        hit = getattr(self, '_obs_uploaded', None)
        if (hit is not None and isinstance(src, torch.Tensor) and hit[0] is src and hit[1] == src._version):
            return hit[2]
        obs = self._d(self.obs)
        if obs.dim() != 2 or obs.shape[1] != self._point_dim + 1:
            raise ValueError("obs must be (M, 4) = [x, y, z, r]" if self._point_dim == 3 else
                             "obs must be (M, 3) = [x, y, r] for a network with n_dof + 2 inputs")
        self.n_obs = obs.shape[0]
        _capi.check(self._lib.dsmppi_set_obstacles(self._ctx, obs.data_ptr(), int(obs.shape[0]), self._stream()))
        if isinstance(src, torch.Tensor):
            self._obs_uploaded = (src, src._version, obs)
        return obs

    def _ignore_mask(self):
        mask = 0
        for link in self.ignored_links:
            mask |= 1 << int(link)
        return mask

    # ------------------------------------------------------------------ reference API
    def reset_DS(self, DS):
        self.DS = DS
        self.qf = DS.q_goal.squeeze()
        self._rebuild_cost()

    def switch_DS_idx(self, idx):
        self.DS_idx = idx
        self.DS = self.DS_ARRAY[idx]
        self.qf = self.DS.q_goal.squeeze()
        self._rebuild_cost()

    def _rebuild_cost(self):
        old = getattr(self, 'Cost', None)
        self.Cost = self._COST_CLASS(self.qf, self.dh_params, backend=self)
        if old is not None:                      # keep limits the caller assigned after construction
            self.Cost.q_min, self.Cost.q_max = old.q_min, old.q_max

    def reset_tensors(self):
        N, H, d = self.N_traj, self.dt_H, self.n_dof
        a = self.tensor_args
        self.all_traj = torch.zeros(N, H, d, **a)
        self.closest_dist_all = 100 + torch.zeros(N, H, **a)
        self.kernel_val_all = torch.zeros(N, H, self.Policy.N_KERNEL_MAX, **a)
        self.dot_products = torch.zeros(N, H, **a)
        self.kernel_activations = torch.zeros(N, H, **a)

    def build_nn_input(self, q_tens, obs_tens):
        self.nn_input = torch.hstack((q_tens.tile(obs_tens.shape[0], 1), obs_tens.repeat_interleave(q_tens.shape[0], 0)))
        return self.nn_input

    def _modulation(self, mod):
        """Fills the constants of the modulation law and the nominal dynamics (read at call time)."""
        if self._TOY:
            self._lib.dsmppi_modulation_toy(_capi.C.byref(mod))
        else:
            self._lib.dsmppi_modulation_default(_capi.C.byref(mod))
        if hasattr(self.DS, 'Mu') and hasattr(self.DS, 'Sigma'):
            mod.ds_kind = _capi.DS_SEDS
            self._upload_seds(self.DS)
        elif hasattr(self.DS, 'lin_thr'):
            mod.ds_kind = _capi.DS_LINEAR_ATTRACTOR
        elif hasattr(self.DS, 'A'):
            mod.ds_kind = _capi.DS_MATRIX
            A = torch.as_tensor(self.DS.A).detach().to('cpu', torch.float32)
            if A.shape != (self.n_dof, self.n_dof):
                raise ValueError("the matrix DS needs A of shape (n_dof, n_dof)")
            for r in range(self.n_dof):
                for c in range(self.n_dof):
                    mod.ds_A[r * _capi.MAX_DOF + c] = float(A[r, c])
        else:
            raise NotImplementedError("the CUDA rollout implements the LinDS attractor (LinDS.py), the SEDS mixture "
                                      "(SEDS.py) and the matrix DS v = (q - qf) @ A (MPPI_toy.py:89) as nominal "
                                      "dynamics")

    def _upload_seds(self, ds):
        """Packs a SEDS object (reference class or optimalmodulationds_b200.SEDS) for the step kernel; re-uploaded
        only when another DS object becomes current."""
        if getattr(self, '_seds_uploaded', None) is ds:
            return
        from .SEDS import SEDS as _SEDS
        src = ds if isinstance(ds, _SEDS) else _SEDS.from_arrays(ds.Mu, ds.Sigma, ds.Priors, ds.q_goal)
        if src.dof != self.n_dof:
            raise ValueError(f"SEDS has {src.dof} joints, the robot {self.n_dof}")
        arrs = [t.detach().to('cpu', torch.float32).contiguous() for t in src.kernel_arrays()]
        sd = _capi.Seds()
        sd.n_gaussians, sd.seds_thr = int(src.n_gaussians), float(getattr(ds, 'seds_thr', 1e-2))
        (sd.priors_host, sd.pdf_den_host, sd.mu_x_host, sd.mu_y_host, sd.sigma_inv_host,
         sd.A_host) = (t.data_ptr() for t in arrs)
        with torch.cuda.device(self._dev):
            _capi.check(self._lib.dsmppi_set_seds(self._ctx, _capi.C.byref(sd), self._stream()))
        self._seds_uploaded = ds

    def _rollout_args(self, N, H, nk, q_cur, mu, sigma, alpha, out):
        a = _capi.RolloutArgs()
        a.N, a.H, a.n_kernels, a.n_closest = N, H, nk, int(self.n_closest_obs)
        a.q_cur_is_batch = 1 if q_cur.dim() == 2 else 0
        a.ignored_link_mask = self._ignore_mask()
        a.dt, a.dst_thr = float(self.dt), float(self.dst_thr)
        self._modulation(a.mod)
        if self.distance_provider == 'fk':
            a.distance_provider, a.fk_n_pts = _capi.DISTANCE_FK, int(self.fk_n_pts)
            for i, v in enumerate(torch.linspace(0.01, 1, int(self.fk_n_pts)).tolist()):
                a.fk_span[i] = v
        elif self.distance_provider != 'nn':
            raise ValueError("distance_provider must be 'nn' or 'fk'")
        a.lin_thr, a.rbf_p = float(getattr(self.DS, 'lin_thr', 0.0)), float(self.Policy.p)
        goal = self._host_vec(self.DS.q_goal)
        for i in range(self.n_dof):
            a.q_goal[i] = goal[i]
        a.q_cur_dev = q_cur.data_ptr()
        a.mu_tmp_dev, a.sigma_tmp_dev, a.alpha_tmp_dev = mu.data_ptr(), sigma.data_ptr(), alpha.data_ptr()
        a.all_traj_dev = out['all_traj'].data_ptr()
        a.closest_dist_all_dev = out['closest'].data_ptr()
        a.kernel_val_all_dev = out['kval'].data_ptr()
        a.dot_products_dev = out['dots'].data_ptr()
        a.kernel_activations_dev = out['acts'].data_ptr()
        a.qdot_dev = out['qdot'].data_ptr()
        a.nn_grad_all_dev = out['grads'].data_ptr()
        a.norm_basis_dev = None
        return a

    # ------------------------------------------------------------------ control tick: one CUDA graph per rollout
    # The integrator process calls propagate() with ONE sample and TWO steps every control tick, on CPU tensors
    # (frankaIntegrator.py:101-121).  At that size the rollout itself is one ~90 us launch and the tick is spent in
    # the wrapper: seven allocations, four uploads, the ctypes call, six downloads (each a stream synchronisation).
    # For small batches of CPU-tensor callers the whole tick -- upload of the state, the policy rows and the obstacles
    # from a pinned staging block, the library's launch sequence, download of every output -- is captured ONCE into a
    # CUDA graph inside the library (dsmppi_tick) and replayed: one C call, one cudaGraphLaunch and one synchronisation
    # per tick.  Kernel arguments are baked into a graph, so the library keys it by the bytes of the argument block
    # (time step, thresholds, goal, n_kernels, obstacle count, ...) and re-captures when a script changes any of them;
    # results are those of the normal path bit for bit (the same launches).  DSMPPI_GRAPH_TICK=0 disables it.
    _TICK_MAX_STATE_STEPS = 4096

    def _tick_eligible(self, q_cur):
        if os.environ.get('DSMPPI_GRAPH_TICK', '1') == '0' or self.tensor_args['device'].type != 'cpu':
            return False
        if self.N_traj * self.dt_H > self._TICK_MAX_STATE_STEPS or self.distance_provider != 'nn':
            return False
        if self._shard is not None or hasattr(self.DS, 'Mu') or getattr(self, '_timing_on', False):
            return False
        if int(self.obs.shape[0]) >= 64 or getattr(self, '_pass1_forced', 'auto') not in ('auto', 'exact'):
            return False            # the prefilter path ends with a host-side verdict: not capturable
        obs = self.obs
        return (isinstance(obs, torch.Tensor) and obs.dim() == 2 and obs.shape[1] == self._point_dim + 1
                and obs.dtype == torch.float32 and q_cur.dtype == torch.float32)

    def _tick_key(self, nk, q_batch):
        """Everything dsmppi_rollout_args bakes into the captured kernel arguments, cheaply (the argument block itself
        is only rebuilt when this changes; the library compares the block's bytes and re-captures its graph)."""
        DS = self.DS
        A = getattr(DS, 'A', None)
        return (nk, q_batch, int(self.n_closest_obs), self._ignore_mask(), float(self.dt), float(self.dst_thr),
                float(self.Policy.p), type(DS), tuple(self._host_vec(DS.q_goal)), float(getattr(DS, 'lin_thr', 0.0)),
                None if A is None else tuple(self._host_vec(A)))

    def _propagate_tick(self, q_cur_user, nk):
        """propagate() of a small CPU-tensor batch through dsmppi_tick: one C call per tick."""
        N, H, d = self.N_traj, self.dt_H, self.n_dof
        P = self.Policy
        q_batch = q_cur_user.dim() == 2
        key = self._tick_key(nk, q_batch)
        t = self.__dict__.get('_tick')
        if t is None or t['key'] != key:
            dummy = torch.empty(1, device=self._dev)
            probe = torch.empty((N, d) if q_batch else (d,), device='meta')
            out = {k: dummy for k in ('all_traj', 'closest', 'kval', 'dots', 'acts', 'qdot', 'grads')}
            ta = _capi.TickArgs()
            ta.rollout = self._rollout_args(N, H, nk, dummy, dummy, dummy, dummy, out)
            ta.rollout.q_cur_is_batch = 1 if probe.dim() == 2 else 0
            t = self._tick = dict(key=key, args=ta, keep=dummy)
        ta = t['args']
        obs = self.obs if self.obs.is_contiguous() else self.obs.contiguous()
        q = q_cur_user if q_cur_user.is_contiguous() else q_cur_user.contiguous()
        ta.n_obs = int(obs.shape[0])
        ta.q_cur_host, ta.obs_host = q.data_ptr(), obs.data_ptr()
        mu, sg, al = P.mu_tmp, P.sigma_tmp, P.alpha_tmp
        if nk > 0:
            if not (mu.is_contiguous() and sg.is_contiguous() and al.is_contiguous()):
                mu, sg, al = mu.contiguous(), sg.contiguous(), al.contiguous()
            ta.mu_tmp_host, ta.sigma_tmp_host, ta.alpha_tmp_host = mu.data_ptr(), sg.data_ptr(), al.data_ptr()
        traj, closest, kv = torch.empty(N, H, d), torch.empty(N, H), torch.empty(N, H, P.N_KERNEL_MAX)
        dots, acts, qdot, grads = torch.empty(N, H), torch.empty(N, H), torch.empty(N, d), torch.empty(N, H, d)
        ta.all_traj_host, ta.closest_dist_all_host, ta.kernel_val_all_host = traj.data_ptr(), closest.data_ptr(), kv.data_ptr()
        ta.dot_products_host, ta.kernel_activations_host = dots.data_ptr(), acts.data_ptr()
        ta.qdot_host, ta.nn_grad_all_host = qdot.data_ptr(), grads.data_ptr()
        _capi.check(self._lib.dsmppi_tick(self._ctx, _capi.C.byref(ta), self._stream()))
        self._mirror = {}
        self._obs_uploaded = None
        self._norm_basis = None
        self._dev_last = dict(grads=None, grads_host=grads, nk=nk)
        self.all_traj, self.closest_dist_all, self.kernel_val_all = traj, closest, kv
        self.dot_products, self.kernel_activations, self.qdot = dots, acts, qdot
        self.nn_grad = grads[:, H - 1, :]
        self.ker_w = kv[:, H - 1, :nk].unsqueeze(2)
        return (traj, closest, kv[:, :, 0:nk], dots, acts)

    def propagate(self):
        N, H, d = self.N_traj, self.dt_H, self.n_dof
        P = self.Policy
        nk = int(P.n_kernels)
        dev = self._dev
        q_user = torch.as_tensor(self.q_cur)
        if self._tick_eligible(q_user):
            if q_user.shape not in ((d,), (N, d)):
                raise ValueError(f"q_cur must be ({d},) or ({N}, {d}), got {tuple(q_user.shape)}")
            with _stage_tags(_ROLLOUT_TAGS):
                return self._propagate_tick(q_user, nk)
        with torch.cuda.device(dev):
            q_cur = self._d(self.q_cur)
            if q_cur.shape not in ((d,), (N, d)):
                raise ValueError(f"q_cur must be ({d},) or ({N}, {d}), got {tuple(q_cur.shape)}")
            mu, sigma, alpha = self._d(P.mu_tmp), self._d(P.sigma_tmp), self._d(P.alpha_tmp)
            if mu.shape != (N, P.N_KERNEL_MAX, d):
                raise ValueError("Policy.mu_tmp must be (N_traj, 50, n_dof)")
            self._upload_obstacles()
            out = dict(all_traj=torch.empty(N, H, d, device=dev), closest=torch.empty(N, H, device=dev),
                       kval=torch.zeros(N, H, P.N_KERNEL_MAX, device=dev), dots=torch.empty(N, H, device=dev),
                       acts=torch.empty(N, H, device=dev), qdot=torch.empty(N, d, device=dev),
                       grads=torch.empty(N, H, d, device=dev))
            args = self._rollout_args(N, H, nk, q_cur, mu, sigma, alpha, out)
            with _stage_tags(_ROLLOUT_TAGS):
                _capi.check(self._lib.dsmppi_rollout(self._ctx, _capi.C.byref(args), self._stream()))
        self._mirror = {}
        self._dev_last = dict(out, mu=mu, sigma=sigma, alpha=alpha, nk=nk)
        self._norm_basis = None
        if self.tensor_args['device'] == dev:
            self.all_traj, self.closest_dist_all, self.kernel_val_all = out['all_traj'], out['closest'], out['kval']
            self.dot_products, self.kernel_activations, self.qdot = out['dots'], out['acts'], out['qdot']
        else:
            self.all_traj, self.closest_dist_all = self._u(out['all_traj']), self._u(out['closest'])
            self.dot_products, self.kernel_activations = self._u(out['dots']), self._u(out['acts'])
            self.qdot = self._u(out['qdot'])
            kv = torch.zeros(N, H, P.N_KERNEL_MAX, **self.tensor_args)
            if nk > 0:
                kv[:, :, :nk] = self._u(out['kval'][:, :, :nk])
            self.kernel_val_all = kv
        for user, key in ((self.all_traj, 'all_traj'), (self.closest_dist_all, 'closest'),
                          (self.kernel_val_all, 'kval'), (self.kernel_activations, 'acts')):
            self._remember(user, out[key])
        self._remember(P.mu_tmp, mu), self._remember(P.sigma_tmp, sigma), self._remember(P.alpha_tmp, alpha)
        self.nn_grad = self._u(out['grads'][:, H - 1, :])
        self.ker_w = self.kernel_val_all[:, H - 1, :nk].unsqueeze(2)
        return (self.all_traj, self.closest_dist_all, self.kernel_val_all[:, :, 0:nk], self.dot_products,
                self.kernel_activations)

    @property
    def norm_basis(self):
        """(N, H, d, d) Householder bases of every state-step (MPPI.py:122-127), materialised on first access
        from the stored blended gradients (SURVEY 7: keeps 4*d*d bytes per state-step off the rollout)."""
        if self._norm_basis is None:
            g = self._dev_last['grads']
            if g is None:
                g = self._d(self._dev_last['grads_host'])
            N, H, d = g.shape
            with torch.cuda.device(self._dev):
                E = torch.empty(N, H, d, d, device=self._dev)
                _capi.check(self._lib.dsmppi_norm_basis(self._ctx, g.data_ptr(), N * H, E.data_ptr(), self._stream()))
            self._norm_basis = self._u(E)
        return self._norm_basis

    @norm_basis.setter
    def norm_basis(self, value):
        self._norm_basis = value

    def distance_repulsion_nn(self, q_prev, aot=False):
        q = self._d(q_prev)
        n = q.shape[0]
        with torch.cuda.device(self._dev):
            self._upload_obstacles()
            dist = torch.empty(n, device=self._dev)
            grad = torch.empty(n, self.n_dof, device=self._dev)
            with _stage_tags(_DISTANCE_TAGS):
                _capi.check(self._lib.dsmppi_distance_grad(self._ctx, q.data_ptr(), n, int(self.n_closest_obs),
                                                           self._ignore_mask(), dist.data_ptr(), grad.data_ptr(),
                                                           self._stream()))
        self.nn_grad = self._u(grad)
        return self._u(dist), self.nn_grad

    def distance_repulsion_fk(self, q_prev, return_indices=False):
        """MPPI.py:306-313: true link-to-sphere distance (10 points per link) and its joint gradient, padded to 7
        columns like the reference's `lambda_rep_vec` (fk_sym_gen.py:265-269)."""
        q = self._d(q_prev)
        n = q.shape[0]
        n_pts = int(self.fk_n_pts)
        span = torch.linspace(0.01, 1, n_pts).contiguous()
        with torch.cuda.device(self._dev):
            self._upload_obstacles()
            dist = torch.empty(n, device=self._dev)
            grad = torch.empty(n, self.n_dof, device=self._dev)
            idx = torch.empty(n, 3, dtype=torch.int32, device=self._dev)
            _capi.check(self._lib.dsmppi_distance_grad_fk(self._ctx, q.data_ptr(), n, n_pts, span.data_ptr(),
                                                          dist.data_ptr(), grad.data_ptr(), idx.data_ptr(),
                                                          self._stream()))
        rep = torch.zeros(n, max(7, self.n_dof), device=self._dev)
        rep[:, :self.n_dof] = grad
        rep = self._u(rep)
        self.nn_grad = rep[:, 0:self.n_dof]
        if return_indices:
            return self._u(dist), rep, self._u(idx)
        return self._u(dist), rep

    def update_kernel_normal_bases(self):
        nk = int(self.Policy.n_kernels)
        if nk > 0:
            _, grad = self.distance_repulsion_nn(self.Policy.mu_c[0:nk], aot=False)
            g = self._d(grad)
            with torch.cuda.device(self._dev):
                E = torch.empty(nk, self.n_dof, self.n_dof, device=self._dev)
                _capi.check(self._lib.dsmppi_norm_basis(self._ctx, g.data_ptr(), nk, E.data_ptr(), self._stream()))
            self.Policy.kernel_obstacle_bases[0:nk] = E.to(self.Policy.kernel_obstacle_bases.device)
        return 0

    # ------------------------------------------------------------------ cost
    def evaluate_costs(self, cost_obj, all_traj, closest_dist_all):
        """Backend of Cost.evaluate_costs (cost.py:13-22)."""
        N, H, d = all_traj.shape
        a = _capi.CostArgs()
        a.N, a.H, a.terms = N, H, self._COST_TERMS
        goal, qmin, qmax = self._host_vec(cost_obj.qf), self._host_vec(cost_obj.q_min), self._host_vec(cost_obj.q_max)
        if len(qmin) < d or len(qmax) < d:
            raise ValueError("Cost.q_min / q_max must have n_dof entries")
        for i in range(d):
            a.q_goal[i], a.q_min[i], a.q_max[i] = goal[i], qmin[i], qmax[i]
        with torch.cuda.device(self._dev):
            tr, cd = self._dev_of(all_traj), self._dev_of(closest_dist_all)
            cost = torch.empty(N, device=self._dev)
            a.all_traj_dev, a.closest_dist_all_dev, a.cost_dev = tr.data_ptr(), cd.data_ptr(), cost.data_ptr()
            _capi.check(self._lib.dsmppi_cost(self._ctx, _capi.C.byref(a), self._stream()))
        user = self._u(cost)
        self._remember(user, cost)
        return user

    def kernel_candidates(self, policy, all_traj, closest_dist_all, dot_products, thr_dist, thr_kernel, thr_dot):
        """Backend of TensorPolicyMPPI.check_traj_for_kernels (policy.py:153-175)."""
        N, H, d = all_traj.shape
        nk = int(policy.n_kernels)
        a = _capi.CandidatesArgs()
        a.N, a.H, a.n_kernels, a.rbf_p = N, H, nk, float(policy.p)
        a.thr_dist, a.thr_kernel, a.thr_dot = float(thr_dist), float(thr_kernel), float(thr_dot)
        with torch.cuda.device(self._dev):
            tr, cd, dp = self._dev_of(all_traj), self._dev_of(closest_dist_all), self._dev_of(dot_products)
            mu_c, sigma_c = self._d(policy.mu_c), self._d(policy.sigma_c)
            count = torch.zeros(1, dtype=torch.int32, device=self._dev)
            cap = min(N * H, 1 << 20)
            while True:
                idx = torch.empty(cap, dtype=torch.int32, device=self._dev)
                a.all_traj_dev, a.closest_dist_all_dev, a.dot_products_dev = tr.data_ptr(), cd.data_ptr(), dp.data_ptr()
                a.mu_c_dev, a.sigma_c_dev = mu_c.data_ptr(), sigma_c.data_ptr()
                a.out_index_dev, a.count_dev, a.capacity = idx.data_ptr(), count.data_ptr(), cap
                _capi.check(self._lib.dsmppi_kernel_candidates(self._ctx, _capi.C.byref(a), self._stream()))
                n = int(count.item())
                if n <= cap:
                    break
                cap = N * H                      # rare: more candidates than the first buffer holds
            order = torch.sort(idx[:n].long())[0]          # the reference returns them in (i, h) order
            cand = tr.reshape(-1, d)[order]
        return self._u(cand)

    def get_cost(self):
        self.cur_cost = self.Cost.evaluate_costs(self.all_traj, self.closest_dist_all)
        return self.cur_cost

    def get_qdot(self, mode='best'):
        qdot = 0
        if mode == 'best':
            qdot = self.qdot[torch.argmin(self.cur_cost), :]
        elif mode == 'weighted':
            beta = self.cur_cost.mean() / 50
            w = torch.exp(-1 / beta * self.cur_cost)
            w = w / w.sum()
            qdot = torch.sum(w.unsqueeze(1) * self.qdot, dim=0)
        return qdot

    # ------------------------------------------------------------------ policy update
    def enable_sample_sharding(self, group=None):
        """Sample-sharded MPPI (SURVEY 8(e)): this object holds N_traj local samples of a job spread over the
        ranks of `group`; shift_policy_means then all-reduces the cost statistics and the packed weighted
        sums (two small NCCL all-reduces per iteration) so every rank applies the identical update."""
        import torch.distributed as dist
        world = dist.get_world_size(group)
        # the global sample count is fixed while the object lives: one all-reduce here, none (and no host
        # synchronisation) per iteration
        n = torch.tensor([float(self.N_traj)], device=self._dev)
        dist.all_reduce(n, group=group)
        self._shard = dict(group=group, rank=dist.get_rank(group), world=world, N_global=int(round(float(n))))

    def shift_policy_means(self):
        P = self.Policy
        nk = int(P.n_kernels)
        N, H, d = self.N_traj, self.dt_H, self.n_dof
        dev = self._dev
        with torch.cuda.device(dev):
            a = _capi.UpdateArgs()
            a.N, a.H, a.n_kernels = N, H, nk
            a.owns_sample0, a.N_global, a.variant = 1, N, self._UPDATE_VARIANT
            a.ker_thr, a.upd_rate = float(self.ker_thr), float(self.policy_upd_rate)
            cost = self._dev_of(self.cur_cost)
            kv, acts = self._dev_of(self.kernel_val_all), self._dev_of(self.kernel_activations)
            mu, sigma, alpha = self._dev_of(P.mu_tmp), self._dev_of(P.sigma_tmp), self._dev_of(P.alpha_tmp)
            mu_c, sigma_c, alpha_c = (self._d(t).clone() for t in (P.mu_c, P.sigma_c, P.alpha_c))
            a.cost_dev, a.kernel_val_all_dev, a.kernel_activations_dev = cost.data_ptr(), kv.data_ptr(), acts.data_ptr()
            a.mu_tmp_dev, a.sigma_tmp_dev, a.alpha_tmp_dev = mu.data_ptr(), sigma.data_ptr(), alpha.data_ptr()
            a.mu_c_dev, a.sigma_c_dev, a.alpha_c_dev = mu_c.data_ptr(), sigma_c.data_ptr(), alpha_c.data_ptr()
            stats = torch.empty(4, device=dev)
            packed = torch.empty(int(self._lib.dsmppi_update_packed_len(nk, d)), device=dev)
            n_upd = torch.zeros(1, dtype=torch.int32, device=dev)
            st = self._stream()
            _capi.check(self._lib.dsmppi_update_cost_stats(self._ctx, cost.data_ptr(), N, stats.data_ptr(), st))
            if self._shard is not None:
                from .parallel import allreduce_cost_stats, allreduce_packed
                a.owns_sample0 = 1 if self._shard['rank'] == 0 else 0
                a.N_global = self._shard['N_global']
                allreduce_cost_stats(stats, self._shard['group'])
            _capi.check(self._lib.dsmppi_update_partial(self._ctx, _capi.C.byref(a), stats.data_ptr(),
                                                        packed.data_ptr(), st))
            if self._shard is not None:
                allreduce_packed(packed, self._shard['group'])
            _capi.check(self._lib.dsmppi_update_finalize(self._ctx, _capi.C.byref(a), packed.data_ptr(),
                                                         n_upd.data_ptr(), st))
        if nk > 0:      # in-place slice assignment keeps aliases of the mean tensors alive (policy.py:108-113)
            P.mu_c[0:nk] = mu_c[0:nk].to(P.mu_c.device)
            P.sigma_c[0:nk] = sigma_c[0:nk].to(P.sigma_c.device)
            P.alpha_c[0:nk] = alpha_c[0:nk].to(P.alpha_c.device)
        self._last_stats = stats
        return 0, n_upd.to(self.tensor_args['device'])[0].to(torch.int64)

    def iteration_host(self, host):
        """One whole MPPI iteration through the C ABI's host-buffer entry point (dsmppi_iteration_host):
        `host` is a dict of CPU tensors (ideally pinned) -- inputs q_cur, mu_tmp, sigma_tmp, alpha_tmp, in/out
        mu_c, sigma_c, alpha_c, outputs all_traj, closest_dist_all, kernel_val_all, dot_products,
        kernel_activations, qdot, cost, n_updated (int32).  Returns (h2d_bytes, d2h_bytes)."""
        N, H, d = self.N_traj, self.dt_H, self.n_dof
        P = self.Policy
        a = _capi.IterationHostArgs()
        dummy = torch.empty(1, device=self._dev)
        out = {k: dummy for k in ('all_traj', 'closest', 'kval', 'dots', 'acts', 'qdot', 'grads')}
        r = self._rollout_args(N, H, int(P.n_kernels), host['q_cur'], dummy, dummy, dummy, out)
        a.rollout = r
        qmin, qmax = self._host_vec(self.Cost.q_min), self._host_vec(self.Cost.q_max)
        for i in range(d):
            a.q_min[i], a.q_max[i] = qmin[i], qmax[i]
        a.ker_thr, a.upd_rate = float(self.ker_thr), float(self.policy_upd_rate)
        a.cost_terms, a.update_variant = self._COST_TERMS, self._UPDATE_VARIANT
        for name in ('q_cur', 'mu_tmp', 'sigma_tmp', 'alpha_tmp', 'mu_c', 'sigma_c', 'alpha_c', 'all_traj',
                     'closest_dist_all', 'kernel_val_all', 'dot_products', 'kernel_activations', 'qdot', 'cost',
                     'n_updated'):
            t = host[name]
            assert t.device.type == 'cpu' and t.is_contiguous(), name
            setattr(a, name + '_host', t.data_ptr())
        with torch.cuda.device(self._dev):
            self._upload_obstacles()
            if self._shard is not None:
                # one shard of a sample-sharded job: the library calls back between its phases and the two small
                # buffers are all-reduced over NCCL on the same stream (SURVEY 8(e)); no host synchronisation
                from .parallel import allreduce_cost_stats, allreduce_packed
                group = self._shard['group']
                stats = torch.empty(4, device=self._dev)
                packed = torch.empty(int(self._lib.dsmppi_update_packed_len(int(P.n_kernels), d)), device=self._dev)

                def exchange(_user, phase):
                    try:
                        if phase == _capi.EXCHANGE_COST_STATS:
                            allreduce_cost_stats(stats, group)
                        else:
                            allreduce_packed(packed, group)
                        return 0
                    except Exception:  # noqa: BLE001 - must not unwind through the C frame
                        import traceback
                        traceback.print_exc()
                        return 1
                hook = _capi.ExchangeFn(exchange)
                a.exchange, a.stats_dev, a.packed_dev = hook, stats.data_ptr(), packed.data_ptr()
                a.owns_sample0 = 1 if self._shard['rank'] == 0 else 0
                a.N_global = self._shard['N_global']
            _capi.check(self._lib.dsmppi_iteration_host(self._ctx, _capi.C.byref(a), self._stream()))
        return int(a.h2d_bytes), int(a.d2h_bytes)

    def update_obstacles(self, obs):
        self.obs = obs
        self.n_obs = obs.shape[0]
        return 0

    # ------------------------------------------------------------------ introspection (bench / tests)
    def launch_count(self):
        return int(self._lib.dsmppi_launch_count(self._ctx))

    def exactness_stats(self):
        """Guard band in effect (metres), the calibration error it was derived from, and how often a rollout had to be
        repeated with a larger candidate list / with every pair scored in fp32 (dsmppi_exactness_stats)."""
        r, f, g, e = _capi.C.c_int64(), _capi.C.c_int64(), _capi.C.c_float(), _capi.C.c_float()
        _capi.check(self._lib.dsmppi_exactness_stats(self._ctx, _capi.C.byref(r), _capi.C.byref(f), _capi.C.byref(g),
                                                     _capi.C.byref(e)))
        return dict(capacity_retries=r.value, exact_fallbacks=f.value, guard_band=g.value, calibration_error=e.value)

    def pass1_stats(self):
        a, b, m = _capi.C.c_int64(), _capi.C.c_int64(), _capi.C.c_int32()
        _capi.check(self._lib.dsmppi_pass1_stats(self._ctx, _capi.C.byref(a), _capi.C.byref(b), _capi.C.byref(m),
                                                 self._stream()))
        return dict(rescored_pairs=a.value, band_overflows=b.value, mode=m.value)

    def debug_pass1(self, q, mode='exact'):
        """Test hook: (n, M) masked minimum link distances of pass 1 from the fp32 or the tensor-core path."""
        code = {'exact': _capi.PASS1_EXACT_FP32, 'tc_f16': _capi.PASS1_TC_F16, 'tc_bf16': _capi.PASS1_TC_BF16}[mode]
        qd = self._d(q)
        with torch.cuda.device(self._dev):
            obs = self._upload_obstacles()
            out = torch.empty(qd.shape[0], obs.shape[0], device=self._dev)
            _capi.check(self._lib.dsmppi_debug_pass1(self._ctx, qd.data_ptr(), int(qd.shape[0]), self._ignore_mask(),
                                                     code, out.data_ptr(), self._stream()))
        return out

    def enable_kernel_timing(self, on=True):
        _capi.check(self._lib.dsmppi_enable_kernel_timing(self._ctx, 1 if on else 0))
        self._timing_on = bool(on)

    def kernel_timing_ex(self):
        """(kernel name, ms per launch, launches) of the dominant kernel in the last rollout."""
        k, ms, n = _capi.C.c_int32(), _capi.C.c_double(), _capi.C.c_int32()
        _capi.check(self._lib.dsmppi_kernel_timing_ex(self._ctx, _capi.C.byref(k), _capi.C.byref(ms), _capi.C.byref(n)))
        name = {0: 'exact_mlp_kernel', 1: 'tc_pass1_kernel', 2: 'rollout_fused_kernel', 3: 'tc_exact_kernel',
                4: 'tc_exact_kernel<whole horizon>'}[k.value]
        return dict(kernel=name, ms=ms.value, launches=n.value)

    def kernel_timing(self):
        p, pn, e, en = _capi.C.c_double(), _capi.C.c_int32(), _capi.C.c_double(), _capi.C.c_int32()
        _capi.check(self._lib.dsmppi_kernel_timing(self._ctx, _capi.C.byref(p), _capi.C.byref(pn), _capi.C.byref(e),
                                                   _capi.C.byref(en)))
        return dict(pass1_ms=p.value, pass1_launches=pn.value, exact_ms=e.value, exact_launches=en.value)
