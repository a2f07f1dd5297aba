"""ctypes binding of libdsmppi_b200.so -- exactly the declarations of include/dsmppi_b200.h.

This is the stub a maintainer of the reference would add to ds_mppi/functions/MPPI.py (INTEGRATION.md):
plain pointers and sizes, no torch types cross the boundary; torch only supplies `tensor.data_ptr()` and
the current stream handle.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DSMPPI_LIB=<path>: another build of the same library (A/B measurements of two builds on one box)
LIB_PATH = os.environ.get("DSMPPI_LIB") or os.path.join(_HERE, "libdsmppi_b200.so")

N_KERNEL_MAX = 50
MAX_DOF = 8
MAX_LINKS = 16
MAX_CLOSEST = 8
MAX_HIDDEN = 256          # widest hidden layer of the distance network
MAX_HIDDEN_LAYERS = 4

PASS1_EXACT_FP32, PASS1_TC_F16, PASS1_TC_BF16, PASS1_AUTO = 0, 1, 2, 3
SCORE_FFMA, SCORE_TC_SPLIT, SCORE_AUTO = 0, 1, 2

_fp = C.c_void_p   # device / host float pointers travel as integers from tensor.data_ptr()


DS_LINEAR_ATTRACTOR, DS_MATRIX, DS_SEDS = 0, 1, 2
DISTANCE_NN, DISTANCE_FK = 0, 1
FK_MAX_PTS = 32
COST_JOINT_LIMITS, COST_TERMINAL_FK, COST_ALL = 1, 2, 3


class Net(C.Structure):
    _fields_ = [("n_dof", C.c_int32), ("n_out", C.c_int32), ("n_point_dim", C.c_int32),
                ("n_hidden", C.c_int16), ("hidden_width", C.c_int16),
                ("W_host", _fp * 5), ("b_host", _fp * 5)]


class Modulation(C.Structure):
    _fields_ = [
        ("ds_kind", C.c_int32), ("fold_activation", C.c_int32),
        ("lvel_mid", C.c_float), ("lvel_k", C.c_float), ("dist_mid", C.c_float), ("dist_k", C.c_float),
        ("ltau_max", C.c_float), ("goal_act_thr", C.c_float), ("repulsion", C.c_float), ("reserved", C.c_float),
        ("ds_A", C.c_float * (MAX_DOF * MAX_DOF)),
    ]


class Seds(C.Structure):
    _fields_ = [("n_gaussians", C.c_int32), ("seds_thr", C.c_float), ("priors_host", _fp), ("pdf_den_host", _fp),
                ("mu_x_host", _fp), ("mu_y_host", _fp), ("sigma_inv_host", _fp), ("A_host", _fp)]


class RolloutArgs(C.Structure):
    _fields_ = [
        ("N", C.c_int32), ("H", C.c_int32), ("q_cur_is_batch", C.c_int32), ("n_kernels", C.c_int32),
        ("n_closest", C.c_int32), ("ignored_link_mask", C.c_uint32),
        ("dt", C.c_float), ("dst_thr", C.c_float), ("lin_thr", C.c_float), ("rbf_p", C.c_float),
        ("q_goal", C.c_float * MAX_DOF), ("mod", Modulation),
        ("distance_provider", C.c_int32), ("fk_n_pts", C.c_int32), ("fk_span", C.c_float * FK_MAX_PTS),
        ("q_cur_dev", _fp), ("mu_tmp_dev", _fp), ("sigma_tmp_dev", _fp), ("alpha_tmp_dev", _fp),
        ("all_traj_dev", _fp), ("closest_dist_all_dev", _fp), ("kernel_val_all_dev", _fp),
        ("dot_products_dev", _fp), ("kernel_activations_dev", _fp), ("qdot_dev", _fp),
        ("nn_grad_all_dev", _fp), ("norm_basis_dev", _fp),
    ]


class CostArgs(C.Structure):
    _fields_ = [
        ("N", C.c_int32), ("H", C.c_int32), ("terms", C.c_int32), ("reserved", C.c_int32),
        ("q_goal", C.c_float * MAX_DOF), ("q_min", C.c_float * MAX_DOF), ("q_max", C.c_float * MAX_DOF),
        ("all_traj_dev", _fp), ("closest_dist_all_dev", _fp), ("cost_dev", _fp),
    ]


class UpdateArgs(C.Structure):
    _fields_ = [
        ("N", C.c_int32), ("H", C.c_int32), ("n_kernels", C.c_int32), ("owns_sample0", C.c_int32),
        ("variant", C.c_int32), ("reserved", C.c_int32), ("N_global", C.c_int64), ("ker_thr", C.c_float), ("upd_rate", C.c_float),
        ("cost_dev", _fp), ("kernel_val_all_dev", _fp), ("kernel_activations_dev", _fp),
        ("mu_tmp_dev", _fp), ("sigma_tmp_dev", _fp), ("alpha_tmp_dev", _fp),
        ("mu_c_dev", _fp), ("sigma_c_dev", _fp), ("alpha_c_dev", _fp),
    ]


class CandidatesArgs(C.Structure):
    _fields_ = [
        ("N", C.c_int32), ("H", C.c_int32), ("n_kernels", C.c_int32), ("rbf_p", C.c_float),
        ("thr_dist", C.c_float), ("thr_kernel", C.c_float), ("thr_dot", C.c_float),
        ("all_traj_dev", _fp), ("closest_dist_all_dev", _fp), ("dot_products_dev", _fp),
        ("mu_c_dev", _fp), ("sigma_c_dev", _fp), ("out_index_dev", _fp), ("count_dev", _fp),
        ("capacity", C.c_int64),
    ]


EXCHANGE_COST_STATS, EXCHANGE_PACKED_SUMS = 0, 1
ExchangeFn = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int32)


class IterationHostArgs(C.Structure):
    _fields_ = [
        ("rollout", RolloutArgs),
        ("q_min", C.c_float * MAX_DOF), ("q_max", C.c_float * MAX_DOF),
        ("ker_thr", C.c_float), ("upd_rate", C.c_float), ("cost_terms", C.c_int32), ("update_variant", C.c_int32),
        ("q_cur_host", _fp), ("mu_tmp_host", _fp), ("sigma_tmp_host", _fp), ("alpha_tmp_host", _fp),
        ("mu_c_host", _fp), ("sigma_c_host", _fp), ("alpha_c_host", _fp),
        ("all_traj_host", _fp), ("closest_dist_all_host", _fp), ("kernel_val_all_host", _fp),
        ("dot_products_host", _fp), ("kernel_activations_host", _fp), ("qdot_host", _fp),
        ("cost_host", _fp), ("n_updated_host", _fp),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("exchange", ExchangeFn), ("exchange_user", C.c_void_p), ("stats_dev", _fp), ("packed_dev", _fp),
        ("owns_sample0", C.c_int32), ("reserved2", C.c_int32), ("N_global", C.c_int64),
    ]


class TickArgs(C.Structure):
    _fields_ = [
        ("rollout", RolloutArgs), ("n_obs", C.c_int32), ("reserved", C.c_int32),
        ("q_cur_host", _fp), ("obs_host", _fp), ("mu_tmp_host", _fp), ("sigma_tmp_host", _fp), ("alpha_tmp_host", _fp),
        ("all_traj_host", _fp), ("closest_dist_all_host", _fp), ("kernel_val_all_host", _fp),
        ("dot_products_host", _fp), ("kernel_activations_host", _fp), ("qdot_host", _fp), ("nn_grad_all_host", _fp),
        ("recaptured", C.c_int32), ("reserved2", C.c_int32),
    ]


EXPORTS = {
    # name: (restype, argtypes)
    "dsmppi_last_error": (C.c_char_p, []),
    "dsmppi_version": (C.c_int, []),
    "dsmppi_modulation_default": (None, [C.POINTER(Modulation)]),
    "dsmppi_modulation_toy": (None, [C.POINTER(Modulation)]),
    "dsmppi_ctx_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Net), _fp, C.c_int32, C.c_int32]),
    "dsmppi_ctx_destroy": (C.c_int, [C.c_void_p]),
    "dsmppi_set_pass1_mode": (C.c_int, [C.c_void_p, C.c_int32, C.c_float]),
    "dsmppi_set_score_mode": (C.c_int, [C.c_void_p, C.c_int32]),
    "dsmppi_set_whole_horizon": (C.c_int, [C.c_void_p, C.c_int32]),
    "dsmppi_set_seds": (C.c_int, [C.c_void_p, C.POINTER(Seds), C.c_void_p]),
    "dsmppi_set_obstacles": (C.c_int, [C.c_void_p, _fp, C.c_int32, C.c_void_p]),
    "dsmppi_set_obstacles_host": (C.c_int, [C.c_void_p, _fp, C.c_int32, C.c_void_p]),
    "dsmppi_rollout": (C.c_int, [C.c_void_p, C.POINTER(RolloutArgs), C.c_void_p]),
    "dsmppi_distance_grad": (C.c_int, [C.c_void_p, _fp, C.c_int32, C.c_int32, C.c_uint32, _fp, _fp, C.c_void_p]),
    "dsmppi_distance_grad_fk": (C.c_int, [C.c_void_p, _fp, C.c_int32, C.c_int32, _fp, _fp, _fp, _fp, C.c_void_p]),
    "dsmppi_debug_pass1": (C.c_int, [C.c_void_p, _fp, C.c_int32, C.c_uint32, C.c_int32, _fp, C.c_void_p]),
    "dsmppi_norm_basis": (C.c_int, [C.c_void_p, _fp, C.c_int64, _fp, C.c_void_p]),
    "dsmppi_cost": (C.c_int, [C.c_void_p, C.POINTER(CostArgs), C.c_void_p]),
    "dsmppi_kernel_candidates": (C.c_int, [C.c_void_p, C.POINTER(CandidatesArgs), C.c_void_p]),
    "dsmppi_update_packed_len": (C.c_int32, [C.c_int32, C.c_int32]),
    "dsmppi_update_cost_stats": (C.c_int, [C.c_void_p, _fp, C.c_int32, _fp, C.c_void_p]),
    "dsmppi_update_partial": (C.c_int, [C.c_void_p, C.POINTER(UpdateArgs), _fp, _fp, C.c_void_p]),
    "dsmppi_update_finalize": (C.c_int, [C.c_void_p, C.POINTER(UpdateArgs), _fp, _fp, C.c_void_p]),
    "dsmppi_iteration_host": (C.c_int, [C.c_void_p, C.POINTER(IterationHostArgs), C.c_void_p]),
    "dsmppi_tick": (C.c_int, [C.c_void_p, C.POINTER(TickArgs), C.c_void_p]),
    "dsmppi_launch_count": (C.c_int64, [C.c_void_p]),
    "dsmppi_pass1_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                     C.c_void_p]),
    "dsmppi_exactness_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float),
                                         C.POINTER(C.c_float)]),
    "dsmppi_score_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                     C.c_void_p]),
    "dsmppi_enable_kernel_timing": (C.c_int, [C.c_void_p, C.c_int32]),
    "dsmppi_kernel_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32),
                                       C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "dsmppi_kernel_timing_ex": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                          C.POINTER(C.c_int32)]),
}

_lib = None


def load():
    """Loads the shared library (no compute, no GPU needed) and types every export."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m optimalmodulationds_b200.build` "
            "(there is no CPU or PyTorch fallback for the MPPI rollout)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)      # AttributeError here == the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().dsmppi_last_error()
        raise RuntimeError("libdsmppi_b200: " + (msg.decode() if msg else f"error {status}"))
