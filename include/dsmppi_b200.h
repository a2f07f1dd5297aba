/*
 * dsmppi_b200.h -- C ABI of the B200-native ds_mppi MPPI rollout library (libdsmppi_b200.so).
 *
 * Drop-in boundary for ONE hot path of epfl-lasa/OptimalModulationDS: the MPPI rollout over N sampled
 * policies x horizon H, its cost and its policy update.  The reference has no FFI (it is pure
 * Python/PyTorch); each entry point below replaces a METHOD of the reference's Python objects, cited as
 * file:line relative to /root/reference/python_scripts/ds_mppi/functions/.  The reference-side binding
 * (a ctypes stub inside MPPI.py) is shown in INTEGRATION.md and implemented in
 * optimalmodulationds_b200/_capi.py.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success, non-zero on error, and
 *     dsmppi_last_error() returns the message of the calling thread's last failure;
 *   - `*_dev` pointers are DEVICE pointers owned by the caller (torch tensors), fp32, contiguous,
 *     row-major; `*_host` pointers are host pointers; the library owns only the opaque context and the
 *     scratch workspace inside it;
 *   - all work is enqueued on the caller's `stream` (a cudaStream_t passed as void*); no call
 *     synchronises the device except the `_host` variants, which must hand back host results;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef DSMPPI_B200_H
#define DSMPPI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSMPPI_N_KERNEL_MAX 50   /* policy.py:18 */
#define DSMPPI_MAX_DOF 8
#define DSMPPI_MAX_LINKS 16      /* network output channels O (<= 16) */
#define DSMPPI_MAX_CLOSEST 8     /* n_closest_obs K (<= 8) */
#define DSMPPI_HIDDEN 256        /* width of the shipped distance MLP, and the largest supported */
#define DSMPPI_MAX_HIDDEN_LAYERS 4  /* hidden layers of the shipped distance MLP, and the most supported */

typedef struct dsmppi_ctx dsmppi_ctx;

/* Network weights as torch stores them: W[l] is (out, in) row-major (mlp_learn/sdf/network_macros_mod.py
 * 137-146 with skips=[]: 3(d+P) -> W -> ... -> W -> O with L hidden layers of one width W, ReLU between; the shipped
 * networks are 256 x 4).  W_host[0..L-1] / b_host[0..L-1] are the hidden layers ((W, 3(d+P)), then (W, W)) and
 * W_host[L] / b_host[L] the output layer (O, W); entries past L are ignored.  HOST pointers. */
typedef struct {
  int32_t n_dof;                 /* d  */
  int32_t n_out;                 /* O  */
  int32_t n_point_dim;           /* P: obstacle coordinates fed to the network (in_channels = d + P); 3 for every
                                  * robot net, 2 for the planar "toy" net (standaloneToy2d.py:30); 0 means 3      */
  int16_t n_hidden;              /* L: hidden layers, 1..4; 0 means 4                                            */
  int16_t hidden_width;          /* W: width of every hidden layer, 1..256; 0 means 256                          */
  const float* W_host[5];
  const float* b_host[5];
} dsmppi_net;

/* Constants of the modulation law.  The reference compiles two sets into its sources: MPPI.py:132-155,194,216
 * (every robot of the live scripts) and MPPI_toy.py:89,114-133,176-180,199 (the 2-D point "toy").
 * dsmppi_modulation_default / dsmppi_modulation_toy fill them; sigmoid(x; y0, y1, x0, x1, k) of MPPI.py:352-353 is
 * passed as its midpoint (x0 + x1) / 2 and slope k. */
enum {
  DSMPPI_DS_LINEAR_ATTRACTOR = 0,  /* LinDS.get_velocity (LinDS.py:11-21): unit speed outside lin_thr              */
  DSMPPI_DS_MATRIX = 1,            /* v = (q - q_goal) @ A (MPPI_toy.py:89), not normalised                         */
  DSMPPI_DS_SEDS = 2               /* Gaussian-mixture regression, SEDS.get_velocity (SEDS.py:61-76); parameters
                                    * uploaded beforehand with dsmppi_set_seds                                    */
};
typedef struct {
  int32_t ds_kind;               /* DSMPPI_DS_*                                                                  */
  int32_t fold_activation;       /* 1: kernel_val_all[:, t, :nk] *= activation (MPPI_toy.py:178-179)             */
  float lvel_mid, lvel_k;        /* l_vel = sigmoid(dot; 0, 1, ..): (-0.5, 10) | toy (-0.1, 100)                  */
  float dist_mid, dist_k;        /* l_n, l_tau over the distance: (0.05, 100) | toy (0.25, 30)                    */
  float ltau_max;                /* 5 | toy 3                                                                    */
  float goal_act_thr;            /* goal activation below this is zeroed: 0.5 | toy 0.3                          */
  float repulsion;               /* collision case: m = 0.1 m + repulsion |v| e0: 0.1 | toy 0.05                 */
  float reserved;
  float ds_A[DSMPPI_MAX_DOF * DSMPPI_MAX_DOF];   /* DSMPPI_DS_MATRIX: A[a][c] at a * DSMPPI_MAX_DOF + c           */
} dsmppi_modulation;

/* Pass-1 precision: how the all-pairs forward pass that ranks obstacles (MPPI.py:231-253) is evaluated. */
enum {
  DSMPPI_PASS1_EXACT_FP32 = 0,   /* fp32 FFMA on every (sample, obstacle) pair                         */
  DSMPPI_PASS1_TC_F16 = 1,       /* tcgen05 fp16 x fp16 -> fp32 prefilter + fp32 re-score of the band   */
  DSMPPI_PASS1_TC_BF16 = 2,      /* same with bf16 operands                                             */
  DSMPPI_PASS1_AUTO = 3          /* TC_F16 when M >= 64, else EXACT                                     */
};

/* Scoring arithmetic: how the rows that produce OUTPUTS (ranking keys, distances, gradients) are evaluated. */
enum {
  DSMPPI_SCORE_FFMA = 0,         /* IEEE fp32 FFMA on the CUDA cores (exact_mlp.cu): the strict mode              */
  DSMPPI_SCORE_TC_SPLIT = 1,     /* tcgen05: operands split into two fp16 halves (22 bits), three MMAs per
                                  * product sum, fp32 accumulation with truncation compensation (tc_exact.cu):
                                  * rms error 2-3e-7 of the rms distance like FFMA; rows whose activations leave
                                  * the fp16 range are re-scored by the FFMA kernel                              */
  DSMPPI_SCORE_AUTO = 2          /* TC_SPLIT whenever the network fits its tiles (3(d+P) <= 32, O <= 16)           */
};

/* Where the per-step distance and its joint gradient come from (MPPI.py:113-115). */
enum {
  DSMPPI_DISTANCE_NN = 0,        /* learned network, distance_repulsion_nn (MPPI.py:227-282) -- the live path     */
  DSMPPI_DISTANCE_FK = 1         /* forward kinematics + sphere distances, distance_repulsion_fk (MPPI.py:306-313) */
};
#define DSMPPI_FK_MAX_PTS 32     /* sample points per link (the reference uses 10, MPPI.py:307) */

typedef struct {
  /* state / problem */
  int32_t N;                     /* samples in this call (<= capacity)                                  */
  int32_t H;                     /* horizon dt_H                                                        */
  int32_t q_cur_is_batch;        /* 0: q_cur_dev is (d,), 1: (N, d)   (MPPI.py:99 broadcast)            */
  int32_t n_kernels;             /* Policy.n_kernels                                                    */
  int32_t n_closest;             /* n_closest_obs K                                                     */
  uint32_t ignored_link_mask;    /* bit l set <=> l in MPPI.ignored_links (MPPI.py:62,241)              */
  float dt;                      /* MPPI.dt                                                             */
  float dst_thr;                 /* MPPI.dst_thr (MPPI.py:117)                                          */
  float lin_thr;                 /* LinDS.lin_thr (LinDS.py:9)                                          */
  float rbf_p;                   /* Policy.p (policy.py:41,186-199)                                     */
  float q_goal[DSMPPI_MAX_DOF];  /* DS.q_goal == MPPI.qf                                                */
  dsmppi_modulation mod;         /* constants of the modulation law (fill with dsmppi_modulation_default)      */
  int32_t distance_provider;     /* DSMPPI_DISTANCE_*                                                           */
  int32_t fk_n_pts;              /* DSMPPI_DISTANCE_FK: points per link (1..32)                                 */
  float fk_span[DSMPPI_FK_MAX_PTS];  /* fractions along a link, torch.linspace(0.01, 1, fk_n_pts) (fk_num.py:79)   */
  /* inputs (device) */
  const float* q_cur_dev;
  const float* mu_tmp_dev;       /* (N, 50, d)  Policy.mu_tmp                                           */
  const float* sigma_tmp_dev;    /* (N, 50)     Policy.sigma_tmp                                        */
  const float* alpha_tmp_dev;    /* (N, 50, d)  Policy.alpha_tmp                                        */
  /* outputs (device) -- the attributes MPPI.propagate fills (MPPI.py:40-51, 224) */
  float* all_traj_dev;           /* (N, H, d)                                                           */
  float* closest_dist_all_dev;   /* (N, H)                                                              */
  float* kernel_val_all_dev;     /* (N, H, 50); only columns [0, n_kernels) are written                 */
  float* dot_products_dev;       /* (N, H)                                                              */
  float* kernel_activations_dev; /* (N, H)                                                              */
  float* qdot_dev;               /* (N, d)                                                              */
  float* nn_grad_all_dev;        /* (N, H, d) blended distance gradient per state-step (basis source)   */
  float* norm_basis_dev;         /* (N, H, d, d) or NULL (lazy: see dsmppi_norm_basis)                  */
} dsmppi_rollout_args;

enum {
  DSMPPI_COST_JOINT_LIMITS = 1,  /* cost.py:16,36-39                                                            */
  DSMPPI_COST_TERMINAL_FK = 2,   /* cost.py:19,27-31                                                            */
  DSMPPI_COST_ALL = 3            /* cost.py:13-21; cost_toy.py:13-19 keeps goal + collision + stagnation only: 0 */
};
typedef struct {
  int32_t N, H;
  int32_t terms;                 /* DSMPPI_COST_* bit mask of the optional terms                                */
  int32_t reserved;
  float q_goal[DSMPPI_MAX_DOF];
  float q_min[DSMPPI_MAX_DOF];   /* Cost.q_min / q_max (cost.py:10-11)                                  */
  float q_max[DSMPPI_MAX_DOF];
  const float* all_traj_dev;         /* (N, H, d) */
  const float* closest_dist_all_dev; /* (N, H)    */
  float* cost_dev;                   /* (N,)      */
} dsmppi_cost_args;

typedef struct {
  int32_t N, H;
  int32_t n_kernels;
  int32_t owns_sample0;          /* 1 when this shard holds global sample 0 (the noise-free rollout)    */
  int32_t variant;               /* 0: MPPI.py:335-342 (max_t kernel_val * activation, and the sample-0 base
                                  * mask); 1: MPPI_toy.py:318-321 (max_t kernel_val, no base mask)            */
  int32_t reserved;
  int64_t N_global;              /* total samples over all shards (for the means)                       */
  float ker_thr;                 /* MPPI.ker_thr                                                        */
  float upd_rate;                /* MPPI.policy_upd_rate (MPPI.py:58,344)                               */
  const float* cost_dev;         /* (N,)                                                                */
  const float* kernel_val_all_dev;     /* (N, H, 50)                                                    */
  const float* kernel_activations_dev; /* (N, H)                                                        */
  const float* mu_tmp_dev;       /* (N, 50, d)                                                          */
  const float* sigma_tmp_dev;    /* (N, 50)                                                             */
  const float* alpha_tmp_dev;    /* (N, 50, d)                                                          */
  float* mu_c_dev;               /* (50, d)  updated in place by _finalize                              */
  float* sigma_c_dev;            /* (50,)                                                               */
  float* alpha_c_dev;            /* (50, d)                                                             */
} dsmppi_update_args;

const char* dsmppi_last_error(void);
int dsmppi_version(void);
void dsmppi_modulation_default(dsmppi_modulation* out);   /* MPPI.py constants, LinDS nominal dynamics   */
void dsmppi_modulation_toy(dsmppi_modulation* out);       /* MPPI_toy.py constants, matrix DS with A = -I */

/* MPPI.__init__ (MPPI.py:22-73): packs the network (fp32 both orientations + fp16/bf16 UMMA smem images),
 * the DH table (dh_params (d+1, 4) = [d, theta, a, alpha], HOST) and sizes the workspace for
 * `capacity` samples.  `device` is the CUDA ordinal.  A network narrower or shallower than 256 x 4 is embedded in
 * that shape (zero rows / columns for the missing features, identity layers for the missing depth), which changes no
 * result: the FFMA scoring kernels run the network's own width and depth, the tensor-core kernels the embedded one.
 * A shape outside 1 <= L <= 4, 1 <= W <= 256 returns 2. */
int dsmppi_ctx_create(dsmppi_ctx** out, const dsmppi_net* net, const float* dh_params_host,
                      int32_t capacity, int32_t device);
int dsmppi_ctx_destroy(dsmppi_ctx* ctx);
/* guard_band > 0 fixes the prefilter's guard band (metres); 0 = calibrate it for the network (dsmppi_exactness_stats).
 * Environment, read by dsmppi_ctx_create: DSMPPI_PASS1_ACC=f32 makes the fp16 prefilter accumulate its hidden layers
 * in fp32 (default: fp16 accumulators -- twice the prefilter error, a wider calibrated band, the same results bit for
 * bit, 8 % less time per prefilter launch); DSMPPI_HALF_TILES=0 keeps the whole-horizon kernel on 128-row tiles;
 * DSMPPI_DISABLE_TC=1 builds no tensor-core images (every mode resolves to the FFMA kernels). */
int dsmppi_set_pass1_mode(dsmppi_ctx* ctx, int32_t mode, float guard_band);
int dsmppi_set_score_mode(dsmppi_ctx* ctx, int32_t mode);     /* DSMPPI_SCORE_*; default AUTO */
/* Small obstacle sets scored in fp32 (M <= 16, or M <= 32 with a latency-bound batch) are rolled out over the whole
 * horizon by ONE launch (rollout_fused_kernel); on = 0 forces the per-step launch sequence (tests compare both). */
int dsmppi_set_whole_horizon(dsmppi_ctx* ctx, int32_t on);

/* MPPI.update_obstacles (MPPI.py:347-350) and the obs argument of __init__: (M, P + 1) = [x, y, z, r], or
 * [x, y, r] for a network created with n_point_dim = 2. */
int dsmppi_set_obstacles(dsmppi_ctx* ctx, const float* obs_dev, int32_t M, void* stream);
int dsmppi_set_obstacles_host(dsmppi_ctx* ctx, const float* obs_host, int32_t M, void* stream);

/* Parameters of a SEDS nominal DS (ds_mppi/functions/SEDS.py:9-27), already in the form its GMR uses (:36-59):
 * for Gaussian j: prior, pdf_den = sqrt(2 pi^d det_j + 1e-100) (the denominator of gaussPDF, :28-34), the input and
 * output means Mu[:d, j] / Mu[d:, j], Sigma_xx^-1 (d, d) and A_j = Sigma_yx Sigma_xx^-1 (d, d), all row-major HOST
 * arrays with the Gaussian index leading.  dsmppi_rollout with mod.ds_kind = DSMPPI_DS_SEDS uses the last upload;
 * lin_thr travels in dsmppi_rollout_args.lin_thr. */
typedef struct {
  int32_t n_gaussians;           /* G <= 32                                                              */
  float seds_thr;                /* SEDS.seds_thr: weaker GMR outputs fall back to the linear DS (:72-75)  */
  const float* priors_host;      /* (G,)      */
  const float* pdf_den_host;     /* (G,)      */
  const float* mu_x_host;        /* (G, d)    */
  const float* mu_y_host;        /* (G, d)    */
  const float* sigma_inv_host;   /* (G, d, d) */
  const float* A_host;           /* (G, d, d) */
} dsmppi_seds;
int dsmppi_set_seds(dsmppi_ctx* ctx, const dsmppi_seds* seds, void* stream);

/* MPPI.propagate (MPPI.py:97-224): the H-step rollout of all N samples. */
int dsmppi_rollout(dsmppi_ctx* ctx, const dsmppi_rollout_args* args, void* stream);

/* MPPI.distance_repulsion_nn (MPPI.py:227-282): q (n, d) -> distance (n,), nn_grad (n, d). */
int dsmppi_distance_grad(dsmppi_ctx* ctx, const float* q_dev, int32_t n, int32_t n_closest,
                         uint32_t ignored_link_mask, float* distance_dev, float* nn_grad_dev, void* stream);

/* MPPI.distance_repulsion_fk (MPPI.py:306-313): true distance between the robot's links (fk_n_pts sample points per
 * link of the modified-DH chain, fk_num.py:78-89) and the obstacle spheres, minimised over (link, obstacle, point)
 * (fk_num.py:142-160), and its analytic gradient w.r.t. the joints: q (n, d) -> distance (n,), grad (n, d).
 * span_host: the fk_n_pts fractions along a link (torch.linspace(0.01, 1, n_pts)) or NULL for the same ramp computed
 * internally; closest_idx_dev: optional (n, 3) = [obstacle, link, point] of the minimum. */
int dsmppi_distance_grad_fk(dsmppi_ctx* ctx, const float* q_dev, int32_t n, int32_t fk_n_pts, const float* span_host,
                            float* distance_dev, float* grad_dev, int32_t* closest_idx_dev, void* stream);

/* Test hook: the per-pair masked minimum link distance of pass 1 (MPPI.py:235-243), (n, M) row-major, from
 * the fp32 path (mode = DSMPPI_PASS1_EXACT_FP32) or the tensor-core prefilter (TC_F16 / TC_BF16).  Any other mode,
 * AUTO included, returns 2. */
int dsmppi_debug_pass1(dsmppi_ctx* ctx, const float* q_dev, int32_t n, uint32_t ignored_link_mask, int32_t mode,
                       float* out_dev, void* stream);

/* The Householder basis the reference stores in MPPI.norm_basis (MPPI.py:122-127), from the blended
 * gradients: grad (n, d) -> basis (n, d, d). */
int dsmppi_norm_basis(dsmppi_ctx* ctx, const float* grad_dev, int64_t n, float* basis_dev, void* stream);

/* MPPI.get_cost -> Cost.evaluate_costs (MPPI.py:315-317, cost.py:13-46). */
int dsmppi_cost(dsmppi_ctx* ctx, const dsmppi_cost_args* args, void* stream);

/* MPPI.shift_policy_means -> TensorPolicyMPPI.update_policy (MPPI.py:331-345, policy.py:88-113), split in
 * the three phases a sample-sharded job needs (SURVEY 8(e)):
 *   cost_stats : stats_dev[0..3] = { sum cost, N, min cost, argmin (as float) }
 *                                                  -> allreduce #1: SUM of stats_dev[0..1] (beta = sum / N / 50)
 *   partial    : packed_dev[L], L = dsmppi_update_packed_len(nk, d)                      -> allreduce #2: SUM
 *   finalize   : EMA of mu_c / sigma_c / alpha_c, n_updated_dev[0] = number of kernels updated.
 * On one GPU call them back to back.  Entries [2..3] (minimum cost and its local index) are per shard; get_qdot
 * reduces them separately when a caller asks for the best sample. */
int32_t dsmppi_update_packed_len(int32_t n_kernels, int32_t n_dof);
int dsmppi_update_cost_stats(dsmppi_ctx* ctx, const float* cost_dev, int32_t N, float* stats_dev, void* stream);
int dsmppi_update_partial(dsmppi_ctx* ctx, const dsmppi_update_args* args, const float* stats_dev,
                          float* packed_dev, void* stream);
int dsmppi_update_finalize(dsmppi_ctx* ctx, const dsmppi_update_args* args, const float* packed_dev,
                           int32_t* n_updated_dev, void* stream);

/* TensorPolicyMPPI.check_traj_for_kernels (policy.py:153-175): state-steps that are close to an obstacle
 * (closest_dist < thr_dist), moving into it (dot < thr_dot) and not covered by any policy kernel
 * (max_k exp(-sigma_k ||q - mu_k||_p^2) < thr_kernel; always true with no kernels).  Appends the flat index
 * i*H + h of every such state-step to out_index_dev (UNORDERED, at most `capacity` entries) and stores their
 * total number in count_dev[0] (which may exceed capacity: the caller re-runs with a larger buffer). */
typedef struct {
  int32_t N, H;
  int32_t n_kernels;
  float rbf_p;                   /* Policy.p                                                            */
  float thr_dist, thr_kernel, thr_dot;
  const float* all_traj_dev;         /* (N, H, d) */
  const float* closest_dist_all_dev; /* (N, H)    */
  const float* dot_products_dev;     /* (N, H)    */
  const float* mu_c_dev;             /* (50, d)   */
  const float* sigma_c_dev;          /* (50,)     */
  int32_t* out_index_dev;            /* (capacity,) */
  int32_t* count_dev;                /* (1,) zeroed by the call */
  int64_t capacity;
} dsmppi_candidates_args;
int dsmppi_kernel_candidates(dsmppi_ctx* ctx, const dsmppi_candidates_args* args, void* stream);

/* One whole MPPI iteration with HOST buffers (what a CPU-tensor caller of the reference API pays):
 * H2D of q_cur / sampled policy, rollout, cost, policy update, D2H of every output.  Host pointers may be
 * pageable or pinned.  Synchronises `stream` before returning.
 * A batch of more than 2 x 131072 samples is pipelined in sample chunks over two internal copy streams (H2D of chunk
 * k+1 and D2H of chunk k-1 under the rollout + cost of chunk k on `stream`; the policy update follows the last
 * chunk); results are bit-identical to the single pass.  Environment: DSMPPI_HOST_CHUNK=<samples> overrides the
 * chunk size, 0 disables the pipeline. */
enum { DSMPPI_EXCHANGE_COST_STATS = 0, DSMPPI_EXCHANGE_PACKED_SUMS = 1 };
typedef int (*dsmppi_exchange_fn)(void* user, int32_t phase);
typedef struct {
  dsmppi_rollout_args rollout;   /* the *_dev fields are ignored; shapes and scalars are used            */
  float q_min[DSMPPI_MAX_DOF];
  float q_max[DSMPPI_MAX_DOF];
  float ker_thr, upd_rate;
  int32_t cost_terms;            /* dsmppi_cost_args.terms                                              */
  int32_t update_variant;        /* dsmppi_update_args.variant                                          */
  const float* q_cur_host;       /* (d,) or (N, d)                                                      */
  const float* mu_tmp_host;      /* (N, 50, d) */
  const float* sigma_tmp_host;   /* (N, 50)    */
  const float* alpha_tmp_host;   /* (N, 50, d) */
  float* mu_c_host;              /* (50, d) in/out */
  float* sigma_c_host;           /* (50,)   in/out */
  float* alpha_c_host;           /* (50, d) in/out */
  float* all_traj_host;          /* (N, H, d)  */
  float* closest_dist_all_host;  /* (N, H)     */
  float* kernel_val_all_host;    /* (N, H, 50) */
  float* dot_products_host;      /* (N, H)     */
  float* kernel_activations_host;/* (N, H)     */
  float* qdot_host;              /* (N, d)     */
  float* cost_host;              /* (N,)       */
  int32_t* n_updated_host;       /* (1,)       */
  int64_t h2d_bytes, d2h_bytes;  /* filled in: bytes moved by this call                                 */
  /* Sample-sharded job (SURVEY 8(e)): when `exchange` is set this call runs ONE SHARD of the iteration and calls
   * exchange(exchange_user, phase) twice, after it has enqueued the producer of the buffer named by `phase` on
   * `stream`; the hook all-reduces (SUM) that caller-owned device buffer over the ranks on the same stream
   * (torch.distributed / NCCL) and returns 0.  NULL = single-GPU iteration (the fields below are ignored). */
  dsmppi_exchange_fn exchange;
  void* exchange_user;
  float* stats_dev;              /* (4,)  DSMPPI_EXCHANGE_COST_STATS: SUM over ranks of stats_dev[0..1]   */
  float* packed_dev;             /* (dsmppi_update_packed_len,)  DSMPPI_EXCHANGE_PACKED_SUMS: SUM of all  */
  int32_t owns_sample0;          /* 1 on the rank holding global sample 0                                 */
  int32_t reserved2;
  int64_t N_global;              /* samples over all ranks                                                */
} dsmppi_iteration_host_args;
int dsmppi_iteration_host(dsmppi_ctx* ctx, dsmppi_iteration_host_args* args, void* stream);

/* One control tick with HOST buffers as ONE replayed CUDA graph (frankaIntegrator.py:101-121: update_obstacles,
 * propagate with one sample and two steps, every tick; frankaPlanner.py's 40 x 10 rollouts fit too).  At such sizes the
 * rollout is a single ~0.1 ms launch and the tick is spent around it, so the whole sequence -- H2D of the state, the
 * obstacles and the FULL (N, 50, ..) policy rows from one pinned staging block, dsmppi_set_obstacles, dsmppi_rollout,
 * D2H of every output into one pinned block -- is captured once per parameter set and then costs one cudaGraphLaunch
 * and one synchronisation.  Kernel arguments are baked into a graph: it is re-captured when any scalar of `rollout`,
 * N, H or n_obs differs from the captured one.  Only for obstacle sets that take the dense fp32 scoring path (the
 * prefilter path ends with a host-side exactness verdict): returns an error otherwise, as it does on a SEDS nominal DS.
 * Runs on an internal stream ordered after `stream`; synchronises before returning. */
typedef struct {
  dsmppi_rollout_args rollout;   /* the *_dev fields are ignored; shapes and scalars are used            */
  int32_t n_obs;                 /* M                                                                    */
  int32_t reserved;
  const float* q_cur_host;       /* (d,) or (N, d)                                                       */
  const float* obs_host;         /* (M, P + 1)                                                           */
  const float* mu_tmp_host;      /* (N, 50, d) or NULL when n_kernels == 0                               */
  const float* sigma_tmp_host;   /* (N, 50)                                                              */
  const float* alpha_tmp_host;   /* (N, 50, d)                                                           */
  float* all_traj_host;          /* (N, H, d)                                                            */
  float* closest_dist_all_host;  /* (N, H)                                                               */
  float* kernel_val_all_host;    /* (N, H, 50): dead columns are written as zeros                        */
  float* dot_products_host;      /* (N, H)                                                               */
  float* kernel_activations_host;/* (N, H)                                                               */
  float* qdot_host;              /* (N, d)                                                               */
  float* nn_grad_all_host;       /* (N, H, d)                                                            */
  int32_t recaptured;            /* filled in: 1 when this call had to (re)capture the graph             */
  int32_t reserved2;
} dsmppi_tick_args;
int dsmppi_tick(dsmppi_ctx* ctx, dsmppi_tick_args* args, void* stream);

/* Introspection used by bench.py / tests: launches issued by the library since ctx creation, pass-1
 * statistics of the last rollout (re-scored pairs; `band_overflows` = sample-steps whose guard band held more than
 * 16 obstacles -- informational: they all get a row), and the resolved pass-1 mode. */
int64_t dsmppi_launch_count(const dsmppi_ctx* ctx);
int dsmppi_pass1_stats(dsmppi_ctx* ctx, int64_t* rescored_pairs, int64_t* band_overflows, int32_t* mode,
                       void* stream);
/* The prefilter path is exact by construction: EVERY obstacle within the guard band of the K-th smallest approximate
 * distance is re-scored in fp32; when a step's candidates do not fit the shared row list the rollout is repeated with
 * a larger list (`capacity_retries`), past 2^27 rows with every pair scored in fp32 (`exact_fallbacks`) -- never
 * truncated; the same repeat in fp32 happens when the prefilter produced inf / NaN for any pair (activations beyond the
 * fp16 range).  `guard_band` is the band in effect (metres): the caller's (dsmppi_set_pass1_mode) or the one
 * calibrated for this network and obstacle set = 3 x `calibration_error`, the largest |prefilter - fp32 scoring|
 * over 256 random joint vectors + the first states of the calling batch x every obstacle. */
int dsmppi_exactness_stats(dsmppi_ctx* ctx, int64_t* capacity_retries, int64_t* exact_fallbacks, float* guard_band,
                           float* calibration_error);
/* Scoring arithmetic in effect (DSMPPI_SCORE_FFMA / _TC_SPLIT) and, for the tensor-core path, how many rows left the
 * fp16 range of its split operands and were re-scored by the FFMA kernel since the context was created
 * (`dropped_rows` > 0 means the re-scoring list overflowed: results of those rows are saturated, not exact). */
int dsmppi_score_stats(dsmppi_ctx* ctx, int32_t* mode, int64_t* range_fixup_rows, int64_t* dropped_rows, void* stream);
/* Average device time (ms) of the dominant kernel over its launches in the last rollout; requires
 * dsmppi_enable_kernel_timing(ctx, 1) beforehand (CUDA events on the launching stream). */
int dsmppi_enable_kernel_timing(dsmppi_ctx* ctx, int32_t on);
int dsmppi_kernel_timing(dsmppi_ctx* ctx, double* pass1_ms_per_launch, int32_t* pass1_launches,
                         double* exact_ms_per_launch, int32_t* exact_launches);
/* Same, naming the kernel: kind 0 = exact_mlp_kernel (FFMA scoring, one launch per step), 1 = tc_pass1_kernel,
 * 2 = rollout_fused_kernel (FFMA, one launch per rollout block: all H steps), 3 = tc_exact_kernel (tensor-core
 * scoring, one launch per step), 4 = tc_exact_kernel in whole-horizon mode (one launch per rollout block). */
int dsmppi_kernel_timing_ex(dsmppi_ctx* ctx, int32_t* kind, double* ms_per_launch, int32_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* DSMPPI_B200_H */
