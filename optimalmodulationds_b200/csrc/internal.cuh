// Internal declarations shared by the translation units of libdsmppi_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "dsmppi_b200.h"

#define HID DSMPPI_HIDDEN
#define MAXL DSMPPI_MAX_HIDDEN_LAYERS
#define MAXD DSMPPI_MAX_DOF
#define MAXO DSMPPI_MAX_LINKS
#define MAXK DSMPPI_MAX_CLOSEST
#define NKMAX DSMPPI_N_KERNEL_MAX
#define CAND_MAX 16            // candidate rows budgeted per sample by the tensor-core prefilter (the band usually
                               // holds K + 1; a sample may take more while the shared row list has room, and a list
                               // that runs out of room makes dsmppi_rollout grow it and run again -- never truncation)
#define N_COUNTERS 16

void dsmppi_set_error(const std::string& msg);

#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      dsmppi_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" __FILE__ + \
                       ":" + std::to_string(__LINE__) + ")");                              \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

#define REQUIRE(cond, msg)                                    \
  do {                                                        \
    if (!(cond)) {                                            \
      dsmppi_set_error(std::string(msg) + " [" #cond "]");    \
      return 2;                                               \
    }                                                         \
  } while (0)

// Device-side view of the distance network (fp32).
struct NetDev {
  int d;        // joints
  int nin;      // d + 3
  int nenc;     // 3 * nin
  int O;        // links
  float scale;  // 0.01 when O == 9 (centimetres -> metres, MPPI.py:236-237), else 1
  int nh;       // hidden layers of the caller's network (1..4); the arrays below hold it embedded in 256 x 4
  int width;    // width of its hidden layers (1..256)
  const float* Wf[4];   // layers 0..3, forward orientation [in][256]
  const float* Wb[4];   // layers 0..3, torch orientation  [256][in]
  const float* W4;      // output layer, torch orientation [O][256]
  const float* b[5];
};

// How a kernel maps a row index to a (sample, obstacle) pair.
enum { ROWS_DENSE = 0, ROWS_SELECTED = 1, ROWS_LIST = 2 };
struct RowSrc {
  int mode;
  int M;                  // obstacles
  int K;                  // ROWS_SELECTED: pairs per sample
  int n_rows;             // host-known row count (upper bound when n_rows_dev != nullptr)
  const int* n_rows_dev;  // ROWS_LIST: device row counter
  const int* sel;         // ROWS_SELECTED: (n, K) obstacle index
  const int* row_sample;  // ROWS_LIST
  const int* row_obs;     // ROWS_LIST
  const int* out_row;     // optional: row r writes its outputs at index out_row[r] (re-scoring of flagged rows)
};

struct DhTable { float v[MAXD + 1][4]; };   // rows [d, theta, a, alpha]

struct dsmppi_ctx {
  int device = 0;
  int d = 0, O = 0, nin = 0, nenc = 0;
  int P = 3;                          // obstacle coordinates fed to the network (nin = d + P)
  int capacity = 0;
  int M = 0;
  int pass1_mode = DSMPPI_PASS1_AUTO;
  float guard_band = 0.f;             // caller-set guard band (dsmppi_set_pass1_mode); 0 = calibrated per network
  float band_cal[2] = {0.f, 0.f};     // calibrated guard band of the fp16 / bf16 prefilter (capi.cu: calibrate_band)
  int band_cal_M[2] = {0, 0};         // obstacle count the calibration ran on (re-run when it changes)
  float band_cal_err[2] = {0.f, 0.f}; // largest |prefilter - fp32 scoring| seen by the calibration
  NetDev net{};
  DhTable dh{};
  float* weights_blob = nullptr;      // all fp32 weights
  void* tc_blob = nullptr;            // tensor-core operand images (tc_pass1.cu)
  size_t tc_blob_bytes = 0;
  void* tcx_blob = nullptr;           // split-fp16 weight images of the tensor-core scoring kernel (tc_exact.cu)
  int* fix_list = nullptr; size_t fix_cap = 0;   // rows whose activations left the fp16 range: (sample, obs, out row)
  int fix_parity = 0;                 // which of counters[4..5] the next tc_exact launch appends to
  int score_mode = DSMPPI_SCORE_AUTO; // which kernel scores / differentiates rows in fp32 accuracy
  // obstacles
  float* obs = nullptr; int obs_cap = 0;   // always (M, 4) = [x, y, z, r] on the device (z = 0 when P == 2)
  float* obs_raw = nullptr; int obs_raw_cap = 0;   // P == 2: the caller's (M, 3) rows before repacking
  void* obs_enc = nullptr; size_t obs_enc_cap = 0;   // tensor path: per-obstacle packed encodings
  // SEDS nominal DS: [priors G | pdf_den G | mu_x G*d | mu_y G*d | sigma_inv G*d*d | A G*d*d]
  float* seds = nullptr; int seds_G = 0; float seds_thr = 0.f;
  // workspace (grown on demand)
  int ws_n = 0, ws_M = 0;
  int ws_mode = -1;                   // resolved pass-1 mode the workspace was sized for (AUTO flips with M)
  size_t cand_rows_want = 0;          // row-list capacity asked for after a rollout ran out of candidate rows
  int* counters_host = nullptr;       // pinned mirror of `counters` for the end-of-rollout exactness check
  int obs_tables_dirty = 1;           // c->obs changed since tc_set_obstacles built the per-obstacle layer-1 table
  int pass1_hacc = 1;                 // fp16 prefilter: hidden layers accumulate in fp16 (DSMPPI_PASS1_ACC=f32: in fp32)
  int half_tiles = 1;                 // whole-horizon tensor-core rollout: 64-row tiles while one wave covers the batch
  int prefilter_used = 0;             // set by distance_pipeline when a call went through the tensor-core prefilter
  int64_t capacity_retries = 0;       // rollouts that were run again with a larger candidate row list
  int64_t exact_fallbacks = 0;        // rollouts that were run again with every pair scored in fp32
  float* q_work = nullptr;            // (n, d) states of the current step
  float* m_rows = nullptr;            // exact masked min distance per scored row
  size_t m_rows_cap = 0;
  float* mdist = nullptr;             // tensor path: approximate (n, M)
  size_t mdist_cap = 0;
  void* enc_q = nullptr; size_t enc_q_cap = 0;       // tensor path: per-sample packed encodings
  int* cand_cnt = nullptr;            // (n)
  int* row_base = nullptr;            // (n)
  int* row_sample = nullptr; int* row_obs = nullptr; size_t rowlist_cap = 0;
  int* counters = nullptr;            // [0] candidate rows reserved this step, [1] samples x steps whose band held more
                                      // than CAND_MAX obstacles (informational), [2..3] rescored pairs (u64), [4..5]
                                      // range-fixup row counts (ping-pong), [6] rows re-scored in FFMA so far, [7] rows
                                      // that did not fit the range-fixup list, [8] largest [0] of any step of this
                                      // rollout (> capacity: the rollout is repeated with a larger list), [9] prefilter
                                      // outputs that were inf / NaN (> 0: the call is repeated with all pairs in fp32)
  int* sel = nullptr;                 // (n, K) selected obstacle indices (two-launch fp32 path)
  int* sel_rows = nullptr;            // (n, K) rows of row_dist / row_grad holding the K closest, ranked
  float* row_dist = nullptr;          // pass-2 distance of every differentiated row
  float* row_grad = nullptr;          // (rows, d)
  size_t row_dist_cap = 0, row_grad_cap = 0;
  float* dist_tmp = nullptr;          // (n)
  float* grad_tmp = nullptr;          // (n, d)
  // policy-update scratch
  float* upd_partials = nullptr; int upd_blocks = 0;
  float* stats_tmp = nullptr;         // 4 floats
  float* stats_part = nullptr;        // cost_stats_kernel: (sum, min, argmin) per CTA
  unsigned int* stats_ticket = nullptr;
  float* packed_tmp = nullptr;
  // host-buffer iteration staging
  float* stage = nullptr; size_t stage_cap = 0;
  int64_t launches = 0;
  int sm_count = 148;
  // kernel timing
  int timing = 0;
  std::vector<cudaEvent_t> ev;        // start/stop pairs around the scoring kernel of each step
  int ev_used = 0;                    // events recorded by the last rollout
  int ev_kind = 0;                    // 0: FFMA dense scoring, 1: tensor-core pass 1, 2: whole-horizon FFMA kernel,
                                      // 3: tensor-core dense scoring, 4: whole-horizon tensor-core kernel
  int fused_rollout = 1;              // 0 disables the single-launch path (tests compare the two)
  // host-buffer iteration of a large batch: copy streams + events of the chunk pipeline (capi.cu)
  cudaStream_t s_in = nullptr, s_out = nullptr;
  std::vector<cudaEvent_t> pipe_ev;
  // control tick (dsmppi_tick): the captured graph, its key and its staging blocks
  cudaStream_t s_tick = nullptr; cudaEvent_t tick_ev = nullptr;
  cudaGraph_t tick_graph = nullptr; cudaGraphExec_t tick_exec = nullptr;
  std::vector<unsigned char> tick_key;
  float* tick_h_in = nullptr; float* tick_h_out = nullptr; float* tick_d_in = nullptr; float* tick_d_out = nullptr;
  size_t tick_in_floats = 0, tick_out_floats = 0;
  int keep_counters = 0;              // 1 while a chunked iteration calls dsmppi_rollout once per chunk
};

// exact_mlp.cu
// q points at the first state; consecutive samples are q_stride floats apart
int launch_exact_forward(dsmppi_ctx* c, const float* q, int q_stride, const RowSrc& src, uint32_t ignore_mask,
                         float* m_rows, cudaStream_t st);
// forward + VJP; when m_rows != nullptr also writes the pass-1 ranking key of every row
// rows_estimate: expected row count when src.n_rows is only an upper bound (device-side counter), else 0
int launch_exact_fwdbwd(dsmppi_ctx* c, const float* q, int q_stride, const RowSrc& src, uint32_t ignore_mask,
                        float* m_rows, float* row_dist, float* row_grad, long long rows_estimate, cudaStream_t st);
// whole-horizon rollout in one launch (M <= 32, fp32 scoring); all_traj[:, 0] must be initialised
int launch_rollout_fused(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st);
// the FFMA kernels over a device-counted row list with remapped outputs (grid-stride; used to re-score the rows the
// tensor-core kernel flags as out of fp16 range)
int launch_exact_fixup(dsmppi_ctx* c, const float* q, int q_stride, const RowSrc& src, uint32_t ignore_mask,
                       float* m_rows, float* row_dist, float* row_grad, bool bwd, cudaStream_t st);
// tc_exact.cu: the same rows / outputs as the two launches above, on the tensor cores (split-fp16 operands)
// (both image builders take the network embedded in the 256 x 4 frame by dsmppi_ctx_create, never the caller's)
int tcx_build_images(dsmppi_ctx* c, const dsmppi_net* frame);
void tcx_free_images(dsmppi_ctx* c);
int launch_tc_exact(dsmppi_ctx* c, const float* q, int q_stride, const RowSrc& src, uint32_t ignore_mask, float* m_rows,
                    float* row_dist, float* row_grad, bool bwd, cudaStream_t st);
int launch_tc_rollout(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st);
inline bool use_tc_scoring(const dsmppi_ctx* c) { return c->tcx_blob && c->score_mode != DSMPPI_SCORE_FFMA; }
// tc_pass1.cu
int tc_build_images(dsmppi_ctx* c, const dsmppi_net* frame);
void tc_free_images(dsmppi_ctx* c);
int tc_set_obstacles(dsmppi_ctx* c, cudaStream_t st);
// table_ready: the per-sample layer-1 table (c->enc_q) of these n states has already been written
int tc_pass1(dsmppi_ctx* c, const float* q, int q_stride, int n, uint32_t ignore_mask, int mode, cudaStream_t st,
             bool table_ready = false);
int tc_reserve_sample_table(dsmppi_ctx* c, int n);
int tc_sample_table(dsmppi_ctx* c, const float* q, int q_stride, int n, int mode, cudaStream_t st);
// rollout_kernels.cu
int launch_rank_dense(dsmppi_ctx* c, int n, int K, bool rows_out, cudaStream_t st);
int launch_identity_rows(dsmppi_ctx* c, int n, int K, cudaStream_t st);
int launch_pack_obstacles(dsmppi_ctx* c, const float* raw, int M, int P, cudaStream_t st);
int launch_select_candidates(dsmppi_ctx* c, int n, int K, float band, size_t cap_rows, cudaStream_t st);
int launch_max_abs_diff(dsmppi_ctx* c, const float* a, const float* b, long long n, float* out, cudaStream_t st);
// exact_mlp.cu: opt the FFMA kernels into their dynamic shared memory on the context's device
int exact_set_attributes();
// rows the candidate list of the prefilter path can hold for a batch of n samples
inline size_t cand_list_cap(const dsmppi_ctx* c, int n) {
  // (fp16 accumulators double the prefilter's error and with it the calibrated band: half a list more per sample)
  const size_t base = (size_t)n * (CAND_MAX + (c->pass1_hacc ? CAND_MAX / 2 : 0));
  return base > c->cand_rows_want ? base : c->cand_rows_want;
}
int launch_rank_candidates(dsmppi_ctx* c, int n, int K, cudaStream_t st);
int launch_blend(dsmppi_ctx* c, int n, int K, float* dist_out, float* grad_out, cudaStream_t st);
int launch_step(dsmppi_ctx* c, const dsmppi_rollout_args* a, int t, cudaStream_t st);
// prefilter path: ranking of the candidate rows + the step + (table_mode >= 0) the layer-1 table of the next state
int launch_rank_step(dsmppi_ctx* c, const dsmppi_rollout_args* a, int t, int table_mode, cudaStream_t st);
int launch_init_traj(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st);
int launch_cost(dsmppi_ctx* c, const dsmppi_cost_args* a, cudaStream_t st);
int launch_basis(dsmppi_ctx* c, const float* grad, int64_t n, float* basis, cudaStream_t st);
int launch_fk_distance(dsmppi_ctx* c, const float* q, int q_stride, int n, int n_pts, const float* span_host,
                       float* dist, float* grad, int grad_stride, int* idx, cudaStream_t st);
int launch_cost_stats(dsmppi_ctx* c, const float* cost, int N, float* stats, cudaStream_t st);
int launch_update_partial(dsmppi_ctx* c, const dsmppi_update_args* a, const float* stats, float* packed,
                          cudaStream_t st);
int launch_update_finalize(dsmppi_ctx* c, const dsmppi_update_args* a, const float* packed, int* n_updated,
                           cudaStream_t st);
int launch_kernel_candidates(dsmppi_ctx* c, const dsmppi_candidates_args* a, cudaStream_t st);
