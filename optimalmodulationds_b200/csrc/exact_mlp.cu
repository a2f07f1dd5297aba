// fp32-exact evaluation of the learned distance network on (sample, obstacle) rows.
//
//   exact_mlp_kernel<false, RPT>: forward only  -> masked minimum link distance per row  (MPPI.py:235-242)
//   exact_mlp_kernel<true,  RPT>: forward + analytic VJP at argmin_l of the raw output   (robot_sdf.py:153-158)
//
// One CTA owns R = 4*RPT rows (RPT = 8, 4 or 2).  Activations live in shared memory feature-major
// (act[k][row]) and are updated in place layer by layer.  A warp owns an R-row x (8*FT)-feature block of the layer
// output, its lanes form a 4 x 8 grid and each thread keeps an RPT-row x FT-feature register tile (FT = 8, 4 or 2
// => 4, 8 or 16 warps per CTA), so one k-step of a warp is FT*RPT FFMAs fed by single-wavefront shared-memory
// loads (broadcast over the row / feature groups).  FT = 8 amortises the loads best and is used whenever there are
// enough row tiles to fill the SMs; the 8- and 16-warp shapes put 2 or 4 warps on every scheduler of an SM that
// holds a single tile, which is what the latency of a small batch (and of the whole-horizon kernel) is made of
// (pick_shape below has the measurements; only 8x8, 8x4 and 4x4 are instantiated).
// The weights of all seven GEMMs (4 forward, 3 backward) are one stream of 8-row stages that the CTA pulls from L2
// through a 4-deep cp.async ring, three stages (24 k-steps) ahead of the FFMAs and straight across layer
// boundaries: a lone CTA on an SM is then FFMA-bound instead of waiting ~500 cycles for L2 every four k-steps,
// which is what set the pace of the first versions whenever there were few rows.  ReLU masks stay in
// registers as bit masks (the forward and backward tilings coincide), so the backward pass needs no extra memory.
// The host picks RPT per launch from the (estimated) row count: big tiles amortise the weight stream, small tiles
// fill the 148 SMs when there are few rows and shorten the tail of the last wave (pick_rpt below).
// A network narrower or shallower than 256 x 4 costs what it computes: the kernels are instantiated for WID = 64, 128
// and 256 features per hidden layer (the smallest that covers the network's width is launched: fewer warps, stages and
// k-steps) and run net.nh hidden layers, i.e. nh forward GEMMs and nh - 1 backward ones plus W_1^T.  The features past
// the network's width are zero in the weights, so every WID >= width gives the same bits (ReLU keeps them at 0 and a
// zero product leaves an fp32 FMA chain unchanged).
// All arithmetic is IEEE fp32 (no fast-math): this is the path that has to agree with the reference's torch-CPU
// numbers to ~1e-6.
#include <cstdlib>

#include "internal.cuh"
#include "step_device.cuh"
#include "exact_tile.cuh"

namespace {
using namespace exact_tile;

// resident CTAs per SM the register budget is sized for: at WID = 256 the 4-warp shape packs 4 (32-row) or 6 (16-row)
// tiles on an SM, the 8-warp shape 2, the 16-warp shape 1; a narrower tile has proportionally fewer warps, so the same
// register budget per thread packs proportionally more of them
__host__ __device__ constexpr int min_ctas(int RPT, int FT, int WID) {
  return (FT == 8 ? (RPT == 8 ? 4 : 6) : (FT == 4 ? (RPT == 8 ? 2 : 3) : 1)) * (HID / WID);
}

template <bool BWD, int RPT, int FT, int WID>
__global__ void __launch_bounds__(nthreads(FT, WID), min_ctas(RPT, FT, WID))
exact_mlp_kernel(NetDev net, RowSrc src, const float* __restrict__ q, int q_stride, const float* __restrict__ obs,
                 uint32_t ignore_mask, float* __restrict__ out_m, float* __restrict__ out_dist,
                 float* __restrict__ out_grad) {
  constexpr int R = 4 * RPT;
  extern __shared__ __align__(16) float smem[];
  const int n_rows = src.n_rows_dev ? min(*src.n_rows_dev, src.n_rows) : src.n_rows;
  const int tiles = (n_rows + R - 1) / R;
  if ((int)blockIdx.x >= tiles) return;
  TileSmem<RPT, WID> sm(smem);
  WeightStream<WID> ws;
  // one tile per CTA in the regular launches; the re-scoring launch (launch_exact_fixup) strides a bounded grid
  stream_begin<BWD, nthreads(FT, WID)>(ws, &net, sm.ring,
                                       (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x);
  int stage = 0;
  for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    mlp_tile<BWD, RPT, FT, WID>(net, src, tile * R, n_rows, q, q_stride, obs, nullptr, 0.f, ignore_mask, out_m, out_dist,
                                out_grad, sm, ws, stage);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Whole-horizon rollout in ONE launch for small obstacle sets (M <= R): a CTA owns S = R / M samples and all of
// their (sample, obstacle) rows, and samples never interact, so it can run all H steps by itself -- network
// forward + VJP on its tile, then one thread per sample ranks its M rows, blends the K closest gradients and takes
// the modulation / policy / Euler step (step_device.cuh) -- with no grid-wide dependency and no launch per step.
// The weight stream simply keeps running across steps.  This is the path of the reference's own CPU-sized
// problems (planar scripts: M = 2..4; Franka integrator tick: N = 1, H = 2) where launch latency, not FLOPs,
// set the pace of the per-step launch sequence.
// MOVE: constant-velocity obstacles -- step t reads obstacle j at obstacle_at(obs, vel, j, c, (t - 1) dt).  A separate
// instantiation, so the static kernels are compiled exactly as without motion.
// ------------------------------------------------------------------------------------------------
template <int RPT, int FT, int WID, bool MOVE>
__global__ void __launch_bounds__(nthreads(FT, WID), (FT == 8 ? 3 : 2) * (HID / WID))
rollout_fused_kernel(NetDev net, StepArgs sa, const float* __restrict__ obs, const float* __restrict__ vel, int M,
                     uint32_t ignore_mask, float* m_rows, float* row_dist, float* row_grad, int* sel_rows) {
  constexpr int R = 4 * RPT;
  extern __shared__ __align__(16) float smem[];
  const int S = R / M;                                  // samples per CTA
  const int i0 = blockIdx.x * S;
  if (i0 >= sa.N) return;
  const int ns = min(S, sa.N - i0);
  const int row0 = i0 * M;                              // dense rows: row = i * M + j
  const int n_rows = row0 + ns * M;
  TileSmem<RPT, WID> sm(smem);
  WeightStream<WID> ws;
  stream_begin<true, nthreads(FT, WID)>(ws, &net, sm.ring, sa.H);
  int stage = 0;
  RowSrc src{};
  src.mode = ROWS_DENSE;
  src.M = M;
  const int d = net.d, K = sa.K;
  const int tid = threadIdx.x;
  for (int t = 1; t <= sa.H; ++t) {
    const float* q = sa.traj + (size_t)(t - 1) * d;     // q_prev = all_traj[:, t-1, :]
    const float tau = MOVE ? __fmul_rn((float)(t - 1), sa.dt) : 0.f;
    mlp_tile<true, RPT, FT, WID>(net, src, row0, n_rows, q, sa.H * d, obs, MOVE ? vel : nullptr, tau, ignore_mask, m_rows,
                                 row_dist, row_grad, sm, ws, stage);
    __syncthreads();                                    // the tile's rows are visible to the whole CTA
    if (tid < ns) {
      const int i = i0 + tid;
      // the K closest obstacles, ascending by (masked distance, obstacle index)  (MPPI.py:243-247)
      const float* mr = m_rows + (size_t)i * M;
      float last_v = -3.4e38f;
      int last_j = -1;
      for (int kk = 0; kk < K; ++kk) {
        float bv = 3.4e38f;
        int bj = -1;
        for (int j = 0; j < M; ++j) {
          const float v = mr[j];
          const bool after = kk == 0 || v > last_v || (v == last_v && j > last_j);
          if (after && (bj < 0 || v < bv)) { bv = v; bj = j; }
        }
        if (bj < 0) bj = last_j < 0 ? 0 : last_j;
        sel_rows[(size_t)i * K + kk] = i * M + bj;
        last_v = bv; last_j = bj;
      }
      step_sample(sa, i, t, step_io_global(sa, i));
    }
    __syncthreads();                                    // next state written before the next tile reads it
  }
}


// Tile shape (rows per thread, features per thread).  Measured on B200 (tools/exact_shape_sweep.py, ms per
// propagate, planar-7 net, M = 4, H = 30; shapes as RPTxFT):
//     rows per step   8x8     4x8     8x4     4x4     8x2     4x2
//        1 000        5.52    4.20    4.79    3.77    5.61    4.13
//        4 000        5.54    5.06    4.86    5.80    5.68    8.19
//        8 000        7.63    7.91    7.84   10.64   11.17   16.19
//       16 000       13.84   13.73   15.29   18.57   22.13   28.28
// While the batch gives an SM at most one 32-row tile, the 8-warp shapes win: two warps per scheduler hide part of
// the shared-memory / FMA latency a lone 4-warp CTA exposes (ncu: 27 % -> 39 % issue-active), 16-row tiles while even
// those leave SMs idle.  16 warps (FT = 2) lose again: 2-feature register tiles need a load per two FFMA2.  From two
// tiles per SM on, the 4-warp 8 x 8 register tile is best (fewest shared-memory loads per FMA; 87 % of the FMA
// peak in steady state with 4 CTAs per SM).
struct Shape { int rpt, ft; };
Shape pick_shape(const dsmppi_ctx* c, long long rows, int min_rows_per_tile) {
  const long long sms = c->sm_count;
  const long long tiles32 = (rows + 31) / 32, tiles16 = (rows + 15) / 16;
  Shape s = {8, 8};
  if (tiles32 <= sms) s = {(min_rows_per_tile <= 16 && tiles16 <= sms) ? 4 : 8, 4};
  const char* fr = std::getenv("DSMPPI_EXACT_RPT");
  const char* ff = std::getenv("DSMPPI_EXACT_FT");
  if (ff) { const int f = std::atoi(ff); if (f == 8 || f == 4) s.ft = f; }
  if (fr) { const int f = std::atoi(fr); if (f == 8 || (f == 4 && min_rows_per_tile <= 16)) s.rpt = f; }
  if (s.ft == 8) s.rpt = 8;
  return s;
}

template <bool BWD, int RPT, int FT, int WID>
int launch_variant(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src,
                   uint32_t ignore_mask, float* out_m, float* out_dist, float* out_grad, cudaStream_t st) {
  constexpr int R = 4 * RPT;
  const long long grid = ((long long)src.n_rows + R - 1) / R;
  exact_mlp_kernel<BWD, RPT, FT, WID><<<(unsigned)grid, nthreads(FT, WID), smem_bytes(R, WID), st>>>(
      c->net, src, q, q_stride, obs, ignore_mask, out_m, out_dist, out_grad);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}

// the smallest instantiated width that covers the network's hidden width
int tile_width(const dsmppi_ctx* c) { return c->net.width <= 64 ? 64 : (c->net.width <= 128 ? 128 : HID); }

#define SHAPE_DISPATCH_W(sh, W, CALL)                             \
  do {                                                            \
    if (sh.ft == 8) return CALL(8, 8, W);                         \
    if (sh.rpt == 8) return CALL(8, 4, W);                        \
    return CALL(4, 4, W);                                         \
  } while (0)
#define SHAPE_DISPATCH(c, sh, CALL)                               \
  do {                                                            \
    const int w_ = tile_width(c);                                 \
    if (w_ == 64) SHAPE_DISPATCH_W(sh, 64, CALL);                 \
    if (w_ == 128) SHAPE_DISPATCH_W(sh, 128, CALL);               \
    SHAPE_DISPATCH_W(sh, HID, CALL);                              \
  } while (0)

template <bool BWD>
int launch(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src, uint32_t ignore_mask,
           float* out_m, float* out_dist, float* out_grad, long long rows_estimate, cudaStream_t st) {
  if (src.n_rows <= 0) return 0;
  if (rows_estimate <= 0 || rows_estimate > src.n_rows) rows_estimate = src.n_rows;
  const Shape sh = pick_shape(c, rows_estimate, 1);
#define CALL(RPT, FT, WID) \
  launch_variant<BWD, RPT, FT, WID>(c, q, q_stride, obs, src, ignore_mask, out_m, out_dist, out_grad, st)
  SHAPE_DISPATCH(c, sh, CALL);
#undef CALL
}

template <int RPT, int FT, int WID>
int launch_fused_variant(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st) {
  constexpr int R = 4 * RPT;
  const int S = R / c->M;
  const long long grid = ((long long)a->N + S - 1) / S;
  const StepArgs sa = make_step_args(c, a, 0);
  if (c->moving)
    rollout_fused_kernel<RPT, FT, WID, true><<<(unsigned)grid, nthreads(FT, WID), smem_bytes(R, WID), st>>>(
        c->net, sa, c->obs, c->vel, c->M, a->ignored_link_mask, c->m_rows, c->row_dist, c->row_grad, c->sel_rows);
  else
    rollout_fused_kernel<RPT, FT, WID, false><<<(unsigned)grid, nthreads(FT, WID), smem_bytes(R, WID), st>>>(
        c->net, sa, c->obs, nullptr, c->M, a->ignored_link_mask, c->m_rows, c->row_dist, c->row_grad, c->sel_rows);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}

template <int RPT, int FT, int WID>
int set_attributes_variant() {
  constexpr int R = 4 * RPT;
  CUDA_TRY(cudaFuncSetAttribute(exact_mlp_kernel<true, RPT, FT, WID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem_bytes(R, WID)));
  CUDA_TRY(cudaFuncSetAttribute(exact_mlp_kernel<false, RPT, FT, WID>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem_bytes(R, WID)));
  CUDA_TRY(cudaFuncSetAttribute(rollout_fused_kernel<RPT, FT, WID, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem_bytes(R, WID)));
  CUDA_TRY(cudaFuncSetAttribute(rollout_fused_kernel<RPT, FT, WID, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem_bytes(R, WID)));
  return 0;
}

template <int WID>
int set_attributes_width() {
  if (set_attributes_variant<8, 8, WID>()) return 1;
  if (set_attributes_variant<8, 4, WID>()) return 1;
  return set_attributes_variant<4, 4, WID>();
}

}  // namespace

// The dynamic shared-memory opt-in is a per-DEVICE function attribute: dsmppi_ctx_create calls this after
// cudaSetDevice, so a second context on another GPU of the same process gets it too (a process-wide "done" flag
// would leave that device without it).
int exact_set_attributes() {
  if (set_attributes_width<64>()) return 1;
  if (set_attributes_width<128>()) return 1;
  return set_attributes_width<HID>();
}

// whole-horizon single launch; the caller has checked M <= 32 and initialised all_traj[:, 0]
int launch_rollout_fused(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st) {
  const int M = c->M;
  // a CTA holds whole samples: S = R / M of them, so the row count that matters is N * (R / S) ~ N * M
  const Shape sh = pick_shape(c, (long long)a->N * M, M);
#define CALL(RPT, FT, WID) launch_fused_variant<RPT, FT, WID>(c, a, st)
  SHAPE_DISPATCH(c, sh, CALL);
#undef CALL
}

namespace {
template <int WID>
int launch_fixup_width(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src,
                       uint32_t ignore_mask, float* m_rows, float* row_dist, float* row_grad, bool bwd, cudaStream_t st) {
  constexpr int RPT = 8, FT = 8, R = 4 * RPT;
  long long grid = ((long long)src.n_rows + R - 1) / R;
  if (grid > 4LL * c->sm_count) grid = 4LL * c->sm_count;       // usually no row is flagged: keep the launch tiny
  if (bwd)
    exact_mlp_kernel<true, RPT, FT, WID><<<(unsigned)grid, nthreads(FT, WID), smem_bytes(R, WID), st>>>(
        c->net, src, q, q_stride, obs, ignore_mask, m_rows, row_dist, row_grad);
  else
    exact_mlp_kernel<false, RPT, FT, WID><<<(unsigned)grid, nthreads(FT, WID), smem_bytes(R, WID), st>>>(
        c->net, src, q, q_stride, obs, ignore_mask, m_rows, nullptr, nullptr);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}
}  // namespace

int launch_exact_fixup(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src,
                       uint32_t ignore_mask, float* m_rows, float* row_dist, float* row_grad, bool bwd, cudaStream_t st) {
#define FIXUP(W) launch_fixup_width<W>(c, q, q_stride, obs, src, ignore_mask, m_rows, row_dist, row_grad, bwd, st)
  const int w = tile_width(c);
  if (w == 64) return FIXUP(64);
  if (w == 128) return FIXUP(128);
  return FIXUP(HID);
#undef FIXUP
}

int launch_exact_forward(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src,
                         uint32_t ignore_mask, float* m_rows, cudaStream_t st) {
  if (use_tc_scoring(c))
    return launch_tc_exact(c, q, q_stride, obs, src, ignore_mask, m_rows, nullptr, nullptr, false, st);
  return launch<false>(c, q, q_stride, obs, src, ignore_mask, m_rows, nullptr, nullptr, 0, st);
}

int launch_exact_fwdbwd(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src,
                        uint32_t ignore_mask, float* m_rows, float* row_dist, float* row_grad, long long rows_estimate,
                        cudaStream_t st) {
  if (use_tc_scoring(c))
    return launch_tc_exact(c, q, q_stride, obs, src, ignore_mask, m_rows, row_dist, row_grad, true, st);
  return launch<true>(c, q, q_stride, obs, src, ignore_mask, m_rows, row_dist, row_grad, rows_estimate, st);
}
