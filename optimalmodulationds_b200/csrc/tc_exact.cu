// fp32-accurate evaluation of the distance network AND its analytic input gradient on the tensor cores.
//
//   tc_exact_kernel<false>: forward only  -> masked minimum link distance per row  (MPPI.py:235-242)
//   tc_exact_kernel<true>:  forward + VJP at argmin_l of the raw output            (robot_sdf.py:153-158)
//
// Same rows, same outputs as exact_mlp.cu (which stays as the strict IEEE-FFMA mode); this is the scoring path of
// every workload by default.  Arithmetic: every operand is split a = hi + lo * 2^-11 with hi = fp16(a),
// lo = fp16((a - hi) * 2^11) -- 22 significant bits, the lo half scaled up so it cannot underflow -- and a product
// sum is three fp16 tcgen05 MMAs with fp32 accumulation in TMEM:
//       D1 += A_hi * B_hi          D2 += A_hi * B_lo + A_lo * B_hi          result = D1 + D2 * 2^-11
// (the lo * lo term is below 2^-24 of the product).  The tensor core truncates its fp32 accumulator toward zero at
// every MMA (K = 16) step, which shrinks a D1 chain of n steps by (1.65e-8 n + 2.1e-8) of its value on average
// (tools/split_precision_probe.py measures both the bias and this fit); uncorrected that bias adds up coherently over
// the layers (rms error 1.4e-6 of the rms distance), so the epilogue multiplies it back: result += D1 * c(n).
// Measured on the shipped nets against an fp64 evaluation: rms error 1.9e-7 .. 3.1e-7 of the rms distance and
// 2.1e-7 .. 3.8e-7 of the rms gradient -- the same as IEEE FFMA (1.5e-7 .. 2.5e-7 / 1.9e-7 .. 2.6e-7); DESIGN.md
// section 3 has the table.
//
// Design (B200, one CTA pair per TPC, persistent over 256-row tiles):
//   * cta_group::2 MMAs, M = 256 (128 rows per CTA = the 128 TMEM lanes): D1 and D2 of a 256-wide layer fill the 512
//     TMEM columns.  The A operand (activations, then back-propagated gradients) lives in shared memory as two K-major
//     fp16 images (hi, lo; 2 x 64 KB) that the epilogue warps rewrite in place.
//   * weights never fit on chip in split form (7 GEMMs x 256 KB), so they stream: each CTA pulls its share of every
//     stage (32 KB: N half x K half, hi | lo) from L2 with one bulk TMA copy into a 3-slot ring, running ahead across
//     layer and tile boundaries.  The pair shares every stage, so a tile of 256 rows costs 816 KB of L2 reads per SM
//     for 41 k cycles of MMAs (20 B/cycle/SM, half the L2 limit).
//   * warp roles: warps 0-7 epilogue (TMEM lane quarter = warp % 4; the two warps of a quarter interleave 32-column
//     chunks): D1/D2 -> bias, ReLU (sign bits kept in registers for the backward pass), hi/lo split, st.shared of the
//     next A operand; warp 8 = TMEM allocator + MMA issuer (leader CTA) / "stage landed" relay (peer CTA);
//     warp 9 = weight loader.
//   * the output layer (N = 32), the one-hot seed g4 = W5[l*, :] * mask and the final W1^T contraction (N = 32)
//     plus the encoding Jacobian (SURVEY Appendix B) run in the same pipeline: 9 GEMMs per tile with BWD.
//   * N-half pipelining.  With TMEM full a layer has no second accumulator to drain under the next GEMM, so every
//     hidden GEMM is issued as two N = 128 halves (same MMA rate, tools/tcx_ss_microbench.cu), each with its own
//     "accumulator complete" barrier:
//       - the epilogue of N half 0 runs under the MMAs of N half 1 and parks its converted operand in 64 registers;
//         it is stored as soon as the last MMAs that read those operand columns have retired (barrier AFREE, after
//         the first K stage of N half 1), i.e. still under N half 1;
//       - the epilogue of N half 1 runs under the NEXT layer's N half 0, which follows the operand K quarter by K
//         quarter (four "operand ready" barriers, 64 columns each);
//       - the issuer opens a weight stage (descriptors, "weights landed") BEFORE it waits for the operand, and builds
//         descriptors from 32-bit low words inside the asm block -- nothing but the MMAs follows a hand-over;
//       - the seed epilogue reads the split rows of W5 from the output layer's weight stage, which the issuer keeps
//         in its ring slot until the first seed quarter is signalled (no global table look-up on the critical path);
//       - the two warps of a lane quarter share the input encoding (h = 0 joint angles, h = 1 obstacle point), and a
//         row's global stores wait until the tile's last hand-over is out: fence.proxy.async is a MEMBAR.ALL.CTA,
//         which would otherwise wait for their round trip.
//     Per-element arithmetic (k order, the three MMAs per step) is unchanged: results are bitwise equal to the
//     unpipelined kernel (tools/tcx_regress.py).  Phase accounting: tools/tcx_prof.py on a -DDSMPPI_TCX_PROF build.
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "internal.cuh"
#include "step_device.cuh"
#include "exact_tile.cuh"
#include "tc_ptx.cuh"

// Experiment switches (tools/tcx_variants.py times the combinations; the defaults are the measured best):
//   TCX_ENC_PIPE   1 = the next tile's encoding is computed before the current tile's last GEMM completes and stored
//                      at the tile end; 0 = computed and stored at the top of the tile
//   TCX_DEFER_STG  1 = a row's results are stored after the tile's last operand hand-over; 0 = where they are produced
#ifndef TCX_ENC_PIPE
#define TCX_ENC_PIPE 1
#endif
#ifndef TCX_DEFER_STG
#define TCX_DEFER_STG 1
#endif

namespace {
using namespace tcx;
using exact_tile::pk2, exact_tile::pk2f, exact_tile::unpk2, exact_tile::fma2, exact_tile::add2, exact_tile::mul2;

constexpr int TROWS = 128;                 // rows per CTA per tile
constexpr int W_MMA = 8, W_LOAD = 9;
// three warpgroups: two of epilogue warps and one holding the two control warps (warps 10-11 only complete it), so
// that setmaxnreg can hand the control group's registers to the epilogue: double-buffered TMEM loads need ~200
constexpr int NTHREADS = 12 * 32;
constexpr int EPI_REGS = 224, CTRL_REGS = 40;   // 8*32*224 + 4*32*40 = 62464 <= 65536
constexpr int NSLOT = 3;
constexpr int SLOT_BYTES = 32768;
constexpr uint32_t A_LBO = TROWS * 16;     // bytes between consecutive 8-element K chunks of the A images
constexpr float SPLIT = 2048.f, INV_SPLIT = 1.f / 2048.f;
// accumulator-truncation compensation of a D1 chain of n MMA steps: 1.65e-8 n + 2.1e-8 (see the header).  Only steps
// with a non-zero product truncate: a GEMM over the hidden features of a W-wide network (embedded in the 256 x 4 frame)
// needs comp_steps(ceil(W / 16)), and an identity layer of the frame, one non-zero product per sum, needs 0.
__host__ __device__ constexpr float comp_steps(int n) { return n > 0 ? 1.65e-8f * n + 2.1e-8f : 0.f; }
constexpr float COMP_K256 = comp_steps(16), COMP_K32 = comp_steps(2);
static_assert(COMP_K256 == 1.65e-8f * 16 + 2.1e-8f && COMP_K32 == 1.65e-8f * 2 + 2.1e-8f, "shipped constants");
// per-GEMM compensation of a pass: [0..3] forward layers, [4] output layer, [5..7] backward W_l^T for l = 3, 2, 1,
// [8] the final W_1^T
constexpr int N_GEMM = 9;
__device__ __forceinline__ float comp_of(const float (&comp)[N_GEMM], int g) {
  float v = comp[0];
#pragma unroll
  for (int i = 1; i < N_GEMM; ++i) v = g == i ? comp[i] : v;
  return v;
}
__device__ __forceinline__ float combine(uint32_t d1, uint32_t d2, float comp) {
  const float a = __uint_as_float(d1);
  return fmaf(a, comp, fmaf(__uint_as_float(d2), INV_SPLIT, a));
}

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi);
__device__ __forceinline__ float2 unpack_h2(uint32_t p);
// D1 + D2 * 2^-11 + D1 * comp for two adjacent columns
__device__ __forceinline__ uint64_t combine2(uint32_t d1a, uint32_t d1b, uint32_t d2a, uint32_t d2b, float comp) {
  const uint64_t a = pk2(d1a, d1b);
  return fma2(a, pk2f(comp, comp), fma2(pk2(d2a, d2b), pk2f(INV_SPLIT, INV_SPLIT), a));
}
// two fp32 values -> their fp16 hi pair and scaled fp16 lo pair (the caller tracks the largest |hi| bit pattern: a
// saturated conversion, 0x7bff = 65504, marks the row as out of fp16 range)
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& h, uint32_t& l) {
  h = pack_h2(v0, v1);
  const float2 f = unpack_h2(h);
  float l0, l1;
  unpk2(mul2(add2(pk2f(v0, v1), pk2f(-f.x, -f.y)), pk2f(SPLIT, SPLIT)), l0, l1);
  l = pack_h2(l0, l1);
}

// ---- shared-memory map (bytes)
constexpr int OFF_AHI = 0;                 // 128 rows x 256 K fp16, canonical K-major (32 chunks x 2 KB)
constexpr int OFF_ALO = 65536;
constexpr int OFF_RING = 131072;           // NSLOT x 32 KB weight stages
constexpr int OFF_BAR = OFF_RING + NSLOT * SLOT_BYTES;
// AREADY0..3: K quarter q (64 columns) of the next A operand is in place (epilogue -> issuer, leader CTA);
// DFULL0 / DFULL1: accumulator columns of N half 0 / 1 are complete (tcgen05.commit -> epilogue, both CTAs).  One
// barrier per quarter / half, so that no barrier can run two phases ahead of a waiter.
// AFREE: the MMAs that read K half 0 of the CURRENT A operand have retired (the first K stage of N half 1 is the last
// of them), so the parked half-0 columns of the next operand may be stored while N half 1 is still running.
enum { BAR_FULL = 0, BAR_PEER = NSLOT, BAR_EMPTY = 2 * NSLOT, BAR_AREADY0 = 3 * NSLOT, BAR_DFULL0 = 3 * NSLOT + 4,
       BAR_DFULL1 = 3 * NSLOT + 5, BAR_AFREE = 3 * NSLOT + 6, NBAR = 3 * NSLOT + 7 };
constexpr int OFF_TMEMPTR = OFF_BAR + 128;  // NBAR * 8 = 128
constexpr int OFF_LST = OFF_TMEMPTR + 16;  // argmin link per row (128 ints)
constexpr int OFF_OVF = OFF_LST + TROWS * 4;   // "left the fp16 range" flag per row (128 ints)
constexpr int OFF_FIXN = OFF_OVF + TROWS * 4;   // whole-horizon kernel: flagged rows of this CTA's tile (count + list)
constexpr int OFF_FIXL = OFF_FIXN + 16;         // (3, 128) ints: samples | obstacles | output rows
constexpr int OFF_B4 = OFF_FIXL + 3 * TROWS * 4;   // output-layer bias (16 floats)
constexpr int SMEM_BYTES = OFF_B4 + 64;
static_assert(exact_tile::smem_bytes(32) <= OFF_RING, "the FFMA fallback tile lives in the A operand images");
constexpr int OFF_SCRATCH = OFF_ALO + 32768;   // final epilogue: a[e][row] fp32 (16 KB) inside the idle A_lo image
// whole-horizon kernel: the tile's rows (ranking key, distance, gradient) and the stepped states, handed from the row
// threads to the CTA's step threads and back through the last 16 KB of the A_lo image (idle between the last GEMM of
// a step and the second half of the next step's first epilogue; the FFMA fallback tile ends below it)
constexpr int OFF_STAGE = OFF_ALO + 49152;
constexpr int STG_M = 0, STG_DIST = TROWS, STG_GRAD = 2 * TROWS, STG_Q = 2 * TROWS + TROWS * MAXD,          // float offsets
              STG_ROWS = STG_Q + TROWS * MAXD;                                                          // (128, MAXK) ints
static_assert((STG_ROWS + TROWS * MAXK) * 4 <= 16384, "row staging exceeds the tail of the A_lo image");
static_assert(exact_tile::smem_bytes(32) <= OFF_STAGE && OFF_SCRATCH + 16384 <= OFF_STAGE, "staging overlaps");
static_assert(NBAR * 8 <= 128, "barrier block");
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared-memory budget");

// ---- weight image of one CTA rank: the stages of one pass in issue order.  A hidden GEMM (N = 256 over the pair) is
// issued as two N = 128 halves x; of half x this CTA holds the 64 output features 128 x + 64 rank + [0, 64).
//   s = 0, 1     GEMM 0  forward layer 1      K = 32   half x = s             8 KB  [hi 4 KB | lo 4 KB]
//   s = 2..13    GEMM 1-3 forward layers 2-4  K = 128  (x, K half) = 4 stages 32 KB [hi 16 KB | lo 16 KB] per GEMM
//   s = 14       GEMM 4  output layer         K = 256  N = 32                 16 KB (16 rows per CTA)
//   s = 15..26   GEMM 5-7 backward W4^T..W2^T K = 128  (x, K half)            32 KB
//   s = 27       GEMM 8  backward W1^T        K = 256  N = 32                 16 KB
constexpr int STAGES_FWD = 15, STAGES_BWD = 28;
constexpr size_t IMG_BYTES = 16384 + 12 * 32768 + 16384 + 12 * 32768 + 16384;   // 835584
__host__ __device__ __forceinline__ void stage_info(int s, uint32_t& off, uint32_t& bytes) {
  if (s <= 1) { off = (uint32_t)s * 8192; bytes = 8192; }
  else if (s <= 13) { off = 16384 + (uint32_t)(s - 2) * 32768; bytes = 32768; }
  else if (s == 14) { off = 16384 + 12 * 32768; bytes = 16384; }
  else if (s <= 26) { off = 2 * 16384 + 12 * 32768 + (uint32_t)(s - 15) * 32768; bytes = 32768; }
  else { off = 2 * 16384 + 24 * 32768; bytes = 16384; }
}

struct TxImages {
  uint8_t* dev = nullptr;      // [rank 0 image | rank 1 image]
};

struct TxArgs {
  const uint8_t* img0; const uint8_t* img1;
  NetDev net;
  RowSrc src;
  const float* q; int q_stride;
  const float* obs;
  const float* vel;                          // whole-horizon kernel with MOVE: (M, 4) obstacle velocities
  uint32_t ignore_mask;
  float* out_m; float* out_dist; float* out_grad;
  int* fix_count;                            // rows appended to fix_list by this launch
  int* fix_next;                             // the counter of the NEXT launch: zeroed here
  int* fix_total;                            // rows handed to the FFMA kernel since the context was created
  int* fix_dropped;                          // rows that did not fit fix_list (both reported by dsmppi_score_stats)
  int* fix_list;                             // (3, fix_cap) = [samples | obstacles | output rows]
  int fix_cap;
  // whole-horizon mode (MODE 2): a CTA owns S = 128 / M samples and all of their (sample, obstacle) rows for all H steps
  StepArgs sa; int M; int S; float* m_rows; float* row_dist; float* row_grad; int* sel_rows;
  float comp[N_GEMM];                        // accumulator-truncation compensation per GEMM (set_compensation)
  int dbg;                                   // DSMPPI_TCX_DEBUG=4: no accumulator-truncation compensation (precision tools)
  long long* prof;                           // -DDSMPPI_TCX_PROF builds: (event id, clock64) pairs of CTA 0's warps
};

// Phase accounting (tools/tcx_prof.py): CTA 0's epilogue warps 0 / 4, its MMA issuer and its weight loader stamp
// (event, clock64) pairs into a.prof -- only in builds with -DDSMPPI_TCX_PROF, the product kernel carries none of it.
#ifdef DSMPPI_TCX_PROF
#define TCX_PROF(region, id)                                                         \
  do {                                                                               \
    if (a.prof && blockIdx.x == 0 && lane == 0 && pcount < 1000) {                   \
      a.prof[(region) * 2048 + 2 * pcount] = (id);                                   \
      a.prof[(region) * 2048 + 2 * pcount + 1] = clock64();                          \
      ++pcount;                                                                      \
    }                                                                                \
  } while (0)
#else
#define TCX_PROF(region, id) do { } while (0)
#endif

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float2 unpack_h2(uint32_t p) {
  return __half22float2(*reinterpret_cast<const __half2*>(&p));
}
// ---- epilogue building blocks: 32 accumulator columns of one row -> 16 packed hi and 16 packed lo operand words
// forward: + bias, ReLU, split; returns the SIGN bits of the pre-activations (set = ReLU off), column 0 in bit 31
__device__ __forceinline__ uint32_t fwd_chunk32(const uint32_t (&r1)[32], const uint32_t (&r2)[32], const float* bias,
                                                float comp, uint32_t (&hw)[16], uint32_t (&lw)[16], uint32_t& range) {
  uint32_t m = 0;
#pragma unroll
  for (int j8 = 0; j8 < 4; ++j8) {
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + 8 * j8));
    const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + 8 * j8 + 4));
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int idx = 8 * j8 + 2 * p;
      float x0, x1;
      unpk2(add2(combine2(r1[idx], r1[idx + 1], r2[idx], r2[idx + 1], comp), pk2f(bb[2 * p], bb[2 * p + 1])), x0, x1);
      m = __funnelshift_l(__float_as_uint(x0), m, 1);
      m = __funnelshift_l(__float_as_uint(x1), m, 1);
      split2(fmaxf(x0, 0.f), fmaxf(x1, 0.f), hw[4 * j8 + p], lw[4 * j8 + p]);
      range = __vmaxu2(range, hw[4 * j8 + p]);
    }
  }
  return m;
}
// backward: columns whose forward ReLU was off (bit set in `bits`, column 0 in bit 31) are zeroed, then split
__device__ __forceinline__ void bwd_chunk32(const uint32_t (&r1)[32], const uint32_t (&r2)[32], uint32_t bits, float comp,
                                            uint32_t (&hw)[16], uint32_t (&lw)[16], uint32_t& range) {
#pragma unroll
  for (int j8 = 0; j8 < 4; ++j8) {
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const int idx = 8 * j8 + 2 * p;
      float x0, x1;
      unpk2(combine2(r1[idx], r1[idx + 1], r2[idx], r2[idx + 1], comp), x0, x1);
      x0 = (bits & (0x80000000u >> idx)) ? 0.f : x0;
      x1 = (bits & (0x40000000u >> idx)) ? 0.f : x1;
      split2(x0, x1, hw[4 * j8 + p], lw[4 * j8 + p]);
      range = __vmaxu2(range, hw[4 * j8 + p] & 0x7fff7fffu);
    }
  }
}
// 32 converted columns -> four 8-column chunks (ch0 ..) of this thread's row in the two A images
template <uint32_t LBO>
__device__ __forceinline__ void store_chunk32(uint8_t* a_hi, uint8_t* a_lo, int ch0, const uint32_t (&hw)[16],
                                              const uint32_t (&lw)[16]) {
#pragma unroll
  for (int j8 = 0; j8 < 4; ++j8) {
    *reinterpret_cast<uint4*>(a_hi + (ch0 + j8) * LBO) = make_uint4(hw[4 * j8], hw[4 * j8 + 1], hw[4 * j8 + 2], hw[4 * j8 + 3]);
    *reinterpret_cast<uint4*>(a_lo + (ch0 + j8) * LBO) = make_uint4(lw[4 * j8], lw[4 * j8 + 1], lw[4 * j8 + 2], lw[4 * j8 + 3]);
  }
}

// MODE 0: forward only, 1: forward + VJP on a list of rows, 2: whole-horizon rollout (forward + VJP + ranking + step, H times)
//
// HM ("half M"): the MMAs run with M = 128 over the CTA pair -- 64 rows per CTA -- instead of 256.  tcgen05's issue
// floor is max(M, 128) N / 512 cycles per K = 16 step at cta_group::2, so a half tile takes half the tensor-pipe time
// (tools/tcx_m128_microbench.cu: 3076 instead of 6148 cycles per split K = 256 layer), and each epilogue thread has
// half the columns: a rollout that is latency-bound on ONE tile per step (planar robots, the control tick, the
// planner's 40 samples) steps in little more than half the time, on twice the CTA pairs.  The accumulator of an
// M = 128 pair MMA uses the "2 x 2" layout: TMEM lanes 0-63 hold the CTA's 64 rows x the first N / 2 columns, lanes
// 64-127 the same rows x the second N / 2 -- which are the output features of CTA rank 0's / rank 1's half of B.  So a
// row has FOUR epilogue threads (lane half fb = feature block, warp half h = 32-column chunk) instead of two, each
// hands over ONE 32-column chunk per N half, and K quarter 2 x + fb of the next operand is complete after 8 (not 16)
// warp arrivals.  Everything else -- weight images, stage order, arithmetic per element -- is the same, so HM results
// are bitwise equal to the full-tile kernel.
//
// MOVE (whole-horizon mode only): constant-velocity obstacles -- step t encodes and re-scores obstacle j at
// obstacle_at(a.obs, a.vel, j, c, (t - 1) dt).  A separate instantiation: the static kernels are compiled as without it.
template <int MODE, bool HM = false, bool MOVE = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1) tc_exact_kernel(TxArgs a) {
  constexpr bool BWD = MODE >= 1;
  constexpr int RPC = HM ? 64 : TROWS;                 // rows per CTA per tile
  constexpr uint32_t ALBO = RPC * 16;                  // bytes between consecutive 8-element K chunks of the A images
  constexpr uint32_t DHALF = HM ? 64 : 128;            // TMEM columns of one N = 128 accumulator half
  constexpr uint32_t D2B = HM ? 128 : 256;             // first TMEM column of D2
  static_assert(!HM || MODE == 2, "half tiles are built for the whole-horizon mode");
  static_assert(!MOVE || MODE == 2, "the per-step launches take the step's obstacle positions in a.obs");
  extern __shared__ __align__(1024) uint8_t smem[];
  const int n_rows = MODE == 2 ? a.sa.N * a.M : (a.src.n_rows_dev ? min(*a.src.n_rows_dev, a.src.n_rows) : a.src.n_rows);
  const int n_tiles = MODE == 2 ? (a.sa.N + 2 * a.S - 1) / (2 * a.S) : (n_rows + 2 * RPC - 1) / (2 * RPC);
  const int n_steps = MODE == 2 ? a.sa.H : 1;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  if (pair >= n_tiles) return;               // both CTAs of the pair leave together, before any allocation

  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + OFF_BAR;
  auto BAR = [&](int i) { return bar0 + (uint32_t)i * 8u; };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEMPTR);
  int* lst = reinterpret_cast<int*>(smem + OFF_LST);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  int pcount = 0;
  (void)pcount;
  constexpr int NG = BWD ? 9 : 5;            // GEMMs per tile
  constexpr int NST = BWD ? STAGES_BWD : STAGES_FWD;

  if (MODE != 2 && blockIdx.x == 0 && tid == 0) *a.fix_next = 0;
  if (tid < 16) reinterpret_cast<float*>(smem + OFF_B4)[tid] = tid < a.net.O ? a.net.b[4][tid] : 0.f;
  if (warp == W_MMA) {
    if (lane == 0) {
      for (int s = 0; s < NSLOT; ++s) {
        mbar_init(BAR(BAR_FULL + s), 1);     // the loader's expect_tx arrival (+ the bytes)
        mbar_init(BAR(BAR_PEER + s), 1);     // leader only: the peer's relay
        mbar_init(BAR(BAR_EMPTY + s), 1);    // tcgen05.commit
      }
      // leader only: 8 epilogue warps x 2 CTAs (half tiles: the 4 warps of the quarter's feature block x 2 CTAs)
      for (int q = 0; q < 4; ++q) mbar_init(BAR(BAR_AREADY0 + q), HM ? 8 : 16);
      mbar_init(BAR(BAR_DFULL0), 1);         // tcgen05.commit
      mbar_init(BAR(BAR_DFULL1), 1);
      mbar_init(BAR(BAR_AFREE), 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc_512_2cta(smem_u32((const void*)tmem_ptr_smem));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  cluster_sync_all();                        // barrier inits visible cluster-wide before any remote arrival

  if (warp < W_MMA) {
    // =================================== epilogue warps ===================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(EPI_REGS));
    const int q4 = warp & 3, h = warp >> 2;
    const int fb = HM ? (q4 >> 1) : 0;                      // half tiles: which 64-feature block of an N half
    const int row = HM ? ((q4 & 1) * 32 + lane) : (q4 * 32 + lane);   // row within the CTA's tile (full tiles: == TMEM lane)
    const uint32_t tD = tmem_base + ((uint32_t)(q4 * 32) << 16);
    uint8_t* a_hi = smem + OFF_AHI + row * 16;
    uint8_t* a_lo = smem + OFF_ALO + row * 16;
    const NetDev& net = a.net;
    const int d = net.d, nin = net.nin, nenc = net.nenc, O = net.O;
    uint32_t d0count = 0, d1count = 0, afcount = 0;         // accumulator halves / operand releases this thread has consumed
    // this thread's columns inside N half x: chunk c = [128 x + 64 c + 32 h, + 32), c = 0, 1 -- interleaved between the
    // two warps of a lane quarter so that K quarter 2 x + c of the next operand is complete when both have stored chunk c
    const int cb = 32 * h;

    auto signal_a = [&](int quarter) {                      // K quarter of the next A operand (or nothing) is in place
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(BAR(BAR_AREADY0 + quarter), 0);
    };
    auto wait_d0 = [&]() {
      mbar_wait(BAR(BAR_DFULL0), d0count & 1);
      ++d0count;
      tc_fence_after();
    };
    auto wait_d1 = [&]() {
      mbar_wait(BAR(BAR_DFULL1), d1count & 1);
      ++d1count;
      tc_fence_after();
    };
    auto wait_afree = [&]() {
      mbar_wait(BAR(BAR_AFREE), afcount & 1);
      ++afcount;
      tc_fence_after();
    };

    // ---- encoded inputs [x, sin x, cos x], split, K = 32 (network_macros_mod.py:139-140).  The two warps of a lane
    //      quarter share a row: h = 0 encodes the joint angles (and keeps sin / cos for the Jacobian), h = 1 the obstacle
    //      point and the zero padding -- every one of the 32 operand columns is written exactly once.  The values of the
    //      NEXT tile are prepared in registers while the last GEMM of the current one runs (rows looked up and their
    //      inputs prefetched one GEMM earlier), so the tile boundary itself only stores them.
    uint32_t en_v[3 * MAXD];                                // element: fp16 hi | fp16 lo << 16
    float en_sn[MAXD], en_cs[MAXD], en_rad = 0.f;
    uint32_t en_range = 0;
    int en_i = 0, en_j = 0;
    bool en_valid = false;
    float en_tau = 0.f;                                     // MOVE: time of the step being encoded
    auto enc_compute = [&](int i, int j, bool valid, const float* qsrc, int qstride) {
      en_i = i; en_j = j; en_valid = valid; en_range = 0;
      if (HM && fb != 0) return;                            // a row's encoding is written by its fb == 0 threads
      auto prep = [&](float v) -> uint32_t {                // saturating like split8, and range-checked
        const uint32_t hh = pack_h2(v, 0.f);
        const uint32_t ll = pack_h2((v - unpack_h2(hh).x) * SPLIT, 0.f);
        en_range = __vmaxu2(en_range, hh & 0x7fff7fffu);
        return (hh & 0xffffu) | (ll << 16);
      };
      if (h == 0) {
        float xq[MAXD];
#pragma unroll
        for (int c = 0; c < MAXD; ++c) {
          xq[c] = (c < d && valid) ? qsrc[(size_t)i * qstride + c] : 0.f;
          en_sn[c] = 0.f; en_cs[c] = 1.f;
        }
        en_rad = valid ? a.obs[j * 4 + 3] : 0.f;
        // a rolled loop over the joints (the arrays it indexes live in local memory): seven inlined sincosf + 21 splits
        // are ~1000 instructions of straight-line code, and at the step boundary of the whole-horizon kernel this
        // runs un-overlapped on warps that are bound by instruction fetch
#pragma unroll
        for (int c = 0; c < MAXD; ++c) {
          if (c < d) {
            float sn_, cs_;
            sincosf(xq[c], &sn_, &cs_);                     // same bits as sinf / cosf (tools/tcx_regress.py)
            en_sn[c] = sn_; en_cs[c] = cs_;
            en_v[3 * c] = prep(xq[c]); en_v[3 * c + 1] = prep(sn_); en_v[3 * c + 2] = prep(cs_);
          }
        }
      } else {
        float xp[3];                                        // nin - d obstacle coordinates: 3, or 2 for the toy variant
#pragma unroll
        for (int c = 0; c < 3; ++c)
          xp[c] = (valid && d + c < nin) ? obstacle_at(a.obs, MOVE ? a.vel : nullptr, j, c, en_tau) : 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c)
          if (d + c < nin) {
            float sp, cp;
            sincosf(xp[c], &sp, &cp);
            en_v[3 * c] = prep(xp[c]); en_v[3 * c + 1] = prep(sp); en_v[3 * c + 2] = prep(cp);
          }
      }
    };
    auto enc_store = [&]() {
      if (HM && fb != 0) return;
      auto st = [&](int e, uint32_t v) {
        const int off = (e >> 3) * ALBO + (e & 7) * 2;
        *reinterpret_cast<uint16_t*>(a_hi + off) = (uint16_t)v;
        *reinterpret_cast<uint16_t*>(a_lo + off) = (uint16_t)(v >> 16);
      };
      if (h == 0) {
#pragma unroll
        for (int c = 0; c < MAXD; ++c)
          if (c < d) { st(c, en_v[3 * c]); st(nin + c, en_v[3 * c + 1]); st(2 * nin + c, en_v[3 * c + 2]); }
      } else {
#pragma unroll
        for (int c = 0; c < 3; ++c)
          if (d + c < nin) { st(d + c, en_v[3 * c]); st(nin + d + c, en_v[3 * c + 1]); st(2 * nin + d + c, en_v[3 * c + 2]); }
        for (int e = 3 * nin; e < 32; ++e) st(e, 0u);
      }
    };
    int nx_i = 0, nx_j = 0;
    bool nx_valid = false;
    auto lookup_tile = [&](int tl) {
      if (tl < n_tiles) {
        nx_valid = row_lookup(a.src, tl * (2 * RPC) + (int)rank * RPC + row, n_rows, nx_i, nx_j);
        if (nx_valid) {
          asm volatile("prefetch.global.L1 [%0];" ::"l"(a.q + (size_t)nx_i * a.q_stride));
          asm volatile("prefetch.global.L1 [%0];" ::"l"(a.obs + nx_j * 4));
        }
      }
    };
    if (MODE != 2) {
      lookup_tile(pair);
      if (TCX_ENC_PIPE) enc_compute(nx_i, nx_j, nx_valid, a.q, a.q_stride);
    }
    uint32_t pass = 0;                                      // (tile, step) passes done: locates the output layer's stage
    float qlane[TROWS / 32] = {0.f, 0.f, 0.f, 0.f};         // whole-horizon kernel, lane-parallel step: this lane's joint
    static_assert(TROWS == 128, "four batches of 32 sample slots");
    float qreg[MAXD];                                       // whole-horizon kernel: the state of this thread's sample
#pragma unroll
    for (int c = 0; c < MAXD; ++c) qreg[c] = 0.f;
    bool enc_stored = false;

    for (int tile = pair; tile < n_tiles; tile += npairs)
    for (int t = 1; t <= n_steps; ++t, ++pass) {
      // global row of this thread: consecutive rows of the list, or (whole-horizon) row j of sample i = dense row i * M + j
      int grow = tile * (2 * RPC) + (int)rank * RPC + row;
      const float* qsrc = MODE == 2 ? a.sa.traj + (size_t)(t - 1) * d : a.q;     // q_prev = all_traj[:, t-1, :]
      const int qstride = MODE == 2 ? a.sa.H * d : a.q_stride;
      float* stg = reinterpret_cast<float*>(smem + OFF_STAGE);
      if (MODE == 2) {                                      // the state was written by the step just before: encode now
        const int sl = row / a.M;
        const int tj = row - sl * a.M;
        const int ti = (tile * 2 + (int)rank) * a.S + sl;
        const bool tv = sl < a.S && ti < a.sa.N;
        grow = tv ? ti * a.M + tj : n_rows;
        if (MOVE) en_tau = __fmul_rn((float)(t - 1), a.sa.dt);
        if (t == 1) enc_compute(ti, tj, tv, qsrc, qstride);
        else enc_compute(sl, tj, tv, stg + STG_Q, MAXD);    // ... and handed over in shared memory: no L2 round trip
      } else if (!TCX_ENC_PIPE) {
        enc_compute(nx_i, nx_j, nx_valid, qsrc, qstride);
      }
      // MODE 2: the rows never leave the SM (they are workspace, not outputs of the rollout)
      float* out_m = MODE == 2 ? stg + STG_M : a.out_m;
      float* out_dist = MODE == 2 ? stg + STG_DIST : a.out_dist;
      float* out_grad = MODE == 2 ? stg + STG_GRAD : a.out_grad;
      const int orow = MODE == 2 ? row : grow;              // where this row's results go
      float sn[MAXD], cs[MAXD];
#pragma unroll
      for (int c = 0; c < MAXD; ++c) { sn[c] = en_sn[c]; cs[c] = en_cs[c]; }
      const float rad = en_rad;
      uint32_t mk[4][4];    // sign bits of the pre-activations (set = ReLU off): layer x 32-column chunk, column 0 in bit 31
      uint32_t range = en_range;                            // largest fp16 magnitude written to the A operand
      const int row_i = en_i, row_j = en_j;
      int* ovf = reinterpret_cast<int*>(smem + OFF_OVF);
      if (h == 0 && fb == 0) ovf[row] = 0;
      if (MODE == 2 || !enc_stored) {                       // otherwise stored at the end of the previous tile
        enc_store();
        if (!HM || fb == 0) signal_a(0);                    // (K = 32 operand: quarter 0 only)
      }
      if (q4 == 0) TCX_PROF(h, 1);
      // this row's results stay in registers until the tile's last hand-over is out: a global store ahead of a
      // fence.proxy.async (MEMBAR.ALL.CTA) would put its round trip on the critical path
      float o_m = 0.f, o_dist = 0.f, o_g[MAXD];

      // ---- hidden layers: h = relu(W h + b), masks kept for the backward pass.  N half 0 is converted under the MMAs
      //      of N half 1 and parked in registers until they retire (they read the operand being replaced); N half 1 is
      //      converted under the next layer's first K half.  Every 64 finished columns are handed over at once.
#pragma unroll 1
      for (int l = 0; l < 4; ++l) {
        const float* bl = net.b[l] + cb;
        const float comp = (a.dbg & 4) ? 0.f : comp_of(a.comp, l);
        if constexpr (HM) {
          // one 32-column chunk per N half: features 128 x + 64 fb + 32 h + [0, 32) -> K quarter 2 x + fb
          wait_d0();
          {
            uint32_t hh0[16], hl0[16];
            {
              uint32_t r1[32], r2[32];
              tmem_ld32(tD + cb, r1);
              tmem_ld32(tD + D2B + cb, r2);
              tc_wait_ld();
              mk[l][0] = fwd_chunk32(r1, r2, bl + 64 * fb, comp, hh0, hl0, range);
            }
            wait_afree();
            store_chunk32<ALBO>(a_hi, a_lo, 8 * fb + 4 * h, hh0, hl0);
            signal_a(fb);
          }
          wait_d1();
          {
            uint32_t r1[32], r2[32], hw[16], lw[16];
            tmem_ld32(tD + DHALF + cb, r1);
            tmem_ld32(tD + D2B + DHALF + cb, r2);
            tc_wait_ld();
            mk[l][1] = fwd_chunk32(r1, r2, bl + 128 + 64 * fb, comp, hw, lw, range);
            store_chunk32<ALBO>(a_hi, a_lo, 16 + 8 * fb + 4 * h, hw, lw);
          }
          signal_a(2 + fb);
          continue;
        }
        wait_d0();
        if (q4 == 0) TCX_PROF(h, 10 + l);
        {
          uint32_t hh0[16], hl0[16], hh1[16], hl1[16];
          {                                                   // one chunk at a time: this half hides under MMAs,
            uint32_t r1[32], r2[32];                          // registers are what is scarce (64 stay parked)
            tmem_ld32(tD + cb, r1);
            tmem_ld32(tD + 256 + cb, r2);
            tc_wait_ld();
            mk[l][0] = fwd_chunk32(r1, r2, bl, comp, hh0, hl0, range);
            tmem_ld32(tD + 64 + cb, r1);
            tmem_ld32(tD + 320 + cb, r2);
            tc_wait_ld();
            mk[l][1] = fwd_chunk32(r1, r2, bl + 64, comp, hh1, hl1, range);
          }
          if (q4 == 0) TCX_PROF(h, 20 + l);
          wait_afree();
          store_chunk32<ALBO>(a_hi, a_lo, 4 * h, hh0, hl0);
          signal_a(0);
          store_chunk32<ALBO>(a_hi, a_lo, 8 + 4 * h, hh1, hl1);
          signal_a(1);
        }
        if (q4 == 0) TCX_PROF(h, 40 + l);
        wait_d1();
        if (q4 == 0) TCX_PROF(h, 30 + l);
        {
          uint32_t r1[2][32], r2[2][32], hw[16], lw[16];
          tmem_ld32(tD + 128 + cb, r1[0]);
          tmem_ld32(tD + 384 + cb, r2[0]);
          tc_wait_ld();
          tmem_ld32(tD + 192 + cb, r1[1]);
          tmem_ld32(tD + 448 + cb, r2[1]);
          mk[l][2] = fwd_chunk32(r1[0], r2[0], bl + 128, comp, hw, lw, range);
          store_chunk32<ALBO>(a_hi, a_lo, 16 + 4 * h, hw, lw);
          signal_a(2);
          tc_wait_ld();
          mk[l][3] = fwd_chunk32(r1[1], r2[1], bl + 192, comp, hw, lw, range);
          store_chunk32<ALBO>(a_hi, a_lo, 24 + 4 * h, hw, lw);
        }
        signal_a(3);
        if (q4 == 0) TCX_PROF(h, 50 + l);
      }

      if (MODE != 2) {
        lookup_tile(tile + npairs);
        if (TCX_ENC_PIPE && !BWD && tile + npairs < n_tiles) enc_compute(nx_i, nx_j, nx_valid, a.q, a.q_stride);
      }
      // ---- output layer (no activation): links 0..15 sit in D columns 0..15
      wait_d0();
      if (q4 == 0) TCX_PROF(h, 60);
      if (h == 0 && fb == 0) {
        uint32_t r1[16], r2[16];
        tmem_ld16(tD, r1);
        tmem_ld16(tD + D2B, r2);
        tc_wait_ld();
        if (q4 == 0) TCX_PROF(h, 64);
        // straight-line; the links the network does not have (o >= O, a launch-wide constant: uniform branches) are
        // skipped -- their IEEE divisions were half of this epilogue for the 7- and 9-link networks
        const float comp_o = (a.dbg & 4) ? 0.f : a.comp[4];
        const float* b4s = reinterpret_cast<const float*>(smem + OFF_B4);
        const bool scaled = net.scale != 1.f;
        float v[16];
#pragma unroll
        for (int o = 0; o < 16; ++o)
          if (o < O) v[o] = combine(r1[o], r2[o], comp_o) + b4s[o];
        int best = 0;
        float bv = v[0], m = 3.0e38f;
#pragma unroll
        for (int o = 1; o < 16; ++o) {                        // argmin of the RAW output (robot_sdf.py:155)
          if (o < O) {
            const bool lt = v[o] < bv;
            bv = lt ? v[o] : bv;
            best = lt ? o : best;
          }
        }
#pragma unroll
        for (int o = 0; o < 16; ++o) {                        // MPPI.py:236-242: /100, minus radius, ignored := 1e6
          if (o < O) {
            float y = scaled ? v[o] / 100.f : v[o];
            y -= rad;
            if ((a.ignore_mask >> o) & 1u) y = 1e6f;
            m = fminf(m, y);
          }
        }
        o_m = m;
        if (BWD) {
          float y = bv;                                       // pass-2 distance of the argmin link (MPPI.py:265-274)
          if (net.scale != 1.f) y = y / 100.f;
          o_dist = y - rad;
        }
        if (!TCX_DEFER_STG && MODE != 2 && grow < n_rows) {
          if (out_m) out_m[grow] = o_m;
          if (BWD) out_dist[grow] = o_dist;
        }
        if (BWD) lst[row] = best;
        if (q4 == 0) TCX_PROF(h, 65);
      }
      if constexpr (BWD) {
        asm volatile("bar.sync 1, 256;" ::: "memory");      // lst visible to the column-half-1 warps
        if (q4 == 0) TCX_PROF(h, 66);
        // ---- g4 = W5[l*, :] * s4, handed over quarter by quarter.  The split rows of W5 are read from the weight stage
        //      of the output layer, which the issuer keeps in its ring slot until the first quarter is signalled: in the
        //      canonical K-major layout the 8 columns of chunk ch of link l* are exactly one 16-byte core-matrix row
        {
          const int ls = lst[row];
          const uint32_t slot4 = (pass * (uint32_t)NST + 14u) % NSLOT;
          const uint8_t* wrow = smem + OFF_RING + slot4 * SLOT_BYTES + ls * 16;
          if constexpr (HM) {
            // this thread's two chunks: K quarters fb and 2 + fb (the columns whose ReLU bits it holds in mk[3][0 / 1])
            uint4 whi[8], wlo[8];
#pragma unroll
            for (int cc = 0; cc < 2; ++cc)
#pragma unroll
              for (int j8 = 0; j8 < 4; ++j8) {
                const int ch = 8 * (2 * cc + fb) + 4 * h + j8;
                whi[4 * cc + j8] = *reinterpret_cast<const uint4*>(wrow + ch * 256);
                wlo[4 * cc + j8] = *reinterpret_cast<const uint4*>(wrow + 8192 + ch * 256);
              }
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
              const int c = 2 * cc + fb;
              const uint32_t bits = mk[3][cc];
#pragma unroll
              for (int j8 = 0; j8 < 4; ++j8) {
                const int ch = 8 * c + 4 * h + j8;
                uint4 hi = whi[4 * cc + j8], lo = wlo[4 * cc + j8];
                const uint32_t on = ~(bits >> (24 - 8 * j8));
                const uint32_t m0 = ((on >> 7) & 1u) * 0xffffu + ((on >> 6) & 1u) * 0xffff0000u;
                const uint32_t m1 = ((on >> 5) & 1u) * 0xffffu + ((on >> 4) & 1u) * 0xffff0000u;
                const uint32_t m2 = ((on >> 3) & 1u) * 0xffffu + ((on >> 2) & 1u) * 0xffff0000u;
                const uint32_t m3 = ((on >> 1) & 1u) * 0xffffu + (on & 1u) * 0xffff0000u;
                hi.x &= m0; hi.y &= m1; hi.z &= m2; hi.w &= m3;
                lo.x &= m0; lo.y &= m1; lo.z &= m2; lo.w &= m3;
                *reinterpret_cast<uint4*>(a_hi + ch * ALBO) = hi;
                *reinterpret_cast<uint4*>(a_lo + ch * ALBO) = lo;
              }
              signal_a(c);
            }
          } else {
          uint4 whi[16], wlo[16];
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              const int ch = 8 * c + 4 * h + j8;
              whi[4 * c + j8] = *reinterpret_cast<const uint4*>(wrow + ch * 256);
              wlo[4 * c + j8] = *reinterpret_cast<const uint4*>(wrow + 8192 + ch * 256);
            }
          if (q4 == 0) TCX_PROF(h, 67);
#pragma unroll
          for (int c = 0; c < 4; ++c) {                       // c = 2 x + chunk: N half x, 32-column chunk of this thread
            const uint32_t bits = mk[3][c];
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
              const int ch = 8 * c + 4 * h + j8;
              uint4 hi = whi[4 * c + j8], lo = wlo[4 * c + j8];
              const uint32_t on = ~(bits >> (24 - 8 * j8));     // column 8 j8 + j of this chunk sits in bit 7 - j
              const uint32_t m0 = ((on >> 7) & 1u) * 0xffffu + ((on >> 6) & 1u) * 0xffff0000u;
              const uint32_t m1 = ((on >> 5) & 1u) * 0xffffu + ((on >> 4) & 1u) * 0xffff0000u;
              const uint32_t m2 = ((on >> 3) & 1u) * 0xffffu + ((on >> 2) & 1u) * 0xffff0000u;
              const uint32_t m3 = ((on >> 1) & 1u) * 0xffffu + (on & 1u) * 0xffff0000u;
              hi.x &= m0; hi.y &= m1; hi.z &= m2; hi.w &= m3;
              lo.x &= m0; lo.y &= m1; lo.z &= m2; lo.w &= m3;
              *reinterpret_cast<uint4*>(a_hi + ch * ALBO) = hi;
              *reinterpret_cast<uint4*>(a_lo + ch * ALBO) = lo;
            }
            signal_a(c);
            if (q4 == 0 && c == 0) TCX_PROF(h, 68);
          }
        }
          }
        if (q4 == 0) TCX_PROF(h, 61);

        // ---- g_{l-1} = (W_l^T g_l) * s_{l-1},  l = 3, 2, 1 (same half-by-half schedule as the forward layers)
#pragma unroll 1
        for (int l = 3; l >= 1; --l) {
          const float comp = (a.dbg & 4) ? 0.f : comp_of(a.comp, 8 - l);
          if constexpr (HM) {
            wait_d0();
            {
              uint32_t hh0[16], hl0[16];
              {
                uint32_t r1[32], r2[32];
                tmem_ld32(tD + cb, r1);
                tmem_ld32(tD + D2B + cb, r2);
                tc_wait_ld();
                bwd_chunk32(r1, r2, mk[l - 1][0], comp, hh0, hl0, range);
              }
              wait_afree();
              store_chunk32<ALBO>(a_hi, a_lo, 8 * fb + 4 * h, hh0, hl0);
              signal_a(fb);
            }
            wait_d1();
            {
              uint32_t r1[32], r2[32], hw[16], lw[16];
              tmem_ld32(tD + DHALF + cb, r1);
              tmem_ld32(tD + D2B + DHALF + cb, r2);
              tc_wait_ld();
              bwd_chunk32(r1, r2, mk[l - 1][1], comp, hw, lw, range);
              store_chunk32<ALBO>(a_hi, a_lo, 16 + 8 * fb + 4 * h, hw, lw);
            }
            signal_a(2 + fb);
            continue;
          }
          wait_d0();
          if (q4 == 0) TCX_PROF(h, 14 + l);
          {
            uint32_t hh0[16], hl0[16], hh1[16], hl1[16];
            {
              uint32_t r1[32], r2[32];
              tmem_ld32(tD + cb, r1);
              tmem_ld32(tD + 256 + cb, r2);
              tc_wait_ld();
              bwd_chunk32(r1, r2, mk[l - 1][0], comp, hh0, hl0, range);
              tmem_ld32(tD + 64 + cb, r1);
              tmem_ld32(tD + 320 + cb, r2);
              tc_wait_ld();
              bwd_chunk32(r1, r2, mk[l - 1][1], comp, hh1, hl1, range);
            }
            if (q4 == 0) TCX_PROF(h, 24 + l);
            wait_afree();
            store_chunk32<ALBO>(a_hi, a_lo, 4 * h, hh0, hl0);
            signal_a(0);
            store_chunk32<ALBO>(a_hi, a_lo, 8 + 4 * h, hh1, hl1);
            signal_a(1);
          }
          if (q4 == 0) TCX_PROF(h, 44 + l);
          wait_d1();
          if (q4 == 0) TCX_PROF(h, 34 + l);
          {
            uint32_t r1[2][32], r2[2][32], hw[16], lw[16];
            tmem_ld32(tD + 128 + cb, r1[0]);
            tmem_ld32(tD + 384 + cb, r2[0]);
            tc_wait_ld();
            tmem_ld32(tD + 192 + cb, r1[1]);
            tmem_ld32(tD + 448 + cb, r2[1]);
            bwd_chunk32(r1[0], r2[0], mk[l - 1][2], comp, hw, lw, range);
            store_chunk32<ALBO>(a_hi, a_lo, 16 + 4 * h, hw, lw);
            signal_a(2);
            tc_wait_ld();
            bwd_chunk32(r1[1], r2[1], mk[l - 1][3], comp, hw, lw, range);
            store_chunk32<ALBO>(a_hi, a_lo, 24 + 4 * h, hw, lw);
          }
          signal_a(3);
          if (q4 == 0) TCX_PROF(h, 54 + l);
        }

        if (TCX_ENC_PIPE && MODE != 2 && tile + npairs < n_tiles) enc_compute(nx_i, nx_j, nx_valid, a.q, a.q_stride);
        // ---- a = W_1^T g_1 (N = 32), then the encoding Jacobian dz/dx_c = a[c] + cos(x_c) a[nin+c] - sin(x_c) a[2nin+c]
        wait_d0();
        if (q4 == 0) TCX_PROF(h, 62);
        if constexpr (HM) {
          // N = 32 over the pair: a[0..15] (rank 0's rows of B) sit on lanes 0-63, a[16..31] on lanes 64-127 -- the
          // row's two h == 0 threads each put their sixteen into the scratch, then the fb == 0 one applies the Jacobian
          if (h == 0) {
            uint32_t r1[16], r2[16];
            tmem_ld16(tD, r1);
            tmem_ld16(tD + D2B, r2);
            tc_wait_ld();
            float* scr = reinterpret_cast<float*>(smem + OFF_SCRATCH) + row;
#pragma unroll
            for (int e = 0; e < 16; ++e) scr[(16 * fb + e) * TROWS] = combine(r1[e], r2[e], (a.dbg & 4) ? 0.f : a.comp[8]);
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (h == 0 && fb == 0) {
            const float* scr = reinterpret_cast<const float*>(smem + OFF_SCRATCH) + row;
#pragma unroll
            for (int c = 0; c < MAXD; ++c)
              if (c < d) o_g[c] = scr[c * TROWS] + cs[c] * scr[(nin + c) * TROWS] - sn[c] * scr[(2 * nin + c) * TROWS];
          }
        } else if (h == 0) {
          uint32_t r1[32], r2[32];
          tmem_ld32(tD, r1);
          tmem_ld32(tD + 256, r2);
          tc_wait_ld();
          float* scr = reinterpret_cast<float*>(smem + OFF_SCRATCH) + row;     // a[e] at scr[e * 128]
#pragma unroll
          for (int e = 0; e < 32; ++e) scr[e * TROWS] = combine(r1[e], r2[e], (a.dbg & 4) ? 0.f : a.comp[8]);
#pragma unroll
          for (int c = 0; c < MAXD; ++c)
            if (c < d) o_g[c] = scr[c * TROWS] + cs[c] * scr[(nin + c) * TROWS] - sn[c] * scr[(2 * nin + c) * TROWS];
          if (!TCX_DEFER_STG && MODE != 2 && grow < n_rows) {
#pragma unroll
            for (int c = 0; c < MAXD; ++c)
              if (c < d) out_grad[(size_t)grow * d + c] = o_g[c];
          }
        }
      }
      (void)nenc;
      int* fixn = reinterpret_cast<int*>(smem + OFF_FIXN);
      int* fixl = reinterpret_cast<int*>(smem + OFF_FIXL);
      if constexpr (MODE == 1) {
        // ---- rows whose activations or gradients saturated fp16 are re-scored in IEEE FFMA right here (round 1 queued
        //      them for a launch of their own after this one -- an empty launch per rollout step in the normal case):
        //      the FFMA tile of exact_mlp.cu on warps 0-3, its shared memory carved out of the A operand images, which
        //      are idle between this tile's last GEMM and the hand-over of the next tile's encoding
        if (((range & 0xffffu) >= 0x7bffu) || ((range >> 16) >= 0x7bffu)) ovf[row] = 1;
        if (tid == 0) *fixn = 0;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (h == 0 && fb == 0 && grow < n_rows && ovf[row]) {
          const int k = atomicAdd(fixn, 1);
          atomicAdd(a.fix_total, 1);
          fixl[k] = row_i;
          fixl[TROWS + k] = row_j;
          fixl[2 * TROWS + k] = grow;            // re-scored straight into the output rows
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const int nfix = *fixn;
        if (nfix > 0) {
          if (tid < exact_tile::nthreads(8)) {
            exact_tile::TileSmem<8> ts(reinterpret_cast<float*>(smem + OFF_AHI));
            exact_tile::WeightStream<> ws;
            const int passes = (nfix + 31) / 32;
            exact_tile::stream_begin<true, exact_tile::nthreads(8)>(ws, &a.net, ts.ring, passes);
            RowSrc fs{};
            fs.mode = ROWS_LIST;
            fs.M = a.src.M;
            fs.n_rows = nfix;
            fs.row_sample = fixl;
            fs.row_obs = fixl + TROWS;
            fs.out_row = fixl + 2 * TROWS;
            int stage = 0;
            for (int r0 = 0; r0 < nfix; r0 += 32) {
              exact_tile::mlp_tile<true, 8, 8>(a.net, fs, r0, nfix, a.q, a.q_stride, a.obs, nullptr, 0.f, a.ignore_mask,
                                              a.out_m, a.out_dist, a.out_grad, ts, ws, stage);
              exact_tile::tile_sync<exact_tile::nthreads(8)>();
            }
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
      }
      // ---- tile end: the next tile's encoding (prepared above) goes out first, then this tile's rows
      if (TCX_ENC_PIPE && MODE != 2 && tile + npairs < n_tiles) {
        enc_store();
        signal_a(0);
        enc_stored = true;
      } else {
        enc_stored = false;
      }
      if ((TCX_DEFER_STG || MODE == 2) && h == 0 && fb == 0 && grow < n_rows && !(MODE == 1 && ovf[row])) {
        if (out_m) out_m[orow] = o_m;
        if (BWD) {
          out_dist[orow] = o_dist;
#pragma unroll
          for (int c = 0; c < MAXD; ++c)
            if (c < d) out_grad[(size_t)orow * d + c] = o_g[c];
        }
      }
      if (q4 == 0) TCX_PROF(h, 63);
      // ---- rows whose activations saturated fp16 are handed to the FFMA arithmetic (forward-only launches: a
      //      device-wide list re-scored by launch_exact_fixup; whole-horizon: this CTA's list, re-scored below)
      if constexpr (MODE != 1) {
      if (((range & 0xffffu) >= 0x7bffu) || ((range >> 16) >= 0x7bffu)) ovf[row] = 1;
      if (MODE == 2 && tid == 0) *fixn = 0;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (h == 0 && fb == 0 && grow < n_rows && ovf[row]) {
        if (MODE != 2) {                       // device-wide list, re-scored by launch_exact_fixup after this kernel
          const int k = atomicAdd(a.fix_count, 1);
          atomicAdd(a.fix_total, 1);
          if (k < a.fix_cap) {
            a.fix_list[k] = row_i;
            a.fix_list[a.fix_cap + k] = row_j;
            a.fix_list[2 * a.fix_cap + k] = grow;
          } else {
            atomicAdd(a.fix_dropped, 1);
          }
        } else {                               // this CTA's list, re-scored right here before the step needs the rows
          const int k = atomicAdd(fixn, 1);
          atomicAdd(a.fix_total, 1);
          fixl[k] = row_i;
          fixl[TROWS + k] = row_j;
          fixl[2 * TROWS + k] = row;           // re-scored into the staged rows
        }
      }
      }
      if constexpr (MODE == 2) {
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (q4 == 0) TCX_PROF(h, 80);
        const int nfix = *fixn;
        if (nfix > 0 && tid < exact_tile::nthreads(8)) {
          // the FFMA tile of exact_mlp.cu on warps 0-3, its shared memory carved out of the (idle) A operand images
          exact_tile::TileSmem<8> ts(reinterpret_cast<float*>(smem + OFF_AHI));
          exact_tile::WeightStream<> ws;
          const int passes = (nfix + 31) / 32;
          exact_tile::stream_begin<true, exact_tile::nthreads(8)>(ws, &a.net, ts.ring, passes);
          RowSrc fs{};
          fs.mode = ROWS_LIST;
          fs.M = a.M;
          fs.n_rows = nfix;
          fs.row_sample = fixl;
          fs.row_obs = fixl + TROWS;
          fs.out_row = fixl + 2 * TROWS;
          int stage = 0;
          for (int r0 = 0; r0 < nfix; r0 += 32) {
            exact_tile::mlp_tile<true, 8, 8>(a.net, fs, r0, nfix, qsrc, qstride, a.obs, MOVE ? a.vel : nullptr, en_tau,
                                            a.ignore_mask, out_m, out_dist, out_grad, ts, ws, stage);
            exact_tile::tile_sync<exact_tile::nthreads(8)>();
          }
        }
        if (nfix > 0) asm volatile("bar.sync 1, 256;" ::: "memory");
        // ---- the K closest obstacles of every sample, ascending by (masked distance, obstacle index)
        //      (MPPI.py:243-247).  With more than a handful of obstacles a warp per sample, lanes over the obstacles:
        //      K serial passes over M = 28 rows on the step thread were 1.4 k instructions -- a third of a control
        //      tick's kernel time.  Same selection as the serial form below (lowest index among equal values).
        const bool warp_rank = a.M > 8;
        if (warp_rank) {
          const int K = a.sa.K, M = a.M;
          for (int sl = warp; sl < a.S; sl += W_MMA) {
            if ((tile * 2 + (int)rank) * a.S + sl >= a.sa.N) break;
            const float* mr = stg + STG_M + sl * M;
            int* rows = reinterpret_cast<int*>(stg + STG_ROWS) + sl * MAXK;
            float last_v = -3.4e38f;
            int last_j = -1;
#pragma unroll 1
            for (int kk = 0; kk < K; ++kk) {
              float bv = 3.4e38f;
              int bj = 0x7fffffff;
              for (int j = lane; j < M; j += 32) {
                const float v = mr[j];
                const bool after = kk == 0 || v > last_v || (v == last_v && j > last_j);
                if (after && (v < bv || (v == bv && j < bj))) { bv = v; bj = j; }
              }
#pragma unroll
              for (int off = 16; off > 0; off >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
                const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
                if (ov < bv || (ov == bv && oj < bj)) { bv = ov; bj = oj; }
              }
              if (bj == 0x7fffffff) bj = last_j < 0 ? 0 : last_j;
              if (lane == 0) rows[kk] = sl * M + bj;
              last_v = bv; last_j = bj;
            }
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        // ---- eight lanes per sample: (ranking of a few obstacles on the first,) then the modulation / policy / Euler
        //      step in its lane-parallel form (step_group_t: a lane per joint / ranked row / policy kernel, bit-identical
        //      to the one-thread step_sample): the step was 13 k of a planar-7 rollout step's 65 k cycles on ONE warp
        if (step_group_supported(a.sa)) {
#pragma unroll
         for (int sb = 0; sb < TROWS / 32; ++sb) {            // 32 sample slots (256 threads) at a time; S <= 128
          if (32 * sb + (warp << 2) < a.S) {                  // warps holding at least one of the CTA's sample slots
            const int g = 32 * sb + (tid >> 3), gl = tid & 7;
            const int i = (tile * 2 + (int)rank) * a.S + g;
            const bool live = g < a.S && i < a.sa.N;
            const int K = a.sa.K, M = a.M;
            int* rows = reinterpret_cast<int*>(stg + STG_ROWS) + (live ? g : 0) * MAXK;
            if (live && gl == 0) {
              asm volatile("prefetch.global.L1 [%0];" ::"l"(a.sa.sigma + (size_t)i * NKMAX));
              for (int b = 0; b < a.sa.nk * d * 4; b += 128) {
                asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.sa.mu + (size_t)i * NKMAX * d) + b));
                asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.sa.alpha + (size_t)i * NKMAX * d) + b));
              }
              const float* mr = stg + STG_M + g * M;
              float last_v = -3.4e38f;
              int last_j = -1;
#pragma unroll 1
              for (int kk = 0; kk < K && !warp_rank; ++kk) {
                float bv = 3.4e38f;
                int bj = -1;
#pragma unroll 1
                for (int j = 0; j < M; ++j) {
                  const float v = mr[j];
                  const bool after = kk == 0 || v > last_v || (v == last_v && j > last_j);
                  if (after && (bj < 0 || v < bv)) { bv = v; bj = j; }
                }
                if (bj < 0) bj = last_j < 0 ? 0 : last_j;
                rows[kk] = g * M + bj;
                last_v = bv; last_j = bj;
              }
            }
            __syncwarp();
            if (tid == 0) TCX_PROF(0, 83);
            if (t == 1) qlane[sb] = (live && gl < d) ? a.sa.traj[(size_t)i * a.sa.H * d + gl] : 0.f;
            const StepIO io{stg + STG_DIST, stg + STG_GRAD, rows, nullptr, live ? stg + STG_Q + g * MAXD : nullptr};
            if (d == 7) step_group_t<7, 8>(a.sa, live ? i : 0, t, io, gl, live, &qlane[sb]);
            else step_group_t<2, 8>(a.sa, live ? i : 0, t, io, gl, live, &qlane[sb]);
          }
         }
        } else if (tid < a.S) {
          const int i = (tile * 2 + (int)rank) * a.S + tid;
          if (i < a.sa.N) {
            const int K = a.sa.K, M = a.M;
            // the sampled policy rows of this sample on their way into L1 while the ranking and the blend run
            asm volatile("prefetch.global.L1 [%0];" ::"l"(a.sa.sigma + (size_t)i * NKMAX));
            for (int b = 0; b < a.sa.nk * d * 4; b += 128) {
              asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.sa.mu + (size_t)i * NKMAX * d) + b));
              asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(a.sa.alpha + (size_t)i * NKMAX * d) + b));
            }
            if (t == 1) {
#pragma unroll
              for (int c = 0; c < MAXD; ++c) qreg[c] = c < d ? a.sa.traj[(size_t)i * a.sa.H * d + c] : 0.f;
            }
            const float* mr = stg + STG_M + tid * M;         // this sample's rows are staged rows tid * M .. + M
            int* rows = reinterpret_cast<int*>(stg + STG_ROWS) + tid * MAXK;   // ranked rows, also in shared memory:
            float last_v = -3.4e38f;                                           // a rolled loop keeps the code short
            int last_j = -1;
#pragma unroll 1
            for (int kk = 0; kk < K && !warp_rank; ++kk) {
              float bv = 3.4e38f;
              int bj = -1;
#pragma unroll 1
              for (int j = 0; j < M; ++j) {
                const float v = mr[j];
                const bool after = kk == 0 || v > last_v || (v == last_v && j > last_j);
                if (after && (bj < 0 || v < bv)) { bv = v; bj = j; }
              }
              if (bj < 0) bj = last_j < 0 ? 0 : last_j;
              rows[kk] = tid * M + bj;
              last_v = bv; last_j = bj;
            }
            if (tid == 0) TCX_PROF(0, 83);
            const StepIO io{stg + STG_DIST, stg + STG_GRAD, rows, qreg, qreg};
            step_sample(a.sa, i, t, io);
#pragma unroll
            for (int c = 0; c < MAXD; ++c)
              if (c < d) stg[STG_Q + tid * MAXD + c] = qreg[c];
          }
        }
        if (q4 == 0) TCX_PROF(h, 81);
        asm volatile("bar.sync 1, 256;" ::: "memory");      // the next state is written before the next encoding reads it
        if (q4 == 0) TCX_PROF(h, 82);
      }
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CTRL_REGS));
  }
  if (warp == W_LOAD) {
    // =================================== weight loader (both CTAs) ===================================
    const uint8_t* img = rank == 0 ? a.img0 : a.img1;
    uint32_t n = 0;
    for (int tile = pair; tile < n_tiles; tile += npairs)
     for (int t = 1; t <= n_steps; ++t)
      for (int s = 0; s < NST; ++s, ++n) {
        const uint32_t slot = n % NSLOT, use = n / NSLOT;
        if (lane == 0) {
          if (use > 0) mbar_wait(BAR(BAR_EMPTY + slot), (use - 1) & 1);
          uint32_t off, bytes;
          stage_info(s, off, bytes);
          mbar_expect_tx(BAR(BAR_FULL + slot), bytes);
          bulk_g2s(sbase + OFF_RING + slot * SLOT_BYTES, img + off, bytes, BAR(BAR_FULL + slot));
        }
        __syncwarp();
      }
  } else if (warp == W_MMA && rank == 1) {
    // =================================== relay (peer CTA): "my half of the stage has landed" ===================
    uint32_t n = 0;
    for (int tile = pair; tile < n_tiles; tile += npairs)
     for (int t = 1; t <= n_steps; ++t)
      for (int s = 0; s < NST; ++s, ++n) {
        const uint32_t slot = n % NSLOT, use = n / NSLOT;
        if (lane == 0) {
          mbar_wait(BAR(BAR_FULL + slot), use & 1);
          mbar_arrive_remote_release(BAR(BAR_PEER + slot), 0);
        }
        __syncwarp();
      }
  } else if (warp == W_MMA) {
    // =================================== MMA issuer (leader CTA) ===================================
    constexpr uint32_t idesc128 = make_idesc(0, HM ? 128 : 256, 128), idesc32 = make_idesc(0, HM ? 128 : 256, 32);
    const uint32_t a_hi = sbase + OFF_AHI, a_lo = sbase + OFF_ALO;
    uint32_t slot = 0, par = 0;                               // ring position of the next weight stage
    uint32_t acount[4] = {0, 0, 0, 0};                        // phases consumed of the four operand-quarter barriers
    uint32_t adh, adl, bdh, bdl, b_step, d1, d2, idesc;       // the open stage: operand descriptors (low words)
    constexpr uint32_t a_step = (2 * ALBO) >> 4;              // one K = 16 step of the A images
    // open a weight stage: its descriptors, then "weights landed in both CTAs" -- all of it before the operand wait, so
    // that nothing but the MMAs themselves follows the moment the epilogue hands a K quarter over
    auto open_stage = [&](uint32_t d_col, uint32_t a_off, uint32_t b_lbo, uint32_t lo_off, uint32_t id) {
      const uint32_t b_base = sbase + OFF_RING + slot * SLOT_BYTES;
      adh = make_desc_lo(a_hi + a_off, ALBO); adl = make_desc_lo(a_lo + a_off, ALBO);
      bdh = make_desc_lo(b_base, b_lbo); bdl = make_desc_lo(b_base + lo_off, b_lbo);
      b_step = (2 * b_lbo) >> 4;
      d1 = tmem_base + d_col; d2 = tmem_base + D2B + d_col;
      idesc = id;
      mbar_wait(BAR(BAR_FULL + slot), par);
      mbar_wait_cluster(BAR(BAR_PEER + slot), par);
      TCX_PROF(2, 100 + (int)d_col + (a_off ? 1 : 0));       // weights landed
    };
    auto wait_a = [&](int q) {                                // K quarter q of the operand is in place
      mbar_wait_cluster(BAR(BAR_AREADY0 + q), acount[q]++ & 1);
      TCX_PROF(2, 92 + q);
    };
    auto steps = [&](int nks, bool first) {                   // nks K = 16 steps of the MMA triple
      tc_fence_after();
      if (elect_one()) {
#pragma unroll 2
        for (int ks = 0; ks < nks; ++ks) {
          const uint32_t acc = (first && ks == 0) ? 0u : 1u;
          mma_ss_2cta_lo(d1, adh, bdh, idesc, acc);          // D1 += A_hi B_hi
          mma_ss_2cta_lo(d2, adh, bdl, idesc, acc);          // D2 += A_hi B_lo
          mma_ss_2cta_lo(d2, adl, bdh, idesc, 1u);           // D2 += A_lo B_hi
          adh += a_step; adl += a_step; bdh += b_step; bdl += b_step;
        }
      }
      __syncwarp();
    };
    uint32_t held_slot = 0;                                   // the output layer's weight stage, read by the seed epilogue
    auto close_stage = [&](int commit_d, bool release = true) {   // commit_d: 0 / 1 = completes N half 0 / 1, 2 = AFREE
      if (elect_one()) {
        if (release) mma_commit_2cta(BAR(BAR_EMPTY + slot)); // the slot may be refilled (both CTAs)
        if (commit_d == 0) mma_commit_2cta(BAR(BAR_DFULL0)); // N half 0 (or a small GEMM) is complete
        if (commit_d == 1) mma_commit_2cta(BAR(BAR_DFULL1));
        if (commit_d == 2) mma_commit_2cta(BAR(BAR_AFREE));  // last reader of the operand's K half 0
      }
      __syncwarp();
      if (++slot == NSLOT) { slot = 0; par ^= 1; }
    };
    constexpr uint32_t KHALF = 8 * 2 * ALBO;                  // byte offset of K = 128 in the A images
    for (int tile = pair; tile < n_tiles; tile += npairs)
    for (int t = 1; t <= n_steps; ++t) {
#pragma unroll 1
      for (int g = 0; g < NG; ++g) {
        if (g == 0) {                          // K = 32: one stage per N half, operand (the encoding) in one piece
          open_stage(0, 0, 64 * 16, 4096, idesc128);
          wait_a(0);
          steps(2, true);
          close_stage(0);
          open_stage(DHALF, 0, 64 * 16, 4096, idesc128);
          steps(2, true);
          if (elect_one()) mma_commit_2cta(BAR(BAR_AFREE));
          __syncwarp();
          close_stage(1);
        } else if (g == 4 || g == 8) {         // N = 32, K = 256: one stage, issued quarter by quarter as the operand lands
          open_stage(0, 0, 16 * 16, 8192, idesc32);
          wait_a(0); steps(4, true);
          wait_a(1); steps(4, false);
          wait_a(2); steps(4, false);
          wait_a(3); steps(4, false);
          held_slot = slot;
          close_stage(0, !(BWD && g == 4));    // W5's stage stays: the seed epilogue reads its rows from the slot
        } else {
          // N half 0 follows the operand quarter by quarter: quarters 0, 1 are the previous layer's half-0 epilogue
          // (parked, stored when that layer's MMAs retired), quarters 2, 3 its half-1 epilogue, whose accumulator
          // columns N half 1 of this layer then overwrites
          open_stage(0, 0, 64 * 16, 16384, idesc128);
          wait_a(0);
          auto release_held = [&]() {          // every seed thread has read W5's rows: hand the slot back in both CTAs
            if (lane == 0) {
              mbar_arrive_remote(BAR(BAR_EMPTY + held_slot), 0);
              mbar_arrive_remote(BAR(BAR_EMPTY + held_slot), 1);
            }
            __syncwarp();
          };
          if (g == 5 && !HM) release_held();
          steps(4, true);
          wait_a(1);
          // (half tiles: quarter 0 is signalled by the fb == 0 warps only; the fb == 1 warps have read their rows of W5
          // once quarter 1 is in as well)
          if (g == 5 && HM) release_held();
          steps(4, false);
          close_stage(-1);
          open_stage(0, KHALF, 64 * 16, 16384, idesc128);
          wait_a(2); steps(4, false);
          wait_a(3); steps(4, false);
          close_stage(0);
          open_stage(DHALF, 0, 64 * 16, 16384, idesc128);
          steps(8, true);
          close_stage(2);
          open_stage(DHALF, KHALF, 64 * 16, 16384, idesc128);
          steps(8, false);
          close_stage(1);
        }
      }
    }
  }
  // ---- teardown
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == W_MMA) {
    __syncwarp();
    tmem_free_512_2cta(tmem_base);
  }
}

// Per-GEMM compensation of the network in hand.  Layer 1 keeps c(2) (K = 3(d+P) <= 32 whatever the width); for the
// 256 x 4 network every other GEMM gets c(16), the constants the kernel had before networks of other shapes existed.
void set_compensation(const dsmppi_ctx* c, float (&comp)[N_GEMM]) {
  const int L = c->net.nh;
  const float hid = comp_steps((c->net.width + 15) / 16);    // a GEMM over the hidden features
  comp[0] = COMP_K32;
  for (int l = 1; l < 4; ++l) comp[l] = l < L ? hid : 0.f;   // forward layer l + 1: hidden, or identity
  comp[4] = hid;
  for (int l = 3; l >= 1; --l) comp[8 - l] = l < L ? hid : 0.f;
  comp[8] = hid;
}

}  // namespace

int tcx_build_images(dsmppi_ctx* c, const dsmppi_net* net) {
  c->tcx_blob = nullptr;
  if (c->nenc > 32 || c->O > 16) return 0;          // layer-1 K and the output N are fixed at 32 / 16: FFMA path only
  const char* dis = std::getenv("DSMPPI_DISABLE_TC");
  if (dis && dis[0] == '1') return 0;
  const size_t total = 2 * IMG_BYTES;
  std::vector<uint8_t> host(total, 0);
  const int nenc = c->nenc, O = c->O;
  auto put = [&](uint8_t* part_hi, uint8_t* part_lo, size_t off, float w) {
    const uint16_t hi = f2h(w);
    const uint16_t lo = f2h((w - h2f(hi)) * 2048.f);
    std::memcpy(part_hi + off, &hi, 2);
    std::memcpy(part_lo + off, &lo, 2);
  };
  for (int rank = 0; rank < 2; ++rank) {
    uint8_t* img = host.data() + (size_t)rank * IMG_BYTES;
    uint32_t off, bytes;
    // GEMM 0: B[n][k] = W0[n][k], k < nenc; N half x, this rank's 64 features
    for (int x = 0; x < 2; ++x) {
      stage_info(x, off, bytes);
      for (int n = 0; n < 64; ++n)
        for (int k = 0; k < 32; ++k)
          put(img + off, img + off + 4096, canon(n, k, 64),
              k < nenc ? net->W_host[0][(size_t)(128 * x + 64 * rank + n) * nenc + k] : 0.f);
    }
    // GEMMs 1-3 (forward): B[n][k] = W_l[n][k];  GEMMs 5-7 (backward, l = 3, 2, 1): B[n][k] = W_l[k][n];
    // stage (x, kh) = N half x, K half kh
    for (int g = 0; g < 3; ++g)
      for (int x = 0; x < 2; ++x)
        for (int kh = 0; kh < 2; ++kh) {
          stage_info(2 + 4 * g + 2 * x + kh, off, bytes);
          const float* W = net->W_host[1 + g];
          for (int n = 0; n < 64; ++n)
            for (int k = 0; k < 128; ++k)
              put(img + off, img + off + 16384, canon(n, k, 64),
                  W[(size_t)(128 * x + 64 * rank + n) * HID + 128 * kh + k]);
          stage_info(15 + 4 * g + 2 * x + kh, off, bytes);
          const float* Wt = net->W_host[3 - g];
          for (int n = 0; n < 64; ++n)
            for (int k = 0; k < 128; ++k)
              put(img + off, img + off + 16384, canon(n, k, 64),
                  Wt[(size_t)(128 * kh + k) * HID + 128 * x + 64 * rank + n]);
        }
    // GEMM 4: N = 32 over the pair.  BOTH ranks carry links 0..15 (rank 1's accumulator columns 16..31 are never
    // read): the seed epilogue of either CTA looks W5[l*, :] up in its own copy of this stage
    stage_info(14, off, bytes);
    for (int n = 0; n < 16; ++n)
      for (int k = 0; k < HID; ++k) {
        const int o = n;
        put(img + off, img + off + 8192, canon(n, k, 16), o < O ? net->W_host[4][(size_t)o * HID + k] : 0.f);
      }
    // GEMM 8: a[e] = sum_k g1[k] W0[k][e], e = 16 * rank + n
    stage_info(27, off, bytes);
    for (int n = 0; n < 16; ++n)
      for (int k = 0; k < HID; ++k) {
        const int e = 16 * rank + n;
        put(img + off, img + off + 8192, canon(n, k, 16), e < nenc ? net->W_host[0][(size_t)k * nenc + e] : 0.f);
      }
  }
  TxImages* t = new TxImages();
  if (cudaMalloc(reinterpret_cast<void**>(&t->dev), total) != cudaSuccess) {
    dsmppi_set_error("cudaMalloc(split weight images) failed");
    delete t;
    return 1;
  }
  CUDA_TRY(cudaMemcpy(t->dev, host.data(), total, cudaMemcpyHostToDevice));
  c->tcx_blob = t;
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  CUDA_TRY(cudaFuncSetAttribute(tc_exact_kernel<2, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  return 0;
}

void tcx_free_images(dsmppi_ctx* c) {
  if (!c->tcx_blob) return;
  TxImages* t = static_cast<TxImages*>(c->tcx_blob);
  if (t->dev) cudaFree(t->dev);
  delete t;
  c->tcx_blob = nullptr;
}

int launch_tc_exact(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const RowSrc& src, uint32_t ignore_mask,
                    float* m_rows, float* row_dist, float* row_grad, bool bwd, cudaStream_t st) {
  REQUIRE(c->tcx_blob, "split weight images not built");
  if (src.n_rows <= 0) return 0;
  TxImages* t = static_cast<TxImages*>(c->tcx_blob);
  TxArgs a;
  a.img0 = t->dev;
  a.img1 = t->dev + IMG_BYTES;
  a.net = c->net;
  a.src = src;
  a.q = q;
  a.q_stride = q_stride;
  a.obs = obs;
  a.vel = nullptr;
  a.ignore_mask = ignore_mask;
  a.out_m = m_rows;
  a.out_dist = row_dist;
  a.out_grad = row_grad;
  // re-scoring list of the rows that leave the fp16 range (normally none): counters[4 + parity] counts this launch's
  // rows, the kernel zeroes the other one for the next launch
  size_t need = (size_t)(src.n_rows < (1 << 24) ? src.n_rows : (1 << 24));
  if (need > c->fix_cap) {
    if (c->fix_list) CUDA_TRY(cudaFree(c->fix_list));
    c->fix_list = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->fix_list), need * 3 * sizeof(int)));
    c->fix_cap = need;
  }
  a.fix_count = c->counters + 4 + c->fix_parity;
  a.fix_next = c->counters + 4 + (c->fix_parity ^ 1);
  a.fix_total = c->counters + 6;
  a.fix_dropped = c->counters + 7;
  a.fix_list = c->fix_list;
  a.fix_cap = (int)c->fix_cap;
  c->fix_parity ^= 1;
  set_compensation(c, a.comp);
  const char* dbg = std::getenv("DSMPPI_TCX_DEBUG");
  a.dbg = dbg ? std::atoi(dbg) : 0;
  a.prof = nullptr;
#ifdef DSMPPI_TCX_PROF
  static long long* prof_buf = nullptr;
  const char* prof_out = std::getenv("DSMPPI_TCX_PROF_OUT");
  if (prof_out && src.n_rows >= 100000) {
    if (!prof_buf) CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&prof_buf), 4 * 2048 * sizeof(long long)));
    CUDA_TRY(cudaMemsetAsync(prof_buf, 0, 4 * 2048 * sizeof(long long), st));
    a.prof = prof_buf;
  }
#endif
  const long long tiles = ((long long)src.n_rows + 2 * TROWS - 1) / (2 * TROWS);
  long long pairs = c->sm_count / 2;
  if (pairs > tiles) pairs = tiles;
  if (pairs < 1) pairs = 1;
  const dim3 grid((unsigned)(2 * pairs));
  if (bwd) tc_exact_kernel<1><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
  else tc_exact_kernel<0><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
#ifdef DSMPPI_TCX_PROF
  if (a.prof) {
    CUDA_TRY(cudaStreamSynchronize(st));
    std::vector<long long> host(4 * 2048);
    CUDA_TRY(cudaMemcpy(host.data(), prof_buf, host.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    if (FILE* f = std::fopen(prof_out, "wb")) {
      std::fwrite(host.data(), sizeof(long long), host.size(), f);
      std::fclose(f);
    }
  }
#endif
  if (bwd) return 0;       // (forward + VJP launches re-score their flagged rows inside the kernel)
  // the flagged rows again, in IEEE fp32, written over the tensor-core results
  RowSrc fix{};
  fix.mode = ROWS_LIST;
  fix.M = src.M;
  fix.K = src.K;
  fix.n_rows = (int)(src.n_rows < a.fix_cap ? src.n_rows : a.fix_cap);
  fix.n_rows_dev = a.fix_count;
  fix.row_sample = c->fix_list;
  fix.row_obs = c->fix_list + c->fix_cap;
  fix.out_row = c->fix_list + 2 * c->fix_cap;
  return launch_exact_fixup(c, q, q_stride, obs, fix, ignore_mask, m_rows, row_dist, row_grad, bwd, st);
}

// whole-horizon rollout in one launch on the tensor cores; the caller has checked M <= 128 / 1 and initialised
// all_traj[:, 0] (same contract as launch_rollout_fused)
int launch_tc_rollout(dsmppi_ctx* c, const dsmppi_rollout_args* ra, cudaStream_t st) {
  REQUIRE(c->tcx_blob, "split weight images not built");
  REQUIRE(c->M >= 1 && c->M <= TROWS, "whole-horizon tensor-core rollout needs M <= 128");
  TxImages* t = static_cast<TxImages*>(c->tcx_blob);
  TxArgs a{};
  a.img0 = t->dev;
  a.img1 = t->dev + IMG_BYTES;
  a.net = c->net;
  a.obs = c->obs;
  a.vel = c->moving ? c->vel : nullptr;
  a.ignore_mask = ra->ignored_link_mask;
  a.sa = make_step_args(c, ra, 0);
  a.M = c->M;
  // Half tiles (64 rows per CTA, tc_exact_kernel<2, true>) while they still cover the batch in one wave of CTA pairs:
  // the rollout is then latency-bound on one tile per step, and a half tile takes about half the time.
  const long long pairs_all = c->sm_count / 2;
  const int s_half = c->M <= 64 ? 64 / c->M : 0;
  const bool half_tiles = c->half_tiles && s_half >= 1 && ((long long)ra->N + 2 * s_half - 1) / (2 * s_half) <= pairs_all;
  a.S = half_tiles ? s_half : TROWS / c->M;
  a.m_rows = c->m_rows;
  a.row_dist = c->row_dist;
  a.row_grad = c->row_grad;
  a.sel_rows = c->sel_rows;
  a.fix_count = c->counters + 4;
  a.fix_next = c->counters + 5;
  a.fix_total = c->counters + 6;
  a.fix_dropped = c->counters + 7;
  a.fix_list = nullptr;
  a.fix_cap = 0;
  set_compensation(c, a.comp);
  const char* dbg = std::getenv("DSMPPI_TCX_DEBUG");
  a.dbg = dbg ? std::atoi(dbg) : 0;
#ifdef DSMPPI_TCX_PROF
  static long long* prof_buf = nullptr;
  const char* prof_out = std::getenv("DSMPPI_TCX_PROF_OUT");
  if (prof_out) {
    if (!prof_buf) CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&prof_buf), 4 * 2048 * sizeof(long long)));
    CUDA_TRY(cudaMemsetAsync(prof_buf, 0, 4 * 2048 * sizeof(long long), st));
    a.prof = prof_buf;
    long long* region3 = prof_buf + 3 * 2048;              // step_sample's own stamps (step_device.cuh)
    int zero = 0;
    CUDA_TRY(cudaMemcpyToSymbolAsync(g_step_prof, &region3, sizeof(region3), 0, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyToSymbolAsync(g_step_prof_n, &zero, sizeof(zero), 0, cudaMemcpyHostToDevice, st));
  }
#endif
  const long long tiles = ((long long)ra->N + 2 * a.S - 1) / (2 * a.S);
  long long pairs = c->sm_count / 2;
  if (pairs > tiles) pairs = tiles;
  if (pairs < 1) pairs = 1;
  const dim3 grid((unsigned)(2 * pairs));
  if (c->moving) {
    if (half_tiles) tc_exact_kernel<2, true, true><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
    else tc_exact_kernel<2, false, true><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
  } else {
    if (half_tiles) tc_exact_kernel<2, true><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
    else tc_exact_kernel<2><<<grid, NTHREADS, SMEM_BYTES, st>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  c->launches++;
#ifdef DSMPPI_TCX_PROF
  if (a.prof) {
    CUDA_TRY(cudaStreamSynchronize(st));
    std::vector<long long> host(4 * 2048);
    CUDA_TRY(cudaMemcpy(host.data(), prof_buf, host.size() * sizeof(long long), cudaMemcpyDeviceToHost));
    if (FILE* f = std::fopen(prof_out, "wb")) {
      std::fwrite(host.data(), sizeof(long long), host.size(), f);
      std::fclose(f);
    }
  }
#endif
  return 0;
}
