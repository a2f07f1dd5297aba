// Tensor-core prefilter for obstacle ranking (pass 1 of MPPI.distance_repulsion_nn, MPPI.py:231-247).
//
// Every (sample, obstacle) pair is pushed through the 5-layer distance MLP on the 5th-generation tensor
// cores (tcgen05.mma, kind::f16; by default fp16 accumulators in the hidden layers and fp32 ones in the output
// layer, see HACC below) to get an APPROXIMATE masked minimum link distance; the fp32-accurate scoring path then
// re-scores only the obstacles inside a (calibrated) guard band of the K-th smallest, so the final ranking,
// distances and gradients are fp32-exact.
//
// Design (B200, one CTA pair per TPC, persistent):
//   * layer 1 is SEPARABLE in its input [q, p]:  W1 enc([q, p]) + b1 = (W1q enc(q) + b1) + W1p enc(p).  The
//     per-sample part A_i (n x 256) and the per-obstacle part B_j (M x 256) are small tables (fp32 arithmetic,
//     stored as fp16 / bf16 pairs); a pair row's first hidden activation is relu(A_i + B_j) -- two packed
//     half-precision instructions per two features, read straight into the layer-2 operand.  The (M N, d + 4)
//     input of MPPI.py:93-95 is never materialised, layer 1 costs no tensor-core time and, above all, no
//     accumulator round trip: a K = 60 GEMM kept the tensor pipe waiting for a full 256-column epilogue per tile
//     (31 % of the pipe's cycles were idle in the first version of this kernel, profiles/r1_tc_pass1_*).  The next
//     tile's operand is prepared under the current tile's last MMAs.
//   * cta_group::2 MMAs with M = 256 (128 pair-rows per CTA): each CTA keeps HALF of every remaining weight
//     matrix resident in shared memory for the whole kernel (3 x 64 + 8 KB of fp16 + 3 KB of biases = 203 KB),
//     loaded once with bulk TMA copies (cp.async.bulk, UBLKCP) -- no weight traffic afterwards.
//   * activations never touch shared memory or HBM: the A operand of every layer lives in TMEM
//     (tcgen05.mma "ts" form); the epilogue warps read the accumulator with tcgen05.ld (fp16 accumulators: two
//     packed features per register), add bias + ReLU (one HFMA2.RELU per feature pair) and write the next layer's
//     A operand back with tcgen05.st.
//   * TMEM (512 columns): A operands of two row tiles X,Y (2 x 128 columns) + two 128-column accumulator
//     halves D_lo/D_hi shared by both tiles.  While the epilogue warps of X drain D_lo/D_hi, the tensor core
//     already works on Y, so in steady state the MMA pipe never waits for an epilogue.
//   * warp roles: warps 0-3 rows of tile X, warps 4-7 rows of tile Y (TMEM lane quarter = warp % 4),
//     warp 8 = TMEM allocator + weight loader + MMA issuer (one elected thread, leader CTA only).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <utility>
#include <vector>

#include "internal.cuh"
#include "l1_table.cuh"
#include "tc_ptx.cuh"

namespace {
using namespace tcx;

constexpr int ROWS = 128;                 // pair-rows per CTA per tile slot
constexpr int NHID = 3;                   // hidden GEMMs on the tensor cores (network layers 2..4)
constexpr int MMA_WARP = 8;               // warps 0..7: rows (2 tile slots x 4 TMEM lane quarters)
// Three warpgroups: two of row warps and one holding the MMA issuer (warp 8; warps 9..11 only exist so that the
// third warpgroup is complete and can hand its registers over with setmaxnreg).  A 9-warp CTA would leave the
// row warps 168 registers (three warps on one scheduler) -- not enough to keep a whole 128-column accumulator
// half in flight, which is what frees D_lo / D_hi early enough for the other tile's MMAs.
constexpr int NTHREADS = 12 * 32;
constexpr int ROW_REGS = 232, ISSUER_REGS = 40;   // 128*(168-40) freed == 2*128*(232-168) claimed

// ---- shared-memory map (bytes); the weight part is a verbatim copy of the per-CTA global image
constexpr int OFF_WH = 0;                          // layers 2..4: 3 x 2 halves x (64 rows x 256) fp16
constexpr int SZ_WHH = 64 * HID * 2;               // 32 KB per half
constexpr int OFF_W5 = OFF_WH + NHID * 2 * SZ_WHH; // output layer: 16 rows x 256 fp16
constexpr int SZ_W5 = 16 * HID * 2;                // 8 KB
constexpr int OFF_BIAS = OFF_W5 + SZ_W5;           // 3 x 256 fp32 (layers 2..4) + 16 fp32 (output)
constexpr int SZ_BIAS = (NHID * HID + 16) * 4;
constexpr int IMG_BYTES = OFF_BIAS + SZ_BIAS;      // 207936
constexpr int OFF_BAR = IMG_BYTES;                 // mbarriers (8 B each)
constexpr int NBAR = 20;
constexpr int OFF_TMEMPTR = OFF_BAR + NBAR * 8;
// hand-over of a tile's 128 distances from the row warps of a slot to that slot's writer warp (warp 9 / 10): two
// buffers per slot, so the row warps never wait for the writer
constexpr int OFF_MBUF = OFF_TMEMPTR + 16;         // [slot][buffer][128] floats
constexpr int OFF_BIASH = OFF_MBUF + 2 * 2 * ROWS * 4;   // hidden-layer biases as fp16 pairs (fp16-accumulator build)
// staging of the two table-A rows a row warp's 32 pair-rows can touch: [warp][2][32] groups of 8 halves
constexpr int OFF_ABUF = OFF_BIASH + NHID * HID * 2;
constexpr int SMEM_BYTES = OFF_ABUF + 8 * 2 * 32 * 16;
static_assert(IMG_BYTES % 16 == 0, "bulk copies need 16-byte granularity");
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB shared-memory budget");

// barrier indices
enum { BAR_W = 0, BAR_AREADY0 = 1, BAR_AREADY1 = 2, BAR_DFREE0 = 3, BAR_DFREE1 = 4,
       BAR_DFULL00 = 5, BAR_DFULL01 = 6, BAR_DFULL10 = 7, BAR_DFULL11 = 8,
       BAR_MFULL = 9,      // + slot * 2 + buffer: the slot's four row warps have written their distances (count 4)
       BAR_MEMPTY = 13 };  // + slot * 2 + buffer: the writer warp has read them (count 1)

// TMEM columns
constexpr uint32_t TM_A0 = 0, TM_A1 = 128, TM_DLO = 256, TM_DHI = 384;

struct TcImages {
  uint8_t* img[2];        // device images, one per CTA rank
  // layers 2..5 of the network in the 256 x 4 frame, laid out as dsmppi_permute_hidden takes them: the images are
  // rebuilt from them whenever the census reorders the hidden features
  std::vector<float> W, b;
  int32_t perm[NHID * HID];            // the order of the images in effect
  uint32_t alive[NHID][HID / 32] = {}; // census: features of hidden layers 2..4 seen active since the last fresh one
};

template <bool BF16>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t r;
  if (BF16) asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// max(x, 0) folded into the conversion (round-to-nearest keeps the sign, so relu commutes with the rounding)
template <bool BF16>
__device__ __forceinline__ uint32_t pack2_relu(uint32_t lo, uint32_t hi) {
  uint32_t r;
  if (BF16) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  else asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(hi)), "f"(__uint_as_float(lo)));
  return r;
}
// two fp32 additions in one issue slot (Blackwell packed fp32 pipe); bit-identical to two add.rn.f32
__device__ __forceinline__ void add2(uint32_t a0, uint32_t a1, float b0, float b1, uint32_t& s0, uint32_t& s1) {
  asm("{\n\t.reg .b64 x, y, z;\n\t"
      "mov.b64 x, {%2, %3};\n\t"
      "mov.b64 y, {%4, %5};\n\t"
      "add.rn.f32x2 z, x, y;\n\t"
      "mov.b64 {%0, %1}, z;\n\t}"
      : "=r"(s0), "=r"(s1)
      : "r"(a0), "r"(a1), "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

// ------------------------------------------------------------------------------------------------
// Layer-1 tables (l1_table.cuh).  A is row-major (a warp's rows share one sample, so its 16-byte reads are
// broadcasts); B is stored [k / 8][j][k % 8] so that the 32 consecutive obstacles of a warp read 32 consecutive
// 16-byte groups (one coalesced 512-byte request per instruction).
// ------------------------------------------------------------------------------------------------
// one CTA of 256 threads per sample / obstacle
template <bool BF16>
__global__ void __launch_bounds__(HID) l1_table_kernel(const float* __restrict__ x, int x_stride, int n, int ncomp,
                                                       int comp0, int nin, const float* __restrict__ Wf0,
                                                       const float* __restrict__ bias, int transposed, int M,
                                                       uint16_t* __restrict__ out) {
  const int i = blockIdx.x, k = threadIdx.x;
  __shared__ float xs[3 * MAXD];
  if (k < ncomp) {
    const float v = x[(size_t)i * x_stride + k];
    float sn, cs;
    sincosf(v, &sn, &cs);
    xs[3 * k] = v; xs[3 * k + 1] = sn; xs[3 * k + 2] = cs;
  }
  __syncthreads();
  const float acc = l1_feature(Wf0, bias, k, xs, ncomp, comp0, nin);
  const size_t o = transposed ? ((size_t)(k >> 3) * M + i) * 8 + (k & 7) : (size_t)i * HID + k;
  out[o] = l1_to_half_bits(acc, BF16);
  (void)n;
}

// Moving obstacles, one launch per rollout step of the per-step paths: obstacle j's position at tau (obstacle_at) into
// pos, and with tab != nullptr also its row of the per-obstacle table B in one format -- the l1_table_kernel<BF16> row
// of that position, computed the same way, so the prefilter sees the table tc_set_obstacles would build for it.
// With a table: one CTA of 256 threads per obstacle; without: one thread per obstacle.
__global__ void __launch_bounds__(HID) obstacles_at_kernel(const float* __restrict__ obs, const float* __restrict__ vel,
                                                           int M, float tau, float* __restrict__ pos, int ncomp,
                                                           int comp0, int nin, const float* __restrict__ Wf0, int bf16,
                                                           uint16_t* __restrict__ tab) {
  if (!tab) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= M) return;
    for (int c = 0; c < 3; ++c) pos[j * 4 + c] = obstacle_at(obs, vel, j, c, tau);
    pos[j * 4 + 3] = obs[j * 4 + 3];
    return;
  }
  const int j = blockIdx.x, k = threadIdx.x;
  __shared__ float xs[3 * MAXD];
  if (k < 4) pos[j * 4 + k] = k < 3 ? obstacle_at(obs, vel, j, k, tau) : obs[j * 4 + 3];
  if (k < ncomp) {
    const float v = obstacle_at(obs, vel, j, k, tau);
    float sn, cs;
    sincosf(v, &sn, &cs);
    xs[3 * k] = v; xs[3 * k + 1] = sn; xs[3 * k + 2] = cs;
  }
  __syncthreads();
  const float acc = l1_feature(Wf0, nullptr, k, xs, ncomp, comp0, nin);
  tab[((size_t)(k >> 3) * M + j) * 8 + (k & 7)] = l1_to_half_bits(acc, bf16 != 0);
}

// Census of the dead-feature skip (tc_census): which features of hidden layers 2..4 have a positive pre-activation
// for any of the n x M pairs of states q (row stride d) and obstacles obs, in fp32 from the fp32 weights.  One CTA
// of 256 threads (one feature each) per CEN_R pair-rows; alive[l][w]: bit f % 32 of word f / 32 for feature f.
constexpr int CEN_R = 32;
__global__ void __launch_bounds__(HID) census_kernel(const NetDev net, const float* __restrict__ q, int n,
                                                     const float* __restrict__ obs, int M,
                                                     uint32_t* __restrict__ alive) {
  __shared__ __align__(16) float h[HID][CEN_R];
  __shared__ float xq[CEN_R][3 * MAXD], xp[CEN_R][9];
  const int k = threadIdx.x, P = net.nin - net.d;
  const long long nrows = (long long)n * M, r0 = (long long)blockIdx.x * CEN_R;
  for (int e = k; e < CEN_R * (MAXD + 3); e += HID) {
    const int r = e / (MAXD + 3), cc = e % (MAXD + 3);
    const long long row = min(r0 + r, nrows - 1);
    float v = 0.f;
    if (cc < net.d) v = q[(row / M) * net.d + cc];
    else if (cc >= MAXD && cc - MAXD < P) v = obs[(row % M) * 4 + cc - MAXD];
    else continue;
    float sn, cs;
    sincosf(v, &sn, &cs);
    float* x = cc < MAXD ? &xq[r][3 * cc] : &xp[r][3 * (cc - MAXD)];
    x[0] = v; x[1] = sn; x[2] = cs;
  }
  __syncthreads();
  float acc[CEN_R];
#pragma unroll 1
  for (int r = 0; r < CEN_R; ++r)
    h[k][r] = fmaxf(l1_feature(net.Wf[0], net.b[0], k, xq[r], net.d, 0, net.nin) +
                        l1_feature(net.Wf[0], nullptr, k, xp[r], P, net.d, net.nin), 0.f);
  __syncthreads();
#pragma unroll 1
  for (int l = 1; l <= NHID; ++l) {
#pragma unroll
    for (int r = 0; r < CEN_R; ++r) acc[r] = net.b[l][k];
    const float* w = net.Wf[l] + k;
#pragma unroll 4
    for (int i = 0; i < HID; ++i) {
      const float wi = w[(size_t)i * HID];
      const float4* hv = reinterpret_cast<const float4*>(h[i]);
#pragma unroll
      for (int r4 = 0; r4 < CEN_R / 4; ++r4) {
        const float4 x = hv[r4];
        acc[4 * r4 + 0] = fmaf(wi, x.x, acc[4 * r4 + 0]);
        acc[4 * r4 + 1] = fmaf(wi, x.y, acc[4 * r4 + 1]);
        acc[4 * r4 + 2] = fmaf(wi, x.z, acc[4 * r4 + 2]);
        acc[4 * r4 + 3] = fmaf(wi, x.w, acc[4 * r4 + 3]);
      }
    }
    __syncthreads();
    bool any = false;
#pragma unroll
    for (int r = 0; r < CEN_R; ++r) {
      any = any || (r0 + r < nrows && acc[r] > 0.f);
      h[k][r] = fmaxf(acc[r], 0.f);
    }
    const uint32_t bits = __ballot_sync(0xffffffffu, any);
    if ((k & 31) == 0 && bits) atomicOr(alive + (l - 1) * (HID / 32) + (k >> 5), bits);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// The prefilter kernel
// ------------------------------------------------------------------------------------------------
struct TcArgs {
  const uint8_t* img0; const uint8_t* img1;    // per-CTA-rank weight images
  const uint4* tabA; const uint4* tabB;        // layer-1 tables: (n, 32) and (32, M) groups of 8 halves
  const float* obs;                            // (M, 4)
  float* mdist;                                // (n * M)
  long long n_rows;                            // n * M
  int n, M, O;
  uint32_t ignore_mask;
  float inv_scale_div;                         // 100 for the 9-link net else 1
  uint32_t zero;                               // 0 (an opaque zero for scheduling dependencies, see first_layer)
  int use_writers;                             // 1: warps 9 / 10 store the distances (0: the row warps do, see there)
  long long* prof;                             // DSMPPI_TC_PROF builds only: [block][warp][8] cycle counters
  int* nonfinite;                              // counts pair-rows whose prefilter output is inf / NaN (see the epilogue)
  // Dead-feature skip: skip[l] of the last K-steps of the GEMM that reads hidden GEMM l's output (network layer 3, 4,
  // output) are not issued (0..8: only features 128..255, the D_hi half, are ever skipped).  Their input features
  // were never active in the calibration's census and come last in the images' feature order (tc_census).
  int skip[NHID];
  int* dead_fired;                             // counts valid pair-rows in which a skipped feature was not +0
};

// Per-phase cycle accounting of the kernel's own pipeline (tools/tc_microbench.cu builds with
// -DDSMPPI_TC_PROF); compiled out of the product library.
#ifdef DSMPPI_TC_PROF
#define PROF_DECL long long _pt = clock64(); long long _pc[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define PROF_ADD(i) do { const long long _n = clock64(); _pc[i] += _n - _pt; _pt = _n; } while (0)
#define PROF_FLUSH(a, w) do { if ((a).prof && (threadIdx.x & 31) == 0) for (int _i = 0; _i < 8; ++_i) \
    (a).prof[((size_t)blockIdx.x * 9 + (w)) * 8 + _i] = _pc[_i]; } while (0)
#else
#define PROF_DECL do { } while (0)
#define PROF_ADD(i) do { } while (0)
#define PROF_FLUSH(a, w) do { } while (0)
#endif

// bias + ReLU + fp16/bf16 pair packing of 32 accumulator columns into pk[OFF .. OFF+16): per pair of columns one
// packed fp32 add and one converting ReLU (the epilogue's issue slots are what the two tile slots compete for)
template <bool BF16, int OFF, int NPK>
__device__ __forceinline__ void relu_pack32(const uint32_t (&v)[32], const float* __restrict__ bias32,
                                            uint32_t (&pk)[NPK]) {
  const float4* b4 = reinterpret_cast<const float4*>(bias32);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 bb = b4[k];
    uint32_t s0, s1, s2, s3;
    add2(v[4 * k + 0], v[4 * k + 1], bb.x, bb.y, s0, s1);
    add2(v[4 * k + 2], v[4 * k + 3], bb.z, bb.w, s2, s3);
    pk[OFF + 2 * k + 0] = pack2_relu<BF16>(s0, s1);
    pk[OFF + 2 * k + 1] = pack2_relu<BF16>(s2, s3);
  }
}

// fp16-accumulator build: 64 accumulator values arrive as 32 packed pairs; bias + ReLU is one HFMA2.RELU per pair.
// No saturation here (a clamping HMNMX2 per pair cost 3.5 % of the kernel): an accumulator that overflowed is inf,
// stays inf / NaN through the remaining layers, and is caught at the output.  The biases come from shared memory as
// fp16 pairs (passed as kernel parameters -- constant bank -- they turned into 192 LDC.64 per tile and cost 4 %).
template <int OFF, int BOFF, int NPK>
__device__ __forceinline__ void relu_h2_32(const uint32_t (&v)[32], const uint4 (&b)[16], uint32_t (&pk)[NPK]) {
  const uint32_t one = 0x3c003c00u;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint4 bb = b[BOFF + k];
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(pk[OFF + 4 * k + 0]) : "r"(v[4 * k + 0]), "r"(one), "r"(bb.x));
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(pk[OFF + 4 * k + 1]) : "r"(v[4 * k + 1]), "r"(one), "r"(bb.y));
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(pk[OFF + 4 * k + 2]) : "r"(v[4 * k + 2]), "r"(one), "r"(bb.z));
    asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(pk[OFF + 4 * k + 3]) : "r"(v[4 * k + 3]), "r"(one), "r"(bb.w));
  }
}
// 16 x 16 bytes of fp16 bias pairs, read BEFORE the wait for the accumulator they belong to: the loads are then off
// the chain accumulator ready -> operand stored (the asm waits carry memory clobbers, nothing moves across them)
__device__ __forceinline__ void load_bias16(const uint4* __restrict__ src, uint4 (&b)[16]) {
  const uint32_t sa = smem_u32(src);
#pragma unroll
  for (int k = 0; k < 16; ++k)      // volatile: the compiler would sink plain loads back to their uses, behind the wait
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(b[k].x), "=r"(b[k].y), "=r"(b[k].z), "=r"(b[k].w) : "r"(sa + 16u * k));
}

// OR of the packed activations (D_hi half, features 128..255, two per word) that the next GEMM does not read when
// its last `s` K-steps (8 words each) are skipped: 0 certifies that every skipped product was an exact zero
__device__ __forceinline__ uint32_t dead_or(const uint32_t (&pk)[64], int s) {
  // straight-line code: a switch over s became indirect branches inside the epilogue and cost spills around them
  uint32_t r = 0;
#pragma unroll
  for (int g = 0; g < 8; ++g)            // words 8g..8g+7 feed K-step 8 + g, skipped when 8 + g >= 16 - s
    if (g >= 8 - s) r |= (pk[8 * g] | pk[8 * g + 1] | pk[8 * g + 2]) | (pk[8 * g + 3] | pk[8 * g + 4] | pk[8 * g + 5]) |
                         (pk[8 * g + 6] | pk[8 * g + 7]);
  return r;
}

// A skipped feature that was active in a valid row: that row's distance lacks its products.  Counted once the
// tile's three hidden epilogues are done (not at the output, where one more live register spilled); the host repeats
// the call without the skip (prefilter_verdict).
__device__ __forceinline__ void dead_count(const TcArgs& a, uint32_t dead, int i) {
  if (dead != 0u && i < a.n) atomicAdd(a.dead_fired, 1);
}

// relu(a + b) on two packed half-precision values: the first hidden activation from the layer-1 tables
template <bool BF16>
__device__ __forceinline__ uint32_t add_relu_h2(uint32_t a, uint32_t b) {
  // one HFMA2.RELU: a * 1 is exact, so fma(a, 1, b) rounds exactly like a + b (an add + a max was two issue slots per
  // feature pair on the tile boundary's critical path)
  uint32_t r;
  if (BF16) asm("fma.rn.relu.bf16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(0x3f803f80u), "r"(b));
  else asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(0x3c003c00u), "r"(b));
  return r;
}

__device__ __forceinline__ uint4 ldg_nc_v4(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

// first hidden activation of pair (sample i, obstacle j): relu(A_i + B_j), 256 features = 128 packed words, the
// layer-2 operand as it goes into TMEM.  64 independent 16-byte loads (the A half is a warp-wide broadcast), issued
// as two halves of 32: all 64 at once would not fit next to the packed result, one small chunk at a time would expose
// the L2 latency many times over (the volatile loads keep that order).  (Free functions, not lambdas: a lambda taking
// the register array by reference that is not inlined would push the array into local memory.)
template <bool BF16>
__device__ __forceinline__ void first_layer(const TcArgs& a, int i, int j, uint32_t dep, uint32_t (&pk)[128]) {
  // `dep` is zero at run time but opaque to ptxas (it is derived from a kernel argument): the load addresses carry it,
  // so the assembler cannot hoist the 64 loads above the value `dep` was derived from, nor merge the two halves
  // (a first build had all 64 loads = 256 registers in flight inside the previous layer's epilogue and spilled 3 KB)
  if (i < a.n) {
    const uint4* ta = a.tabA + (size_t)i * 32 + dep;
    const uint4* tb = a.tabB + j + dep;
    // the row stride of table B carries `dep` too: as a loop invariant its 32 multiples (64 registers of addresses)
    // would be hoisted out of the tile loop and held across the hidden-layer epilogues
    const uint32_t strideM = (uint32_t)a.M + dep;
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      uint4 x[16], y[16];
#pragma unroll
      for (int kb = 0; kb < 16; ++kb) {
        x[kb] = ldg_nc_v4(ta + 16 * hf + kb);
        y[kb] = ldg_nc_v4(tb + (size_t)((16 * hf + kb) * strideM));
      }
#pragma unroll
      for (int kb = 0; kb < 16; ++kb) {
        pk[64 * hf + 4 * kb + 0] = add_relu_h2<BF16>(x[kb].x, y[kb].x);
        pk[64 * hf + 4 * kb + 1] = add_relu_h2<BF16>(x[kb].y, y[kb].y);
        pk[64 * hf + 4 * kb + 2] = add_relu_h2<BF16>(x[kb].z, y[kb].z);
        pk[64 * hf + 4 * kb + 3] = add_relu_h2<BF16>(x[kb].w, y[kb].w);
      }
      if (hf == 0) {
        const uint32_t d2 = (pk[3] | pk[11] | pk[19] | pk[27] | pk[35] | pk[43] | pk[51] | pk[59] | pk[63]) & a.zero;
        ta += d2;
        tb += d2;
      }
    }
  } else {
#pragma unroll
    for (int k = 0; k < 128; ++k) pk[k] = 0u;
  }
}
// The same, with the per-sample half read through shared memory: the 32 consecutive pair-rows of a warp belong to at
// most two samples (M >= 32), so the warp copies those two 512-byte rows once (one coalesced 16-byte load per lane and
// row) instead of every lane loading its own copy -- 2 instead of 32 global loads per thread, and the whole per-obstacle
// half (32 loads, 128 registers) fits in flight at once: one L2 latency per tile instead of two.
// Issued in two parts so that the loads are in flight while the caller drains the output layer.
struct TableLoads {
  uint4 y[32];        // this thread's per-obstacle half (256 features)
  uint4 a0, a1;       // lane-th 16-byte group of the warp's two per-sample rows
  int i0;
};
__device__ __forceinline__ void first_layer_issue(const TcArgs& a, int i, int j, uint32_t dep, int lane, TableLoads& t) {
  // Every load is unconditional: pair-rows past the end of the batch (i == n; only in the last tile) read the tables
  // of sample n - 1 and of their own, valid, obstacle index, and compute a row nobody stores.  (Predicated loads made
  // the compiler zero all 132 destination registers first, on every tile.)
  t.i0 = __shfl_sync(0xffffffffu, i, 0);
  const uint4* ta = a.tabA + dep;
  t.a0 = ldg_nc_v4(ta + (size_t)min(t.i0, a.n - 1) * 32 + lane);
  t.a1 = ldg_nc_v4(ta + (size_t)min(t.i0 + 1, a.n - 1) * 32 + lane);
  const uint4* tb = a.tabB + j + dep;
  const uint32_t strideM = (uint32_t)a.M + dep;
#pragma unroll
  for (int kb = 0; kb < 32; ++kb) t.y[kb] = ldg_nc_v4(tb + (size_t)(kb * strideM));
}
template <bool BF16>
__device__ __forceinline__ void first_layer_finish(const TcArgs& a, int i, const TableLoads& t, uint4* abuf, int lane,
                                                   uint32_t (&pk)[128]) {
  abuf[lane] = t.a0;
  abuf[32 + lane] = t.a1;
  __syncwarp();
  const uint4* ar = abuf + (i - t.i0) * 32;          // 0 or 1: a warp's rows span at most two samples
#pragma unroll
  for (int kb = 0; kb < 32; ++kb) {
    const uint4 x = ar[kb];
    pk[4 * kb + 0] = add_relu_h2<BF16>(x.x, t.y[kb].x);
    pk[4 * kb + 1] = add_relu_h2<BF16>(x.y, t.y[kb].y);
    pk[4 * kb + 2] = add_relu_h2<BF16>(x.z, t.y[kb].z);
    pk[4 * kb + 3] = add_relu_h2<BF16>(x.w, t.y[kb].w);
  }
  __syncwarp();
}
__device__ __forceinline__ void store_operand(uint32_t tA, const uint32_t (&pk)[128]) {
  tmem_st32<0>(tA, pk);
  tmem_st32<32>(tA + 32, pk);
  tmem_st32<64>(tA + 64, pk);
  tmem_st32<96>(tA + 96, pk);
}

// HACC: the hidden layers accumulate in fp16 (tcgen05 D format f16) instead of fp32.  The prefilter only has to be
// right to within its calibrated guard band, and an fp16 accumulator halves the epilogue (half the tcgen05.ld
// traffic, one HFMA2.RELU instead of an FADD2 + a converting ReLU per two features) and costs the tensor pipe less
// energy per MMA -- which is what this power-capped kernel is short of.  The output layer keeps fp32 accumulators.
template <bool BF16, bool HACC = false, bool ASM = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
tc_pass1_kernel(const __grid_constant__ TcArgs a) {
  static_assert(!(BF16 && HACC), "bf16 operands accumulate in fp32");
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar0 = sbase + OFF_BAR;
  auto BAR = [&](int i) { return bar0 + (uint32_t)i * 8u; };
  const float* bias = reinterpret_cast<const float*>(smem + OFF_BIAS);
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + OFF_TMEMPTR);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  // ---- one-time setup: barriers, TMEM, resident weights
  float* mbuf = reinterpret_cast<float*>(smem + OFF_MBUF);
  if (warp == MMA_WARP) {
    if (lane == 0) {
      mbar_init(BAR(BAR_W), 1);
      mbar_init(BAR(BAR_AREADY0), 8);     // 4 row warps of the slot x 2 CTAs (used in the leader CTA)
      mbar_init(BAR(BAR_AREADY1), 8);
      mbar_init(BAR(BAR_DFREE0), 8);      // 4 draining warps x 2 CTAs
      mbar_init(BAR(BAR_DFREE1), 8);
      for (int i = BAR_DFULL00; i <= BAR_DFULL11; ++i) mbar_init(BAR(i), 1);   // tcgen05.commit arrives
      for (int i = 0; i < 4; ++i) { mbar_init(BAR(BAR_MFULL + i), 4); mbar_init(BAR(BAR_MEMPTY + i), 1); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc_512_2cta(smem_u32((const void*)tmem_ptr_smem));
    if (lane == 0) {
      const uint8_t* img = rank == 0 ? a.img0 : a.img1;
      mbar_expect_tx(BAR(BAR_W), IMG_BYTES);
      constexpr int CH = 32768;
      for (int off = 0; off < IMG_BYTES; off += CH) {
        const int n = IMG_BYTES - off < CH ? IMG_BYTES - off : CH;
        bulk_g2s(sbase + off, img + off, n, BAR(BAR_W));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  mbar_wait(BAR(BAR_W), 0);            // this CTA's weights have landed
  if constexpr (HACC) {
    uint32_t* bh = reinterpret_cast<uint32_t*>(smem + OFF_BIASH);
    for (int k = tid; k < NHID * HID / 2; k += NTHREADS) bh[k] = pack2<false>(bias[2 * k], bias[2 * k + 1]);
    __syncthreads();
  }
  cluster_sync_all();                  // ... and so have the peer's; barrier inits visible cluster-wide

  const long long n_tiles = (a.n_rows + 2 * ROWS - 1) / (2 * ROWS);     // 256 pair-rows per tile

  if (warp < MMA_WARP) {
    // =================================== row warps ===================================
    // warp = slot*4 + quarter; a thread owns one pair-row (TMEM lane).  Per hidden layer it pulls a whole
    // 128-column accumulator half into registers with four back-to-back tcgen05.ld, releases that half to the
    // tensor core at once (the other tile's MMAs are waiting for it), and only then does bias / ReLU / fp16
    // packing; the packed low half waits in registers until the D_hi MMAs have retired the old A operand.
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(ROW_REGS));
    const int slot = warp >> 2;                          // 0: tile X, 1: tile Y
    const int row = ((warp & 3) << 5) | lane;            // TMEM lane == row within the CTA's 128
    const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
    const uint32_t tA = tmem_base + lane_addr + (slot ? TM_A1 : TM_A0);
    const uint32_t tDlo = tmem_base + lane_addr + TM_DLO, tDhi = tmem_base + lane_addr + TM_DHI;
    const uint32_t bar_aready = BAR(slot ? BAR_AREADY1 : BAR_AREADY0);
    const uint32_t bar_full_lo = BAR(slot ? BAR_DFULL10 : BAR_DFULL00);
    const uint32_t bar_full_hi = BAR(slot ? BAR_DFULL11 : BAR_DFULL01);
    uint4* abuf = reinterpret_cast<uint4*>(smem + OFF_ABUF) + warp * 64;

    auto signal = [&](uint32_t bar) {       // one arrival per warp on the leader CTA's barrier
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(bar, 0);
    };
    // pair-row of this thread: r = tile*256 + rank*128 + row = i*M + j, advanced by a constant stride per
    // iteration (no 64-bit division inside the loop)
    const long long stride = 2LL * npairs * (2 * ROWS);
    const int di = (int)(stride / a.M), dj = (int)(stride % a.M);
    const long long r0 = ((long long)slot * npairs + pair) * (2 * ROWS) + (long long)rank * ROWS + row;
    int i_cur = (int)min(r0 / a.M, (long long)a.n), j_cur = (int)(r0 % a.M);
    if ((long long)pair < n_tiles) {
      uint32_t pk[128];
      if constexpr (ASM) {
        TableLoads t;
        first_layer_issue(a, i_cur, j_cur, a.zero, lane, t);
        first_layer_finish<BF16>(a, i_cur, t, abuf, lane, pk);
      } else {
        first_layer<BF16>(a, i_cur, j_cur, a.zero, pk);
      }
      store_operand(tA, pk);
      tc_wait_st();
      signal(bar_aready);
    }
    PROF_DECL;
    for (long long it = 0;; ++it) {
      const long long tX = (it * 2) * npairs + pair;
      if (tX >= n_tiles) break;
      const bool more = ((it + 1) * 2) * npairs + pair < n_tiles;
      int i_next = min(i_cur + di, a.n), j_next = j_cur + dj;
      if (j_next >= a.M) { j_next -= a.M; i_next = min(i_next + 1, a.n); }
      uint32_t tile_dep = 0;
      uint32_t dead = 0;                     // dead_or over this tile's three hidden epilogues
      // fp16-accumulator build: one hidden layer's epilogue
      auto hacc_layer = [&](auto L) {
        constexpr int l = decltype(L)::value;
        PROF_ADD(7);
        uint32_t pk[64], raw[2][32];
        const uint4* bsm = reinterpret_cast<const uint4*>(smem + OFF_BIASH) + l * (HID / 8);
        uint4 bq[16];
        load_bias16(bsm, bq);
        mbar_wait(bar_full_lo, (uint32_t)(l & 1));
        tc_fence_after();
        PROF_ADD(0);
        tmem_ld32p(tDlo, raw[0]);
        tmem_ld32p(tDlo + 64, raw[1]);
        tc_wait_ld();
        signal(BAR(BAR_DFREE0));
        PROF_ADD(1);
        relu_h2_32<0, 0>(raw[0], bq, pk);
        relu_h2_32<32, 8>(raw[1], bq, pk);
        PROF_ADD(2);
        load_bias16(bsm + 16, bq);
        mbar_wait(bar_full_hi, (uint32_t)((it + l) & 1));
        tc_fence_after();
        PROF_ADD(3);
        tmem_ld32p(tDhi, raw[0]);
        tmem_ld32p(tDhi + 64, raw[1]);
        tmem_st32<0>(tA, pk);
        tmem_st32<32>(tA + 32, pk);
        tc_wait_ld();
        signal(BAR(BAR_DFREE1));
        PROF_ADD(4);
        relu_h2_32<0, 0>(raw[0], bq, pk);
        relu_h2_32<32, 8>(raw[1], bq, pk);
        tmem_st32<0>(tA + 64, pk);
        tmem_st32<32>(tA + 96, pk);
        dead |= dead_or(pk, a.skip[l]);      // under the store's latency
        tc_wait_st();
        signal(bar_aready);
        if (l == NHID - 1) {
          tile_dep = (pk[7] | pk[23] | pk[39] | pk[63]) & a.zero;
          dead_count(a, dead, i_cur);
        }
        PROF_ADD(5);
      };
      if constexpr (HACC) {
        hacc_layer(std::integral_constant<int, 0>{});
        hacc_layer(std::integral_constant<int, 1>{});
        hacc_layer(std::integral_constant<int, 2>{});
        static_assert(NHID == 3, "three hidden GEMMs");
      } else {
#pragma unroll
      for (int l = 0; l < NHID; ++l) {       // network layers 2..4
        const float* bl = bias + l * HID;
        PROF_ADD(7);
        uint32_t pk[64], raw[4][32];
        // ---- D_lo (features 0..127) while the tensor core is still producing D_hi.  Per tile a slot uses D_lo four
        //      times (three hidden layers + the output layer) and D_hi three times: phase parities below
        mbar_wait(bar_full_lo, (uint32_t)(l & 1));
        tc_fence_after();
        PROF_ADD(0);
        tmem_ld32(tDlo, raw[0]);
        tmem_ld32(tDlo + 32, raw[1]);
        tmem_ld32(tDlo + 64, raw[2]);
        tmem_ld32(tDlo + 96, raw[3]);
        tc_wait_ld();
        signal(BAR(BAR_DFREE0));                                    // D_lo drained: the other tile may use it
        PROF_ADD(1);
        relu_pack32<BF16, 0>(raw[0], bl, pk);
        relu_pack32<BF16, 16>(raw[1], bl + 32, pk);
        relu_pack32<BF16, 32>(raw[2], bl + 64, pk);
        relu_pack32<BF16, 48>(raw[3], bl + 96, pk);
        PROF_ADD(2);
        // ---- D_hi (features 128..255); its completion also retires every MMA that read the old A operand
        mbar_wait(bar_full_hi, (uint32_t)((it + l) & 1));          // phase 3*it + l of this slot's D_hi
        tc_fence_after();
        PROF_ADD(3);
        tmem_ld32(tDhi, raw[0]);
        tmem_ld32(tDhi + 32, raw[1]);
        tmem_ld32(tDhi + 64, raw[2]);
        tmem_ld32(tDhi + 96, raw[3]);
        tmem_st32<0>(tA, pk);
        tmem_st32<32>(tA + 32, pk);
        tc_wait_ld();
        signal(BAR(BAR_DFREE1));                                    // D_hi drained
        PROF_ADD(4);
        relu_pack32<BF16, 0>(raw[0], bl + 128, pk);
        relu_pack32<BF16, 16>(raw[1], bl + 160, pk);
        relu_pack32<BF16, 32>(raw[2], bl + 192, pk);
        relu_pack32<BF16, 48>(raw[3], bl + 224, pk);
        tmem_st32<0>(tA + 64, pk);
        tmem_st32<32>(tA + 96, pk);
        dead |= dead_or(pk, a.skip[l]);
        tc_wait_st();
        signal(bar_aready);                                         // next layer's A operand is in TMEM
        if (l == NHID - 1) {
          tile_dep = (pk[7] | pk[23] | pk[39] | pk[63]) & a.zero;
          dead_count(a, dead, i_cur);
        }
        PROF_ADD(5);
      }
      }
      // ---- output layer of this tile; under its MMAs (and the other tile's last hidden layer) the NEXT tile's
      //      first activation is read from the tables, so that the tile boundary costs one tcgen05.st
      const bool valid = i_cur < a.n;
      float rad = 0.f;
      if (valid) rad = __ldg(a.obs + (size_t)j_cur * 4 + 3);
      // the tile's result: masked minimum link distance (MPPI.py:236-242), handed to the writer warp
      auto finish_tile = [&](const uint32_t (&v)[16]) {
        float m = 3.0e38f;
        if (valid) {
          bool finite = true;
#pragma unroll
          for (int o = 0; o < 16; ++o) {
            if (o < a.O) {
              float y = __uint_as_float(v[o]) + bias[NHID * HID + o];
              finite = finite && (fabsf(y) <= 3.0e38f);
              y = y / a.inv_scale_div - rad;
              if ((a.ignore_mask >> o) & 1u) y = 1e6f;
              m = fminf(m, y);
            }
          }
          // An activation beyond the fp16 range (an fp16 accumulator that overflowed, or a saturated conversion feeding
          // inf - inf) surfaces here as inf / NaN.  Such a value says nothing about the pair: it is counted, and the
          // host repeats the whole call with every pair scored in fp32 (prefilter_verdict); the finite stand-in only
          // keeps the selection kernel's arithmetic defined until then.
          if (!finite) {
            m = -3.0e38f;
            atomicAdd(a.nonfinite, 1);
          }
        }
        if (a.use_writers) {
          // hand the distance to this slot's writer warp through shared memory (one st.shared + one mbarrier arrival
          // per warp): this warp is on the tensor core's critical path, a global store and its address arithmetic are
          // not free there (2.51 -> 2.39 ms per launch)
          const int b = (int)(it & 1);
          if (it >= 2) mbar_wait(BAR(BAR_MEMPTY + slot * 2 + b), (uint32_t)(((it >> 1) - 1) & 1));
          mbuf[(slot * 2 + b) * ROWS + row] = m;
          __syncwarp();
          if (lane == 0) mbar_arrive_local(BAR(BAR_MFULL + slot * 2 + b));
        } else if (valid) {
          a.mdist[(size_t)i_cur * a.M + j_cur] = m;
        }
      };
      uint32_t v[16];
      // (one branch holds the whole life of the 128-register operand: split into two `if (more)` blocks around the
      // wait, the compiler kept it conditionally live through the hidden-layer epilogues and spilled 3 KB per thread)
      if (more) {
        // D_lo is released as soon as the output layer has completed, with the next tile's table loads in flight and
        // before they are consumed: the other slot's next layer waits for D_lo (profiles/tc_pass1_schedule_ab.txt)
        uint32_t nxt[128];
        if constexpr (ASM) {
          TableLoads t;
          first_layer_issue(a, i_next, j_next, tile_dep, lane, t);
          PROF_ADD(6);
          mbar_wait(bar_full_lo, 1u);                               // fourth use of D_lo in this tile
          tc_fence_after();
          PROF_ADD(0);
          tmem_ld16(tDlo, v);
          tc_wait_ld();
          signal(BAR(BAR_DFREE0));
          first_layer_finish<BF16>(a, i_next, t, abuf, lane, nxt);
          store_operand(tA, nxt);               // the output-layer MMA has retired: A may be overwritten
        } else {
          first_layer<BF16>(a, i_next, j_next, tile_dep, nxt);
          PROF_ADD(6);
          mbar_wait(bar_full_lo, 1u);
          tc_fence_after();
          PROF_ADD(0);
          tmem_ld16(tDlo, v);
          store_operand(tA, nxt);
          tc_wait_ld();
          signal(BAR(BAR_DFREE0));
        }
        tc_wait_st();
        signal(bar_aready);
        finish_tile(v);
      } else {
        PROF_ADD(6);
        mbar_wait(bar_full_lo, 1u);
        tc_fence_after();
        PROF_ADD(0);
        tmem_ld16(tDlo, v);
        tc_wait_ld();
        signal(BAR(BAR_DFREE0));
        finish_tile(v);
      }
      i_cur = i_next;
      j_cur = j_next;
      PROF_ADD(6);
    }
    PROF_FLUSH(a, warp);
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(ISSUER_REGS));
  }
  if (warp == MMA_WARP && rank == 0) {
    // =================================== MMA issuer (warp 8 of the leader CTA) ===================================
    // The whole warp runs this loop convergently and one elected lane issues: every operand is then warp-uniform
    // and the (layer, slot, half) groups are fully unrolled, so one MMA costs a handful of issue slots.  (The
    // first version issued from a single divergent thread inside rolled loops: ~18 dependent instructions per
    // MMA, and the issue loop -- not the tensor pipe, not the epilogue -- set the pace of the whole kernel.)
    constexpr int fmt = BF16 ? 1 : 0;
    constexpr uint32_t idesc128 = make_idesc(fmt, 256, 128, !HACC);
    constexpr uint32_t idesc32 = make_idesc(fmt, 256, 32);
    const uint32_t sb4 = sbase >> 4;
    uint32_t ph_a[2] = {0, 0}, ph_free[2] = {0, 0};
    PROF_DECL;
    // one (layer L, slot S, half H) group: wait for the operands, issue its K-steps, commit
    auto group = [&](auto L, auto S, auto H) {
      constexpr int l = decltype(L)::value, s = decltype(S)::value, h = decltype(H)::value;
      PROF_ADD(2);
      mbar_wait(BAR(h ? BAR_DFREE1 : BAR_DFREE0), ph_free[h] ^ 1);
      ph_free[h] ^= 1;
      tc_fence_after();
      PROF_ADD(1);
      constexpr uint32_t boff = l < NHID ? OFF_WH + (l * 2 + h) * SZ_WHH : OFF_W5;
      constexpr uint32_t lbo = l < NHID ? 64 * 16 : 16 * 16;
      constexpr int ksteps = HID / 16;
      constexpr uint32_t idesc = l < NHID ? idesc128 : idesc32;
      constexpr uint32_t dcol = h ? TM_DHI : TM_DLO, acol = s ? TM_A1 : TM_A0;
      // K-steps 8..15 of the GEMMs after layer 2 may be skipped (their features come last, see TcArgs::skip)
      constexpr int fixed = l == 0 ? ksteps : ksteps / 2;
      const uint32_t nk = l == 0 ? ksteps : ksteps - a.skip[l > 0 ? l - 1 : 0];
      if (elect_one()) {
        mma_group<dcol, acol, boff, lbo, idesc, fixed>(tmem_base, sb4, nk, std::make_integer_sequence<int, ksteps>{});
        mma_commit_2cta(BAR(BAR_DFULL00 + s * 2 + h));
      }
      __syncwarp();
    };
    // one (slot, layer) step: wait for the slot's operand, then its accumulator halves
    auto step = [&](auto S, auto L) {
      constexpr int l = decltype(L)::value, s = decltype(S)::value;
      PROF_ADD(2);
      mbar_wait(BAR(s ? BAR_AREADY1 : BAR_AREADY0), ph_a[s]);
      ph_a[s] ^= 1;
      tc_fence_after();
      PROF_ADD(0);
      group(L, S, std::integral_constant<int, 0>{});
      if constexpr (l < NHID) group(L, S, std::integral_constant<int, 1>{});
    };
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;
    using I3 = std::integral_constant<int, 3>;
    // The two tile slots run HALF A TILE APART: X is two layers ahead of Y.  A slot's tile boundary -- drain the output
    // layer, read the next tile's first activation from the tables (L2 latency), store it -- takes ~2.5 k cycles during
    // which that slot has no MMA to offer; with both slots at the boundary together the tensor pipe idled for it (27 %
    // of its cycles in the ncu capture of the un-staggered order).  Staggered, one slot's boundary falls under a full
    // hidden layer (2.1 k cycles of MMAs) of the other.
    const long long n_it = (n_tiles - pair + 2LL * npairs - 1) / (2LL * npairs);   // iterations of this pair
    if (n_it > 0) {
      step(I0{}, I0{});
      step(I0{}, I1{});
    }
    for (long long it = 0; it < n_it; ++it) {
      const bool more = it + 1 < n_it;
      step(I0{}, I2{}); step(I1{}, I0{});
      step(I0{}, I3{}); step(I1{}, I1{});
      if (more) step(I0{}, I0{});
      step(I1{}, I2{});
      if (more) step(I0{}, I1{});
      step(I1{}, I3{});
    }
    PROF_ADD(2);
    PROF_FLUSH(a, MMA_WARP);
  }
  if ((warp == MMA_WARP + 1 || warp == MMA_WARP + 2) && a.use_writers) {
    // =================================== distance writers (warps 9, 10: one per tile slot) ========================
    // Per tile: the slot's 128 distances from shared memory to the (n, M) scratch matrix, 128 bytes per store
    // instruction; the matrix stays in L2 for select_candidates_kernel, which follows.
    //
    // Measured alternatives (B200, Franka shelf 2064, 4096 samples; ms per launch): row warps store directly 2.51;
    // writer warps 2.39 (this form).  Taking the guard band of a sample INSIDE this kernel as soon as its M distances
    // are complete (one atomic per sample and tile on a writer warp: free, 2.36) was tried three ways and lost each
    // time: on the writer warp itself 6.1 (while it selects, its slot's row warps run out of hand-over buffers and,
    // the issuer alternating the slots strictly, the whole CTA pair stops); on a dedicated warp with the sample staged
    // in shared memory 7.4 (the 24 KB of staging came out of the L1 that serves the table loads and the spills); on a
    // dedicated warp at this warpgroup's 40 registers 20 (spilled loop variables, every spill an L2 round trip).  The
    // stand-alone kernel takes 36 us per step with sixteen warps per SM hiding that latency.
    const int slot = warp - (MMA_WARP + 1);
    for (long long it = 0;; ++it) {
      const long long tX = (it * 2) * npairs + pair;
      if (tX >= n_tiles) break;                              // the row warps of both slots loop on slot X's tile
      const long long tile = (it * 2 + slot) * npairs + pair;
      const int b = (int)(it & 1);
      mbar_wait(BAR(BAR_MFULL + slot * 2 + b), (uint32_t)((it >> 1) & 1));
      float vals[4];
#pragma unroll
      for (int w = 0; w < 4; ++w) vals[w] = mbuf[(slot * 2 + b) * ROWS + 32 * w + lane];
      __syncwarp();
      if (lane == 0) mbar_arrive_local(BAR(BAR_MEMPTY + slot * 2 + b));
      const long long r0 = tile * (2 * ROWS) + (long long)rank * ROWS;       // pair-row r = i * M + j: mdist index
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const long long r = r0 + 32 * w + lane;
        if (r < a.n_rows) a.mdist[r] = vals[w];
      }
    }
  }
  // ---- teardown
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == MMA_WARP) {
    __syncwarp();
    tmem_free_512_2cta(tmem_base);
  }
}

// host: bf16 conversion (round to nearest even), no device needed
uint16_t f2bf(float f) {
  __nv_bfloat16 h = __float2bfloat16_rn(f);
  uint16_t u;
  std::memcpy(&u, &h, 2);
  return u;
}

}  // namespace

// Layers 2..5 of a network in the 256 x 4 frame (W: three 256 x 256 then O x 256, b: three 256 then O; torch
// orientation, concatenated) with the hidden features of layers 2..4 reordered: feature f of hidden layer 2 + l
// becomes the network's feature perm[l * 256 + f].  An exact transform of the network: the rows and biases of the
// layer 2..4 GEMMs and the matching input columns of the layer 3, layer 4 and output GEMMs move together (layer 1
// keeps its order).
int dsmppi_permute_hidden(int32_t n_out, const float* W, const float* b, const int32_t* perm, float* W_out,
                          float* b_out) {
  REQUIRE(W && b && perm && W_out && b_out, "null argument");
  REQUIRE(n_out >= 1 && n_out <= MAXO, "n_out out of range (1..16)");
  for (int l = 0; l < NHID; ++l) {
    std::vector<int> seen(HID, 0);
    for (int f = 0; f < HID; ++f) {
      REQUIRE(perm[l * HID + f] >= 0 && perm[l * HID + f] < HID && !seen[perm[l * HID + f]], "perm is not a permutation");
      seen[perm[l * HID + f]] = 1;
    }
  }
  auto in_feat = [&](int l, int k) { return l == 0 ? k : perm[(l - 1) * HID + k]; };
  for (int l = 0; l <= NHID; ++l) {
    const size_t wo = (size_t)l * HID * HID, bo = (size_t)l * HID;
    const int rows = l < NHID ? HID : n_out;
    for (int o = 0; o < rows; ++o) {
      const int src = l < NHID ? perm[l * HID + o] : o;
      for (int k = 0; k < HID; ++k) W_out[wo + (size_t)o * HID + k] = W[wo + (size_t)src * HID + in_feat(l, k)];
      b_out[bo + o] = b[bo + src];
    }
  }
  return 0;
}

namespace {

// The four weight images (fp16 / bf16 x CTA rank) of layers 2..5 of the network, W / b as dsmppi_permute_hidden
// lays them out
std::vector<uint8_t> image_bytes(const std::vector<float>& W, const std::vector<float>& b, int O) {
  std::vector<uint8_t> host((size_t)4 * IMG_BYTES, 0);
  for (int fmt = 0; fmt < 2; ++fmt)
    for (int rank = 0; rank < 2; ++rank) {
      uint8_t* img = host.data() + (size_t)(fmt * 2 + rank) * IMG_BYTES;
      auto put = [&](size_t off, float v) {
        const uint16_t u = fmt ? f2bf(v) : f2h(v);
        std::memcpy(img + off, &u, 2);
      };
      for (int h = 0; h < 2; ++h)
        for (int n = 0; n < 64; ++n) {
          const int feat = 128 * h + 64 * rank + n;        // output feature held by this CTA in half h
          for (int l = 0; l < NHID; ++l)                   // network layers 2..4 (layer 1 comes from the tables)
            for (int k = 0; k < HID; ++k)
              put(OFF_WH + (l * 2 + h) * SZ_WHH + canon(n, k, 64), W[(size_t)l * HID * HID + (size_t)feat * HID + k]);
        }
      for (int n = 0; n < 16; ++n) {
        const int o = 16 * rank + n;                       // N = 32 over the pair: links 0..15 | 16..31 (padding)
        for (int k = 0; k < HID; ++k)
          put(OFF_W5 + canon(n, k, 16), o < O ? W[(size_t)NHID * HID * HID + (size_t)o * HID + k] : 0.f);
      }
      float* bias = reinterpret_cast<float*>(img + OFF_BIAS);
      for (int k = 0; k < NHID * HID; ++k) bias[k] = b[k];
      for (int o = 0; o < 16; ++o) bias[NHID * HID + o] = o < O ? b[NHID * HID + o] : 0.f;
    }
  return host;
}

}  // namespace

int tc_build_images(dsmppi_ctx* c, const dsmppi_net* net) {
  c->tc_blob = nullptr;
  if (c->O > 16) return 0;                          // output N is fixed at 16 links; fall back to fp32
  const char* dis = std::getenv("DSMPPI_DISABLE_TC");
  if (dis && dis[0] == '1') return 0;
  TcImages* t = new TcImages();
  for (int l = 1; l <= 4; ++l) {
    const int rows = l < 4 ? HID : c->O;
    t->W.insert(t->W.end(), net->W_host[l], net->W_host[l] + (size_t)rows * HID);
    t->b.insert(t->b.end(), net->b_host[l], net->b_host[l] + rows);
  }
  for (int l = 0; l < NHID; ++l)
    for (int f = 0; f < HID; ++f) t->perm[l * HID + f] = f;
  // two formats x two CTA ranks
  uint8_t* dev = nullptr;
  if (cudaMalloc(reinterpret_cast<void**>(&dev), (size_t)4 * IMG_BYTES) != cudaSuccess) {
    dsmppi_set_error("cudaMalloc(tc images) failed");
    delete t;
    return 1;
  }
  const std::vector<uint8_t> host = image_bytes(t->W, t->b, c->O);
  if (cudaMemcpy(dev, host.data(), host.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
    dsmppi_set_error("cudaMemcpy(tc images) failed");
    cudaFree(dev);
    delete t;
    return 1;
  }
  t->img[0] = dev;
  t->img[1] = nullptr;
  c->tc_blob = t;
  c->tc_blob_bytes = host.size();
  auto opt_in = [](auto kernel) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
  };
  CUDA_TRY(opt_in(tc_pass1_kernel<false, false, false>));
  CUDA_TRY(opt_in(tc_pass1_kernel<false, false, true>));
  CUDA_TRY(opt_in(tc_pass1_kernel<true, false, false>));
  CUDA_TRY(opt_in(tc_pass1_kernel<true, false, true>));
  CUDA_TRY(opt_in(tc_pass1_kernel<false, true, false>));
  CUDA_TRY(opt_in(tc_pass1_kernel<false, true, true>));
  return 0;
}

void tc_free_images(dsmppi_ctx* c) {
  if (!c->tc_blob) return;
  TcImages* t = static_cast<TcImages*>(c->tc_blob);
  if (t->img[0]) cudaFree(t->img[0]);
  delete t;
  c->tc_blob = nullptr;
}

// Census of the dead-feature skip, over the n states q (row stride d) x every current obstacle: features of hidden
// layers 2..4 that never had a positive pre-activation go last in the images' order, and whole K = 16 steps of them
// are not issued by the GEMM that reads them (c->pass1_skip; at most 8 per GEMM, the D_hi half).  Each prefiltered row
// proves its skip (the kernel's dead_or): a row in which a skipped feature was active makes the host repeat the call
// without the skip and mark the census stale.  A census at the same obstacle count adds to the features seen active
// before; one that finds nothing new after such a repeat turns the skip off until the next fresh census (the active
// feature is then one the census rows do not reach).  *changed: the images' order changed.
int tc_census(dsmppi_ctx* c, const float* q, int n, cudaStream_t st, bool* changed) {
  TcImages* t = static_cast<TcImages*>(c->tc_blob);
  *changed = false;
  uint32_t* dev = nullptr;
  uint32_t alive[NHID][HID / 32];
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dev), sizeof(alive)));
  cudaError_t e = cudaMemsetAsync(dev, 0, sizeof(alive), st);
  const long long rows = (long long)n * c->M;
  if (e == cudaSuccess) {
    census_kernel<<<(unsigned)((rows + CEN_R - 1) / CEN_R), HID, 0, st>>>(c->net, q, n, c->obs, c->M, dev);
    c->launches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(alive, dev, sizeof(alive), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(dev);
  CUDA_TRY(e);
  const bool fresh = c->census_M != c->M;
  bool woke = false;
  for (int l = 0; l < NHID; ++l)
    for (int w = 0; w < HID / 32; ++w) {
      if (!fresh) {
        woke = woke || (alive[l][w] & ~t->alive[l][w]) != 0;
        alive[l][w] |= t->alive[l][w];
      }
      t->alive[l][w] = alive[l][w];
    }
  // active features first, each group in the network's order
  int32_t perm[NHID * HID];
  for (int l = 0; l < NHID; ++l) {
    int p = 0;
    for (int pass = 0; pass < 2; ++pass)
      for (int f = 0; f < HID; ++f)
        if (((alive[l][f >> 5] >> (f & 31)) & 1u) == (pass == 0 ? 1u : 0u)) perm[l * HID + p++] = f;
  }
  for (int l = 0; l < NHID; ++l) {
    int n_alive = 0;
    for (int w = 0; w < HID / 32; ++w) n_alive += __builtin_popcount(alive[l][w]);
    const int s = (HID - n_alive) / 16;
    c->pass1_skip[l] = (fresh || woke) ? (s < 8 ? s : 8) : 0;
  }
  c->census_M = c->M;
  c->census_stale = 0;
  if (std::memcmp(perm, t->perm, sizeof(perm)) != 0) {
    std::vector<float> W(t->W.size()), b(t->b.size());
    if (const int rc = dsmppi_permute_hidden(c->O, t->W.data(), t->b.data(), perm, W.data(), b.data())) return rc;
    const std::vector<uint8_t> host = image_bytes(W, b, c->O);
    CUDA_TRY(cudaMemcpyAsync(t->img[0], host.data(), host.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    std::memcpy(t->perm, perm, sizeof(perm));
    *changed = true;
  }
  return 0;
}

int tc_set_obstacles(dsmppi_ctx* c, cudaStream_t st) {
  // per-obstacle layer-1 table B, both formats (fp16 first, bf16 after it): M x 256 halves each
  const size_t need = (size_t)2 * c->M * HID * 2;
  if (need > c->obs_enc_cap) {
    if (c->obs_enc) CUDA_TRY(cudaFree(c->obs_enc));
    c->obs_enc = nullptr;
    CUDA_TRY(cudaMalloc(&c->obs_enc, need));
    c->obs_enc_cap = need;
  }
  uint16_t* out = static_cast<uint16_t*>(c->obs_enc);
  l1_table_kernel<false><<<c->M, HID, 0, st>>>(c->obs, 4, c->M, c->P, c->d, c->nin, c->net.Wf[0], nullptr, 1, c->M, out);
  l1_table_kernel<true><<<c->M, HID, 0, st>>>(c->obs, 4, c->M, c->P, c->d, c->nin, c->net.Wf[0], nullptr, 1, c->M,
                                              out + (size_t)c->M * HID);
  CUDA_TRY(cudaGetLastError());
  c->launches += 2;
  return 0;
}

// the per-sample layer-1 table A of n states (row stride q_stride floats) in the format of `mode`
int tc_reserve_sample_table(dsmppi_ctx* c, int n) {
  const size_t need = (size_t)n * HID * 2;
  if (need > c->enc_q_cap) {
    if (c->enc_q) CUDA_TRY(cudaFree(c->enc_q));
    c->enc_q = nullptr;
    CUDA_TRY(cudaMalloc(&c->enc_q, need + need / 8));
    c->enc_q_cap = need + need / 8;
  }
  return 0;
}

int tc_sample_table(dsmppi_ctx* c, const float* q, int q_stride, int n, int mode, cudaStream_t st) {
  const bool bf16 = mode == DSMPPI_PASS1_TC_BF16;
  if (tc_reserve_sample_table(c, n)) return 1;
  uint16_t* ta = static_cast<uint16_t*>(c->enc_q);
  if (bf16) l1_table_kernel<true><<<n, HID, 0, st>>>(q, q_stride, n, c->d, 0, c->nin, c->net.Wf[0], c->net.b[0], 0, 0, ta);
  else l1_table_kernel<false><<<n, HID, 0, st>>>(q, q_stride, n, c->d, 0, c->nin, c->net.Wf[0], c->net.b[0], 0, 0, ta);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}

int launch_obstacles_at(dsmppi_ctx* c, float tau, int mode, cudaStream_t st) {
  const int M = c->M;
  if (M > c->obs_step_cap) {
    if (c->obs_step) CUDA_TRY(cudaFree(c->obs_step));
    c->obs_step = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->obs_step), (size_t)M * 4 * sizeof(float)));
    c->obs_step_cap = M;
  }
  if (mode == DSMPPI_PASS1_EXACT_FP32) {
    obstacles_at_kernel<<<(M + 127) / 128, 128, 0, st>>>(c->obs, c->vel, M, tau, c->obs_step, 0, 0, 0, nullptr, 0,
                                                         nullptr);
  } else {
    const size_t need = (size_t)M * HID * 2;
    if (need > c->obs_enc_step_cap) {
      if (c->obs_enc_step) CUDA_TRY(cudaFree(c->obs_enc_step));
      c->obs_enc_step = nullptr;
      CUDA_TRY(cudaMalloc(&c->obs_enc_step, need));
      c->obs_enc_step_cap = need;
    }
    obstacles_at_kernel<<<M, HID, 0, st>>>(c->obs, c->vel, M, tau, c->obs_step, c->P, c->d, c->nin, c->net.Wf[0],
                                           mode == DSMPPI_PASS1_TC_BF16 ? 1 : 0,
                                           static_cast<uint16_t*>(c->obs_enc_step));
  }
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}

int tc_pass1(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const void* obs_tab, int n,
             uint32_t ignore_mask, int mode, cudaStream_t st, bool table_ready) {
  REQUIRE(c->tc_blob, "tensor-core images not built");
  TcImages* t = static_cast<TcImages*>(c->tc_blob);
  const bool bf16 = mode == DSMPPI_PASS1_TC_BF16;
  if (!obs_tab && c->obs_tables_dirty) {  // (small obstacle sets never get here: they are scored densely in fp32)
    if (tc_set_obstacles(c, st)) return 1;
    c->obs_tables_dirty = 0;
  }
  // the per-sample table of these states: written by the fused step kernel of the previous rollout step, else here
  if (!table_ready && tc_sample_table(c, q, q_stride, n, mode, st)) return 1;
  TcArgs a;
  const uint8_t* base = t->img[0] + (size_t)(bf16 ? 2 : 0) * IMG_BYTES;
  a.img0 = base;
  a.img1 = base + IMG_BYTES;
  a.tabA = reinterpret_cast<const uint4*>(c->enc_q);
  a.tabB = obs_tab ? static_cast<const uint4*>(obs_tab)
                   : reinterpret_cast<const uint4*>(static_cast<uint16_t*>(c->obs_enc) + (bf16 ? (size_t)c->M * HID : 0));
  a.obs = obs;
  a.mdist = c->mdist;
  a.n_rows = (long long)n * c->M;
  a.n = n;
  a.M = c->M;
  a.O = c->O;
  a.ignore_mask = ignore_mask;
  a.inv_scale_div = (c->O == 9) ? 100.f : 1.f;
  a.zero = 0u;
  a.use_writers = 1;
  a.nonfinite = c->counters + 9;
  a.dead_fired = c->counters + 10;
  for (int l = 0; l < NHID; ++l) a.skip[l] = c->pass1_noskip ? 0 : c->pass1_skip[l];
  a.prof = nullptr;
#ifdef DSMPPI_TC_PROF
  a.prof = reinterpret_cast<long long*>(c->stage);   // the micro-benchmark parks its counter buffer here
#endif
  const long long n_tiles = (a.n_rows + 2 * ROWS - 1) / (2 * ROWS);
  long long pairs = c->sm_count / 2;
  if (pairs > (n_tiles + 1) / 2) pairs = (n_tiles + 1) / 2;     // each pair takes two tiles per iteration
  if (pairs < 1) pairs = 1;
  const dim3 grid((unsigned)(2 * pairs));
  // (the shared-memory staging of table A needs a warp's 32 consecutive pair-rows to span at most two samples)
  const bool stage_a = c->M >= 32;
  auto launch = [&](auto kernel) { kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(a); };
  if (bf16) stage_a ? launch(tc_pass1_kernel<true, false, true>) : launch(tc_pass1_kernel<true, false, false>);
  else if (c->pass1_hacc) stage_a ? launch(tc_pass1_kernel<false, true, true>) : launch(tc_pass1_kernel<false, true, false>);
  else stage_a ? launch(tc_pass1_kernel<false, false, true>) : launch(tc_pass1_kernel<false, false, false>);
  CUDA_TRY(cudaGetLastError());
  c->launches++;
  return 0;
}
