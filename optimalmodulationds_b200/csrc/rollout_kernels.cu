// Per-sample stages of the MPPI rollout around the distance network: obstacle ranking, gradient blend,
// modulation + policy blend + Euler step, cost with terminal FK, Householder basis, policy update.
// One thread (or one warp, for ranking) per sample; every per-sample vector (d <= 8) lives in registers.
#include <cfloat>

#include "internal.cuh"
#include "step_device.cuh"
#include "select_device.cuh"
#include "l1_table.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// Ranking: the K closest obstacles per sample, ascending by (distance, obstacle index)
// (MPPI.py:243-247: sort over obstacles, first K).  One warp per sample.
// ------------------------------------------------------------------------------------------------
__global__ void rank_kernel(const float* __restrict__ m_rows, const int* __restrict__ row_base,
                            const int* __restrict__ cnt, const int* __restrict__ row_obs, int M, int n, int K,
                            int rows_out, int* __restrict__ sel) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n) return;
  const int base = row_base ? row_base[w] : w * M;
  const int c = cnt ? cnt[w] : M;
  float last_v = -FLT_MAX;
  int last_j = -1, last_t = 0;
  bool first = true;
  for (int kk = 0; kk < K; ++kk) {
    float bv = FLT_MAX;
    int bj = 0x7fffffff, bt = 0;
    for (int t = lane; t < c; t += 32) {
      const float v = m_rows[base + t];
      const int j = row_obs ? row_obs[base + t] : t;
      const bool after = first || v > last_v || (v == last_v && j > last_j);
      if (after && (v < bv || (v == bv && j < bj))) { bv = v; bj = j; bt = t; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
      const int ot = __shfl_xor_sync(0xffffffffu, bt, off);
      if (ov < bv || (ov == bv && oj < bj)) { bv = ov; bj = oj; bt = ot; }
    }
    if (bj == 0x7fffffff) { bj = last_j < 0 ? 0 : last_j; bt = last_t; }   // fewer than K candidates: repeat
    if (lane == 0) sel[w * K + kk] = rows_out ? base + bt : bj;
    last_v = bv; last_j = bj; last_t = bt; first = false;
  }
}

// The same ranking for a handful of obstacles scored densely (M <= 16: the planar and dense-field workloads): one
// THREAD per sample scans its M rows K times -- a warp per sample would idle 30 lanes and, at 10^6 samples, launch
// 10^6 warps for 2 x 10^6 floats.  Same order as the warp form: ascending by (distance, obstacle index).
__global__ void __launch_bounds__(256) rank_small_kernel(const float* __restrict__ m_rows, int M, int n, int K,
                                                         int rows_out, int* __restrict__ sel) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= n) return;
  const float* mr = m_rows + (size_t)w * M;
  float last_v = -FLT_MAX;
  int last_j = -1;
  for (int kk = 0; kk < K; ++kk) {
    float bv = FLT_MAX;
    int bj = -1;
    for (int j = 0; j < M; ++j) {
      const float v = mr[j];
      const bool after = kk == 0 || v > last_v || (v == last_v && j > last_j);
      if (after && (bj < 0 || v < bv)) { bv = v; bj = j; }
    }
    if (bj < 0) bj = last_j < 0 ? 0 : last_j;            // fewer than K candidates: repeat
    sel[(size_t)w * K + kk] = rows_out ? w * M + bj : bj;
    last_v = bv; last_j = bj;
  }
}

// ------------------------------------------------------------------------------------------------
// Candidate band from the approximate (tensor-core) distances: every obstacle within `band` of the
// K-th smallest approximate distance is re-scored in fp32.  One warp per sample.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) select_candidates_kernel(const float* __restrict__ mdist, int M, int n, int K,
                                                                float band, int cap_rows, int* __restrict__ cand_cnt,
                                                                int* __restrict__ row_base, int* __restrict__ row_sample,
                                                                int* __restrict__ row_obs, int* __restrict__ counters) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n) return;
  const float* md = mdist + (size_t)w * M;
  select_candidates_warp([md](int t) { return md[t]; }, M, K, band, cap_rows, w, lane, cand_cnt, row_base, row_sample,
                         row_obs, counters);
}

// largest |a - b| over n elements (guard-band calibration of the prefilter); out[0] must be zeroed beforehand.
// Non-negative floats order like their bit patterns, so the grid-wide maximum is an integer atomicMax.
__global__ void max_abs_diff_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n,
                                    float* __restrict__ out) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float df = fabsf(a[i] - b[i]);
    if (df == df) m = fmaxf(m, df);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(m));
}

__global__ void pack_obstacles_kernel(const float* __restrict__ raw, int M, int P, float* __restrict__ obs) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= M) return;
  float o[4] = {0.f, 0.f, 0.f, 0.f};
  for (int c = 0; c < P; ++c) o[c] = raw[j * (P + 1) + c];
  o[3] = raw[j * (P + 1) + P];
  for (int c = 0; c < 4; ++c) obs[j * 4 + c] = o[c];
}

__global__ void identity_rows_kernel(int total, int* __restrict__ rows) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) rows[i] = i;
}

__global__ void blend_kernel(const float* __restrict__ row_dist, const float* __restrict__ row_grad,
                             const int* __restrict__ sel_rows, int n, int K, int d, float* __restrict__ dist_out,
                             float* __restrict__ grad_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float dist, g[MAXD];
  blend(row_dist, row_grad, sel_rows + (size_t)i * K, K, d, dist, g);
  dist_out[i] = dist;
  for (int a = 0; a < d; ++a) grad_out[(size_t)i * d + a] = g[a];
}

__global__ void __launch_bounds__(128) step_kernel(StepArgs s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < s.N) step_sample(s, i, s.t, step_io_global(s, i));
}

// ------------------------------------------------------------------------------------------------
// Prefilter path, ONE launch after the scoring kernel: a WARP per sample
//   1. ranks the sample's re-scored candidate rows -- the K closest, ascending by (fp32 key, obstacle index): the
//      second half of MPPI.py:245-253's sort (the body of rank_kernel);
//   2. the group's lanes run the modulation / policy / Euler step (step_group_t, MPPI.py:101-223) on those rows: lane a
//      owns joint a, lane k row k and the policy kernels k, k + GL, ... -- bit-identical to the one-thread step_sample;
//   3. all lanes write the layer-1 table row of the NEXT state for the next step's prefilter (l1_table.cuh).
// Replaces rank_kernel + step_kernel + l1_table_kernel.  The step is a 5 k-instruction dependent chain per sample:
// with one sample per warp an SM holds ~28 such chains on 28 warps instead of one warp with 28 active lanes, so the
// schedulers have something to switch to.
// ------------------------------------------------------------------------------------------------
struct RankStepArgs {
  const float* m_rows; const int* row_base; const int* cand_cnt; const int* row_obs;
  const float* Wf0; const float* b0; uint16_t* tabA;      // tabA == nullptr: no table (last step, or no prefilter next)
  int nin; int bf16;
};

// GL lanes per sample (a power of two <= 32): 128 / GL samples per CTA.  With GL = 32 the step's registers (~128 per
// thread, allocated for all 32 lanes of a warp that uses one) allow 16 samples per SM and 4096 samples need two waves
// of the 26 us chain; GL = 8 runs four chains per warp and fits them in one.
template <int GL>
__global__ void __launch_bounds__(128) rank_step_kernel(StepArgs s, RankStepArgs r) {
  constexpr int SPB = 128 / GL;                     // samples per CTA
  __shared__ int rows_s[SPB][MAXK];
  __shared__ float qn_s[SPB][MAXD];
  __shared__ float xs_s[SPB][3 * MAXD];
  const int g = threadIdx.x / GL, gl = threadIdx.x % GL;
  const int w = blockIdx.x * SPB + g;
  const bool live = w < s.N;                        // (no early return: the shuffles below are warp-wide)
  const int K = s.K;
  {
    const int base = live ? r.row_base[w] : 0, c = live ? r.cand_cnt[w] : 0;
    float last_v = -FLT_MAX;
    int last_j = -1, last_t = 0;
    bool first = true;
    for (int kk = 0; kk < K; ++kk) {
      float bv = FLT_MAX;
      int bj = 0x7fffffff, bt = 0;
      for (int t = gl; t < c; t += GL) {
        const float v = r.m_rows[base + t];
        const int j = r.row_obs[base + t];
        const bool after = first || v > last_v || (v == last_v && j > last_j);
        if (after && (v < bv || (v == bv && j < bj))) { bv = v; bj = j; bt = t; }
      }
#pragma unroll
      for (int off = GL / 2; off > 0; off >>= 1) {   // xor offsets below GL stay inside the aligned group
        const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, off);
        const int ot = __shfl_xor_sync(0xffffffffu, bt, off);
        if (ov < bv || (ov == bv && oj < bj)) { bv = ov; bj = oj; bt = ot; }
      }
      if (bj == 0x7fffffff) { bj = last_j < 0 ? 0 : last_j; bt = last_t; }   // fewer than K candidates: repeat
      if (gl == 0) rows_s[g][kk] = base + bt;
      last_v = bv; last_j = bj; last_t = bt; first = false;
    }
  }
  __syncwarp();
  // the step: on all GL lanes where the lane-parallel form exists (bit-identical, step_device.cuh), else on lane 0
  if (step_group_supported(s)) {
    const StepIO io{s.row_dist, s.row_grad, rows_s[g], nullptr, qn_s[g]};
    if (s.d == 7) step_group_t<7, GL>(s, live ? w : 0, s.t, io, gl, live);
    else step_group_t<2, GL>(s, live ? w : 0, s.t, io, gl, live);
  } else if (gl == 0 && live) {
    step_sample(s, w, s.t, StepIO{s.row_dist, s.row_grad, rows_s[g], nullptr, qn_s[g]});
  }
  __syncwarp();
  // ---- the next state's layer-1 table rows, by the whole CTA: a thread owns two adjacent features, keeps their 3 d
  //      weights in registers and walks the CTA's samples (inputs broadcast from shared memory).  (Each group writing
  //      its own row -- 32 features per lane, the weights re-read from L2 inside every feature's dependent FMA chain --
  //      took 29 of this kernel's 39 us.)  Same FMA order as l1_feature, so a table does not depend on who wrote it.
  const bool table = r.tabA != nullptr && s.t < s.H;
  if (table && live) {
    const int d = s.d;
    if (gl < d) {
      const float v = qn_s[g][gl];
      float sn, cs;
      sincosf(v, &sn, &cs);
      xs_s[g][3 * gl] = v; xs_s[g][3 * gl + 1] = sn; xs_s[g][3 * gl + 2] = cs;
    }
  }
  __syncthreads();
  if (table) {
    const int d = s.d;
    static_assert(HID == 2 * 128, "two features per thread of a 128-thread CTA");
    const int k = 2 * threadIdx.x;
    float2 wq[MAXD], ws[MAXD], wc[MAXD];
#pragma unroll
    for (int c = 0; c < MAXD; ++c) {
      if (c < d) {
        wq[c] = *reinterpret_cast<const float2*>(r.Wf0 + (size_t)c * HID + k);
        ws[c] = *reinterpret_cast<const float2*>(r.Wf0 + (size_t)(r.nin + c) * HID + k);
        wc[c] = *reinterpret_cast<const float2*>(r.Wf0 + (size_t)(2 * r.nin + c) * HID + k);
      }
    }
    const float2 bias = r.b0 ? *reinterpret_cast<const float2*>(r.b0 + k) : make_float2(0.f, 0.f);
    const int n_here = min(SPB, s.N - blockIdx.x * SPB);
    for (int gg = 0; gg < n_here; ++gg) {
      float a0 = bias.x, a1 = bias.y;
#pragma unroll
      for (int c = 0; c < MAXD; ++c) {
        if (c < d) {
          const float x = xs_s[gg][3 * c], sn = xs_s[gg][3 * c + 1], cs = xs_s[gg][3 * c + 2];
          a0 = fmaf(wq[c].x, x, a0); a1 = fmaf(wq[c].y, x, a1);
          a0 = fmaf(ws[c].x, sn, a0); a1 = fmaf(ws[c].y, sn, a1);
          a0 = fmaf(wc[c].x, cs, a0); a1 = fmaf(wc[c].y, cs, a1);
        }
      }
      const uint32_t packed = (uint32_t)l1_to_half_bits(a0, r.bf16 != 0) | ((uint32_t)l1_to_half_bits(a1, r.bf16 != 0) << 16);
      *reinterpret_cast<uint32_t*>(r.tabA + ((size_t)(blockIdx.x * SPB + gg)) * HID + k) = packed;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel-candidate detection (policy.py:153-175): one thread per state-step, unordered atomic append
// ------------------------------------------------------------------------------------------------
struct CandArgs {
  long long total;            // N * H
  int d, nk;
  float p, thr_dist, thr_kernel, thr_dot;
  const float* traj; const float* closest; const float* dots; const float* mu; const float* sigma;
  int* out_index; int* count; long long capacity;
};

__global__ void __launch_bounds__(256) kernel_candidates_kernel(CandArgs c) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  if (idx < c.total && c.closest[idx] < c.thr_dist && c.dots[idx] < c.thr_dot) {
    keep = true;
    if (c.nk > 0) {
      float q[MAXD];
#pragma unroll
      for (int a = 0; a < MAXD; ++a) q[a] = a < c.d ? c.traj[idx * c.d + a] : 0.f;
      float cover = -FLT_MAX;
      for (int k = 0; k < c.nk; ++k) {
        float acc = 0.f;
        if (c.p == 2.f) {
#pragma unroll
          for (int a = 0; a < MAXD; ++a)
            if (a < c.d) { const float df = q[a] - c.mu[k * c.d + a]; acc += df * df; }
          acc = sqrtf(acc);
        } else {
#pragma unroll
          for (int a = 0; a < MAXD; ++a)
            if (a < c.d) acc += powf(fabsf(q[a] - c.mu[k * c.d + a]), c.p);
          acc = powf(acc, 1.f / c.p);
        }
        cover = fmaxf(cover, expf(-c.sigma[k] * (acc * acc)));          // eval_rbf_simple, policy.py:201-214
      }
      keep = cover < c.thr_kernel;
    }
  }
  // warp-aggregated append
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  if (bal) {
    const int lane = threadIdx.x & 31, leader = __ffs(bal) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(c.count, __popc(bal));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (keep) {
      const long long pos = base + __popc(bal & ((1u << lane) - 1u));
      if (pos < c.capacity) c.out_index[pos] = (int)idx;
    }
  }
}

__global__ void init_traj_kernel(const float* __restrict__ q_cur, int is_batch, int N, int H, int d,
                                 float* __restrict__ traj) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * d) return;
  const int i = idx / d, a = idx - i * d;
  traj[(size_t)i * H * d + a] = is_batch ? q_cur[idx] : q_cur[a];   // MPPI.py:99
}

// ------------------------------------------------------------------------------------------------
// Cost (cost.py:13-46) with the terminal forward kinematics (fk_num.py:7-75)
// ------------------------------------------------------------------------------------------------
struct CostArgs {
  int N, H, d, terms;
  float goal[MAXD], qmin[MAXD], qmax[MAXD];
  DhTable dh;
  const float* traj; const float* closest; float* cost;
};

// link end points P_link = T_{link+1}[:3,3] + T_{link+1}[:3,0] * a_{link+1}
__device__ __forceinline__ void fk_points(const float* q, int d, const DhTable& dh, float (*pts)[3]) {
  float Rm[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  float tv[3] = {0, 0, 0};
#pragma unroll
  for (int i = 0; i < MAXD; ++i) {
    if (i < d) {
      const float dd = dh.v[i][0], th = dh.v[i][1], aa = dh.v[i][2], al = dh.v[i][3];
      const float sa = sinf(al), ca = cosf(al), sq = sinf(q[i] + th), cq = cosf(q[i] + th);
      // modified-DH transform (fk_num.py:17-26)
      const float A[3][4] = {{cq, -sq, 0.f, aa}, {sq * ca, cq * ca, -sa, -dd * sa}, {sq * sa, cq * sa, ca, dd * ca}};
      float Rn[3][3], tn[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) Rn[r][c] = Rm[r][0] * A[0][c] + Rm[r][1] * A[1][c] + Rm[r][2] * A[2][c];
        tn[r] = Rm[r][0] * A[0][3] + Rm[r][1] * A[1][3] + Rm[r][2] * A[2][3] + tv[r];
      }
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) Rm[r][c] = Rn[r][c];
        tv[r] = tn[r];
      }
      const float an = dh.v[i + 1][2];
#pragma unroll
      for (int r = 0; r < 3; ++r) pts[i][r] = Rm[r][0] * an + tv[r];
    }
  }
}

__global__ void __launch_bounds__(128) cost_kernel(CostArgs c) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.N) return;
  const int d = c.d, H = c.H;
  const float* tr = c.traj + (size_t)i * H * d;
  float qT[MAXD], q0[MAXD];
  float sg = 0.f, s0 = 0.f;
#pragma unroll
  for (int a = 0; a < MAXD; ++a) {
    qT[a] = a < d ? tr[(size_t)(H - 1) * d + a] : 0.f;
    q0[a] = a < d ? tr[a] : 0.f;
    const float dg = a < d ? qT[a] - c.goal[a] : 0.f;
    const float d0 = a < d ? q0[a] - qT[a] : 0.f;
    sg += dg * dg;
    s0 += d0 * d0;
  }
  const float goal_cost = 10.f * sqrtf(sg);                           // cost.py:14
  int ncoll = 0, nviol = 0;
  for (int t = 0; t < H; ++t) {
    ncoll += c.closest[(size_t)i * H + t] < 0.f ? 1 : 0;              // cost.py:33-34
    for (int a = 0; a < d; ++a) {
      const float x = tr[(size_t)t * d + a];
      nviol += (x < c.qmin[a]) ? 1 : 0;
      nviol += (x > c.qmax[a]) ? 1 : 0;                               // cost.py:36-39
    }
  }
  const float coll_cost = 100.f * (float)ncoll;
  const float jl_cost = (c.terms & DSMPPI_COST_JOINT_LIMITS) ? 100.f * (nviol > 0 ? 1.f : 0.f) : 0.f;
  float inv = 1.f / sqrtf(s0);
  if (isnan(inv)) inv = 0.f;                                          // nan_to_num(0): nan -> 0,
  else if (isinf(inv)) inv = inv > 0.f ? FLT_MAX : -FLT_MAX;          // +-inf -> +-FLT_MAX
  const float stag_cost = 10.f * goal_cost * inv;                     // cost.py:17,41-43
  float fk = 0.f;
  if (c.terms & DSMPPI_COST_TERMINAL_FK) {
    float pT[MAXD][3], pG[MAXD][3];
    fk_points(qT, d, c.dh, pT);
    fk_points(c.goal, d, c.dh, pG);
#pragma unroll
    for (int l = 0; l < MAXD; ++l)
      if (l < d) {
        const float dx = pT[l][0] - pG[l][0], dy = pT[l][1] - pG[l][1], dz = pT[l][2] - pG[l][2];
        fk += sqrtf(dx * dx + dy * dy + dz * dz);                      // cost.py:27-31
      }
    c.cost[i] = goal_cost + coll_cost + jl_cost + stag_cost + 10.f * fk;   // cost.py:21
  } else {
    c.cost[i] = (c.terms & DSMPPI_COST_JOINT_LIMITS) ? goal_cost + coll_cost + jl_cost + stag_cost
                                                      : goal_cost + coll_cost + stag_cost;   // cost_toy.py:18
  }
}

// ------------------------------------------------------------------------------------------------
// True-distance provider (MPPI.distance_repulsion_fk, MPPI.py:306-313): batched modified-DH forward kinematics
// (fk_num.py:78-89: n_pts sample points on every link, at fractions linspace(0.01, 1, n_pts) of the next link's `a`),
// minimum sphere distance over (link, obstacle, point) (dist_tens, fk_num.py:142-160) and the analytic gradient of
// that distance w.r.t. the joints.  The reference differentiates sympy-generated planar closed forms
// (fk_sym_gen.py:r1..r7); here the same derivative comes from the geometric Jacobian of the DH chain,
// d|P - y|/dq_j = (P - y)/|P - y| . (z_j x (P - o_j)) for every joint j at or before the point's link, which is valid
// for any modified-DH arm (the reference marks this path "not implemented for Franka").
// LANES = 1: one thread per sample; LANES = 32: one warp per sample, lanes stride over the obstacles.
// ------------------------------------------------------------------------------------------------
constexpr int FK_MAX_PTS = 32;
struct FkDistArgs {
  int n, d, M, n_pts;
  float span[FK_MAX_PTS];    // torch.linspace(0.01, 1, n_pts), computed on the host with torch's own formula
  DhTable dh;
  const float* q; int q_stride;
  const float* obs;          // (M, 4)
  float* dist;               // (n)
  float* grad; int grad_stride;   // (n, grad_stride): first d entries written
  int* idx;                  // (n, 3) = [obstacle, link, point] or nullptr
};

template <int LANES>
__global__ void __launch_bounds__(128) fk_distance_kernel(FkDistArgs a) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = gid / LANES, lane = gid % LANES;
  if (i >= a.n) return;
  const int d = a.d;
  // frames of every joint: R[k], o[k] = rotation / origin of frame k+1 (its z axis is the axis of joint k)
  float R[MAXD][3][3], o[MAXD][3], q[MAXD];
  {
    float Rm[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
    float tv[3] = {0, 0, 0};
#pragma unroll
    for (int k = 0; k < MAXD; ++k) {
      if (k < d) {
        q[k] = a.q[(size_t)i * a.q_stride + k];
        const float dd = a.dh.v[k][0], th = a.dh.v[k][1], aa = a.dh.v[k][2], al = a.dh.v[k][3];
        const float sa = sinf(al), ca = cosf(al), sq = sinf(q[k] + th), cq = cosf(q[k] + th);
        const float A[3][4] = {{cq, -sq, 0.f, aa}, {sq * ca, cq * ca, -sa, -dd * sa}, {sq * sa, cq * sa, ca, dd * ca}};
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
          for (int c = 0; c < 3; ++c) R[k][r][c] = Rm[r][0] * A[0][c] + Rm[r][1] * A[1][c] + Rm[r][2] * A[2][c];
          o[k][r] = Rm[r][0] * A[0][3] + Rm[r][1] * A[1][3] + Rm[r][2] * A[2][3] + tv[r];
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
          for (int c = 0; c < 3; ++c) Rm[r][c] = R[k][r][c];
          tv[r] = o[k][r];
        }
      }
    }
  }
  // minimum over (link, obstacle, point); ties: first in that order, like the nested torch.min of dist_tens
  float best = FLT_MAX;
  int bl = 0, bj = 0, bp = 0;
  for (int l = 0; l < d; ++l) {
    const float an = a.dh.v[l + 1][2];
    for (int j = lane; j < a.M; j += LANES) {
      const float ox = a.obs[j * 4], oy = a.obs[j * 4 + 1], oz = a.obs[j * 4 + 2], orad = a.obs[j * 4 + 3];
      for (int p = 0; p < a.n_pts; ++p) {
        const float x = an * a.span[p];
        const float dx = R[l][0][0] * x + o[l][0] - ox, dy = R[l][1][0] * x + o[l][1] - oy,
                    dz = R[l][2][0] * x + o[l][2] - oz;
        const float dist = sqrtf(dx * dx + dy * dy + dz * dz) - orad;
        if (dist < best) { best = dist; bl = l; bj = j; bp = p; }
      }
    }
  }
  if (LANES > 1) {
    // warp argmin with the (link, obstacle, point) order as tie-break
#pragma unroll
    for (int off = LANES / 2; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, off);
      const int ol = __shfl_xor_sync(0xffffffffu, bl, off), oj = __shfl_xor_sync(0xffffffffu, bj, off),
                op = __shfl_xor_sync(0xffffffffu, bp, off);
      const bool earlier = ol < bl || (ol == bl && (oj < bj || (oj == bj && op < bp)));
      if (ov < best || (ov == best && earlier)) { best = ov; bl = ol; bj = oj; bp = op; }
    }
    if (lane != 0) return;
  }
  // gradient at the closest (link, obstacle, point)
  const float x = a.dh.v[bl + 1][2] * a.span[bp];
  float P[3], u[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) P[r] = R[bl][r][0] * x + o[bl][r];
  u[0] = P[0] - a.obs[bj * 4]; u[1] = P[1] - a.obs[bj * 4 + 1]; u[2] = P[2] - a.obs[bj * 4 + 2];
  const float un = sqrtf(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
  a.dist[i] = best;
#pragma unroll
  for (int k = 0; k < MAXD; ++k) {
    if (k < d) {
      float g = 0.f;
      if (k <= bl) {
        const float zx = R[k][0][2], zy = R[k][1][2], zz = R[k][2][2];
        const float rx = P[0] - o[k][0], ry = P[1] - o[k][1], rz = P[2] - o[k][2];
        const float cx = zy * rz - zz * ry, cy = zz * rx - zx * rz, cz = zx * ry - zy * rx;
        g = (u[0] * cx + u[1] * cy + u[2] * cz) / un;
      }
      a.grad[(size_t)i * a.grad_stride + k] = g;
    }
  }
  if (a.idx) { a.idx[i * 3] = bj; a.idx[i * 3 + 1] = bl; a.idx[i * 3 + 2] = bp; }
}

// ------------------------------------------------------------------------------------------------
// Householder basis: Q of the unblocked QR (geqr2 + org2r) of [g | e_2 .. e_d], column 0 := g/|g|
// (MPPI.py:122-127).  One thread per state-step, D compile-time so the d x d tiles stay in registers.
// ------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(128) basis_kernel(const float* __restrict__ grad, long long n,
                                                    float* __restrict__ basis) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float A[D][D], tau[D], g[D];
#pragma unroll
  for (int r = 0; r < D; ++r) {
    g[r] = grad[i * D + r];
#pragma unroll
    for (int c = 0; c < D; ++c) A[r][c] = (r == c) ? 1.f : 0.f;
  }
#pragma unroll
  for (int r = 0; r < D; ++r) A[r][0] = g[r];
#pragma unroll
  for (int k = 0; k < D; ++k) {
    // slarfg
    const float alpha = A[k][k];
    float xs = 0.f;
#pragma unroll
    for (int r = k + 1; r < D; ++r) xs += A[r][k] * A[r][k];
    const float xnorm = sqrtf(xs);
    if (xnorm == 0.f) {
      tau[k] = 0.f;
    } else {
      const float beta = -copysignf(sqrtf(alpha * alpha + xnorm * xnorm), alpha);
      tau[k] = (beta - alpha) / beta;
      const float sc = 1.f / (alpha - beta);
#pragma unroll
      for (int r = k + 1; r < D; ++r) A[r][k] *= sc;
      A[k][k] = beta;
    }
    // apply H_k to the trailing columns
#pragma unroll
    for (int c = k + 1; c < D; ++c) {
      float w = A[k][c];
#pragma unroll
      for (int r = k + 1; r < D; ++r) w += A[r][k] * A[r][c];
      w *= tau[k];
      A[k][c] -= w;
#pragma unroll
      for (int r = k + 1; r < D; ++r) A[r][c] -= A[r][k] * w;
    }
  }
  // org2r: Q = H_0 ... H_{D-1} applied to I, backwards
  float Q[D][D];
#pragma unroll
  for (int r = 0; r < D; ++r)
#pragma unroll
    for (int c = 0; c < D; ++c) Q[r][c] = (r == c) ? 1.f : 0.f;
#pragma unroll
  for (int k = D - 1; k >= 0; --k) {
#pragma unroll
    for (int c = 0; c < D; ++c) {
      float w = Q[k][c];
#pragma unroll
      for (int r = k + 1; r < D; ++r) w += A[r][k] * Q[r][c];
      w *= tau[k];
      Q[k][c] -= w;
#pragma unroll
      for (int r = k + 1; r < D; ++r) Q[r][c] -= A[r][k] * w;
    }
  }
  float ss = 0.f;
#pragma unroll
  for (int r = 0; r < D; ++r) ss += g[r] * g[r];
  const float gn = sqrtf(ss);
#pragma unroll
  for (int r = 0; r < D; ++r) Q[r][0] = g[r] / gn;                    // MPPI.py:126
  float* out = basis + i * D * D;
#pragma unroll
  for (int r = 0; r < D; ++r)
#pragma unroll
    for (int c = 0; c < D; ++c) out[r * D + c] = Q[r][c];
}

// ------------------------------------------------------------------------------------------------
// Policy update (MPPI.py:331-345, policy.py:88-113) as three reductions (SURVEY 8(e))
// ------------------------------------------------------------------------------------------------
// stats = { sum cost, N, min cost, argmin }: the two entries a sample-sharded job SUM-all-reduces are adjacent.
// Fixed order => deterministic: every CTA reduces a contiguous chunk of
// samples to (sum, min, argmin) and the last CTA to finish (ticket counter) combines the chunks in index order.
// HBM-bound: 4 B per sample, read once, coalesced.
constexpr int STATS_MAX_BLOCKS = 1024;
__global__ void __launch_bounds__(1024) cost_stats_kernel(const float* __restrict__ cost, int N,
                                                          float* __restrict__ stats, float* __restrict__ part,
                                                          unsigned int* __restrict__ ticket) {
  __shared__ float ssum[32], smin[32];
  __shared__ int sidx[32];
  __shared__ bool last;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb = gridDim.x;
  const long long chunk = ((long long)N + nb - 1) / nb;
  const long long i0 = blockIdx.x * chunk, i1 = min((long long)N, i0 + chunk);
  float s = 0.f, mn = FLT_MAX;
  int mi = 0x7fffffff;
  auto fold = [&](float om, int oi) { if (om < mn || (om == mn && oi < mi)) { mn = om; mi = oi; } };
  auto block_reduce = [&]() {          // result valid in warp 0
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, off);
      const float om = __shfl_xor_sync(0xffffffffu, mn, off);
      const int oi = __shfl_xor_sync(0xffffffffu, mi, off);
      fold(om, oi);
    }
    if (lane == 0) { ssum[w] = s; smin[w] = mn; sidx[w] = mi; }
    __syncthreads();
    if (w == 0) {
      const int nw = blockDim.x >> 5;
      s = lane < nw ? ssum[lane] : 0.f;
      mn = lane < nw ? smin[lane] : FLT_MAX;
      mi = lane < nw ? sidx[lane] : 0x7fffffff;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        const float om = __shfl_xor_sync(0xffffffffu, mn, off);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, off);
        fold(om, oi);
      }
    }
  };
  for (long long i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
    const float c = cost[i];
    s += c;
    fold(c, (int)i);
  }
  block_reduce();
  if (nb == 1) {
    if (threadIdx.x == 0) { stats[0] = s; stats[1] = (float)N; stats[2] = mn; stats[3] = (float)mi; }
    return;
  }
  if (threadIdx.x == 0) {
    part[3 * blockIdx.x + 0] = s;
    part[3 * blockIdx.x + 1] = mn;
    part[3 * blockIdx.x + 2] = __int_as_float(mi);
    __threadfence();
    last = atomicAdd(ticket, 1u) == (unsigned)nb - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  s = 0.f; mn = FLT_MAX; mi = 0x7fffffff;
  if ((int)threadIdx.x < nb) {                 // nb <= 1024 == blockDim.x: one chunk per thread, combined in index order
    s = part[3 * threadIdx.x + 0];
    mn = part[3 * threadIdx.x + 1];
    mi = __float_as_int(part[3 * threadIdx.x + 2]);
  }
  __syncthreads();
  block_reduce();
  if (threadIdx.x == 0) {
    stats[0] = s; stats[1] = (float)N; stats[2] = mn; stats[3] = (float)mi;
    *ticket = 0;                               // ready for the next launch
  }
}

struct UpdArgs {
  int N, H, d, nk, owns0, L, variant;
  const float* cost; const float* kval; const float* acts; const float* mu; const float* sigma; const float* alpha;
  const float* stats;
  float* partials;
};

constexpr int UPD_T = 256, UPD_W = UPD_T / 32;
constexpr int UPD_LMAX = 1 + NKMAX * (2 * MAXD + 3);
constexpr int UPD_EMAX = (UPD_LMAX + 31) / 32;                             // packed elements per lane, worst case

// packed = [ sum w | sum w mu (nk*d) | sum w sigma (nk) | sum w alpha (nk*d) | sum_i max_t kv*act (nk) |
//            mean_t kv[sample 0] (nk) ],  w = exp(-cost / beta),  beta = mean(cost) / 50
// A CTA owns a contiguous chunk of samples, a warp takes every 8th sample of it (two at a time, so twice the loads
// are in flight), and the lanes run over the packed elements: the live columns of a sample's (50, d) policy rows are
// contiguous, so every load is a coalesced segment (the old one-CTA-per-sample walk reached 150 GB/s at 10^6
// samples).  E = elements per lane is a template parameter so the common small policies (nk = 10) keep the register
// count, and with it the number of resident warps, where a latency-bound kernel needs them.  Fixed order: per-warp
// sums over its samples, warps combined in index order, CTAs combined by update_block_sum_kernel.
template <int E>
__global__ void __launch_bounds__(UPD_T, E <= 3 ? 4 : 2) update_partial_kernel(UpdArgs u) {
  __shared__ float red[UPD_W][32 * E];
  const int nk = u.nk, d = u.d, H = u.H, L = u.L;
  const int o_mu = 1, o_sg = o_mu + nk * d, o_al = o_sg + nk, o_mx = o_al + nk * d, o_b0 = o_mx + nk;
  const float beta = (u.stats[0] / u.stats[1]) / 50.f;               // MPPI.py:332
  const float nib = -1.f / beta;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long chunk = ((long long)u.N + gridDim.x - 1) / gridDim.x;
  const long long i0 = blockIdx.x * chunk, i1 = min((long long)u.N, i0 + chunk);
  // Branch-free address selection: the lanes of a warp fall into different segments of the packed vector, and a
  // divergent if-chain would serialise one DRAM latency per segment (that, not bandwidth, set the pace of the first
  // version: 5 us per sample pair).  Every lane issues ONE load from its own segment (lane 0 and the max_t / base
  // lanes re-read the sample's cost as a dummy), all of them before the first use.
  auto seg_ptr = [&](long long i, int idx) -> const float* {
    const float* p = u.cost + i;
    p = (idx >= o_mu && idx < o_sg) ? u.mu + (size_t)i * NKMAX * d + (idx - o_mu) : p;
    p = (idx >= o_sg && idx < o_al) ? u.sigma + (size_t)i * NKMAX + (idx - o_sg) : p;
    p = (idx >= o_al && idx < o_mx) ? u.alpha + (size_t)i * NKMAX * d + (idx - o_al) : p;
    return p;
  };
  auto max_t = [&](long long i, int k) -> float {          // max_t kernel_val * activation  (MPPI.py:336)
    const float* kv = u.kval + (size_t)i * H * NKMAX + k;
    const float* ac = u.acts + (size_t)i * H;
    float mx = -FLT_MAX;
    if (u.variant == 0) {
#pragma unroll 4
      for (int t = 0; t < H; ++t) mx = fmaxf(mx, kv[t * NKMAX] * ac[t]);
    } else {
#pragma unroll 4
      for (int t = 0; t < H; ++t) mx = fmaxf(mx, kv[t * NKMAX]);                                    // MPPI_toy.py:318
    }
    return mx;
  };
  auto base_mean = [&](long long i, int k) -> float {      // mean_t kernel_val of the noise-free sample 0  (MPPI.py:341)
    if (i != 0 || !u.owns0) return 0.f;
    float sm = 0.f;
    for (int t = 0; t < H; ++t) sm += u.kval[(size_t)t * NKMAX + k];
    return sm / (float)H;
  };
  auto finish = [&](long long i, int idx, float w, float x) -> float {
    if (idx == 0) return w;
    if (idx < o_mx) return w * x;
    if (idx < o_b0) return max_t(i, idx - o_mx);
    return base_mean(i, idx - o_b0);
  };
  float acc[E];
#pragma unroll
  for (int e = 0; e < E; ++e) acc[e] = 0.f;
  long long i = i0 + warp;
  for (; i + UPD_W < i1; i += 2 * UPD_W) {
    const float w0 = expf(nib * u.cost[i]), w1 = expf(nib * u.cost[i + UPD_W]);                      // MPPI.py:333
    float x0[E], x1[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int idx = min(lane + 32 * e, L - 1);
      x0[e] = *seg_ptr(i, idx);
      x1[e] = *seg_ptr(i + UPD_W, idx);
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int idx = lane + 32 * e;
      if (idx < L) {
        const float v0 = finish(i, idx, w0, x0[e]), v1 = finish(i + UPD_W, idx, w1, x1[e]);
        acc[e] += v0;
        acc[e] += v1;
      }
    }
  }
  if (i < i1) {
    const float w0 = expf(nib * u.cost[i]);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int idx = lane + 32 * e;
      if (idx < L) acc[e] += finish(i, idx, w0, *seg_ptr(i, idx));
    }
  }
#pragma unroll
  for (int e = 0; e < E; ++e) red[warp][lane + 32 * e] = acc[e];
  __syncthreads();
  for (int idx = threadIdx.x; idx < L; idx += UPD_T) {
    float sum = 0.f;
#pragma unroll
    for (int w2 = 0; w2 < UPD_W; ++w2) sum += red[w2][idx];
    u.partials[(size_t)blockIdx.x * L + idx] = sum;
  }
}

__global__ void update_block_sum_kernel(const float* __restrict__ partials, int blocks, int L,
                                        float* __restrict__ packed) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= L) return;
  float s = 0.f;
  for (int b = 0; b < blocks; ++b) s += partials[(size_t)b * L + idx];
  packed[idx] = s;
}

__global__ void update_finalize_kernel(const float* __restrict__ packed, int nk, int d, int variant, float n_global,
                                       float ker_thr, float rate, float* __restrict__ mu_c,
                                       float* __restrict__ sigma_c, float* __restrict__ alpha_c,
                                       int* __restrict__ n_updated) {
  const int o_mu = 1, o_sg = o_mu + nk * d, o_al = o_sg + nk, o_mx = o_al + nk * d, o_b0 = o_mx + nk;
  const float wsum = packed[0];
  int cnt = 0;
  for (int k = threadIdx.x; k < nk; k += blockDim.x) {
    // MPPI.py:338-342; MPPI_toy.py:319-320 has no sample-0 base mask
    const bool on = (packed[o_mx + k] / n_global > ker_thr) && (variant != 0 || packed[o_b0 + k] > ker_thr);
    const float r = on ? rate : 0.f;                                   // policy.py:97-99
    for (int a = 0; a < d; ++a) {
      mu_c[k * d + a] = (1.f - r) * mu_c[k * d + a] + r * (packed[o_mu + k * d + a] / wsum);
      alpha_c[k * d + a] = (1.f - r) * alpha_c[k * d + a] + r * (packed[o_al + k * d + a] / wsum);
    }
    sigma_c[k] = (1.f - r) * sigma_c[k] + r * (packed[o_sg + k] / wsum);
    cnt += on ? 1 : 0;
  }
  __shared__ int total;
  if (threadIdx.x == 0) total = 0;
  __syncthreads();
  if (cnt) atomicAdd(&total, cnt);
  __syncthreads();
  if (threadIdx.x == 0) n_updated[0] = total;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------------
#define LAUNCH_CHECK(c)              \
  do {                               \
    CUDA_TRY(cudaGetLastError());    \
    (c)->launches++;                 \
  } while (0)

int launch_rank_dense(dsmppi_ctx* c, int n, int K, bool rows_out, cudaStream_t st) {
  if (c->M <= 16) {
    rank_small_kernel<<<(n + 255) / 256, 256, 0, st>>>(c->m_rows, c->M, n, K, rows_out ? 1 : 0,
                                                       rows_out ? c->sel_rows : c->sel);
    LAUNCH_CHECK(c);
    return 0;
  }
  const int threads = 128, warps = threads / 32;
  rank_kernel<<<(n + warps - 1) / warps, threads, 0, st>>>(c->m_rows, nullptr, nullptr, nullptr, c->M, n, K,
                                                          rows_out ? 1 : 0, rows_out ? c->sel_rows : c->sel);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_identity_rows(dsmppi_ctx* c, int n, int K, cudaStream_t st) {
  identity_rows_kernel<<<(n * K + 255) / 256, 256, 0, st>>>(n * K, c->sel_rows);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_pack_obstacles(dsmppi_ctx* c, const float* raw, int M, int P, cudaStream_t st) {
  pack_obstacles_kernel<<<(M + 127) / 128, 128, 0, st>>>(raw, M, P, c->obs);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_select_candidates(dsmppi_ctx* c, int n, int K, float band, size_t cap_rows, cudaStream_t st) {
  CUDA_TRY(cudaMemsetAsync(c->counters, 0, sizeof(int), st));   // row counter only; stats accumulate
  const int threads = 128, warps = threads / 32;
  const int cap = (int)(cap_rows < 0x7fffffffu ? cap_rows : 0x7fffffffu);
  select_candidates_kernel<<<(n + warps - 1) / warps, threads, 0, st>>>(
      c->mdist, c->M, n, K, band, cap, c->cand_cnt, c->row_base, c->row_sample, c->row_obs, c->counters);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_max_abs_diff(dsmppi_ctx* c, const float* a, const float* b, long long n, float* out, cudaStream_t st) {
  CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(float), st));
  long long blocks = (n + 255) / 256;
  if (blocks > 4LL * c->sm_count) blocks = 4LL * c->sm_count;
  if (blocks < 1) blocks = 1;
  max_abs_diff_kernel<<<(unsigned)blocks, 256, 0, st>>>(a, b, n, out);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_rank_candidates(dsmppi_ctx* c, int n, int K, cudaStream_t st) {
  const int threads = 128, warps = threads / 32;
  rank_kernel<<<(n + warps - 1) / warps, threads, 0, st>>>(c->m_rows, c->row_base, c->cand_cnt, c->row_obs, c->M, n,
                                                          K, 1, c->sel_rows);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_blend(dsmppi_ctx* c, int n, int K, float* dist_out, float* grad_out, cudaStream_t st) {
  blend_kernel<<<(n + 127) / 128, 128, 0, st>>>(c->row_dist, c->row_grad, c->sel_rows, n, K, c->d, dist_out,
                                                grad_out);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_kernel_candidates(dsmppi_ctx* c, const dsmppi_candidates_args* a, cudaStream_t st) {
  CandArgs k;
  k.total = (long long)a->N * a->H;
  k.d = c->d; k.nk = a->n_kernels; k.p = a->rbf_p;
  k.thr_dist = a->thr_dist; k.thr_kernel = a->thr_kernel; k.thr_dot = a->thr_dot;
  k.traj = a->all_traj_dev; k.closest = a->closest_dist_all_dev; k.dots = a->dot_products_dev;
  k.mu = a->mu_c_dev; k.sigma = a->sigma_c_dev;
  k.out_index = a->out_index_dev; k.count = a->count_dev; k.capacity = a->capacity;
  CUDA_TRY(cudaMemsetAsync(a->count_dev, 0, sizeof(int), st));
  kernel_candidates_kernel<<<(unsigned)((k.total + 255) / 256), 256, 0, st>>>(k);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_init_traj(dsmppi_ctx* c, const dsmppi_rollout_args* a, cudaStream_t st) {
  const int total = a->N * c->d;
  init_traj_kernel<<<(total + 255) / 256, 256, 0, st>>>(a->q_cur_dev, a->q_cur_is_batch, a->N, a->H, c->d,
                                                       a->all_traj_dev);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_step(dsmppi_ctx* c, const dsmppi_rollout_args* a, int t, cudaStream_t st) {
  const StepArgs s = make_step_args(c, a, t);
  // one thread per sample, a long dependent chain each: spread small batches over all SMs (one warp per CTA)
  const int bs = a->N <= c->sm_count * 128 ? 32 : 128;
  step_kernel<<<(a->N + bs - 1) / bs, bs, 0, st>>>(s);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_rank_step(dsmppi_ctx* c, const dsmppi_rollout_args* a, int t, int table_mode, cudaStream_t st) {
  const StepArgs s = make_step_args(c, a, t);
  RankStepArgs r;
  r.m_rows = c->m_rows; r.row_base = c->row_base; r.cand_cnt = c->cand_cnt; r.row_obs = c->row_obs;
  r.Wf0 = c->net.Wf[0]; r.b0 = c->net.b[0];
  r.tabA = (table_mode >= 0 && t < a->H) ? static_cast<uint16_t*>(c->enc_q) : nullptr;
  r.nin = c->nin; r.bf16 = table_mode == DSMPPI_PASS1_TC_BF16 ? 1 : 0;
  static_assert(MAXD <= 8, "the table part reads one joint per lane of an 8-lane group");
  rank_step_kernel<8><<<(a->N + 15) / 16, 128, 0, st>>>(s, r);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_cost(dsmppi_ctx* c, const dsmppi_cost_args* a, cudaStream_t st) {
  CostArgs k;
  k.N = a->N; k.H = a->H; k.d = c->d; k.terms = a->terms;
  for (int i = 0; i < MAXD; ++i) { k.goal[i] = a->q_goal[i]; k.qmin[i] = a->q_min[i]; k.qmax[i] = a->q_max[i]; }
  k.dh = c->dh;
  k.traj = a->all_traj_dev; k.closest = a->closest_dist_all_dev; k.cost = a->cost_dev;
  cost_kernel<<<(a->N + 127) / 128, 128, 0, st>>>(k);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_fk_distance(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, int n, int n_pts,
                       const float* span_host, float* dist, float* grad, int grad_stride, int* idx, cudaStream_t st) {
  FkDistArgs a;
  if (n_pts < 1 || n_pts > FK_MAX_PTS) { dsmppi_set_error("n_pts out of range (1..32)"); return 2; }
  a.n = n; a.d = c->d; a.M = c->M; a.n_pts = n_pts;
  // fractions along a link: the caller's torch.linspace(0.01, 1, n_pts) (fk_num.py:79), or the same ramp computed
  // here (start + i * step in the lower half, end - (n - 1 - i) * step above; may differ from torch by one ulp)
  const float start = 0.01f, end = 1.f;
  const float step = n_pts > 1 ? (end - start) / (float)(n_pts - 1) : 0.f;
  for (int p = 0; p < n_pts; ++p)
    a.span[p] = span_host ? span_host[p]
                          : (p < n_pts / 2 ? start + step * (float)p : end - step * (float)(n_pts - 1 - p));
  a.dh = c->dh;
  a.q = q; a.q_stride = q_stride; a.obs = obs;
  a.dist = dist; a.grad = grad; a.grad_stride = grad_stride; a.idx = idx;
  if (c->M >= 32) {
    const long long threads = (long long)n * 32;
    fk_distance_kernel<32><<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(a);
  } else {
    fk_distance_kernel<1><<<(n + 127) / 128, 128, 0, st>>>(a);
  }
  LAUNCH_CHECK(c);
  return 0;
}

int launch_basis(dsmppi_ctx* c, const float* grad, int64_t n, float* basis, cudaStream_t st) {
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (n <= 0) return 0;
  switch (c->d) {
#define CASE(D) case D: basis_kernel<D><<<grid, 128, 0, st>>>(grad, (long long)n, basis); break;
    CASE(1) CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8)
#undef CASE
    default: dsmppi_set_error("unsupported n_dof"); return 2;
  }
  LAUNCH_CHECK(c);
  return 0;
}

int launch_cost_stats(dsmppi_ctx* c, const float* cost, int N, float* stats, cudaStream_t st) {
  // one CTA per 16 K samples, at most STATS_MAX_BLOCKS; small batches keep the single-CTA latency
  int blocks = (N + 16383) / 16384;
  if (blocks > STATS_MAX_BLOCKS) blocks = STATS_MAX_BLOCKS;
  if (blocks < 1) blocks = 1;
  cost_stats_kernel<<<blocks, 1024, 0, st>>>(cost, N, stats, c->stats_part, c->stats_ticket);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_update_partial(dsmppi_ctx* c, const dsmppi_update_args* a, const float* stats, float* packed,
                          cudaStream_t st) {
  UpdArgs u;
  u.N = a->N; u.H = a->H; u.d = c->d; u.nk = a->n_kernels; u.owns0 = a->owns_sample0; u.variant = a->variant;
  u.L = dsmppi_update_packed_len(a->n_kernels, c->d);
  u.cost = a->cost_dev; u.kval = a->kernel_val_all_dev; u.acts = a->kernel_activations_dev;
  u.mu = a->mu_tmp_dev; u.sigma = a->sigma_tmp_dev; u.alpha = a->alpha_tmp_dev; u.stats = stats;
  u.partials = c->upd_partials;
  int blocks = c->upd_blocks;
  if (blocks > (a->N + UPD_W - 1) / UPD_W) blocks = (a->N + UPD_W - 1) / UPD_W;     // at least one sample per warp
  if (blocks < 1) blocks = 1;
  if (u.L <= 32 * 3) update_partial_kernel<3><<<blocks, UPD_T, 0, st>>>(u);
  else if (u.L <= 32 * 6) update_partial_kernel<6><<<blocks, UPD_T, 0, st>>>(u);
  else update_partial_kernel<UPD_EMAX><<<blocks, UPD_T, 0, st>>>(u);
  LAUNCH_CHECK(c);
  update_block_sum_kernel<<<(u.L + 127) / 128, 128, 0, st>>>(c->upd_partials, blocks, u.L, packed);
  LAUNCH_CHECK(c);
  return 0;
}

int launch_update_finalize(dsmppi_ctx* c, const dsmppi_update_args* a, const float* packed, int* n_updated,
                           cudaStream_t st) {
  update_finalize_kernel<<<1, 64, 0, st>>>(packed, a->n_kernels, c->d, a->variant, (float)a->N_global, a->ker_thr, a->upd_rate,
                                          a->mu_c_dev, a->sigma_c_dev, a->alpha_c_dev, n_updated);
  LAUNCH_CHECK(c);
  return 0;
}
