// The fp32 (IEEE FFMA) network tile shared by exact_mlp.cu (its kernels) and tc_exact.cu (which re-scores, inside its
// whole-horizon kernel, the rows that left the fp16 range): rows -> encoded inputs -> net.nh hidden layers -> output
// layer -> analytic VJP, on R = 4 * RPT rows held feature-major in shared memory.  See exact_mlp.cu for the design notes.
// WID is the number of features the tile computes per hidden layer (64, 128 or 256, at least the network's width; the
// weights are read from the 256 x 4 frame, whose features past the network's width are zero).
// Every barrier is the named barrier 2 over the NT = nthreads(FT, WID) threads that run the tile, so a kernel may hand
// the tile to a subset of its warps (threadIdx.x < NT) while the others do something else.
#pragma once
#include "internal.cuh"

namespace exact_tile {

template <int NT>
__device__ __forceinline__ void tile_sync() { asm volatile("bar.sync 2, %0;" ::"n"(NT) : "memory"); }

// a warp computes 8 * FT features: 128 / 256 / 512 threads for FT = 8 / 4 / 2 at WID = 256
__host__ __device__ constexpr int nthreads(int FT, int WID = HID) { return 32 * (WID / (8 * FT)); }
constexpr int XS = 12;    // padded row stride of the raw-input scratch (nin <= 11)
constexpr int WS = 8;     // k-rows of weights per pipeline stage (8 KB at WID = 256)
constexpr int NSTAGE = 4; // ring depth

__device__ __forceinline__ bool row_lookup(const RowSrc& s, int r, int n_rows, int& i, int& j) {
  if (r >= n_rows) return false;
  if (s.mode == ROWS_DENSE) {
    i = r / s.M;
    j = r - i * s.M;
  } else if (s.mode == ROWS_SELECTED) {
    i = r / s.K;
    j = s.sel[r];
  } else {
    i = s.row_sample[r];
    j = s.row_obs[r];
  }
  return true;
}

// Thread tile: rows r0 .. r0+RPT-1 and FT features: FT = 8: {fa .. fa+3} (j = 0..3) and {fa+32 .. fa+35} (j = 4..7);
// FT = 4 / 2: {fa .. fa+FT-1}.
template <int FT>
struct Tile {
  int r0, fa;
  __device__ __forceinline__ void init(int tid, int RPT) {
    r0 = ((tid & 31) >> 3) * RPT;                                  // lane / 8: one of four RPT-row groups
    fa = (tid >> 5) * (8 * FT) + (tid & 7) * (FT == 8 ? 4 : FT);   // warp: feature block; lane % 8: feature group
  }
  __device__ __forceinline__ int feat(int j) const { return FT == 8 ? fa + (j & 3) + ((j >> 2) << 5) : fa + j; }
};

// FT consecutive-group values of a feature row (weights of one k, or a bias vector) for this thread's tile
template <int FT>
__device__ __forceinline__ void load_feats(const float* p, float (&w)[FT]) {
  if constexpr (FT == 8) {
    const float4 w0 = *reinterpret_cast<const float4*>(p), w1 = *reinterpret_cast<const float4*>(p + 32);
    w[0] = w0.x; w[1] = w0.y; w[2] = w0.z; w[3] = w0.w; w[4] = w1.x; w[5] = w1.y; w[6] = w1.z; w[7] = w1.w;
  } else if constexpr (FT == 4) {
    const float4 w0 = *reinterpret_cast<const float4*>(p);
    w[0] = w0.x; w[1] = w0.y; w[2] = w0.z; w[3] = w0.w;
  } else {
    const float2 w0 = *reinterpret_cast<const float2*>(p);
    w[0] = w0.x; w[1] = w0.y;
  }
}

template <int RPT>
__device__ __forceinline__ void load_rows(const float* p, float (&a)[RPT]) {
  if constexpr (RPT == 8) {
    const float4 a0 = *reinterpret_cast<const float4*>(p), a1 = *reinterpret_cast<const float4*>(p + 4);
    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
  } else if constexpr (RPT == 4) {
    const float4 a0 = *reinterpret_cast<const float4*>(p);
    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
  } else {
    const float2 a0 = *reinterpret_cast<const float2*>(p);
    a[0] = a0.x; a[1] = a0.y;
  }
}

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Packed fp32 FMA (Blackwell fma.rn.f32x2): two IEEE fused multiply-adds per issue slot, bit-identical to two
// fmaf().  The inner loop is issue-bound with scalar FFMAs (ncu: issue 68 %, fma pipe 51 %), so halving the FFMA
// issue count is what lets the pipe fill.
__device__ __forceinline__ uint64_t pack2f(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2f(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// The weight stream: GEMM g = 0..L-1 are the forward layers (Wf[g], K = nenc or WID), g = L..2L-2 the backward ones
// (Wb[L-1], .., Wb[1]), L = net->nh; stage indices run through all of them.  A stage is WS k-rows of WID features,
// taken from the 256-wide rows of the frame.
template <int WID = HID>
struct WeightStream {
  const NetDev* net;
  float* ring;            // [NSTAGE][WS][WID]
  int n0;                 // stages of GEMM 0 = ceil(nenc / WS)
  int per_pass;           // stages of one pass over a row tile (forward, or forward + backward)
  int total;              // stages in the whole stream: per_pass x number of passes this CTA makes
  int issued;             // next stage to request

  __device__ __forceinline__ void locate(int stage, const float*& src, int& rows) const {
    int g, st;
    stage %= per_pass;
    if (stage < n0) { g = 0; st = stage; }
    else { g = 1 + (stage - n0) / (WID / WS); st = (stage - n0) % (WID / WS); }
    const int K = g == 0 ? net->nenc : WID;
    const int L = net->nh;
    const float* W = g < L ? net->Wf[g] : net->Wb[2 * L - 1 - g];
    src = W + (size_t)st * WS * HID;
    rows = min(WS, K - st * WS);
  }
  // every thread requests its share of the next stage (or nothing past the end) and closes one group
  template <int NT>
  __device__ __forceinline__ void request_next() {
    if (issued < total) {
      const float* src;
      int rows;
      locate(issued, src, rows);
      float* dst = ring + (size_t)(issued % NSTAGE) * WS * WID;
      for (int c = threadIdx.x; c < rows * (WID / 4); c += NT) {
        const int kk = c / (WID / 4), f = c - kk * (WID / 4);
        cp_async16(dst + kk * WID + f * 4, src + (size_t)kk * HID + f * 4);
      }
    }
    ++issued;
    cp_async_commit();
  }
};

// acc[i][j] = sum_k act[k][r0+i] * W[k*WID + feat(j)], W arriving through the ring; `stage` is the stream position
// of this GEMM's first stage and is advanced past its last one
template <int RPT, int FT, int WID>
__device__ __forceinline__ void gemm_tile(WeightStream<WID>& ws, int& stage, int K, const float (*act)[4 * RPT],
                                          const Tile<FT>& t, float (&acc)[RPT][FT]) {
  constexpr int NT = nthreads(FT, WID);
  uint64_t acc2[RPT][FT / 2];             // acc2[i][p] = (acc[i][2p], acc[i][2p+1])
#pragma unroll
  for (int i = 0; i < RPT; ++i)
#pragma unroll
    for (int p = 0; p < FT / 2; ++p) acc2[i][p] = 0ull;
  for (int k0 = 0; k0 < K; k0 += WS, ++stage) {
    cp_async_wait<NSTAGE - 2>();          // this thread's share of `stage` has landed ...
    tile_sync<NT>();                      // ... and everybody's; the buffer of stage-1 is free again
    ws.template request_next<NT>();       // refill it with stage + NSTAGE - 1
    const float* wb = ws.ring + (size_t)(stage % NSTAGE) * WS * WID + t.fa;
    const int rows = min(WS, K - k0);
    if (rows == WS) {
#pragma unroll
      for (int kk = 0; kk < WS; ++kk) {
        float a[RPT], w[FT];
        load_rows<RPT>(&act[k0 + kk][t.r0], a);
        load_feats<FT>(wb + kk * WID, w);
        uint64_t wp[FT / 2];
#pragma unroll
        for (int p = 0; p < FT / 2; ++p) wp[p] = pack2f(w[2 * p], w[2 * p + 1]);
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const uint64_t ad = pack2f(a[i], a[i]);
#pragma unroll
          for (int p = 0; p < FT / 2; ++p) acc2[i][p] = fma2(ad, wp[p], acc2[i][p]);
        }
      }
    } else {
      for (int kk = 0; kk < rows; ++kk) {
        float a[RPT], w[FT];
        load_rows<RPT>(&act[k0 + kk][t.r0], a);
        load_feats<FT>(wb + kk * WID, w);
        uint64_t wp[FT / 2];
#pragma unroll
        for (int p = 0; p < FT / 2; ++p) wp[p] = pack2f(w[2 * p], w[2 * p + 1]);
#pragma unroll
        for (int i = 0; i < RPT; ++i) {
          const uint64_t ad = pack2f(a[i], a[i]);
#pragma unroll
          for (int p = 0; p < FT / 2; ++p) acc2[i][p] = fma2(ad, wp[p], acc2[i][p]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < RPT; ++i)
#pragma unroll
    for (int p = 0; p < FT / 2; ++p) unpack2f(acc2[i][p], acc[i][2 * p], acc[i][2 * p + 1]);
}

template <int RPT, int FT>
__device__ __forceinline__ void store_tile(float (*act)[4 * RPT], const Tile<FT>& t, const float (&v)[RPT][FT]) {
#pragma unroll
  for (int j = 0; j < FT; ++j) {
    float* p = &act[t.feat(j)][t.r0];
    if constexpr (RPT == 8) {
      *reinterpret_cast<float4*>(p) = make_float4(v[0][j], v[1][j], v[2][j], v[3][j]);
      *reinterpret_cast<float4*>(p + 4) = make_float4(v[4][j], v[5][j], v[6][j], v[7][j]);
    } else if constexpr (RPT == 4) {
      *reinterpret_cast<float4*>(p) = make_float4(v[0][j], v[1][j], v[2][j], v[3][j]);
    } else {
      *reinterpret_cast<float2*>(p) = make_float2(v[0][j], v[1][j]);
    }
  }
}

template <int RPT, int WID = HID>
struct TileSmem {
  static constexpr int R = 4 * RPT;
  static_assert(WID >= 3 * (MAXD + 3), "the encoded inputs share the activation rows");
  float (*act)[R];   // [WID][R]
  float* ring;       // [NSTAGE][WS][WID] weight stages
  float* xs;         // [R][XS]  raw inputs x = [q, p]
  float* zs;         // [R][MAXO] raw outputs
  float* rad;        // [R]
  int* lst;          // [R] argmin link
  __device__ __forceinline__ explicit TileSmem(float* smem) {
    act = reinterpret_cast<float (*)[R]>(smem);
    ring = smem + WID * R;
    xs = ring + NSTAGE * WS * WID;
    zs = xs + R * XS;
    rad = zs + R * MAXO;
    lst = reinterpret_cast<int*>(rad + R);
  }
};

// starts the weight stream of a CTA that will make `passes` passes over row tiles: the first three stages fly
// while the inputs are encoded
template <bool BWD, int NT, int WID>
__device__ __forceinline__ void stream_begin(WeightStream<WID>& ws, const NetDev* net, float* ring, int passes) {
  ws.net = net;
  ws.ring = ring;
  ws.n0 = (net->nenc + WS - 1) / WS;
  ws.per_pass = ws.n0 + (BWD ? 2 : 1) * (net->nh - 1) * (WID / WS);
  ws.total = ws.per_pass * passes;
  ws.issued = 0;
#pragma unroll
  for (int i = 0; i < NSTAGE - 1; ++i) ws.template request_next<NT>();
}

// One pass of the network over the R rows [row0, row0 + R) of `src` (rows >= n_rows are padding): forward, and with
// BWD the analytic VJP.  Called by all NT threads of the CTA; `ws` / `stage` carry the weight stream across calls.
template <bool BWD, int RPT, int FT, int WID = HID>
__device__ __forceinline__ void mlp_tile(const NetDev& net, const RowSrc& src, int row0, int n_rows,
                                         const float* q, int q_stride, const float* __restrict__ obs,
                                         uint32_t ignore_mask, float* out_m, float* out_dist, float* out_grad,
                                         const TileSmem<RPT, WID>& sm, WeightStream<WID>& ws, int& stage) {
  constexpr int R = 4 * RPT;
  constexpr int NT = nthreads(FT, WID);
  float (*act)[R] = sm.act;
  float* xs = sm.xs;
  float* zs = sm.zs;
  float* rad = sm.rad;
  int* lst = sm.lst;
  const int tid = threadIdx.x;
  Tile<FT> t;
  t.init(tid, RPT);
  const int d = net.d, nin = net.nin, nenc = net.nenc, O = net.O, L = net.nh;

  // ---- rows -> encoded inputs [x, sin x, cos x]  (network_macros_mod.py:139-140)
  for (int idx = tid; idx < R * nin; idx += NT) {
    const int r = idx % R, c = idx / R;
    int i = 0, j = 0;
    const bool valid = row_lookup(src, row0 + r, n_rows, i, j);
    float x = 0.f;
    if (valid) x = (c < d) ? q[(size_t)i * q_stride + c] : obs[j * 4 + (c - d)];
    xs[r * XS + c] = x;
    act[c][r] = x;
    act[nin + c][r] = sinf(x);
    act[2 * nin + c][r] = cosf(x);
    if (c == 0) rad[r] = valid ? obs[j * 4 + 3] : 0.f;
  }
  tile_sync<NT>();

  uint64_t mk[MAXL];       // ReLU masks of this thread's tile, bit i*FT+j
  float acc[RPT][FT];
  // ---- hidden layers: h = relu(W h + b)
#pragma unroll 1
  for (int l = 0; l < L; ++l) {
    gemm_tile<RPT, FT, WID>(ws, stage, l == 0 ? nenc : WID, act, t, acc);
    tile_sync<NT>();
    float bb[FT];
    load_feats<FT>(net.b[l] + t.fa, bb);
    uint64_t m = 0;
#pragma unroll
    for (int i = 0; i < RPT; ++i)
#pragma unroll
      for (int j = 0; j < FT; ++j) {
        const float v = acc[i][j] + bb[j];
        const bool on = v > 0.f;
        if (BWD) m |= (uint64_t)(on ? 1u : 0u) << (i * FT + j);
        acc[i][j] = on ? v : 0.f;
      }
    mk[l] = m;
    store_tile<RPT, FT>(act, t, acc);
    tile_sync<NT>();
  }

  // ---- output layer (no activation)
  for (int idx = tid; idx < R * O; idx += NT) {
    const int r = idx % R, o = idx / R;
    const float* w = net.W4 + o * HID;
    float s = 0.f;
#pragma unroll 8
    for (int k = 0; k < WID; ++k) s = fmaf(act[k][r], __ldg(w + k), s);
    zs[r * MAXO + o] = s + __ldg(net.b[4] + o);
  }
  tile_sync<NT>();

  if constexpr (!BWD) {
    // MPPI.py:236-242: /100 for the 9-link Franka net, minus radius, ignored links := 1e6, min over links
    if (tid < R && row0 + tid < n_rows) {
      float m = 3.0e38f;
      for (int o = 0; o < O; ++o) {
        float y = zs[tid * MAXO + o];
        if (net.scale != 1.f) y = y / 100.f;
        y -= rad[tid];
        if ((ignore_mask >> o) & 1u) y = 1e6f;
        m = fminf(m, y);
      }
      out_m[src.out_row ? src.out_row[row0 + tid] : row0 + tid] = m;
    }
  } else {
  // ---- pass 2: l* = argmin of the RAW output (robot_sdf.py:155), distance of that link (MPPI.py:265-274);
  //      optionally also the pass-1 ranking key (masked minimum) so one launch serves both passes
  if (tid < R) {
    int best = 0;
    float bv = zs[tid * MAXO];
    float m = 3.0e38f;
    for (int o = 0; o < O; ++o) {
      const float v = zs[tid * MAXO + o];
      if (v < bv) { bv = v; best = o; }
      float y = v;
      if (net.scale != 1.f) y = y / 100.f;
      y -= rad[tid];
      if ((ignore_mask >> o) & 1u) y = 1e6f;
      m = fminf(m, y);
    }
    lst[tid] = best;
    if (row0 + tid < n_rows) {
      float y = bv;
      if (net.scale != 1.f) y = y / 100.f;
      const int orow = src.out_row ? src.out_row[row0 + tid] : row0 + tid;
      out_dist[orow] = y - rad[tid];
      if (out_m) out_m[orow] = m;
    }
  }
  tile_sync<NT>();

  // g4 = W5[l*, :] * s4
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    const float* w = net.W4 + lst[t.r0 + i] * HID;
    const uint32_t bits = (uint32_t)(mk[L - 1] >> (i * FT)) & 0xffu;
#pragma unroll
    for (int j = 0; j < FT; ++j) acc[i][j] = ((bits >> j) & 1u) ? __ldg(w + t.feat(j)) : 0.f;
  }
  store_tile<RPT, FT>(act, t, acc);
  tile_sync<NT>();

  // g_{l-1} = (W_l^T g_l) * s_{l-1},  l = L-1, .., 1   (Wb[l] is torch's [out][in]: out = k, in = n)
#pragma unroll 1
  for (int l = L - 1; l >= 1; --l) {
    gemm_tile<RPT, FT, WID>(ws, stage, WID, act, t, acc);
    tile_sync<NT>();
    const uint64_t m = mk[l - 1];
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      const uint32_t bits = (uint32_t)(m >> (i * FT)) & 0xffu;
#pragma unroll
      for (int j = 0; j < FT; ++j) acc[i][j] = ((bits >> j) & 1u) ? acc[i][j] : 0.f;
    }
    store_tile<RPT, FT>(act, t, acc);
    tile_sync<NT>();
  }

  // a = W_1^T g_1 (only the three entries per joint that are consumed), then the encoding Jacobian:
  // dz/dx_c = a[c] + cos(x_c) a[nin+c] - sin(x_c) a[2nin+c]                       (SURVEY Appendix B)
  for (int idx = tid; idx < R * d; idx += NT) {
    const int r = idx % R, c = idx / R;
    const float* w = net.Wb[0];
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 4
    for (int k = 0; k < WID; ++k) {
      const float g = act[k][r];
      a0 = fmaf(g, __ldg(w + k * nenc + c), a0);
      a1 = fmaf(g, __ldg(w + k * nenc + nin + c), a1);
      a2 = fmaf(g, __ldg(w + k * nenc + 2 * nin + c), a2);
    }
    const float x = xs[r * XS + c];
    if (row0 + r < n_rows) {
      const int orow = src.out_row ? src.out_row[row0 + r] : row0 + r;
      out_grad[(size_t)orow * d + c] = a0 + cosf(x) * a1 - sinf(x) * a2;
    }
  }
  }  // BWD
}


constexpr size_t smem_bytes(int R, int WID = HID) {
  return (size_t)(WID * R + NSTAGE * WS * WID + R * XS + R * MAXO + R + R) * sizeof(float);
}

}  // namespace exact_tile
