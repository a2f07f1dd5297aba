// extern "C" surface of libdsmppi_b200.so (see include/dsmppi_b200.h) and the host-side orchestration of
// one rollout: per step  [tensor-core prefilter -> candidate band ->] fp32 scoring -> ranking ->
// fp32 forward+VJP on the K closest -> modulation/integration step.  Everything is stream-ordered; the
// host never waits inside the horizon loop.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "internal.cuh"

static thread_local std::string g_last_error;
void dsmppi_set_error(const std::string& msg) { g_last_error = msg; }

namespace {

template <typename T>
int grow(T*& p, size_t& cap, size_t need) {
  if (need <= cap) return 0;
  if (p) CUDA_TRY(cudaFree(p));
  p = nullptr;
  const size_t n = need + need / 8;
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&p), n * sizeof(T)));
  cap = n;
  return 0;
}

template <typename T>
int alloc(T*& p, size_t n) {
  if (p) CUDA_TRY(cudaFree(p));
  p = nullptr;
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&p), (n ? n : 1) * sizeof(T)));
  return 0;
}

constexpr int FUSE_M_MAX = 16;   // up to this many obstacles the fp32 path differentiates every pair in one launch

// The pass-1 mode that runs when `requested` is asked for with M obstacles: AUTO takes the fp16 prefilter from 64
// obstacles on, and every tensor-core mode needs the prefilter's weight images.  Each entry point resolves once and
// passes the result down; the context's own mode and obstacle count are only written by their setters.
int resolve_mode(const dsmppi_ctx* c, int requested, int M) {
  int m = requested;
  if (m == DSMPPI_PASS1_AUTO) m = (M >= 64 && c->tc_blob) ? DSMPPI_PASS1_TC_F16 : DSMPPI_PASS1_EXACT_FP32;
  if (m != DSMPPI_PASS1_EXACT_FP32 && !c->tc_blob) m = DSMPPI_PASS1_EXACT_FP32;
  return m;
}

// which of band_cal / band_cal_M / band_cal_err holds the guard band of a prefilter mode
int band_slot(int mode) { return mode == DSMPPI_PASS1_TC_BF16 ? 1 : 0; }

// Samples never interact, so a very large batch is processed in blocks of samples: it bounds the workspace
// (the (n, M) prefilter matrix is the big one: <= 1 GiB) and keeps every row index inside 31 bits.
long long sample_block(const dsmppi_ctx* c) {
  const long long block = (1LL << 28) / c->M;
  return block > (1 << 18) ? 1 << 18 : block < 1 ? 1 : block;
}

// the arguments of samples [off, off + n) of a batch
dsmppi_rollout_args slice_samples(const dsmppi_rollout_args& a, int d, long long off, int n) {
  dsmppi_rollout_args b = a;
  b.N = n;
  if (a.q_cur_is_batch) b.q_cur_dev = a.q_cur_dev + off * d;
  if (a.mu_tmp_dev) b.mu_tmp_dev = a.mu_tmp_dev + off * NKMAX * d;
  if (a.sigma_tmp_dev) b.sigma_tmp_dev = a.sigma_tmp_dev + off * NKMAX;
  if (a.alpha_tmp_dev) b.alpha_tmp_dev = a.alpha_tmp_dev + off * NKMAX * d;
  b.all_traj_dev = a.all_traj_dev + off * a.H * d;
  b.closest_dist_all_dev = a.closest_dist_all_dev + off * a.H;
  b.kernel_val_all_dev = a.kernel_val_all_dev + off * a.H * NKMAX;
  b.dot_products_dev = a.dot_products_dev + off * a.H;
  b.kernel_activations_dev = a.kernel_activations_dev + off * a.H;
  b.qdot_dev = a.qdot_dev + off * d;
  b.nn_grad_all_dev = a.nn_grad_all_dev + off * a.H * d;
  return b;
}

constexpr int WHOLE_M_MAX = 32;  // largest obstacle set a row tile of the whole-horizon kernel can hold

// Whole-horizon single launch: fp32 scoring with every (sample, obstacle) pair differentiated.  Always for
// M <= 16 (same FLOPs as the per-step launches); for 17..32 obstacles only while the batch is latency-bound,
// because differentiating all M pairs instead of the K closest costs up to 1.5x the FLOPs.
bool use_whole_horizon(const dsmppi_ctx* c, int n, int mode) {
  if (!c->fused_rollout || mode != DSMPPI_PASS1_EXACT_FP32) return false;
  if (use_tc_scoring(c)) {
    // tensor-core scoring: a CTA pair holds 2 * (128 / M) samples for the whole horizon.  Worth it while one wave of
    // pairs covers the batch (the step then costs no launch); with more tiles per pair the per-step launches win,
    // because their step kernel runs on all SMs instead of 128 / M threads per CTA
    if (c->M > WHOLE_M_MAX) return false;
    const long long per_pair = 2LL * (128 / c->M);
    return (n + per_pair - 1) / per_pair <= c->sm_count / 2;
  }
  if (c->M <= FUSE_M_MAX) return true;
  return c->M <= WHOLE_M_MAX && n <= 2 * c->sm_count;
}

// records one event of a start/stop pair on the launching stream (no host synchronisation)
int timing_mark(dsmppi_ctx* c, int kind, cudaStream_t st) {
  if (!c->timing) return 0;
  if (c->ev_used >= (int)c->ev.size()) {
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreate(&e));
    c->ev.push_back(e);
  }
  c->ev_kind = kind;
  CUDA_TRY(cudaEventRecord(c->ev[c->ev_used++], st));
  return 0;
}

// mean time of the start/stop event pairs the last call recorded
int average_event_pairs(dsmppi_ctx* c, double* avg_ms, int* pairs) {
  double tot = 0.0;
  int n = 0;
  for (int i = 0; i + 1 < c->ev_used; i += 2) {
    CUDA_TRY(cudaEventSynchronize(c->ev[i + 1]));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, c->ev[i], c->ev[i + 1]));
    tot += ms;
    ++n;
  }
  *avg_ms = n ? tot / n : 0.0;
  *pairs = n;
  return 0;
}

// The sizes below depend on the resolved pass-1 mode, and AUTO flips with the obstacle count (prefilter from 64
// obstacles on, dense fp32 scoring below): a workspace sized for one mode must not be taken for the other.
int ensure_workspace(dsmppi_ctx* c, int n, int M, int mode) {
  const size_t list_rows_now = cand_list_cap(c, n);
  if (n <= c->ws_n && M <= c->ws_M && mode == c->ws_mode && list_rows_now <= c->rowlist_cap) return 0;
  const int nn = n > c->ws_n ? n : c->ws_n;
  const int mm = M > c->ws_M ? M : c->ws_M;
  const int d = c->d;
  if (nn > c->ws_n) {
    if (alloc(c->q_work, (size_t)nn * d) || alloc(c->cand_cnt, (size_t)nn) ||
        alloc(c->row_base, (size_t)nn) || alloc(c->sel, (size_t)nn * MAXK) ||
        alloc(c->sel_rows, (size_t)nn * MAXK) || alloc(c->dist_tmp, (size_t)nn) || alloc(c->grad_tmp, (size_t)nn * d))
      return 1;
  }
  // rows scored in fp32: dense n*M when the prefilter is off, the candidate list when it is on
  const size_t list_rows = cand_list_cap(c, nn);
  size_t rows = (mode == DSMPPI_PASS1_EXACT_FP32) ? (size_t)nn * mm : list_rows;
  if (rows < list_rows) rows = list_rows;
  if (grow(c->m_rows, c->m_rows_cap, rows)) return 1;
  // rows that get a distance + gradient: all candidates (fused single launch) or the K selected
  size_t drows = list_rows;
  if (mm <= WHOLE_M_MAX && (size_t)nn * mm > drows) drows = (size_t)nn * mm;
  if (grow(c->row_dist, c->row_dist_cap, drows)) return 1;
  if (grow(c->row_grad, c->row_grad_cap, drows * d)) return 1;
  size_t cap = c->rowlist_cap;
  if (grow(c->row_sample, cap, list_rows)) return 1;
  if (grow(c->row_obs, c->rowlist_cap, list_rows)) return 1;
  if (mode != DSMPPI_PASS1_EXACT_FP32) {
    if (grow(c->mdist, c->mdist_cap, (size_t)nn * mm)) return 1;
  }
  c->ws_n = nn;
  c->ws_M = mm;
  c->ws_mode = mode;
  return 0;
}

// The caller's network (L hidden layers of width W) in the shipped 256 x 4 shape, the one storage format of every
// weight image.  Missing features get zero weights and biases: their pre-activation is 0, ReLU keeps it 0, and they
// add exact zeros downstream.  Missing layers L+1..4 are the identity on the first W features with zero bias: their
// input is already >= 0, so relu(I h) = h exactly, and their ReLU mask equals layer L's, which leaves the VJP unchanged.
struct Frame {
  std::vector<float> W[5], b[5];
  dsmppi_net net{};
};

Frame embed_net(const dsmppi_net* src, int nenc, int L, int W) {
  Frame f;
  const int O = src->n_out;
  for (int l = 0; l < 4; ++l) {
    const int in = l == 0 ? nenc : HID, in_src = l == 0 ? nenc : W;
    f.W[l].assign((size_t)HID * in, 0.f);
    f.b[l].assign(HID, 0.f);
    for (int o = 0; o < W; ++o) {
      if (l < L) {
        for (int k = 0; k < in_src; ++k) f.W[l][(size_t)o * in + k] = src->W_host[l][(size_t)o * in_src + k];
        f.b[l][o] = src->b_host[l][o];
      } else {
        f.W[l][(size_t)o * in + o] = 1.f;
      }
    }
  }
  f.W[4].assign((size_t)O * HID, 0.f);
  for (int o = 0; o < O; ++o)
    for (int k = 0; k < W; ++k) f.W[4][(size_t)o * HID + k] = src->W_host[L][(size_t)o * W + k];
  f.b[4].assign(src->b_host[L], src->b_host[L] + O);
  f.net = *src;
  f.net.n_hidden = MAXL;
  f.net.hidden_width = HID;
  for (int l = 0; l < 5; ++l) {
    f.net.W_host[l] = f.W[l].data();
    f.net.b_host[l] = f.b[l].data();
  }
  return f;
}

void tick_free(dsmppi_ctx* c);

}  // namespace

extern "C" {

const char* dsmppi_last_error(void) { return g_last_error.c_str(); }
int dsmppi_version(void) { return 103; }   // 103: dsmppi_set_obstacle_velocities

void dsmppi_modulation_default(dsmppi_modulation* m) {
  if (!m) return;
  std::memset(m, 0, sizeof(*m));
  m->ds_kind = DSMPPI_DS_LINEAR_ATTRACTOR;
  m->lvel_mid = (-1.f + 0.f) / 2.f; m->lvel_k = 10.f;       // MPPI.py:132
  m->dist_mid = (0.0f + 0.1f) / 2.f; m->dist_k = 100.f;     // MPPI.py:148-151 (the "franka" set, used by all robots)
  m->ltau_max = 5.f;                                        // MPPI.py:152
  m->goal_act_thr = 0.5f;                                   // MPPI.py:194
  m->repulsion = 0.1f;                                      // MPPI.py:216
}

void dsmppi_modulation_toy(dsmppi_modulation* m) {
  if (!m) return;
  std::memset(m, 0, sizeof(*m));
  m->ds_kind = DSMPPI_DS_MATRIX;
  for (int i = 0; i < MAXD; ++i) m->ds_A[i * MAXD + i] = -1.f;   // standaloneToy2d.py:70 (callers overwrite)
  m->fold_activation = 1;                                   // MPPI_toy.py:178-179
  m->lvel_mid = (float)((-0.2 + 0.0) / 2); m->lvel_k = 100.f;    // MPPI_toy.py:114
  m->dist_mid = (0.0f + 0.5f) / 2.f; m->dist_k = 30.f;      // MPPI_toy.py:124-127
  m->ltau_max = 3.f;                                        // MPPI_toy.py:133
  m->goal_act_thr = 0.3f;                                   // MPPI_toy.py:176
  m->repulsion = 0.05f;                                     // MPPI_toy.py:199
}

int dsmppi_ctx_create(dsmppi_ctx** out, const dsmppi_net* net, const float* dh_params_host, int32_t capacity,
                      int32_t device) {
  REQUIRE(out && net && dh_params_host, "null argument");
  REQUIRE(net->n_dof >= 1 && net->n_dof <= MAXD, "n_dof out of range (1..8)");
  REQUIRE(net->n_out >= 1 && net->n_out <= MAXO, "n_out out of range (1..16)");
  REQUIRE(capacity >= 1, "capacity must be positive");
  const int P = net->n_point_dim == 0 ? 3 : net->n_point_dim;
  REQUIRE(P == 2 || P == 3, "n_point_dim must be 2 or 3");
  const int L = net->n_hidden == 0 ? MAXL : net->n_hidden;
  const int W = net->hidden_width == 0 ? HID : net->hidden_width;
  REQUIRE(L >= 1 && L <= MAXL && W >= 1 && W <= HID,
          "unsupported network shape: the supported family is 1..4 hidden layers of one width 1..256 (n_hidden, "
          "hidden_width)");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  REQUIRE(ndev > 0 && device < ndev, "no such CUDA device (this library has no CPU fallback)");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  REQUIRE(prop.major == 10, "libdsmppi_b200 is built for sm_100a (B200) only");
  dsmppi_ctx* c = new dsmppi_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->d = net->n_dof;
  c->O = net->n_out;
  c->P = P;
  c->nin = c->d + P;
  c->nenc = 3 * c->nin;
  c->capacity = capacity;
  for (int i = 0; i <= c->d; ++i)
    for (int j = 0; j < 4; ++j) c->dh.v[i][j] = dh_params_host[i * 4 + j];
  // Every image below is built from the 256 x 4 frame, never from the caller's arrays
  const Frame fr = embed_net(net, c->nenc, L, W);
  const dsmppi_net* fnet = &fr.net;
  // fp32 weight blob: Wf[l] = W_l^T ([in][256]) and Wb[l] = W_l ([256][in]) for the hidden layers, W4, biases
  const int in_dim[5] = {c->nenc, HID, HID, HID, HID};
  auto pad = [](size_t x) { return (x + 63) / 64 * 64; };
  size_t total = 0, off_f[4], off_b[4], off_w4, off_bias[5];
  for (int l = 0; l < 4; ++l) { off_f[l] = total; total += pad((size_t)in_dim[l] * HID); }
  for (int l = 0; l < 4; ++l) { off_b[l] = total; total += pad((size_t)in_dim[l] * HID); }
  off_w4 = total; total += pad((size_t)c->O * HID);
  for (int l = 0; l < 5; ++l) { off_bias[l] = total; total += pad(HID); }
  std::vector<float> blob(total, 0.f);
  for (int l = 0; l < 4; ++l) {
    const float* Wl = fnet->W_host[l];
    for (int o = 0; o < HID; ++o)
      for (int k = 0; k < in_dim[l]; ++k) {
        blob[off_f[l] + (size_t)k * HID + o] = Wl[(size_t)o * in_dim[l] + k];
        blob[off_b[l] + (size_t)o * in_dim[l] + k] = Wl[(size_t)o * in_dim[l] + k];
      }
    std::memcpy(&blob[off_bias[l]], fnet->b_host[l], HID * sizeof(float));
  }
  std::memcpy(&blob[off_w4], fnet->W_host[4], (size_t)c->O * HID * sizeof(float));
  std::memcpy(&blob[off_bias[4]], fnet->b_host[4], (size_t)c->O * sizeof(float));
  if (cudaMalloc(reinterpret_cast<void**>(&c->weights_blob), total * sizeof(float)) != cudaSuccess) {
    delete c;
    dsmppi_set_error("cudaMalloc(weights) failed");
    return 1;
  }
  CUDA_TRY(cudaMemcpy(c->weights_blob, blob.data(), total * sizeof(float), cudaMemcpyHostToDevice));
  c->net.d = c->d; c->net.nin = c->nin; c->net.nenc = c->nenc; c->net.O = c->O;
  c->net.scale = (c->O == 9) ? 0.01f : 1.f;            // MPPI.py:236-237
  c->net.nh = L;
  c->net.width = W;
  for (int l = 0; l < 4; ++l) {
    c->net.Wf[l] = c->weights_blob + off_f[l];
    c->net.Wb[l] = c->weights_blob + off_b[l];
  }
  c->net.W4 = c->weights_blob + off_w4;
  for (int l = 0; l < 5; ++l) c->net.b[l] = c->weights_blob + off_bias[l];
  if (exact_set_attributes()) { delete c; return 1; }
  if (tc_build_images(c, fnet)) { delete c; return 1; }
  if (tcx_build_images(c, fnet)) { delete c; return 1; }
  if (const char* e = std::getenv("DSMPPI_HALF_TILES")) c->half_tiles = std::atoi(e) != 0;
  if (const char* e = std::getenv("DSMPPI_PASS1_ACC")) c->pass1_hacc = std::strcmp(e, "f32") != 0;
  c->upd_blocks = c->sm_count * 4;       // update_partial_kernel: four 256-thread CTAs per SM (56 registers per thread)
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->upd_partials),
                      (size_t)c->upd_blocks * dsmppi_update_packed_len(NKMAX, MAXD) * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->stats_tmp), 4 * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->stats_part), 3 * 1024 * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->stats_ticket), sizeof(unsigned int)));
  CUDA_TRY(cudaMemset(c->stats_ticket, 0, sizeof(unsigned int)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->packed_tmp), dsmppi_update_packed_len(NKMAX, MAXD) * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->counters), N_COUNTERS * sizeof(int)));
  CUDA_TRY(cudaMemset(c->counters, 0, N_COUNTERS * sizeof(int)));
  CUDA_TRY(cudaMallocHost(reinterpret_cast<void**>(&c->counters_host), N_COUNTERS * sizeof(int)));
  *out = c;
  return 0;
}

int dsmppi_ctx_destroy(dsmppi_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  tc_free_images(c);
  tcx_free_images(c);
  void* ptrs[] = {c->weights_blob, c->seds, c->obs, c->obs_raw, c->obs_enc, c->vel, c->obs_step, c->obs_enc_step,
                  c->q_work, c->m_rows, c->mdist, c->enc_q,
                  c->cand_cnt, c->row_base, c->row_sample, c->row_obs, c->counters, c->sel, c->fix_list,
                  c->sel_rows, c->row_dist, c->row_grad, c->dist_tmp, c->grad_tmp, c->upd_partials, c->stats_tmp, c->stats_part,
                  c->stats_ticket,
                  c->packed_tmp, c->stage};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  tick_free(c);
  if (c->s_tick) cudaStreamDestroy(c->s_tick);
  if (c->tick_ev) cudaEventDestroy(c->tick_ev);
  if (c->counters_host) cudaFreeHost(c->counters_host);
  for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
  for (cudaEvent_t e : c->pipe_ev) cudaEventDestroy(e);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  delete c;
  return 0;
}

int dsmppi_set_pass1_mode(dsmppi_ctx* c, int32_t mode, float guard_band) {
  REQUIRE(c, "null ctx");
  REQUIRE(mode >= 0 && mode <= 3, "bad pass-1 mode");
  c->pass1_mode = mode;
  c->guard_band = guard_band > 0.f ? guard_band : 0.f;   // 0: the band calibrated for this network (calibrate_band)
  return 0;       // ensure_workspace re-sizes when the resolved mode differs from the one it sized for
}

int dsmppi_set_score_mode(dsmppi_ctx* c, int32_t mode) {
  REQUIRE(c, "null ctx");
  REQUIRE(mode >= 0 && mode <= 2, "bad score mode");
  REQUIRE(mode != DSMPPI_SCORE_TC_SPLIT || c->tcx_blob, "this network does not fit the tensor-core scoring tiles");
  c->score_mode = mode;
  return 0;
}

int dsmppi_set_whole_horizon(dsmppi_ctx* c, int32_t on) {
  REQUIRE(c, "null ctx");
  c->fused_rollout = on ? 1 : 0;
  return 0;
}

int dsmppi_set_seds(dsmppi_ctx* c, const dsmppi_seds* sd, void* stream) {
  REQUIRE(c && sd, "null argument");
  REQUIRE(sd->n_gaussians >= 1 && sd->n_gaussians <= 32, "n_gaussians out of range (1..32)");
  REQUIRE(sd->priors_host && sd->pdf_den_host && sd->mu_x_host && sd->mu_y_host && sd->sigma_inv_host && sd->A_host,
          "null SEDS array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  const int G = sd->n_gaussians, d = c->d;
  std::vector<float> blob;
  blob.insert(blob.end(), sd->priors_host, sd->priors_host + G);
  blob.insert(blob.end(), sd->pdf_den_host, sd->pdf_den_host + G);
  blob.insert(blob.end(), sd->mu_x_host, sd->mu_x_host + G * d);
  blob.insert(blob.end(), sd->mu_y_host, sd->mu_y_host + G * d);
  blob.insert(blob.end(), sd->sigma_inv_host, sd->sigma_inv_host + G * d * d);
  blob.insert(blob.end(), sd->A_host, sd->A_host + G * d * d);
  if (G > c->seds_G || !c->seds) {
    if (c->seds) CUDA_TRY(cudaFree(c->seds));
    c->seds = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->seds), blob.size() * sizeof(float)));
  }
  // the host vector dies with this call: a synchronous copy ordered after earlier work on the stream
  CUDA_TRY(cudaStreamSynchronize(st));
  CUDA_TRY(cudaMemcpy(c->seds, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice));
  c->seds_G = G;
  c->seds_thr = sd->seds_thr;
  return 0;
}

int dsmppi_set_obstacles(dsmppi_ctx* c, const float* obs_dev, int32_t M, void* stream) {
  REQUIRE(c && obs_dev, "null argument");
  REQUIRE(M >= 1, "need at least one obstacle");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  if (M > c->obs_cap) {
    if (c->obs) CUDA_TRY(cudaFree(c->obs));
    c->obs = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->obs), (size_t)M * 4 * sizeof(float)));
    c->obs_cap = M;
  }
  if (c->P == 3) {
    CUDA_TRY(cudaMemcpyAsync(c->obs, obs_dev, (size_t)M * 4 * sizeof(float), cudaMemcpyDefault, st));
  } else {
    // (M, P + 1) rows [x, y, r] -> the device layout [x, y, 0, r]; the staging copy also serves host sources
    if (M > c->obs_raw_cap) {
      if (c->obs_raw) CUDA_TRY(cudaFree(c->obs_raw));
      c->obs_raw = nullptr;
      CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->obs_raw), (size_t)M * (c->P + 1) * sizeof(float)));
      c->obs_raw_cap = M;
    }
    CUDA_TRY(cudaMemcpyAsync(c->obs_raw, obs_dev, (size_t)M * (c->P + 1) * sizeof(float), cudaMemcpyDefault, st));
    if (launch_pack_obstacles(c, c->obs_raw, M, c->P, st)) return 1;
  }
  c->M = M;
  c->obs_tables_dirty = 1;      // the prefilter's per-obstacle table is rebuilt by the next launch that needs it
  c->moving = 0;                // a new obstacle set is static until its velocities are set
  return 0;
}

int dsmppi_set_obstacle_velocities(dsmppi_ctx* c, const float* vel, int32_t M, void* stream) {
  REQUIRE(c, "null ctx");
  REQUIRE(M == c->M, "velocities need one row per obstacle: M differs from the obstacle count of dsmppi_set_obstacles");
  if (!vel) {
    c->moving = 0;
    return 0;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  if (M > c->vel_cap) {
    if (c->vel) CUDA_TRY(cudaFree(c->vel));
    c->vel = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->vel), (size_t)M * 4 * sizeof(float)));
    c->vel_cap = M;
  }
  // the caller's (M, P) rows -> the (M, 4) layout of c->obs, the components past P zero
  CUDA_TRY(cudaMemsetAsync(c->vel, 0, (size_t)M * 4 * sizeof(float), st));
  CUDA_TRY(cudaMemcpy2DAsync(c->vel, 4 * sizeof(float), vel, c->P * sizeof(float), c->P * sizeof(float), M,
                             cudaMemcpyDefault, st));
  c->moving = 1;
  return 0;
}

int dsmppi_set_obstacles_host(dsmppi_ctx* c, const float* obs_host, int32_t M, void* stream) {
  return dsmppi_set_obstacles(c, obs_host, M, stream);   // cudaMemcpyDefault handles host sources
}

}  // extern "C"

// ---- guard band of the prefilter, calibrated per network ------------------------------------------------------
// The tensor-core prefilter ranks obstacles on reduced-precision distances; every obstacle within `band` of the
// K-th smallest is re-scored in fp32.  The band must exceed twice the prefilter's error, which depends on the
// network's weights: it is MEASURED for the network (and obstacle set) in hand instead of assumed -- CAL_Q random
// joint vectors in [-pi, pi]^d plus the first states of the calling batch, against every current obstacle, fp32
// scoring kernel vs prefilter; band = CAL_SAFETY x the largest difference.  One-off (re-run when the obstacle count
// changes); costs two launches and one host synchronisation.  dsmppi_set_pass1_mode(.., band > 0) overrides it.
// With `census`, the same states first take the dead-feature census (tc_census), so that the band is measured on the
// reordered, skipping kernel that will run; a new feature order voids the band of the other format too.  Should a
// calibration row itself prove a skipped feature active, the skip is dropped and the band measured again without it.
constexpr int CAL_Q = 256;
constexpr float CAL_SAFETY = 3.f;

static int calibrate_band(dsmppi_ctx* c, const float* q, int q_stride, int n, uint32_t ignore_mask, int mode,
                          cudaStream_t st, bool census) {
  const int slot = band_slot(mode);
  const int d = c->d, M = c->M;
  const int n_act = n < CAL_Q ? n : CAL_Q;
  const int nq = CAL_Q + n_act;
  std::vector<float> hq((size_t)nq * d);
  uint64_t lcg = 0x9E3779B97F4A7C15ull;
  for (size_t i = 0; i < (size_t)CAL_Q * d; ++i) {
    lcg = lcg * 6364136223846793005ull + 1442695040888963407ull;
    hq[i] = ((float)((lcg >> 40) & 0xFFFFFF) / 16777216.f * 2.f - 1.f) * 3.14159265f;
  }
  float *dq = nullptr, *ref = nullptr, *err = nullptr;
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dq), (size_t)nq * d * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&ref), (size_t)nq * M * sizeof(float)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&err), sizeof(float)));
  CUDA_TRY(cudaMemcpyAsync(dq, hq.data(), (size_t)CAL_Q * d * sizeof(float), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpy2DAsync(dq + (size_t)CAL_Q * d, d * sizeof(float), q, (size_t)q_stride * sizeof(float),
                             d * sizeof(float), n_act, cudaMemcpyDeviceToDevice, st));
  int rc = ensure_workspace(c, nq, M, mode);
  bool reordered = false;
  if (!rc && census) rc = tc_census(c, dq, nq, st, &reordered);
  if (reordered) c->band_cal[0] = c->band_cal[1] = 0.f;
  const bool measure = c->guard_band <= 0.f && (c->band_cal[slot] <= 0.f || c->band_cal_M[slot] != M);
  RowSrc src{};
  src.mode = ROWS_DENSE; src.M = M; src.n_rows = nq * M;
  if (!rc && measure) rc = launch_exact_forward(c, dq, d, c->obs, src, ignore_mask, ref, st);
  auto ck = [](cudaError_t e) {
    if (e == cudaSuccess) return 0;
    dsmppi_set_error(std::string("guard-band calibration: ") + cudaGetErrorString(e));
    return 1;
  };
  float h = 0.f;
  for (int pass = 0; !rc && measure && pass < 2; ++pass) {
    int fired = 0;                         // counter 10 of this measurement alone, cleared for the call that follows
    rc = ck(cudaMemsetAsync(c->counters + 10, 0, sizeof(int), st));
    if (!rc) rc = tc_pass1(c, dq, d, c->obs, nullptr, nq, ignore_mask, mode, st);
    if (!rc) rc = launch_max_abs_diff(c, ref, c->mdist, (long long)nq * M, err, st);
    if (!rc) rc = ck(cudaMemcpyAsync(&h, err, sizeof(float), cudaMemcpyDeviceToHost, st));
    if (!rc) rc = ck(cudaMemcpyAsync(&fired, c->counters + 10, sizeof(int), cudaMemcpyDeviceToHost, st));
    if (!rc) rc = ck(cudaMemsetAsync(c->counters + 10, 0, sizeof(int), st));
    if (!rc) rc = ck(cudaStreamSynchronize(st));
    if (rc || fired == 0) break;
    for (int l = 0; l < 3; ++l) c->pass1_skip[l] = 0;
  }
  cudaFree(dq); cudaFree(ref); cudaFree(err);
  if (rc) return rc;
  if (!measure) return 0;
  c->band_cal_err[slot] = h;
  float band = CAL_SAFETY * h;
  const float floor_band = (c->O == 9 ? 1e-3f : 1e-2f);      // never below 1 mm (cm-scaled net) / 1 cm
  if (!(band > floor_band)) band = floor_band;
  c->band_cal[slot] = band;
  c->band_cal_M[slot] = M;
  return 0;
}

// distance + gradient of n states q (row stride q_stride floats) against the obstacle rows obs, scored in the
// resolved pass-1 `mode`: fills c->row_dist / c->row_grad and the ranked row indices c->sel_rows (n, K)
// obs / obs_tab: c->obs and nullptr (the context's prefilter table), or one rollout step's positions and their table
// (launch_obstacles_at); the guard-band calibration always runs on c->obs
// table_ready / defer_rank: the rollout loop of the prefilter path hands the per-sample layer-1 table over from the
// previous step and ranks inside its fused step launch (launch_rank_step)
static int distance_pipeline(dsmppi_ctx* c, const float* q, int q_stride, const float* obs, const void* obs_tab, int n,
                             int K, uint32_t ignore_mask, int mode, cudaStream_t st, bool table_ready = false,
                             bool defer_rank = false) {
  REQUIRE(c->M >= 1, "obstacles not set");
  REQUIRE(K >= 1 && K <= MAXK, "n_closest_obs out of range (1..8)");
  REQUIRE(K <= c->M, "n_closest_obs exceeds the number of obstacles");
  if (mode != DSMPPI_PASS1_EXACT_FP32) {
    const int slot = band_slot(mode);
    const bool band_due = c->guard_band <= 0.f && (c->band_cal[slot] <= 0.f || c->band_cal_M[slot] != c->M);
    // (not while a call is repeated without the skip: the census is taken again by the next call)
    const bool census_due = !c->pass1_noskip && (c->census_M != c->M || c->census_stale);
    if (band_due || census_due) {
      if (calibrate_band(c, q, q_stride, n, ignore_mask, mode, st, census_due)) return 1;
      table_ready = false;                 // the calibration wrote ITS states' table over the one handed in
    }
  }
  if (ensure_workspace(c, n, c->M, mode)) return 1;
  RowSrc src{};
  src.M = c->M;
  src.K = K;
  if (mode == DSMPPI_PASS1_EXACT_FP32 && c->M <= FUSE_M_MAX) {
    // few obstacles: one launch scores AND differentiates every (sample, obstacle) pair
    src.mode = ROWS_DENSE;
    src.n_rows = n * c->M;
    if (timing_mark(c, use_tc_scoring(c) ? 3 : 0, st)) return 1;
    if (launch_exact_fwdbwd(c, q, q_stride, obs, src, ignore_mask, c->m_rows, c->row_dist, c->row_grad, 0, st))
      return 1;
    if (timing_mark(c, use_tc_scoring(c) ? 3 : 0, st)) return 1;
    return launch_rank_dense(c, n, K, true, st);
  }
  if (mode == DSMPPI_PASS1_EXACT_FP32) {
    // many obstacles, no tensor-core prefilter: fp32 forward on every pair, then forward + VJP on the K closest
    src.mode = ROWS_DENSE;
    src.n_rows = n * c->M;
    if (timing_mark(c, use_tc_scoring(c) ? 3 : 0, st)) return 1;
    if (launch_exact_forward(c, q, q_stride, obs, src, ignore_mask, c->m_rows, st)) return 1;
    if (timing_mark(c, use_tc_scoring(c) ? 3 : 0, st)) return 1;
    if (launch_rank_dense(c, n, K, false, st)) return 1;
    RowSrc s2{};
    s2.mode = ROWS_SELECTED;
    s2.M = c->M;
    s2.K = K;
    s2.n_rows = n * K;
    s2.sel = c->sel;
    if (launch_exact_fwdbwd(c, q, q_stride, obs, s2, ignore_mask, nullptr, c->row_dist, c->row_grad, 0, st)) return 1;
    return launch_identity_rows(c, n, K, st);
  }
  // tensor-core prefilter -> candidate band -> one fp32 launch (ranking key + distance + gradient) -> rank
  c->prefilter_used = 1;
  const float band = c->guard_band > 0.f ? c->guard_band : c->band_cal[band_slot(mode)];
  const size_t cap_rows = cand_list_cap(c, n);
  if (timing_mark(c, 1, st)) return 1;
  if (tc_pass1(c, q, q_stride, obs, obs_tab, n, ignore_mask, mode, st, table_ready)) return 1;
  if (timing_mark(c, 1, st)) return 1;
  if (launch_select_candidates(c, n, K, band, cap_rows, st)) return 1;
  src.mode = ROWS_LIST;
  src.n_rows = (int)(cap_rows < 0x7fffffffu ? cap_rows : 0x7fffffffu);
  src.n_rows_dev = c->counters;
  src.row_sample = c->row_sample;
  src.row_obs = c->row_obs;
  // the candidate count lives on the device; K + 1 per sample is what the guard band typically lets through
  if (launch_exact_fwdbwd(c, q, q_stride, obs, src, ignore_mask, c->m_rows, c->row_dist, c->row_grad,
                          (long long)n * (K + 1), st))
    return 1;
  if (defer_rank) return 0;
  return launch_rank_candidates(c, n, K, st);
}

// After a call that went through the prefilter: did every step's candidate list fit, and did every row that left the
// fp16 range of the split operands get its FFMA re-score?  One small D2H copy + a stream synchronisation -- only on the
// prefilter path, whose rollouts take milliseconds.  verdict: 0 exact, 1 repeat (the list has been re-budgeted, or the
// call must fall back to scoring every pair in fp32: *exact_mode = 1).
static int prefilter_verdict(dsmppi_ctx* c, int n_max, cudaStream_t st, int* verdict, int* exact_mode) {
  *verdict = 0;
  *exact_mode = 0;
  if (!c->prefilter_used) return 0;
  CUDA_TRY(cudaMemcpyAsync(c->counters_host, c->counters, N_COUNTERS * sizeof(int), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  const int* h = c->counters_host;
  REQUIRE(h[7] == 0, "tensor-core scoring: rows left the fp16 range and did not fit the FFMA re-scoring list "
                     "(use dsmppi_set_score_mode(DSMPPI_SCORE_FFMA) for this network)");
  if (h[9] != 0) {       // prefilter outputs that were inf / NaN (activations beyond fp16): nothing to rank them by
    *verdict = 1;
    *exact_mode = 1;
    c->exact_fallbacks++;
    return 0;
  }
  if (h[10] != 0) {      // a row proved a skipped dead feature active: the same prefilter without the skip
    *verdict = 1;
    c->pass1_noskip = 1;
    c->census_stale = 1;
    c->skip_repeats++;
    return 0;
  }
  const size_t high = (size_t)(unsigned)h[8];
  if (high <= cand_list_cap(c, n_max)) return 0;
  *verdict = 1;
  // room for the worst step seen plus a quarter; the list costs 44 bytes per row (indices, key, distance, gradient)
  const size_t want = high + high / 4;
  if (want > ((size_t)1 << 27)) {          // > 5.9 GB of rows: score every pair of this call in fp32 instead
    *exact_mode = 1;
    c->exact_fallbacks++;
  } else {
    c->cand_rows_want = want;
    c->capacity_retries++;
  }
  return 0;
}

// The prefilter path is exact by construction: a call whose candidates did not all fit the row list is detected after
// it ran (high-water mark, prefilter_verdict) and run again with a list that holds them -- or, past 2^27 rows or on
// prefilter outputs beyond fp16, once more with every pair scored in fp32 -- or, when a row proved a skipped dead feature
// active (counter 10), once more with the same prefilter and no skip.  The repeat recomputes from the same inputs.
// run(mode, attempt) does the work of one call in the resolved pass-1 `mode`; attempt is 0, 1, .. for the runs the
// verdict checks and -1 for the fp32 fallback.
template <typename Run>
static int run_exact_attempts(dsmppi_ctx* c, int mode, int n_max, cudaStream_t st, Run&& run) {
  for (int attempt = 0;; ++attempt) {
    c->prefilter_used = 0;
    CUDA_TRY(cudaMemsetAsync(c->counters + 8, 0, 3 * sizeof(int), st));
    if (const int rc = run(mode, attempt)) return rc;
    int verdict = 0, exact = 0;
    if (const int rc = prefilter_verdict(c, n_max, st, &verdict, &exact)) return rc;
    if (!verdict) return 0;
    REQUIRE(attempt < 4, "candidate row list still too small after four attempts");
    if (exact) return run(DSMPPI_PASS1_EXACT_FP32, -1);
  }
}
// (a repeat without the dead-feature skip lasts for the rest of this call only)
template <typename Run>
static int run_exact(dsmppi_ctx* c, int mode, int n_max, cudaStream_t st, Run&& run) {
  c->pass1_noskip = 0;
  const int rc = run_exact_attempts(c, mode, n_max, st, run);
  c->pass1_noskip = 0;
  return rc;
}

// The obstacle rows step t of a per-step path scores against: c->obs, or with moving obstacles their positions at
// tau = (t - 1) dt, written by one launch before the step's work (with the prefilter's per-obstacle table of `mode`)
static int step_obstacles(dsmppi_ctx* c, const dsmppi_rollout_args* a, int t, int mode, cudaStream_t st,
                          const float** obs, const void** obs_tab) {
  *obs = c->obs;
  *obs_tab = nullptr;
  if (!c->moving) return 0;
  if (launch_obstacles_at(c, (float)(t - 1) * a->dt, mode, st)) return 1;
  *obs = c->obs_step;
  if (mode != DSMPPI_PASS1_EXACT_FP32) *obs_tab = c->obs_enc_step;
  return 0;
}

// one pass over the batch (in blocks of samples) in the resolved pass-1 `mode` with the context's list budget
static int rollout_once(dsmppi_ctx* c, const dsmppi_rollout_args* a, int mode, cudaStream_t st) {
  const int d = c->d;
  const float* obs = nullptr;
  const void* obs_tab = nullptr;
  const long long block = sample_block(c);
  for (long long off = 0; off < a->N; off += block) {
    dsmppi_rollout_args b = slice_samples(*a, d, off, (int)(a->N - off < block ? a->N - off : block));
    if (launch_init_traj(c, &b, st)) return 1;
    if (a->distance_provider == DSMPPI_DISTANCE_FK) {
      // true-distance provider: FK + sphere distances write one (distance, gradient) row per sample, K = 1
      if (ensure_workspace(c, b.N, c->M, mode)) return 1;
      if (launch_identity_rows(c, b.N, 1, st)) return 1;
      b.n_closest = 1;
      for (int t = 1; t <= b.H; ++t) {
        const float* q = b.all_traj_dev + (size_t)(t - 1) * d;
        if (step_obstacles(c, &b, t, DSMPPI_PASS1_EXACT_FP32, st, &obs, &obs_tab)) return 1;
        if (launch_fk_distance(c, q, b.H * d, obs, b.N, b.fk_n_pts, b.fk_span, c->row_dist, c->row_grad, d, nullptr,
                               st))
          return 1;
        if (launch_step(c, &b, t, st)) return 1;
      }
      continue;
    }
    if (use_whole_horizon(c, b.N, mode)) {
      REQUIRE(b.n_closest >= 1 && b.n_closest <= MAXK, "n_closest_obs out of range (1..8)");
      REQUIRE(b.n_closest <= c->M, "n_closest_obs exceeds the number of obstacles");
      if (ensure_workspace(c, b.N, c->M, mode)) return 1;
      const bool tcx = use_tc_scoring(c);
      if (timing_mark(c, tcx ? 4 : 2, st)) return 1;
      if (tcx ? launch_tc_rollout(c, &b, st) : launch_rollout_fused(c, &b, st)) return 1;
      if (timing_mark(c, tcx ? 4 : 2, st)) return 1;
      continue;
    }
    if (mode != DSMPPI_PASS1_EXACT_FP32) {
      // prefilter path, four launches per step: tc_pass1 (all-pairs prefilter) -> select_candidates (guard band) ->
      // tc_exact / exact_mlp (fp32 scoring + VJP of the band; + its normally empty FFMA range fix-up) -> rank_step
      // (ranking, modulation step, and the next step's per-sample layer-1 table)
      if (tc_reserve_sample_table(c, b.N)) return 1;
      for (int t = 1; t <= b.H; ++t) {
        const float* q = b.all_traj_dev + (size_t)(t - 1) * d;        // q_prev = all_traj[:, t-1, :]
        // from step 2 on, the previous step's rank_step launch wrote the layer-1 table of these states
        if (step_obstacles(c, &b, t, mode, st, &obs, &obs_tab)) return 1;
        if (distance_pipeline(c, q, b.H * d, obs, obs_tab, b.N, b.n_closest, b.ignored_link_mask, mode, st, t > 1,
                              true))
          return 1;
        if (launch_rank_step(c, &b, t, mode, st)) return 1;
      }
      continue;
    }
    for (int t = 1; t <= b.H; ++t) {
      const float* q = b.all_traj_dev + (size_t)(t - 1) * d;          // q_prev = all_traj[:, t-1, :]
      if (step_obstacles(c, &b, t, mode, st, &obs, &obs_tab)) return 1;
      if (distance_pipeline(c, q, b.H * d, obs, obs_tab, b.N, b.n_closest, b.ignored_link_mask, mode, st)) return 1;
      if (launch_step(c, &b, t, st)) return 1;
    }
  }
  if (a->norm_basis_dev)
    if (launch_basis(c, a->nn_grad_all_dev, (int64_t)a->N * a->H, a->norm_basis_dev, st)) return 1;
  return 0;
}

extern "C" {

int dsmppi_rollout(dsmppi_ctx* c, const dsmppi_rollout_args* a, void* stream) {
  REQUIRE(c && a, "null argument");
  REQUIRE(a->N >= 1 && a->H >= 1, "N and H must be positive");
  REQUIRE(a->n_kernels >= 0 && a->n_kernels <= NKMAX, "n_kernels out of range");
  REQUIRE(a->q_cur_dev && a->all_traj_dev && a->closest_dist_all_dev && a->kernel_val_all_dev &&
              a->dot_products_dev && a->kernel_activations_dev && a->qdot_dev && a->nn_grad_all_dev,
          "null device pointer");
  REQUIRE(a->n_kernels == 0 || (a->mu_tmp_dev && a->sigma_tmp_dev && a->alpha_tmp_dev), "null policy pointer");
  REQUIRE(a->distance_provider == DSMPPI_DISTANCE_NN || a->distance_provider == DSMPPI_DISTANCE_FK,
          "unknown distance_provider");
  REQUIRE(a->distance_provider != DSMPPI_DISTANCE_FK || (c->P == 3 && a->fk_n_pts >= 1 && a->fk_n_pts <= DSMPPI_FK_MAX_PTS),
          "the FK distance provider needs 3-D obstacles and 1..32 points per link");
  REQUIRE(a->mod.ds_kind == DSMPPI_DS_LINEAR_ATTRACTOR || a->mod.ds_kind == DSMPPI_DS_MATRIX ||
              a->mod.ds_kind == DSMPPI_DS_SEDS, "unknown mod.ds_kind");
  REQUIRE(a->mod.ds_kind != DSMPPI_DS_SEDS || (c->seds && c->seds_G > 0), "SEDS parameters not set (dsmppi_set_seds)");
  REQUIRE(a->mod.lvel_k != 0.f && a->mod.dist_k != 0.f,
          "rollout_args.mod is not initialised (dsmppi_modulation_default / _toy)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  REQUIRE(c->M >= 1, "obstacles not set");
  if (!c->keep_counters) c->ev_used = 0;
  const int ev_start = c->ev_used;
  const long long block = sample_block(c);
  const int n_max = (int)(a->N < block ? a->N : block);
  // The whole call is repeated.  Counters 1..3 restart with each run the verdict checks, except that the first run
  // of a chunk of a chunked iteration adds to the earlier chunks' counts; the fp32 fallback keeps the counts of the
  // run it replaces.
  return run_exact(c, resolve_mode(c, c->pass1_mode, c->M), n_max, st, [&](int mode, int attempt) {
    c->ev_used = ev_start;
    if (attempt > 0 || (attempt == 0 && !c->keep_counters))
      CUDA_TRY(cudaMemsetAsync(c->counters + 1, 0, 3 * sizeof(int), st));
    return rollout_once(c, a, mode, st);
  });
}

int dsmppi_distance_grad(dsmppi_ctx* c, const float* q_dev, int32_t n, int32_t n_closest, uint32_t ignored_link_mask,
                         float* distance_dev, float* nn_grad_dev, void* stream) {
  REQUIRE(c && q_dev && distance_dev && nn_grad_dev, "null argument");
  REQUIRE(n >= 1, "n must be positive");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  REQUIRE(c->M >= 1, "obstacles not set");
  const long long block = sample_block(c);
  const int mode = resolve_mode(c, c->pass1_mode, c->M);
  for (long long off = 0; off < n; off += block) {
    const int nb = (int)(n - off < block ? n - off : block);
    // each block is repeated on its own
    const int rc = run_exact(c, mode, nb, st, [&](int m, int) {
      const int r = distance_pipeline(c, q_dev + off * c->d, c->d, c->obs, nullptr, nb, n_closest, ignored_link_mask, m,
                                      st);
      return r ? r : launch_blend(c, nb, n_closest, distance_dev + off, nn_grad_dev + off * c->d, st);
    });
    if (rc) return rc;
  }
  return 0;
}

int dsmppi_distance_grad_fk(dsmppi_ctx* c, const float* q_dev, int32_t n, int32_t fk_n_pts, const float* span_host,
                            float* distance_dev, float* grad_dev, int32_t* closest_idx_dev, void* stream) {
  REQUIRE(c && q_dev && distance_dev && grad_dev, "null argument");
  REQUIRE(n >= 1, "n must be positive");
  REQUIRE(c->M >= 1, "obstacles not set");
  REQUIRE(c->P == 3, "the FK distance provider needs 3-D obstacles");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_fk_distance(c, q_dev, c->d, c->obs, n, fk_n_pts, span_host, distance_dev, grad_dev, c->d,
                            closest_idx_dev, static_cast<cudaStream_t>(stream));
}

int dsmppi_debug_pass1(dsmppi_ctx* c, const float* q_dev, int32_t n, uint32_t ignored_link_mask, int32_t mode,
                       float* out_dev, void* stream) {
  REQUIRE(c && q_dev && out_dev, "null argument");
  REQUIRE(mode >= DSMPPI_PASS1_EXACT_FP32 && mode <= DSMPPI_PASS1_TC_BF16,
          "bad pass-1 mode (EXACT_FP32, TC_F16 or TC_BF16; AUTO is not a kernel)");
  REQUIRE(c->M >= 1, "obstacles not set");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  if (ensure_workspace(c, n, c->M, resolve_mode(c, mode, c->M))) return 1;
  const size_t bytes = (size_t)n * c->M * sizeof(float);
  if (mode == DSMPPI_PASS1_EXACT_FP32) {
    RowSrc src{};
    src.mode = ROWS_DENSE; src.M = c->M; src.n_rows = n * c->M;
    if (launch_exact_forward(c, q_dev, c->d, c->obs, src, ignored_link_mask, c->m_rows, st)) return 1;
    CUDA_TRY(cudaMemcpyAsync(out_dev, c->m_rows, bytes, cudaMemcpyDeviceToDevice, st));
  } else {
    REQUIRE(c->tc_blob, "tensor-core path unavailable for this network");
    if (tc_pass1(c, q_dev, c->d, c->obs, nullptr, n, ignored_link_mask, mode, st)) return 1;
    CUDA_TRY(cudaMemcpyAsync(out_dev, c->mdist, bytes, cudaMemcpyDeviceToDevice, st));
  }
  return 0;                // the next rollout re-sizes for its own mode (ensure_workspace keys on it)
}

int dsmppi_norm_basis(dsmppi_ctx* c, const float* grad_dev, int64_t n, float* basis_dev, void* stream) {
  REQUIRE(c && grad_dev && basis_dev, "null argument");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_basis(c, grad_dev, n, basis_dev, static_cast<cudaStream_t>(stream));
}

int dsmppi_kernel_candidates(dsmppi_ctx* c, const dsmppi_candidates_args* a, void* stream) {
  REQUIRE(c && a && a->all_traj_dev && a->closest_dist_all_dev && a->dot_products_dev && a->out_index_dev &&
              a->count_dev,
          "null argument");
  REQUIRE(a->N >= 1 && a->H >= 1 && (long long)a->N * a->H < (1LL << 31), "N * H must fit 31 bits");
  REQUIRE(a->n_kernels >= 0 && a->n_kernels <= NKMAX, "n_kernels out of range");
  REQUIRE(a->n_kernels == 0 || (a->mu_c_dev && a->sigma_c_dev), "null policy pointer");
  REQUIRE(a->capacity >= 1, "capacity must be positive");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_kernel_candidates(c, a, static_cast<cudaStream_t>(stream));
}

int dsmppi_cost(dsmppi_ctx* c, const dsmppi_cost_args* a, void* stream) {
  REQUIRE(c && a && a->all_traj_dev && a->closest_dist_all_dev && a->cost_dev, "null argument");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_cost(c, a, static_cast<cudaStream_t>(stream));
}

int32_t dsmppi_update_packed_len(int32_t nk, int32_t d) { return 1 + nk * (2 * d + 3); }

int dsmppi_update_cost_stats(dsmppi_ctx* c, const float* cost_dev, int32_t N, float* stats_dev, void* stream) {
  REQUIRE(c && cost_dev && stats_dev, "null argument");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_cost_stats(c, cost_dev, N, stats_dev, static_cast<cudaStream_t>(stream));
}

int dsmppi_update_partial(dsmppi_ctx* c, const dsmppi_update_args* a, const float* stats_dev, float* packed_dev,
                          void* stream) {
  REQUIRE(c && a && stats_dev && packed_dev, "null argument");
  REQUIRE(a->n_kernels >= 0 && a->n_kernels <= NKMAX, "n_kernels out of range");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_update_partial(c, a, stats_dev, packed_dev, static_cast<cudaStream_t>(stream));
}

int dsmppi_update_finalize(dsmppi_ctx* c, const dsmppi_update_args* a, const float* packed_dev,
                           int32_t* n_updated_dev, void* stream) {
  REQUIRE(c && a && packed_dev && n_updated_dev, "null argument");
  CUDA_TRY(cudaSetDevice(c->device));
  return launch_update_finalize(c, a, packed_dev, n_updated_dev, static_cast<cudaStream_t>(stream));
}

int dsmppi_iteration_host(dsmppi_ctx* c, dsmppi_iteration_host_args* h, void* stream) {
  REQUIRE(c && h, "null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaSetDevice(c->device));
  const dsmppi_rollout_args& r = h->rollout;
  const size_t N = r.N, H = r.H, d = c->d;
  REQUIRE(N >= 1 && H >= 1, "N and H must be positive");
  const size_t nk = r.n_kernels;
  // staging layout (floats)
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += (n + 3) / 4 * 4; return o; };
  const size_t o_q = take(r.q_cur_is_batch ? N * d : d), o_mu = take(N * NKMAX * d), o_sg = take(N * NKMAX),
               o_al = take(N * NKMAX * d), o_tr = take(N * H * d), o_cd = take(N * H), o_kv = take(N * H * NKMAX),
               o_dp = take(N * H), o_ka = take(N * H), o_qd = take(N * d), o_gr = take(N * H * d), o_co = take(N),
               o_muc = take(NKMAX * d), o_sgc = take(NKMAX), o_alc = take(NKMAX * d), o_nu = take(4);
  if (grow(c->stage, c->stage_cap, off)) return 1;
  float* S = c->stage;
  int64_t h2d = 0, d2h = 0;
  auto up = [&](size_t o, const float* src, size_t n) {
    h2d += (int64_t)(n * sizeof(float));
    return cudaMemcpyAsync(S + o, src, n * sizeof(float), cudaMemcpyHostToDevice, st);
  };
  auto down = [&](float* dst, size_t o, size_t n) {
    d2h += (int64_t)(n * sizeof(float));
    return cudaMemcpyAsync(dst, S + o, n * sizeof(float), cudaMemcpyDeviceToHost, st);
  };
  // A batch of more than two chunks is pipelined (below); DSMPPI_HOST_CHUNK overrides the chunk size (0 = never).
  size_t CHUNK = (size_t)1 << 17;
  if (const char* e = std::getenv("DSMPPI_HOST_CHUNK")) CHUNK = (size_t)std::atoll(e);
  const bool pipelined = CHUNK > 0 && N > 2 * CHUNK;
  h2d += (int64_t)((r.q_cur_is_batch ? N * d : d) * sizeof(float)) + (int64_t)(N * nk * (2 * d + 1) * sizeof(float));
  if (!pipelined || !r.q_cur_is_batch)
    CUDA_TRY(cudaMemcpyAsync(S + o_q, h->q_cur_host, (r.q_cur_is_batch ? N * d : d) * sizeof(float),
                             cudaMemcpyHostToDevice, st));
  if (nk > 0 && !pipelined) {
    // only the live kernel columns travel: (N, 50, d) rows are strided, so copy with a 2-D memcpy
    CUDA_TRY(cudaMemcpy2DAsync(S + o_mu, NKMAX * d * sizeof(float), h->mu_tmp_host, NKMAX * d * sizeof(float),
                               nk * d * sizeof(float), N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpy2DAsync(S + o_al, NKMAX * d * sizeof(float), h->alpha_tmp_host, NKMAX * d * sizeof(float),
                               nk * d * sizeof(float), N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpy2DAsync(S + o_sg, NKMAX * sizeof(float), h->sigma_tmp_host, NKMAX * sizeof(float),
                               nk * sizeof(float), N, cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(up(o_muc, h->mu_c_host, NKMAX * d));
  CUDA_TRY(up(o_sgc, h->sigma_c_host, NKMAX));
  CUDA_TRY(up(o_alc, h->alpha_c_host, NKMAX * d));
  dsmppi_rollout_args a = r;
  a.q_cur_dev = S + o_q; a.mu_tmp_dev = S + o_mu; a.sigma_tmp_dev = S + o_sg; a.alpha_tmp_dev = S + o_al;
  a.all_traj_dev = S + o_tr; a.closest_dist_all_dev = S + o_cd; a.kernel_val_all_dev = S + o_kv;
  a.dot_products_dev = S + o_dp; a.kernel_activations_dev = S + o_ka; a.qdot_dev = S + o_qd;
  a.nn_grad_all_dev = S + o_gr; a.norm_basis_dev = nullptr;
  dsmppi_cost_args ca{};
  ca.N = r.N; ca.H = r.H; ca.terms = h->cost_terms;
  for (int i = 0; i < MAXD; ++i) { ca.q_goal[i] = r.q_goal[i]; ca.q_min[i] = h->q_min[i]; ca.q_max[i] = h->q_max[i]; }
  ca.all_traj_dev = a.all_traj_dev; ca.closest_dist_all_dev = a.closest_dist_all_dev; ca.cost_dev = S + o_co;
  if (!pipelined) {
    if (dsmppi_rollout(c, &a, stream)) return 1;
    if (launch_cost(c, &ca, st)) return 1;
  } else {
    // ---- large batch: samples never interact before the policy update, so the batch moves through
    //      [H2D on s_in] -> [rollout + cost on the caller's stream] -> [D2H on s_out] in chunks of samples; with the
    //      copies of neighbouring chunks under the compute of this one the iteration costs max(copy, compute), not the sum
    const size_t n_chunks = (N + CHUNK - 1) / CHUNK;
    if (!c->s_in) CUDA_TRY(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
    if (!c->s_out) CUDA_TRY(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
    while (c->pipe_ev.size() < 2 * n_chunks + 2) {
      cudaEvent_t e;
      CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      c->pipe_ev.push_back(e);
    }
    cudaEvent_t ev_start = c->pipe_ev[2 * n_chunks], ev_drained = c->pipe_ev[2 * n_chunks + 1];
    CUDA_TRY(cudaEventRecord(ev_start, st));              // the small uploads above, and whatever the caller queued
    CUDA_TRY(cudaStreamWaitEvent(c->s_in, ev_start, 0));
    CUDA_TRY(cudaStreamWaitEvent(c->s_out, ev_start, 0));
    c->ev_used = 0;
    CUDA_TRY(cudaMemsetAsync(c->counters + 1, 0, 3 * sizeof(int), st));
    struct KeepCounters {                                   // cleared on every exit path, error returns included
      dsmppi_ctx* c;
      explicit KeepCounters(dsmppi_ctx* ctx) : c(ctx) { c->keep_counters = 1; }
      ~KeepCounters() { c->keep_counters = 0; }
    } keep(c);
    int rc = 0;
    for (size_t k = 0; k < n_chunks && !rc; ++k) {
      const size_t o = k * CHUNK, n = N - o < CHUNK ? N - o : CHUNK;
      cudaEvent_t ev_in = c->pipe_ev[2 * k], ev_out = c->pipe_ev[2 * k + 1];
      if (r.q_cur_is_batch)
        CUDA_TRY(cudaMemcpyAsync(S + o_q + o * d, h->q_cur_host + o * d, n * d * sizeof(float), cudaMemcpyHostToDevice,
                                 c->s_in));
      if (nk > 0) {
        CUDA_TRY(cudaMemcpy2DAsync(S + o_mu + o * NKMAX * d, NKMAX * d * sizeof(float), h->mu_tmp_host + o * NKMAX * d,
                                   NKMAX * d * sizeof(float), nk * d * sizeof(float), n, cudaMemcpyHostToDevice, c->s_in));
        CUDA_TRY(cudaMemcpy2DAsync(S + o_al + o * NKMAX * d, NKMAX * d * sizeof(float), h->alpha_tmp_host + o * NKMAX * d,
                                   NKMAX * d * sizeof(float), nk * d * sizeof(float), n, cudaMemcpyHostToDevice, c->s_in));
        CUDA_TRY(cudaMemcpy2DAsync(S + o_sg + o * NKMAX, NKMAX * sizeof(float), h->sigma_tmp_host + o * NKMAX,
                                   NKMAX * sizeof(float), nk * sizeof(float), n, cudaMemcpyHostToDevice, c->s_in));
      }
      CUDA_TRY(cudaEventRecord(ev_in, c->s_in));
      CUDA_TRY(cudaStreamWaitEvent(st, ev_in, 0));
      const dsmppi_rollout_args b = slice_samples(a, c->d, (long long)o, (int)n);
      rc = dsmppi_rollout(c, &b, stream);
      if (rc) break;
      dsmppi_cost_args cb = ca;
      cb.N = (int)n;
      cb.all_traj_dev = b.all_traj_dev; cb.closest_dist_all_dev = b.closest_dist_all_dev; cb.cost_dev = ca.cost_dev + o;
      rc = launch_cost(c, &cb, st);
      if (rc) break;
      CUDA_TRY(cudaEventRecord(ev_out, st));
      CUDA_TRY(cudaStreamWaitEvent(c->s_out, ev_out, 0));
      auto down_c = [&](float* dst, size_t off_f, size_t per_sample) {
        return cudaMemcpyAsync(dst + o * per_sample, S + off_f + o * per_sample, n * per_sample * sizeof(float),
                               cudaMemcpyDeviceToHost, c->s_out);
      };
      CUDA_TRY(down_c(h->all_traj_host, o_tr, H * d));
      CUDA_TRY(down_c(h->closest_dist_all_host, o_cd, H));
      if (nk > 0)
        CUDA_TRY(cudaMemcpy2DAsync(h->kernel_val_all_host + o * H * NKMAX, NKMAX * sizeof(float),
                                   S + o_kv + o * H * NKMAX, NKMAX * sizeof(float), nk * sizeof(float), n * H,
                                   cudaMemcpyDeviceToHost, c->s_out));
      CUDA_TRY(down_c(h->dot_products_host, o_dp, H));
      CUDA_TRY(down_c(h->kernel_activations_host, o_ka, H));
      CUDA_TRY(down_c(h->qdot_host, o_qd, d));
      CUDA_TRY(down_c(h->cost_host, o_co, 1));
    }
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(ev_drained, c->s_out));
    CUDA_TRY(cudaStreamWaitEvent(st, ev_drained, 0));      // the caller's stream is done when the last copy-out is
  }
  // sample-sharded caller: the two exchanges of SURVEY 8(e) happen inside this call through the caller's hook (it
  // all-reduces its own device buffers on `stream`); without a hook this is the single-GPU iteration
  const bool sharded = h->exchange != nullptr;
  REQUIRE(!sharded || (h->stats_dev && h->packed_dev && h->N_global >= r.N),
          "a sharded iteration needs stats_dev, packed_dev and N_global");
  float* stats_buf = sharded ? h->stats_dev : c->stats_tmp;
  float* packed_buf = sharded ? h->packed_dev : c->packed_tmp;
  dsmppi_update_args ua{};
  ua.N = r.N; ua.H = r.H; ua.n_kernels = r.n_kernels; ua.variant = h->update_variant;
  ua.owns_sample0 = sharded ? h->owns_sample0 : 1;
  ua.N_global = sharded ? h->N_global : r.N;
  ua.ker_thr = h->ker_thr; ua.upd_rate = h->upd_rate;
  ua.cost_dev = S + o_co; ua.kernel_val_all_dev = a.kernel_val_all_dev;
  ua.kernel_activations_dev = a.kernel_activations_dev;
  ua.mu_tmp_dev = a.mu_tmp_dev; ua.sigma_tmp_dev = a.sigma_tmp_dev; ua.alpha_tmp_dev = a.alpha_tmp_dev;
  ua.mu_c_dev = S + o_muc; ua.sigma_c_dev = S + o_sgc; ua.alpha_c_dev = S + o_alc;
  if (launch_cost_stats(c, ua.cost_dev, r.N, stats_buf, st)) return 1;
  if (sharded) REQUIRE(h->exchange(h->exchange_user, DSMPPI_EXCHANGE_COST_STATS) == 0, "exchange hook failed (cost stats)");
  if (launch_update_partial(c, &ua, stats_buf, packed_buf, st)) return 1;
  if (sharded) REQUIRE(h->exchange(h->exchange_user, DSMPPI_EXCHANGE_PACKED_SUMS) == 0, "exchange hook failed (packed sums)");
  if (launch_update_finalize(c, &ua, packed_buf, reinterpret_cast<int*>(S + o_nu), st)) return 1;
  if (!pipelined) {
    CUDA_TRY(down(h->all_traj_host, o_tr, N * H * d));
    CUDA_TRY(down(h->closest_dist_all_host, o_cd, N * H));
    if (nk > 0) {
      CUDA_TRY(cudaMemcpy2DAsync(h->kernel_val_all_host, NKMAX * sizeof(float), S + o_kv, NKMAX * sizeof(float),
                                 nk * sizeof(float), N * H, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(down(h->dot_products_host, o_dp, N * H));
    CUDA_TRY(down(h->kernel_activations_host, o_ka, N * H));
    CUDA_TRY(down(h->qdot_host, o_qd, N * d));
    CUDA_TRY(down(h->cost_host, o_co, N));
  } else {
    d2h += (int64_t)((N * H * d + 3 * N * H + N * d + N) * sizeof(float));
  }
  if (nk > 0) d2h += (int64_t)(N * H * nk * sizeof(float));
  CUDA_TRY(down(h->mu_c_host, o_muc, NKMAX * d));
  CUDA_TRY(down(h->sigma_c_host, o_sgc, NKMAX));
  CUDA_TRY(down(h->alpha_c_host, o_alc, NKMAX * d));
  CUDA_TRY(cudaMemcpyAsync(h->n_updated_host, S + o_nu, sizeof(int), cudaMemcpyDeviceToHost, st));
  d2h += sizeof(int);
  CUDA_TRY(cudaStreamSynchronize(st));
  h->h2d_bytes = h2d;
  h->d2h_bytes = d2h;
  return 0;
}

int64_t dsmppi_launch_count(const dsmppi_ctx* c) { return c ? c->launches : 0; }

int dsmppi_pass1_stats(dsmppi_ctx* c, int64_t* rescored_pairs, int64_t* band_overflows, int32_t* mode, void* stream) {
  REQUIRE(c, "null ctx");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int host[4] = {0, 0, 0, 0};
  CUDA_TRY(cudaMemcpyAsync(host, c->counters, sizeof(host), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (band_overflows) *band_overflows = host[1];
  if (rescored_pairs) {
    unsigned long long v;
    std::memcpy(&v, &host[2], sizeof(v));
    *rescored_pairs = (int64_t)v;
  }
  if (mode) *mode = resolve_mode(c, c->pass1_mode, c->M);
  return 0;
}

int dsmppi_prefilter_skip_stats(dsmppi_ctx* c, int32_t* skipped_ksteps, int64_t* repeated_calls) {
  REQUIRE(c, "null argument");
  if (skipped_ksteps)
    for (int l = 0; l < 3; ++l) skipped_ksteps[l] = c->pass1_skip[l];
  if (repeated_calls) *repeated_calls = c->skip_repeats;
  return 0;
}

int dsmppi_exactness_stats(dsmppi_ctx* c, int64_t* capacity_retries, int64_t* exact_fallbacks, float* guard_band,
                           float* calibration_error) {
  REQUIRE(c, "null ctx");
  const int slot = band_slot(resolve_mode(c, c->pass1_mode, c->M));
  if (capacity_retries) *capacity_retries = c->capacity_retries;
  if (exact_fallbacks) *exact_fallbacks = c->exact_fallbacks;
  if (guard_band) *guard_band = c->guard_band > 0.f ? c->guard_band : c->band_cal[slot];
  if (calibration_error) *calibration_error = c->band_cal_err[slot];
  return 0;
}

int dsmppi_score_stats(dsmppi_ctx* c, int32_t* mode, int64_t* range_fixup_rows, int64_t* dropped_rows, void* stream) {
  REQUIRE(c, "null ctx");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int host[2] = {0, 0};
  CUDA_TRY(cudaMemcpyAsync(host, c->counters + 6, sizeof(host), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (mode) *mode = use_tc_scoring(c) ? DSMPPI_SCORE_TC_SPLIT : DSMPPI_SCORE_FFMA;
  if (range_fixup_rows) *range_fixup_rows = host[0];
  if (dropped_rows) *dropped_rows = host[1];
  return 0;
}

int dsmppi_enable_kernel_timing(dsmppi_ctx* c, int32_t on) {
  REQUIRE(c, "null ctx");
  c->timing = on;
  return 0;
}

int dsmppi_kernel_timing_ex(dsmppi_ctx* c, int32_t* kind, double* ms_per_launch, int32_t* launches) {
  REQUIRE(c, "null ctx");
  double avg;
  int n;
  if (average_event_pairs(c, &avg, &n)) return 1;
  if (kind) *kind = c->ev_kind;
  if (ms_per_launch) *ms_per_launch = avg;
  if (launches) *launches = n;
  return 0;
}

int dsmppi_kernel_timing(dsmppi_ctx* c, double* pass1_ms, int32_t* pass1_n, double* exact_ms, int32_t* exact_n) {
  REQUIRE(c, "null ctx");
  double avg;
  int n;
  if (average_event_pairs(c, &avg, &n)) return 1;
  if (pass1_ms) *pass1_ms = c->ev_kind == 1 ? avg : 0.0;
  if (pass1_n) *pass1_n = c->ev_kind == 1 ? n : 0;
  if (exact_ms) *exact_ms = c->ev_kind == 0 ? avg : 0.0;
  if (exact_n) *exact_n = c->ev_kind == 0 ? n : 0;
  return 0;
}

}  // extern "C"

// ---- control tick ------------------------------------------------------------------------------------------------
namespace {
struct TickLayout {
  size_t q, obs, mu, sg, al, in_total;
  size_t tr, cd, dp, ka, qd, gr, kv, out_total;
};
TickLayout tick_layout(const dsmppi_ctx* c, const dsmppi_rollout_args& r, int M) {
  TickLayout L{};
  const size_t N = r.N, H = r.H, d = c->d, P1 = c->P + 1;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += (n + 3) / 4 * 4; return o; };
  L.q = take(r.q_cur_is_batch ? N * d : d); L.obs = take((size_t)M * P1);
  L.mu = take(N * NKMAX * d); L.sg = take(N * NKMAX); L.al = take(N * NKMAX * d);
  L.in_total = off;
  off = 0;
  L.tr = take(N * H * d); L.cd = take(N * H); L.dp = take(N * H); L.ka = take(N * H); L.qd = take(N * d);
  L.gr = take(N * H * d); L.kv = take(N * H * NKMAX);
  L.out_total = off;
  return L;
}
void tick_free(dsmppi_ctx* c) {
  if (c->tick_exec) cudaGraphExecDestroy(c->tick_exec);
  if (c->tick_graph) cudaGraphDestroy(c->tick_graph);
  c->tick_exec = nullptr; c->tick_graph = nullptr;
  if (c->tick_h_in) cudaFreeHost(c->tick_h_in);
  if (c->tick_h_out) cudaFreeHost(c->tick_h_out);
  if (c->tick_d_in) cudaFree(c->tick_d_in);
  if (c->tick_d_out) cudaFree(c->tick_d_out);
  c->tick_h_in = c->tick_h_out = c->tick_d_in = c->tick_d_out = nullptr;
  c->tick_in_floats = c->tick_out_floats = 0;
  c->tick_key.clear();
}
}  // namespace

extern "C" int dsmppi_tick(dsmppi_ctx* c, dsmppi_tick_args* t, void* stream) {
  REQUIRE(c && t, "null argument");
  const dsmppi_rollout_args& r = t->rollout;
  REQUIRE(r.N >= 1 && r.H >= 1 && t->n_obs >= 1, "N, H and n_obs must be positive");
  REQUIRE(t->q_cur_host && t->obs_host && t->all_traj_host && t->closest_dist_all_host && t->kernel_val_all_host &&
              t->dot_products_host && t->kernel_activations_host && t->qdot_host && t->nn_grad_all_host,
          "null host pointer");
  REQUIRE(r.n_kernels == 0 || (t->mu_tmp_host && t->sigma_tmp_host && t->alpha_tmp_host), "null policy pointer");
  REQUIRE(r.mod.ds_kind != DSMPPI_DS_SEDS && r.distance_provider == DSMPPI_DISTANCE_NN,
          "the graphed tick covers the linear / matrix nominal DS with the network distance");
  REQUIRE(!c->moving, "the graphed tick covers static obstacles (clear the velocities, or call dsmppi_rollout)");
  CUDA_TRY(cudaSetDevice(c->device));
  // the prefilter path cannot be captured (it ends with a host-side verdict)
  REQUIRE(resolve_mode(c, c->pass1_mode, t->n_obs) == DSMPPI_PASS1_EXACT_FP32,
          "the graphed tick needs the dense fp32 scoring path (few obstacles)");
  REQUIRE(!c->timing, "kernel timing events cannot be recorded into a graph");
  cudaStream_t caller = static_cast<cudaStream_t>(stream);
  if (!c->s_tick) {
    CUDA_TRY(cudaStreamCreateWithFlags(&c->s_tick, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&c->tick_ev, cudaEventDisableTiming));
  }
  const TickLayout L = tick_layout(c, r, t->n_obs);
  const size_t d = c->d, N = r.N, H = r.H, P1 = c->P + 1;
  // key: every scalar of the argument block (device pointers zeroed) + M
  dsmppi_rollout_args k = r;
  k.q_cur_dev = k.mu_tmp_dev = k.sigma_tmp_dev = k.alpha_tmp_dev = nullptr;
  k.all_traj_dev = k.closest_dist_all_dev = k.kernel_val_all_dev = k.dot_products_dev = k.kernel_activations_dev = nullptr;
  k.qdot_dev = k.nn_grad_all_dev = k.norm_basis_dev = nullptr;
  std::vector<unsigned char> key(sizeof(k) + sizeof(int32_t) + 3 * sizeof(int));
  std::memcpy(key.data(), &k, sizeof(k));
  std::memcpy(key.data() + sizeof(k), &t->n_obs, sizeof(int32_t));
  const int modes[3] = {c->pass1_mode, c->score_mode, c->fused_rollout};
  std::memcpy(key.data() + sizeof(k) + sizeof(int32_t), modes, sizeof(modes));
  const bool rebuild = !c->tick_exec || key != c->tick_key;
  t->recaptured = rebuild ? 1 : 0;
  if (rebuild) {
    CUDA_TRY(cudaStreamSynchronize(c->s_tick));
    if (L.in_total != c->tick_in_floats || L.out_total != c->tick_out_floats) {
      tick_free(c);
      CUDA_TRY(cudaMallocHost(reinterpret_cast<void**>(&c->tick_h_in), L.in_total * sizeof(float)));
      CUDA_TRY(cudaMallocHost(reinterpret_cast<void**>(&c->tick_h_out), L.out_total * sizeof(float)));
      CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->tick_d_in), L.in_total * sizeof(float)));
      CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c->tick_d_out), L.out_total * sizeof(float)));
      std::memset(c->tick_h_in, 0, L.in_total * sizeof(float));
      c->tick_in_floats = L.in_total; c->tick_out_floats = L.out_total;
    } else {
      if (c->tick_exec) cudaGraphExecDestroy(c->tick_exec);
      if (c->tick_graph) cudaGraphDestroy(c->tick_graph);
      c->tick_exec = nullptr; c->tick_graph = nullptr;
    }
    CUDA_TRY(cudaMemset(c->tick_d_out, 0, L.out_total * sizeof(float)));     // dead kernel_val columns stay zero
    CUDA_TRY(cudaDeviceSynchronize());
  }
  // inputs -> pinned staging
  float* hi = c->tick_h_in;
  std::memcpy(hi + L.q, t->q_cur_host, (r.q_cur_is_batch ? N * d : d) * sizeof(float));
  std::memcpy(hi + L.obs, t->obs_host, (size_t)t->n_obs * P1 * sizeof(float));
  if (r.n_kernels > 0) {
    std::memcpy(hi + L.mu, t->mu_tmp_host, N * NKMAX * d * sizeof(float));
    std::memcpy(hi + L.sg, t->sigma_tmp_host, N * NKMAX * sizeof(float));
    std::memcpy(hi + L.al, t->alpha_tmp_host, N * NKMAX * d * sizeof(float));
  }
  dsmppi_rollout_args a = r;
  float* di = c->tick_d_in; float* do_ = c->tick_d_out;
  a.q_cur_dev = di + L.q; a.mu_tmp_dev = di + L.mu; a.sigma_tmp_dev = di + L.sg; a.alpha_tmp_dev = di + L.al;
  a.all_traj_dev = do_ + L.tr; a.closest_dist_all_dev = do_ + L.cd; a.kernel_val_all_dev = do_ + L.kv;
  a.dot_products_dev = do_ + L.dp; a.kernel_activations_dev = do_ + L.ka; a.qdot_dev = do_ + L.qd;
  a.nn_grad_all_dev = do_ + L.gr; a.norm_basis_dev = nullptr;
  auto sequence = [&](cudaStream_t st) -> int {
    CUDA_TRY(cudaMemcpyAsync(di, hi, L.in_total * sizeof(float), cudaMemcpyHostToDevice, st));
    if (dsmppi_set_obstacles(c, di + L.obs, t->n_obs, st)) return 1;
    if (dsmppi_rollout(c, &a, st)) return 1;
    CUDA_TRY(cudaMemcpyAsync(c->tick_h_out, do_, L.out_total * sizeof(float), cudaMemcpyDeviceToHost, st));
    return 0;
  };
  CUDA_TRY(cudaEventRecord(c->tick_ev, caller));                 // ordered after whatever the caller has queued
  CUDA_TRY(cudaStreamWaitEvent(c->s_tick, c->tick_ev, 0));
  if (rebuild) {
    if (sequence(c->s_tick)) return 1;                           // eager pass: sizes the workspace outside the capture
    CUDA_TRY(cudaStreamSynchronize(c->s_tick));
    CUDA_TRY(cudaStreamBeginCapture(c->s_tick, cudaStreamCaptureModeThreadLocal));
    const int rc = sequence(c->s_tick);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(c->s_tick, &g);
    if (rc || e != cudaSuccess) {
      if (g) cudaGraphDestroy(g);
      if (!rc) dsmppi_set_error(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
      return 1;
    }
    c->tick_graph = g;
    CUDA_TRY(cudaGraphInstantiate(&c->tick_exec, g, 0));
    c->tick_key = key;
  }
  CUDA_TRY(cudaGraphLaunch(c->tick_exec, c->s_tick));
  CUDA_TRY(cudaStreamSynchronize(c->s_tick));
  const float* ho = c->tick_h_out;
  std::memcpy(t->all_traj_host, ho + L.tr, N * H * d * sizeof(float));
  std::memcpy(t->closest_dist_all_host, ho + L.cd, N * H * sizeof(float));
  std::memcpy(t->dot_products_host, ho + L.dp, N * H * sizeof(float));
  std::memcpy(t->kernel_activations_host, ho + L.ka, N * H * sizeof(float));
  std::memcpy(t->qdot_host, ho + L.qd, N * d * sizeof(float));
  std::memcpy(t->nn_grad_all_host, ho + L.gr, N * H * d * sizeof(float));
  std::memcpy(t->kernel_val_all_host, ho + L.kv, N * H * NKMAX * sizeof(float));
  return 0;
}
