// Micro-benchmarks behind the tiling decisions of tc_pass1.cu (run on a B200 through gpurun):
//   1. tcgen05.ld / tcgen05.st throughput per SM for 4 and 8 warps,
//   2. tcgen05.mma cta_group::2 "ts" issue floor for the two shapes the kernel uses (M=256, N=128 / 256, K=16),
//   3. both at once (does draining an accumulator slow the tensor pipe down?),
//   4. the production kernel itself built with -DDSMPPI_TC_PROF: per-phase cycle accounting of the row
//      warps and of the MMA issuer on a Franka-shelf-sized problem.
// Build:  nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -DDSMPPI_TC_PROF \
//              -I include -I optimalmodulationds_b200/csrc tools/tc_microbench.cu -o tools/tc_microbench
// Run:    tc_microbench [n [M]]        all of the above, random-init net, random obstacles
//         tc_microbench power           the bare MMA loop at full power (fp32 / fp16 accumulators)
//         tc_microbench phase FILE [n]  only 4., on the net and obstacles of FILE (tools/tc_phase_inputs.py writes it),
//                                       after the dead-feature census of the library (tc_census) on 128 of the states
#include <cstdio>
#include <random>
#include <string>

#include "../optimalmodulationds_b200/csrc/tc_pass1.cu"

void dsmppi_set_error(const std::string& msg) { fprintf(stderr, "error: %s\n", msg.c_str()); }

namespace {

constexpr int MB_SMEM = 2 * SZ_WHH + 1024;   // two 32 KB B halves + barriers

// mode 0: LDTM (x32 loads, `per_wait` loads in flight), mode 1: STTM, mode 2: MMA N=128 (two halves), mode 3:
// MMA N=256, mode 4: MMA N=128 with warps 0..3 draining the other accumulator half all the time.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NTHREADS, 1)
mb_kernel(int mode, int iters, int nwarps, int per_wait, long long* out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const uint32_t bar = sbase + 2 * SZ_WHH;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + 2 * SZ_WHH + 64);
  volatile int* stop = reinterpret_cast<volatile int*>(smem + 2 * SZ_WHH + 128);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  // operands: pseudo-random fp16 in (-1, 1) (a constant operand toggles few wires and understates the power draw)
  for (int i = tid; i < 2 * SZ_WHH / 4; i += NTHREADS) {
    uint32_t x = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
    x ^= x >> 13; x *= 0x5bd1e995u; x ^= x >> 15;
    reinterpret_cast<uint32_t*>(smem)[i] = (x & 0x83ff83ffu) | 0x38003800u;   // sign + mantissa, exponent of 0.5..1
  }
  if (tid == 0) *stop = 0;
  if (warp == MMA_WARP) {
    if (lane == 0) {
      mbar_init(bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc_512_2cta(smem_u32((const void*)tmem_ptr_smem));
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  cluster_sync_all();
  const uint32_t lane_addr = (uint32_t)((warp & 3) * 32) << 16;
  long long cyc = 0;
  uint32_t sink = 0;
  if (mode >= 2 && warp < 4) {            // the A operand (TMEM) gets the same kind of data
    uint32_t v[32];
    for (int g = 0; g < 4; ++g) {
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        uint32_t x = (uint32_t)(tid * 131 + g * 32 + k) * 2654435761u;
        x ^= x >> 13; x *= 0x5bd1e995u; x ^= x >> 15;
        v[k] = (x & 0x83ff83ffu) | 0x38003800u;
      }
      tmem_st32<0>(tmem_base + lane_addr + TM_A0 + g * 32, v);
    }
    tc_wait_st();
    tc_fence_before();
  }
  __syncthreads();
  tc_fence_after();
  if (mode <= 1 && warp < nwarps) {
    const uint32_t t0 = tmem_base + lane_addr + (warp >> 2) * 128;
    uint32_t v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = k;
    const long long c0 = clock64();
    for (int it = 0; it < iters; ++it) {
      if (mode == 0) {
        for (int g = 0; g < 4; g += per_wait) {
          for (int j = 0; j < per_wait; ++j) {
            tmem_ld32(t0 + (g + j) * 32, v);
            sink ^= v[0] ^ v[31];
          }
          tc_wait_ld();
        }
      } else {
        for (int g = 0; g < 4; ++g) tmem_st32<0>(t0 + g * 32, v);
        tc_wait_st();
      }
    }
    cyc = clock64() - c0;
    if (lane == 0) out[(size_t)blockIdx.x * 9 + warp] = cyc;
  }
  if (mode >= 2) {
    if (warp == MMA_WARP && rank == 0 && lane == 0) {
      // modes 5 / 6: the loop of mode 2 with an fp16 (instead of fp32) accumulator, for the power comparison below
      const uint32_t acc_bit = (mode == 5) ? (1u << 4) : 0u;
      const uint32_t idesc128 = make_idesc(0, 256, 128) ^ acc_bit, idesc256 = make_idesc(0, 256, 256);
      const long long c0 = clock64();
      for (int it = 0; it < iters; ++it) {
        if (mode == 3) {
          for (uint32_t ks = 0; ks < 16; ++ks)
            mma_ts_2cta(tmem_base + TM_DLO, tmem_base + TM_A0 + ks * 8, make_desc(sbase + ks * 2 * 128 * 16, 128 * 16),
                        idesc256, ks > 0);
        } else {
          for (int h = 0; h < (mode == 4 ? 1 : 2); ++h)
            for (uint32_t ks = 0; ks < 16; ++ks)
              mma_ts_2cta(tmem_base + (h ? TM_DHI : TM_DLO), tmem_base + TM_A0 + ks * 8,
                          make_desc(sbase + h * SZ_WHH + ks * 2 * 64 * 16, 64 * 16), idesc128, ks > 0);
        }
      }
      mma_commit_2cta(bar);
      mbar_wait(bar, 0);
      cyc = clock64() - c0;
      out[(size_t)blockIdx.x * 9 + MMA_WARP] = cyc;
      *stop = 1;
    } else if (mode == 4 && warp < 4) {
      // drain D_hi continuously while the tensor pipe accumulates into D_lo
      uint32_t v[32];
      long long n = 0;
      const long long c0 = clock64();
      while (!*stop && rank == 0) {
        for (int g = 0; g < 4; ++g) {
          tmem_ld32(tmem_base + lane_addr + TM_DHI + g * 32, v);
          sink ^= v[0];
        }
        tc_wait_ld();
        ++n;
      }
      cyc = clock64() - c0;
      if (lane == 0 && rank == 0) { out[(size_t)blockIdx.x * 9 + warp] = cyc; out[(size_t)(blockIdx.x + 1) * 9 + warp] = n; }
    }
  }
  if (sink == 0x12345678u) out[0] = sink;
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == MMA_WARP) {
    __syncwarp();
    tmem_free_512_2cta(tmem_base);
  }
}

// Sustained rate under the power cap: the MMA loop alone on every SM for a few seconds, fp32 against fp16 accumulators.
void run_power(const char* name, int mode, int iters, long long* dout) {
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  mb_kernel<<<148, NTHREADS, MB_SMEM>>>(mode, iters / 20, 0, 0, dout);   // warm-up
  cudaEventRecord(e0);
  mb_kernel<<<148, NTHREADS, MB_SMEM>>>(mode, iters, 0, 0, dout);
  cudaEventRecord(e1);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(e)); exit(1); }
  float ms;
  cudaEventElapsedTime(&ms, e0, e1);
  const double flops = (double)iters * 32 * 2.0 * 256 * 128 * 16 * 74;
  printf("%-44s : %8.1f ms -> %.1f TFLOP/s sustained\n", name, ms, flops / ms * 1e-9);
}

void run_mb(const char* name, int mode, int iters, int nwarps, int per_wait, long long* dout, double unit_bytes_or_mma) {
  cudaMemset(dout, 0, 2 * 148 * 9 * sizeof(long long));
  mb_kernel<<<2, NTHREADS, MB_SMEM>>>(mode, iters, nwarps, per_wait, dout);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("%s: %s\n", name, cudaGetErrorString(e)); exit(1); }
  long long h[18];
  cudaMemcpy(h, dout, sizeof(h), cudaMemcpyDeviceToHost);
  if (mode <= 1) {
    long long mx = 0;
    for (int w = 0; w < nwarps; ++w) mx = h[w] > mx ? h[w] : mx;
    const double bytes = (double)iters * nwarps * 4 * 32 * 32 * 4;
    printf("%-44s warps=%d per_wait=%d : %8lld cyc  -> %.1f B/cyc/SM\n", name, nwarps, per_wait, mx, bytes / mx);
  } else {
    const double n_mma = (double)iters * (mode == 3 ? 16 : (mode == 4 ? 16 : 32));
    printf("%-44s : %8lld cyc for %.0f MMAs -> %.1f cyc/MMA", name, h[MMA_WARP], n_mma, h[MMA_WARP] / n_mma);
    if (mode == 4) printf("   drain warps: %lld x 16 KB in %lld cyc -> %.1f B/cyc/SM", h[9], h[0], (double)h[9] * 4 * 16384 / h[0]);
    printf("\n");
  }
}

}  // namespace

// FILE of `phase`: int32 M, then float32 W0 (256 x 30), b0, W1..W3 (256 x 256 each), b1..b3, W4 (9 x 256), b4 in
// torch orientation, then the (M, 4) obstacles
bool read_phase_inputs(const char* path, std::vector<float> (&W)[5], std::vector<float> (&b)[5], std::vector<float>& obs,
                       int& M) {
  FILE* f = fopen(path, "rb");
  if (!f) return false;
  const int in_dim[5] = {30, 256, 256, 256, 256}, out_dim[5] = {256, 256, 256, 256, 9};
  bool ok = fread(&M, 4, 1, f) == 1 && M > 0;
  for (int l = 0; ok && l < 5; ++l) {
    W[l].resize((size_t)in_dim[l] * out_dim[l]);
    b[l].resize(out_dim[l]);
    ok = fread(W[l].data(), 4, W[l].size(), f) == W[l].size() && fread(b[l].data(), 4, b[l].size(), f) == b[l].size();
  }
  if (ok) {
    obs.resize((size_t)M * 4);
    ok = fread(obs.data(), 4, obs.size(), f) == obs.size();
  }
  fclose(f);
  return ok;
}

float* upload(const std::vector<float>& h) {
  float* d = nullptr;
  cudaMalloc(&d, h.size() * 4);
  cudaMemcpy(d, h.data(), h.size() * 4, cudaMemcpyHostToDevice);
  return d;
}

int main(int argc, char** argv) {
  const bool phase = argc > 2 && std::string(argv[1]) == "phase";
  const int n = phase ? (argc > 3 ? atoi(argv[3]) : 4096) : argc > 1 ? atoi(argv[1]) : 4096;
  int M = phase ? 0 : argc > 2 ? atoi(argv[2]) : 2064;
  cudaFuncSetAttribute(mb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MB_SMEM);
  long long* dout;
  cudaMalloc(&dout, 2 * 148 * 9 * sizeof(long long));
  if (argc > 1 && std::string(argv[1]) == "power") {
    for (int rep = 0; rep < 2; ++rep) {
      run_power("MMA loop, fp32 accumulators, 148 SMs", 2, 2500000, dout);
      run_power("MMA loop, fp16 accumulators, 148 SMs", 5, 2500000, dout);
    }
    return 0;
  }
  std::vector<float> W[5], b[5], obs;
  if (phase) {
    if (!read_phase_inputs(argv[2], W, b, obs, M)) { fprintf(stderr, "cannot read %s\n", argv[2]); return 1; }
  } else {
    for (int nw : {4, 8})
      for (int pw : {1, 2, 4}) run_mb("tcgen05.ld 32x32b.x32", 0, 2000, nw, pw, dout, 0);
    for (int nw : {4, 8}) run_mb("tcgen05.st 32x32b.x32", 1, 2000, nw, 4, dout, 0);
    run_mb("tcgen05.mma cg2 ts M256 N128 K16 (2 halves)", 2, 200, 0, 0, dout, 0);
    run_mb("tcgen05.mma cg2 ts M256 N256 K16", 3, 200, 0, 0, dout, 0);
    run_mb("tcgen05.mma N128 + 4 warps draining D_hi", 4, 400, 0, 0, dout, 0);
  }

  // ---- the production kernel with phase accounting
  dsmppi_ctx c;
  c.d = 7; c.O = 9; c.nin = 10; c.nenc = 30; c.M = M; c.sm_count = 148;
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, 0);
  c.sm_count = prop.multiProcessorCount;
  std::mt19937 rng(0);
  std::normal_distribution<float> nd(0.f, 1.f);
  const int in_dim[5] = {30, 256, 256, 256, 256}, out_dim[5] = {256, 256, 256, 256, 9};
  dsmppi_net net;
  net.n_dof = 7; net.n_out = 9;
  for (int l = 0; l < 5; ++l) {
    if (!phase) {
      W[l].resize((size_t)in_dim[l] * out_dim[l]);
      b[l].resize(out_dim[l]);
      for (auto& x : W[l]) x = nd(rng) / sqrtf((float)in_dim[l]);
      for (auto& x : b[l]) x = 0.1f * nd(rng);
    }
    net.W_host[l] = W[l].data();
    net.b_host[l] = b[l].data();
  }
  if (tc_build_images(&c, &net)) return 1;
  // the layer-1 tables are computed from the fp32 weights (W1^T, [3 nin][256]) and the layer-1 bias on the device;
  // the census reads layers 2..4 the same way (forward orientation [in][256])
  for (int l = 0; l < 4; ++l) {
    std::vector<float> wf((size_t)in_dim[l] * 256);
    for (int o = 0; o < 256; ++o)
      for (int k = 0; k < in_dim[l]; ++k) wf[(size_t)k * 256 + o] = W[l][(size_t)o * in_dim[l] + k];
    c.net.Wf[l] = upload(wf);
    c.net.b[l] = upload(b[l]);
  }
  c.net.d = 7; c.net.nin = 10; c.net.nenc = 30; c.net.O = 9; c.P = 3;
  std::vector<float> q((size_t)n * 7);
  if (!phase) {
    obs.resize((size_t)M * 4);
    for (auto& x : obs) x = 0.5f * nd(rng);
  }
  // joint vectors uniform in [-pi, pi]^7 (tools/dead_feature_study.py: the census features stay dead on them)
  std::uniform_real_distribution<float> ud(-3.14159265f, 3.14159265f);
  for (auto& x : q) x = phase ? ud(rng) : nd(rng);
  cudaMalloc(&c.obs, obs.size() * 4);
  cudaMemcpy(c.obs, obs.data(), obs.size() * 4, cudaMemcpyHostToDevice);
  float* dq;
  cudaMalloc(&dq, q.size() * 4);
  cudaMemcpy(dq, q.data(), q.size() * 4, cudaMemcpyHostToDevice);
  cudaMalloc(&c.mdist, (size_t)n * M * 4);
  cudaMalloc(reinterpret_cast<void**>(&c.counters), N_COUNTERS * sizeof(int));   // (the kernel counts non-finite outputs)
  cudaMemset(c.counters, 0, N_COUNTERS * sizeof(int));
  if (phase) {
    bool reordered = false;
    if (tc_census(&c, dq, n < 128 ? n : 128, 0, &reordered)) return 1;
    printf("census: %d / %d / %d K-steps skipped in the layer 3 / layer 4 / output GEMMs\n", c.pass1_skip[0],
           c.pass1_skip[1], c.pass1_skip[2]);
  }
  const size_t prof_n = (size_t)c.sm_count * 9 * 8;
  cudaMalloc(reinterpret_cast<void**>(&c.stage), prof_n * sizeof(long long));
  cudaMemset(c.stage, 0, prof_n * sizeof(long long));
  cudaEvent_t e0, e1;                                   // (tc_pass1 builds the per-obstacle table on first use)
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 3; ++rep) {
    cudaEventRecord(e0);
    if (tc_pass1(&c, dq, 7, c.obs, nullptr, n, 0x7, DSMPPI_PASS1_TC_F16, 0)) return 1;
    cudaEventRecord(e1);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("tc_pass1: %s\n", cudaGetErrorString(e)); return 1; }
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    const double fl = (double)n * M * 2.0 * (30 * 256 + 3 * 256 * 256 + 256 * 9);
    printf("tc_pass1 (PROF build) n=%d M=%d: %.3f ms  %.1f TFLOP/s algorithmic\n", n, M, ms, fl / ms * 1e-9);
  }
  int counters[N_COUNTERS];
  cudaMemcpy(counters, c.counters, sizeof(counters), cudaMemcpyDeviceToHost);
  printf("rows with a skipped feature active: %d, non-finite rows: %d\n", counters[10], counters[9]);
  std::vector<long long> prof(prof_n);
  cudaMemcpy(prof.data(), c.stage, prof_n * sizeof(long long), cudaMemcpyDeviceToHost);
  const char* row_names[8] = {"wait D_lo full", "drain D_lo (ld+pack 64)", "pack lo 64..127", "wait D_hi full",
                              "drain D_hi (ld+st+pack)", "pack+st+wait_st+signal A", "out layer + next tile's tables",
                              "loop top"};
  const char* iss_names[8] = {"wait A ready", "wait D free", "issue", "", "", "", "", ""};
  for (int blk : {0, 1, 146}) {
    printf("block %d (rank %d)\n", blk, blk & 1);
    for (int w : {0, 4, 8}) {
      const long long* p = &prof[((size_t)blk * 9 + w) * 8];
      long long tot = 0;
      for (int i = 0; i < 8; ++i) tot += p[i];
      if (!tot) continue;
      printf("  warp %d total %lld cyc:", w, tot);
      for (int i = 0; i < 8; ++i)
        if (p[i]) printf("  [%s] %.1f%%", w == 8 ? iss_names[i] : row_names[i], 100.0 * p[i] / tot);
      printf("\n");
    }
  }
  return 0;
}
