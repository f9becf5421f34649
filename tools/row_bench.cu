// Micro-benchmark of the three DMMA row kernels at the C4 upper-layer shape (development tool, not product code):
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 [-DROW_TIMING] -o tools/row_bench tools/row_bench.cu
//   tools/row_bench [R=65536] [M=256] [S=64] [reps=10]
// Prints CUDA-event times of mobo_layer_rows_fwd (training, saving t / u), the backward product + covariance-gradient
// kernels and the SYRK, their algorithmic TFLOP/s and fraction of the measured DMMA peak; with -DROW_TIMING also
// the forward kernel's per-phase cycle shares (thread 0 of every CTA, averaged).
#include <cstdlib>
#include "../mobocmf_b200/csrc/abi.cu"
#include <cstdlib>
#include <cstdio>
#include <vector>

static double* dev_rand(size_t n, double lo, double hi) {
  std::vector<double> h(n);
  for (auto& v : h) v = lo + (hi - lo) * (rand() / (double)RAND_MAX);
  double* d; cudaMalloc(&d, n * 8); cudaMemcpy(d, h.data(), n * 8, cudaMemcpyHostToDevice);
  return d;
}

int main(int argc, char** argv) {
  const long long R = argc > 1 ? atoll(argv[1]) : 65536;
  const int M = argc > 2 ? atoi(argv[2]) : 256, S = argc > 3 ? atoi(argv[3]) : 64, reps = argc > 4 ? atoi(argv[4]) : 10;
  const int d = 6, MP = ((M + 31) / 32) * 32;
  const long long B = R / S;
  srand(1);
  double* Zx = dev_rand((size_t)M * d, 0, 1);
  double* zf = dev_rand(M, -1, 1);
  std::vector<double> th = {1.0, 1.0, 1.0, 1.0, 0.01};
  for (int c = 0; c < d; ++c) th.push_back(3.0);
  for (int c = 0; c < d; ++c) th.push_back(0.3);
  double* theta; cudaMalloc(&theta, 64 * 8); cudaMemcpy(theta, th.data(), th.size() * 8, cudaMemcpyHostToDevice);
  double* m = dev_rand(M, -0.5, 0.5);
  std::vector<double> Lq((size_t)M * M, 0.0);
  for (int i = 0; i < M; ++i) for (int j = 0; j <= i; ++j) Lq[(size_t)i * M + j] = i == j ? 0.1 : 0.01 * (rand() / (double)RAND_MAX - 0.5);
  double* dLq; cudaMalloc(&dLq, Lq.size() * 8); cudaMemcpy(dLq, Lq.data(), Lq.size() * 8, cudaMemcpyHostToDevice);
  double* ops; cudaMalloc(&ops, mobo_ops_doubles(M) * 8); cudaMemset(ops, 0, mobo_ops_doubles(M) * 8);
  double* gops; cudaMalloc(&gops, mobo_ops_doubles(M) * 8); cudaMemset(gops, 0, mobo_ops_doubles(M) * 8);
  int rc = mobo_layer_precompute(1, d, M, Zx, zf, theta, m, dLq, 1e-6, ops, nullptr);
  double* x = dev_rand((size_t)B * d, 0, 1);
  double* mu_prev = dev_rand(B, -1, 1);
  double* var_prev = dev_rand(B, 0.01, 0.1);
  double* eps = dev_rand(R, -1, 1);
  double *mu, *var, *craw, *Ts, *Us, *dmu, *dvar, *df, *dtheta, *dzf, *work;
  unsigned int* clamp; cudaMalloc(&clamp, 64); cudaMemset(clamp, 0, 64);
  cudaMalloc(&mu, R * 8); cudaMalloc(&var, R * 8); cudaMalloc(&craw, R * 8); cudaMalloc(&df, R * 8);
  cudaMalloc(&Ts, mobo_rows_save_doubles(M, R) * 8); cudaMalloc(&Us, mobo_rows_save_doubles(M, R) * 8);
  dmu = dev_rand(R, -1, 1); dvar = dev_rand(R, -1, 1);
  cudaMalloc(&dtheta, 64 * 8); cudaMalloc(&dzf, MP * 8); cudaMalloc(&work, mobo_rows_bwd_work_doubles(M, R) * 8);
  cudaEvent_t e[5]; for (auto& v : e) cudaEventCreate(&v);
  float t_f = 0, t_fe = 0, t_b = 0;
  mobo_profile_enable(1);
  for (int it = 0; it < reps + 2; ++it) {
    cudaEventRecord(e[0]);
    rc |= mobo_layer_rows_fwd(1, d, M, Zx, zf, theta, ops, x, S, mu_prev, var_prev, S, eps, R, nullptr, R, 1, mu, var, craw,
                              clamp, Ts, Us, nullptr);
    cudaEventRecord(e[1]);
    rc |= mobo_layer_rows_fwd(1, d, M, Zx, zf, theta, ops, x, S, mu_prev, var_prev, S, eps, R, nullptr, R, 0, mu, var, nullptr,
                              nullptr, nullptr, nullptr, nullptr);
    cudaEventRecord(e[2]);
    rc |= mobo_layer_rows_bwd(1, d, M, Zx, zf, theta, ops, x, S, mu_prev, var_prev, S, eps, R, nullptr, R, 1, dmu, dvar, craw,
                              clamp, Ts, Us, 1, df, nullptr, dtheta, dzf, gops, work, nullptr);
    cudaEventRecord(e[3]);
    cudaEventSynchronize(e[3]);
    float a, b, c;
    cudaEventElapsedTime(&a, e[0], e[1]); cudaEventElapsedTime(&b, e[1], e[2]); cudaEventElapsedTime(&c, e[2], e[3]);
    if (it >= 2) { t_f += a; t_fe += b; t_b += c; }
  }
  const double peak = 37.1, F = 2.0 * M * M + 2.0 * M + 3.0 * (d + 1) * M;
  t_f /= reps; t_fe /= reps; t_b /= reps;
  printf("rc=%d err=%s  R=%lld M=%d S=%d\n", rc, cudaGetErrorString(cudaGetLastError()), R, M, S);
  printf("rows_fwd (train, saves t/u): %8.1f us  %6.2f TF  %.3f of peak\n", t_f * 1e3, F * R / t_f / 1e9, F * R / t_f / 1e9 / peak);
  printf("rows_fwd (eval)            : %8.1f us  %6.2f TF  %.3f of peak\n", t_fe * 1e3, F * R / t_fe / 1e9, F * R / t_fe / 1e9 / peak);
  printf("rows_bwd (all kernels)     : %8.1f us\n", t_b * 1e3);
  {
    std::vector<char> names(1 << 20); std::vector<float> ms(1 << 16);
    const int n = mobo_profile_collect(names.data(), names.size(), ms.data(), (int)ms.size());
    struct Acc { const char* name; double t; int c; }; std::vector<Acc> acc;
    const char* p = names.data();
    for (int i = 0; i < n; ++i) {
      bool hit = false;
      for (auto& a : acc) if (!strcmp(a.name, p)) { a.t += ms[i]; a.c++; hit = true; break; }
      if (!hit) acc.push_back({p, ms[i], 1});
      p += strlen(p) + 1;
    }
    const int iters = reps + 2;
    for (auto& a : acc) {
      double alg = 0;
      if (!strcmp(a.name, "row_bwd_gemm_kernel")) alg = (2.0 * M * M + 2.0 * M) * R;
      if (!strcmp(a.name, "syrk_kernel")) alg = (double)M * M * R;
      const double us = a.t / iters * 1e3;
      if (alg > 0) printf("  %-28s %8.1f us / iteration  %6.2f TF  %.3f of peak\n", a.name, us, alg / us / 1e6, alg / us / 1e6 / peak);
      else printf("  %-28s %8.1f us / iteration (%d launches)\n", a.name, us, a.c / iters);
    }
  }
  {   // SYRK alone, with and without the b = sum dmu t accumulation of set 0 (no clamp count: the clamped-rows set's
      // CTAs exit at once, as in a step where no row was clamped)
    double* part; cudaMalloc(&part, (mobo::syrk_part_doubles(MP, R) + mobo::syrk_alpha_doubles(MP, mobo::syrk_nchunk(MP, R))) * 8);
    double* pal = part + mobo::syrk_part_doubles(MP, R);
    for (int variant = 0; variant < 2; ++variant) {
      float tt = 0;
      for (int it = 0; it < reps + 2; ++it) {
        cudaEventRecord(e[0]);
        mobo::launch_syrk_both(Ts, dvar, craw, MP, R, part, nullptr, nullptr, variant ? nullptr : dmu, pal, nullptr);
        cudaEventRecord(e[1]); cudaEventSynchronize(e[1]);
        float x; cudaEventElapsedTime(&x, e[0], e[1]);
        if (it >= 2) tt += x;
      }
      tt /= reps;
      printf("syrk_kernel alone %-18s %8.1f us  %6.2f TF  %.3f of peak\n", variant ? "(no b accumulation)" : "(with b)", tt * 1e3,
             (double)M * M * R / tt / 1e9, (double)M * M * R / tt / 1e9 / peak);
    }
  }
#ifdef ROW_TIMING
  {   // backward product kernel: phases of thread 0 (rows_bwd above was the last launch of it)
    cudaDeviceSynchronize();
    static unsigned long long tb[3][512][16];
    cudaMemcpyFromSymbol(tb, mobo::row_times, sizeof(tb));
    const char* nb[8] = {"(top: row scalars -> smem)", "WAIT: staged u / t, sync", "y = H u (warp 0)", "dt, dt -> tile", "sync", "stage next tile (warp 0)", "dk = W^T dt (warp 0)", "dk stores"};
    double tt = 0, ss[8] = {0};
    for (int b = 0; b < 148; ++b) for (int k = 0; k < 8; ++k) { ss[k] += (double)tb[1][b][k]; tt += (double)tb[1][b][k]; }
    printf("backward product kernel, cycles of thread 0 summed over the CTAs: share per phase\n");
    for (int k = 0; k < 8; ++k) printf("  %-30s %6.2f %%   %9.0f cycles per CTA\n", nb[k], 100.0 * ss[k] / tt, ss[k] / 148);
  }
  {
    mobo_layer_rows_fwd(1, d, M, Zx, zf, theta, ops, x, S, mu_prev, var_prev, S, eps, R, nullptr, R, 1, mu, var, craw, clamp,
                        Ts, Us, nullptr);
    cudaDeviceSynchronize();
    static unsigned long long t[3][512][16];
    cudaMemcpyFromSymbol(t, mobo::row_times, sizeof(t));
    const char* names[12] = {"load_inducing (once)", "load_tile_rows+sync", "build K", "sync after build", "gemm1 (warp 0)",
                             "sums after gemm1", "sync (K free)", "t -> tile + sync", "gemm2 (warp 0)", "sums + U stores",
                             "sync", "epilogue + bulk wait + sync"};
    const bool pp = S >= mobo::XSHARE_MIN_REP;   // product warps of the warp-specialised kernel
    const char* pp_names[12] = {"setup (once)", "WAIT: K ready", "gemm1 (warp 0)", "sync, t -> tile, sync, signal",
                                "gemm2 (warp 0)", "WAIT: t sums / store done", "u -> tile, sync, signal", "-", "-", "-", "-", "-"};
    if (pp) for (int k = 0; k < 12; ++k) names[k] = pp_names[k];
    const int grid = pp ? 148 : 148 * mobo::ROW_CTAS_PER_SM;
    double tot = 0, s[12] = {0};
    for (int b = 0; b < grid; ++b) for (int k = 0; k < 12; ++k) { s[k] += (double)t[0][b][k]; tot += (double)t[0][b][k]; }
    printf("forward kernel (training launch: saves t / u), cycles of thread 0 summed over %d CTAs: share per phase\n", grid);
    for (int k = 0; k < 12; ++k) printf("  %-30s %6.2f %%   %9.0f cycles per CTA\n", names[k], 100.0 * s[k] / tot, s[k] / grid);
    if (pp) {
      const char* bnames[10] = {"(loop top)", "WAIT: buffer free", "stage 2: K of tile i", "sync, signal K ready", "stage 1: x-kernels of tile i+1", "sync", "-", "-", "-", "-"};
      const char* fnames[10] = {"(loop top)", "WAIT: t ready", "t sums", "bulk wait t, signal", "WAIT: u ready", "u sums, epilogue", "bulk wait u, signal", "-", "-", "-"};
      for (int w = 1; w <= 2; ++w) {
        double tt = 0, ss[10] = {0};
        for (int b = 0; b < grid; ++b) for (int k = 0; k < 10; ++k) { ss[k] += (double)t[w][b][k]; tt += (double)t[w][b][k]; }
        printf("%s warps (thread 0 of the role):\n", w == 1 ? "build" : "finish");
        for (int k = 0; k < 10; ++k) printf("  %-30s %6.2f %%   %9.0f cycles per CTA\n", w == 1 ? bnames[k] : fnames[k], 100.0 * ss[k] / tt, ss[k] / grid);
      }
    }
  }
#endif
  return 0;
}
