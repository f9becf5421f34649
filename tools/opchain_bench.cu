// Timing / correctness harness of the cooperative operator-chain kernel (development tool, not product code).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -DOC_TIMING -o tools/opchain_bench tools/opchain_bench.cu
#include "../mobocmf_b200/csrc/matrix_ops.cu"
#include "../mobocmf_b200/csrc/opchain.cu"
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
using namespace mobo;
int main(int argc, char** argv) {
  const int M = argc > 1 ? atoi(argv[1]) : 256, d = 6, nl = argc > 2 ? atoi(argv[2]) : 3;
  const int MP = ((M + 31) / 32) * 32;
  srand(1);
  std::vector<double> Z(M * d), th0 = {1.0, 0.3, 0.3, 0.3, 0.3, 0.3, 0.3}, m(M), Lq((size_t)M * M, 0.0);
  for (auto& v : Z) v = rand() / (double)RAND_MAX;
  for (auto& v : m) v = rand() / (double)RAND_MAX - 0.5;
  for (int i = 0; i < M; ++i) for (int j = 0; j <= i; ++j) Lq[(size_t)i * M + j] = i == j ? 0.1 : 0.01 * (rand() / (double)RAND_MAX - 0.5);
  std::vector<double> th1 = {1.0, 1.0, 1.0, 1.0, 0.01}; for (int c = 0; c < d; ++c) th1.push_back(3.0); for (int c = 0; c < d; ++c) th1.push_back(0.3);
  double *dZ, *dth0, *dth1, *dm, *dLq; cudaMalloc(&dZ, Z.size() * 8); cudaMalloc(&dth0, 64 * 8); cudaMalloc(&dth1, 64 * 8); cudaMalloc(&dm, M * 8); cudaMalloc(&dLq, Lq.size() * 8);
  cudaMemcpy(dZ, Z.data(), Z.size() * 8, cudaMemcpyHostToDevice); cudaMemcpy(dth0, th0.data(), th0.size() * 8, cudaMemcpyHostToDevice);
  cudaMemcpy(dth1, th1.data(), th1.size() * 8, cudaMemcpyHostToDevice); cudaMemcpy(dm, m.data(), M * 8, cudaMemcpyHostToDevice); cudaMemcpy(dLq, Lq.data(), Lq.size() * 8, cudaMemcpyHostToDevice);
  LayerBatch b; b.n = nl; b.d = d; b.M = M; b.MP = MP;
  std::vector<double*> ops(nl);
  for (int l = 0; l < kMaxLayers; ++l) {
    const bool ok = l < nl;
    if (ok) { cudaMalloc(&ops[l], ops_size(MP) * 8); cudaMemset(ops[l], 0xff, ops_size(MP) * 8); }
    b.kind[l] = ok && l > 0 ? 1 : 0; b.Zx[l] = dZ; b.zf[l] = dm; b.theta[l] = (ok && l > 0) ? dth1 : dth0; b.m[l] = dm; b.Lq[l] = dLq; b.ops[l] = ok ? ops[l] : nullptr;
  }
  double jitter = 1e-6;
  const int nb = MP / 32, nblk = nb * (nb + 1) / 2;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0);
    opchain_reset_kernel<<<nl, 128>>>(b);
    void* args[] = {(void*)&b, (void*)&jitter};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)opchain_kernel, dim3(nl * nblk), dim3(OC_THREADS), args, 0, 0);
    cudaEventRecord(e1); cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    printf("M=%d layers=%d CTAs=%d: %.1f us (%s)\n", M, nl, nl * nblk, ms * 1e3, cudaGetErrorString(e));
  }
#ifdef OC_TIMING
  unsigned long long t[64][8]; cudaMemcpyFromSymbol(t, oc_times, sizeof(t));
  unsigned long long t0 = ~0ull; for (int q = 0; q < nblk && q < 64; ++q) if (t[q][0] < t0) t0 = t[q][0];
  printf("layer 0 CTAs, times in us since first start: start P-done updates-done factor-done(L signalled for panels) W-done H-done stats\n");
  for (int q = 0; q < nblk && q < 64; ++q) {
    int bi = 0, rem = q; while (rem > bi) { rem -= bi + 1; ++bi; }
    printf("(%d,%d):", bi, rem); for (int k = 0; k < 7; ++k) printf(" %7.1f", (t[q][k] - t0) * 1e-3); printf("\n");
  }
#endif
  std::vector<double> out(ops_size(MP)); cudaMemcpy(out.data(), ops[nl - 1], out.size() * 8, cudaMemcpyDeviceToHost);
  const double* L = out.data() + ops_block(MP, OPS_L); const double* W = out.data() + ops_block(MP, OPS_W); const double* P = out.data() + ops_block(MP, OPS_P);
  double e1m = 0, e2m = 0;
  for (int i = 0; i < MP; ++i) for (int j = 0; j <= i; ++j) {
    double s = 0, w = 0; for (int k = 0; k < MP; ++k) { s += L[i * MP + k] * L[j * MP + k]; w += W[i * MP + k] * L[k * MP + j]; }
    e1m = fmax(e1m, fabs(s - P[i * MP + j])); e2m = fmax(e2m, fabs(w - (i == j)));
  }
  printf("max |LL^T - P| %.2e   max |WL - I| %.2e  KL %.6f status %.0f\n", e1m, e2m, out[ops_scal(MP) + SC_KL], out[ops_scal(MP) + SC_STATUS]);
  return 0;
}
