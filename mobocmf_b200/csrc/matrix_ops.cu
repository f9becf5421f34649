// Per-step M x M operator chain of the sparse-GP layers (forward and backward) for sm_100a.
//
// Forward (what the reference reaches through UnwhitenedVariationalStrategy.forward / kl_mvn_mvn [upstream gpytorch],
// called from mobocmf/layers/mfdgp_hidden_layer.py:286 and mobocmf/mlls/variational_elbo_mf.py:40):
//   P = K(Z_l, Z_l) + jitter I      (CovarianceMatrixMF.add_jitter, layers/mfdgp_hidden_layer.py:17-20)
//   L = chol(P);  W = L^-1;  H = W tril(L_q);  beta = W m
//   KL = 1/2 [ 2 sum log L_ii - sum log L_q,ii^2 + |beta|^2 + |H|_F^2 - M ]
// Backward: the loss depends on P only through P^-1 = W^T W and P^-1 S P^-1 = W^T G2 W (G2 = H H^T), so with the
// row pass's WHITENED statistics A2 = sum dvar t t^T (A1 = A2 minus the clamped rows), b = sum dmu t (t = W k) and
// g = dLoss/dKL everything is assembled in whitened space (moderate magnitudes) and mapped back by one congruence:
//   dP  = W^T [ A1 - A2 G2 - G2 A2 - 1/2 (beta b^T + b beta^T) + g/2 (I - beta beta^T - G2) ] W
//   dLq = tril(W^T (2 A2 + g I) H) - g diag(1 / L_q,ii),      dm = W^T (b + g beta)
// (no differentiation through the Cholesky factor is needed), then dP goes through K(Z,Z) to d theta and d zf —
// the gradient through the inducing inputs [Z, m_{l-1}] (SURVEY.md §7).
//
// All matrices are MP x MP row-major (MP = M rounded up to 32, identity/zero padded) and L2-resident; products run
// on the DMMA pipe.  The layers' chains are independent: the forward of all layers of a model is one launch
// (opchain.cu, LayerBatch); the backward below is enqueued one layer at a time.
#include "common.cuh"

namespace mobo {

struct LayerBatch {
  int n;
  int d, M, MP;
  int kind[kMaxLayers];
  const double* Zx[kMaxLayers];
  const double* zf[kMaxLayers];
  const double* theta[kMaxLayers];
  const double* m[kMaxLayers];
  const double* Lq[kMaxLayers];
  double* ops[kMaxLayers];
};

// backward through K(Z,Z): dP symmetric.  One warp per inducing point i.
//   dtheta += sum_ij dP_ij dk_ij/dtheta ;  dzf_i = 2 sum_j dP_ij dk(z_i,z_j)/d f_i
//   part_theta: [gridDim.x][kMaxTheta];  dzf: M or NULL
constexpr int KZB_WARPS = 8;
__global__ void __launch_bounds__(KZB_WARPS * 32)
kzz_bwd_kernel(int kind, int d, int M, int MP, const double* Zx, const double* zf, const double* theta,
               const double* dP, double* part_theta, double* dzf) {
  __shared__ KernParams kp;
  __shared__ double accw[KZB_WARPS][kMaxTheta];
  if (threadIdx.x == 0) load_kern_params(kp, kind, d, theta);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * KZB_WARPS + warp;
  double th_s[5], th_l1[kMaxD], th_l2[kMaxD];
#pragma unroll
  for (int q = 0; q < 5; ++q) th_s[q] = 0.0;
#pragma unroll
  for (int c = 0; c < kMaxD; ++c) { th_l1[c] = 0.0; th_l2[c] = 0.0; }
  double dzi = 0.0;
  if (i < M) {
    const double fi = kind == 1 ? zf[i] : 0.0;
    double zi[kMaxD];
#pragma unroll
    for (int c = 0; c < kMaxD; ++c) zi[c] = c < d ? Zx[(size_t)i * d + c] : 0.0;
    for (int j = lane; j < M; j += 32) {
      const double gk = dP[(size_t)i * MP + j];
      if (i == j) {
        if (kind == 0) {
          th_s[0] += gk;
        } else {
          th_s[0] += gk * (kp.vlin * fi * fi + kp.af);
          th_s[1] += gk * kp.a1 * fi * fi;
          th_s[2] += gk * kp.a1;
          th_s[4] += gk;
          dzi += gk * kp.a1 * kp.vlin * fi;     // doubled below -> 2 a1 v f
        }
        continue;
      }
      double D1 = 0.0, D2 = 0.0, diff[kMaxD];
#pragma unroll
      for (int c = 0; c < kMaxD; ++c) {
        diff[c] = c < d ? zi[c] - Zx[(size_t)j * d + c] : 0.0;
        D1 = fma(diff[c] * diff[c], kp.il1[c], D1);
        D2 = fma(diff[c] * diff[c], kp.il2[c], D2);
      }
      const double E1 = exp(-0.5 * D1);
      if (kind == 0) {
        const double gkk = gk * kp.a1 * E1;
        th_s[0] = fma(gk, E1, th_s[0]);
#pragma unroll
        for (int c = 0; c < kMaxD; ++c) th_l1[c] = fma(gkk, diff[c] * diff[c], th_l1[c]);
      } else {
        const double fj = zf[j], dff = fi - fj;
        const double Ef = exp(-0.5 * dff * dff * kp.ilf), E2 = exp(-0.5 * D2);
        const double gg = kp.vlin * fi * fj + kp.af * Ef;
        const double s1 = kp.a1 * E1, s2 = kp.a2 * E2;
        const double dEf = s1 * kp.af * Ef * dff * kp.ilf;
        dzi = fma(gk, s1 * kp.vlin * fj - dEf, dzi);
        th_s[0] = fma(gk, E1 * gg, th_s[0]);
        th_s[1] = fma(gk, s1 * fi * fj, th_s[1]);
        th_s[2] = fma(gk, s1 * Ef, th_s[2]);
        th_s[3] = fma(gk, dEf * dff, th_s[3]);
        th_s[4] = fma(gk, E2, th_s[4]);
        const double g1 = gk * s1 * gg, g2 = gk * s2;
#pragma unroll
        for (int c = 0; c < kMaxD; ++c) {
          const double d2 = diff[c] * diff[c];
          th_l1[c] = fma(g1, d2, th_l1[c]);
          th_l2[c] = fma(g2, d2, th_l2[c]);
        }
      }
    }
  }
  dzi = warp_sum(dzi);
  if (lane == 0 && i < M && kind == 1 && dzf) dzf[i] = 2.0 * dzi;
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const double s = warp_sum(th_s[q]);
    if (lane == 0) accw[warp][q] = s;
  }
#pragma unroll
  for (int c = 0; c < kMaxD; ++c) {
    double s = warp_sum(th_l1[c]);
    if (lane == 0) accw[warp][5 + c] = s;
    s = warp_sum(th_l2[c]);
    if (lane == 0) accw[warp][5 + kMaxD + c] = s;
  }
  __syncthreads();
  const int tid = threadIdx.x;
  if (tid < kMaxTheta) {
    double s = 0.0;
    for (int w = 0; w < KZB_WARPS; ++w) s += accw[w][tid];
    double out = 0.0;
    int slot = -1;
    if (kind == 0) {
      if (tid == 0) { slot = 0; out = s; }
      else if (tid >= 5 && tid < 5 + d) { slot = 1 + (tid - 5); out = s * kp.il1[tid - 5] * sqrt(kp.il1[tid - 5]); }
    } else {
      if (tid < 5) { slot = tid; out = tid == 3 ? s * sqrt(kp.ilf) : s; }
      else if (tid < 5 + d) { slot = tid; out = s * kp.il1[tid - 5] * sqrt(kp.il1[tid - 5]); }
      else if (tid >= 5 + kMaxD && tid < 5 + kMaxD + d) {
        const int c = tid - 5 - kMaxD;
        slot = 5 + d + c;
        out = s * kp.il2[c] * sqrt(kp.il2[c]);
      }
    }
    if (slot >= 0) part_theta[(size_t)blockIdx.x * kMaxTheta + slot] = out;
  }
}

// out[i] = sum_b part[b][i], i < n  (sequential in b: a fixed order)
__global__ void reduce_batch_kernel(const double* part, int nblocks, int stride, int n, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0.0;
  for (int b = 0; b < nblocks; ++b) s += part[(size_t)b * stride + i];
  out[i] = s;
}

// ---------------------------------------------------------------------------------------------------
// 32 x 32 Cholesky factor in registers of one warp (lane = row, columns exchanged by shuffles); used by the
// diagonal CTAs of the operator-chain kernel (opchain.cu).
// ---------------------------------------------------------------------------------------------------

__device__ __forceinline__ void chol32_inwarp(double (&row)[32], double& rinv, int lane, int& fail) {
  // row[c] = A[lane][c] (lower part valid).  On exit row[c] = L[lane][c] for c <= lane and rinv = 1 / L[lane][lane].
  // Right-looking; the pivot's reciprocal square root (1 ulp) replaces the square root and the division of the
  // textbook form, which sit on the critical path of the whole operator chain.
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const double djj = __shfl_sync(0xffffffffu, row[j], j);
    if (!(djj > 0.0)) fail = 1;
    const double r = rsqrt(djj);
    if (lane == j) { row[j] = djj * r; rinv = r; }
    else if (lane > j) row[j] = row[j] * r;
#pragma unroll
    for (int c = j + 1; c < 32; ++c) {
      const double lcj = __shfl_sync(0xffffffffu, row[j], c);   // L[c][j]
      if (lane >= c) row[c] = fma(-row[j], lcj, row[c]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// strided GEMM  C = op(A) op(B)  (n x n x n, n multiple of 32), 32x32 tiles, BK = 32,
// register-prefetched double buffering.  Triangular operands shorten the k range:
//   a_tri: 1 = op(A)[m][k] == 0 for k > m (lower), 2 = == 0 for k < m (upper);  b_tri likewise on op(B)[k][n]:
//   1 = lower (== 0 for n > k), 2 = upper (== 0 for n < k).
// element (m,k) of op(A) = A[m*rsA + k*csA];  element (k,n) of op(B) = B[k*rsB + n*csB]
// ---------------------------------------------------------------------------------------------------
constexpr int GM_T = 32, GM_K = 32, GM_THREADS = 128, GM_LD = GM_T + 4;

struct GemmArgs {
  int n;
  int rsA, csA, rsB, csB;
  int a_tri, b_tri;
  const double* A;
  const double* B;
  double* C;
};

__global__ void __launch_bounds__(GM_THREADS) gemm_kernel(const __grid_constant__ GemmArgs a) {
  __shared__ double As[2][GM_K][GM_LD];   // [k][m]
  __shared__ double Bs[2][GM_K][GM_LD];   // [k][n]
  const double* __restrict__ A = a.A;
  const double* __restrict__ B = a.B;
  double* __restrict__ C = a.C;
  const int n = a.n;
  const int m0 = blockIdx.y * GM_T, n0 = blockIdx.x * GM_T;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int wi = warp >> 1, wj = warp & 1;          // 16 x 16 per warp
  int kbeg = 0, kend = n;
  if (a.a_tri == 1) kend = min(kend, m0 + GM_T);
  if (a.a_tri == 2) kbeg = max(kbeg, m0);
  if (a.b_tri == 1) kbeg = max(kbeg, n0);
  if (a.b_tri == 2) kend = min(kend, n0 + GM_T);
  double acc[2][2][2] = {};
  // each thread moves 8 elements of each operand per k-tile; index order chosen so global reads coalesce
  double ra[8], rb[8];
  auto gload = [&](int k0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int idx = tid + q * GM_THREADS;
      int kk, mm, kb, nn;
      if (a.csA == 1) { mm = idx >> 5; kk = idx & 31; } else { kk = idx >> 5; mm = idx & 31; }
      if (a.rsB == 1) { nn = idx >> 5; kb = idx & 31; } else { kb = idx >> 5; nn = idx & 31; }
      ra[q] = A[(size_t)(m0 + mm) * a.rsA + (size_t)(k0 + kk) * a.csA];
      rb[q] = B[(size_t)(k0 + kb) * a.rsB + (size_t)(n0 + nn) * a.csB];
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int idx = tid + q * GM_THREADS;
      int kk, mm, kb, nn;
      if (a.csA == 1) { mm = idx >> 5; kk = idx & 31; } else { kk = idx >> 5; mm = idx & 31; }
      if (a.rsB == 1) { nn = idx >> 5; kb = idx & 31; } else { kb = idx >> 5; nn = idx & 31; }
      As[buf][kk][mm] = ra[q];
      Bs[buf][kb][nn] = rb[q];
    }
  };
  if (kbeg < kend) {
    gload(kbeg);
    sstore(0);
    __syncthreads();
    int buf = 0;
    for (int k0 = kbeg; k0 < kend; k0 += GM_K) {
      const bool more = k0 + GM_K < kend;
      if (more) gload(k0 + GM_K);
#pragma unroll
      for (int kk = 0; kk < GM_K; kk += 4) {
        double af[2], bf[2];
#pragma unroll
        for (int x = 0; x < 2; ++x) af[x] = As[buf][kk + t][16 * wi + 8 * x + g];
#pragma unroll
        for (int y = 0; y < 2; ++y) bf[y] = Bs[buf][kk + t][16 * wj + 8 * y + g];
#pragma unroll
        for (int x = 0; x < 2; ++x)
#pragma unroll
          for (int y = 0; y < 2; ++y) dmma884(acc[x][y][0], acc[x][y][1], af[x], bf[y]);
      }
      if (more) sstore(buf ^ 1);
      __syncthreads();
      buf ^= 1;
    }
  }
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int i = m0 + 16 * wi + 8 * x + g, j = n0 + 16 * wj + 8 * y + 2 * t + e;
        C[(size_t)i * n + j] = acc[x][y][e];
      }
}

// an operand of gemm(): op(p) = p^T when trans; tri as a_tri / b_tri above
struct GemmOperand { const double* p; bool trans; int tri; };

static int gemm(int n, const GemmOperand& A, const GemmOperand& B, double* C, cudaStream_t st) {
  GemmArgs a;
  a.n = n;
  a.rsA = A.trans ? 1 : n; a.csA = A.trans ? n : 1;
  a.rsB = B.trans ? 1 : n; a.csB = B.trans ? n : 1;
  a.a_tri = A.tri; a.b_tri = B.tri;
  a.A = A.p; a.B = B.p; a.C = C;
  MOBO_LAUNCH("gemm_kernel", st, gemm_kernel<<<dim3(n / GM_T, n / GM_T), GM_THREADS, 0, st>>>(a));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// dm = W^T (b + g beta).  Warp per row of W^T.
__global__ void __launch_bounds__(256) white_vec_kernel(const double* WT, const double* b, const double* beta,
                                                        const double* dkl, double* dm, int M, int MP) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * 8 + warp;
  if (j >= M) return;
  const double* row = WT + (size_t)j * MP;
  const double g = dkl[0];
  double s = 0.0;
  for (int i = j + lane; i < MP; i += 32) s = fma(row[i], b[i] + g * beta[i], s);
  s = warp_sum(s);
  if (lane == 0) dm[j] = s;
}

// whitened gradient core  N = A1 - V - V^T - 1/2 (beta b^T + b beta^T) + g/2 (I - beta beta^T - G2)  (dP = W^T N W)
// and F = 2 A2 + g I  (dLq = tril(W^T F H) - g diag(1/Lq_ii));  A1 = A2 - Ac when some row was clamped.
//   clamp_flag: number of clamped rows (scal[SC_CLAMP] of the gradient buffer)
__global__ void combine_kernel(const double* A2, const double* Ac, const double* V, const double* G2, const double* b,
                               const double* beta, const double* dkl, const double* clamp_flag, double* N, double* F,
                               int MP) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= MP * MP) return;
  const int i = idx / MP, j = idx - i * MP;
  const size_t tr = (size_t)j * MP + i;
  const double g = dkl[0];
  const bool clamped = *clamp_flag != 0.0;
  const double a2 = 0.5 * (A2[idx] + A2[tr]);
  const double a1 = clamped ? a2 - 0.5 * (Ac[idx] + Ac[tr]) : a2;
  const double bi_ = b[i], bj_ = b[j], be_i = beta[i], be_j = beta[j];
  const double eye = i == j ? 1.0 : 0.0;
  N[idx] = a1 - V[idx] - V[tr] - 0.5 * (be_i * bj_ + bi_ * be_j) + 0.5 * g * (eye - be_i * be_j - G2[idx]);
  F[idx] = 2.0 * a2 + g * eye;
}

// dLq (M x M, ld M) = tril(E)[:M,:M] - g diag(1 / Lq_ii)
__global__ void dlq_extract_kernel(const double* E, const double* LQ, const double* dkl, double* dLq, int M, int MP) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * M) return;
  const int i = idx / M, j = idx - i * M;
  double v = j <= i ? E[(size_t)i * MP + j] : 0.0;
  if (i == j) v -= dkl[0] / LQ[(size_t)i * MP + i];
  dLq[idx] = v;
}

}  // namespace mobo
